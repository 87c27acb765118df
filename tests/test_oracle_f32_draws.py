"""The float64 restatement of the fp32 draw contract (oracle/f32_draws.py), checked without a GPU: its vectorised
Philox word for word against the C oracle, its transforms against scipy and the fp64 Box-Muller, its retry rule against
the reference's control flow."""
import numpy as np
import pytest
from scipy import special

from oracle import c_oracle, dr_port, f32_draws


def test_vectorised_philox_matches_the_c_oracle_word_for_word():
    rs = np.random.RandomState(0)
    ctr = rs.randint(0, 2 ** 32, size=(4, 200), dtype=np.uint64)
    ctr[:, :4] = [[0, 0xFFFFFFFF, 0, 1], [0, 0xFFFFFFFF, 0xFFFFFFFF, 0], [0, 0xFFFFFFFF, 5, 7], [0, 0xFFFFFFFF, 0, 3]]
    for key in ((0, 0), (0xFFFFFFFF, 0xFFFFFFFF), (123456789, 987654321)):
        got = f32_draws.philox(*ctr, *key)
        for i in range(ctr.shape[1]):
            want = c_oracle.philox(tuple(int(v) for v in ctr[:, i]), key)
            assert tuple(int(w[i]) for w in got) == want, (key, i)


@pytest.mark.parametrize("sample_id,tick", [(0, 0), (5, 1), ((1 << 32) + 9, 3), (77, (1 << 32) + 2), ((3 << 40) + 1, (5 << 36) + 11)])
def test_draw_block_follows_the_counter_layout_of_the_c_oracle(sample_id, tick):
    """ids and ticks above 2^32 included: their high words share counter word 1."""
    seed = (7 << 32) | 99
    for purpose in (f32_draws.PURPOSE_XI, f32_draws.PURPOSE_TASKS):
        for attempt in range(3):
            u = c_oracle.uniforms(seed, sample_id, tick, purpose, attempt, 12, np.float32)
            for j in range(3):
                w = f32_draws.draw_block(seed, [sample_id], tick, purpose, attempt * 16 + j)
                mine = np.array([(int(v[0]) >> 8) * 2.0 ** -24 for v in w], np.float32)
                assert np.array_equal(mine, u[4 * j:4 * j + 4]), (purpose, attempt, j)


def test_transforms_match_scipy_and_the_fp64_box_muller():
    r = np.random.RandomState(1).randint(0, 2 ** 32, size=5000, dtype=np.uint64).astype(np.uint32)
    r[:4] = [0, 0xFFFFFFFF, 0x80000000, 255]
    u = (r >> 8).astype(np.float64) * 2.0 ** -24
    assert np.max(np.abs(f32_draws.tn_z(r) - dr_port.truncnorm_ppf(u, 0.0, 1.0))) < 1e-13
    assert f32_draws.tn_z(np.uint32(0)) == pytest.approx(-2.0, abs=1e-12)
    assert np.all(np.abs(f32_draws.tn_z(r)) <= 2.0 + 1e-12)
    rb = r[::-1].copy()
    z0, z1, b0, b1 = f32_draws.normal_pair(r, rb)
    w0, w1 = dr_port.box_muller_f64(u + 2.0 ** -24, (rb >> 8).astype(np.float64) * 2.0 ** -24 - 0.5)
    assert np.max(np.abs(z0 - w0)) < 1e-12 and np.max(np.abs(z1 - w1)) < 1e-12
    # the radius reaches 0 (u1 = 1) and sqrt(48 ln 2) (u1 = 2^-24); the bound covers radius, angle and the product
    assert f32_draws.radius(np.uint32(0xFFFFFFFF)) == 0.0
    assert f32_draws.radius(np.uint32(0)) == pytest.approx(np.sqrt(48 * np.log(2.0)), rel=1e-15)
    assert np.all(b0 >= f32_draws.RADIUS_BOUND) and np.all(b0 <= 1e-5)


def test_retry_rule_and_ambiguity():
    """First of attempts 0..2 at or above the floor, else the floor; a give-up is flagged; draws near the floor are
    ambiguous and carry every candidate."""
    seed, ids = 5, np.arange(20000, dtype=np.uint64)
    mean, std = np.array([0.1, 1.0, 0.3, 2.0, 0.1]), np.array([1.0, 0.1, 0.5, 0.01, 0.01])
    floor = np.array([0.5, 0.9, 0.2, 1.0, 0.1])
    ref = f32_draws.sample_dr("truncnorm", seed, ids, 3, f32_draws.PURPOSE_TASKS, mean, std, floor)
    v, cand = ref["value"], ref["candidates"]
    for i in (0, 1, 17, 19999):
        for d in range(5):
            want = dr_port.sample_truncnorm_dim(None, None, float(np.float32(floor[d])),
                                                iter(list(cand[i, d, :3]) + [np.nan]).__next__)
            assert v[i, d] == want
    assert np.all(v >= f32_draws.f32(floor))
    # dim 0: an attempt falls below the floor with p = P(TN(-2, 2) < 0.4); all three do with p^3
    p = (special.ndtr(0.4) - special.ndtr(-2.0)) / (special.ndtr(2.0) - special.ndtr(-2.0))
    assert abs(np.mean(ref["gave_up"][:, 0]) - p ** 3) < 0.01
    assert np.mean(ref["ambiguous"]) < 1e-4
    # a floor placed on an attempt's value makes exactly the draws that reach that attempt ambiguous
    fl = floor.copy(); fl[1] = float(np.float32(cand[0, 1, 0]))
    amb = f32_draws.sample_dr("truncnorm", seed, ids[:1], 3, f32_draws.PURPOSE_TASKS, mean, std, fl)["ambiguous"]
    assert amb[0, 1] and not amb[0, [0, 2, 3]].any()
    g = f32_draws.sample_dr("gaussian", seed, ids, 3, f32_draws.PURPOSE_TASKS, mean[:4], std[:4], np.full(4, 0.1))
    assert np.all(g["bound"][~g["gave_up"]] > 0) and np.all(g["bound"][~g["gave_up"]] < 1e-5)
