"""T0: pin the oracle restatements (Python port, C port) to the REAL reference.

Live against /root/reference when it is mounted, and against tests/golden/ (produced by
oracle/make_golden.py from the real reference) everywhere else.  Bit-exact: `==`, not allclose.
"""
import json
import math
import os

import numpy as np
import pytest

from oracle import c_oracle, cartpole_port as port, reference_loader as rl

needs_ref = pytest.mark.skipif(not rl.available(), reason=rl.UNAVAILABLE)


def _episodes(t):
    off = 0
    for e in range(len(t["length"])):
        T = int(t["length"][e])
        yield e, slice(off, off + T)
        off += T


def test_known_answers_port_and_c(golden_dir):
    rows = json.load(open(os.path.join(golden_dir, "cartpole_known_answers.json")))
    assert len(rows) == 8
    for r in rows:
        s0 = tuple(float(v) for v in r["s0"])
        want = tuple(float(v) for v in r["s1"])
        euler = r["integrator"] == "euler"
        got, term = port.dynamics_step(s0, tuple(r["xi"]), r["action"], euler)
        assert got == want and term == r["done"]
        st = np.array(s0, np.float64).reshape(4, 1).copy()
        term_c = c_oracle.step_batch(st, np.array(r["xi"]).reshape(4, 1), np.array([r["action"]], np.uint8), euler)
        assert tuple(st[:, 0]) == want and bool(term_c[0]) == r["done"]
        assert r["polemass_length"] == 0.05       # SURVEY section 0.4: stale after set_task


def test_survey_table_row():
    """First row of SURVEY.md section 8c, typed in by hand (independent of the generated json)."""
    s0 = (0.004881350392732478, 0.021518936637241942, 0.010276337607164385, 0.004488318299689688)
    got, term = port.dynamics_step(s0, port.NOMINAL_TASK, 1, True)
    assert got == (0.005311729125477317, 0.21649201419928263, 0.010366103973158179, -0.28493466577473725)
    assert not term


def test_golden_trajectories_bit_exact(golden_traj):
    t = golden_traj
    n_steps = 0
    for e, sl in _episodes(t):
        s = tuple(t["s0"][e])
        xi = tuple(t["xi"][e])
        sc = np.array(s).reshape(4, 1).copy()
        xic = np.array(xi).reshape(4, 1)
        for k in range(sl.start, sl.stop):
            s, term = port.dynamics_step(s, xi, int(t["actions"][k]), bool(t["euler"][e]))
            term_c = c_oracle.step_batch(sc, xic, t["actions"][k:k + 1], bool(t["euler"][e]))
            assert s == tuple(t["states"][k]), (e, k)
            assert tuple(sc[:, 0]) == tuple(t["states"][k]), (e, k)
            assert term == bool(t["dones"][k]) == bool(term_c[0])
            assert t["rewards"][k] == 1.0
            n_steps += 1
        assert bool(t["dones"][sl.stop - 1]) or (sl.stop - sl.start) == 500
    assert n_steps == len(t["actions"]) > 4000


def test_beyond_done_reward_rule(golden_dir):
    g = np.load(os.path.join(golden_dir, "cartpole_beyond_done.npz"))
    env = port.CartPolePort()
    env.state = tuple(g["s0"]); env.set_task(*g["xi"])
    for k in range(len(g["actions"])):
        obs, r, d, _ = env.step(int(g["actions"][k]))
        assert tuple(obs) == tuple(g["states"][k])
        assert r == g["rewards"][k] and d == bool(g["dones"][k])
        assert (-1 if env.steps_beyond_done is None else env.steps_beyond_done) == g["beyond"][k]
    # the scenario leaves, re-enters (reward 1.0 again, done False) and leaves the thresholds
    assert list(g["rewards"][:6]) == [1, 1, 0, 0, 0, 1]


def test_timelimit_survivor(golden_dir):
    g = np.load(os.path.join(golden_dir, "cartpole_timelimit.npz"))
    env = port.TimeLimitPort(port.CartPolePort())
    env.env.seed(0)
    env.reset()
    env.env.state = tuple(g["s0"]); env.set_task(*g["xi"])
    for k in range(500):
        obs, r, d, info = env.step(int(g["actions"][k]))
        assert tuple(obs) == tuple(g["states"][k])
        if k < 499:
            assert not d and "TimeLimit.truncated" not in info
    assert d and info["TimeLimit.truncated"] is True
    # C closed loop reproduces it with its own in-loop policy (left-to-right dot product)
    st = g["s0"].reshape(4, 1).copy(); xi = g["xi"].reshape(4, 1).copy()
    el = np.zeros(1, np.int32); ep = np.ones(1, np.uint32)
    out = c_oracle.closed_loop(st, xi, el, ep, seed=7, env_id0=0, tick0=1, K=500, w=g["w"], b=0.0, log=True)
    assert np.array_equal(out["states"][:499, :, 0], g["states"][:499])
    assert out["done"][:499].sum() == 0 and out["done"][499, 0] and out["truncated"][499, 0]
    assert list(out["stats"]) == [1.0, 500.0, 250000.0, 500.0, 500.0, 500.0]
    assert ep[0] == 2 and el[0] == 0


def test_action_check_matches_gym_021():
    env = port.CartPolePort(); env.state = (0.0, 0.0, 0.0, 0.0)
    env.step(1); env.step(np.int64(0))
    for bad in (2, -1, 1.0, np.float32(1.0), "1"):
        with pytest.raises(AssertionError):
            env.step(bad)


def test_constants(golden_dir):
    assert port.THETA_THRESHOLD == 0.20943951023931953
    assert port.POLEMASS_LENGTH == 0.05
    assert port.SEARCH_BOUNDS == ((2.0, 20.0), (0.5, 3.0), (0.05, 0.3), (0.1, 1.0))
    # the reference's own get_task_lower_bound(i), recorded by oracle/make_golden.py
    ref_lb = np.load(os.path.join(golden_dir, "sampler_reference_draws.npz"))["truncnorm_lb"]
    assert tuple(float(v) for v in ref_lb) == tuple(port.LOWER_BOUNDS)


def test_philox_known_answers():
    """Random123 kat vectors for philox4x32-10."""
    assert c_oracle.philox((0, 0, 0, 0), (0, 0)) == (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)
    assert c_oracle.philox((0xffffffff,) * 4, (0xffffffff,) * 2) == (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)
    assert c_oracle.philox((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == \
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)


def test_c_draw_spec():
    s = c_oracle.init_state(3, 11, 1)
    assert s.shape == (4,) and np.all(s >= -0.05) and np.all(s < 0.05)
    assert not np.array_equal(s, c_oracle.init_state(3, 11, 2))
    assert not np.array_equal(s, c_oracle.init_state(3, 12, 1))
    # 48-bit env ids and 48-bit ticks both reach the Philox counter
    assert not np.array_equal(c_oracle.init_state(3, 11, 5), c_oracle.init_state(3, 11, (1 << 32) + 5))
    assert not np.array_equal(c_oracle.init_state(3, 11, 5), c_oracle.init_state(3, (1 << 32) + 11, 5))
    assert not np.array_equal(c_oracle.init_state(3, (1 << 32) + 11, 5), c_oracle.init_state(3, 11, (1 << 32) + 5))
    s32 = c_oracle.init_state(3, 11, 1, np.float32)
    assert s32.dtype == np.float32 and np.all(np.abs(s32) <= 0.05)
    a = c_oracle.random_actions(4096, 0, 0, 0)
    assert set(np.unique(a)) == {0, 1} and 0.45 < a.mean() < 0.55
    # sharding invariance of the action stream: a shard starting at env 1000 sees the same bits
    assert np.array_equal(c_oracle.random_actions(500, 1000, 0, 5), c_oracle.random_actions(1500, 0, 0, 5)[1000:])


# ------------------------------------------------------------------ live against the real reference
@needs_ref
def test_reference_quirks_still_there():
    env = rl.make_cartpole()
    env.set_task(5.0, 2.0, 0.2, 0.8)
    assert env.polemass_length == 0.05 and env.total_mass == 2.2          # section 0.4
    env.set_dr_distribution("uniform", [2, 20, 0.5, 3, 0.05, 0.3, 0.1, 1.0])
    env.set_dr_training(True)
    before = env.get_task().copy()
    env.reset()
    assert np.array_equal(env.get_task(), before)                          # section 0.5: no resample on reset
    assert env.theta_threshold_radians == port.THETA_THRESHOLD and env.x_threshold == port.X_THRESHOLD
    assert (env.force_mag, env.tau, env.kinematics_integrator) == (port.FORCE_MAG, port.TAU, "euler")
    for i in range(4):
        assert env.get_search_bounds_mean(i) == port.SEARCH_BOUNDS[i]
        assert env.get_task_lower_bound(i) == port.LOWER_BOUNDS[i]


@needs_ref
def test_port_and_c_vs_live_reference_random_policy():
    rs = np.random.RandomState(99)
    lo = np.array([b[0] for b in port.SEARCH_BOUNDS]); hi = np.array([b[1] for b in port.SEARCH_BOUNDS])
    steps = 0
    for e in range(300):
        env = rl.make_cartpole()
        euler = bool(e % 2)
        env.kinematics_integrator = "euler" if euler else "semi"
        xi = lo + (hi - lo) * rs.uniform(size=4)
        s0 = rs.uniform(-0.05, 0.05, 4)
        env.state = s0.copy(); env.steps_beyond_done = None; env.set_task(*xi)
        s = tuple(s0); sc = s0.reshape(4, 1).copy(); xic = xi.reshape(4, 1).copy()
        for k in range(500):
            a = int(rs.randint(2))
            obs, r, d, _ = env.step(a)
            s, term = port.dynamics_step(s, tuple(xi), a, euler)
            tc = c_oracle.step_batch(sc, xic, np.array([a], np.uint8), euler)
            assert tuple(obs) == s == tuple(sc[:, 0]) and d == term == bool(tc[0])
            steps += 1
            if d:
                break
    assert steps > 5000


def test_port_episode_length_law_matches_the_references_demo_loop(golden_dir):
    """The Python port under the SyncVectorEnv-style harness (the CPU baseline of bench.py) reproduces the law of the
    reference's own demo loop: 4 000 port episodes vs the 20 000 golden ones, two-sample KS at alpha = 0.001."""
    import math
    import os
    from oracle import dr_port
    ref = np.load(os.path.join(golden_dir, "cartpole_episode_lengths.npz"))["euler"].astype(np.float64)
    lo = np.array([b[0] for b in port.SEARCH_BOUNDS]); hi = np.array([b[1] for b in port.SEARCH_BOUNDS])
    rs = np.random.RandomState(5)
    env = port.TimeLimitPort(port.CartPolePort())
    env.env.seed(5)
    got = []
    for _ in range(4000):
        env.set_task(*dr_port.sample_task("uniform", lo, hi, rng=rs))
        env.reset()
        T = 0
        while True:
            _, _, d, _ = env.step(int(rs.randint(2)))
            T += 1
            if d:
                break
        got.append(T)
    got = np.array(got, np.float64)
    grid = np.arange(1, 501)
    d = np.max(np.abs(np.searchsorted(np.sort(got), grid, side="right") / got.size
                      - np.searchsorted(np.sort(ref), grid, side="right") / ref.size))
    assert d < 1.95 * math.sqrt((got.size + ref.size) / (got.size * ref.size)), d
    assert abs(got.mean() - ref.mean()) < 5 * math.sqrt(ref.var() / ref.size + got.var() / got.size)
