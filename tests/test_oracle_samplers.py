"""T0 for the DR samplers: the port's control flow and target laws vs the REAL reference.

Golden inputs: tests/golden/sampler_control_flow.json (scripted draws through the reference's own
retry loops) and sampler_reference_draws.npz (iid draws of the reference's sample_task).
"""
import json
import os

import numpy as np
import pytest
from scipy import stats

from oracle import dr_port, reference_loader as rl

needs_ref = pytest.mark.skipif(not rl.available(), reason=rl.UNAVAILABLE)


def _script(values):
    it = iter(values)
    used = [0]

    def draw():
        used[0] += 1
        return next(it)
    return draw, used


def test_retry_loops_match_reference_known_answers(golden_dir):
    rows = json.load(open(os.path.join(golden_dir, "sampler_control_flow.json")))
    assert sum(r["kind"] == "truncnorm" for r in rows) >= 5 and sum(r["kind"] == "gaussian" for r in rows) >= 4
    for r in rows:
        draw, used = _script(r["script"])
        if r["kind"] == "truncnorm":
            got = dr_port.sample_truncnorm_dim(1.0, 0.5, r["lb"], draw)
            assert got == r["result"] and used[0] == r["consumed"]
        else:
            if r["error"] is None:
                assert dr_port.sample_gaussian_dim(0.0, 1.0, draw) == r["result"]
            else:
                with pytest.raises(Exception, match="Not all samples were above > 0.1 after 2 attempts"):
                    dr_port.sample_gaussian_dim(0.0, 1.0, draw)
            assert used[0] == r["consumed"]


def test_target_laws_fit_the_references_own_draws(golden_dir):
    """The analytic CDFs (what the GPU samples are KS-tested against) describe the reference's output."""
    g = np.load(os.path.join(golden_dir, "sampler_reference_draws.npz"))
    n = g["uniform"].shape[0]
    crit = 1.95 / np.sqrt(n)          # alpha = 0.001
    lo, hi = dr_port.split_interleaved(list(g["uniform_params"]))
    for d in range(4):
        assert dr_port.ks_distance(g["uniform"][:, d], dr_port.uniform_cdf(lo[d], hi[d])) < crit
        assert abs(dr_port.ks_distance(g["uniform"][:, d], dr_port.uniform_cdf(lo[d], hi[d]))
                   - stats.kstest(g["uniform"][:, d], dr_port.uniform_cdf(lo[d], hi[d])).statistic) < 1e-12
    mu, sd = dr_port.split_interleaved(list(g["gaussian_params"]))
    for d in range(4):
        cdf, q = dr_port.gaussian_floor_cdf(mu[d], sd[d])
        assert dr_port.ks_distance(g["gaussian"][:, d], cdf) < crit
        assert g["gaussian"][:, d].min() >= 0.1
    mu, sd = dr_port.split_interleaved(list(g["truncnorm_params"]))
    for d in range(4):
        cdf, p = dr_port.truncnorm_lb_cdf(mu[d], sd[d], g["truncnorm_lb"][d])
        x = g["truncnorm"][:, d]
        assert dr_port.ks_distance(x, cdf) < crit
        assert x.min() >= g["truncnorm_lb"][d] and x.max() <= mu[d] + 2 * sd[d]
        mass = np.mean(x == g["truncnorm_lb"][d])
        assert abs(mass - p ** 3) < 4 * np.sqrt(max(p ** 3 * (1 - p ** 3), 1e-9) / n) + 1e-12
    # dim 2 was set up with mean == lb: p = 1/2, point mass 1/8 at the bound
    assert abs(np.mean(g["truncnorm"][:, 2] == 0.1) - 0.125) < 0.02


def test_truncnorm_moments_closed_form():
    assert abs(dr_port.TN_VAR - 0.7737413035499232) < 1e-15
    assert abs(dr_port.TN_EXCESS_KURT - (-0.6344632828703505)) < 1e-12
    u = (np.arange(200000) + 0.5) / 200000
    x = dr_port.truncnorm_ppf(u, 0.0, 1.0)
    assert abs(x.var() - dr_port.TN_VAR) < 1e-4 and abs(x.min() + 2) < 1e-3 and abs(x.max() - 2) < 1e-3


def test_split_interleaved_prefix_rule():
    a, b = dr_port.split_interleaved([1, 2, 3, 4, 5])      # odd tail ignored: range(len//2)
    assert list(a) == [1, 3] and list(b) == [2, 4]


def test_port_sample_task_shapes_and_errors():
    rs = np.random.RandomState(0)
    lo, hi = np.array([2.0, 0.5, 0.05, 0.1]), np.array([20.0, 3.0, 0.3, 1.0])
    x = dr_port.sample_task("uniform", lo, hi, rng=rs)
    assert x.shape == (4,) and np.all(x >= lo) and np.all(x < hi)
    x = dr_port.sample_task("truncnorm", [9.8, 1.0], [0.5, 0.1], lb=[0.1, 0.1], rng=rs)
    assert abs(x[0] - 9.8) <= 1.0 and abs(x[1] - 1.0) <= 0.2
    with pytest.raises(Exception, match="after 2 attempts"):
        dr_port.sample_task("gaussian", [-50.0], [1.0], rng=rs)
    with pytest.raises(ValueError, match="sampling value of random env needs to be set"):
        dr_port.sample_task(None, [1.0], [1.0])


def test_truncnorm_rvs_is_inverse_cdf_of_one_uniform():
    """scipy's truncnorm.rvs == ppf(U): the GPU sampler's inverse-CDF design reproduces the same map."""
    import scipy.stats
    rs1, rs2 = np.random.RandomState(5), np.random.RandomState(5)
    a = scipy.stats.truncnorm.rvs(-2, 2, loc=3.0, scale=0.5, size=64, random_state=rs1)
    b = dr_port.truncnorm_ppf(rs2.uniform(size=64), 3.0, 0.5)
    assert np.allclose(a, b, rtol=0, atol=1e-12)


@needs_ref
def test_live_reference_30dim_humanoid_table():
    lb = [0.2] * 13 + [0.8] * 6 + [0.15] + [0.8] * 3 + [0.15] * 7
    env = rl.make_sampler_env(30, lb)
    nu = np.array([8.322, 2.036, 5.853, 4.526, 2.632, 1.767, 4.526, 2.632, 1.767, 1.594, 1.198, 1.594, 1.198]
                  + [5, 5, 5, 5, 5, 5, 1, 5, 5, 5, 1, 1, 1, 1, 1, 1, 1], float)
    distr = np.stack([nu, 0.1 * nu], 1).reshape(-1)
    env.set_dr_distribution("truncnorm", list(distr))
    np.random.seed(1)
    x = env.sample_tasks(50)
    assert x.shape == (50, 30) and np.all(np.abs(x - nu) <= 0.2 * nu + 1e-12)
    env.set_dr_distribution("nope", []) if False else None
    with pytest.raises(Exception, match="Unknown dr_type:nope"):
        env.set_dr_distribution("nope", [])


def test_fullgaussian_port_describes_the_references_draws(golden_dir):
    """denormalize(clip(mean + F z)) with F F^T = cov has the law of the reference's fullgaussian sample_task."""
    from random_envs_b200.random_env import covariance_factor
    g = np.load(os.path.join(golden_dir, "sampler_reference_draws.npz"))
    mean, cov, ref = g["fullgaussian_mean"], g["fullgaussian_cov"], g["fullgaussian"]
    lo, hi = np.array([2.0, 0.5, 0.05, 0.1]), np.array([20.0, 3.0, 0.3, 1.0])     # random_cartpole.py:127-132
    f = covariance_factor(cov)
    assert np.allclose(f @ f.T, cov, atol=1e-14)
    z = np.random.RandomState(3).randn(200000, 4)
    x = dr_port.sample_fullgaussian_from_z(mean, f, lo, hi, z)
    assert np.all(x >= lo) and np.all(x <= hi)
    for d in range(4):
        assert stats.ks_2samp(x[:, d], ref[:, d]).pvalue > 1e-3, d
    # clipping on both sides of dim 3 shows up as atoms at the search bounds, in the port and in the reference
    for v in (lo[3], hi[3]):
        assert abs(np.mean(x[:, 3] == v) - np.mean(ref[:, 3] == v)) < 0.02 and np.mean(ref[:, 3] == v) > 0.02
    assert np.max(np.abs(np.corrcoef(x.T) - np.corrcoef(ref.T))) < 0.05
    # singular covariance still factors (eigen fallback)
    s = np.array([[1.0, 1.0], [1.0, 1.0]])
    fs = covariance_factor(s)
    assert np.allclose(fs @ fs.T, s, atol=1e-12)


@needs_ref
def test_fullgaussian_port_vs_live_reference_denormalisation():
    env = rl.make_cartpole()
    p = np.array([0.0, 4.0, 2.0, 1.0])
    lo, hi = env.get_task_search_bounds()
    assert np.array_equal(env.denormalize_parameters(p), dr_port.denormalize(p, lo, hi))
