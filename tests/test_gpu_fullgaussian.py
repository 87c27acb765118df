"""SURVEY section 8f rank 1: `fullgaussian` DR (random_env.py:123-127,192-220) on the GPU.

x = mean + F z (F F^T = cov) in the normalised [0,4] space, clipped, denormalised to the search bounds.
"""
import os

import numpy as np
import pytest
import torch
from scipy import stats

import random_envs_b200 as random_envs
from random_envs_b200.random_env import covariance_factor
from oracle import c_oracle, dr_port, f32_draws

pytestmark = pytest.mark.gpu

LO = np.array([2.0, 0.5, 0.05, 0.1]); HI = np.array([20.0, 3.0, 0.3, 1.0])


def _golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "sampler_reference_draws.npz"))
    return g["fullgaussian_mean"], g["fullgaussian_cov"], g["fullgaussian"]


def test_fp64_values_follow_the_contract(golden_dir):
    """Sample i = denormalize(clip(mean + F z_i)), z_i = Box-Muller of the oracle's Philox uniforms."""
    mean, cov, _ = _golden(golden_dir)
    s = random_envs.TaskSampler("RandomCartPole-v0"); s.seed_dr(5)
    s.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
    x = s.sample_tasks(300)
    f = covariance_factor(cov)
    for i in (0, 1, 63, 64, 299):
        z = np.zeros(4)
        for j in range(2):                                   # fp64: one Philox block = 2 uniforms = 1 normal pair
            u = c_oracle.uniforms(5, i, 0, c_oracle.PURPOSE_TASKS, 0, 4, np.float64)[2 * j:2 * j + 2]
            z[2 * j], z[2 * j + 1] = dr_port.box_muller_f64(u[0] + 2.0 ** -53, u[1])
        want = dr_port.sample_fullgaussian_from_z(mean, f, LO, HI, z)
        assert np.max(np.abs(x[i] - want) / (HI - LO)) < 1e-12, i


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_moments_clipping_and_reference_draws(dtype, golden_dir):
    mean, cov, ref = _golden(golden_dir)
    n = 1 << 20
    s = random_envs.TaskSampler("RandomCartPole-v0"); s.seed_dr(9)
    s.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
    x = s.sample_tasks_tensor(n, dtype=dtype).double().cpu().numpy()
    assert np.all(x >= LO - 1e-6) and np.all(x <= HI + 1e-6)
    scale = (HI - LO) / 4
    # dims 0..2 are (practically) never clipped: mean and covariance of the affine image
    mu = LO + scale * mean
    c = np.cov(x[:, :3].T)
    want = (scale[:3, None] * cov[:3, :3]) * scale[None, :3]
    assert np.all(np.abs(x[:, :3].mean(0) - mu[:3]) < 6 * np.sqrt(np.diag(want) / n) + 1e-6 * mu[:3])
    assert np.max(np.abs(c - want) / np.sqrt(np.outer(np.diag(want), np.diag(want)))) < 0.01
    # dim 3: sigma = 1.58 around 2 -> both clips active; atoms match the normal tail mass
    sd3 = np.sqrt(cov[3, 3])
    lo32, hi32 = (float(np.float32(LO[3])), float(np.float32(HI[3]))) if dtype == torch.float32 else (LO[3], HI[3])
    for v, p in ((lo32, stats.norm.cdf((0 - mean[3]) / sd3)), (hi32, stats.norm.sf((4 - mean[3]) / sd3))):
        assert abs(np.mean(np.abs(x[:, 3] - v) < 1e-7) - p) < 5 * np.sqrt(p * (1 - p) / n) + 1e-4
    xa = x.copy()                                         # fp32: map the clip atoms back onto the fp64 bounds
    for d in range(4):
        xa[np.abs(xa[:, d] - LO[d]) < 1e-7, d] = LO[d]
        xa[np.abs(xa[:, d] - HI[d]) < 1e-7, d] = HI[d]
        assert stats.ks_2samp(xa[:50000, d], ref[:, d]).pvalue > 1e-4, d
    assert np.max(np.abs(np.corrcoef(x[:200000].T) - np.corrcoef(ref.T))) < 0.06


def test_30dim_humanoid_fullgaussian_runs_and_is_correlated():
    s = random_envs.TaskSampler("RandomHumanoid-v0"); s.seed_dr(1)
    rs = np.random.RandomState(0)
    a = 0.05 * rs.randn(30, 30) + 0.3 * np.eye(30)
    cov = a @ a.T
    s.set_dr_distribution("fullgaussian", {"mean": np.full(30, 2.0), "cov": cov})
    x = s.sample_tasks_tensor(1 << 18, dtype=torch.float32).double().cpu().numpy()
    lo, hi = s.get_task_search_bounds()
    assert x.shape == (1 << 18, 30) and np.all(x >= lo - 1e-5) and np.all(x <= hi + 1e-5)
    scale = (hi - lo) / 4
    want = (scale[:, None] * cov) * scale[None, :]
    got = np.cov(x.T)
    assert np.max(np.abs(got - want) / np.sqrt(np.outer(np.diag(want), np.diag(want)))) < 0.02


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_vector_env_resamples_fullgaussian_xi_on_reset(dtype, golden_dir):
    mean, cov, ref = _golden(golden_dir)
    n = 1 << 17
    env = random_envs.RandomCartPoleVecEnv(n, dtype=dtype, seed=4)
    env.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
    env.set_dr_training(True)
    env.reset()
    xi = env.get_task().double().cpu().numpy()
    for d in range(4):
        xi[np.abs(xi[:, d] - LO[d]) < 1e-7, d] = LO[d]
        xi[np.abs(xi[:, d] - HI[d]) < 1e-7, d] = HI[d]
        assert stats.ks_2samp(xi[:50000, d], ref[:, d]).pvalue > 1e-4, d
    assert np.max(np.abs(np.corrcoef(xi.T) - np.corrcoef(ref.T))) < 0.06
    before = env.get_task().clone()
    obs, rew, done, _ = env.step(env.sample_actions())
    for _ in range(30):
        obs, rew, done, _ = env.step(env.sample_actions())
    changed = (env.get_task() != before).any(1)
    assert 0.2 < float(changed.float().mean()) <= 1.0          # envs that finished an episode got a new xi
    env.rollout((0.1, 0.1, 1.0, 0.3), 0.0, 100)
    xi2 = env.get_task().double().cpu().numpy()
    assert np.all(xi2 >= LO - 1e-6) and np.all(xi2 <= HI + 1e-6)


@pytest.mark.parametrize("env_id,n", [("RandomHumanoid-v0", 100000 + 77), ("RandomHumanoidUnmodeled-v0", 128 * 5), ("RandomHumanoid-v0", 37)])
def test_tensor_core_contraction_matches_the_fma_chain_kernel(env_id, n):
    """dim > 16, fp32: X = Z F^T runs as tcgen05.mma kind::tf32 on head/tail-split operands (renv_fullgauss_tc.cuh).
    Same Philox draws as the CUDA-core kernel, so the two differ only by the rounding of the contraction: stated
    tolerance 4e-6 of the search-bound width (3xTF32 products, fp32 accumulation)."""
    dim = len(random_envs.XI_TABLES[env_id].names)
    rs = np.random.RandomState(3)
    a = 0.2 * rs.randn(dim, dim) + 0.5 * np.eye(dim)
    cov, mean = a @ a.T, rs.uniform(1.0, 3.0, dim)

    def draw(tensor):
        old = os.environ.get("RENV_FULLGAUSS_TENSOR")
        os.environ["RENV_FULLGAUSS_TENSOR"] = "1" if tensor else "0"
        try:
            s = random_envs.TaskSampler(env_id); s.seed_dr(21)
            s.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
            x = s.sample_tasks_tensor(n, dtype=torch.float32)
            y = s.sample_tasks_tensor(n, dtype=torch.float32)          # second call: another Philox tick
            s.check_dr_violations()
            return x.double().cpu().numpy(), y.double().cpu().numpy(), s.get_task_search_bounds()
        finally:
            if old is None:
                os.environ.pop("RENV_FULLGAUSS_TENSOR", None)
            else:
                os.environ["RENV_FULLGAUSS_TENSOR"] = old
    xt, yt, (lo, hi) = draw(True)
    xc, yc, _ = draw(False)
    assert xt.shape == (n, dim)
    assert np.max(np.abs(xt - xc) / (hi - lo)) <= 4e-6 and np.max(np.abs(yt - yc) / (hi - lo)) <= 4e-6
    assert not np.array_equal(xt, yt)
    assert np.mean(xt == xc) > 0.2          # many entries even agree to the last bit
    # and both against the float64 restatement of the fp32 contract (fp32 takes 4 normals per Philox block, fp64 2,
    # so the fp64 sampler draws other values): every entry within its stated bound
    f = covariance_factor(cov)
    for got, tick, tc in ((xt, 0, True), (yt, 1, True), (xc, 0, False), (yc, 1, False)):
        value, bound = f32_draws.fullgaussian_sample(21, np.arange(n, dtype=np.uint64), tick, f32_draws.PURPOSE_TASKS,
                                                     mean, f, lo, hi, tensor_core=tc)
        assert np.all(np.abs(got - value) <= bound), (tick, tc, np.max(np.abs(got - value) - bound))
