"""Every fp32 normal / truncated-normal transform of renv_dr.cuh over all 2^24 inputs (tests/normal_transforms_harness.cu):

  * the packed attempt-0 transforms of the sampler (truncnorm_pair, gaussian_pair) equal the scalar Num<float> path
    (retries, env resets, observation noise, both fullgaussian kernels) bit for bit;
  * tn_z_bits, the Box-Muller radius and the angle stay within the bounds stated in renv_dr.cuh, which are the
    constants of oracle/f32_draws.py that every value-level test of the fp32 draws uses.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import f32_draws
from random_envs_b200 import build as lib_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "normal_transforms_harness.cu")
N = 1 << 24
M = np.arange(N, dtype=np.uint32)


def _compile(out):
    cmd = [lib_build._nvcc()] + lib_build.NVCC_FLAGS + ["-I", lib_build.CSRC, "-o", out, SRC]
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


def test_harness_compiles_for_sm_100a(tmp_path):
    res = _compile(str(tmp_path / "libharness.so"))
    assert res.returncode == 0, res.stdout


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("harness") / "libharness.so")
    res = _compile(path)
    assert res.returncode == 0, res.stdout
    lib = ctypes.CDLL(path)
    for f in (lib.harness_tn_z, lib.harness_normal_pair, lib.harness_packed):
        f.restype = ctypes.c_int
    lib.harness_normal_pair.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int]
    lib.harness_packed.argtypes = [ctypes.c_int] + [ctypes.c_float] * 4 + [ctypes.c_void_p, ctypes.c_void_p]
    return lib


def _words(m):
    return np.asarray(m, dtype=np.uint32) << np.uint32(8)


def _partner(m):
    return ((np.asarray(m, dtype=np.uint64) * np.uint64(2654435761) + np.uint64(12345)) & np.uint64(N - 1)).astype(np.uint32)


def _run(fn, *args):
    import torch
    torch.cuda.synchronize()
    rc = fn(*args)
    assert rc == 0, "CUDA error %d" % rc


@pytest.mark.gpu
def test_tn_z_bits_within_its_bound_over_all_inputs(harness):
    import torch
    out = torch.empty(N, dtype=torch.float32, device="cuda")
    _run(harness.harness_tn_z, ctypes.c_void_p(out.data_ptr()))
    err = np.abs(out.cpu().numpy().astype(np.float64) - f32_draws.tn_z(_words(M)))
    assert err.max() <= f32_draws.TN_Z_BOUND, (err.max(), int(err.argmax()))


# fixed partner words: angle 0 (cos = 1, sin = 0 exactly: z0 IS the radius), -pi/2, an arbitrary one, and -pi
ANGLES = [1 << 23, 1 << 22, 0x5A5A5A, 0]
# fixed radius words: the largest radius (u1 = 2^-24), u1 = 1/2, a radius near 1, and u1 = 1 (radius 0)
RADII = [0, (1 << 23) - 1, 0x9B4C35, N - 1]


@pytest.mark.gpu
@pytest.mark.parametrize("b", ANGLES)
def test_box_muller_radius_within_its_bound_over_all_inputs(harness, b):
    import torch
    z0 = torch.empty(N, dtype=torch.float32, device="cuda"); z1 = torch.empty_like(z0)
    _run(harness.harness_normal_pair, z0.data_ptr(), z1.data_ptr(), b, 0)
    w0, w1, b0, b1 = f32_draws.normal_pair(_words(M), _words(np.full(N, b)))
    g0, g1 = z0.cpu().numpy().astype(np.float64), z1.cpu().numpy().astype(np.float64)
    if b == 1 << 23:
        rad = f32_draws.radius(_words(M))
        assert np.array_equal(g1, np.zeros(N))
        err = np.abs(g0 - rad)
        assert err.max() <= f32_draws.RADIUS_BOUND, ("radius", err.max(), int(err.argmax()))
    assert np.all(np.abs(g0 - w0) <= b0), np.max(np.abs(g0 - w0) - b0)
    assert np.all(np.abs(g1 - w1) <= b1), np.max(np.abs(g1 - w1) - b1)


@pytest.mark.gpu
@pytest.mark.parametrize("a", RADII)
def test_box_muller_angle_within_its_bound_over_all_inputs(harness, a):
    import torch
    z0 = torch.empty(N, dtype=torch.float32, device="cuda"); z1 = torch.empty_like(z0)
    _run(harness.harness_normal_pair, z0.data_ptr(), z1.data_ptr(), a, 1)
    w0, w1, b0, b1 = f32_draws.normal_pair(_words(np.full(N, a)), _words(M))
    g0, g1 = z0.cpu().numpy().astype(np.float64), z1.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(g0 - w0) <= b0), np.max(np.abs(g0 - w0) - b0)
    assert np.all(np.abs(g1 - w1) <= b1), np.max(np.abs(g1 - w1) - b1)
    rad = float(f32_draws.radius(_words(a)))
    if rad > 1.0:                      # the angle alone: |(z0, z1) / rad - (cos, sin)| within the trig bound
        trig = np.maximum(np.abs(g0 - w0), np.abs(g1 - w1)) - f32_draws.RADIUS_BOUND - 2 ** -24 * rad
        assert np.max(trig) / rad <= f32_draws.TRIG_BOUND


@pytest.mark.gpu
@pytest.mark.parametrize("law", ["truncnorm", "gaussian"])
@pytest.mark.parametrize("mean,std", [((0.0, 0.0), (1.0, 1.0)), ((9.81, 0.1), (0.5, 0.01)), ((-3.0, 1e4), (0.0625, 300.0))])
def test_packed_pair_equals_the_scalar_path_bit_for_bit(harness, law, mean, std):
    import torch
    out = torch.empty(2 * N, dtype=torch.float32, device="cuda")
    bad = torch.zeros(1, dtype=torch.int64, device="cuda")
    code = harness.harness_dr_truncnorm() if law == "truncnorm" else harness.harness_dr_gaussian()
    _run(harness.harness_packed, code, mean[0], std[0], mean[1], std[1], out.data_ptr(), bad.data_ptr())
    assert int(bad.item()) == 0
    # and the packed values against the float64 contract
    p = out.cpu().numpy().astype(np.float64).reshape(N, 2)
    m32, s32 = f32_draws.f32(mean), f32_draws.f32(std)
    ra, rb = _words(M), _words(_partner(M))
    if law == "truncnorm":
        z = [f32_draws.tn_z(ra), f32_draws.tn_z(rb)]
        bz = [f32_draws.TN_Z_BOUND] * 2
    else:
        w0, w1, b0, b1 = f32_draws.normal_pair(ra, rb)
        z, bz = [w0, w1], [b0, b1]
    for q in range(2):
        want = m32[q] + s32[q] * z[q]
        bound = s32[q] * bz[q] + 2 ** -24 * (np.abs(want) + abs(m32[q]))
        assert np.all(np.abs(p[:, q] - want) <= bound), (q, np.max(np.abs(p[:, q] - want) - bound))
