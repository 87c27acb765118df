"""Float64 restatement of the fp32 draw contract: normal, truncated-normal, full-Gaussian and observation-noise draws.

TEST INFRASTRUCTURE (see oracle/__init__.py).

The fp32 kernels turn each 32-bit Philox word r into the 24-bit integer m = r >> 8 and push it through MUFU-based
transforms (renv_dr.cuh).  Here the same integers go through the exact transforms in float64:

  truncated normal   z = ndtri(Phi(-2) + m 2^-24 (Phi(2) - Phi(-2)))
  Box-Muller pair    rad = sqrt(-2 ln((m_a + 1) 2^-24)),  ang = 2 pi (m_b 2^-24 - 1/2),  (rad cos ang, rad sin ang)

Every function returns the float64 value together with a per-element bound on |fp32 kernel - float64 value| derived
from the transform errors stated in renv_dr.cuh (the constants below), so a test can compare every output value.
A draw whose accept / reject decision against a floor lies within its bound of the floor is flagged AMBIGUOUS: fp32
and float64 may legitimately take different branches there.

Counters follow DESIGN section 3: key = (seed lo, seed hi), counter = (id lo, id[47:32] | tick[47:32] << 16, tick lo,
purpose << 24 | slot), slot = attempt * 16 + dim block; fp32 takes 4 values per block, dim d from block d // 4, word
d % 4; the Box-Muller pairs are (word 0, word 1) and (word 2, word 3), radius from the first word of a pair.
"""
import numpy as np
from scipy import special

PURPOSE_XI, PURPOSE_TASKS, PURPOSE_OBS = 1, 3, 4
GAUSSIAN_FLOOR = 0.1

# Transform error bounds of the fp32 kernels (absolute), as stated in renv_dr.cuh and DESIGN section 3 and measured
# over all 2^24 inputs by tests/test_gpu_normal_transforms.py.
TN_Z_BOUND = 7e-7          # Num<float>::tn_z_bits
RADIUS_BOUND = 2e-6        # Box-Muller radius sqrt(-2 ln u)
TRIG_BOUND = 1e-6          # cos / sin of the fixed-point angle, including the rounding of the angle itself

_PHI_M2 = special.ndtr(-2.0)
_PHI_SPAN = special.ndtr(2.0) - _PHI_M2
_EPS = 2.0 ** -24          # unit roundoff of fp32

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays of counters (broadcast together); key words are Python ints.  Returns 4 uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & _MASK for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c[0]                      # < 2^64: exact in uint64
        p1 = _M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return [v.astype(np.uint32) for v in c]


def draw_block(seed, ids, tick, purpose, slot):
    """The 4 words of block (seed, id, tick, purpose, slot) for every id (and / or tick) of the broadcast arrays."""
    ids = np.asarray(ids, dtype=np.uint64)
    tick = np.asarray(tick, dtype=np.uint64)
    c1 = ((ids >> np.uint64(32)) & np.uint64(0xFFFF)) | (((tick >> np.uint64(32)) & np.uint64(0xFFFF)) << np.uint64(16))
    c3 = (int(purpose) << 24) | int(slot)
    return philox(ids & _MASK, c1, tick & _MASK, c3, int(seed) & 0xFFFFFFFF, int(seed) >> 32)


# ----------------------------------------------------------------------------- transforms
def tn_z(r):
    """Standard normal truncated to [-2, 2] by inverse CDF of the 24-bit uniform of word r."""
    m = (np.asarray(r, dtype=np.uint32) >> np.uint32(8)).astype(np.float64)
    return special.ndtri(_PHI_M2 + m * 2.0 ** -24 * _PHI_SPAN)


def radius(ra):
    """Box-Muller radius sqrt(-2 ln u1), u1 = ((ra >> 8) + 1) 2^-24 in (0, 1]."""
    k = (np.asarray(ra, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) + 1.0
    return np.sqrt(-2.0 * np.log(k * 2.0 ** -24))


def angle(rb):
    m = (np.asarray(rb, dtype=np.uint32) >> np.uint32(8)).astype(np.float64)
    return 2.0 * np.pi * (m * 2.0 ** -24 - 0.5)


def normal_pair(ra, rb):
    """(z0, z1, bound): both branches of one Box-Muller pair and the bound on each fp32 branch."""
    rad, ang = radius(ra), angle(rb)
    z0, z1 = rad * np.cos(ang), rad * np.sin(ang)
    # |rad_f trig_f - rad trig| <= |rad_f - rad| |trig_f| + rad |trig_f - trig|, |trig_f| <= 1 + TRIG_BOUND
    bound = RADIUS_BOUND * (1.0 + TRIG_BOUND) + rad * TRIG_BOUND
    return z0, z1, bound + _EPS * np.abs(z0), bound + _EPS * np.abs(z1)


def standard_block(words, law):
    """(z, bound), each a list of 4 arrays: the standard draws of one Philox block under `law`."""
    if law == "truncnorm":
        z = [tn_z(w) for w in words]
        return z, [TN_Z_BOUND + 0.0 * v for v in z]
    a0, a1, b0, b1 = normal_pair(words[0], words[1])
    c0, c1, d0, d1 = normal_pair(words[2], words[3])
    return [a0, a1, c0, c1], [b0, b1, d0, d1]


def normals(seed, ids, tick, purpose, dim, slot0=0):
    """(z, bound), each (len(ids), dim): dim d from block slot0 + d // 4, word d % 4."""
    ids = np.atleast_1d(np.asarray(ids, dtype=np.uint64))
    z = np.zeros((ids.size, dim)); bz = np.zeros((ids.size, dim))
    for j in range((dim + 3) // 4):
        zs, bs = standard_block(draw_block(seed, ids, tick, purpose, slot0 + j), "gaussian")
        for q in range(4):
            if 4 * j + q < dim:
                z[:, 4 * j + q], bz[:, 4 * j + q] = zs[q], bs[q]
    return z, bz


def f32(x):
    """The fp32 image (as float64) of a parameter: the host casts every double parameter to float once."""
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


# ----------------------------------------------------------------------------- laws
def sample_dr(law, seed, ids, tick, purpose, mean, std, floor):
    """fp32 `truncnorm` / `gaussian` DR draws: mean + std z, the first of attempts 0..2 (slot attempt * 16 + j) that is
    not below the floor, else the floor.  mean / std / floor: (dim,) as the caller passes them (rounded to fp32 here).

    Returns a dict of (n, dim) arrays:
      value, bound      the float64 value and the bound on the kernel's deviation from it (0 at the floor)
      ambiguous         some attempt up to the deciding one lies within its bound of the floor
      candidates, cand_bound  (n, dim, 4): the three attempts and the floor, any of which an ambiguous draw may yield
      gave_up           no attempt reached the floor (gaussian: a violation)
    """
    mean, std, floor = f32(mean), f32(std), f32(floor)
    ids = np.atleast_1d(np.asarray(ids, dtype=np.uint64))
    n, dim = ids.size, mean.size
    cand = np.zeros((n, dim, 4)); cb = np.zeros((n, dim, 4))
    for t in range(3):
        for j in range((dim + 3) // 4):
            zs, bs = standard_block(draw_block(seed, ids, tick, purpose, t * 16 + j), law)
            for q in range(4):
                d = 4 * j + q
                if d < dim:
                    x = mean[d] + std[d] * zs[q]
                    cand[:, d, t] = x
                    cb[:, d, t] = abs(std[d]) * bs[q] + _EPS * (np.abs(x) + abs(mean[d]))
    cand[:, :, 3] = floor
    value = np.broadcast_to(floor, (n, dim)).copy(); bound = np.zeros((n, dim))
    decided = np.zeros((n, dim), bool); ambiguous = np.zeros((n, dim), bool)
    for t in range(3):
        x, b = cand[:, :, t], cb[:, :, t]
        near = np.abs(x - floor) <= b
        ambiguous |= ~decided & near
        take = ~decided & (x >= floor)
        value[take], bound[take] = x[take], b[take]
        decided |= take
    return dict(value=value, bound=bound, ambiguous=ambiguous, candidates=cand, cand_bound=cb, gave_up=~decided)


def check_dr(got, ref):
    """Asserts every element of the kernel's fp32 output `got` (n, dim) matches `ref` = sample_dr(...): unambiguous
    elements within their bound of the value, ambiguous ones within the bound of one of the candidates."""
    got = np.asarray(got, dtype=np.float64)
    amb = ref["ambiguous"]
    err = np.abs(got - ref["value"]) - ref["bound"]
    bad = ~amb & (err > 0)
    assert not bad.any(), "%d values off, first at %s: got %r want %r +- %r" % (
        bad.sum(), np.argwhere(bad)[0], got[bad][0], ref["value"][bad][0], ref["bound"][bad][0])
    if amb.any():
        ok = (np.abs(got[amb][:, None] - ref["candidates"][amb]) <= ref["cand_bound"][amb]).any(1)
        assert ok.all(), "an ambiguous draw matches none of its attempts nor the floor"


def fullgaussian(z, bz, mean, factor, lo, hi, tensor_core=False):
    """`fullgaussian` in fp32: denormalize(clip(mean + F z, 0, 4), lo, hi) on standard normals z (n, dim) with bounds bz.

    The FMA chain (and the tensor-core contraction, whose 3xTF32 products and fp32 accumulation are looser) rounds each
    of its dim + 1 partial sums; clipping is 1-Lipschitz; denormalize rounds twice more.  Returns (value, bound)."""
    mean, factor, lo, hi = f32(mean), f32(factor), f32(lo), f32(hi)
    x = mean + z @ factor.T
    mag = np.abs(mean) + np.abs(z) @ np.abs(factor).T
    dim = mean.size
    # FMA chain: one rounding per partial sum.  Tensor cores: 3xTF32 drops Z_lo F_lo (2^-22 of each product) and the
    # TF32 operands keep 11 bits of the tails (another 2^-22 each), about 4 eps per product on top of an fp32
    # accumulation whose rounding mode is not specified; 8 eps per term covers both.
    rounding = (dim + 2) * _EPS * mag * (8.0 if tensor_core else 1.0)
    bx = bz @ np.abs(factor).T + rounding
    w = f32(hi - lo)                                  # the kernels round hi - lo once
    value = (np.clip(x, 0.0, 4.0) * w) / 4.0 + lo
    bound = bx * np.abs(w) / 4.0 + 4.0 * _EPS * (np.abs(value) + np.abs(w) + np.abs(lo))
    return value, bound


def fullgaussian_sample(seed, ids, tick, purpose, mean, cov_factor, lo, hi, tensor_core=False):
    z, bz = normals(seed, ids, tick, purpose, len(mean))
    return fullgaussian(z, bz, mean, cov_factor, lo, hi, tensor_core)


def obs_noise(seed, ids, tick, which, state, std):
    """Observation of a Noisy env: state + std z, z from block (kObs, which * 16).  state (n, 4) fp32 values."""
    z, bz = normals(seed, ids, tick, PURPOSE_OBS, 4, slot0=16 * int(which))
    s, std = np.asarray(state, dtype=np.float64), float(f32(std))
    value = s + std * z
    return value, std * bz + _EPS * (np.abs(value) + np.abs(s))
