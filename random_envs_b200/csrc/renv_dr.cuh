// Domain-randomisation samplers: device-side equivalent of RandomEnv.sample_task
// (reference random_envs/random_env.py:148-190), one Philox block (4 floats / 2 doubles) at a time.
//
//   uniform    :150-151  lo + (hi-lo)*U
//   truncnorm  :153-171  X = mean + std*Phi^-1(Phi(-2) + U*(Phi(2)-Phi(-2)))  -- scipy's truncnorm.rvs IS
//                        the inverse CDF of one uniform; while X < lb redraw; after the 3rd redraw X = lb.
//                        (The reference consumes a 4th draw before giving up and discards it; with a
//                        counter-based generator an unused draw has no effect, so attempts 0..2 suffice.)
//   gaussian   :173-190  X = randn*std + mean; while X < 0.1 redraw; three failures -> the reference raises;
//                        here the dim is counted in `violations` and set to the floor, the host raises.
//
// double: library normcdfinv / log / sincospi with explicitly rounded affine maps (parity path).
// float:  the truncation to [-2, 2] keeps the inverse CDF in its central region, so Phi^-1 is one MUFU.LG2 and a
//         degree-6 polynomial (no tail branches, no sign select, max abs error 7e-7); Box-Muller takes its radius
//         from MUFU.LG2, or a series of ln(1 - v) near u1 = 1 (max abs error 2e-6), and its angle from MUFU sin / cos
//         (max abs error 1e-6, angle rounding included).  Both transforms start from the integer draw (r >> 8).  These bounds hold over all 2^24 inputs
//         (tests/test_gpu_normal_transforms.py) and are the ones oracle/f32_draws.py checks every fp32 draw against.
#pragma once
#include "renv_philox.cuh"
#include "renv_pack.cuh"

namespace renv {

constexpr double kPhiMinus2 = 0.022750131948179195;      // Phi(-2)
constexpr double kPhiSpan = 0.9544997361036416;          // Phi(2) - Phi(-2)
constexpr double kGaussianFloor = 0.1;                   // random_env.py:181 (hard-coded)

enum DrType : int { kDrNone = 0, kDrUniform = 1, kDrTruncnorm = 2, kDrGaussian = 3, kDrFullGaussian = 4 };

// Compact 4-dim image of renv_dr_cfg for the cart-pole kernels (passed by value as a kernel parameter), already
// converted to the element type on the host (renv_abi.cu to_cfg4) so that a reset pays no F2F conversions:
//   uniform:            a = lo, b = hi - lo (fp32: times 2^-24, see Pack<float>::uniform_affine)
//   truncnorm/gaussian: a = mean, b = std, floor = lower bound / 0.1
//   fullgaussian (random_env.py:192-198): a = mean in the normalised [0,4] space, b / floor = search-bound lo / hi,
//                       factor = any F with F F^T = cov (row-major 4x4).
template <typename T> struct DrCfg4 {
    int dr_type;
    int dim;
    T a[4], b[4], floor[4];
    T factor[16];
};

template <typename T> struct Num;
// MUFU.LG2 without the denormal-input scaling of lg2.approx.f32 (3 extra instructions): arguments here are >= 2^-24.
__device__ __forceinline__ float lg2_approx(float x)
{
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

template <> struct Num<float> {
    __device__ static __forceinline__ float affine(float scale, float u, float off) { return fmaf(scale, u, off); }
    __device__ static __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    // z = Phi^-1(Phi(-2) + u * (Phi(2) - Phi(-2))) for u = (r >> 8) * 2^-24 in [0, 1).  With X = Phi(2) - Phi(-2) and
    // x = 2p - 1 = X (2u - 1) in [-X, X):  z = sqrt(2) erfinv(x) = x * g(w), w = -ln(1 - x^2) in [0, 2.42]; g is fitted
    // (Chebyshev nodes, degree 6 in t = w - 1.25, max abs error of z 2.9e-7).  1 - x^2 >= 0.089, so forming it with
    // one FMA loses nothing that matters (<= 2e-7 in z).  11 FMA-pipe + 1 MUFU + 2 ALU instructions per value.
    // Max abs error of z over all 2^24 inputs, float(Phi(2) - Phi(-2)) included: 7e-7 (measured 6.1e-7 on the B200,
    // tests/test_gpu_normal_transforms.py).
    __device__ static __forceinline__ float tn_z_bits(uint32_t r)
    {
        const float X = (float)kPhiSpan;
        const float x = fmaf((float)(r >> 8), 2.0f * X / 16777216.0f, -X);
        const float t = fmaf(lg2_approx(fmaf(-x, x, 1.0f)), -0.69314718056f, -1.25f);
        float g = -6.496782899e-06f;
        g = fmaf(g, t, 4.291892561e-05f);
        g = fmaf(g, t, 2.023686373e-04f);
        g = fmaf(g, t, -3.186480695e-03f);
        g = fmaf(g, t, 3.552299202e-03f);
        g = fmaf(g, t, 3.528738932e-01f);
        g = fmaf(g, t, 1.682294103e+00f);
        return __fmul_rn(g, x);
    }
    __device__ static __forceinline__ void tn_z4(uint4 r, float z[4])
    {
        z[0] = tn_z_bits(r.x); z[1] = tn_z_bits(r.y); z[2] = tn_z_bits(r.z); z[3] = tn_z_bits(r.w);
    }
    // Box-Muller radius sqrt(-2 ln u1), u1 = ((r >> 8) + 1) 2^-24 in (0, 1].  Near u1 = 1 the radius -> 0 and the square
    // root turns an absolute error e of the logarithm into sqrt(2 e), so MUFU.LG2 (absolute error ~2^-22 there) cannot
    // be used on its own: for v = 1 - u1 < 1/16 (exact: v = (~r >> 8) 2^-24) -ln(1 - v) is its series to v^6 (relative
    // truncation error v^6 / 7 < 1e-8); below, lg2(u1) <= -0.093 and MUFU.LG2's absolute error is harmless.  (The
    // former (24 - lg2(k)) 2 ln 2, k = 2^24 u1, cancelled near k = 2^24: off by up to 1.28e-3 on the B200.)  Max abs
    // error over all 2^24 inputs: 2e-6 (measured 6.3e-7 on the B200, tests/test_gpu_normal_transforms.py).  Cost:
    // 5 FFMA + FMUL + FSETP + FSEL more per pair than the cancelling form, 11 % of the gaussian sampler's rate.
    __device__ static __forceinline__ float bm_radius(uint32_t ra)
    {
        const float v = __fmul_rn((float)(~ra >> 8), 1.0f / 16777216.0f);
        float p = fmaf(v, 1.0f / 6.0f, 0.2f);
        p = fmaf(p, v, 0.25f);
        p = fmaf(p, v, 1.0f / 3.0f);
        p = fmaf(p, v, 0.5f);
        p = fmaf(p, v, 1.0f);
        const float near1 = __fmul_rn(2.0f * v, p);                                         // -2 ln(1 - v)
        const float far = __fmul_rn(lg2_approx(__fsub_rn(1.0f, v)), -1.3862943611198906f);  // -2 ln 2 lg2(u1)
        return sqrt_approx(v < 0.0625f ? near1 : far);
    }
    // 4 standard normals from one Philox block: Box-Muller on the pairs (x,y) and (z,w), both branches used.
    // angle = 2 pi (u2 - 1/2), u2 = (r >> 8) 2^-24, with MUFU sin / cos: together with the rounding of the angle, off
    // by at most 1e-6 absolute; each normal is within 2e-6 + 1e-6 rad (+ its own rounding) of the float64 value.
    __device__ static __forceinline__ void normal_pair(uint32_t ra, uint32_t rb, float *z)
    {
        const float two_pi = 6.283185307179586f;
        const float rad = bm_radius(ra);
        const float ang = fmaf((float)(rb >> 8), two_pi / 16777216.0f, -0.5f * two_pi);
        z[0] = __fmul_rn(rad, __cosf(ang));
        z[1] = __fmul_rn(rad, __sinf(ang));
    }
    __device__ static __forceinline__ void normals(uint4 r, float z[4])
    {
        normal_pair(r.x, r.y, z);
        normal_pair(r.z, r.w, z + 2);
    }
};
template <> struct Num<double> {
    // separately rounded multiply and add: the numpy expression lo + (hi-lo)*u, bit for bit
    __device__ static __forceinline__ double affine(double scale, double u, double off)
    {
        return __dadd_rn(off, __dmul_rn(scale, u));
    }
    __device__ static __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    __device__ static __forceinline__ double tn_z(double u) { return normcdfinv(affine(kPhiSpan, u, kPhiMinus2)); }
    __device__ static __forceinline__ void tn_z4(uint4 r, double z[2])
    {
        Pack<double>::uniforms(r, z);
        z[0] = tn_z(z[0]); z[1] = tn_z(z[1]);
    }
    __device__ static __forceinline__ void normals(uint4 r, double z[2]) { Pack<double>::normals(r, z); }
};

// fullgaussian tail (random_env.py:194-198 + denormalize_parameters :205-220): clip to [0, 4], then
// (p * (hi - lo)) / 4 + lo in that operator order.
__device__ __forceinline__ float denormalize(float x, float lo, float hi)
{
    x = fminf(fmaxf(x, 0.0f), 4.0f);
    return fmaf(__fmul_rn(x, __fsub_rn(hi, lo)), 0.25f, lo);
}
__device__ __forceinline__ double denormalize(double x, double lo, double hi)
{
    x = fmin(fmax(x, 0.0), 4.0);
    return __dadd_rn(__ddiv_rn(__dmul_rn(x, __dsub_rn(hi, lo)), 4.0), lo);
}

// Parameters of one dim block (dims j*P .. j*P+P-1) held in registers, already converted to T.
template <typename T> struct DimBlock {
    static constexpr int P = Pack<T>::kPerBlock;
    T a[P], b[P], floor[P];      // floor: lower bound (truncnorm) / 0.1 (gaussian) / unused (uniform)
    unsigned valid;              // bit k set <=> dim j*P + k exists
};

// The same parameters already converted on the host (dr_sample launcher): a thread's set-up is 12 constant-bank loads
// instead of 12 loads + 12 F2F.F32.F64 conversions + the uniform pre-scaling.
template <typename T> struct DrCfgPrepared {
    int dr_type, dim;
    T a[32], b[32], floor[32];       // b: (hi - lo) [* 2^-24 for fp32] (uniform) or std; floor: lb (truncnorm) / 0.1 (gaussian)
};
template <typename T> __device__ __forceinline__ DimBlock<T> load_dim_block(const DrCfg4<T> &cfg, int j)
{
    constexpr int P = Pack<T>::kPerBlock;
    DimBlock<T> blk;
    blk.valid = (1u << P) - 1u;
#pragma unroll
    for (int k = 0; k < P; ++k) {
        blk.a[k] = cfg.a[j * P + k]; blk.b[k] = cfg.b[j * P + k]; blk.floor[k] = cfg.floor[j * P + k];
    }
    return blk;
}
template <typename T> __device__ __forceinline__ DimBlock<T> load_dim_block(const DrCfgPrepared<T> &cfg, int j)
{
    constexpr int P = Pack<T>::kPerBlock;
    DimBlock<T> blk;
    blk.valid = 0;
#pragma unroll
    for (int k = 0; k < P; ++k) {
        const int d = j * P + k;
        const bool ok = d < cfg.dim;
        blk.a[k] = ok ? cfg.a[d] : T(0);
        blk.b[k] = ok ? cfg.b[d] : T(0);
        blk.floor[k] = ok ? cfg.floor[d] : T(0);
        if (ok) blk.valid |= 1u << k;
    }
    return blk;
}

// One standard draw per dim of the block for attempt `t`: truncnorm -> TN(-2,2) by inverse CDF, gaussian -> N(0,1).
template <typename T>
__device__ __forceinline__ void standard_draws(bool tn, uint64_t seed, uint64_t id, uint64_t tick, uint32_t purpose,
                                               uint32_t slot, T *z)
{
    const uint4 r = draw_block(seed, id, tick, purpose, slot);
    if (tn) {
        Num<T>::tn_z4(r, z);
    } else {
        Num<T>::normals(r, z);
    }
}

// Attempt 0 for the whole block, branch-free (the common case: every dim accepted).  Returns the mask of dims
// whose draw fell below the floor and must be redrawn.  uniform: out is final, mask 0.
template <typename T>
__device__ __forceinline__ unsigned first_attempt(int dr_type, const DimBlock<T> &blk, uint64_t seed, uint64_t id,
                                                  uint64_t tick, uint32_t purpose, int j, T *out)
{
    unsigned pending = 0;
    if (dr_type == kDrUniform) {
        // dims beyond `dim` have a = b = 0 and are never stored by the caller
        Pack<T>::uniform_affine(draw_block(seed, id, tick, purpose, (uint32_t)j), blk.b, blk.a, out);
    } else if (dr_type == kDrTruncnorm || dr_type == kDrGaussian) {
        constexpr int P = Pack<T>::kPerBlock;
        T z[P];
        standard_draws<T>(dr_type == kDrTruncnorm, seed, id, tick, purpose, (uint32_t)j, z);
#pragma unroll
        for (int k = 0; k < P; ++k) {
            out[k] = Num<T>::affine(blk.b[k], z[k], blk.a[k]);
            if (out[k] < blk.floor[k]) pending |= 1u << k;      // the reference's loop condition: `obs < bound`
        }
        pending &= blk.valid;
    }
    return pending;
}

// Redraws (attempts 1 and 2) for the rejected dims only, then the reference's give-up rule.  Returns the number
// of gaussian violations.
template <typename T>
__device__ __forceinline__ unsigned redraws(int dr_type, const DimBlock<T> &blk, uint64_t seed, uint64_t id,
                                            uint64_t tick, uint32_t purpose, int j, unsigned pending, T *out)
{
    constexpr int P = Pack<T>::kPerBlock;
    const bool tn = dr_type == kDrTruncnorm;
    unsigned violations = 0;
    for (int t = 1; t < 3 && pending; ++t) {
        T z[P];
        standard_draws<T>(tn, seed, id, tick, purpose, (uint32_t)(t * 16 + j), z);
#pragma unroll
        for (int k = 0; k < P; ++k) {
            if (pending & (1u << k)) {
                const T x = Num<T>::affine(blk.b[k], z[k], blk.a[k]);
                if (!(x < blk.floor[k])) {
                    out[k] = x;
                    pending &= ~(1u << k);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < P; ++k) {
        if (pending & (1u << k)) {
            out[k] = blk.floor[k];
            if (!tn) ++violations;
        }
    }
    return violations;
}

// Fills out[k] for the valid dims of the block.  Returns the number of gaussian violations.
template <typename T>
__device__ __forceinline__ unsigned sample_dim_block(int dr_type, const DimBlock<T> &blk, uint64_t seed, uint64_t id,
                                                     uint64_t tick, uint32_t purpose, int j, T *out)
{
    const unsigned pending = first_attempt<T>(dr_type, blk, seed, id, tick, purpose, j, out);
    return pending ? redraws<T>(dr_type, blk, seed, id, tick, purpose, j, pending, out) : 0u;
}

template <typename T, typename Cfg>
__device__ __forceinline__ unsigned sample_dim_block(const Cfg &cfg, uint64_t seed, uint64_t id, uint64_t tick,
                                                     uint32_t purpose, int j, T *out)
{
    return sample_dim_block<T>(cfg.dr_type, load_dim_block(cfg, j), seed, id, tick, purpose, j, out);
}

// ---- fp32 sampler hot path: the transforms of one Philox block on PACKED pairs (FFMA2 / FMUL2) ------------------
// Same operations, operands and rounding as the scalar Num<float> / Pack<float> code above, lane for lane (a packed
// lane rounds like the scalar instruction; -x is produced by a second FMA with negated constants, which is exact
// because rounding is sign-symmetric) -- so the values are bit-identical -- in half the FMA-pipe issue slots.
struct DimBlockPacked {
    u64 a01, a23, b01, b23;         // uniform: off / scale * 2^-24;  truncnorm, gaussian: mean / std
    float floor[4];
    unsigned valid;
};
__device__ __forceinline__ DimBlockPacked pack_dim_block(const DimBlock<float> &b)
{
    DimBlockPacked p;
    p.a01 = pk(b.a[0], b.a[1]); p.a23 = pk(b.a[2], b.a[3]);
    p.b01 = pk(b.b[0], b.b[1]); p.b23 = pk(b.b[2], b.b[3]);
#pragma unroll
    for (int k = 0; k < 4; ++k) p.floor[k] = b.floor[k];
    p.valid = b.valid;
    return p;
}
__device__ __forceinline__ u64 bits24_pair(uint32_t ra, uint32_t rb) { return pk((float)(ra >> 8), (float)(rb >> 8)); }

// Pack<float>::uniform_affine
__device__ __forceinline__ void uniform4_packed(uint4 r, const DimBlockPacked &p, float out[4])
{
    unpk(fma2(p.b01, bits24_pair(r.x, r.y), p.a01), out[0], out[1]);
    unpk(fma2(p.b23, bits24_pair(r.z, r.w), p.a23), out[2], out[3]);
}
// Num<float>::tn_z_bits for two draws, then the affine map mean + std * z
__device__ __forceinline__ u64 truncnorm_pair(uint32_t ra, uint32_t rb, u64 std2, u64 mean2)
{
    const float X = (float)kPhiSpan;
    const u64 F = bits24_pair(ra, rb);
    const u64 x = fma2(F, splat(2.0f * X / 16777216.0f), splat(-X));
    const u64 nx = fma2(F, splat(-2.0f * X / 16777216.0f), splat(X));          // == -x exactly
    float w0, w1;
    unpk(fma2(nx, x, splat(1.0f)), w0, w1);
    const u64 t = fma2(pk(lg2_approx(w0), lg2_approx(w1)), splat(-0.69314718056f), splat(-1.25f));
    u64 g = splat(-6.496782899e-06f);
    g = fma2(g, t, splat(4.291892561e-05f));
    g = fma2(g, t, splat(2.023686373e-04f));
    g = fma2(g, t, splat(-3.186480695e-03f));
    g = fma2(g, t, splat(3.552299202e-03f));
    g = fma2(g, t, splat(3.528738932e-01f));
    g = fma2(g, t, splat(1.682294103e+00f));
    return fma2(std2, mul2(g, x), mean2);
}
// Num<float>::normal_pair for one (radius, angle) draw pair, then the affine map
__device__ __forceinline__ u64 gaussian_pair(uint32_t ra, uint32_t rb, u64 std2, u64 mean2)
{
    const float two_pi = 6.283185307179586f;
    const float rad = Num<float>::bm_radius(ra);
    const float ang = fmaf((float)(rb >> 8), two_pi / 16777216.0f, -0.5f * two_pi);
    return fma2(std2, mul2(splat(rad), pk(__cosf(ang), __sinf(ang))), mean2);
}
// Attempt 0 for a whole block.  Returns true when some valid dim fell below its floor (the caller then takes the
// scalar first_attempt / redraws path for this block: the reference's retry loop, random_env.py:158-171,177-190).
template <int kDrType>
__device__ __forceinline__ bool first_attempt_packed(uint4 r, const DimBlockPacked &p, float out[4])
{
    if (kDrType == kDrUniform) {
        uniform4_packed(r, p, out);
        return false;
    }
    if (kDrType == kDrTruncnorm) {
        unpk(truncnorm_pair(r.x, r.y, p.b01, p.a01), out[0], out[1]);
        unpk(truncnorm_pair(r.z, r.w, p.b23, p.a23), out[2], out[3]);
    } else {
        unpk(gaussian_pair(r.x, r.y, p.b01, p.a01), out[0], out[1]);
        unpk(gaussian_pair(r.z, r.w, p.b23, p.a23), out[2], out[3]);
    }
    // dims beyond `dim` have mean = std = floor = 0: 0 < 0 is false, no mask needed
    return out[0] < p.floor[0] || out[1] < p.floor[1] || out[2] < p.floor[2] || out[3] < p.floor[3];
}

}  // namespace renv
