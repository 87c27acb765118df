// Log-likelihood of candidate task distributions on recorded cart-pole transitions (include/renv.h
// renv_cartpole_transition_loglik_f64): the objective DROPO-style offline DR fitting scores, in fp64.
//
// For window w (start t), candidate c and sample m, s_m is obs[t] pushed through lam applications of dynamics<double>
// (the parity path of renv_cartpole.cuh, termination ignored) under xi[c, m] and the recorded actions a[t .. t+lam-1].
// With y = next_obs[t+lam-1], mu = mean_m s_m, Sigma = cov_m(s_m) (ddof 1) and S = Sigma + diag(eps):
//     loglik[c, w] = -1/2 (y - mu)' S^-1 (y - mu) - 1/2 log det S - 2 log(2 pi)
// (-inf when the Cholesky factorisation of S meets a pivot <= 0 or NaN; NaN when the window leaves [0, T)).
//
// Launch: one CTA per (candidate, tile of kLlWindowsPerCta windows), kLlThreads threads.  A window's M samples are
// split over a fixed group of kLlLanes lanes, sample m on lane m mod kLlLanes.  Each lane accumulates the shifted sums
// sum d and sum d d' (4 + 10 doubles) of d = s_m - s_0: the shift s_0, the prediction under sample 0, is computed by
// every lane, so partial sums of different lanes simply add, and the cancellation in the covariance stays at the scale
// of the spread instead of the scale of the state.  A fixed xor-shuffle tree combines the lanes; lane 0 of the group
// forms mu, S, its Cholesky factor and the log-density.  The candidate's xi and derive() (total mass and its
// reciprocal) are staged in shared memory in chunks of kLlChunk samples, so a warp reads kLlLanes consecutive
// doubles per field and the 32 / kLlLanes groups share them.  Nothing depends on C, on the other candidates or on the
// grid: the order of every sum is fixed by (M, kLlLanes) alone.
//
// The per-candidate totals are a second kernel: one CTA per candidate sums its W values in a fixed order (strided
// per thread, then a fixed tree) with error-free transformations (TwoSum), so total[c] is the fp64 rounding of the
// exact sum up to a few ulp; a NaN or -inf value is passed through as a plain sum would.
#pragma once
#include "renv_cartpole.cuh"
#include <math_constants.h>

namespace renv {

constexpr int kLlLanes = 4;                              // lanes per window (fixed: results must not depend on M or W)
constexpr int kLlThreads = 256;
constexpr int kLlWindowsPerCta = kLlThreads / kLlLanes;
constexpr int kLlChunk = 256;                            // samples of xi staged per pass (12 KB)
constexpr int kLlSumThreads = 256;
static_assert(kLlChunk % kLlLanes == 0 && 32 % kLlLanes == 0, "a group of lanes lies in one warp");

struct LoglikArgs {
    const double *obs, *next_obs;          // (T, 4) rows
    const uint8_t *action;                 // (T)
    const int32_t *window;                 // (W) start indices
    const double *xi;                      // (C, M, 4) rows
    double *loglik;                        // (C, W)
    int64_t T;
    int W, C, M, lam;
    int64_t tiles;                         // window tiles per candidate
    double eps[4];
};

struct LoglikSmem {
    double g[kLlChunk], mc[kLlChunk], mp[kLlChunk], l[kLlChunk], total[kLlChunk], inv[kLlChunk];
};

// A 4-double row, 16-byte aligned (two 128-bit loads).
__device__ __forceinline__ State<double> ll_row(const double *p)
{
    const double2 a = *reinterpret_cast<const double2 *>(p), b = *reinterpret_cast<const double2 *>(p + 2);
    return State<double>{ a.x, a.y, b.x, b.y };
}

// Stage samples [m0, m0 + kLlChunk) of the candidate (rows past M are left alone and never read).
__device__ __forceinline__ void ll_stage(LoglikSmem &sm, const double *xi, int M, int m0)
{
    for (int j = threadIdx.x; j < kLlChunk && m0 + j < M; j += kLlThreads) {
        const State<double> v = ll_row(xi + 4 * (int64_t)(m0 + j));
        const Derived<double> d = derive(Xi<double>{ v.x, v.x_dot, v.theta, v.theta_dot });
        sm.g[j] = v.x; sm.mc[j] = v.x_dot; sm.mp[j] = v.theta; sm.l[j] = v.theta_dot;
        sm.total[j] = d.total_mass; sm.inv[j] = d.inv_total;
    }
}

__device__ __forceinline__ void ll_sample(const LoglikSmem &sm, int j, Xi<double> &p, Derived<double> &d)
{
    p = Xi<double>{ sm.g[j], sm.mc[j], sm.mp[j], sm.l[j] };
    d = Derived<double>{ sm.total[j], sm.inv[j] };
}

// Prediction of one sample: lam dynamics steps from s; the actions come from `bits` (step k < 64) or from memory.
template <bool kEuler>
__device__ __forceinline__ void ll_predict(State<double> &s, const Xi<double> &p, const Derived<double> &d,
                                           uint64_t bits, const uint8_t *act, int lam)
{
    for (int k = 0; k < lam; ++k) {
        const int a = k < 64 ? (int)((bits >> k) & 1u) : (int)act[k];
        dynamics(s, p, d, a, kEuler);
    }
}

struct LlSums { double d[4], dd[10]; };     // dd: (0,0) (0,1) (0,2) (0,3) (1,1) (1,2) (1,3) (2,2) (2,3) (3,3)

__device__ __forceinline__ void ll_accumulate(LlSums &acc, const State<double> &s, const State<double> &s0)
{
    const double d[4] = { s.x - s0.x, s.x_dot - s0.x_dot, s.theta - s0.theta, s.theta_dot - s0.theta_dot };
    int q = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        acc.d[i] += d[i];
#pragma unroll
        for (int j = i; j < 4; ++j, ++q) acc.dd[q] = fma(d[i], d[j], acc.dd[q]);
    }
}

// -1/2 r' S^-1 r - 1/2 log det S - 2 log 2 pi by a Cholesky factorisation of S (packed as LlSums::dd); -inf when a
// pivot is <= 0 or NaN.
__device__ __forceinline__ double ll_gauss(const double S[10], const double r[4])
{
    const int idx[4][4] = { { 0, 1, 2, 3 }, { 1, 4, 5, 6 }, { 2, 5, 7, 8 }, { 3, 6, 8, 9 } };
    double L[4][4], z[4], quad = 0.0, logdet = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        double piv = S[idx[j][j]];
#pragma unroll
        for (int k = 0; k < j; ++k) piv -= L[j][k] * L[j][k];
        if (!(piv > 0.0)) return -CUDART_INF;
        const double ljj = sqrt(piv);
        L[j][j] = ljj;
        logdet += log(ljj);
#pragma unroll
        for (int i = j + 1; i < 4; ++i) {
            double v = S[idx[i][j]];
#pragma unroll
            for (int k = 0; k < j; ++k) v -= L[i][k] * L[j][k];
            L[i][j] = v / ljj;
        }
        double zj = r[j];
#pragma unroll
        for (int k = 0; k < j; ++k) zj -= L[j][k] * z[k];
        z[j] = zj / ljj;
        quad += z[j] * z[j];
    }
    return -0.5 * quad - logdet - 3.6757541328186907;    // 2 log(2 pi)
}

template <bool kEuler>
__global__ void __launch_bounds__(kLlThreads) cartpole_transition_loglik_kernel(const __grid_constant__ LoglikArgs a)
{
    __shared__ LoglikSmem sm;
    const int64_t c = blockIdx.x / a.tiles;
    const int64_t w = (blockIdx.x - c * a.tiles) * kLlWindowsPerCta + threadIdx.x / kLlLanes;
    const int lane = threadIdx.x % kLlLanes;
    const double *xi = a.xi + c * (int64_t)a.M * 4;
    const bool live = w < a.W;
    const int64_t t = live ? (int64_t)a.window[w] : 0;
    const bool valid = live && t >= 0 && t <= a.T - a.lam;      // device-side guard: NaN for a bad start index

    State<double> start{ 0.0, 0.0, 0.0, 0.0 };
    uint64_t bits = 0;
    const uint8_t *act = a.action + (valid ? t : 0);
    if (valid) {
        start = ll_row(a.obs + 4 * t);
        const int n = a.lam < 64 ? a.lam : 64;
        for (int k = 0; k < n; ++k) bits |= (uint64_t)(act[k] != 0) << k;
    }
    State<double> s0 = start;
    LlSums acc;
#pragma unroll
    for (int i = 0; i < 4; ++i) acc.d[i] = 0.0;
#pragma unroll
    for (int q = 0; q < 10; ++q) acc.dd[q] = 0.0;

    for (int m0 = 0; m0 < a.M; m0 += kLlChunk) {
        if (m0) __syncthreads();
        ll_stage(sm, xi, a.M, m0);
        __syncthreads();
        const int n = a.M - m0 < kLlChunk ? a.M - m0 : kLlChunk;
        Xi<double> p;
        Derived<double> d;
        if (m0 == 0) {                                        // the shift: the prediction under sample 0, on every lane
            ll_sample(sm, 0, p, d);
            ll_predict<kEuler>(s0, p, d, bits, act, a.lam);
        }
        if (a.lam == 1 && fabs(start.theta) <= kSmallAngleF64) {
            // one step from one start state: with the small-angle branch known, sin / cos of the start are the same
            // for every sample and the compiler takes them out of the loop
            const int a0 = (int)(bits & 1u);
            for (int j = lane; j < n; j += kLlLanes) {
                State<double> s = start;
                ll_sample(sm, j, p, d);
                dynamics<true>(s, p, d, a0, kEuler);
                ll_accumulate(acc, s, s0);
            }
        } else {
            for (int j = lane; j < n; j += kLlLanes) {
                State<double> s = start;
                ll_sample(sm, j, p, d);
                ll_predict<kEuler>(s, p, d, bits, act, a.lam);
                ll_accumulate(acc, s, s0);
            }
        }
    }

    // fixed xor tree over the kLlLanes lanes of the group: every lane ends with the same bits
#pragma unroll
    for (int off = 1; off < kLlLanes; off <<= 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) acc.d[i] += __shfl_xor_sync(0xffffffffu, acc.d[i], off);
#pragma unroll
        for (int q = 0; q < 10; ++q) acc.dd[q] += __shfl_xor_sync(0xffffffffu, acc.dd[q], off);
    }
    if (!live || lane != 0) return;
    double out = CUDART_NAN;
    if (valid) {
        const double M = (double)a.M, inv_m = 1.0 / M, inv_m1 = 1.0 / (M - 1.0);
        const State<double> y = ll_row(a.next_obs + 4 * (t + a.lam - 1));
        // r = y - mu = (y - s0) - mean(d)
        const double r[4] = { (y.x - s0.x) - acc.d[0] * inv_m, (y.x_dot - s0.x_dot) - acc.d[1] * inv_m,
                              (y.theta - s0.theta) - acc.d[2] * inv_m, (y.theta_dot - s0.theta_dot) - acc.d[3] * inv_m };
        double S[10];
        int q = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = i; j < 4; ++j, ++q)
                S[q] = (acc.dd[q] - acc.d[i] * acc.d[j] * inv_m) * inv_m1 + (i == j ? a.eps[i] : 0.0);
        out = ll_gauss(S, r);
    }
    a.loglik[c * a.W + w] = out;
}

// total[c] = sum_w loglik[c, w] in a fixed order: thread i sums w = i, i + kLlSumThreads, ... with TwoSum, then a
// fixed tree over the threads.  The plain sum decides non-finite results (NaN, -inf).
__device__ __forceinline__ void two_sum(double &s, double &e, double x)
{
    const double t = s + x, bp = t - s, err = (s - (t - bp)) + (x - bp);
    s = t;
    e += err;
}

__global__ void __launch_bounds__(kLlSumThreads) loglik_total_kernel(const double *loglik, int W, double *total)
{
    __shared__ double ss[kLlSumThreads], se[kLlSumThreads], sp[kLlSumThreads];
    const double *row = loglik + (int64_t)blockIdx.x * W;
    double s = 0.0, e = 0.0, plain = 0.0;
    for (int w = threadIdx.x; w < W; w += kLlSumThreads) {
        const double v = row[w];
        two_sum(s, e, v);
        plain += v;
    }
    ss[threadIdx.x] = s; se[threadIdx.x] = e; sp[threadIdx.x] = plain;
    __syncthreads();
    for (int half = kLlSumThreads / 2; half > 0; half >>= 1) {
        if (threadIdx.x < half) {
            double a = ss[threadIdx.x], ea = se[threadIdx.x] + se[threadIdx.x + half];
            two_sum(a, ea, ss[threadIdx.x + half]);
            ss[threadIdx.x] = a; se[threadIdx.x] = ea;
            sp[threadIdx.x] += sp[threadIdx.x + half];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) total[blockIdx.x] = isfinite(sp[0]) ? ss[0] + se[0] : sp[0];
}

}  // namespace renv
