// Exhaustive device harness for the fp32 transforms of renv_dr.cuh: every launcher sweeps all 2^24 values of the
// 24-bit integer a transform reads (r >> 8), so the B200's MUFU.LG2 / __sinf / __cosf errors are measured over their
// whole input range (tests/test_gpu_normal_transforms.py compares the outputs with oracle/f32_draws.py).
//
// Compiled at test time with random_envs_b200.build.NVCC_FLAGS into a shared library; the launchers take device
// pointers (torch tensors) and synchronise before they return the CUDA error code.
#include <stdint.h>
#include "renv_dr.cuh"

using namespace renv;

namespace {

constexpr uint32_t kN = 1u << 24;

// a fixed bijection of the 24-bit integers: the partner word of m in a packed pair (odd multiplier mod 2^24)
__device__ __forceinline__ uint32_t partner(uint32_t m) { return (m * 2654435761u + 12345u) & (kN - 1u); }

__global__ void tn_z_kernel(float *out)
{
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < kN) out[m] = Num<float>::tn_z_bits((m << 8) | (m & 0xffu));     // the low 8 bits are ignored
}

// normal_pair(ra, rb) with one of the two words swept over all 2^24 values and the other fixed
__global__ void normal_pair_kernel(float *z0, float *z1, uint32_t fixed, int sweep_angle)
{
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= kN) return;
    float z[2];
    if (sweep_angle) Num<float>::normal_pair(fixed << 8, m << 8, z);
    else Num<float>::normal_pair(m << 8, fixed << 8, z);
    z0[m] = z[0];
    z1[m] = z[1];
}

// the packed attempt-0 transforms against the scalar Num<float> path, bit for bit, on the pairs (m, partner(m))
__global__ void packed_kernel(int law, float mean0, float std0, float mean1, float std1, float *out,
                              unsigned long long *mismatches)
{
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= kN) return;
    const uint32_t ra = m << 8, rb = partner(m) << 8;
    const u64 std2 = pk(std0, std1), mean2 = pk(mean0, mean1);
    float p0, p1, s[2];
    if (law == kDrTruncnorm) {
        unpk(truncnorm_pair(ra, rb, std2, mean2), p0, p1);
        s[0] = Num<float>::tn_z_bits(ra);
        s[1] = Num<float>::tn_z_bits(rb);
    } else {
        unpk(gaussian_pair(ra, rb, std2, mean2), p0, p1);
        Num<float>::normal_pair(ra, rb, s);
    }
    s[0] = Num<float>::affine(std0, s[0], mean0);
    s[1] = Num<float>::affine(std1, s[1], mean1);
    out[2 * m] = p0;
    out[2 * m + 1] = p1;
    const unsigned bad = (__float_as_uint(p0) != __float_as_uint(s[0])) + (__float_as_uint(p1) != __float_as_uint(s[1]));
    if (bad) atomicAdd(mismatches, (unsigned long long)bad);
}

int finish()
{
    const cudaError_t e = cudaDeviceSynchronize();
    return e == cudaSuccess ? (int)cudaGetLastError() : (int)e;
}

}  // namespace

extern "C" {

int harness_tn_z(float *out)
{
    tn_z_kernel<<<kN / 256, 256>>>(out);
    return finish();
}

int harness_normal_pair(float *z0, float *z1, uint32_t fixed, int sweep_angle)
{
    normal_pair_kernel<<<kN / 256, 256>>>(z0, z1, fixed, sweep_angle);
    return finish();
}

int harness_packed(int law, float mean0, float std0, float mean1, float std1, float *out, unsigned long long *mismatches)
{
    packed_kernel<<<kN / 256, 256>>>(law, mean0, std0, mean1, std1, out, mismatches);
    return finish();
}

int harness_dr_truncnorm() { return kDrTruncnorm; }
int harness_dr_gaussian() { return kDrGaussian; }

}
