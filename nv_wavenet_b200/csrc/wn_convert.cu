// wn_convert.cu -- dtype conversion / fill helpers (replaces nv_wavenet_conversions.cuh:28-116).
#include "wn_common.h"

namespace {
__global__ void f32_to_f16_kernel(__half* __restrict__ dst, const float* __restrict__ src, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    // 4 elements per thread per trip when aligned
    const size_t n4 = ((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) ? n / 4 : 0;
    for (size_t j = i; j < n4; j += stride) {
        const float4 v = reinterpret_cast<const float4*>(src)[j];
        __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
        uint2 o;
        o.x = *reinterpret_cast<unsigned*>(&lo);
        o.y = *reinterpret_cast<unsigned*>(&hi);
        reinterpret_cast<uint2*>(dst)[j] = o;
    }
    for (size_t j = n4 * 4 + i; j < n; j += stride) dst[j] = __float2half_rn(src[j]);
}
// mu-law decode of sampled indices, table-driven: out[b * out_pitch + j] = lut[yOut[b * N + offset + j]]
__global__ void mulaw_decode_kernel(const int* __restrict__ y, int N, int offset, int size, size_t out_pitch, size_t total, int A,
                                    const float* __restrict__ lut_f, const short* __restrict__ lut_s, float* __restrict__ out_f,
                                    short* __restrict__ out_s)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / (size_t)size, j = i % (size_t)size, o = b * out_pitch + j;
        int v = y[b * (size_t)N + offset + j];
        v = v < 0 ? 0 : (v >= A ? A - 1 : v);
        if (out_f) out_f[o] = lut_f[v];
        if (out_s) out_s[o] = lut_s[v];
    }
}
__global__ void fill_int_kernel(int* dst, int v, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = v;
}
}  // namespace

cudaError_t wn_f32_to_f16(__half* dst, const float* src_dev, size_t n, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    const int threads = 256;
    size_t blocks = (n / 4 + threads - 1) / threads;
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 16) blocks = 148 * 16;
    f32_to_f16_kernel<<<(unsigned)blocks, threads, 0, stream>>>(dst, src_dev, n);
    return cudaGetLastError();
}

__global__ void f16_to_f32_kernel(float* __restrict__ dst, const __half* __restrict__ src, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = __half2float(src[i]);
}
cudaError_t wn_f16_to_f32(float* dst, const __half* src_dev, size_t n, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    f16_to_f32_kernel<<<(unsigned)blocks, 256, 0, stream>>>(dst, src_dev, n);
    return cudaGetLastError();
}

// Counter-based selectors (SURVEY.md 8f next-1: "device-side Philox selectors"): element i of the [N][B] selector array is the
// first 32-bit output of Philox-4x32-10 with counter (i_lo, i_hi, 0, 0) and key (seed_lo, seed_hi), mapped to [0, 1) with
// 24 bits: (x >> 8) * 2^-24.  Stateless, order-independent, reproducible on the host (tests/test_gpu_zz_selectors.py).
// dst[i] takes counter first + i, so a range of samples can be drawn on its own: first = first_sample * B.
__host__ __device__ inline unsigned wn_philox_first(unsigned long long ctr, unsigned long long seed)
{
    unsigned c0 = (unsigned)ctr, c1 = (unsigned)(ctr >> 32), c2 = 0, c3 = 0;
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
    for (int r = 0; r < 10; r++) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
        const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0, n1 = (unsigned)p1, n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1, n3 = (unsigned)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}
__global__ void selectors_kernel(float* __restrict__ dst, size_t n, unsigned long long first, unsigned long long seed)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = (float)(wn_philox_first(first + i, seed) >> 8) * (1.0f / 16777216.0f);
}
cudaError_t wn_fill_selectors(float* dst, size_t n, unsigned long long first, unsigned long long seed, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    selectors_kernel<<<(unsigned)blocks, 256, 0, stream>>>(dst, n, first, seed);
    return cudaGetLastError();
}

cudaError_t wn_fill_int(int* dst, int value, size_t n, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    fill_int_kernel<<<(unsigned)blocks, 256, 0, stream>>>(dst, value, n);
    return cudaGetLastError();
}

cudaError_t wn_mulaw_decode(const int* yOut, int N, int offset, int size, int B, int A, const float* lut_f, const short* lut_s, float* out_f,
                            short* out_s, size_t out_pitch, cudaStream_t stream)
{
    const size_t total = (size_t)B * size;
    if (total == 0) return cudaSuccess;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    mulaw_decode_kernel<<<(unsigned)blocks, 256, 0, stream>>>(yOut, N, offset, size, out_pitch, total, A, lut_f, lut_s, out_f, out_s);
    return cudaGetLastError();
}
