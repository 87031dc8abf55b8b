// wn_common.h -- shared declarations of the B200 WaveNet inference engine (host + device).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

// Everything a kernel launch needs.  Device pointers only.
// Replaces nv_wavenet_params<T_weight,T_data> (nv_wavenet.cuh:40-85) of the reference.
struct WnParams {
    int L, R, S, A, maxDil;
    int B;              // batch size of this run (stride of Lh / selectors / ring, nv_wavenet.cuh:144)
    int N;              // row stride of yOut: num_samples of this run (singleblock.cuh:245), the window W on windowed engines
    int init_sample, count;
    // window origin: the absolute sample held in slot 0 of every per-sample store (Lh, sel, forced, yOut); sample t lives in slot
    // t - origin.  0 on full engines.  The sample index t itself stays absolute (dilation mask, history-ring slot).
    int origin;
    int tanhEmbed, dump;
    // model (TD = float in fp32 mode, __half in fp16 mode)
    const void *embPrev, *embCur;                       // TD [A][R]
    const void *Wprev, *Wcur, *Wres, *Wskip;            // TD col-major, [L][M*K]
    const void *Wzs, *Wza;                              // TD col-major A x S, A x A
    const void *Bh, *Bres, *Bskip, *Bzs, *Bza;          // TD [L][2R], [L][R], [L][S], [A], [A]
    // inputs
    const void* Lh;                                     // TD [N][L][B][2R]
    const float* sel;                                   // [N][B]
    const int* forced;                                  // [B][N] or NULL
    // state
    int *yPrev, *yCur;                                  // [B]
    void* ring;                                         // TD [(maxDil+1)][L][B][R]  layer inputs
    int* yOut;                                          // [B][N]
    // last-sample activation dumps (fp32)
    float *xtOut, *skipOut, *Zs, *Za, *P;               // [L][B][R], [L][B][S], [B][A] x3
    // optional timeline trace of one sample (debug): 3 x 1024 (tag << 48 | clock) words, or NULL
    unsigned long long* trace;
    int trace_t;
};

struct WnLaunchInfo {
    int kernel, grid, block, smem_bytes, batch_per_cta, cluster;
};

// stream kernel (wn_stream_kernel.cu): CUDA-core, one CTA per batch tile, weights streamed from L2.
cudaError_t wn_launch_stream(const WnParams& p, int contract, cudaStream_t stream, WnLaunchInfo* info);   // 0 fp32 exact, 1 fp16, 2 fp32 fast
bool wn_stream_supported(int R, int S, int A, bool fp16);

// conversions (wn_convert.cu)
cudaError_t wn_f32_to_f16(__half* dst, const float* src_dev, size_t n, cudaStream_t stream);
cudaError_t wn_f16_to_f32(float* dst, const __half* src_dev, size_t n, cudaStream_t stream);
cudaError_t wn_fill_selectors(float* dst, size_t n, unsigned long long first, unsigned long long seed, cudaStream_t stream);   // counters first..first+n-1
cudaError_t wn_fill_int(int* dst, int value, size_t n, cudaStream_t stream);
