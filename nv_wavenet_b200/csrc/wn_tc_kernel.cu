// wn_tc_kernel.cu -- fp16 tensor-core kernel of the WaveNet inference loop (sm_100a: tcgen05 + TMEM + bulk TMA).
//
// ONE persistent CTA (12 warps) per tile of 32 / 64 / 128 utterances runs the whole autoregressive loop for `count` samples:
//
//   warps 0-7  "epilogue": 2, 4 or 8 threads per utterance (an utterance occupies 1, 2 or 4 rows = TMEM lanes of every tile).
//              embed -> per layer: [Dx + Bres + x -> x tile] [D1 + Lh + Bh -> tanh * sigmoid -> h tile]
//              -> relu(skip) tile -> relu(Zs) tile -> softmax + categorical sample, all row-local
//              (the reference spreads these over CTAs/threads: nv_wavenet_persistent.cuh:223-462, softmax.cuh:36-191).
//   warp 8     TMA producer.  Streams the pre-tiled fp16 weight image (and the x[t-d] history tiles) from L2 through an
//              NSTAGE x 16 KB shared-memory ring, and the conditioning tiles, with cp.async.bulk + mbarrier complete_tx.
//   warp 9     MMA issuer A (and the only issuer of the unfused schedule): D[128 rows x N channels] (fp32, TMEM) +=
//              X[128 x 64] . W[N x 64]^T with tcgen05.mma (activations = A operand, weights = B operand, both K-major
//              SWIZZLE_128B); tcgen05.commit signals the epilogue and frees ring stages.
//   warp 10    MMA issuer B of the fused schedule (skip and dilated-history GEMMs, half of the output GEMMs).
//   warp 11    history copy of the fused schedule (x tile: shared -> global ring, one bulk copy).
//
// Replaces nv_wavenet_persistent.cuh + matrix_math.cuh + softmax.cuh of the reference for T_data = half.
// Numerical contract (oracle/wavenet_oracle.c, WNO_PREC_FP16): weights, biases, embeddings, Lh and every GEMM
// input rounded to fp16; fp32 accumulation; residual stream, skip sum, softmax in fp32 (logits parked as fp16 offsets from the row max).  The fused schedule folds
// Wcur_l . Wres_{l-1} into one fp16 matrix (see the kernel) -- same tolerance, checked by the same tests.
#include "wn_common.h"
#include "wn_math.cuh"
#include "wn_sm100.cuh"

#include <stdlib.h>

namespace {

using namespace sm100;

constexpr int R = 64, A = 256;
constexpr int TILE = 16384;                 // [128 rows x 64 fp16] K-major SW128
constexpr int NT = 384;                     // 8 epilogue warps + TMA producer warp + 2 MMA issuer warps + history-copy warp
constexpr int NEPI = 256;

struct TcImage {                            // byte offsets inside the packed image
    size_t layer_bytes, off_out, off_bias, total;
    size_t b_bh, b_bres, b_bskp, b_bzs, b_bza, b_bhf;     // float offsets inside the bias block
    size_t l_wf;                                   // byte offset of the folded matrix Wcur_l . Wres_{l-1} inside a layer block
};
__host__ __device__ inline TcImage tc_image(int S, int L)
{
    TcImage im;
    im.l_wf = (size_t)TILE * 2 + TILE / 2 + (size_t)(S / 128) * TILE;
    im.layer_bytes = im.l_wf + TILE;
    im.off_out = (size_t)L * im.layer_bytes;
    im.off_bias = im.off_out + (size_t)(S / 64) * 2 * TILE + (size_t)(A / 64) * 2 * TILE;
    im.b_bh = 0;
    im.b_bres = im.b_bh + (size_t)L * 128;
    im.b_bskp = im.b_bres + (size_t)L * 64;
    im.b_bzs = im.b_bskp + (size_t)L * S;
    im.b_bza = im.b_bzs + A;
    im.b_bhf = im.b_bza + A;
    im.total = im.off_bias + (im.b_bhf + (size_t)L * 128) * sizeof(float);
    return im;
}

__host__ __device__ inline size_t tc_smem_bytes(int S, int L, int nstage)
{
    // 4 activation tiles + weight ring + conditioning buffers (2 tiles) + biases (Bh, Bres, Bskip-sum, Bzs, Bza) + dilations + barriers
    return 1024 + 4 * (size_t)TILE + (size_t)nstage * TILE + 2 * TILE + ((size_t)L * 192 + S + 2 * A) * sizeof(float) + (size_t)L * 4 +
           128 * 5 * sizeof(float) + (2 * nstage + 20) * 8 + 16;
}

// Conditioning in the tensor-core layout: fp16 [N][L][Bpad rows][2 halves of 64 channels], tiled per 128 utterances;
// inside a tile: [half][row][128 B], 16-byte chunks XOR-swizzled with (row & 7) -- i.e. exactly the K-major
// SWIZZLE_128B image of an MMA A-operand tile, so a 1-D bulk TMA copy of rows*128 bytes needs no further shuffling.
// TU = utterances per tile: 64 (four threads per utterance, the lower-latency variant) while the batch fits the SMs
// that way, 128 otherwise.
__host__ __device__ inline int cond_rows(int B, int tile, int TU) { const int r = B - tile * TU; return r >= TU ? TU : ((r + 7) & ~7); }
__host__ __device__ inline size_t cond_bpad(int B, int TU) { const int nt = (B + TU - 1) / TU; return (size_t)(nt - 1) * TU + cond_rows(B, nt - 1, TU); }

__global__ void tc_cond_kernel(unsigned char* __restrict__ dst, const float* __restrict__ src, int first_sample, int nsamples, int L, int B, int TU)
{
    // one thread per (sample, layer, utterance, 8-channel chunk): 32 B in, 16 B out
    const size_t total = (size_t)nsamples * L * B * 16;
    const size_t bpad = cond_bpad(B, TU);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i & 15);
        const size_t rowi = i >> 4;                       // (s * L + l) * B + b
        const int b = (int)(rowi % B);
        const size_t sl = rowi / B;                       // s * L + l
        const float4 f0 = *reinterpret_cast<const float4*>(src + rowi * 128 + c * 8);
        const float4 f1 = *reinterpret_cast<const float4*>(src + rowi * 128 + c * 8 + 4);
        __half2 h0 = __floats2half2_rn(f0.x, f0.y), h1 = __floats2half2_rn(f0.z, f0.w), h2 = __floats2half2_rn(f1.x, f1.y), h3 = __floats2half2_rn(f1.z, f1.w);
        uint4 o;
        o.x = *reinterpret_cast<unsigned*>(&h0); o.y = *reinterpret_cast<unsigned*>(&h1);
        o.z = *reinterpret_cast<unsigned*>(&h2); o.w = *reinterpret_cast<unsigned*>(&h3);
        const int tile = b / TU, r = b % TU, half = c >> 3, q = c & 7;
        const size_t off = (((size_t)first_sample * L + sl) * bpad + (size_t)tile * TU) * 256 + (size_t)half * cond_rows(B, tile, TU) * 128 +
                           (size_t)r * 128 + (size_t)((q ^ (r & 7)) << 4);
        *reinterpret_cast<uint4*>(dst + off) = o;
    }
}

// inverse of tc_cond_kernel (debug / tests): conditioning store -> fp32 [n][L][B][2R]
__global__ void tc_cond_readback_kernel(float* __restrict__ dst, const unsigned char* __restrict__ src, int first_sample, int nsamples, int L, int B, int TU)
{
    const size_t total = (size_t)nsamples * L * B * 16;
    const size_t bpad = cond_bpad(B, TU);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i & 15);
        const size_t rowi = i >> 4;
        const int b = (int)(rowi % B);
        const size_t sl = rowi / B;
        const int tile = b / TU, r = b % TU, half = c >> 3, q = c & 7;
        const size_t off = (((size_t)first_sample * L + sl) * bpad + (size_t)tile * TU) * 256 + (size_t)half * cond_rows(B, tile, TU) * 128 +
                           (size_t)r * 128 + (size_t)((q ^ (r & 7)) << 4);
        const __half2* v = reinterpret_cast<const __half2*>(src + off);
#pragma unroll
        for (int k = 0; k < 4; k++) { dst[rowi * 128 + c * 8 + 2 * k] = __low2float(v[k]); dst[rowi * 128 + c * 8 + 2 * k + 1] = __high2float(v[k]); }
    }
}

// ------------------------------------------------------------------------------------------------ pack
// blob (fp16, column-major matrices as uploaded) -> tiled / swizzled weight image + fp32 bias block
__global__ void tc_pack_kernel(WnParams p, unsigned char* __restrict__ img, TcImage im)
{
    const int S = p.S, L = p.L;
    const __half* Wprev = static_cast<const __half*>(p.Wprev);
    const __half* Wcur = static_cast<const __half*>(p.Wcur);
    const __half* Wres = static_cast<const __half*>(p.Wres);
    const __half* Wskip = static_cast<const __half*>(p.Wskip);
    const __half* Wzs = static_cast<const __half*>(p.Wzs);
    const __half* Wza = static_cast<const __half*>(p.Wza);
    const size_t gstride = (size_t)gridDim.x * blockDim.x;
    const size_t g0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto put = [&](size_t chunk_off, int row, int k, __half v) { *reinterpret_cast<__half*>(img + chunk_off + sw128_offset(row, k)) = v; };
    // per layer
    for (size_t i = g0; i < (size_t)L * 128 * 64; i += gstride) {
        const int l = (int)(i / (128 * 64)), c = (int)(i % (128 * 64)) / 64, k = (int)(i % 64);
        const size_t lb = (size_t)l * im.layer_bytes;
        put(lb, c, k, Wprev[(size_t)l * 128 * 64 + c + (size_t)k * 128]);
        put(lb + TILE, c, k, Wcur[(size_t)l * 128 * 64 + c + (size_t)k * 128]);
        if (c < 64) put(lb + 2 * TILE, c, k, Wres[(size_t)l * 64 * 64 + c + (size_t)k * 64]);
    }
    for (size_t i = g0; i < (size_t)L * S * 64; i += gstride) {
        const int l = (int)(i / ((size_t)S * 64)), s = (int)((i / 64) % S), k = (int)(i % 64);
        put((size_t)l * im.layer_bytes + 2 * TILE + TILE / 2 + (size_t)(s / 128) * TILE, s % 128, k, Wskip[(size_t)l * S * 64 + s + (size_t)k * S]);
    }
    // folded matrix of the fused schedule: Wf_l = Wcur_l . Wres_{l-1} (fp32 accumulation of the fp16 factors, one rounding),
    // so that Wcur_l . x_l = Wcur_l . x_{l-1} + Wf_l . h_{l-1} + Wcur_l . Bres_{l-1}
    for (size_t i = g0; i < (size_t)L * 128 * 64; i += gstride) {
        const int l = (int)(i / (128 * 64)), c = (int)(i % (128 * 64)) / 64, k = (int)(i % 64);
        if (l == 0) continue;
        float acc = 0.f;
        for (int j = 0; j < 64; j++)
            acc = fmaf(__half2float(Wcur[(size_t)l * 128 * 64 + c + (size_t)j * 128]), __half2float(Wres[(size_t)(l - 1) * 64 * 64 + j + (size_t)k * 64]), acc);
        put((size_t)l * im.layer_bytes + im.l_wf, c, k, __float2half_rn(acc));
    }
    // output layers: chunk (kt, nh) = rows a in [128 nh, +128), k in [64 kt, +64)
    for (size_t i = g0; i < (size_t)A * S; i += gstride) {
        const int a = (int)(i / S), s = (int)(i % S);
        put(im.off_out + (size_t)((s / 64) * 2 + a / 128) * TILE, a % 128, s % 64, Wzs[a + (size_t)s * A]);
    }
    const size_t off_wza = im.off_out + (size_t)(S / 64) * 2 * TILE;
    for (size_t i = g0; i < (size_t)A * A; i += gstride) {
        const int a = (int)(i / A), z = (int)(i % A);
        put(off_wza + (size_t)((z / 64) * 2 + a / 128) * TILE, a % 128, z % 64, Wza[a + (size_t)z * A]);
    }
    // biases -> fp32; running prefix of the skip biases (the skip sum is kept in TMEM without biases)
    float* bias = reinterpret_cast<float*>(img + im.off_bias);
    const __half* Bh = static_cast<const __half*>(p.Bh);
    const __half* Bres = static_cast<const __half*>(p.Bres);
    const __half* Bskip = static_cast<const __half*>(p.Bskip);
    for (size_t i = g0; i < (size_t)L * 128; i += gstride) {
        const int l = (int)(i / 128), c = (int)(i % 128);
        const float bh = __half2float(Bh[i]);
        bias[im.b_bh + i] = bh;
        float acc = 0.f;                                        // Wcur_l . Bres_{l-1}
        if (l > 0)
            for (int j = 0; j < 64; j++)
                acc = fmaf(__half2float(Wcur[(size_t)l * 128 * 64 + c + (size_t)j * 128]), __half2float(Bres[(size_t)(l - 1) * 64 + j]), acc);
        bias[im.b_bhf + i] = bh + acc;
    }
    for (size_t i = g0; i < (size_t)L * 64; i += gstride) bias[im.b_bres + i] = __half2float(Bres[i]);
    for (size_t s = g0; s < (size_t)S; s += gstride) {
        float acc = 0.f;
        for (int l = 0; l < L; l++) { acc += __half2float(Bskip[(size_t)l * S + s]); bias[im.b_bskp + (size_t)l * S + s] = acc; }
    }
    for (size_t i = g0; i < (size_t)A; i += gstride) {
        bias[im.b_bzs + i] = __half2float(static_cast<const __half*>(p.Bzs)[i]);
        bias[im.b_bza + i] = __half2float(static_cast<const __half*>(p.Bza)[i]);
    }
}

// ------------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ uint32_t pack_h2(float a, float b)
{
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t v)
{
    return __half22float2(*reinterpret_cast<__half2*>(&v));
}
// chunk q (16 bytes = 8 fp16) of row `row` inside a SW128 tile
__device__ __forceinline__ uint32_t chunk_off(int row, int q) { return (uint32_t)row * 128u + (uint32_t)((q ^ (row & 7)) << 4); }

// DUP (tiles with <= 64 live utterances, e.g. the 64-per-GPU headline case): every utterance occupies TWO rows (u and u+64)
// of each activation tile / TMEM accumulator, so that all four TMEM lane quadrants -- and with them all four warp
// schedulers and their MUFU pipes -- work for it: 4 threads per utterance instead of 2, each on 16 of the 64 channels.
//
// FUSED (default schedule): ONE MMA <-> epilogue round trip per layer instead of two.  The pre-activation of layer l is
// accumulated as  (Lh + Bh') [tcgen05.st] + Wprev_l.x_l[t-d] + Wcur_l.x_{l-1} [both in the background, one layer early]
// + Wf_l.h_{l-1} [the only GEMM on the critical path], Wf_l = Wcur_l.Wres_{l-1} folded at pack time.  The residual GEMM
// Wres_{l-1}.h_{l-1} still produces x_l (history ring, next layer's background GEMM, dump) but nothing waits on it
// before the next gate.
template <int S, int CP, bool FUSED>
__global__ void __launch_bounds__(NT, 1) wn_tc_kernel(const WnParams p, const unsigned char* __restrict__ img, const int nstage)
{
    // CP = row copies per utterance (1, 2, 4): tiles of 128 / CP utterances, 2 CP threads per utterance.  CP = 4 spreads a
    // small batch over twice the SMs of CP = 2 and halves the per-thread gate / residual / softmax work once more.
    constexpr bool DUP = CP > 1;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // 1024-byte alignment by OFFSET (not by pointer round-trip through an integer): the compiler keeps knowing these
    // are shared-memory addresses and emits LDS/STS instead of generic LD/ST
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int L = p.L, B = p.B;
    const TcImage im = tc_image(S, L);

    unsigned char* t_xc = smem;                    // x tile of the current layer        (= BIG k-tile 0)
    unsigned char* t_x1 = smem + 3 * TILE;         // FUSED: x tiles ping-pong by layer parity (t_xc, t_x1 = BIG k-tile 3)
    unsigned char* t_h = smem + TILE;              // gated activation tiles, double buffered by layer parity (= BIG k-tiles 1, 2)
    unsigned char* t_big = smem;                   // [128 x 256] as 4 k-tiles: relu(skip), relu(Zs), then fp16 logits scratch
    unsigned char* ring = smem + 4 * TILE;
    // conditioning buffers: one Lh[t][l] tile = [2 halves][rows][128 B]; DUP tiles (<= 64 rows, 16 KB) are double
    // buffered, full tiles (32 KB) single buffered
    unsigned char* t_cond = ring + (size_t)nstage * TILE;
    constexpr int NC = DUP ? 2 : 1;
    constexpr int CB = DUP ? TILE : 2 * TILE;
    float* s_bh = reinterpret_cast<float*>(t_cond + 2 * TILE);
    float* s_bres = s_bh + (size_t)L * 128;
    float* s_bsk = s_bres + (size_t)L * 64;
    float* s_bzs = s_bsk + S;
    float* s_bza = s_bzs + A;
    int* s_dil = reinterpret_cast<int*>(s_bza + A);
    float* s_pair = reinterpret_cast<float*>(s_dil + L + (L & 1));      // [128 rows][2 halves][max, sum] softmax exchange
    int* s_y = reinterpret_cast<int*>(s_pair + 128 * 4);                // [128] sampled index per utterance
    uint64_t* w_full = reinterpret_cast<uint64_t*>(s_y + 128);
    uint64_t* w_empty = w_full + nstage;
    uint64_t* epi_done = w_empty + nstage;      // [2] at +0, +17: tile-published phases alternate between the two barriers
    uint64_t* d1_full = epi_done + 1;
    uint64_t* dx_full = epi_done + 2;
    uint64_t* skip_full = epi_done + 3;
    uint64_t* out_full = epi_done + 4;
    uint64_t* pre_done = epi_done + 5;          // accumulator of the coming layer initialised with Lh + bias
    uint64_t* cond_full = epi_done + 6;         // [NC]
    uint64_t* cond_empty = epi_done + 8;        // [NC]
    uint64_t* cx_done = epi_done + 10;          // fused schedule, see the issuer roles
    uint64_t* b_done = epi_done + 11;           // [2] at +11, +14: alternating by layer parity, so that the signalling role can
    uint64_t* hx_full = epi_done + 12;          //     never complete a barrier twice before its waiter has looked once
    uint64_t* hx_done = epi_done + 13;          // [2] at +13, +15
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(epi_done + 16);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile = blockIdx.x, ntiles = gridDim.x;
    const int slots = p.maxDil + 1;
    const int t_begin = p.init_sample, t_end = p.init_sample + p.count;
    unsigned char* gring = static_cast<unsigned char*>(p.ring);
    auto ring_tile = [&](int t, int l) -> unsigned char* {
        return gring + (((size_t)(t % slots) * L + l) * ntiles + tile) * (size_t)TILE;
    };

    if (tid == 0) {
        for (int s = 0; s < nstage; s++) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
        mbar_init(epi_done, NEPI); mbar_init(epi_done + 17, NEPI);
        mbar_init(d1_full, 1); mbar_init(dx_full, 1); mbar_init(skip_full, FUSED ? 2 : 1); mbar_init(out_full, FUSED ? 2 : 1);
        mbar_init(cx_done, 1); mbar_init(b_done, 1); mbar_init(b_done + 3, 1); mbar_init(hx_full, NEPI); mbar_init(hx_done, 1); mbar_init(hx_done + 2, 1);
        mbar_init(pre_done, NEPI);
        for (int i = 0; i < NC; i++) { mbar_init(&cond_full[i], 1); mbar_init(&cond_empty[i], NEPI); }
        fence_mbar_init();
        // dilation of layer l (nv_wavenet.cuh:99-111): 1,2,4..maxDil,1,2,...
        int d = 1;
        for (int l = 0; l < L; l++) { s_dil[l] = d; d <<= 1; if (d > p.maxDil) d = 1; }
    }
    if (warp == 8) tmem_alloc<512>(tmem_slot);
    {   // biases and the identity tile -> shared memory
        const float* gb = reinterpret_cast<const float*>(img + im.off_bias);
        for (int i = tid; i < L * 128; i += NT) s_bh[i] = gb[(FUSED ? im.b_bhf : im.b_bh) + i];
        for (int i = tid; i < L * 64; i += NT) s_bres[i] = gb[im.b_bres + i];
        for (int i = tid; i < S; i += NT) s_bsk[i] = gb[im.b_bskp + (size_t)(L - 1) * S + i];
        for (int i = tid; i < A; i += NT) { s_bzs[i] = gb[im.b_bzs + i]; s_bza[i] = gb[im.b_bza + i]; }
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns: [0,128) and [128,256) = pre-activation accumulators, ping-pong by layer parity; the residual GEMM of
    // layer l writes columns [0,64) of the buffer the gate of layer l has just drained; [256,512) = skip sum over layers
    // (then Zs); Za reuses [0,256).
    const uint32_t D1B = tmem_base, DSKIP = tmem_base + 256, DZS = tmem_base + 256, DZA = tmem_base;

    // conditioning tile geometry (see tc_cond_kernel)
    constexpr int TU = 128 / CP;                    // utterances per tile
    const int c_rows = cond_rows(B, tile, TU);
    const uint32_t c_bytes = (uint32_t)c_rows * 128u;
    const size_t c_bpad = cond_bpad(B, TU);
    const unsigned char* gcond = static_cast<const unsigned char*>(p.Lh);
    auto cond_ptr = [&](int t, int l, int half) -> const unsigned char* {
        return gcond + (((size_t)(t - p.origin) * L + l) * c_bpad + (size_t)tile * TU) * 256 + (size_t)half * c_bytes;
    };

    // debug timeline: role r (0 epilogue thread 0, 1 MMA issuer, 2 producer) appends (tag << 48 | clock) words
    unsigned long long* trc = (p.trace && blockIdx.x == 0) ? p.trace : nullptr;
    int trn = 0;
    const int tr_t = p.trace_t & 0xFFFF, tr_tid = p.trace_t >> 16;     // sample and epilogue thread to trace
#define TRACE(role, tag) do { if (trc && t == tr_t && trn < 1023) trc[(role) * 1024 + trn++] = ((unsigned long long)(tag) << 48) | (clock64() & 0xFFFFFFFFFFFFull); } while (0)

    if (warp == 8) {
        // =============================================================== TMA producer (whole warp converged, one lane issues)
        {
            int stage = 0;
            uint32_t ph = 1;
            auto put = [&](const void* src, uint32_t bytes) {
                mbar_wait(&w_empty[stage], ph);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&w_full[stage], bytes);
                    tma_load_1d(ring + (size_t)stage * TILE, src, bytes, &w_full[stage]);
                }
                __syncwarp();
                if (++stage == nstage) { stage = 0; ph ^= 1; }
            };
            // history tile: `bytes` of rows from row 0; with DUP the same rows again from row 64
            auto put_act = [&](const void* src, uint32_t bytes) {
                if (!DUP) { put(src, bytes); return; }
                mbar_wait(&w_empty[stage], ph);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&w_full[stage], CP * bytes);
#pragma unroll
                    for (int k = 0; k < CP; k++) tma_load_1d(ring + (size_t)stage * TILE + (size_t)k * (TILE / CP), src, bytes, &w_full[stage]);
                }
                __syncwarp();
                if (++stage == nstage) { stage = 0; ph ^= 1; }
            };
            // conditioning tile g (g counts layers since the start of the launch) -> buffer g % NC
            int g_cond = 0;
            auto put_cond = [&](int t, int l) {
                const int cbuf = g_cond % NC;
                mbar_wait(&cond_empty[cbuf], ((g_cond / NC) & 1) ^ 1);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&cond_full[cbuf], 2 * c_bytes);
                    tma_load_1d(t_cond + (size_t)cbuf * CB, cond_ptr(t, l, 0), 2 * c_bytes, &cond_full[cbuf]);   // both halves are contiguous
                    // pull the tiles a few layers ahead from HBM into L2 (sample and layer kept apart: t * L overflows an int
                    // at sample indices a windowed engine reaches)
                    const int ta = t + (l + 4) / L, la = (l + 4) % L;
                    if (ta < t_end) tma_prefetch_l2(cond_ptr(ta, la, 0), 2 * c_bytes);
                }
                __syncwarp();
                g_cond++;
            };
            // Weight-ring chunk order = consumption order of the MMA issuer (see there):
            //   prev(0) | cur(0) res(0) prev(1) | cur(1) skip(0) res(1) prev(2) | ... | cur(L-1) skip(L-2) res(L-1) | skip(L-1) | Wzs | Wza
            // where prev(l) = the x[t-d_l] history tile + Wprev_l, present only if t >= d_l.
            auto put_prev = [&](int t, int l, int d) {
                if (t >= d) { put_act(ring_tile(t - d, l), TILE / CP); put(img + (size_t)l * im.layer_bytes, TILE); }
            };
            auto put_skip = [&](int l) {
                for (int c = 0; c < S / 128; c++) put(img + (size_t)l * im.layer_bytes + 2 * TILE + TILE / 2 + (size_t)c * TILE, TILE);
            };
            if (FUSED) {
                // chunk order of the fused schedule (see the MMA issuer):
                //   prev(0) cur(0) prev(1) cur(1) | res(0) Wf(1) skip(0) prev(2) cur(2) | ... | res(L-2) Wf(L-1) skip(L-2) | skip(L-1) | Wzs | Wza
                // (on the dumping sample skip(l-1) precedes Wf(l), and res(L-1) is computed as well)
                for (int t = t_begin; t < t_end; t++) {
                    const bool dstep = p.dump && (t == t_end - 1);
                    put_cond(t, 0);
                    put_prev(t, 0, 1);
                    put(img + TILE, TILE);                              // Wcur_0
                    if (L > 1) {
                        put_cond(t, 1);
                        put_prev(t, 1, s_dil[1]);
                        put(img + im.layer_bytes + TILE, TILE);         // Wcur_1
                    }
                    for (int l = 1; l < L; l++) {
                        const unsigned char* lw = img + (size_t)l * im.layer_bytes;
                        if (lane == 0) TRACE(2, 100 + l);
                        if (NC == 2 && l + 1 < L) put_cond(t, l + 1);
                        put(lw - im.layer_bytes + 2 * TILE, TILE / 2);  // Wres_{l-1}
                        if (dstep) put_skip(l - 1);
                        put(lw + im.l_wf, TILE);                        // Wf_l
                        if (!dstep) put_skip(l - 1);
                        if (l + 1 < L) {
                            // single conditioning buffer: its consumer (gate l) first needs the residual of layer l-1 above
                            if (NC == 1) put_cond(t, l + 1);
                            put_prev(t, l + 1, s_dil[l + 1]);
                            put(lw + im.layer_bytes + TILE, TILE);      // Wcur_{l+1}
                        }
                    }
                    if (dstep) put(img + (size_t)(L - 1) * im.layer_bytes + 2 * TILE, TILE / 2);
                    put_skip(L - 1);
                    const unsigned char* ow = img + im.off_out;
                    for (int c = 0; c < (S / 64) * 2 + (A / 64) * 2; c++) put(ow + (size_t)c * TILE, TILE);
                }
            } else
            for (int t = t_begin; t < t_end; t++) {
                int d = 1;
                put_cond(t, 0);
                put_prev(t, 0, 1);
                for (int l = 0; l < L; l++) {
                    const unsigned char* lw = img + (size_t)l * im.layer_bytes;
                    int dn = d << 1; if (dn > p.maxDil) dn = 1;
                    if (lane == 0) TRACE(2, 100 + l);
                    if (l + 1 < L) put_cond(t, l + 1);
                    put(lw + TILE, TILE);                               // Wcur_l
                    if (l > 0) put_skip(l - 1);
                    put(lw + 2 * TILE, TILE / 2);                       // Wres_l
                    if (l + 1 < L) put_prev(t, l + 1, dn);
                    d = dn;
                }
                put_skip(L - 1);
                const unsigned char* ow = img + im.off_out;
                for (int c = 0; c < (S / 64) * 2 + (A / 64) * 2; c++) put(ow + (size_t)c * TILE, TILE);
            }
        }
    } else if (warp >= 9) {
        // =============================================================== MMA issuer(s) (whole warp converged, one lane issues)
        {
            const uint32_t idesc128 = make_idesc_f16(128, 128), idesc64 = make_idesc_f16(128, 64);
            int stage = 0;
            uint32_t ph_full = 0, ph_epi = 0;
            const uint64_t d_ring = make_desc_kmajor_sw128(smem_u32(ring)), d_xc = make_desc_kmajor_sw128(smem_u32(t_xc)),
                           d_h = make_desc_kmajor_sw128(smem_u32(t_h)), d_big = make_desc_kmajor_sw128(smem_u32(t_big));
            uint32_t ph_pre = 0;
            constexpr uint64_t TILE_D = TILE >> 4;                      // one tile further, in descriptor address units
            auto wait_stage = [&]() -> uint64_t {                       // descriptor of the next ring stage once its data landed
                mbar_wait(&w_full[stage], ph_full);
                return d_ring + (uint64_t)stage * TILE_D;
            };
            auto advance = [&]() { if (++stage == nstage) { stage = 0; ph_full ^= 1; } };
            // 4 K-slices of one 64-deep chunk, then (optionally) up to two commits; single elected lane
            auto mma4 = [&](uint64_t da, uint64_t db, uint32_t d, uint32_t idesc, bool acc0, uint64_t* bar0, uint64_t* bar1) {
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; k++) umma_f16(d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (acc0 || k) ? 1u : 0u);
                    if (bar0) umma_commit(bar0);
                    if (bar1) umma_commit(bar1);
                }
                __syncwarp();
            };
            // the epilogue's "tile published" phases alternate between two barriers (role B may be a whole gate behind role A:
            // on a single barrier it could find TWO completions past the one it waits for, which a parity wait cannot see)
            int n_epi = 0;
            auto wait_epi = [&]() {
                const int k = n_epi & 1;
                mbar_wait(epi_done + k * 17, (ph_epi >> k) & 1u);
                ph_epi ^= 1u << k;
                n_epi++;
                tc_fence_after_sync();
            };
            // open(l): the epilogue has initialised D1[l&1] with Lh[t][l] + Bh (tcgen05.st); add Wprev_l . x[t-d]
            auto open_layer = [&](int l, bool has_prev) {
                const uint32_t d1 = D1B + (uint32_t)(l & 1) * 128;
                mbar_wait(pre_done, ph_pre); ph_pre ^= 1;
                tc_fence_after_sync();
                if (has_prev) {
                    const uint64_t da = wait_stage();
                    const int sa = stage;
                    advance();
                    const uint64_t db = wait_stage();
                    tc_fence_after_sync();
                    mma4(da, db, d1, idesc128, true, &w_empty[sa], &w_empty[stage]);
                    advance();
                }
            };
            // fused schedule: the conditioning and the bias are added by the gate itself, so the FIRST GEMM into an
            // accumulator overwrites it: Wprev_l . x[t-d] if the history reaches back that far, else the Wcur GEMM
            auto open_f = [&](int l, bool has_prev, bool wait_x) {
                if (wait_x) { mbar_wait(pre_done, ph_pre); ph_pre ^= 1; tc_fence_after_sync(); }
                if (has_prev) {
                    const uint64_t da = wait_stage();
                    const int sa = stage;
                    advance();
                    const uint64_t db = wait_stage();
                    tc_fence_after_sync();
                    mma4(da, db, D1B + (uint32_t)(l & 1) * 128, idesc128, false, &w_empty[sa], &w_empty[stage]);
                    advance();
                }
            };
            // skip(l): Dskip (+)= Wskip_l . h_l, h_l in the H buffer of parity l
            auto skip_layer = [&](int l, uint64_t* done_bar) {
                const uint64_t dh = d_h + (uint64_t)(l & 1) * TILE_D;
                // all S/128 chunks as ONE issue block: a single election, the commits at the end
                uint64_t dws[S / 128];
                int sts[S / 128];
#pragma unroll
                for (int c = 0; c < S / 128; c++) { dws[c] = wait_stage(); sts[c] = stage; advance(); }
                tc_fence_after_sync();
                if (elect_one()) {
#pragma unroll
                    for (int c = 0; c < S / 128; c++)
#pragma unroll
                        for (int k = 0; k < 4; k++) umma_f16(DSKIP + c * 128, dh + (uint64_t)(2 * k), dws[c] + (uint64_t)(2 * k), idesc128, (l > 0 || k) ? 1u : 0u);
#pragma unroll
                    for (int c = 0; c < S / 128; c++) umma_commit(&w_empty[sts[c]]);
                    if (done_bar) umma_commit(done_bar);
                }
                __syncwarp();
            };
            // Issue order per layer: cur(l) | skip(l-1) in the shadow of the gate epilogue | res(l) | prev(l+1) in the shadow
            // of the residual epilogue.  Nothing but cur / res sits between an epilogue arrival and the accumulator it
            // waits for.
            auto out_gemms = [&]() {
                wait_epi();                                             // relu(skip) tile ready
                for (int kt = 0; kt < S / 64; kt++)
                    for (int nh = 0; nh < 2; nh++) {
                        const uint64_t dw = wait_stage();
                        tc_fence_after_sync();
                        const bool last = (kt == S / 64 - 1) && nh == 1;
                        mma4(d_big + (uint64_t)kt * TILE_D, dw, DZS + nh * 128, idesc128, kt > 0, &w_empty[stage], last ? out_full : nullptr);
                        advance();
                    }
                wait_epi();                                             // relu(Zs) tile ready
                for (int kt = 0; kt < A / 64; kt++)
                    for (int nh = 0; nh < 2; nh++) {
                        const uint64_t dw = wait_stage();
                        tc_fence_after_sync();
                        const bool last = (kt == A / 64 - 1) && nh == 1;
                        mma4(d_big + (uint64_t)kt * TILE_D, dw, DZA + nh * 128, idesc128, kt > 0, &w_empty[stage], last ? out_full : nullptr);
                        advance();
                    }
            };
            if (FUSED) {
                // Three single-lane roles share the issue work, which -- not the tensor pipe -- bounds a one-CTA layer
                // (every group of 4 MMAs + commits costs its issuing thread ~350 cycles, every mbarrier wait ~100):
                //   A (warp 9)  critical path: per gate h_{l-1}: res(l-1) -> dx_full | Wf(l) -> d1_full | Wcur_{l+1}.x_l
                //   B (warp 10) background:    skip(l-1) | Wprev_{l+1}.x_{l+1}[t-d]      (+ the nh = 1 half of Zs / Za)
                //   C (warp 11) history ring:  published x_l tile -> global, one bulk copy (async proxy on both ends)
                // All walk the same chunk sequence of the weight ring and wait only for their own chunks.
                //   cx_done  A -> B: Wcur_{l+1}.x_l (which OVERWRITES D1) has completed, Wprev may accumulate
                //   b_done   B -> gate threads: skip(l-1) [h tile of that parity reusable] and prev(l+1) completed; awaited next to
                //                    d1_full(l+1), which also bounds how far B can fall behind
                //   hx_full  epilogue -> C, hx_done C -> A: the copy of x_{l-1} has fully completed before A commits dx_full(l-1)
                //                    (whose consumer overwrites an x tile) and before the commits that let the producer run on
                const uint64_t d_x[2] = {d_xc, d_big + 3 * TILE_D};
                const int role = warp - 9;
                uint32_t ph_cx = 0, ph_hx = 0;                     // ph_hx: bit k = phase of barrier k of the pair
                auto wait2 = [&](uint64_t* pair, int stride, uint32_t& ph, int k) {
                    mbar_wait(pair + (k & 1) * stride, (ph >> (k & 1)) & 1u);
                    ph ^= 1u << (k & 1);
                };
                auto skipc = [&](int n) { for (int i = 0; i < n; i++) advance(); };
                constexpr int SKC = S / 128;
                if (role == 2) {
                    const uint32_t hist_bytes = (uint32_t)(TILE / CP);
                    for (int t = t_begin; t < t_end; t++)
                        for (int l = 0; l < L; l++) {
                            mbar_wait(hx_full, ph_hx); ph_hx ^= 1;
                            if (lane == 0) {
                                tma_store_1d(ring_tile(t, l), (l & 1) ? t_x1 : t_xc, hist_bytes);
                                tma_store_wait_all();
                                mbar_arrive(hx_done + (l & 1) * 2);
                            }
                            __syncwarp();
                        }
                } else if (role == 0) {
                    for (int t = t_begin; t < t_end; t++) {
                        const bool dstep = p.dump && (t == t_end - 1);
                        uint64_t dw;
                        wait_epi();                                     // x_0 tile ready (and Dza of the previous sample consumed)
                        if (lane == 0) TRACE(1, 20);
                        open_f(0, t >= 1, false);                       // Wprev_0 . x_0[t-1] stays with A (start of the chain)
                        dw = wait_stage();
                        tc_fence_after_sync();
                        mma4(d_x[0], dw, D1B, idesc128, t >= 1, d1_full, &w_empty[stage]);          // D1[0] (+)= Wcur_0 . x_0
                        advance();
                        if (L > 1) {
                            const bool hp = t >= s_dil[1];
                            if (hp) skipc(2);                           // B: Wprev_1
                            dw = wait_stage();
                            tc_fence_after_sync();
                            mma4(d_x[0], dw, D1B + 128, idesc128, false, hp ? cx_done : nullptr, &w_empty[stage]);   // D1[1] = Wcur_1 . x_0
                            advance();
                        }
                        for (int l = 1; l < L; l++) {
                            const uint64_t dh = d_h + (uint64_t)((l - 1) & 1) * TILE_D;
                            const bool hpn = (l + 1 < L) && t >= s_dil[l + 1];
                            dw = wait_stage();                          // Wres_{l-1} already landed when h arrives
                            if (!dstep) {                               // ... and so has Wf_l, the next chunk of the sequence
                                const int s1 = (stage + 1 == nstage) ? 0 : stage + 1;
                                mbar_wait(&w_full[s1], s1 ? ph_full : (ph_full ^ 1u));
                            }
                            wait_epi();                                 // h_{l-1} ready, D1[(l-1)&1] drained
                            if (lane == 0) TRACE(1, 22);
                            // (every tcgen05.commit sits in the election block of the MMAs it tracks: issued with nothing of its
                            // thread outstanding it never arrives)
                            mma4(dh, dw, D1B + (uint32_t)((l - 1) & 1) * 128, idesc64, false, dx_full, &w_empty[stage]);      // Dx = Wres . h
                            advance();
                            if (lane == 0) TRACE(1, 25);
                            if (dstep) skip_layer(l - 1, nullptr);      // dumping sample: the skip sum through l-1 must be complete at gate l
                            dw = wait_stage();
                            tc_fence_after_sync();
                            // D1[l] += Wf_l . h; B's share of D1[l] / the free h tile are awaited by the gate threads, not here
                            mma4(dh, dw, D1B + (uint32_t)(l & 1) * 128, idesc128, true, d1_full, &w_empty[stage]);
                            advance();
                            if (lane == 0) TRACE(1, 21);
                            if (!dstep) skipc(SKC);                     // B: skip(l-1)
                            // history copy of x_{l-1} complete: before dx_full(l), whose consumer overwrites that x tile, and
                            // before any further commit lets the producer run on
                            wait2(hx_done, 2, ph_hx, l - 1);
                            mbar_wait(pre_done, ph_pre); ph_pre ^= 1;   // x_l tile published, Dx of layer l-1 consumed
                            tc_fence_after_sync();
                            if (l + 1 < L) {
                                if (hpn) skipc(2);                      // B: Wprev_{l+1}
                                dw = wait_stage();
                                tc_fence_after_sync();
                                mma4(d_x[l & 1], dw, D1B + (uint32_t)((l + 1) & 1) * 128, idesc128, false, hpn ? cx_done : nullptr, &w_empty[stage]);   // = Wcur_{l+1} . x_l
                                advance();
                            }
                            if (lane == 0) TRACE(1, 24);
                        }
                        wait_epi();                                     // h_{L-1}
                        wait2(hx_done, 2, ph_hx, L - 1);                // x_{L-1} copied: the activation tiles may be reused
                        if (dstep) {
                            dw = wait_stage();
                            tc_fence_after_sync();
                            mma4(d_h + (uint64_t)((L - 1) & 1) * TILE_D, dw, D1B + (uint32_t)((L - 1) & 1) * 128, idesc64, false, dx_full, &w_empty[stage]);
                            advance();
                            skip_layer(L - 1, skip_full);
                        } else {
                            skipc(SKC);
                        }
                        if (lane == 0) mbar_arrive(skip_full);          // second arrival: this role's conditions for the output phase
                        __syncwarp();
                        // output GEMMs: A takes the nh = 0 half of the columns, B the other
                        for (int g = 0; g < 2; g++) {
                            wait_epi();                                 // relu(skip) / relu(Zs) tile ready
                            const int KT = g ? A / 64 : S / 64;
                            for (int kt = 0; kt < KT; kt++) {
                                dw = wait_stage();
                                tc_fence_after_sync();
                                mma4(d_big + (uint64_t)kt * TILE_D, dw, (g ? DZA : DZS), idesc128, kt > 0, &w_empty[stage], kt == KT - 1 ? out_full : nullptr);
                                advance();
                                skipc(1);
                            }
                        }
                    }
                } else {
                    for (int t = t_begin; t < t_end; t++) {
                        const bool dstep = p.dump && (t == t_end - 1);
                        // b_done of iteration j (0 at the start of the sample, l in the loop) is committed inside the LAST issue
                        // block of the iteration, or -- if this role issued nothing -- signalled by a plain arrival
                        auto bsig = [&](int j) { return b_done + (j & 1) * 3; };
                        auto prev_b = [&](int l, uint64_t* done_bar) {  // D1[l&1] += Wprev_l . x_l[t-d], after A's overwrite has completed
                            mbar_wait(cx_done, ph_cx); ph_cx ^= 1;
                            const uint64_t da = wait_stage();
                            const int sa = stage;
                            advance();
                            const uint64_t db = wait_stage();
                            tc_fence_after_sync();
                            if (elect_one()) {
#pragma unroll
                                for (int k = 0; k < 4; k++) umma_f16(D1B + (uint32_t)(l & 1) * 128, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc128, 1u);
                                umma_commit(&w_empty[sa]);
                                umma_commit(&w_empty[stage]);
                                if (done_bar) umma_commit(done_bar);
                            }
                            __syncwarp();
                            advance();
                        };
                        auto arrive_b = [&](int j) { if (elect_one()) mbar_arrive(bsig(j)); __syncwarp(); };
                        wait_epi();                                     // x_0
                        if (t >= 1) skipc(2);                           // A: Wprev_0
                        skipc(1);                                       // A: Wcur_0
                        if (L > 1) {
                            if (t >= s_dil[1]) prev_b(1, bsig(0)); else arrive_b(0);
                            skipc(1);                                   // A: Wcur_1
                        }
                        for (int l = 1; l < L; l++) {
                            skipc(1);                                   // A: Wres_{l-1}
                            wait_epi();                                 // h_{l-1}
                            const bool hpn = (l + 1 < L) && t >= s_dil[l + 1];
                            if (dstep) skipc(SKC + 1);                  // A: skip(l-1), Wf_l
                            else { skipc(1); skip_layer(l - 1, hpn ? nullptr : bsig(l)); }
                            if (l + 1 < L) {
                                if (hpn) prev_b(l + 1, bsig(l));
                                skipc(1);                               // A: Wcur_{l+1}
                            }
                            if (dstep && !hpn) arrive_b(l);             // nothing issued in this iteration
                        }
                        wait_epi();                                     // h_{L-1}
                        if (dstep) skipc(1 + SKC);
                        else skip_layer(L - 1, skip_full);
                        for (int g = 0; g < 2; g++) {
                            wait_epi();
                            const int KT = g ? A / 64 : S / 64;
                            for (int kt = 0; kt < KT; kt++) {
                                skipc(1);
                                const uint64_t dw = wait_stage();
                                tc_fence_after_sync();
                                mma4(d_big + (uint64_t)kt * TILE_D, dw, (g ? DZA : DZS) + 128, idesc128, kt > 0, &w_empty[stage], kt == KT - 1 ? out_full : nullptr);
                                advance();
                            }
                        }
                    }
                }
            } else if (warp == 9)
            for (int t = t_begin; t < t_end; t++) {
                int d = 1;                                              // dilation of layer l (nv_wavenet.cuh:99-111)
                for (int l = 0; l < L; l++) {
                    int dn = d << 1; if (dn > p.maxDil) dn = 1;         // dilation of layer l + 1
                    const uint32_t d1 = D1B + (uint32_t)(l & 1) * 128;
                    uint64_t dw = 0;
                    if (l > 0) dw = wait_stage();                       // Wcur_l is already in flight: wait for it before x_l
                    wait_epi();                                         // x_l tile ready (and, for l = 0, Dza consumed)
                    if (lane == 0) TRACE(1, 20);
                    if (l == 0) { open_layer(0, t >= 1); dw = wait_stage(); }
                    tc_fence_after_sync();
                    mma4(d_xc, dw, d1, idesc128, true, d1_full, &w_empty[stage]);       // D1 += Wcur . x[t]
                    advance();
                    if (lane == 0) TRACE(1, 21);
                    if (l > 0) skip_layer(l - 1, nullptr);              // in the shadow of the gate epilogue
                    dw = wait_stage();                                  // Wres_l
                    wait_epi();                                         // h tile ready, D1 consumed
                    if (lane == 0) TRACE(1, 22);
                    mma4(d_h + (uint64_t)(l & 1) * TILE_D, dw, d1, idesc64, false, dx_full, &w_empty[stage]);   // Dx = Wres . h
                    advance();
                    if (lane == 0) TRACE(1, 23);
                    if (l + 1 < L) open_layer(l + 1, t >= dn);          // in the shadow of the residual epilogue
                    if (lane == 0) TRACE(1, 24);
                    d = dn;
                }
                skip_layer(L - 1, skip_full);
                out_gemms();
            }
        }
    } else {
        // =============================================================== epilogue: 8 warps, TWO threads per utterance
        // Warp w works on TMEM lane quadrant w % 4 (hardware rule) and on channel half w / 4: thread (quad, lane, ch)
        // owns row 32*quad + lane and channels [32 ch, 32 ch + 32) of the 64-wide residual / gate, i.e. 16-byte chunks
        // 4 ch .. 4 ch + 3 of its row in every 128-byte tile row.  Two warps per scheduler hide each other's latencies.
        constexpr int NS = 2 * CP;                      // threads per utterance
        constexpr int CW = 64 / NS;                     // residual / gate channels per thread
        constexpr int CQ = CW / 8;                      // 16-byte chunks per thread in a 128-byte tile row
        const int quad = warp & 3, ch = warp >> 2;
        const int row = quad * 32 + lane;               // TMEM lane / tile row this thread reads
        const int u = row & (TU - 1);                   // utterance of the tile
        const int sub = ch * CP + row / TU;             // which CW-wide slice of the channels is mine
        const int b = tile * TU + u;
        const bool valid = b < B;
        const bool wv = tile * TU + ((quad * 32) & (TU - 1)) < B;   // warp has a live utterance: dead warps only keep
                                                        // the barrier protocol going (their rows are never read back)
        const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
        const int c32 = CW * sub, q4 = CQ * sub;        // first channel / first chunk of this thread
        // rows of the activation tiles this thread writes: its own row, and with DUP the twin row of the utterance
        auto st_tile = [&](unsigned char* tile_base, int q, uint4 v) {
#pragma unroll
            for (int k = 0; k < CP; k++) *reinterpret_cast<uint4*>(tile_base + chunk_off(u + k * TU, q)) = v;   // same (row & 7): same swizzle
        };
        auto tmem_ldc = [&](uint32_t addr, uint32_t (&r)[32]) {       // CW columns into r[0..CW)
            if constexpr (CW == 32) { tmem_ld32(addr, r); }
            else if constexpr (CW == 16) {
                uint32_t t16[16];
                tmem_ld16(addr, t16);
#pragma unroll
                for (int i = 0; i < 16; i++) r[i] = t16[i];
            } else {
                uint32_t t8[8];
                tmem_ld8(addr, t8);
#pragma unroll
                for (int i = 0; i < 8; i++) r[i] = t8[i];
            }
        };
        uint32_t ph_d1 = 0, ph_dx = 0, ph_skip = 0, ph_out = 0, ph_bd = 0;
        const __half* embPrev = static_cast<const __half*>(p.embPrev);
        const __half* embCur = static_cast<const __half*>(p.embCur);
        const float* gbias = reinterpret_cast<const float*>(img + im.off_bias);
        int yp = valid ? p.yPrev[b] : 0, yc = valid ? p.yCur[b] : 0;
        float x[CW];                                  // this thread's slice of the residual stream (fp32)
#pragma unroll
        for (int i = 0; i < CW; i++) x[i] = 0.f;
        // History ring (global, read back d samples later by TMA): written AFTER the barrier arrival that publishes the
        // shared-memory tile, then fenced towards the async proxy while this thread would be waiting for the MMA anyway.
        auto store_history = [&](unsigned char* grow) {
#pragma unroll
            for (int q = 0; q < CQ; q++) {
                uint32_t o[4];
#pragma unroll
                for (int j = 0; j < 4; j++) o[j] = pack_h2(x[8 * q + 2 * j], x[8 * q + 2 * j + 1]);
                *reinterpret_cast<uint4*>(grow + chunk_off(u, q4 + q)) = make_uint4(o[0], o[1], o[2], o[3]);   // one copy: row u
            }
            fence_proxy_async_global();
        };
        int n_pub = 0;                                 // tiles published so far: selects the barrier of the pair
        auto publish = [&]() {                         // smem tile written -> visible to the MMA (async proxy), then signal
            tc_fence_before_sync();
            fence_proxy_async_smem();
            mbar_arrive(epi_done + (n_pub & 1) * 17);
            n_pub++;
        };
        auto epi_bar = [&]() { asm volatile("bar.sync 1, 256;" ::: "memory"); };
        // Initialise the pre-activation accumulator of layer `ln` with Lh[tn][ln] + Bh (fp32) straight from the TMA-fed
        // conditioning buffer: tcgen05.st, done while this thread would otherwise wait for the residual GEMM.  Each row
        // needs all 128 columns from the two threads that may touch its TMEM lane: channel half `ch`, both gate halves.
        int g_pre = 0;
        bool tr_on = false;
        auto prestore = [&](int ln) {
            const int cbuf = g_pre % NC;
            mbar_wait(&cond_full[cbuf], (g_pre / NC) & 1);
            if (tid == tr_tid && trc && tr_on && trn < 1023) trc[trn++] = (14ull << 48) | (clock64() & 0xFFFFFFFFFFFFull);
            if (wv) {
                const unsigned char* cb = t_cond + (size_t)cbuf * CB;
                const uint32_t d1n = D1B + (uint32_t)(ln & 1) * 128 + lane_off;
                // only the columns the gate thread of THIS row reads: [c32, c32 + CW) of both gate halves (with DUP the other
                // columns of the row belong to the twin row's thread and are never read from this one)
#pragma unroll
                for (int half = 0; half < 2; half++) {
                    const float* bh = s_bh + (size_t)ln * 128 + 64 * half + c32;
                    uint32_t v[CW];
#pragma unroll
                    for (int q = 0; q < CQ; q++) {
                        const uint4 w = *reinterpret_cast<const uint4*>(cb + (size_t)half * c_bytes + chunk_off(u, q4 + q));
                        const uint32_t wv4[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const float2 f = unpack_h2(wv4[j]);
                            v[8 * q + 2 * j] = __float_as_uint(f.x + bh[8 * q + 2 * j]);
                            v[8 * q + 2 * j + 1] = __float_as_uint(f.y + bh[8 * q + 2 * j + 1]);
                        }
                    }
                    if constexpr (CW == 32) tmem_st32(d1n + 64 * half + c32, v);
                    else if constexpr (CW == 16) tmem_st16(d1n + 64 * half + c32, v);
                    else tmem_st8(d1n + 64 * half + c32, v);
                }
                tmem_st_wait();
            }
            if (tid == tr_tid && trc && tr_on && trn < 1023) trc[trn++] = (15ull << 48) | (clock64() & 0xFFFFFFFFFFFFull);
            tc_fence_before_sync();
            mbar_arrive(&cond_empty[cbuf]);
            mbar_arrive(pre_done);
            g_pre++;
        };
        // relu(acc + bias) of this thread's half of a 256(or S)-wide accumulator -> fp16 rows of the 4-k-tile activation tile
        auto relu_to_tile = [&](uint32_t dacc, const float* bias, int width, float* dump_dst) {
            const int c_lo = sub * (width / NS);
#pragma unroll 1
            for (int c0 = c_lo; c0 < c_lo + width / NS; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(dacc + lane_off + c0, v);
                tmem_ld_wait();
                uint32_t o[16];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bb = *reinterpret_cast<const float4*>(bias + c0 + j);
                    float v0 = fmaxf(__uint_as_float(v[j]) + bb.x, 0.f), v1 = fmaxf(__uint_as_float(v[j + 1]) + bb.y, 0.f);
                    float v2 = fmaxf(__uint_as_float(v[j + 2]) + bb.z, 0.f), v3 = fmaxf(__uint_as_float(v[j + 3]) + bb.w, 0.f);
                    if (!valid) { v0 = 0.f; v1 = 0.f; v2 = 0.f; v3 = 0.f; }
                    o[j >> 1] = pack_h2(v0, v1);
                    o[(j >> 1) + 1] = pack_h2(v2, v3);
                }
                if (dump_dst && valid) {                                // last sample of a dumping launch only
#pragma unroll
                    for (int j = 0; j < 32; j++) dump_dst[c0 + j] = fmaxf(__uint_as_float(v[j]) + bias[c0 + j], 0.f);
                }
                unsigned char* kt = t_big + (size_t)(c0 >> 6) * TILE;
                const int q = (c0 & 63) >> 3;
#pragma unroll
                for (int i = 0; i < 4; i++) st_tile(kt, q + i, make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]));
            }
        };

        for (int t = t_begin; t < t_end; t++) {
            const bool dump = p.dump && (t == t_end - 1);
            tr_on = (t == tr_t);
            const float sel = valid ? __ldg(p.sel + (size_t)(t - p.origin) * B + b) : 0.5f;
            if (!FUSED) prestore(0);                                    // D1[0] <- Lh[t][0] + Bh (Dza of the previous sample is consumed)
            // ---------------- embedding: x0 = tanh(embPrev[yPrev] + embCur[yCur])   (reference.cpp:42-57)
            if (wv) {
                const uint4* ep = reinterpret_cast<const uint4*>(embPrev + (size_t)yp * R + c32);
                const uint4* ec = reinterpret_cast<const uint4*>(embCur + (size_t)yc * R + c32);
#pragma unroll
                for (int q = 0; q < CQ; q++) {
                    const uint4 a = __ldg(ep + q), c = __ldg(ec + q);
                    const uint32_t av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
                    uint32_t o[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const float2 fa = unpack_h2(av[j]), fc = unpack_h2(cv[j]);
                        float e0 = fa.x + fc.x, e1 = fa.y + fc.y;
                        if (p.tanhEmbed) { e0 = wn::tanhf_fast(e0); e1 = wn::tanhf_fast(e1); }
                        if (!valid) { e0 = 0.f; e1 = 0.f; }
                        x[8 * q + 2 * j] = e0; x[8 * q + 2 * j + 1] = e1;
                        o[j] = pack_h2(e0, e1);
                    }
                    st_tile(t_xc, q4 + q, make_uint4(o[0], o[1], o[2], o[3]));
                }
            }
            publish();                                                  // x_0 ready
            if (FUSED) mbar_arrive(hx_full);
            if (tid == tr_tid) TRACE(0, 1);
            if (!FUSED && wv) store_history(ring_tile(t, 0));

            // fused schedule: Lh[t][l] + Bh' of this thread's channels from the TMA-fed conditioning buffer -> registers
            // (done BEFORE waiting for the accumulator)
            float cnd[2 * CW];
            auto load_cond = [&](int ln) {
                const int cbuf = g_pre % NC;
                mbar_wait(&cond_full[cbuf], (g_pre / NC) & 1);
                if (tid == tr_tid) TRACE(0, 14);
                if (wv) {
                    const unsigned char* cb = t_cond + (size_t)cbuf * CB;
#pragma unroll
                    for (int half = 0; half < 2; half++) {
                        const float* bh = s_bh + (size_t)ln * 128 + 64 * half + c32;
#pragma unroll
                        for (int q = 0; q < CQ; q++) {
                            const uint4 w = *reinterpret_cast<const uint4*>(cb + (size_t)half * c_bytes + chunk_off(u, q4 + q));
                            const uint32_t wv4[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                const float2 f = unpack_h2(wv4[j]);
                                cnd[half * CW + 8 * q + 2 * j] = f.x + bh[8 * q + 2 * j];
                                cnd[half * CW + 8 * q + 2 * j + 1] = f.y + bh[8 * q + 2 * j + 1];
                            }
                        }
                    }
                }
                mbar_arrive(&cond_empty[cbuf]);
                g_pre++;
            };
            // gate of layer l: D1[l&1] -> h tile of parity l
            auto gate = [&](int l) {
                const uint32_t d1 = D1B + (uint32_t)(l & 1) * 128 + lane_off;
                unsigned char* th = t_h + (size_t)(l & 1) * TILE;
                uint32_t ta[32], sa[32];
                tmem_ldc(d1 + c32, ta);
                tmem_ldc(d1 + 64 + c32, sa);
                tmem_ld_wait();
                if (tid == tr_tid) TRACE(0, 16);
                uint32_t hp[CW / 2];
#pragma unroll
                for (int j = 0; j < CW; j += 2) {
                    float a0 = __uint_as_float(ta[j]), a1 = __uint_as_float(ta[j + 1]);
                    float g0 = __uint_as_float(sa[j]), g1 = __uint_as_float(sa[j + 1]);
                    if (FUSED) {
                        // the gate is MUFU-bound (2 transcendental per channel): evaluate both as packed fp16 pairs, one
                        // MUFU.TANH per TWO values; h is rounded to fp16 for the next GEMM anyway
                        a0 += cnd[j]; a1 += cnd[j + 1]; g0 += cnd[CW + j]; g1 += cnd[CW + j + 1];
                        const __half2 th = wn::tanh_h2(__floats2half2_rn(a0, a1));
                        const __half2 tg = wn::tanh_h2(__floats2half2_rn(0.5f * g0, 0.5f * g1));
                        const __half2 hh = __hmul2(th, __hfma2(tg, __float2half2_rn(0.5f), __float2half2_rn(0.5f)));
                        hp[j >> 1] = *reinterpret_cast<const uint32_t*>(&hh);
                    } else {
                        const float h0 = wn::tanhf_fast(a0) * wn::sigmoidf_fast(g0);
                        const float h1 = wn::tanhf_fast(a1) * wn::sigmoidf_fast(g1);
                        hp[j >> 1] = pack_h2(h0, h1);
                    }
                }
#pragma unroll
                for (int q = 0; q < CQ; q++) st_tile(th, q4 + q, make_uint4(hp[4 * q], hp[4 * q + 1], hp[4 * q + 2], hp[4 * q + 3]));
                if (tid == tr_tid) TRACE(0, 12);
            };
            // residual of layer l: x += Dx + Bres (Dx in columns [0,64) of D1[l&1]); optionally -> x tile `xt`
            auto residual = [&](int l, unsigned char* xt) {
                const uint32_t d1 = D1B + (uint32_t)(l & 1) * 128 + lane_off;
                const float* br = s_bres + (size_t)l * 64 + c32;
                uint32_t v[32];
                tmem_ldc(d1 + c32, v);
                tmem_ld_wait();
                uint32_t o[CW / 2];
#pragma unroll
                for (int j = 0; j < CW; j += 2) {
                    const float2 bb = *reinterpret_cast<const float2*>(br + j);
                    float v0 = x[j] + (__uint_as_float(v[j]) + bb.x), v1 = x[j + 1] + (__uint_as_float(v[j + 1]) + bb.y);
                    if (!valid) { v0 = 0.f; v1 = 0.f; }
                    x[j] = v0; x[j + 1] = v1;
                    o[j >> 1] = pack_h2(v0, v1);
                }
                if (xt) {
#pragma unroll
                    for (int q = 0; q < CQ; q++) st_tile(xt, q4 + q, make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]));
                }
                if (dump && valid) {                                    // last sample of a dumping launch only
#pragma unroll
                    for (int j = 0; j < CW; j++) p.xtOut[((size_t)l * B + b) * R + c32 + j] = x[j];
                }
            };
            // dump only: skip sum through layer l (complete, and the next contribution not yet issued, at the call sites)
            auto dump_skip = [&](int l) {
                const int c_lo = sub * (S / NS);
                for (int c0 = c_lo; c0 < c_lo + S / NS; c0 += 16) {
                    uint32_t w[16];
                    tmem_ld16(DSKIP + lane_off + c0, w);
                    tmem_ld_wait();
                    if (valid)
                        for (int j = 0; j < 16; j++)
                            p.skipOut[((size_t)l * B + b) * S + c0 + j] = __uint_as_float(w[j]) + gbias[im.b_bskp + (size_t)l * S + c0 + j];
                }
            };

            if (FUSED) {
                for (int l = 0; l < L; l++) {
                    load_cond(l);                                       // in the shadow of the residual GEMM
                    if (tid == tr_tid) TRACE(0, 5);
                    if (l > 0) {
                        // x_l = x_{l-1} + Wres_{l-1}.h_{l-1} + Bres_{l-1}: needed by the NEXT layer's background GEMM and the history
                        mbar_wait(dx_full, ph_dx); ph_dx ^= 1;
                        tc_fence_after_sync();
                        if (tid == tr_tid) TRACE(0, 4);
                        if (wv) residual(l - 1, (l & 1) ? t_x1 : t_xc);
                        tc_fence_before_sync();                         // x_l tile published, Dx consumed
                        fence_proxy_async_smem();
                        mbar_arrive(pre_done);
                        mbar_arrive(hx_full);
                        if (tid == tr_tid) TRACE(0, 13);
                        // B's share of this layer's accumulator (Wprev . x[t-d]) is complete and skip(l-2) has released the h tile
                        mbar_wait(b_done + ((l - 1) & 1) * 3, (ph_bd >> ((l - 1) & 1)) & 1u); ph_bd ^= 1u << ((l - 1) & 1);
                    }
                    mbar_wait(d1_full, ph_d1); ph_d1 ^= 1;
                    tc_fence_after_sync();
                    if (tid == tr_tid) TRACE(0, 2);
                    if (wv) gate(l);
                    if (dump && l > 0 && wv) dump_skip(l - 1);
                    publish();                                          // h_l ready, D1[l&1] drained
                    if (tid == tr_tid) TRACE(0, 3);
                }
                if (L > 1) { mbar_wait(b_done + ((L - 1) & 1) * 3, (ph_bd >> ((L - 1) & 1)) & 1u); ph_bd ^= 1u << ((L - 1) & 1); }
                if (dump) {
                    mbar_wait(dx_full, ph_dx); ph_dx ^= 1;
                    tc_fence_after_sync();
                    if (wv) residual(L - 1, nullptr);
                }
            } else
            for (int l = 0; l < L; l++) {
                // ---------------- gate: h = tanh(a[0:R]) * sigmoid(a[R:2R]); D1 already holds the complete pre-activation
                // a = (Lh[t][l] + Bh) + Wprev.x[t-d] + Wcur.x[t]   (reference.cpp:67-80)
                mbar_wait(d1_full, ph_d1); ph_d1 ^= 1;
                tc_fence_after_sync();
                if (tid == tr_tid) TRACE(0, 2);
                if (wv) gate(l);
                publish();                                              // h ready, D1 drained
                if (tid == tr_tid) TRACE(0, 3);
                if (l + 1 < L) prestore(l + 1);                         // while the residual GEMM runs
                // ---------------- residual: x += Dx + Bres   (reference.cpp:82-84)
                mbar_wait(dx_full, ph_dx); ph_dx ^= 1;
                tc_fence_after_sync();
                if (tid == tr_tid) TRACE(0, 4);
                if (wv) {
                    residual(l, (l + 1 < L) ? t_xc : nullptr);
                    // skip sum through layer l-1 is complete here (its MMAs precede this layer's residual GEMM) and the
                    // next contribution is only issued after the arrival below: no extra barrier needed
                    if (dump && l > 0) dump_skip(l - 1);
                }
                if (l + 1 < L) {
                    publish();                                          // x_{l+1} ready
                    if (tid == tr_tid) TRACE(0, 5);
                    if (wv) store_history(ring_tile(t, l + 1));
                }
            }

            // ---------------- relu(skip) -> GEMM input of the first output layer   (reference.cpp:88-90)
            mbar_wait(skip_full, ph_skip); ph_skip ^= 1;
            tc_fence_after_sync();
            if (tid == tr_tid) TRACE(0, 6);
            if (wv) relu_to_tile(DSKIP, s_bsk, S, dump ? p.skipOut + ((size_t)(L - 1) * B + b) * S : nullptr);
            publish();                                                  // relu(skip) tile ready
            if (tid == tr_tid) TRACE(0, 7);

            // ---------------- Zs = relu(Wzs . skip + Bzs)   (reference.cpp:96-98)
            mbar_wait(out_full, ph_out); ph_out ^= 1;
            tc_fence_after_sync();
            if (wv) relu_to_tile(DZS, s_bzs, A, dump ? p.Zs + (size_t)b * A : nullptr);
            publish();                                                  // relu(Zs) tile ready
            if (tid == tr_tid) TRACE(0, 9);

            // ---------------- Za, softmax, categorical sample   (reference.cpp:100-121)
            // The two threads of an utterance each take 128 logits: a first TMEM pass finds the local max in fp32, a second one parks
            // (z - max) as fp16 in the thread's own row of the (now dead) activation tiles -- the rounding error is proportional to the
            // distance from the row's true max, i.e. negligible where the probability mass is; exp / sums / scan run from shared memory; the
            // halves meet through s_pair (local max, local sum) and s_y.
            mbar_wait(out_full, ph_out); ph_out ^= 1;
            tc_fence_after_sync();
            if (tid == tr_tid) TRACE(0, 10);
            constexpr int PART = A / NS, NCH = PART / 16;               // logits per thread, 16-logit chunks per thread
            const int a_lo = sub * PART;
            float mx = -INFINITY;                                       // the true row max (DESIGN.md §3)
            float csum[NCH];
            float lsum = 0.f;
            auto expz = [&](uint32_t packed, float& e0, float& e1) {       // packed = (z - local max) in fp16
                const float2 z = unpack_h2(packed);
                e0 = wn::exp2f_fast(z.x * 1.4426950408889634f);
                e1 = wn::exp2f_fast(z.y * 1.4426950408889634f);
            };
            if (wv) {
#pragma unroll 1
                for (int c0 = a_lo; c0 < a_lo + PART; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(DZA + lane_off + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        const float z0 = __uint_as_float(v[j]) + s_bza[c0 + j], z1 = __uint_as_float(v[j + 1]) + s_bza[c0 + j + 1];
                        mx = fmaxf(mx, fmaxf(z0, z1));
                        if (dump && valid) { p.Za[(size_t)b * A + c0 + j] = z0; p.Za[(size_t)b * A + c0 + j + 1] = z1; }
                    }
                }
#pragma unroll 1
                for (int c0 = a_lo; c0 < a_lo + PART; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(DZA + lane_off + c0, v);
                    tmem_ld_wait();
                    uint32_t o[16];
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        const float z0 = __uint_as_float(v[j]) + s_bza[c0 + j], z1 = __uint_as_float(v[j + 1]) + s_bza[c0 + j + 1];
                        o[j >> 1] = pack_h2(z0 - mx, z1 - mx);
                    }
                    unsigned char* kt = t_big + (size_t)(c0 >> 6) * TILE;      // scratch: own row only
                    const int q = (c0 & 63) >> 3;
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        *reinterpret_cast<uint4*>(kt + chunk_off(row, q + i)) = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                }
#pragma unroll
                for (int c = 0; c < NCH; c++) {
                    const int c0 = a_lo + 16 * c;
                    const unsigned char* kt = t_big + (size_t)(c0 >> 6) * TILE;
                    const int q = (c0 & 63) >> 3;
                    const uint4 u0 = *reinterpret_cast<const uint4*>(kt + chunk_off(row, q)), u1 = *reinterpret_cast<const uint4*>(kt + chunk_off(row, q + 1));
                    const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
                    float sacc = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; j++) { float e0, e1; expz(w[j], e0, e1); sacc += e0; sacc += e1; }
                    csum[c] = sacc;
                    lsum += sacc;
                }
                s_pair[(u * NS + sub) * 2] = mx;
                s_pair[(u * NS + sub) * 2 + 1] = lsum;
            }
            epi_bar();
            int y = A - 1;
            if (wv) {
                float pm[NS], ps[NS];
                float M = -INFINITY;
#pragma unroll
                for (int i = 0; i < NS; i++) { pm[i] = s_pair[(u * NS + i) * 2]; ps[i] = s_pair[(u * NS + i) * 2 + 1]; M = fmaxf(M, pm[i]); }
                float total = 0.f, off = 0.f, fme = 1.f, mine_hi = 0.f;
#pragma unroll
                for (int i = 0; i < NS; i++) {
                    const float f = wn::exp2f_fast((pm[i] - M) * 1.4426950408889634f);
                    if (i == sub) { off = total; fme = f; }
                    total += ps[i] * f;
                    if (i == sub) mine_hi = total;
                }
                const float target = sel * total;
                // owner = first part whose scaled running sum exceeds the target; the last part takes what is left
                const bool mine = (sub == 0 || !(target < off)) && (target < mine_hi || sub == NS - 1);
                if (mine) {
                    int cb = NCH - 1;
                    float base = off;
                    {
                        float run = off;
                        bool found = false;
#pragma unroll
                        for (int c = 0; c < NCH; c++) {
                            const float nxt = run + csum[c] * fme;
                            if (!found && target < nxt) { cb = c; base = run; found = true; }
                            run = nxt;
                        }
                        if (!found) base = run - csum[NCH - 1] * fme;
                    }
                    const int c0 = a_lo + 16 * cb;
                    const unsigned char* kt = t_big + (size_t)(c0 >> 6) * TILE;
                    const int q = (c0 & 63) >> 3;
                    const uint4 u0 = *reinterpret_cast<const uint4*>(kt + chunk_off(row, q)), u1 = *reinterpret_cast<const uint4*>(kt + chunk_off(row, q + 1));
                    const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
                    float run = base;
                    bool found = false;
                    int yy = (cb == NCH - 1 && sub == NS - 1) ? A - 1 : c0 + 15;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        float e0, e1;
                        expz(w[j], e0, e1);
                        run += e0 * fme;
                        if (!found && target < run) { yy = c0 + 2 * j; found = true; }
                        run += e1 * fme;
                        if (!found && target < run) { yy = c0 + 2 * j + 1; found = true; }
                    }
                    s_y[u] = yy;
                    if (valid) p.yOut[(size_t)b * p.N + (t - p.origin)] = yy;
                }
                if (dump && valid) {
                    const float inv = fme / total;
                    for (int a = a_lo; a < a_lo + PART; a++) {
                        const unsigned char* kt = t_big + (size_t)(a >> 6) * TILE;
                        const float z = __half2float(*reinterpret_cast<const __half*>(kt + chunk_off(row, (a & 63) >> 3) + (a & 7) * 2));
                        p.P[(size_t)b * A + a] = wn::exp2f_fast(z * 1.4426950408889634f) * inv;
                    }
                }
            }
            epi_bar();
            if (wv) y = s_y[u];
            if (valid) {
                const int fb = p.forced ? p.forced[(size_t)b * p.N + (t - p.origin)] : y;
                yp = yc;
                yc = fb;
            }
            if (tid == tr_tid) TRACE(0, 11);
            // Dza is consumed: the x_0-ready arrival of the next sample (or kernel end) releases it
        }
        if (valid && sub == 0) { p.yPrev[b] = yp; p.yCur[b] = yc; }
        tc_fence_before_sync();
    }
#undef TRACE

    __syncthreads();
    if (warp == 8) tmem_dealloc<512>(tmem_base);
}

int pick_nstage(int S, int L)
{
    for (int n = 8; n >= 3; n--)
        if (tc_smem_bytes(S, L, n) <= 227 * 1024) return n;
    return 0;
}

}  // namespace

bool wn_tc_supported(int R_, int S, int A_, int L, int)
{
    return R_ == R && A_ == A && (S == 128 || S == 256) && pick_nstage(S, L) >= 3;
}

size_t wn_tc_image_bytes(int, int S, int, int L) { return tc_image(S, L).total; }

// 64-utterance tiles (the lower-latency four-threads-per-utterance variant) as long as one wave of CTAs covers the batch
// Utterances per CTA tile: 32 (eight threads per utterance) while that keeps the launch small enough to stay latency-bound,
// 64 as long as one wave of CTAs covers the batch, else full 128-row tiles.  NVWN_TC_TILE / NVWN_TC_NODUP force a shape.
int wn_tc_tile_utt(int B, int S)
{
    if (getenv("NVWN_TC_NODUP")) return 128;
    if (const char* v = getenv("NVWN_TC_TILE")) { const int t = atoi(v); if (t == 128 || t == 64 || (t == 32 && S == 256)) return t; }
    // Round 2: the soak test (tests/test_gpu_parity.py::test_fp16_soak_determinism_and_chunking, tools/diag_determinism.py) shows
    // rare run-to-run flips of a sampled index (about one per 1e5 utterance-samples) with the FUSED schedule (32- / 64-utterance
    // tiles) and with the 128-row tiles; the unfused schedule on 64-utterance tiles is clean over the same soak.  Those variants
    // stay reachable through NVWN_TC_TILE / NVWN_TC_NODUP / NVWN_TC_FUSED for investigation but are never selected automatically
    // (the latency-mode kernel, wn_lat_kernel.cu, serves the batches they were meant for).
    return 64;
}

// schedule of an engine, resolved once at creation: "0" / "1" in NVWN_TC_FUSED force one (tests); see wn_tc_tile_utt() for the default
bool wn_tc_fused_default()
{
    const char* fv = getenv("NVWN_TC_FUSED");
    return fv ? fv[0] != '0' : false;
}

size_t wn_tc_ring_bytes(int TU, int L, int maxDil, int B)
{
    return (size_t)(maxDil + 1) * L * ((B + TU - 1) / TU) * TILE;
}

size_t wn_tc_cond_bytes(int TU, int L, int B, int N) { return (size_t)N * L * cond_bpad(B, TU) * 256; }

cudaError_t wn_tc_cond_convert(void* dst, const float* src_dev, int first_sample, int nsamples, int TU, int L, int B, cudaStream_t stream)
{
    if (nsamples <= 0) return cudaSuccess;
    const size_t total = (size_t)nsamples * L * B * 16;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    tc_cond_kernel<<<(unsigned)blocks, 256, 0, stream>>>(static_cast<unsigned char*>(dst), src_dev, first_sample, nsamples, L, B, TU);
    return cudaGetLastError();
}

cudaError_t wn_tc_cond_readback(float* dst_dev, const void* store, int first_sample, int nsamples, int TU, int L, int B, cudaStream_t stream)
{
    if (nsamples <= 0) return cudaSuccess;
    const size_t total = (size_t)nsamples * L * B * 16;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    tc_cond_readback_kernel<<<(unsigned)blocks, 256, 0, stream>>>(dst_dev, static_cast<const unsigned char*>(store), first_sample, nsamples, L, B, TU);
    return cudaGetLastError();
}

cudaError_t wn_tc_pack(void* image, const WnParams& p, cudaStream_t stream)
{
    const TcImage im = tc_image(p.S, p.L);
    cudaError_t e = cudaMemsetAsync(image, 0, im.total, stream);
    if (e != cudaSuccess) return e;
    tc_pack_kernel<<<296, 256, 0, stream>>>(p, static_cast<unsigned char*>(image), im);
    return cudaGetLastError();
}

cudaError_t wn_launch_tc(const WnParams& p, const void* tc_image_, int TU, bool fused, cudaStream_t stream, WnLaunchInfo* info)
{
    const int nstage = pick_nstage(p.S, p.L);
    if (nstage < 3) return cudaErrorInvalidValue;
    const size_t smem = tc_smem_bytes(p.S, p.L, nstage);
    const int grid = (p.B + TU - 1) / TU;
    cudaError_t e = cudaErrorInvalidValue;
    const int cp = 128 / TU;                                    // row copies per utterance: 2 cp threads work for each
    const unsigned char* im8 = static_cast<const unsigned char*>(tc_image_);
    // Fused schedule (one MMA<->epilogue round trip per layer, +1 weight chunk per layer) while the launch is latency-bound;
    // with (nearly) every SM streaming the weights from L2 the extra chunk costs more than the round trip saves
    // (measured, 64-utterance tiles: 2048 utt. 50.9M vs 44.5M samples/s fused; 9472 utt. 175.6M fused vs 196.4M unfused).
#define WN_TC_LAUNCH(SV, DV, FV)                                                                                     \
    do {                                                                                                             \
        e = cudaFuncSetAttribute(wn_tc_kernel<SV, DV, FV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
        if (e != cudaSuccess) return e;                                                                              \
        wn_tc_kernel<SV, DV, FV><<<grid, NT, smem, stream>>>(p, im8, nstage);                                       \
    } while (0)
#define WN_TC_LAUNCH2(SV, DV) do { if (fused) WN_TC_LAUNCH(SV, DV, true); else WN_TC_LAUNCH(SV, DV, false); } while (0)
    if (p.S == 256) {
        if (cp == 4) WN_TC_LAUNCH(256, 4, true);                // 32-utterance tiles exist for the fused schedule only (NVWN_TC_TILE=32)
        else if (cp == 2) WN_TC_LAUNCH2(256, 2);
        else WN_TC_LAUNCH2(256, 1);
    } else {
        if (cp == 2) WN_TC_LAUNCH2(128, 2); else WN_TC_LAUNCH2(128, 1);
    }
#undef WN_TC_LAUNCH2
#undef WN_TC_LAUNCH
    if (info) { info->kernel = 17; info->grid = grid; info->block = NT; info->smem_bytes = (int)smem; info->batch_per_cta = TU; info->cluster = 1; }
    return cudaGetLastError();
}
