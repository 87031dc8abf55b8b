// wn_stream_kernel.cu -- "stream" kernel family: one persistent CTA per batch tile runs the WHOLE
// autoregressive loop (embed -> L x (dilated 2x1 conv + gated tanh*sigmoid + 1x1 residual + 1x1 skip
// accumulate) -> two output layers -> softmax -> categorical sample -> feed back) for `count`
// consecutive samples.  Weights are streamed from L2 every step with coalesced column-major reads;
// activations never leave shared memory; the only HBM streams are the conditioning Lh (prefetched one
// layer ahead into registers) and the dilation history ring.
//
// Replaces nv_wavenet_{singleblock,dualblock,persistent}.cuh + matrix_math.cuh + softmax.cuh of the
// reference for
//   * fp32 (TD=float): the BIT-EXACT path.  Operation order is the reference CPU model's
//     (nv_wavenet_reference.cpp:59-121, matrix.cpp:85-183): left-to-right dot products with separately
//     rounded multiply and add, ((a_prev + a_cur) + Bh) + Lh, (Wres.h + Bres) + x, (Wskip.h + skip) + Bskip,
//     softmax with max initialised to 0, sequential sum and p = e / sum, first index with sel < cumsum(p).
//     exp/tanh are the portable double-precision forms of wn_math.cuh.  A CPU evaluation of the same
//     formulas (oracle/wavenet_oracle.c, PORTABLE mode) gives identical bits.
//   * fp16 storage (TD=__half): weights / Lh / ring in fp16, GEMM inputs rounded to fp16, fp32 FMA
//     accumulate, fast MUFU transcendentals.  Fallback for shapes the tensor-core kernel does not cover.
//
// RING = true (fp32, A <= threads): the weights do not come through per-thread L2 loads but through a shared-memory ring of
// bulk-TMA pieces (cp.async.bulk + mbarrier complete_tx), issued by one lane of an extra warp in exactly the order the stages
// consume them: per layer the column slabs [Wprev | Wcur] of stage 1 and [Wres | Wskip] of stage 3, per sample the slabs of Wzs
// and Wza.  A slab of a column-major matrix is contiguous, so every piece is one or two plain 1-D copies; a thread reads its row
// of the slab with conflict-free 4-byte shared loads.  The arithmetic and its order are untouched (same bits).
#include "wn_common.h"
#include "wn_math.cuh"
#include "wn_sm100.cuh"

#include <type_traits>

namespace {

template <typename TD> struct Num;
template <> struct Num<float> {
    static constexpr bool exact = true;
    static constexpr bool true_max = false;
    static __device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
    static __device__ __forceinline__ float ldcg(const float* p) { return __ldcg(p); }
    static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
    static __device__ __forceinline__ float q(float v) { return v; }
    static __device__ __forceinline__ float mac(float acc, float w, float x) { return __fadd_rn(acc, __fmul_rn(w, x)); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float tanh_(float v) { return wn::tanhf_portable(v); }
    static __device__ __forceinline__ float sigmoid_(float v) { return wn::sigmoidf_portable(v); }
};
template <> struct Num<__half> {
    static constexpr bool exact = false;
    static constexpr bool true_max = true;      // softmax from the true row max, not from max(0, logits) as the reference does
    static __device__ __forceinline__ float ld(const __half* p) { return __half2float(__ldg(p)); }
    static __device__ __forceinline__ float ldcg(const __half* p) { return __half2float(__ldcg(p)); }
    static __device__ __forceinline__ void st(__half* p, float v) { *p = __float2half_rn(v); }
    static __device__ __forceinline__ float q(float v) { return __half2float(__float2half_rn(v)); }
    static __device__ __forceinline__ float mac(float acc, float w, float x) { return fmaf(w, x, acc); }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float tanh_(float v) { return wn::tanhf_fast(v); }
    static __device__ __forceinline__ float sigmoid_(float v) { return wn::sigmoidf_fast(v); }
};

// fp32 in the REFERENCE GPU KERNELS' arithmetic (NVWN_FP32_FAST): fused multiply-add, two interleaved partial sums per dot
// product (GEMM<R,2>, matrix_math.cuh:80-117), single-precision libm tanh / exp.  Not bit-identical to the CPU model -- it
// agrees with it like the reference's own kernels do (sampled indices equal unless a selector falls within rounding of a
// class boundary; nv_wavenet_test.cu:273-298 tolerances on the activations) -- but free of the 8-cycle-per-term serial chain.
struct NumFast32 {
    static constexpr bool exact = false;
    static constexpr bool true_max = false;     // the reference GPU kernels' softmax, max starting at 0
    static __device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
    static __device__ __forceinline__ float ldcg(const float* p) { return __ldcg(p); }
    static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
    static __device__ __forceinline__ float q(float v) { return v; }
    static __device__ __forceinline__ float mac(float acc, float w, float x) { return fmaf(w, x, acc); }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float tanh_(float v) { return tanhf(v); }
    static __device__ __forceinline__ float sigmoid_(float v) { return 1.f / (1.f + expf(-v)); }
};
template <typename TD, bool FAST> struct NumSel { using type = Num<TD>; };
template <> struct NumSel<float, true> { using type = NumFast32; };

// acc[b] = sum_k W[row + k*M] * xs[b][k], k ascending (matrix.cpp:85-102 order).
// KB weights are requested back to back before the first use, so the L2 latency is paid once per
// KB columns instead of once per 8.
template <typename TD, int BT, int KB, bool FAST>
__device__ __forceinline__ void dot_cols(const TD* __restrict__ W, int M, int K, int row,
                                         const float* __restrict__ xs, float (&acc)[BT])
{
    using N = typename NumSel<TD, FAST>::type;
    float odd[BT];                                   // second partial sum of the non-exact contracts (odd k)
#pragma unroll
    for (int b = 0; b < BT; b++) { acc[b] = 0.f; odd[b] = 0.f; }
    const TD* wp = W + row;
#pragma unroll 1
    for (int k0 = 0; k0 < K; k0 += KB) {
        float w[KB];
#pragma unroll
        for (int j = 0; j < KB; j++) w[j] = N::ld(wp + (size_t)(k0 + j) * M);
#pragma unroll
        for (int j = 0; j < KB; j += 4) {
#pragma unroll
            for (int b = 0; b < BT; b++) {
                const float4 xa = *reinterpret_cast<const float4*>(xs + b * K + k0 + j);
                if (N::exact) {
                    float a = acc[b];
                    a = N::mac(a, w[j], xa.x); a = N::mac(a, w[j + 1], xa.y); a = N::mac(a, w[j + 2], xa.z); a = N::mac(a, w[j + 3], xa.w);
                    acc[b] = a;
                } else {
                    float a = acc[b], o = odd[b];
                    a = N::mac(a, w[j], xa.x); o = N::mac(o, w[j + 1], xa.y); a = N::mac(a, w[j + 2], xa.z); o = N::mac(o, w[j + 3], xa.w);
                    acc[b] = a; odd[b] = o;
                }
            }
        }
    }
    if (!N::exact) {
#pragma unroll
        for (int b = 0; b < BT; b++) acc[b] += odd[b];
    }
}

// the same sum continued over one column slab held in shared memory: ws[k * M + row], k < KS; xs points at column k0 of the inputs
// (MC = M when it is a compile-time constant: the shared loads then carry immediate offsets)
__device__ __forceinline__ float lds_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
template <int BT, int KS, int MC, bool FAST, typename N>
__device__ __forceinline__ void dot_slab(const float* __restrict__ ws, int Mrt, int row, const float* __restrict__ xs, int K,
                                         float (&acc)[BT], float (&odd)[BT])
{
    const int M = MC ? MC : Mrt;
    const uint32_t wp = sm100::smem_u32(ws + row);
#pragma unroll
    for (int j = 0; j < KS; j += 4) {
        const float w0 = lds_f32(wp + (j + 0) * M * 4), w1 = lds_f32(wp + (j + 1) * M * 4), w2 = lds_f32(wp + (j + 2) * M * 4), w3 = lds_f32(wp + (j + 3) * M * 4);
#pragma unroll
        for (int b = 0; b < BT; b++) {
            const float4 xa = *reinterpret_cast<const float4*>(xs + b * K + j);
            if (N::exact) {
                float a = acc[b];
                a = N::mac(a, w0, xa.x); a = N::mac(a, w1, xa.y); a = N::mac(a, w2, xa.z); a = N::mac(a, w3, xa.w);
                acc[b] = a;
            } else {
                float a = acc[b], o = odd[b];
                a = N::mac(a, w0, xa.x); o = N::mac(o, w1, xa.y); a = N::mac(a, w2, xa.z); o = N::mac(o, w3, xa.w);
                acc[b] = a; odd[b] = o;
            }
        }
    }
}

constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int cmin(int a, int b) { return a < b ? a : b; }

// geometry of the weight ring (RING kernels): slab widths so that a piece stays at or below 40 KB
template <int R, int S> struct RingCfg {
    static constexpr int PIECE = 40960, SLOTS = 4;
    static constexpr int pow2_le(int v) { int k = 4; while (2 * k <= v) k *= 2; return k; }
    static constexpr int KS1 = cmin(cmin(R, 32), pow2_le(PIECE / (4 * R * 4)));      // [Wprev | Wcur]: 4R rows of floats per column
    static constexpr int KS3 = cmin(cmin(R, 32), pow2_le(PIECE / ((R + S) * 4)));    // [Wres | Wskip]: R + S rows per column
    static constexpr int NS1 = R / KS1, NS3 = R / KS3;
    static_assert(KS1 >= 4 && KS3 >= 4 && R % KS1 == 0 && R % KS3 == 0 && (R + S) * KS3 * 4 <= PIECE && 4 * R * KS1 * 4 <= PIECE, "piece geometry");
    static __host__ __device__ int kso(int A) { int k = 32; while (k > 4 && A * k * 4 > PIECE) k >>= 1; return k; }   // output layers: A rows per column
};

template <int R, int S> struct Shape {
    static constexpr int NT = cmax(cmax(4 * R, R + S), 128);       // threads per CTA
};

template <int R, int S, int BT>
__host__ __device__ constexpr size_t stream_smem_floats(int A, int L)
{
    return (size_t)BT * (3 * R + 4 * R + R + 2 * S + 3 * A) + BT * 4 + BT * 2 + L + 4;
}

template <typename TD, int R, int S, int BT, bool FAST, bool RING>
__global__ void __launch_bounds__(Shape<R, S>::NT + (RING ? 32 : 0), 1) wn_stream_kernel(const WnParams p)
{
    using N = typename NumSel<TD, FAST>::type;
    using RC = RingCfg<R, S>;
    static_assert(!RING || std::is_same<TD, float>::value, "the weight ring is the fp32 kernels'");
    constexpr int NT = Shape<R, S>::NT;
    constexpr int NACT = 2 * R * BT;
    constexpr int ACT_PER = (NACT + NT - 1) / NT;
    constexpr int KBR = R < 64 ? R : 64;          // weight columns in flight per thread in the R-deep dots
    static_assert(R * BT <= NT, "one x-task per thread");

    const int tid = threadIdx.x;
    const int A = p.A, L = p.L, B = p.B;
    const int b0 = blockIdx.x * BT;
    const int slots = p.maxDil + 1;

    extern __shared__ __align__(16) float sm[];
    float* x = sm;                         // [BT][R]   residual stream, fp32
    float* xq = x + BT * R;                // [BT][R]   GEMM input of the current layer
    float* xp = xq + BT * R;               // [BT][R]   GEMM input x[t-d]
    float* ap = xp + BT * R;               // [BT][2R]  Wprev . x[t-d]
    float* ac = ap + BT * 2 * R;           // [BT][2R]  Wcur . x[t]   -> overwritten by tanh / sigmoid values
    float* hq = ac + BT * 2 * R;           // [BT][R]   gated activation, GEMM input
    float* skip = hq + BT * R;             // [BT][S]   running skip sum, fp32
    float* skq = skip + BT * S;            // [BT][S]   relu(skip) as GEMM input
    float* zsq = skq + BT * S;             // [BT][A]
    float* za = zsq + BT * A;              // [BT][A]   logits
    float* ex = za + BT * A;               // [BT][A]   exp / p
    float* red = ex + BT * A;              // [BT][4]   max, sum
    int* ysm = reinterpret_cast<int*>(red + BT * 4);   // [BT][2]  yPrev, yCur
    int* dil = ysm + BT * 2;               // [L]
    // RING: [SLOTS] pieces, 128-byte aligned behind the activations, then full[SLOTS] / empty[SLOTS] barriers
    float* ring_w = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(dil + L + 4) + 127) & ~uintptr_t(127));
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(ring_w + RC::SLOTS * (RC::PIECE / 4));
    uint64_t* bar_empty = bar_full + RC::SLOTS;
    // all compute threads (the producer warp of the RING kernels is not among them)
    auto SYNC = [&]() { if (RING) asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); else __syncthreads(); };

    const TD* embPrev = static_cast<const TD*>(p.embPrev);
    const TD* embCur = static_cast<const TD*>(p.embCur);
    const TD* Wprev = static_cast<const TD*>(p.Wprev);
    const TD* Wcur = static_cast<const TD*>(p.Wcur);
    const TD* Wres = static_cast<const TD*>(p.Wres);
    const TD* Wskip = static_cast<const TD*>(p.Wskip);
    const TD* Wzs = static_cast<const TD*>(p.Wzs);
    const TD* Wza = static_cast<const TD*>(p.Wza);
    const TD* Bh = static_cast<const TD*>(p.Bh);
    const TD* Bres = static_cast<const TD*>(p.Bres);
    const TD* Bskip = static_cast<const TD*>(p.Bskip);
    const TD* Bzs = static_cast<const TD*>(p.Bzs);
    const TD* Bza = static_cast<const TD*>(p.Bza);
    const TD* Lh = static_cast<const TD*>(p.Lh);
    TD* ring = static_cast<TD*>(p.ring);

    // dilation schedule 1,2,4..maxDil,1,2..  (nv_wavenet.cuh:99-111, reference.cpp:285-289)
    if (tid == 0) {
        int d = 1;
        for (int l = 0; l < L; l++) { dil[l] = d; d <<= 1; if (d > p.maxDil) d = 1; }
    }
    if (tid < BT) { ysm[tid * 2] = p.yPrev[b0 + tid]; ysm[tid * 2 + 1] = p.yCur[b0 + tid]; }
    if (RING && tid == 0) {
        for (int i = 0; i < RC::SLOTS; i++) { sm100::mbar_init(bar_full + i, 1); sm100::mbar_init(bar_empty + i, NT / 32); }
        sm100::fence_mbar_init();
    }
    __syncthreads();

    const int kso = RC::kso(A);
    if (RING && tid >= NT) {
        // ---- producer warp: one lane streams the pieces in consumption order ----
        if (tid == NT) {
            const float* fWprev = reinterpret_cast<const float*>(p.Wprev); const float* fWcur = reinterpret_cast<const float*>(p.Wcur);
            const float* fWres = reinterpret_cast<const float*>(p.Wres); const float* fWskip = reinterpret_cast<const float*>(p.Wskip);
            const float* fWzs = reinterpret_cast<const float*>(p.Wzs); const float* fWza = reinterpret_cast<const float*>(p.Wza);
            uint32_t n = 0;
            auto put = [&](const float* s0, uint32_t f0, const float* s1, uint32_t f1) {       // floats of the one or two parts of a piece
                const uint32_t sl = n % RC::SLOTS;
                sm100::mbar_wait(bar_empty + sl, ((n / RC::SLOTS) & 1) ^ 1);
                sm100::mbar_arrive_expect_tx(bar_full + sl, (f0 + f1) * 4);
                float* dst = ring_w + sl * (RC::PIECE / 4);
                sm100::tma_load_1d(dst, s0, f0 * 4, bar_full + sl);
                if (f1) sm100::tma_load_1d(dst + f0, s1, f1 * 4, bar_full + sl);
                n++;
            };
            for (int t = p.init_sample; t < p.init_sample + p.count; t++) {
                for (int l = 0; l < L; l++) {
                    for (int j = 0; j < RC::NS1; j++)
                        put(fWprev + (size_t)l * 2 * R * R + (size_t)j * RC::KS1 * 2 * R, 2 * R * RC::KS1, fWcur + (size_t)l * 2 * R * R + (size_t)j * RC::KS1 * 2 * R, 2 * R * RC::KS1);
                    for (int j = 0; j < RC::NS3; j++)
                        put(fWres + (size_t)l * R * R + (size_t)j * RC::KS3 * R, R * RC::KS3, fWskip + (size_t)l * S * R + (size_t)j * RC::KS3 * S, S * RC::KS3);
                }
                for (int j = 0; j < S / kso; j++) put(fWzs + (size_t)j * kso * A, (uint32_t)(A * kso), nullptr, 0);
                for (int j = 0; j < A / kso; j++) put(fWza + (size_t)j * kso * A, (uint32_t)(A * kso), nullptr, 0);
            }
        }
        return;
    }
    // consumer side of the ring: every compute warp takes every piece (whether or not its threads have rows in that stage)
    uint32_t pcn = 0;
    auto piece_wait = [&]() -> const float* {
        const uint32_t sl = pcn % RC::SLOTS;
        sm100::mbar_wait(bar_full + sl, (pcn / RC::SLOTS) & 1);
        return ring_w + sl * (RC::PIECE / 4);
    };
    auto piece_done = [&]() {
        __syncwarp();
        if ((tid & 31) == 0) sm100::mbar_arrive(bar_empty + pcn % RC::SLOTS);
        pcn++;
    };

    // fixed per-thread roles
    const bool has_x = tid < R * BT;
    const int xb = has_x ? tid / R : 0, xr = has_x ? tid % R : 0;

    const int t_end = p.init_sample + p.count;
    auto ring_at = [&](int t, int l, int b, int r) -> TD* {
        return ring + (((size_t)(t % slots) * L + l) * B + (b0 + b)) * R + r;
    };
    auto lh_at = [&](int t, int l, int idx) -> const TD* {
        const int b = idx / (2 * R), row = idx % (2 * R);
        return Lh + (((size_t)t * L + l) * B + (b0 + b)) * (2 * R) + row;
    };

    // prefetch registers for (t = init, l = 0)
    float lh_nxt[ACT_PER], bh_nxt[ACT_PER];
    float xp_nxt = 0.f;
    {
        const int t = p.init_sample;
#pragma unroll
        for (int j = 0; j < ACT_PER; j++) {
            const int idx = tid + j * NT;
            lh_nxt[j] = (idx < NACT && t < t_end) ? N::ldcg(lh_at(t, 0, idx)) : 0.f;
            bh_nxt[j] = (idx < NACT) ? N::ld(Bh + idx % (2 * R)) : 0.f;
        }
        if (has_x) xp_nxt = (t >= 1) ? N::ldcg(ring_at(t - 1, 0, xb, xr)) : 0.f;
    }

    for (int t = p.init_sample; t < t_end; t++) {
        const bool dump = p.dump && (t == t_end - 1);
        // ---- embedding (nv_wavenet_reference.cpp:42-57) ----
        if (has_x) {
            const int yp = ysm[xb * 2], yc = ysm[xb * 2 + 1];
            float e = N::add(N::ld(embPrev + (size_t)yp * R + xr), N::ld(embCur + (size_t)yc * R + xr));
            if (p.tanhEmbed) e = N::tanh_(e);
            x[xb * R + xr] = e;
            xq[xb * R + xr] = N::q(e);
            N::st(ring_at(t, 0, xb, xr), e);
            xp[xb * R + xr] = xp_nxt;
        }
        for (int i = tid; i < S * BT; i += NT) skip[i] = 0.f;     // zero matrix (reference.cpp:290)
        SYNC();

        for (int l = 0; l < L; l++) {
            // ---- conditioning / history prefetch for the next layer (or layer 0 of the next sample) ----
            float lh_cur[ACT_PER], bh_cur[ACT_PER];
#pragma unroll
            for (int j = 0; j < ACT_PER; j++) { lh_cur[j] = lh_nxt[j]; bh_cur[j] = bh_nxt[j]; }
            {
                const bool wrap = (l + 1 == L);
                const int tn = wrap ? t + 1 : t, ln = wrap ? 0 : l + 1;
                const bool live = tn < t_end;
#pragma unroll
                for (int j = 0; j < ACT_PER; j++) {
                    const int idx = tid + j * NT;
                    lh_nxt[j] = (live && idx < NACT) ? N::ldcg(lh_at(tn, ln, idx)) : 0.f;
                    bh_nxt[j] = (idx < NACT) ? N::ld(Bh + (size_t)ln * 2 * R + idx % (2 * R)) : 0.f;
                }
                // x[t-d] of the next layer.  For (t+1, layer 0) the source is this sample's embedding,
                // written above by this CTA and ordered by the barriers in between.
                const int dn = dil[ln];
                xp_nxt = (live && has_x && tn >= dn) ? N::ldcg(ring_at(tn - dn, ln, xb, xr)) : 0.f;
            }

            // ---- stage 1: a_prev = Wprev.x[t-d], a_cur = Wcur.x[t]  (reference.cpp:61-65) ----
            if (RING) {
                const bool cur = tid >= 2 * R;
                const int row = cur ? tid - 2 * R : tid;
                float acc[BT], odd[BT];
#pragma unroll
                for (int b = 0; b < BT; b++) { acc[b] = 0.f; odd[b] = 0.f; }
                for (int j = 0; j < RC::NS1; j++) {
                    const float* pw = piece_wait();
                    if (tid < 4 * R)
                        dot_slab<BT, RC::KS1, 2 * R, FAST, N>(pw + (cur ? 2 * R * RC::KS1 : 0), 2 * R, row, (cur ? xq : xp) + j * RC::KS1, R, acc, odd);
                    piece_done();
                }
                if (tid < 4 * R) {
                    float* dst = cur ? ac : ap;
#pragma unroll
                    for (int b = 0; b < BT; b++) dst[b * 2 * R + row] = N::exact ? acc[b] : acc[b] + odd[b];
                }
            } else if (tid < 4 * R) {
                const bool cur = tid >= 2 * R;
                const int row = cur ? tid - 2 * R : tid;
                const TD* W = (cur ? Wcur : Wprev) + (size_t)l * 2 * R * R;
                float acc[BT];
                dot_cols<TD, BT, KBR, FAST>(W, 2 * R, R, row, cur ? xq : xp, acc);
                float* dst = cur ? ac : ap;
#pragma unroll
                for (int b = 0; b < BT; b++) dst[b * 2 * R + row] = acc[b];
            }
            SYNC();

            // ---- pre-activation adds and tanh / sigmoid (reference.cpp:67-72, 76-78) ----
#pragma unroll
            for (int j = 0; j < ACT_PER; j++) {
                const int idx = tid + j * NT;
                if (idx < NACT) {
                    const int row = idx % (2 * R);
                    float v = N::add(ap[idx], ac[idx]);
                    v = N::add(v, bh_cur[j]);
                    v = N::add(v, lh_cur[j]);
                    ac[idx] = (row < R) ? N::tanh_(v) : N::sigmoid_(v);
                }
            }
            SYNC();

            // ---- h = tanh * sigmoid; stage-1 inputs are dead, install x[t-d] of the next layer ----
            if (has_x) {
                const float h = N::mul(ac[xb * 2 * R + xr], ac[xb * 2 * R + xr + R]);
                hq[xb * R + xr] = N::q(h);
                xp[xb * R + xr] = xp_nxt;
            }
            SYNC();

            // ---- stage 3: residual (reference.cpp:82-84) and skip (reference.cpp:86-90) ----
            float acc[BT];
            if (RING) {
                const bool is_res = tid < R;
                const int row = is_res ? tid : tid - R;
                float odd[BT];
#pragma unroll
                for (int b = 0; b < BT; b++) { acc[b] = 0.f; odd[b] = 0.f; }
                for (int j = 0; j < RC::NS3; j++) {
                    const float* pw = piece_wait();
                    if (tid < R) dot_slab<BT, RC::KS3, R, FAST, N>(pw, R, row, hq + j * RC::KS3, R, acc, odd);
                    else if (tid < R + S) dot_slab<BT, RC::KS3, S, FAST, N>(pw + R * RC::KS3, S, row, hq + j * RC::KS3, R, acc, odd);
                    piece_done();
                }
                if (!N::exact) {
#pragma unroll
                    for (int b = 0; b < BT; b++) acc[b] += odd[b];
                }
            }
            if (tid < R + S) {
                const bool is_res = tid < R;
                const int row = is_res ? tid : tid - R;
                const TD* W = is_res ? Wres + (size_t)l * R * R : Wskip + (size_t)l * S * R;
                const float bias = is_res ? N::ld(Bres + (size_t)l * R + row) : N::ld(Bskip + (size_t)l * S + row);
                if (!RING) dot_cols<TD, BT, KBR, FAST>(W, is_res ? R : S, R, row, hq, acc);
                if (is_res) {
#pragma unroll
                    for (int b = 0; b < BT; b++) {
                        float v = N::add(acc[b], bias);
                        v = N::add(v, x[b * R + row]);
                        x[b * R + row] = v;
                        xq[b * R + row] = N::q(v);
                        if (l + 1 < L) N::st(ring_at(t, l + 1, b, row), v);
                        if (dump) p.xtOut[((size_t)l * B + b0 + b) * R + row] = v;
                    }
                } else {
#pragma unroll
                    for (int b = 0; b < BT; b++) {
                        float v = N::add(acc[b], skip[b * S + row]);
                        v = N::add(v, bias);
                        if (l == L - 1) { v = (v < 0.f) ? 0.f : v; skq[b * S + row] = N::q(v); }
                        skip[b * S + row] = v;
                        if (dump) p.skipOut[((size_t)l * B + b0 + b) * S + row] = v;
                    }
                }
            }
            SYNC();
        }

        // ---- output layers (reference.cpp:93-104) ----
        // (RING kernels: A <= NT, one row per thread; the slabs of Wzs, then of Wza, come through the ring)
        auto out_dot = [&](const TD* W, int K, int row, const float* xs, float (&acc)[BT]) {
            if (RING) {
                float odd[BT];
#pragma unroll
                for (int b = 0; b < BT; b++) { acc[b] = 0.f; odd[b] = 0.f; }
                for (int j = 0; j < K / kso; j++) {
                    const float* pw = piece_wait();
                    if (row < A) {
                        if (A == 256 && kso == 32) dot_slab<BT, 32, 256, FAST, N>(pw, A, row, xs + j * 32, K, acc, odd);
                        else if (kso == 32) dot_slab<BT, 32, 0, FAST, N>(pw, A, row, xs + j * 32, K, acc, odd);
                        else if (kso == 16) dot_slab<BT, 16, 0, FAST, N>(pw, A, row, xs + j * 16, K, acc, odd);
                        else if (kso == 8) dot_slab<BT, 8, 0, FAST, N>(pw, A, row, xs + j * 8, K, acc, odd);
                        else dot_slab<BT, 4, 0, FAST, N>(pw, A, row, xs + j * 4, K, acc, odd);
                    }
                    piece_done();
                }
                if (!N::exact) {
#pragma unroll
                    for (int b = 0; b < BT; b++) acc[b] += odd[b];
                }
            } else {
                dot_cols<TD, BT, 32, FAST>(W, A, K, row, xs, acc);
            }
        };
        for (int row = tid; row < (RING ? NT : A); row += NT) {
            float acc[BT];
            out_dot(Wzs, S, row, skq, acc);
            if (row < A) {
                const float bias = N::ld(Bzs + row);
#pragma unroll
                for (int b = 0; b < BT; b++) {
                    float v = N::add(acc[b], bias);
                    v = (v < 0.f) ? 0.f : v;
                    zsq[b * A + row] = N::q(v);
                    if (dump) p.Zs[(size_t)(b0 + b) * A + row] = v;
                }
            }
        }
        SYNC();
        for (int row = tid; row < (RING ? NT : A); row += NT) {
            float acc[BT];
            out_dot(Wza, A, row, zsq, acc);
            if (row < A) {
                const float bias = N::ld(Bza + row);
#pragma unroll
                for (int b = 0; b < BT; b++) {
                    const float v = N::add(acc[b], bias);
                    za[b * A + row] = v;
                    if (dump) p.Za[(size_t)(b0 + b) * A + row] = v;
                }
            }
        }
        SYNC();

        // ---- softmax + categorical sample ----
        const int warp = tid >> 5, lane = tid & 31;
        if (N::exact) {
            // matrix.cpp:167-183 and reference.cpp:106-121, bit for bit
            if (warp < BT) {
                float mx = 0.f;                                      // "float max = 0.f"
                for (int a = lane; a < A; a += 32) mx = fmaxf(mx, za[warp * A + a]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                if (lane == 0) red[warp * 4] = mx;
            }
            SYNC();
            for (int i = tid; i < A * BT; i += NT) ex[i] = wn::expf_portable(__fsub_rn(za[i], red[(i / A) * 4]));
            SYNC();
            if (tid < BT) {
                float s = 0.f;
                const float* e = ex + tid * A;
                for (int a = 0; a < A; a += 4) {
                    const float4 v = *reinterpret_cast<const float4*>(e + a);
                    s = __fadd_rn(s, v.x); s = __fadd_rn(s, v.y); s = __fadd_rn(s, v.z); s = __fadd_rn(s, v.w);
                }
                red[tid * 4 + 1] = s;
            }
            SYNC();
            for (int i = tid; i < A * BT; i += NT) {
                const float pr = __fdiv_rn(ex[i], red[(i / A) * 4 + 1]);
                ex[i] = pr;
                if (dump) p.P[(size_t)(b0 + i / A) * A + (i % A)] = pr;
            }
            SYNC();
            if (tid < BT) {
                const float sel = p.sel[(size_t)t * B + b0 + tid];
                const float* pr = ex + tid * A;
                float cs = 0.f;
                int y = -1;
                for (int a = 0; a < A; a++) {
                    cs = __fadd_rn(cs, pr[a]);
                    if (sel < cs) { y = a; break; }
                }
                if (y < 0) y = A - 1;       // the reference asserts here (reference.cpp:119)
                p.yOut[(size_t)(b0 + tid) * p.N + t] = y;
                const int fb = p.forced ? p.forced[(size_t)(b0 + tid) * p.N + t] : y;
                ysm[tid * 2] = ysm[tid * 2 + 1];
                ysm[tid * 2 + 1] = fb;
            }
        } else {
            // one warp per utterance; lane owns A/32 consecutive rows so that the scan is in row order
            if (warp < BT) {
                const int per = A / 32;
                const float* z = za + warp * A + lane * per;
                float mx = N::true_max ? -INFINITY : 0.f;          // fp16: the true row max (DESIGN.md §3)
                for (int j = 0; j < per; j++) mx = fmaxf(mx, z[j]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                float* e = ex + warp * A + lane * per;
                float ls = 0.f;
                for (int j = 0; j < per; j++) {
                    const float v = wn::exp2f_fast((z[j] - mx) * 1.4426950408889634f);
                    e[j] = v;
                    ls += v;
                }
                float inc = ls;                                     // inclusive scan over lanes
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float v = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += v;
                }
                const float total = __shfl_sync(0xffffffffu, inc, 31);
                const float target = p.sel[(size_t)t * B + b0 + warp] * total;
                const unsigned hit = __ballot_sync(0xffffffffu, target < inc);
                int y = A - 1;
                if (hit) {
                    const int first = __ffs(hit) - 1;
                    if (lane == first) {
                        float cs = inc - ls;
                        y = lane * per + per - 1;
                        for (int j = 0; j < per; j++) {
                            cs += e[j];
                            if (target < cs) { y = lane * per + j; break; }
                        }
                    }
                    y = __shfl_sync(0xffffffffu, y, first);
                }
                if (dump) {
                    const float inv = 1.f / total;
                    for (int j = 0; j < per; j++) p.P[(size_t)(b0 + warp) * A + lane * per + j] = e[j] * inv;
                }
                if (lane == 0) {
                    p.yOut[(size_t)(b0 + warp) * p.N + t] = y;
                    const int fb = p.forced ? p.forced[(size_t)(b0 + warp) * p.N + t] : y;
                    ysm[warp * 2] = ysm[warp * 2 + 1];
                    ysm[warp * 2 + 1] = fb;
                }
            }
        }
        SYNC();
    }

    if (tid < BT) { p.yPrev[b0 + tid] = ysm[tid * 2]; p.yCur[b0 + tid] = ysm[tid * 2 + 1]; }
}

template <typename TD, int R, int S, int BT, bool FAST, bool RING>
cudaError_t launch_kernel(const WnParams& p, cudaStream_t stream, WnLaunchInfo* info)
{
    constexpr int NT = Shape<R, S>::NT;
    using RC = RingCfg<R, S>;
    size_t smem = stream_smem_floats<R, S, BT>(p.A, p.L) * sizeof(float);
    if (RING) smem += 128 + (size_t)RC::SLOTS * RC::PIECE + 2 * RC::SLOTS * sizeof(uint64_t);
    auto kfn = wn_stream_kernel<TD, R, S, BT, FAST, RING>;
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int grid = p.B / BT, block = NT + (RING ? 32 : 0);
    kfn<<<grid, block, smem, stream>>>(p);
    if (info) { info->grid = grid; info->block = block; info->smem_bytes = (int)smem; info->batch_per_cta = BT; info->cluster = 1; }
    return cudaGetLastError();
}

// fp32: weights through the shared-memory ring when the output layers fit one row per thread and every matrix starts on a
// 16-byte boundary (bulk copies); NVWN_STREAM_RING=0 keeps the per-thread L2 loads
template <typename TD, int R, int S, int BT, bool FAST>
cudaError_t launch_one(const WnParams& p, cudaStream_t stream, WnLaunchInfo* info)
{
    if constexpr (std::is_same<TD, float>::value && R <= 64) {                 // (R = 128: measured slower than the per-thread loads)
        static const bool want = [] { const char* v = getenv("NVWN_STREAM_RING"); return !v || atoi(v) != 0; }();
        const void* mats[] = {p.Wprev, p.Wcur, p.Wres, p.Wskip, p.Wzs, p.Wza};
        bool ok = want && p.A <= Shape<R, S>::NT && p.A % 32 == 0;
        for (const void* m : mats) ok = ok && (reinterpret_cast<uintptr_t>(m) & 15) == 0;
        const size_t smem = stream_smem_floats<R, S, BT>(p.A, p.L) * sizeof(float) + 128 + (size_t)RingCfg<R, S>::SLOTS * RingCfg<R, S>::PIECE + 64;
        if (ok && smem <= 232448) return launch_kernel<TD, R, S, BT, FAST, true>(p, stream, info);
    }
    return launch_kernel<TD, R, S, BT, FAST, false>(p, stream, info);
}

template <typename TD, int R, int S, bool FAST>
cudaError_t launch_bt(const WnParams& p, int bt, cudaStream_t stream, WnLaunchInfo* info)
{
    switch (bt) {
        case 4: return launch_one<TD, R, S, 4, FAST>(p, stream, info);
        case 2: return launch_one<TD, R, S, 2, FAST>(p, stream, info);
        default: return launch_one<TD, R, S, 1, FAST>(p, stream, info);
    }
}

template <typename TD, bool FAST>
cudaError_t launch_shape(const WnParams& p, int bt, cudaStream_t stream, WnLaunchInfo* info)
{
    if (p.R == 32 && p.S == 128) return launch_bt<TD, 32, 128, FAST>(p, bt, stream, info);
    if (p.R == 64 && p.S == 128) return launch_bt<TD, 64, 128, FAST>(p, bt, stream, info);
    if (p.R == 64 && p.S == 256) return launch_bt<TD, 64, 256, FAST>(p, bt, stream, info);
    if (p.R == 128 && p.S == 256) return launch_bt<TD, 128, 256, FAST>(p, bt, stream, info);
    return cudaErrorInvalidValue;
}

}  // namespace

bool wn_stream_supported(int R, int S, int A, bool)
{
    const bool shape = (R == 32 && S == 128) || (R == 64 && S == 128) || (R == 64 && S == 256) || (R == 128 && S == 256);
    return shape && A % 32 == 0 && A >= 32 && A <= 4096;
}

// Batch tile per CTA: every CTA re-reads all weights from L2 each sample, so L2 traffic per step is
// (B / BT) * weight_bytes; keep that under ~128 MB/step while using as many SMs as possible.
static int pick_bt(const WnParams& p, bool fp16)
{
    if (const char* env = getenv("NVWN_STREAM_BT")) {
        const int v = atoi(env);
        if ((v == 1 || v == 2 || v == 4) && p.B % v == 0) return v;
    }
    const double wbytes = (fp16 ? 2.0 : 4.0) * ((double)p.L * (5.0 * p.R * p.R + (double)p.S * p.R) + (double)p.A * p.S + (double)p.A * p.A);
    int bt = 1;
    while (bt < 4 && p.B % (bt * 2) == 0 && ((double)(p.B / bt) * wbytes > 128e6 || p.B / bt > 296)) bt *= 2;
    return bt;
}

// contract: 0 = fp32 bit-exact (CPU model's operation order), 1 = fp16 storage, 2 = fp32 in the reference GPU kernels' arithmetic
cudaError_t wn_launch_stream(const WnParams& p, int contract, cudaStream_t stream, WnLaunchInfo* info)
{
    const bool fp16 = contract == 1;
    if (!wn_stream_supported(p.R, p.S, p.A, fp16)) return cudaErrorInvalidValue;
    const int bt = pick_bt(p, fp16);
    if (info) info->kernel = 16;
    if (fp16) return launch_shape<__half, false>(p, bt, stream, info);
    return contract == 2 ? launch_shape<float, true>(p, bt, stream, info) : launch_shape<float, false>(p, bt, stream, info);
}
