// wn_lat_kernel.cu -- latency-mode fp16 kernel of the WaveNet inference loop (sm_100a).
//
// The autoregressive loop is a chain of ~45 tiny dependent GEMMs per sample (M = utterances, N <= 256, K <= 256).  On such a
// chain the tcgen05 round trip (MMA -> commit -> mbarrier -> tcgen05.ld, ~500 cycles) is the cost, not the tensor pipe
// (wn_tc_kernel.cu: 2.4 k cycles per layer).  This kernel keeps the whole chain in REGISTERS: warp-level mma.sync
// (m16n8k16, fp16 x fp16 -> fp32) with the utterances as the M dimension, so that the accumulator fragment of one GEMM is
// -- after the row-local epilogue -- exactly the A fragment of the next one; the only exchange between the eight compute
// warps is one 2 KB shared-memory tile + one named barrier per GEMM stage.
//
//   one persistent CTA per tile of 16 utterances (B = 64 -> 4 SMs), 8 compute warps + 1 producer warp:
//   compute warp w  owns output channels [8w, 8w+8) (+R for the sigmoid half) of every layer GEMM, [32w, 32w+32) of the skip
//                   sum / Zs / Za; residual stream (fp32) and skip sum (fp32) never leave its registers.
//                   per layer:  a = Wcur.x + Wprev.x[t-d] + (Bh + Lh)  ->  h = tanh * sigmoid  -> [h tile, barrier]
//                               x' = Wres.h + Bres + x -> [x tile, history ring, barrier];  skip += Wskip.h
//                   per sample: relu(skip) -> Zs -> Za -> softmax + categorical sample (warp-local, two utterances per warp)
//                               -> embedding gather from the shared-memory resident table.
//   producer warp   streams the weight image (pre-arranged in mma B-fragment order, so that every weight load of a warp is one
//                   conflict-free 512-byte LDS.128) from L2 through a shared-memory ring with bulk TMA + mbarriers: two pieces
//                   per layer ([Wcur_l | Wprev_l+1] 32 KB, [Wres_l | Wskip_l] 40 KB), two slots per piece type, every slot
//                   refilled as soon as its occupant is consumed -- each piece is in flight two layers before its use.
//   Lh (the only HBM stream), biases and the dilated history x[t-d] are prefetched into registers one / two layers ahead.
//
// wn_lat2_kernel (second half of this file, the default up to ~720 utterances) spreads the same data flow over a cluster of three
// CTAs per tile -- chain / tail / prep -- that hand tiles over through distributed shared memory; see the comment there.
//
// Replaces nv_wavenet_{singleblock,dualblock,persistent}.cuh + matrix_math.cuh + softmax.cuh of the reference for
// T_data = half while the batch is small enough to be latency-bound.  Numerical contract: oracle/wavenet_oracle.c
// WNO_PREC_FP16 (GEMM inputs fp16, fp32 accumulation, fp32 residual stream / skip sum / softmax), gate evaluated with
// tanh.approx.f16x2; no weight folding.
#include "wn_common.h"
#include "wn_math.cuh"
#include "wn_sm100.cuh"

#include <stdlib.h>

namespace {

using namespace sm100;

constexpr int R = 64, A = 256;
constexpr int NCW = 8;                      // compute warps
constexpr int NCT = NCW * 32;
constexpr int NT = NCT + 32;                // + producer warp
constexpr int TU = 16;                      // utterances per tile = M of mma.m16n8k16
constexpr int LROW = 264;                   // padded row (floats) of the transposed-logits buffer
constexpr int EROW = 33;                    // padded row (32-bit words) of the shared-memory embedding table
constexpr int MAXL = 64;

template <int S>
struct Cfg {
    // one layer block of the weight image = two ring pieces, in consumption order:
    //   P1 = [ Wcur_l | Wprev_{(l+1) mod L} ]  (32 KB)      P2 = [ Wres_l | Wskip_l ]  (8 KB + S x 128 B)
    static constexpr int W_CUR = 0, W_PREV = 16384, W_RES = 32768, W_SKIP = 40960;
    static constexpr int P1_BYTES = 32768, P2_BYTES = 8192 + S * 128;
    // output GEMMs: 4 + 4 ring pieces per sample, each all 32 n-tiles x OJP k-step pairs
    static constexpr int NQ_ZS = 4, NQ_ZA = 4;
    static constexpr int OJP_ZS = S / 128, OJP_ZA = A / 128;         // k-step pairs per piece
    static constexpr int ZS_PIECE = 32 * OJP_ZS * 512, ZA_PIECE = 32 * OJP_ZA * 512;
    static constexpr int OPIECE = ZA_PIECE > ZS_PIECE ? ZA_PIECE : ZS_PIECE;
    static constexpr int NSK = S / 64;                               // skip n-tiles per warp
    // ring: two slots per piece type; output pieces alternate between the two types
    static constexpr int SLOT1 = P1_BYTES, SLOT2 = P2_BYTES > OPIECE ? P2_BYTES : OPIECE;
    // shared memory map
    static constexpr uint32_t O_RING1 = 0;                           // 2 x SLOT1
    static constexpr uint32_t O_RING2 = 2 * SLOT1;                   // 2 x SLOT2
    static constexpr uint32_t O_EMB = O_RING2 + 2 * SLOT2;
    static constexpr uint32_t O_BOUT = O_EMB + A * EROW * 4;         // fp32: Bskip total [S], Bzs [A], Bza [A]
    static constexpr uint32_t O_EPBUF = O_BOUT + (S + 2 * A) * 4;           // two [16 rows][33 words] buffers (sample parity)
    static constexpr uint32_t O_PST = O_EPBUF + 2 * TU * EROW * 4;          // 3 x 2 KB: staged history tiles x[t-d] (A-fragment order)
    static constexpr uint32_t O_OB0 = O_PST + 3 * 2048;
    static constexpr uint32_t O_OB1 = O_OB0 + (S / 16) * 512;
    static constexpr uint32_t O_LBUF = O_OB1 + (A / 16) * 512;              // transposed logits; its first 4 KB double as ...
    static constexpr uint32_t O_XBUF = O_LBUF, O_HBUF = O_LBUF + 2048;      // ... the x and h exchange tiles (dead while the logits live)
    static constexpr uint32_t O_DIL = O_LBUF + TU * LROW * 4;
    static constexpr uint32_t O_YS = O_DIL + MAXL * 4;
    static constexpr uint32_t O_BAR = O_YS + 2 * TU * 4;
    static constexpr uint32_t SMEM = O_BAR + 16 * 8;
};

struct LatImage {
    size_t layer_bytes, off_zs, off_za, off_bias, total;
    size_t b_layer, b_skpre, b_bzs, b_bza;      // float offsets inside the bias block
};
__host__ __device__ inline LatImage lat_image(int S, int L)
{
    LatImage im;
    im.layer_bytes = 40960 + (size_t)S * 128;
    im.off_zs = (size_t)L * im.layer_bytes;
    im.off_za = im.off_zs + (size_t)A * S * 2;
    im.off_bias = im.off_za + (size_t)A * A * 2;
    im.b_layer = 0;                             // [L][8 warps][4 t][8]: Bh tanh pair, Bh sigmoid pair, Bres pair, 0, 0
    im.b_skpre = (size_t)L * 256;               // [L][S] running sum of the skip biases
    im.b_bzs = im.b_skpre + (size_t)L * S;
    im.b_bza = im.b_bzs + A;
    im.total = im.off_bias + (im.b_bza + A) * sizeof(float);
    return im;
}

// ------------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ void hmma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b)
{
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void load_a(uint32_t (&a)[4], uint32_t addr)
{
    const uint4 v = lds128(addr);
    a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
}
// predicated load into an existing register quad: no select on the loaded value, so nothing waits for the load here
__device__ __forceinline__ void ldg_nc_v4_if(uint4& d, const void* p, bool pred)
{
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
                 : "+r"(d.x), "+r"(d.y), "+r"(d.z), "+r"(d.w) : "l"(p), "r"((uint32_t)pred) : "memory");
}
__device__ __forceinline__ void stg_v2(void* p, uint32_t a, uint32_t b) { asm volatile("st.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory"); }
__device__ __forceinline__ void bar_compute() { asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory"); }
__device__ __forceinline__ uint32_t pack_h2(float a, float b)
{
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t v) { return __half22float2(*reinterpret_cast<__half2*>(&v)); }
__device__ __forceinline__ uint32_t u32(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 h2(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }

__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory"); }
// the mbarrier receives one arrival once every cp.async this thread has issued so far has landed
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) { asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_pending() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// mbarrier by shared-memory address
__device__ __forceinline__ void mbar_init_a(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) { asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_a(uint32_t bar, uint32_t bytes) { asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ bool mbar_try_a(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// a look that never suspends the thread (try_wait parks it until a time limit when the phase is still running)
__device__ __forceinline__ bool mbar_probe_a(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// three looks issued back to back: their ~90-cycle latencies overlap
__device__ __forceinline__ void mbar_try3_a(uint32_t b1, uint32_t p1, uint32_t b2, uint32_t p2, uint32_t b3, uint32_t p3, bool& o1, bool& o2, bool& o3)
{
    uint32_t r1, r2, r3;
    asm volatile("{\n\t.reg .pred q1, q2, q3;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 q1, [%3], %4;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 q2, [%5], %6;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 q3, [%7], %8;\n\t"
                 "selp.u32 %0, 1, 0, q1;\n\tselp.u32 %1, 1, 0, q2;\n\tselp.u32 %2, 1, 0, q3;\n\t}"
                 : "=r"(r1), "=r"(r2), "=r"(r3) : "r"(b1), "r"(p1), "r"(b2), "r"(p2), "r"(b3), "r"(p3) : "memory");
    o1 = r1 != 0; o2 = r2 != 0; o3 = r3 != 0;
}
static __device__ __noinline__ void lat_timeout(uint32_t bar, uint32_t parity)
{
    printf("wn_lat: mbarrier wait timed out: block %d thread %d barrier@0x%x parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
    __trap();
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity)
{
    uint32_t spins = 0;
    while (!mbar_try_a(bar, parity))
        if (++spins > (1u << 24)) lat_timeout(bar, parity);
}
__device__ __forceinline__ void tma_load_a(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// ------------------------------------------------------------------------------------------------ conditioning layout
// fp16, [N][L][tiles][8 warps][32 lanes][16 B]: the uint4 of thread (w, lane = 4 g + t) holds, as half2 pairs of channels
// (c, c+1), c = 8 w + 2 t:  .x = (row g, tanh c) .y = (row g+8, tanh c) .z = (row g, sigmoid R+c) .w = (row g+8, sigmoid R+c)
// i.e. exactly the accumulator fragment the thread adds it to.  Rows past the batch are zero.
__global__ void lat_cond_kernel(unsigned char* __restrict__ dst, const float* __restrict__ src, int first_sample, int nsamples, int L, int B, int ntiles)
{
    const size_t total = (size_t)nsamples * L * ntiles * 256;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int th = (int)(i & 255), w = th >> 5, lane = th & 31, g = lane >> 2, t = lane & 3;
        const size_t slt = i >> 8;                       // (s * L + l) * ntiles + tile
        const int tile = (int)(slt % ntiles);
        const size_t sl = slt / ntiles;                  // s * L + l
        const int c = 8 * w + 2 * t;
        uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
        for (int hi = 0; hi < 2; hi++) {
            const int b = tile * TU + g + 8 * hi;
            if (b < B) {
                const float* row = src + (sl * B + b) * 128;
                const float2 ft = *reinterpret_cast<const float2*>(row + c), fs = *reinterpret_cast<const float2*>(row + 64 + c);
                __half2 a = __floats2half2_rn(ft.x, ft.y), s = __floats2half2_rn(fs.x, fs.y);
                o[hi] = *reinterpret_cast<uint32_t*>(&a);
                o[2 + hi] = *reinterpret_cast<uint32_t*>(&s);
            }
        }
        const size_t off = (((size_t)first_sample * L * ntiles) + slt) * 4096 + (size_t)th * 16;
        *reinterpret_cast<uint4*>(dst + off) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// inverse of lat_cond_kernel (debug / tests): conditioning store -> fp32 [n][L][B][2R]
__global__ void lat_cond_readback_kernel(float* __restrict__ dst, const unsigned char* __restrict__ src, int first_sample, int nsamples, int L, int B, int ntiles)
{
    const size_t total = (size_t)nsamples * L * B * 64;            // one thread per channel pair
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c2 = (int)(i & 63);
        const size_t row = i >> 6;                                  // (s * L + l) * B + b
        const int b = (int)(row % B);
        const size_t sl = row / B;
        const int tile = b / TU, r = b % TU, g = r & 7, hi = r >> 3;
        const int sig = c2 >= 32, cc = (c2 & 31) * 2, w = cc >> 3, t = (cc & 7) >> 1;
        const size_t off = (((size_t)first_sample * L + sl) * ntiles + tile) * 4096 + (size_t)(w * 32 + g * 4 + t) * 16 + (size_t)(2 * sig + hi) * 4;
        const __half2 v = *reinterpret_cast<const __half2*>(src + off);
        dst[row * 128 + sig * 64 + cc] = __low2float(v);
        dst[row * 128 + sig * 64 + cc + 1] = __high2float(v);
    }
}

// ------------------------------------------------------------------------------------------------ pack
// blob (fp16, column-major M x K matrices as uploaded) -> weight image in mma.m16n8k16 B-fragment order.
// Element (n-tile nt, k-step pair jp, lane = 4 g + t) of a matrix W[M][K] is the uint4
//   { W[8nt+g][32jp+2t .. +1], W[8nt+g][32jp+8+2t ..], W[8nt+g][32jp+16+2t ..], W[8nt+g][32jp+24+2t ..] }
// = (b0, b1) of k-step 2jp and (b0, b1) of k-step 2jp+1.
__device__ __forceinline__ void frag_pos(int row, int k, int njp, size_t& byte_off)
{
    const int nt = row >> 3, g = row & 7, jp = k >> 5, kk = k & 31, comp = kk >> 3, t = (kk & 7) >> 1, e = kk & 1;
    byte_off = ((size_t)(nt * njp + jp) * 32 + (g * 4 + t)) * 16 + comp * 4 + e * 2;
}
__global__ void lat_pack_kernel(WnParams p, unsigned char* __restrict__ img, LatImage im)
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
    auto put = [&](size_t base, int row, int k, int njp, __half v) {
        size_t o;
        frag_pos(row, k, njp, o);
        *reinterpret_cast<__half*>(img + base + o) = v;
    };
    for (size_t i = g0; i < (size_t)L * 128 * 64; i += gstride) {
        const int l = (int)(i / (128 * 64)), c = (int)(i % (128 * 64)) / 64, k = (int)(i % 64);
        const size_t lb = (size_t)l * im.layer_bytes;
        put(lb, c, k, 2, Wcur[(size_t)l * 128 * 64 + c + (size_t)k * 128]);
        put((size_t)((l + L - 1) % L) * im.layer_bytes + 16384, c, k, 2, Wprev[(size_t)l * 128 * 64 + c + (size_t)k * 128]);   // rides with the layer before it
        if (c < 64) put(lb + 32768, c, k, 2, Wres[(size_t)l * 64 * 64 + c + (size_t)k * 64]);
    }
    for (size_t i = g0; i < (size_t)L * S * 64; i += gstride) {
        const int l = (int)(i / ((size_t)S * 64)), s = (int)((i / 64) % S), k = (int)(i % 64);
        put((size_t)l * im.layer_bytes + 40960, s, k, 2, Wskip[(size_t)l * S * 64 + s + (size_t)k * S]);
    }
    // output matrices: ring piece q holds k-step pairs [q OJP, (q+1) OJP) of all 32 n-tiles
    {
        const int ojp = S / 128;
        const size_t piece = (size_t)32 * ojp * 512;
        for (size_t i = g0; i < (size_t)A * S; i += gstride) {
            const int a = (int)(i / S), s = (int)(i % S);
            const int jp = s >> 5, q = jp / ojp;
            put(im.off_zs + (size_t)q * piece, a, (s & 31) + 32 * (jp % ojp), ojp, Wzs[a + (size_t)s * A]);
        }
    }
    {
        const int ojp = A / 128;
        const size_t piece = (size_t)32 * ojp * 512;
        for (size_t i = g0; i < (size_t)A * A; i += gstride) {
            const int a = (int)(i / A), z = (int)(i % A);
            const int jp = z >> 5, q = jp / ojp;
            put(im.off_za + (size_t)q * piece, a, (z & 31) + 32 * (jp % ojp), ojp, Wza[a + (size_t)z * A]);
        }
    }
    float* bias = reinterpret_cast<float*>(img + im.off_bias);
    const __half* Bh = static_cast<const __half*>(p.Bh);
    const __half* Bres = static_cast<const __half*>(p.Bres);
    const __half* Bskip = static_cast<const __half*>(p.Bskip);
    for (size_t i = g0; i < (size_t)L * 256; i += gstride) {
        const int l = (int)(i / 256), w = (int)(i % 256) / 32, t = (int)(i % 32) / 8, e = (int)(i % 8);
        const int c = 8 * w + 2 * t + (e & 1);
        float v = 0.f;
        if (e < 2) v = __half2float(Bh[(size_t)l * 128 + c]);
        else if (e < 4) v = __half2float(Bh[(size_t)l * 128 + 64 + c]);
        else if (e < 6) v = __half2float(Bres[(size_t)l * 64 + c]);
        bias[im.b_layer + i] = v;
    }
    for (size_t s = g0; s < (size_t)S; s += gstride) {
        float acc = 0.f;
        for (int l = 0; l < L; l++) { acc += __half2float(Bskip[(size_t)l * S + s]); bias[im.b_skpre + (size_t)l * S + s] = acc; }
    }
    for (size_t i = g0; i < (size_t)A; i += gstride) {
        bias[im.b_bzs + i] = __half2float(static_cast<const __half*>(p.Bzs)[i]);
        bias[im.b_bza + i] = __half2float(static_cast<const __half*>(p.Bza)[i]);
    }
}

// ------------------------------------------------------------------------------------------------ the kernel
struct StepIt { int t, l, slot; };       // coordinates of a layer step: sample, layer, history-ring slot of that sample

// DUMP: write the last-sample activations (the host runs the final sample of a dumping launch with this variant).
// TRC:  record the clock64 timeline (debug; tools/lat_trace.py).
template <int S, bool DUMP, bool TRC>
__global__ void __launch_bounds__(NT, 1) wn_lat_kernel(const WnParams p, const unsigned char* __restrict__ img, const int ntiles_alloc)
{
    using C = Cfg<S>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t sm = smem_u32(smem_raw);
    const int L = p.L, B = p.B;
    const LatImage im = lat_image(S, L);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile = blockIdx.x;
    const int slots = p.maxDil + 1;
    const int t_begin = p.init_sample, t_end = p.init_sample + p.count;
    const float* gbias = reinterpret_cast<const float*>(img + im.off_bias);

    // mbarriers of the weight ring: piece n lives in slot (n >> 1) & 1 of slot type n & 1; one full / empty pair per slot
    const uint32_t s_full = sm + C::O_BAR, s_empty = s_full + 32, s_pfull = s_full + 64;       // [4], [4], [3]
    int* dil = reinterpret_cast<int*>(smem_raw + C::O_DIL);
    int* ys = reinterpret_cast<int*>(smem_raw + C::O_YS);      // [TU] current index, [TU] previous index
    float* s_bout = reinterpret_cast<float*>(smem_raw + C::O_BOUT);
    constexpr int NQ = C::NQ_ZS + C::NQ_ZA;
    static_assert(NQ == 8, "the ring bookkeeping assumes 8 output pieces per sample");

    // debug timeline: role 0 = compute thread 0, role 2 = producer; words (tag << 48 | clock)
    unsigned long long* trc = (TRC && p.trace && blockIdx.x == 0) ? p.trace : nullptr;
    int trn = 0;
    const int tr_t = p.trace_t & 0xFFFF;
#define TRACE(role, tag) do { if (TRC && trc && t == tr_t && trn < 1023) trc[(role) * 1024 + trn++] = ((unsigned long long)(tag) << 48) | (clock64() & 0xFFFFFFFFFFFFull); } while (0)

    if (tid == 0) {
        for (int i = 0; i < 4; i++) { mbar_init_a(s_full + 8 * i, 1); mbar_init_a(s_empty + 8 * i, NCW); }
        for (int i = 0; i < 3; i++) mbar_init_a(s_pfull + 8 * i, 128);
        fence_mbar_init();
        int d = 1;                                     // dilation of layer l (nv_wavenet.cuh:99-111): 1,2,4..maxDil,1,2,...
        for (int l = 0; l < L; l++) { dil[l] = d; d <<= 1; if (d > p.maxDil) d = 1; }
    }
    {   // current-index embedding table -> shared memory (rows padded to 33 words: gathers of different rows fall into
        // different banks); output-layer biases; feedback state
        const uint32_t* ec = static_cast<const uint32_t*>(p.embCur);
        for (int i = tid; i < A * 32; i += NT) sts32(sm + C::O_EMB + ((i >> 5) * EROW + (i & 31)) * 4, ec[i]);
        for (int i = tid; i < S; i += NT) s_bout[i] = gbias[im.b_skpre + (size_t)(L - 1) * S + i];
        for (int i = tid; i < A; i += NT) { s_bout[S + i] = gbias[im.b_bzs + i]; s_bout[S + A + i] = gbias[im.b_bza + i]; }
        if (tid < TU) {
            const int b = tile * TU + tid;
            ys[tid] = b < B ? p.yCur[b] : 128;
            ys[TU + tid] = b < B ? p.yPrev[b] : 128;
        }
    }
    __syncthreads();

    if (warp == NCW) {
        // =============================================================== TMA producer (one lane): the pieces in consumption order,
        // each refilled as soon as ITS previous occupant has been consumed (two layers of lead for every piece)
        if (lane == 0) {
            uint32_t pc = 0;
            auto put = [&](const unsigned char* src, uint32_t bytes) {
                const uint32_t idx = (pc >> 1) & 1, bo = ((pc & 1) * 2 + idx) * 8;
                const uint32_t dst = (pc & 1) ? sm + C::O_RING2 + idx * C::SLOT2 : sm + C::O_RING1 + idx * C::SLOT1;
                mbar_wait_a(s_empty + bo, ((pc >> 2) & 1) ^ 1);
                mbar_expect_a(s_full + bo, bytes);
                tma_load_a(dst, src, bytes, s_full + bo);
                pc++;
            };
            for (int t = t_begin; t < t_end; t++) {
                for (int l = 0; l < L; l++) {
                    const unsigned char* src = img + (size_t)l * im.layer_bytes;
                    put(src, C::P1_BYTES);
                    put(src + C::P1_BYTES, C::P2_BYTES);
                    TRACE(2, 100 + l);
                }
                for (int q = 0; q < NQ; q++) {
                    put(q < C::NQ_ZS ? img + im.off_zs + (size_t)q * C::ZS_PIECE : img + im.off_za + (size_t)(q - C::NQ_ZS) * C::ZA_PIECE,
                        q < C::NQ_ZS ? C::ZS_PIECE : C::ZA_PIECE);
                    TRACE(2, 200 + q);
                }
            }
        }
    } else {
        // =============================================================== compute warps
        const int w = warp, g = lane >> 2, t4 = lane & 3;
        const int b0 = tile * TU + g, b1 = b0 + 8;
        const bool v0 = b0 < B, v1 = b1 < B;
        const uint32_t cstride = (uint32_t)ntiles_alloc * 4096u, rstride = (uint32_t)ntiles_alloc * 2048u;
        const unsigned char* gcond = static_cast<const unsigned char*>(p.Lh) + (size_t)tile * 4096 + (size_t)(w * 32 + lane) * 16;
        unsigned char* gring = static_cast<unsigned char*>(p.ring) + (size_t)tile * 2048 + (size_t)lane * 16;
        const float* gbl = gbias + im.b_layer + (size_t)(w * 4 + t4) * 8;
        const int jw = w >> 1, hw = w & 1;             // this warp's 8 channels = k-step jw, half hw of an activation tile
        const uint32_t lane16 = (uint32_t)lane * 16;
        const uint32_t xchg = (uint32_t)(jw * 512 + hw * 8) + lane16;
        const int cw = 8 * w + 2 * t4;                 // first of the thread's two channels inside the warp's slice
        // this thread's B-fragment offsets inside the ring pieces
        const uint32_t o_t0 = (uint32_t)(w * 2) * 512 + lane16, o_g0 = (uint32_t)((8 + w) * 2) * 512 + lane16;   // + 512 for the second k-step pair
        const uint32_t o_res = (uint32_t)(w * 2) * 512 + lane16, o_skip = 8192u + (uint32_t)(w * C::NSK * 2) * 512 + lane16;
        const uint32_t o_out = (uint32_t)(4 * w) * 512;                                                         // output pieces: x OJP, + lane16

        auto advance = [&](StepIt& it) { if (++it.l == L) { it.l = 0; it.t++; if (++it.slot == slots) it.slot = 0; } };
        auto release = [&](uint32_t bar) { __syncwarp(); if (lane == 0) mbar_arrive_a(bar); };
        // Every mbarrier wait costs ~90 cycles even when the phase completed long ago (TRYWAIT latency).  The barriers of the coming
        // step are therefore looked at once, at the end of the running step (measured: 40.1 kHz at C3 B=64 against 38.4 kHz with
        // plain waits at the point of use, and 35.9 kHz with blocking waits moved behind the preceding HMMA batches).
        auto probe = [&](uint32_t bar, uint32_t parity) -> bool { return mbar_try_a(bar, parity); };
        auto ensure = [&](bool ok, uint32_t bar, uint32_t parity) { if (!ok) mbar_wait_a(bar, parity); };

        // dilated history x_l[t - d] (zero before the start of the utterance, nv_wavenet.cuh:106) of the step `itp`: staged three
        // steps ahead into a 3-slot shared-memory ring by warps 0-3 (128 threads x 16 B, cp.async; completion on an mbarrier)
        StepIt itp{t_begin, 0, t_begin % slots};
        uint32_t pcnt = 0;                             // tiles staged so far (slot = pcnt % 3)
        auto stage_history = [&]() {
            if (w < 4) {
                const uint32_t slot3 = pcnt % 3;
                const int d = dil[itp.l];
                const uint32_t dst = sm + C::O_PST + slot3 * 2048 + (uint32_t)(w * 32 + lane) * 16;
                if (itp.t >= t_end || itp.t < d) {
                    sts128(dst, make_uint4(0, 0, 0, 0));
                    mbar_arrive_a(s_pfull + 8 * slot3);
                } else {
                    int sl = itp.slot - d; if (sl < 0) sl += slots;
                    cp_async16(dst, gring - lane16 + (size_t)(sl * L + itp.l) * rstride + (size_t)(w * 32 + lane) * 16);
                    cp_async_arrive_noinc(s_pfull + 8 * slot3);
                }
            }
            pcnt++;
            advance(itp);
        };

        uint32_t xa[4][4];
        uint4 cbA = make_uint4(0, 0, 0, 0), cbB = make_uint4(0, 0, 0, 0);
        float accp[2][4];                              // pre-activation of the coming step: Wprev.x[t-d] + Bh + Lh
        float2 brn;                                    // Bres pair of the coming step
        float4 bh_next; float2 br_next;                // Bh / Bres pairs of the step after (prefetched a layer ahead)
        float xres[4] = {0.f, 0.f, 0.f, 0.f};
        float sk[C::NSK][4];
#pragma unroll
        for (int i = 0; i < C::NSK; i++) sk[i][0] = sk[i][1] = sk[i][2] = sk[i][3] = 0.f;
        const unsigned char* cptr = gcond + (size_t)t_begin * L * cstride;      // conditioning of step it3 (steps are consecutive in memory)

        // accp <- (Bh + Lh) + Wprev . x[t-d] for the coming step `it1` (its staged history tile is number `pn`, its conditioning
        // sits in cbA / cbB by parity); Wprev rides in the SAME ring piece as the current layer's Wcur (`p1`; the very first
        // one comes from global memory).  Then the conditioning of step it3 is fetched.  Independent of the current layer's data.
        StepIt it1{0, 0, 0}, it3{0, 0, 0};
        uint32_t pn = 0, kp = 0;                       // kp = parity of the running step
        auto prep = [&](const uint32_t p1, const bool from_global, const bool pf_ok) {
            brn = br_next;
            const uint4 cb = kp ? cbA : cbB;           // step k consumes the buffer of parity (k + 1) & 1 ...
            {
                const float2 c0 = unpack_h2(cb.x), c1 = unpack_h2(cb.y), c2 = unpack_h2(cb.z), c3 = unpack_h2(cb.w);
                accp[0][0] = bh_next.x + c0.x; accp[0][1] = bh_next.y + c0.y; accp[0][2] = bh_next.x + c1.x; accp[0][3] = bh_next.y + c1.y;
                accp[1][0] = bh_next.z + c2.x; accp[1][1] = bh_next.w + c2.y; accp[1][2] = bh_next.z + c3.x; accp[1][3] = bh_next.w + c3.y;
            }
            const uint32_t slot3 = pn % 3;
            if (it1.t < t_end) {
                uint4 bt0, bg0, bt1, bg1;
                if (from_global) {
                    const unsigned char* gp = img + (size_t)(L - 1) * im.layer_bytes + C::W_PREV;
                    bt0 = ldg_nc_v4(gp + o_t0); bg0 = ldg_nc_v4(gp + o_g0); bt1 = ldg_nc_v4(gp + o_t0 + 512); bg1 = ldg_nc_v4(gp + o_g0 + 512);
                } else {
                    bt0 = lds128(p1 + C::W_PREV + o_t0); bg0 = lds128(p1 + C::W_PREV + o_g0);
                    bt1 = lds128(p1 + C::W_PREV + o_t0 + 512); bg1 = lds128(p1 + C::W_PREV + o_g0 + 512);
                }
                ensure(pf_ok, s_pfull + 8 * slot3, (pn / 3) & 1);
                uint32_t pb[4][4];
#pragma unroll
                for (int j = 0; j < 4; j++) load_a(pb[j], sm + C::O_PST + slot3 * 2048 + j * 512 + lane16);
                float u0[4] = {0.f, 0.f, 0.f, 0.f}, u1[4] = {0.f, 0.f, 0.f, 0.f};         // second half of K: independent chains
                hmma(accp[0], pb[0], bt0.x, bt0.y); hmma(accp[1], pb[0], bg0.x, bg0.y); hmma(u0, pb[2], bt1.x, bt1.y); hmma(u1, pb[2], bg1.x, bg1.y);
                hmma(accp[0], pb[1], bt0.z, bt0.w); hmma(accp[1], pb[1], bg0.z, bg0.w); hmma(u0, pb[3], bt1.z, bt1.w); hmma(u1, pb[3], bg1.z, bg1.w);
#pragma unroll
                for (int i = 0; i < 4; i++) { accp[0][i] += u0[i]; accp[1][i] += u1[i]; }
            }
            pn++;
            {   // ... and refills it with the conditioning of step k + 3
                const unsigned char* src = cptr;
                cptr += cstride;
                const bool live = it3.t < t_end;       // past the end the stale value is never used (the prep of such a step is skipped)
                ldg_nc_v4_if(cbA, src, live && kp != 0);
                ldg_nc_v4_if(cbB, src, live && kp == 0);
            }
            advance(it1); advance(it3);
            bh_next = *reinterpret_cast<const float4*>(gbl + it1.l * 256);
            br_next = *reinterpret_cast<const float2*>(gbl + it1.l * 256 + 4);
        };

        // ---------------- prologue: previous-index rows of the first sample, prefetch pipeline
        {
            const uint32_t* ep = static_cast<const uint32_t*>(p.embPrev);
            sts32(sm + C::O_EPBUF + (g * EROW + 4 * w + t4) * 4, ep[ys[TU + g] * 32 + 4 * w + t4]);
            sts32(sm + C::O_EPBUF + ((g + 8) * EROW + 4 * w + t4) * 4, ep[ys[TU + g + 8] * 32 + 4 * w + t4]);
        }
        StepIt it0{t_begin, 0, t_begin % slots};
        stage_history(); stage_history(); stage_history();              // history tiles of steps 0, 1, 2
        {
            it1 = it0; it3 = it0;
            kp = 1;                                                     // the prologue plays "step -1": consumes cbA (step 0), refills it with step 2
            cbA = ldg_nc_v4(cptr); cptr += cstride;
            { StepIt i1 = it0; advance(i1); cbB = i1.t < t_end ? ldg_nc_v4(cptr) : make_uint4(0, 0, 0, 0); cptr += cstride; }
            advance(it3); advance(it3);
            bh_next = *reinterpret_cast<const float4*>(gbl); br_next = *reinterpret_cast<const float2*>(gbl + 4);
            prep(0, true, false);                                       // leaves it1 = step 1, it3 = step 3
            kp = 0;
        }
        bar_compute();

        // ring bookkeeping: a layer step uses slot `sb` of both piece types; the parity of its barriers is `fph`
        uint32_t sb = 0, fph = 0;

        bool ok_f1 = false, ok_f2 = false, ok_pf = false;          // what the look at the coming step's barriers returned
        // one layer step
        auto step = [&](const int t, const int l) {
            const uint32_t p1 = sm + C::O_RING1 + sb * C::SLOT1, p2 = sm + C::O_RING2 + sb * C::SLOT2;
            const uint32_t f1 = s_full + sb * 8, f2 = s_full + 16 + sb * 8, e1 = s_empty + sb * 8, e2 = s_empty + 16 + sb * 8;
            const float2 br = brn;
            // ---- a = Wcur.x + [Wprev.x[t-d] + Bh + Lh]   (nv_wavenet.cuh:131-157); the two halves of K as independent chains
            ensure(ok_f1, f1, fph);
            {
                const uint4 bt0 = lds128(p1 + o_t0), bg0 = lds128(p1 + o_g0), bt1 = lds128(p1 + o_t0 + 512), bg1 = lds128(p1 + o_g0 + 512);
                float u0[4] = {0.f, 0.f, 0.f, 0.f}, u1[4] = {0.f, 0.f, 0.f, 0.f};
                hmma(accp[0], xa[0], bt0.x, bt0.y); hmma(accp[1], xa[0], bg0.x, bg0.y); hmma(u0, xa[2], bt1.x, bt1.y); hmma(u1, xa[2], bg1.x, bg1.y);
                hmma(accp[0], xa[1], bt0.z, bt0.w); hmma(accp[1], xa[1], bg0.z, bg0.w); hmma(u0, xa[3], bt1.z, bt1.w); hmma(u1, xa[3], bg1.z, bg1.w);
#pragma unroll
                for (int i = 0; i < 4; i++) { accp[0][i] += u0[i]; accp[1][i] += u1[i]; }
            }
            // ---- h = tanh(a[:R]) * sigmoid(a[R:])   (packed fp16 MUFU; sigmoid(x) = 0.5 tanh(x/2) + 0.5)
            {
                const __half2 half = __floats2half2_rn(0.5f, 0.5f);
                const __half2 tg0 = wn::tanh_h2(h2(pack_h2(accp[0][0], accp[0][1]))), tg1 = wn::tanh_h2(h2(pack_h2(accp[0][2], accp[0][3])));
                const __half2 sg0 = __hfma2(wn::tanh_h2(h2(pack_h2(0.5f * accp[1][0], 0.5f * accp[1][1]))), half, half);
                const __half2 sg1 = __hfma2(wn::tanh_h2(h2(pack_h2(0.5f * accp[1][2], 0.5f * accp[1][3]))), half, half);
                sts64(sm + C::O_HBUF + xchg, u32(__hmul2(tg0, sg0)), u32(__hmul2(tg1, sg1)));
            }
            if (tid == 0) TRACE(0, 12);
            // ---- while the other warps finish their part of h: the dilated-history half of the next step's pre-activation
            // (after the last layer: layer 0 of the next sample); then this piece of the ring is free
            prep(p1, false, ok_pf);
            release(e1);
            bar_compute();
            uint32_t ha[4][4];
#pragma unroll
            for (int j = 0; j < 4; j++) load_a(ha[j], sm + C::O_HBUF + j * 512 + lane16);
            if (tid == 0) TRACE(0, 10);
            // ---- x' = Wres.h + Bres + x   (nv_wavenet.cuh:185-207); two half-K chains
            float ra[4] = {0.f, 0.f, 0.f, 0.f}, rb[4] = {0.f, 0.f, 0.f, 0.f};
            ensure(ok_f2, f2, fph);
            {
                const uint4 bw0 = lds128(p2 + o_res), bw1 = lds128(p2 + o_res + 512);
                hmma(ra, ha[0], bw0.x, bw0.y); hmma(rb, ha[2], bw1.x, bw1.y);
                hmma(ra, ha[1], bw0.z, bw0.w); hmma(rb, ha[3], bw1.z, bw1.w);
            }
            xres[0] = ((ra[0] + rb[0]) + br.x) + xres[0]; xres[1] = ((ra[1] + rb[1]) + br.y) + xres[1];
            xres[2] = ((ra[2] + rb[2]) + br.x) + xres[2]; xres[3] = ((ra[3] + rb[3]) + br.y) + xres[3];
            if (l + 1 < L) {
                const uint32_t x01 = pack_h2(xres[0], xres[1]), x23 = pack_h2(xres[2], xres[3]);
                sts64(sm + C::O_XBUF + xchg, x01, x23);
                stg_v2(gring + (size_t)(it0.slot * L + l + 1) * rstride + jw * 512 + hw * 8, x01, x23);
            }
            if (tid == 0) TRACE(0, 14);
            if (DUMP) {
                if (v0) { p.xtOut[((size_t)l * B + b0) * R + cw] = xres[0]; p.xtOut[((size_t)l * B + b0) * R + cw + 1] = xres[1]; }
                if (v1) { p.xtOut[((size_t)l * B + b1) * R + cw] = xres[2]; p.xtOut[((size_t)l * B + b1) * R + cw + 1] = xres[3]; }
            }
            // ---- while the other warps finish their part of x': skip += Wskip.h   (biases are added once, after the last layer)
#pragma unroll
            for (int jp = 0; jp < 2; jp++) {
                uint4 bw[C::NSK];
#pragma unroll
                for (int i = 0; i < C::NSK; i++) bw[i] = lds128(p2 + o_skip + (i * 2 + jp) * 512);
#pragma unroll
                for (int i = 0; i < C::NSK; i++) hmma(sk[i], ha[2 * jp], bw[i].x, bw[i].y);
#pragma unroll
                for (int i = 0; i < C::NSK; i++) hmma(sk[i], ha[2 * jp + 1], bw[i].z, bw[i].w);
            }
            release(e2);
            stage_history();                           // the history tile of three steps ahead
            {   // look at the coming step's barriers now; the answers are consumed a barrier later
                const uint32_t nsb = sb ^ 1, nph = fph ^ sb;
                mbar_try3_a(s_full + nsb * 8, nph, s_full + 16 + nsb * 8, nph, s_pfull + 8 * (pn % 3), (pn / 3) & 1, ok_f1, ok_f2, ok_pf);
            }
            if (tid == 0) TRACE(0, 15);
            if (DUMP) {
                const float* pre = gbias + im.b_skpre + (size_t)l * S;
#pragma unroll
                for (int i = 0; i < C::NSK; i++) {
                    const int c = 8 * (w * C::NSK + i) + 2 * t4;
                    float o0 = sk[i][0] + pre[c], o1 = sk[i][1] + pre[c + 1], o2 = sk[i][2] + pre[c], o3 = sk[i][3] + pre[c + 1];
                    if (l == L - 1) { o0 = fmaxf(o0, 0.f); o1 = fmaxf(o1, 0.f); o2 = fmaxf(o2, 0.f); o3 = fmaxf(o3, 0.f); }
                    if (v0) { p.skipOut[((size_t)l * B + b0) * S + c] = o0; p.skipOut[((size_t)l * B + b0) * S + c + 1] = o1; }
                    if (v1) { p.skipOut[((size_t)l * B + b1) * S + c] = o2; p.skipOut[((size_t)l * B + b1) * S + c + 1] = o3; }
                }
            }
            if (l + 1 < L) {
                bar_compute();
#pragma unroll
                for (int j = 0; j < 4; j++) load_a(xa[j], sm + C::O_XBUF + j * 512 + lane16);
            }
            if (tid == 0) TRACE(0, 11);
            fph ^= sb; sb ^= 1; kp ^= 1;               // slot alternates every step, barrier parity every second step
        };

        uint32_t epar = 0;                             // parity of the sample (epbuf buffer)
        for (int t = t_begin; t < t_end; t++) {
            // ---------------- embedding (reference.cpp:42-57): x0 = [tanh](embPrev[yPrev] + embCur[yCur]), this warp's 8 channels
            if (tid == 0) TRACE(0, 1);
            const float sel0 = (2 * w + 0 + tile * TU) < B ? p.sel[(size_t)t * B + tile * TU + 2 * w] : 0.5f;
            const float sel1 = (2 * w + 1 + tile * TU) < B ? p.sel[(size_t)t * B + tile * TU + 2 * w + 1] : 0.5f;
            {
                const int yc0 = ys[g], yc1 = ys[g + 8];
                const uint32_t eo = sm + C::O_EPBUF + epar * (TU * EROW * 4);
                const float2 a0 = unpack_h2(lds32(eo + (g * EROW + 4 * w + t4) * 4)), a1 = unpack_h2(lds32(eo + ((g + 8) * EROW + 4 * w + t4) * 4));
                const float2 c0 = unpack_h2(lds32(sm + C::O_EMB + (yc0 * EROW + 4 * w + t4) * 4)), c1 = unpack_h2(lds32(sm + C::O_EMB + (yc1 * EROW + 4 * w + t4) * 4));
                xres[0] = a0.x + c0.x; xres[1] = a0.y + c0.y; xres[2] = a1.x + c1.x; xres[3] = a1.y + c1.y;
                if (p.tanhEmbed) {
#pragma unroll
                    for (int i = 0; i < 4; i++) xres[i] = wn::tanhf_fast(xres[i]);
                }
                const uint32_t x01 = pack_h2(xres[0], xres[1]), x23 = pack_h2(xres[2], xres[3]);
                sts64(sm + C::O_XBUF + xchg, x01, x23);
                stg_v2(gring + (size_t)(it0.slot * L) * rstride + jw * 512 + hw * 8, x01, x23);
                // previous-index rows of the NEXT sample (= this sample's current index): global -> shared, asynchronously
                const unsigned char* ep = static_cast<const unsigned char*>(p.embPrev);
                const uint32_t en = sm + C::O_EPBUF + (epar ^ 1) * (TU * EROW * 4);
                cp_async4(en + (g * EROW + 4 * w + t4) * 4, ep + (size_t)yc0 * 128 + (4 * w + t4) * 4);
                cp_async4(en + ((g + 8) * EROW + 4 * w + t4) * 4, ep + (size_t)yc1 * 128 + (4 * w + t4) * 4);
                cp_async_commit();
            }
            bar_compute();
#pragma unroll
            for (int j = 0; j < 4; j++) load_a(xa[j], sm + C::O_XBUF + j * 512 + lane16);
            if (tid == 0) TRACE(0, 2);

            for (int l = 0; l < L; l++) step(t, l);
            ok_f1 = ok_f2 = false;                     // those looks were at slots the output pieces use first (same parity): stale

            // ---------------- relu(skip + bias) -> Zs -> Za   (reference.cpp:93-104)
#pragma unroll
            for (int i = 0; i < C::NSK; i++) {
                const int nt = w * C::NSK + i, c = 8 * nt + 2 * t4;
                const float b0f = s_bout[c], b1f = s_bout[c + 1];
                sts64(sm + C::O_OB0 + (nt >> 1) * 512 + lane16 + (nt & 1) * 8,
                      pack_h2(fmaxf(sk[i][0] + b0f, 0.f), fmaxf(sk[i][1] + b1f, 0.f)), pack_h2(fmaxf(sk[i][2] + b0f, 0.f), fmaxf(sk[i][3] + b1f, 0.f)));
                sk[i][0] = sk[i][1] = sk[i][2] = sk[i][3] = 0.f;
            }
            bar_compute();
            if (tid == 0) TRACE(0, 20);
            float zz[4][4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int c = 32 * w + 8 * i + 2 * t4;
                zz[i][0] = zz[i][2] = s_bout[S + c]; zz[i][1] = zz[i][3] = s_bout[S + c + 1];
            }
            // the 8 output pieces continue the ring sequence: piece q sits in slot type q & 1, slot sb ^ (q >> 1 & 1)
            auto out_gemm = [&](const int q, const int ojp, const uint32_t abuf, const int kp0) {
                const uint32_t idx = sb ^ ((q >> 1) & 1), bo = ((q & 1) * 2 + idx) * 8;
                const uint32_t st = ((q & 1) ? sm + C::O_RING2 + idx * C::SLOT2 : sm + C::O_RING1 + idx * C::SLOT1) + o_out * ojp + lane16;
                mbar_wait_a(s_full + bo, fph ^ (((sb + (q >> 1)) >> 1) & 1));
                for (int jp = 0; jp < ojp; jp++) {
                    uint32_t a0[4], a1[4];
                    load_a(a0, abuf + ((kp0 + jp) * 2) * 512 + lane16);
                    load_a(a1, abuf + ((kp0 + jp) * 2 + 1) * 512 + lane16);
                    uint4 bw[4];
#pragma unroll
                    for (int i = 0; i < 4; i++) bw[i] = lds128(st + (i * ojp + jp) * 512);
#pragma unroll
                    for (int i = 0; i < 4; i++) hmma(zz[i], a0, bw[i].x, bw[i].y);
#pragma unroll
                    for (int i = 0; i < 4; i++) hmma(zz[i], a1, bw[i].z, bw[i].w);
                }
                release(s_empty + bo);
            };
#pragma unroll
            for (int q = 0; q < C::NQ_ZS; q++) out_gemm(q, C::OJP_ZS, sm + C::O_OB0, q * C::OJP_ZS);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int nt = 4 * w + i, c = 8 * nt + 2 * t4;
                const float z0 = fmaxf(zz[i][0], 0.f), z1 = fmaxf(zz[i][1], 0.f), z2 = fmaxf(zz[i][2], 0.f), z3 = fmaxf(zz[i][3], 0.f);
                sts64(sm + C::O_OB1 + (nt >> 1) * 512 + lane16 + (nt & 1) * 8, pack_h2(z0, z1), pack_h2(z2, z3));
                if (DUMP) {
                    if (v0) { p.Zs[(size_t)b0 * A + c] = z0; p.Zs[(size_t)b0 * A + c + 1] = z1; }
                    if (v1) { p.Zs[(size_t)b1 * A + c] = z2; p.Zs[(size_t)b1 * A + c + 1] = z3; }
                }
                zz[i][0] = zz[i][2] = s_bout[S + A + c]; zz[i][1] = zz[i][3] = s_bout[S + A + c + 1];
            }
            bar_compute();
            if (tid == 0) TRACE(0, 21);
#pragma unroll
            for (int q = 0; q < C::NQ_ZA; q++) out_gemm(C::NQ_ZS + q, C::OJP_ZA, sm + C::O_OB1, q * C::OJP_ZA);
            // 8 pieces = 4 slot pairs later: same slot, same barrier parity as before the output phase
            // logits (fp32) -> transposed buffer: row = utterance, 256 contiguous classes
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int c = 32 * w + 8 * i + 2 * t4;
                sts64(sm + C::O_LBUF + (g * LROW + c) * 4, __float_as_uint(zz[i][0]), __float_as_uint(zz[i][1]));
                sts64(sm + C::O_LBUF + ((g + 8) * LROW + c) * 4, __float_as_uint(zz[i][2]), __float_as_uint(zz[i][3]));
                if (DUMP) {
                    if (v0) { p.Za[(size_t)b0 * A + c] = zz[i][0]; p.Za[(size_t)b0 * A + c + 1] = zz[i][1]; }
                    if (v1) { p.Za[(size_t)b1 * A + c] = zz[i][2]; p.Za[(size_t)b1 * A + c + 1] = zz[i][3]; }
                }
            }
            bar_compute();
            if (tid == 0) TRACE(0, 22);
            if (t + 1 < t_end) {                       // every output piece is consumed: the first pieces of the next sample
                ok_f1 = probe(s_full + sb * 8, fph);
                ok_f2 = probe(s_full + 16 + sb * 8, fph);
            }
            // ---------------- softmax + categorical sample (matrix.cpp:167-183, reference.cpp:106-121): warp w serves
            // utterances 2w and 2w+1; lane holds 8 consecutive classes of each
            {
                float e[2][8], m[2] = {-INFINITY, -INFINITY};              // the true row max (DESIGN.md §3)
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const uint4 u0 = lds128(sm + C::O_LBUF + ((2 * w + r) * LROW + 8 * lane) * 4), u1 = lds128(sm + C::O_LBUF + ((2 * w + r) * LROW + 8 * lane + 4) * 4);
                    e[r][0] = __uint_as_float(u0.x); e[r][1] = __uint_as_float(u0.y); e[r][2] = __uint_as_float(u0.z); e[r][3] = __uint_as_float(u0.w);
                    e[r][4] = __uint_as_float(u1.x); e[r][5] = __uint_as_float(u1.y); e[r][6] = __uint_as_float(u1.z); e[r][7] = __uint_as_float(u1.w);
#pragma unroll
                    for (int k = 0; k < 8; k++) m[r] = fmaxf(m[r], e[r][k]);
                }
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) {
                    m[0] = fmaxf(m[0], __shfl_xor_sync(0xffffffffu, m[0], o));
                    m[1] = fmaxf(m[1], __shfl_xor_sync(0xffffffffu, m[1], o));
                }
                float incl[2];
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const float ms = m[r] * 1.4426950408889634f;
                    float run = 0.f;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        const float ev = wn::exp2f_fast(fmaf(e[r][k], 1.4426950408889634f, -ms));
                        run += ev;
                        e[r][k] = run;                                     // inclusive running sum inside the lane
                    }
                    incl[r] = run;
                }
                const float tot_lane[2] = {incl[0], incl[1]};
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float a0 = __shfl_up_sync(0xffffffffu, incl[0], o), a1 = __shfl_up_sync(0xffffffffu, incl[1], o);
                    if (lane >= o) { incl[0] += a0; incl[1] += a1; }
                }
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const float total = __shfl_sync(0xffffffffu, incl[r], 31);
                    const float excl = incl[r] - tot_lane[r];
                    const float target = (r == 0 ? sel0 : sel1) * total;
                    int cntk = 0;
#pragma unroll
                    for (int k = 0; k < 8; k++) cntk += (target < excl + e[r][k]) ? 0 : 1;
                    const unsigned ball = __ballot_sync(0xffffffffu, target < incl[r]);
                    const int lf = ball ? __ffs(ball) - 1 : 31;
                    const int ck = __shfl_sync(0xffffffffu, cntk, lf);
                    const int y = ball ? 8 * lf + (ck < 7 ? ck : 7) : A - 1;
                    const int b = tile * TU + 2 * w + r;
                    if (DUMP && b < B) {
                        const float inv = 1.f / total;
                        float prevv = 0.f;
#pragma unroll
                        for (int k = 0; k < 8; k++) { p.P[(size_t)b * A + 8 * lane + k] = (e[r][k] - prevv) * inv; prevv = e[r][k]; }
                    }
                    if (lane == 0) {
                        int fbk = y;
                        if (b < B) {
                            p.yOut[(size_t)b * p.N + t] = y;
                            if (p.forced) fbk = p.forced[(size_t)b * p.N + t];
                        } else fbk = 128;
                        ys[TU + 2 * w + r] = ys[2 * w + r];
                        ys[2 * w + r] = fbk;
                    }
                }
            }
            cp_async_wait_all();                       // the next sample's previous-index rows have landed
            bar_compute();
            if (tid == 0) TRACE(0, 23);
            epar ^= 1;
            if (++it0.slot == slots) it0.slot = 0;
            it0.t++;
        }
        if (tid < TU && tile * TU + tid < B) { p.yCur[tile * TU + tid] = ys[tid]; p.yPrev[tile * TU + tid] = ys[TU + tid]; }
    }
#undef TRACE
}

// ================================================================================================ three-CTA cluster variant
// The single-CTA kernel above runs at ~83 % of its SM's shared-memory bandwidth (per layer step: 72 KB written by TMA, 72 KB of
// B fragments and 48 KB of A fragments read back; ncu: 0.57 LSU wavefronts per cycle + the TMA writes).  Here one 16-utterance tile
// is served by a CLUSTER OF THREE CTAs on three SMs, and only what depends on the previous sample stays on the first one:
//   rank 0 "chain": embedding, cur / res GEMMs, gate, history ring writes             ring pieces [Wcur_l | Wres_l] (24 KB)
//   rank 1 "tail":  skip GEMM of every step (off the chain), Zs, Za, softmax, sampling ring pieces Wskip_l and the output pieces
//   rank 2 "prep":  (Bh + Lh) + Wprev . x[t-d] of the steps to come, up to NAP ahead   ring pieces Wprev_l (16 KB)
// Distributed shared memory carries three flows, all as st.async with complete_tx on a transaction barrier that the receiver arms
// one phase ahead (data and signal travel together, no release fence on the sender), buffers handed back with relaxed remote arrives:
// h (2 KB per step, chain -> tail), the pre-activation before the current-sample GEMM (8 KB per step, prep -> chain), the 16 sampled
// indices (once per sample, tail -> chain).  Each CTA moves less than ~100 KB per step through its shared memory; a single CTA
// doing all of it moves ~190 KB per step and is bound by that.
constexpr int NTC = NCT + 32;

template <int S>
struct CfgC {
    using C = Cfg<S>;
    static constexpr uint32_t PIECE0 = 24576;                              // chain: [Wcur | Wres]
    static constexpr uint32_t SLOT1 = 32768;                               // tail: Wskip_l (S x 128 B) or an output piece
    static constexpr int NSLOT1 = 4;
    static constexpr int NAP = 4;                                          // pre-activation tiles in flight from the prep CTA to the chain CTA
    static constexpr int NPS = 8;                                          // staged history / conditioning tiles of the prep CTA
    // chain CTA
    static constexpr uint32_t C_RING = 0;                                  // 2 x PIECE0
    static constexpr uint32_t C_EMB = 2 * PIECE0;
    static constexpr uint32_t C_EPBUF = C_EMB + A * EROW * 4;
    static constexpr uint32_t C_XBUF = C_EPBUF + 2 * TU * EROW * 4;
    static constexpr uint32_t C_HBUF = C_XBUF + 2048;
    static constexpr uint32_t C_AP = C_HBUF + 2048;                        // NAP x 8 KB: (Bh + Lh) + Wprev . x[t-d] of the coming steps, written by the prep CTA
    static constexpr uint32_t C_BIAS = C_AP + NAP * 8192;                  // [L][8 warps][4][8] fp32: Bh / Bres pairs per thread (Bres is read here)
    static constexpr uint32_t C_END = C_BIAS + MAXL * 1024;
    // tail CTA
    static constexpr uint32_t T_RING = 0;                                  // NSLOT1 x SLOT1
    static constexpr uint32_t T_BOUT = NSLOT1 * SLOT1;
    static constexpr uint32_t T_HBUF = T_BOUT + (S + 2 * A) * 4;           // 2 x 2 KB, written by the chain CTA
    static constexpr uint32_t T_OB0 = T_HBUF + 2 * 2048;
    static constexpr uint32_t T_OB1 = T_OB0 + (S / 16) * 512;
    static constexpr uint32_t T_LBUF = T_OB1 + (A / 16) * 512;
    static constexpr uint32_t T_END = T_LBUF + TU * LROW * 4;
    // prep CTA
    static constexpr uint32_t P_RING = 0;                                  // 4 x 16 KB: Wprev_l
    static constexpr uint32_t P_PST = 4 * 16384;                           // NPS x 2 KB: staged history tiles x[t-d] (A-fragment order)
    static constexpr uint32_t P_COND = P_PST + NPS * 2048;                 // NPS x 4 KB: conditioning tiles, staged with the history tiles (cp.async)
    static constexpr uint32_t P_BIAS = P_COND + NPS * 4096;                // [L][8 warps][4][4] fp32: this thread's Bh
    static constexpr uint32_t P_DIL = P_BIAS + MAXL * 512;
    static constexpr uint32_t P_END = P_DIL + MAXL * 4;
    // common tail of the maps (same offsets in every CTA, so that remote addresses are computed with mapa on local ones)
    static constexpr uint32_t O_YS = (C_END > T_END ? (C_END > P_END ? C_END : P_END) : (T_END > P_END ? T_END : P_END));
    static constexpr uint32_t O_BAR = O_YS + 2 * TU * 4;
    static constexpr uint32_t SMEM = O_BAR + 32 * 8;
};
constexpr int NCL = 3;                       // CTAs per cluster

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// remote stores that complete bytes on a remote mbarrier (data and signal travel together: no release fence on the sender)
__device__ __forceinline__ void st_async_v2(uint32_t raddr, uint32_t a, uint32_t b, uint32_t rbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1,%2}, [%3];" ::"r"(raddr), "r"(a), "r"(b), "r"(rbar) : "memory");
}
__device__ __forceinline__ void st_async_v4(uint32_t raddr, float a, float b, float c, float d, uint32_t rbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1,%2,%3,%4}, [%5];"
                 ::"r"(raddr), "r"(__float_as_uint(a)), "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d)), "r"(rbar) : "memory");
}
__device__ __forceinline__ void st_async_u32(uint32_t raddr, uint32_t a, uint32_t rbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(raddr), "r"(a), "r"(rbar) : "memory");
}
// "this buffer is free again": no data behind it, so no release ordering is paid for
__device__ __forceinline__ void mbar_arrive_remote(uint32_t raddr) { asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory"); }
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int S, bool DUMP, bool TRC>
__global__ void __launch_bounds__(NTC, 1) wn_lat2_kernel(const WnParams p, const unsigned char* __restrict__ img, const int ntiles_alloc)
{
    // debug timeline (tools/lat_trace.py): role 0 = chain CTA thread 0, role 1 = tail CTA thread 0, of the first cluster
    unsigned long long* trc = (TRC && p.trace && blockIdx.x < 2) ? p.trace : nullptr;
    int trn = 0;
    const int tr_t = p.trace_t & 0xFFFF;
#define TRACE2(role, tag) do { if (TRC && trc && threadIdx.x == 0 && t == tr_t && trn < 1023) trc[(role) * 1024 + trn++] = ((unsigned long long)(tag) << 48) | (clock64() & 0xFFFFFFFFFFFFull); } while (0)
    using C = Cfg<S>;
    using M = CfgC<S>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t sm = smem_u32(smem_raw);
    const int L = p.L, B = p.B;
    const LatImage im = lat_image(S, L);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint32_t crank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const bool is_chain = crank == 0, is_tail = crank == 1;
    const int tile = blockIdx.x / NCL;
    const int slots = p.maxDil + 1;
    const int t_begin = p.init_sample, t_end = p.init_sample + p.count;
    const float* gbias = reinterpret_cast<const float*>(img + im.off_bias);
    constexpr int NQ = C::NQ_ZS + C::NQ_ZA;

    // barriers (same offsets in every CTA): ring full[4] / empty[4] (the chain uses two of each); pfull[NPS] (prep: staged history
    // tiles); hfull[2] (tail: h tiles, bytes from the chain); hfree[2], yfull, apfull[NAP] (chain: bytes from the tail / the prep CTA);
    // apfree[NAP] (prep: arrived by the chain's warps)
    const uint32_t s_full = sm + M::O_BAR, s_empty = s_full + 32, s_pfull = s_full + 64, s_hfull = s_full + 128, s_hfree = s_full + 144, s_yfull = s_full + 160;
    const uint32_t s_apfull = s_full + 168, s_apfree = s_full + 200;
    int* ys = reinterpret_cast<int*>(smem_raw + M::O_YS);

    if (tid == 0) {
        for (int i = 0; i < 4; i++) { mbar_init_a(s_full + 8 * i, 1); mbar_init_a(s_empty + 8 * i, NCW); }
        for (int i = 0; i < M::NPS; i++) mbar_init_a(s_pfull + 8 * i, 128);
        for (int i = 0; i < 2; i++) { mbar_init_a(s_hfull + 8 * i, 1); mbar_init_a(s_hfree + 8 * i, NCW); }
        for (int i = 0; i < M::NAP; i++) { mbar_init_a(s_apfull + 8 * i, 1); mbar_init_a(s_apfree + 8 * i, NCW); }
        mbar_init_a(s_yfull, 1);
        fence_mbar_init();
        // transaction barriers are armed by their owner one phase ahead: the tail expects 2 KB per h tile, the chain 128 B of indices
        // and 8 KB per pre-activation tile
        if (is_chain) { mbar_expect_a(s_yfull, 2 * TU * 4); for (int i = 0; i < M::NAP; i++) mbar_expect_a(s_apfull + 8 * i, 8192); }
        else if (is_tail) { mbar_expect_a(s_hfull, 2048); mbar_expect_a(s_hfull + 8, 2048); }
    }
    if (tid < TU) {
        const int b = tile * TU + tid;
        ys[tid] = b < B ? p.yCur[b] : 128;
        ys[TU + tid] = b < B ? p.yPrev[b] : 128;
    }
    if (is_chain) {
        const uint32_t* ec = static_cast<const uint32_t*>(p.embCur);
        for (int i = tid; i < A * 32; i += NTC) sts32(sm + M::C_EMB + ((i >> 5) * EROW + (i & 31)) * 4, ec[i]);
        for (int i = tid; i < L * 256; i += NTC) sts32(sm + M::C_BIAS + i * 4, __float_as_uint(gbias[im.b_layer + i]));
    } else if (is_tail) {
        float* s_bout = reinterpret_cast<float*>(smem_raw + M::T_BOUT);
        for (int i = tid; i < S; i += NTC) s_bout[i] = gbias[im.b_skpre + (size_t)(L - 1) * S + i];
        for (int i = tid; i < A; i += NTC) { s_bout[S + i] = gbias[im.b_bzs + i]; s_bout[S + A + i] = gbias[im.b_bza + i]; }
    } else {
        int* dil = reinterpret_cast<int*>(smem_raw + M::P_DIL);
        if (tid == 0) { int d = 1; for (int l = 0; l < L; l++) { dil[l] = d; d <<= 1; if (d > p.maxDil) d = 1; } }   // nv_wavenet.cuh:99-111
        for (int i = tid; i < L * 128; i += NTC) sts32(sm + M::P_BIAS + i * 4, __float_as_uint(gbias[im.b_layer + (i >> 2) * 8 + (i & 3)]));
    }
    __syncthreads();
    cluster_sync_all();                                    // every CTA's barriers are initialised before anybody signals a peer

    const int w = warp, g = lane >> 2, t4 = lane & 3;
    const int b0 = tile * TU + g, b1 = b0 + 8;
    const bool v0 = b0 < B, v1 = b1 < B;
    const uint32_t lane16 = (uint32_t)lane * 16;
    const int jw = w >> 1, hw = w & 1;
    const uint32_t xchg = (uint32_t)(jw * 512 + hw * 8) + lane16;
    auto release = [&](uint32_t bar) { __syncwarp(); if (lane == 0) mbar_arrive_a(bar); };
    auto release_remote = [&](uint32_t local_bar, uint32_t rank) { __syncwarp(); if (lane == 0) mbar_arrive_remote(mapa_u32(local_bar, rank)); };

    if (is_chain) {
        // ===================================================================================== chain CTA
        if (warp == NCW) {
            if (lane == 0) {
                uint32_t pc = 0;
                for (int t = t_begin; t < t_end; t++)
                    for (int l = 0; l < L; l++, pc++) {
                        const uint32_t sl = pc & 1;
                        mbar_wait_a(s_empty + 8 * sl, ((pc >> 1) & 1) ^ 1);
                        mbar_expect_a(s_full + 8 * sl, M::PIECE0);
                        tma_load_a(sm + M::C_RING + sl * M::PIECE0, img + (size_t)l * im.layer_bytes + C::W_CUR, 16384, s_full + 8 * sl);
                        tma_load_a(sm + M::C_RING + sl * M::PIECE0 + 16384, img + (size_t)l * im.layer_bytes + C::W_RES, 8192, s_full + 8 * sl);
                    }
            }
        } else {
            const uint32_t rstride = (uint32_t)ntiles_alloc * 2048u;
            unsigned char* gring = static_cast<unsigned char*>(p.ring) + (size_t)tile * 2048;
            const int cw = 8 * w + 2 * t4;
            const uint32_t o_t0 = (uint32_t)(w * 2) * 512 + lane16, o_g0 = (uint32_t)((8 + w) * 2) * 512 + lane16, o_res = 16384u + (uint32_t)(w * 2) * 512 + lane16;
            const uint32_t r_hbuf = mapa_u32(sm + M::T_HBUF + xchg, 1);            // this thread's slot of the tail CTA's h tiles
            const uint32_t r_hfull = mapa_u32(s_hfull, 1);
            const uint32_t s_bias = sm + M::C_BIAS + (uint32_t)(w * 4 + t4) * 32;   // this thread's Bh / Bres pairs of layer 0 (+ 1 KB per layer)
            const uint32_t s_ap = sm + M::C_AP + (uint32_t)(w * 32 + lane) * 32;    // this thread's 8 floats of a pre-activation tile (+ 8 KB per buffer)
            uint32_t xa[4][4];
            float accp[2][4];
            float2 brn = make_float2(0.f, 0.f);
            float xres[4] = {0.f, 0.f, 0.f, 0.f};
            int t1 = t_begin, l1 = 0;                          // the coming step (number pn)
            uint32_t pn = 0;
            // accp <- (Bh + Lh) + Wprev . x[t-d] of the coming step: computed by the prep CTA, read from this CTA's shared memory
            auto prep = [&](const bool ap_ok) {
                if (t1 < t_end) {
                    const uint2 b2 = lds64(s_bias + l1 * 1024 + 16);
                    if (!ap_ok) mbar_wait_a(s_apfull + 8 * (pn & 3), (pn >> 2) & 1);
                    const uint4 a0 = lds128(s_ap + (pn & 3) * 8192), a1 = lds128(s_ap + (pn & 3) * 8192 + 16);
                    brn = make_float2(__uint_as_float(b2.x), __uint_as_float(b2.y));
                    accp[0][0] = __uint_as_float(a0.x); accp[0][1] = __uint_as_float(a0.y); accp[0][2] = __uint_as_float(a0.z); accp[0][3] = __uint_as_float(a0.w);
                    accp[1][0] = __uint_as_float(a1.x); accp[1][1] = __uint_as_float(a1.y); accp[1][2] = __uint_as_float(a1.z); accp[1][3] = __uint_as_float(a1.w);
                    // the tile has been read: arm its barrier for the tile NAP steps on (one thread, ordered before this warp's "free"
                    // signal), then hand the buffer back to the prep CTA
                    if (tid == 0) mbar_expect_a(s_apfull + 8 * (pn & 3), 8192);
                    release_remote(s_apfree + 8 * (pn & 3), 2);
                }
                pn++;
                if (++l1 == L) { l1 = 0; t1++; }
            };
            {   // prologue: previous-index rows of the first sample; staging of steps 0, 1, 2; pre-activation of step 0
                const uint32_t* ep = static_cast<const uint32_t*>(p.embPrev);
                sts32(sm + M::C_EPBUF + (g * EROW + 4 * w + t4) * 4, ep[ys[TU + g] * 32 + 4 * w + t4]);
                sts32(sm + M::C_EPBUF + ((g + 8) * EROW + 4 * w + t4) * 4, ep[ys[TU + g + 8] * 32 + 4 * w + t4]);
            }
            StepIt it0{t_begin, 0, t_begin % slots};
            prep(false);                                       // step 0
            bar_compute();

            uint32_t pc = 0, epar = 0, hcnt = 0;               // ring piece counter, sample parity, h tiles handed over
            bool ok_f = false, ok_ap = false, ok_hf = false;
            for (int t = t_begin; t < t_end; t++) {
                TRACE2(0, 1);
                if (t > t_begin) {                             // the tail CTA has written this sample's indices into ys
                    mbar_wait_a(s_yfull, (uint32_t)(t - t_begin - 1) & 1);
                    if (tid == 0 && t + 1 < t_end) mbar_expect_a(s_yfull, 2 * TU * 4);          // arm the next hand-back
                }
                {   // embedding (reference.cpp:42-57), this warp's 8 channels
                    const int yc0 = ys[g], yc1 = ys[g + 8];
                    const uint32_t eo = sm + M::C_EPBUF + epar * (TU * EROW * 4);
                    const float2 a0 = unpack_h2(lds32(eo + (g * EROW + 4 * w + t4) * 4)), a1 = unpack_h2(lds32(eo + ((g + 8) * EROW + 4 * w + t4) * 4));
                    const float2 c0 = unpack_h2(lds32(sm + M::C_EMB + (yc0 * EROW + 4 * w + t4) * 4)), c1 = unpack_h2(lds32(sm + M::C_EMB + (yc1 * EROW + 4 * w + t4) * 4));
                    xres[0] = a0.x + c0.x; xres[1] = a0.y + c0.y; xres[2] = a1.x + c1.x; xres[3] = a1.y + c1.y;
                    if (p.tanhEmbed) {
#pragma unroll
                        for (int i = 0; i < 4; i++) xres[i] = wn::tanhf_fast(xres[i]);
                    }
                    const uint32_t x01 = pack_h2(xres[0], xres[1]), x23 = pack_h2(xres[2], xres[3]);
                    sts64(sm + M::C_XBUF + xchg, x01, x23);
                    stg_v2(gring + lane16 + (size_t)(it0.slot * L) * rstride + jw * 512 + hw * 8, x01, x23);
                    const unsigned char* ep = static_cast<const unsigned char*>(p.embPrev);
                    const uint32_t en = sm + M::C_EPBUF + (epar ^ 1) * (TU * EROW * 4);
                    cp_async4(en + (g * EROW + 4 * w + t4) * 4, ep + (size_t)yc0 * 128 + (4 * w + t4) * 4);
                    cp_async4(en + ((g + 8) * EROW + 4 * w + t4) * 4, ep + (size_t)yc1 * 128 + (4 * w + t4) * 4);
                    cp_async_commit();                         // landed long before the next sample starts (waited for at the end of this one)
                }
                bar_compute();
#pragma unroll
                for (int j = 0; j < 4; j++) load_a(xa[j], sm + M::C_XBUF + j * 512 + lane16);
                TRACE2(0, 2);

                for (int l = 0; l < L; l++, pc++) {
                    const uint32_t sl = pc & 1, p1 = sm + M::C_RING + sl * M::PIECE0, fph = (pc >> 1) & 1;
                    const float2 br = brn;
                    if (!ok_f) mbar_wait_a(s_full + 8 * sl, fph);
                    {
                        const uint4 bt0 = lds128(p1 + o_t0), bg0 = lds128(p1 + o_g0), bt1 = lds128(p1 + o_t0 + 512), bg1 = lds128(p1 + o_g0 + 512);
                        float u0[4] = {0.f, 0.f, 0.f, 0.f}, u1[4] = {0.f, 0.f, 0.f, 0.f};
                        hmma(accp[0], xa[0], bt0.x, bt0.y); hmma(accp[1], xa[0], bg0.x, bg0.y); hmma(u0, xa[2], bt1.x, bt1.y); hmma(u1, xa[2], bg1.x, bg1.y);
                        hmma(accp[0], xa[1], bt0.z, bt0.w); hmma(accp[1], xa[1], bg0.z, bg0.w); hmma(u0, xa[3], bt1.z, bt1.w); hmma(u1, xa[3], bg1.z, bg1.w);
#pragma unroll
                        for (int i = 0; i < 4; i++) { accp[0][i] += u0[i]; accp[1][i] += u1[i]; }
                    }
                    {
                        const __half2 half = __floats2half2_rn(0.5f, 0.5f);
                        const __half2 tg0 = wn::tanh_h2(h2(pack_h2(accp[0][0], accp[0][1]))), tg1 = wn::tanh_h2(h2(pack_h2(accp[0][2], accp[0][3])));
                        const __half2 sg0 = __hfma2(wn::tanh_h2(h2(pack_h2(0.5f * accp[1][0], 0.5f * accp[1][1]))), half, half);
                        const __half2 sg1 = __hfma2(wn::tanh_h2(h2(pack_h2(0.5f * accp[1][2], 0.5f * accp[1][3]))), half, half);
                        const uint32_t h01 = u32(__hmul2(tg0, sg0)), h23 = u32(__hmul2(tg1, sg1));
                        sts64(sm + M::C_HBUF + xchg, h01, h23);
                        // the tail CTA's copy: buffer hcnt & 1, free once the tail has read the tile of two steps ago
                        if (!ok_hf) mbar_wait_a(s_hfree + 8 * (hcnt & 1), ((hcnt >> 1) & 1) ^ 1);
                        st_async_v2(r_hbuf + (hcnt & 1) * 2048, h01, h23, r_hfull + 8 * (hcnt & 1));
                        hcnt++;
                    }
                    TRACE2(0, 12);
                    prep(ok_ap);
                    bar_compute();
                    uint32_t ha[4][4];
#pragma unroll
                    for (int j = 0; j < 4; j++) load_a(ha[j], sm + M::C_HBUF + j * 512 + lane16);
                    TRACE2(0, 10);
                    float ra[4] = {0.f, 0.f, 0.f, 0.f}, rb[4] = {0.f, 0.f, 0.f, 0.f};
                    {
                        const uint4 bw0 = lds128(p1 + o_res), bw1 = lds128(p1 + o_res + 512);
                        hmma(ra, ha[0], bw0.x, bw0.y); hmma(rb, ha[2], bw1.x, bw1.y);
                        hmma(ra, ha[1], bw0.z, bw0.w); hmma(rb, ha[3], bw1.z, bw1.w);
                    }
                    release(s_empty + 8 * sl);
                    xres[0] = ((ra[0] + rb[0]) + br.x) + xres[0]; xres[1] = ((ra[1] + rb[1]) + br.y) + xres[1];
                    xres[2] = ((ra[2] + rb[2]) + br.x) + xres[2]; xres[3] = ((ra[3] + rb[3]) + br.y) + xres[3];
                    if (l + 1 < L) {
                        const uint32_t x01 = pack_h2(xres[0], xres[1]), x23 = pack_h2(xres[2], xres[3]);
                        sts64(sm + M::C_XBUF + xchg, x01, x23);
                        stg_v2(gring + lane16 + (size_t)(it0.slot * L + l + 1) * rstride + jw * 512 + hw * 8, x01, x23);
                    }
                    TRACE2(0, 14);
                    if (DUMP) {
                        if (v0) { p.xtOut[((size_t)l * B + b0) * R + cw] = xres[0]; p.xtOut[((size_t)l * B + b0) * R + cw + 1] = xres[1]; }
                        if (v1) { p.xtOut[((size_t)l * B + b1) * R + cw] = xres[2]; p.xtOut[((size_t)l * B + b1) * R + cw + 1] = xres[3]; }
                    }
                    {   // look at the coming step's barriers
                        const uint32_t npc = pc + 1;
                        ok_f = mbar_probe_a(s_full + 8 * (npc & 1), (npc >> 1) & 1);
                        ok_ap = mbar_probe_a(s_apfull + 8 * (pn & 3), (pn >> 2) & 1);
                        ok_hf = mbar_probe_a(s_hfree + 8 * (hcnt & 1), ((hcnt >> 1) & 1) ^ 1);
                    }
                    TRACE2(0, 13);
                    if (l + 1 < L) {
                        bar_compute();
#pragma unroll
                        for (int j = 0; j < 4; j++) load_a(xa[j], sm + M::C_XBUF + j * 512 + lane16);
                    }
                    TRACE2(0, 11);
                }
                cp_async_wait_all();                           // the previous-index rows of the next sample
                epar ^= 1;
                if (++it0.slot == slots) it0.slot = 0;
                it0.t++;
            }
        }
    } else if (is_tail) {
        // ===================================================================================== tail CTA
        if (warp == NCW) {
            if (lane == 0) {
                uint32_t pc = 0;
                auto put = [&](const unsigned char* src, uint32_t bytes) {
                    const uint32_t sl = pc & 3;
                    mbar_wait_a(s_empty + 8 * sl, ((pc >> 2) & 1) ^ 1);
                    mbar_expect_a(s_full + 8 * sl, bytes);
                    tma_load_a(sm + M::T_RING + sl * M::SLOT1, src, bytes, s_full + 8 * sl);
                    pc++;
                };
                for (int t = t_begin; t < t_end; t++) {
                    for (int l = 0; l < L; l++) put(img + (size_t)l * im.layer_bytes + C::W_SKIP, S * 128);
                    for (int q = 0; q < NQ; q++)
                        put(q < C::NQ_ZS ? img + im.off_zs + (size_t)q * C::ZS_PIECE : img + im.off_za + (size_t)(q - C::NQ_ZS) * C::ZA_PIECE,
                            q < C::NQ_ZS ? C::ZS_PIECE : C::ZA_PIECE);
                }
            }
        } else {
            float* s_bout = reinterpret_cast<float*>(smem_raw + M::T_BOUT);
            const uint32_t o_skip = (uint32_t)(w * C::NSK * 2) * 512 + lane16, o_out = (uint32_t)(4 * w) * 512;
            float sk[C::NSK][4];
#pragma unroll
            for (int i = 0; i < C::NSK; i++) sk[i][0] = sk[i][1] = sk[i][2] = sk[i][3] = 0.f;
            uint32_t pc = 0, hcnt = 0;
            for (int t = t_begin; t < t_end; t++) {
                const float sel0 = (2 * w + 0 + tile * TU) < B ? p.sel[(size_t)t * B + tile * TU + 2 * w] : 0.5f;
                const float sel1 = (2 * w + 1 + tile * TU) < B ? p.sel[(size_t)t * B + tile * TU + 2 * w + 1] : 0.5f;
                for (int l = 0; l < L; l++, pc++, hcnt++) {
                    const uint32_t hb = sm + M::T_HBUF + (hcnt & 1) * 2048;
                    mbar_wait_a(s_hfull + 8 * (hcnt & 1), (hcnt >> 1) & 1);
                    TRACE2(1, 16);
                    uint32_t ha[4][4];
#pragma unroll
                    for (int j = 0; j < 4; j++) load_a(ha[j], hb + j * 512 + lane16);
                    const uint32_t sl = pc & 3, p2 = sm + M::T_RING + sl * M::SLOT1;
                    mbar_wait_a(s_full + 8 * sl, (pc >> 2) & 1);
#pragma unroll
                    for (int jp = 0; jp < 2; jp++) {
                        uint4 bw[C::NSK];
#pragma unroll
                        for (int i = 0; i < C::NSK; i++) bw[i] = lds128(p2 + o_skip + (i * 2 + jp) * 512);
#pragma unroll
                        for (int i = 0; i < C::NSK; i++) hmma(sk[i], ha[2 * jp], bw[i].x, bw[i].y);
#pragma unroll
                        for (int i = 0; i < C::NSK; i++) hmma(sk[i], ha[2 * jp + 1], bw[i].z, bw[i].w);
                    }
                    // the h tile has been read (the HMMAs above hold its values): arm its barrier for the tile after next (one thread,
                    // ordered before this warp's "free" signal), then hand the buffer back to the chain CTA
                    if (tid == 0) mbar_expect_a(s_hfull + 8 * (hcnt & 1), 2048);
                    release_remote(s_hfree + 8 * (hcnt & 1), 0);
                    release(s_empty + 8 * sl);
                    TRACE2(1, 15);
                    if (DUMP) {
                        const float* pre = gbias + im.b_skpre + (size_t)l * S;
#pragma unroll
                        for (int i = 0; i < C::NSK; i++) {
                            const int c = 8 * (w * C::NSK + i) + 2 * t4;
                            float o0 = sk[i][0] + pre[c], o1 = sk[i][1] + pre[c + 1], o2 = sk[i][2] + pre[c], o3 = sk[i][3] + pre[c + 1];
                            if (l == L - 1) { o0 = fmaxf(o0, 0.f); o1 = fmaxf(o1, 0.f); o2 = fmaxf(o2, 0.f); o3 = fmaxf(o3, 0.f); }
                            if (v0) { p.skipOut[((size_t)l * B + b0) * S + c] = o0; p.skipOut[((size_t)l * B + b0) * S + c + 1] = o1; }
                            if (v1) { p.skipOut[((size_t)l * B + b1) * S + c] = o2; p.skipOut[((size_t)l * B + b1) * S + c + 1] = o3; }
                        }
                    }
                }
                // ---------------- relu(skip + bias) -> Zs -> Za   (reference.cpp:93-104)
#pragma unroll
                for (int i = 0; i < C::NSK; i++) {
                    const int nt = w * C::NSK + i, c = 8 * nt + 2 * t4;
                    const float b0f = s_bout[c], b1f = s_bout[c + 1];
                    sts64(sm + M::T_OB0 + (nt >> 1) * 512 + lane16 + (nt & 1) * 8,
                          pack_h2(fmaxf(sk[i][0] + b0f, 0.f), fmaxf(sk[i][1] + b1f, 0.f)), pack_h2(fmaxf(sk[i][2] + b0f, 0.f), fmaxf(sk[i][3] + b1f, 0.f)));
                    sk[i][0] = sk[i][1] = sk[i][2] = sk[i][3] = 0.f;
                }
                bar_compute();
                TRACE2(1, 20);
                float zz[4][4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int c = 32 * w + 8 * i + 2 * t4;
                    zz[i][0] = zz[i][2] = s_bout[S + c]; zz[i][1] = zz[i][3] = s_bout[S + c + 1];
                }
                auto out_gemm = [&](const int ojp, const uint32_t abuf, const int kp0) {
                    const uint32_t sl = pc & 3, st = sm + M::T_RING + sl * M::SLOT1 + o_out * ojp + lane16;
                    mbar_wait_a(s_full + 8 * sl, (pc >> 2) & 1);
                    for (int jp = 0; jp < ojp; jp++) {
                        uint32_t a0[4], a1[4];
                        load_a(a0, abuf + ((kp0 + jp) * 2) * 512 + lane16);
                        load_a(a1, abuf + ((kp0 + jp) * 2 + 1) * 512 + lane16);
                        uint4 bw[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) bw[i] = lds128(st + (i * ojp + jp) * 512);
#pragma unroll
                        for (int i = 0; i < 4; i++) hmma(zz[i], a0, bw[i].x, bw[i].y);
#pragma unroll
                        for (int i = 0; i < 4; i++) hmma(zz[i], a1, bw[i].z, bw[i].w);
                    }
                    release(s_empty + 8 * sl);
                    pc++;
                };
#pragma unroll
                for (int q = 0; q < C::NQ_ZS; q++) out_gemm(C::OJP_ZS, sm + M::T_OB0, q * C::OJP_ZS);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int nt = 4 * w + i, c = 8 * nt + 2 * t4;
                    const float z0 = fmaxf(zz[i][0], 0.f), z1 = fmaxf(zz[i][1], 0.f), z2 = fmaxf(zz[i][2], 0.f), z3 = fmaxf(zz[i][3], 0.f);
                    sts64(sm + M::T_OB1 + (nt >> 1) * 512 + lane16 + (nt & 1) * 8, pack_h2(z0, z1), pack_h2(z2, z3));
                    if (DUMP) {
                        if (v0) { p.Zs[(size_t)b0 * A + c] = z0; p.Zs[(size_t)b0 * A + c + 1] = z1; }
                        if (v1) { p.Zs[(size_t)b1 * A + c] = z2; p.Zs[(size_t)b1 * A + c + 1] = z3; }
                    }
                    zz[i][0] = zz[i][2] = s_bout[S + A + c]; zz[i][1] = zz[i][3] = s_bout[S + A + c + 1];
                }
                bar_compute();
                TRACE2(1, 21);
#pragma unroll
                for (int q = 0; q < C::NQ_ZA; q++) out_gemm(C::OJP_ZA, sm + M::T_OB1, q * C::OJP_ZA);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int c = 32 * w + 8 * i + 2 * t4;
                    sts64(sm + M::T_LBUF + (g * LROW + c) * 4, __float_as_uint(zz[i][0]), __float_as_uint(zz[i][1]));
                    sts64(sm + M::T_LBUF + ((g + 8) * LROW + c) * 4, __float_as_uint(zz[i][2]), __float_as_uint(zz[i][3]));
                    if (DUMP) {
                        if (v0) { p.Za[(size_t)b0 * A + c] = zz[i][0]; p.Za[(size_t)b0 * A + c + 1] = zz[i][1]; }
                        if (v1) { p.Za[(size_t)b1 * A + c] = zz[i][2]; p.Za[(size_t)b1 * A + c + 1] = zz[i][3]; }
                    }
                }
                bar_compute();
                TRACE2(1, 22);
                {   // softmax + categorical sample: warp w serves utterances 2w and 2w+1; lane holds 8 consecutive classes of each
                    float e[2][8], m[2] = {-INFINITY, -INFINITY};          // the true row max (DESIGN.md §3)
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        const uint4 u0 = lds128(sm + M::T_LBUF + ((2 * w + r) * LROW + 8 * lane) * 4), u1 = lds128(sm + M::T_LBUF + ((2 * w + r) * LROW + 8 * lane + 4) * 4);
                        e[r][0] = __uint_as_float(u0.x); e[r][1] = __uint_as_float(u0.y); e[r][2] = __uint_as_float(u0.z); e[r][3] = __uint_as_float(u0.w);
                        e[r][4] = __uint_as_float(u1.x); e[r][5] = __uint_as_float(u1.y); e[r][6] = __uint_as_float(u1.z); e[r][7] = __uint_as_float(u1.w);
#pragma unroll
                        for (int k = 0; k < 8; k++) m[r] = fmaxf(m[r], e[r][k]);
                    }
#pragma unroll
                    for (int o = 16; o >= 1; o >>= 1) {
                        m[0] = fmaxf(m[0], __shfl_xor_sync(0xffffffffu, m[0], o));
                        m[1] = fmaxf(m[1], __shfl_xor_sync(0xffffffffu, m[1], o));
                    }
                    float incl[2];
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        const float ms = m[r] * 1.4426950408889634f;
                        float run = 0.f;
#pragma unroll
                        for (int k = 0; k < 8; k++) { run += wn::exp2f_fast(fmaf(e[r][k], 1.4426950408889634f, -ms)); e[r][k] = run; }
                        incl[r] = run;
                    }
                    const float tot_lane[2] = {incl[0], incl[1]};
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const float a0 = __shfl_up_sync(0xffffffffu, incl[0], o), a1 = __shfl_up_sync(0xffffffffu, incl[1], o);
                        if (lane >= o) { incl[0] += a0; incl[1] += a1; }
                    }
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        const float total = __shfl_sync(0xffffffffu, incl[r], 31);
                        const float excl = incl[r] - tot_lane[r];
                        const float target = (r == 0 ? sel0 : sel1) * total;
                        int cntk = 0;
#pragma unroll
                        for (int k = 0; k < 8; k++) cntk += (target < excl + e[r][k]) ? 0 : 1;
                        const unsigned ball = __ballot_sync(0xffffffffu, target < incl[r]);
                        const int lf = ball ? __ffs(ball) - 1 : 31;
                        const int ck = __shfl_sync(0xffffffffu, cntk, lf);
                        const int y = ball ? 8 * lf + (ck < 7 ? ck : 7) : A - 1;
                        const int b = tile * TU + 2 * w + r;
                        if (DUMP && b < B) {
                            const float inv = 1.f / total;
                            float prevv = 0.f;
#pragma unroll
                            for (int k = 0; k < 8; k++) { p.P[(size_t)b * A + 8 * lane + k] = (e[r][k] - prevv) * inv; prevv = e[r][k]; }
                        }
                        if (lane == 0) {
                            int fbk = y;
                            if (b < B) {
                                p.yOut[(size_t)b * p.N + t] = y;
                                if (p.forced) fbk = p.forced[(size_t)b * p.N + t];
                            } else fbk = 128;
                            const int yold = ys[2 * w + r];
                            ys[TU + 2 * w + r] = yold;
                            ys[2 * w + r] = fbk;
                            // the chain CTA's copy (it reads it after waiting for yfull)
                            if (t + 1 < t_end) {                  // the chain CTA's copy: data + completion on its yfull barrier
                                const uint32_t rb = mapa_u32(s_yfull, 0);
                                st_async_u32(mapa_u32(sm + M::O_YS + (TU + 2 * w + r) * 4, 0), (uint32_t)yold, rb);
                                st_async_u32(mapa_u32(sm + M::O_YS + (2 * w + r) * 4, 0), (uint32_t)fbk, rb);
                            }
                        }
                    }
                }
                TRACE2(1, 23);
                bar_compute();
            }
            if (tid < TU && tile * TU + tid < B) { p.yCur[tile * TU + tid] = ys[tid]; p.yPrev[tile * TU + tid] = ys[TU + tid]; }
        }
    } else {
        // ===================================================================================== prep CTA
        // (Bh + Lh) + Wprev . x[t-d] of every step, as far ahead of the chain CTA as its NAP tile buffers allow.  Nothing here depends on
        // the current sample: the history it reads was written by the chain CTA at least L - 9 steps earlier (wn_launch_lat asks for L >= 12).
        const int nsteps = p.count * L;
        if (warp == NCW) {
            if (lane == 0) {
                int l = 0;
                for (int n = 0; n < nsteps; n++) {
                    const uint32_t sl = n & 3;
                    mbar_wait_a(s_empty + 8 * sl, ((n >> 2) & 1) ^ 1);
                    mbar_expect_a(s_full + 8 * sl, 16384);
                    // Wprev of layer l lives in the block of the layer before it (lat_pack_kernel)
                    tma_load_a(sm + M::P_RING + sl * 16384, img + (size_t)((l + L - 1) % L) * im.layer_bytes + C::W_PREV, 16384, s_full + 8 * sl);
                    if (++l == L) l = 0;
                }
            }
        } else {
            int* dil = reinterpret_cast<int*>(smem_raw + M::P_DIL);
            const uint32_t rstride = (uint32_t)ntiles_alloc * 2048u, cstride = (uint32_t)ntiles_alloc * 4096u;
            const unsigned char* gring = static_cast<const unsigned char*>(p.ring) + (size_t)tile * 2048;
            const uint32_t o_t0 = (uint32_t)(w * 2) * 512 + lane16, o_g0 = (uint32_t)((8 + w) * 2) * 512 + lane16;
            const uint32_t r_ap = mapa_u32(sm + M::C_AP + (uint32_t)(w * 32 + lane) * 32, 0);   // this thread's 8 floats of the chain CTA's tiles
            const uint32_t r_apfull = mapa_u32(s_apfull, 0);
            const uint32_t s_cond = sm + M::P_COND + (uint32_t)(w * 32 + lane) * 16;  // this thread's 16 B of a conditioning tile (+ 4 KB per slot)
            const uint32_t s_bias = sm + M::P_BIAS + (uint32_t)(w * 4 + t4) * 16;     // this thread's Bh of layer 0 (+ 512 B per layer)
            // Staging of the step `itp`, three steps before its use, no register and no scoreboard involved:
            //  * its conditioning tile: every thread copies the 16 bytes it will read back itself (cp.async; completion = the thread's
            //    own cp.async group, no barrier);
            //  * its dilated history x_l[t-d] (zero before the start of the utterance, nv_wavenet.cuh:106): warps 0-3, 128 x 16 B,
            //    completion on an mbarrier (every warp reads the whole tile).
            // NPS = 8 slots: a slot is staged again five steps after its use, and the weight ring (4 pieces) keeps the warps within four.
            StepIt itp{t_begin, 0, t_begin % slots};
            uint32_t pcnt = 0;
            const unsigned char* cptr = static_cast<const unsigned char*>(p.Lh) + (size_t)tile * 4096 + (size_t)(w * 32 + lane) * 16 + (size_t)t_begin * L * cstride;
            auto stage = [&]() {
                const uint32_t slot = pcnt & (M::NPS - 1);
                if (itp.t < t_end) cp_async16(s_cond + slot * 4096, cptr);
                cptr += cstride;
                if (w < 4) {
                    const int d = dil[itp.l];
                    const uint32_t dst = sm + M::P_PST + slot * 2048 + (uint32_t)(w * 32 + lane) * 16;
                    if (itp.t >= t_end || itp.t < d) {
                        sts128(dst, make_uint4(0, 0, 0, 0));
                        mbar_arrive_a(s_pfull + 8 * slot);
                    } else {
                        int sl = itp.slot - d; if (sl < 0) sl += slots;
                        cp_async16(dst, gring + (size_t)(sl * L + itp.l) * rstride + (size_t)(w * 32 + lane) * 16);
                        cp_async_arrive_noinc(s_pfull + 8 * slot);
                    }
                }
                cp_async_commit();
                pcnt++;
                if (++itp.l == L) { itp.l = 0; itp.t++; if (++itp.slot == slots) itp.slot = 0; }
            };
            stage(); stage(); stage();
            int l1 = 0;
            for (int n = 0; n < nsteps; n++) {
                const uint32_t sl = n & 3, pa = sm + M::P_RING + sl * 16384, slot = n & (M::NPS - 1), buf = n & (M::NAP - 1);
                cp_async_wait_pending<2>();                    // this thread's conditioning of step n has landed (two later groups may be in flight)
                const uint4 cb = lds128(s_cond + slot * 4096);
                const uint4 bq = lds128(s_bias + l1 * 512);
                mbar_wait_a(s_full + 8 * sl, (n >> 2) & 1);
                const uint4 bt0 = lds128(pa + o_t0), bg0 = lds128(pa + o_g0), bt1 = lds128(pa + o_t0 + 512), bg1 = lds128(pa + o_g0 + 512);
                mbar_wait_a(s_pfull + 8 * slot, (n >> 3) & 1);
                uint32_t pb[4][4];
#pragma unroll
                for (int j = 0; j < 4; j++) load_a(pb[j], sm + M::P_PST + slot * 2048 + j * 512 + lane16);
                const float4 bh = make_float4(__uint_as_float(bq.x), __uint_as_float(bq.y), __uint_as_float(bq.z), __uint_as_float(bq.w));
                const float2 c0 = unpack_h2(cb.x), c1 = unpack_h2(cb.y), c2 = unpack_h2(cb.z), c3 = unpack_h2(cb.w);
                float a0[4] = {bh.x + c0.x, bh.y + c0.y, bh.x + c1.x, bh.y + c1.y}, a1[4] = {bh.z + c2.x, bh.w + c2.y, bh.z + c3.x, bh.w + c3.y};
                float u0[4] = {0.f, 0.f, 0.f, 0.f}, u1[4] = {0.f, 0.f, 0.f, 0.f};
                hmma(a0, pb[0], bt0.x, bt0.y); hmma(a1, pb[0], bg0.x, bg0.y); hmma(u0, pb[2], bt1.x, bt1.y); hmma(u1, pb[2], bg1.x, bg1.y);
                hmma(a0, pb[1], bt0.z, bt0.w); hmma(a1, pb[1], bg0.z, bg0.w); hmma(u0, pb[3], bt1.z, bt1.w); hmma(u1, pb[3], bg1.z, bg1.w);
                release(s_empty + 8 * sl);
                // the chain CTA's tile buffer n % NAP is free once it has read tile n - NAP
                mbar_wait_a(s_apfree + 8 * buf, ((n / M::NAP) & 1) ^ 1);
                st_async_v4(r_ap + buf * 8192, a0[0] + u0[0], a0[1] + u0[1], a0[2] + u0[2], a0[3] + u0[3], r_apfull + 8 * buf);
                st_async_v4(r_ap + buf * 8192 + 16, a1[0] + u1[0], a1[1] + u1[1], a1[2] + u1[2], a1[3] + u1[3], r_apfull + 8 * buf);
                stage();
                if (++l1 == L) l1 = 0;
            }
            cp_async_wait_all();
        }
    }
#undef TRACE2
    // nobody leaves while the peer may still write into this CTA's shared memory or arrive on its barriers
    cluster_sync_all();
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
bool wn_lat_supported(int R_, int S, int A_, int L)
{
    return R_ == R && A_ == A && (S == 128 || S == 256) && L >= 4 && L <= MAXL;     // L >= 4: history prefetch runs 3 steps ahead (single-CTA kernel)
}
int wn_lat_tiles(int B) { return (B + TU - 1) / TU; }
size_t wn_lat_image_bytes(int S, int L) { return lat_image(S, L).total; }
size_t wn_lat_ring_bytes(int L, int maxDil, int B) { return (size_t)(maxDil + 1) * L * wn_lat_tiles(B) * 2048; }
size_t wn_lat_cond_bytes(int L, int B, int N) { return (size_t)N * L * wn_lat_tiles(B) * 4096; }

cudaError_t wn_lat_cond_convert(void* dst, const float* src_dev, int first_sample, int nsamples, int L, int B, cudaStream_t stream)
{
    if (nsamples <= 0) return cudaSuccess;
    const int ntiles = wn_lat_tiles(B);
    const size_t total = (size_t)nsamples * L * ntiles * 256;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    lat_cond_kernel<<<(unsigned)blocks, 256, 0, stream>>>(static_cast<unsigned char*>(dst), src_dev, first_sample, nsamples, L, B, ntiles);
    return cudaGetLastError();
}

cudaError_t wn_lat_cond_readback(float* dst_dev, const void* store, int first_sample, int nsamples, int L, int B, cudaStream_t stream)
{
    if (nsamples <= 0) return cudaSuccess;
    const size_t total = (size_t)nsamples * L * B * 64;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    lat_cond_readback_kernel<<<(unsigned)blocks, 256, 0, stream>>>(dst_dev, static_cast<const unsigned char*>(store), first_sample, nsamples, L, B, wn_lat_tiles(B));
    return cudaGetLastError();
}

cudaError_t wn_lat_pack(void* image, const WnParams& p, cudaStream_t stream)
{
    const LatImage im = lat_image(p.S, p.L);
    cudaError_t e = cudaMemsetAsync(image, 0, im.total, stream);
    if (e != cudaSuccess) return e;
    lat_pack_kernel<<<296, 256, 0, stream>>>(p, static_cast<unsigned char*>(image), im);
    return cudaGetLastError();
}

// p.B = utterances of this run; engine_B = batch size the conditioning store / history ring were laid out for
template <int S>
static cudaError_t lat_launch_S(const WnParams& p, const unsigned char* im8, int grid, int ntiles_alloc, cudaStream_t stream, size_t* smem_out)
{
    const size_t smem = Cfg<S>::SMEM;
    *smem_out = smem;
    cudaError_t e;
#define LAT_GO(DUMPV, TRCV, PP)                                                                                                    \
    do {                                                                                                                           \
        e = cudaFuncSetAttribute(wn_lat_kernel<S, DUMPV, TRCV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        if (e != cudaSuccess) return e;                                                                                            \
        wn_lat_kernel<S, DUMPV, TRCV><<<grid, NT, smem, stream>>>(PP, im8, ntiles_alloc);                                          \
        e = cudaGetLastError();                                                                                                    \
        if (e != cudaSuccess) return e;                                                                                            \
    } while (0)
    // a dumping launch = every sample but the last with the plain kernel, then the last one with the dumping variant
    // (a continuation is bit-identical to one launch: the whole state lives in global memory between launches)
    WnParams head = p, tail = p;
    if (p.dump) { head.count = p.count - 1; head.dump = 0; tail.init_sample = p.init_sample + p.count - 1; tail.count = 1; }
    if (head.count > 0) {
        if (p.trace) LAT_GO(false, true, head); else LAT_GO(false, false, head);
    }
    if (p.dump) LAT_GO(true, false, tail);
#undef LAT_GO
    return cudaSuccess;
}

// the cluster variant: grid = NCL x tiles, cluster (NCL, 1, 1)
template <int S, bool DUMP, bool TRC>
static cudaError_t lat2_go(const WnParams& pp, const unsigned char* im8, int tiles, int ntiles_alloc, cudaStream_t stream)
{
    const size_t smem = CfgC<S>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(wn_lat2_kernel<S, DUMP, TRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(NCL * tiles, 1, 1);
    cfg.blockDim = dim3(NTC, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = NCL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, wn_lat2_kernel<S, DUMP, TRC>, pp, im8, ntiles_alloc);
    return e != cudaSuccess ? e : cudaGetLastError();
}
// how many clusters the device runs at once (a cluster needs NCL SMs of one GPC: fewer than 148 / NCL fit); 0 if the query fails
template <int S>
static int lat2_max_clusters()
{
    static int cached = -1;
    if (cached >= 0) return cached;
    const size_t smem = CfgC<S>::SMEM;
    if (cudaFuncSetAttribute(wn_lat2_kernel<S, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return cached = 0; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(NCL * 48, 1, 1);
    cfg.blockDim = dim3(NTC, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = NCL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, wn_lat2_kernel<S, false, false>, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
    return cached = n;
}
template <int S>
static cudaError_t lat2_launch_S(const WnParams& p, const unsigned char* im8, int tiles, int ntiles_alloc, cudaStream_t stream, size_t* smem_out)
{
    *smem_out = CfgC<S>::SMEM;
    WnParams head = p, tail = p;
    if (p.dump) { head.count = p.count - 1; head.dump = 0; tail.init_sample = p.init_sample + p.count - 1; tail.count = 1; }
    cudaError_t e = cudaSuccess;
    if (head.count > 0) e = p.trace ? lat2_go<S, false, true>(head, im8, tiles, ntiles_alloc, stream) : lat2_go<S, false, false>(head, im8, tiles, ntiles_alloc, stream);
    if (e == cudaSuccess && p.dump) e = lat2_go<S, true, false>(tail, im8, tiles, ntiles_alloc, stream);
    return e;
}

int wn_lat_max_clusters(int S) { return S == 256 ? lat2_max_clusters<256>() : S == 128 ? lat2_max_clusters<128>() : 0; }

// cluster: serve every 16-utterance tile with a cluster of three CTAs (chain / tail / prep) instead of one
cudaError_t wn_launch_lat(const WnParams& p, const void* image, int engine_B, bool cluster, cudaStream_t stream, WnLaunchInfo* info)
{
    const int grid = wn_lat_tiles(p.B), ntiles_alloc = wn_lat_tiles(engine_B);
    const unsigned char* im8 = static_cast<const unsigned char*>(image);
    size_t smem = 0;
    cudaError_t e;
    // the cluster kernel's prep CTA reads history tiles the chain CTA wrote at least L - 9 steps earlier: it wants a few steps of margin
    const int fit = cluster ? wn_lat_max_clusters(p.S) : 0;
    if (cluster && p.L >= 12 && grid <= fit) {               // every cluster must be resident at once: a second wave would halve the rate
        if (p.S == 256) e = lat2_launch_S<256>(p, im8, grid, ntiles_alloc, stream, &smem);
        else if (p.S == 128) e = lat2_launch_S<128>(p, im8, grid, ntiles_alloc, stream, &smem);
        else return cudaErrorInvalidValue;
        if (e != cudaSuccess) return e;
        if (info) { info->kernel = 18; info->grid = NCL * grid; info->block = NTC; info->smem_bytes = (int)smem; info->batch_per_cta = TU; info->cluster = NCL; }
        return cudaGetLastError();
    }
    if (p.S == 256) e = lat_launch_S<256>(p, im8, grid, ntiles_alloc, stream, &smem);
    else if (p.S == 128) e = lat_launch_S<128>(p, im8, grid, ntiles_alloc, stream, &smem);
    else return cudaErrorInvalidValue;
    if (e != cudaSuccess) return e;
    if (info) { info->kernel = 18; info->grid = grid; info->block = NT; info->smem_bytes = (int)smem; info->batch_per_cta = TU; info->cluster = 1; }
    return cudaGetLastError();
}
