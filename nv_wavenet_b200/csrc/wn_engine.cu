// wn_engine.cu -- host side of the B200 WaveNet inference engine + the handle C-ABI (include/nvwn_b200.h).
//
// Owns every device buffer, uploads / converts weights and inputs, picks the kernel and launches it.
// Re-design of the reference host class nvWavenetInfer<T_weight,T_data,R,S,A> (nv_wavenet.cuh:220-640):
//   * all weights live in ONE packed device blob (so a multi-GPU job broadcasts it with a single NCCL call);
//   * fp32 -> fp16 conversion runs on the device from a pinned/device staging area, asynchronously;
//   * every buffer is freed; pointer kinds are detected with cudaPointerGetAttributes().type
//     (the reference's attributes.memoryType no longer compiles, nv_wavenet_conversions.cuh:41);
//   * yOut copies use cudaMemcpyDefault, so `samples` may be host or device memory.
#include "../../include/nvwn_b200.h"
#include "wn_common.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

cudaError_t wn_launch_tc(const WnParams& p, const void* tc_image, int TU, bool fused, cudaStream_t stream, WnLaunchInfo* info);   // wn_tc_kernel.cu
int wn_tc_tile_utt(int B, int S);
bool wn_tc_fused_default();
bool wn_tc_supported(int R, int S, int A, int L, int B);
cudaError_t wn_cond_transpose_wu(float* WuT, const float* Wu, int C, int K, cudaStream_t stream);              // wn_cond_producer.cu
cudaError_t wn_cond_produce(float* out, float* U, const float* feat, const float* WuT, const float* bu, const float* Wc, const float* bc,
                            int B, int C, int T, int K, int stride, int L, int R, int n0, int m, cudaStream_t stream);
void wn_cond_host(float* Lh, const float* feat, const float* Wu, const float* bu, const float* Wc, const float* bc,
                  int B, int C, int T, int K, int stride, int L, int R);
cudaError_t wn_mulaw_decode(const int* yOut, int N, int offset, int size, int B, int A, const float* lut_f, const short* lut_s, float* out_f,
                            short* out_s, size_t out_pitch, cudaStream_t stream);                                // wn_convert.cu
size_t wn_tc_image_bytes(int R, int S, int A, int L);
cudaError_t wn_tc_pack(void* image, const WnParams& p, cudaStream_t stream);
size_t wn_tc_ring_bytes(int TU, int L, int maxDil, int B);
size_t wn_tc_cond_bytes(int TU, int L, int B, int N);
cudaError_t wn_tc_cond_convert(void* dst, const float* src_dev, int first_sample, int nsamples, int TU, int L, int B, cudaStream_t stream);
// latency-mode fp16 kernel (wn_lat_kernel.cu)
bool wn_lat_supported(int R, int S, int A, int L);
size_t wn_lat_image_bytes(int S, int L);
size_t wn_lat_ring_bytes(int L, int maxDil, int B);
size_t wn_lat_cond_bytes(int L, int B, int N);
cudaError_t wn_lat_cond_convert(void* dst, const float* src_dev, int first_sample, int nsamples, int L, int B, cudaStream_t stream);
cudaError_t wn_lat_pack(void* image, const WnParams& p, cudaStream_t stream);
cudaError_t wn_lat_cond_readback(float* dst_dev, const void* store, int first_sample, int nsamples, int L, int B, cudaStream_t stream);
cudaError_t wn_tc_cond_readback(float* dst_dev, const void* store, int first_sample, int nsamples, int TU, int L, int B, cudaStream_t stream);
cudaError_t wn_launch_lat(const WnParams& p, const void* image, int engine_B, bool cluster, cudaStream_t stream, WnLaunchInfo* info);
int wn_lat_max_clusters(int S);

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}

#define CK(call)                                                                                             \
    do {                                                                                                     \
        cudaError_t _e = (call);                                                                             \
        if (_e != cudaSuccess)                                                                               \
            return fail((int)_e, std::string(cudaGetErrorString(_e)) + " at " __FILE__ ":" + std::to_string(__LINE__)); \
    } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

bool is_device_ptr(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

}  // namespace

struct nvwn_engine {
    int dtype, R, S, A, L, maxDil, B, N, impl, tanhEmbed, device;
    size_t td;                               // sizeof(TD)
    // windowed engine (nvwn_create_windowed): every per-sample store holds N = W samples, sample t in slot t % W; 0 = full engine
    int W = 0;
    long long gen_lo = 0, gen_hi = -1;       // windowed: samples [gen_lo, gen_hi) generated back to back since nvwn_reset_history

    // packed weight blob (TD elements), offsets in bytes
    char* blob = nullptr;
    size_t blob_bytes = 0;
    size_t o_embPrev, o_embCur, o_Wprev, o_Wcur, o_Wres, o_Wskip, o_Wzs, o_Wza, o_Bh, o_Bres, o_Bskip, o_Bzs, o_Bza;

    void* Lh = nullptr;                      // TD [N][L][B][2R]
    float* sel = nullptr;                    // [N][B]
    int* forced = nullptr;                   // [B][N]; not allocated on windowed engines
    bool use_forced = false;
    int *yPrev = nullptr, *yCur = nullptr, *yOut = nullptr;
    void* ring = nullptr;
    float *xtOut = nullptr, *skipOut = nullptr, *Zs = nullptr, *Za = nullptr, *P = nullptr;

    float* stage_dev = nullptr;              // device fp32 staging for host->fp16 uploads
    size_t stage_elems = 0;

    void* tc_image = nullptr;                // tensor-core kernel's pre-tiled weight image
    bool tc_dirty = true;
    bool tc_mode = false;                    // decided once at creation: conditioning + history use the tiled layouts
    int tc_tile = 64;                        // utterances per tensor-core tile and its schedule: resolved ONCE at creation (the
    bool tc_fused = false;                   // conditioning store, the history ring and every launch depend on them)
    bool lat_cluster = true;                 // latency mode: a three-CTA cluster per tile while 3 x tiles fit one wave (NVWN_LAT_CLUSTER=0 disables; read once)
    bool lat_mode = false;                   // decided once at creation: latency-mode kernel (fragment-ordered layouts); tc_image holds its weight image

    // conditioning producer (nvwn_cond_producer_load / _run): features | Wu | WuT | bu | Wc | bc | U chunk | Lh chunk in one allocation
    float* cp_scratch = nullptr;
    size_t cp_floats = 0;
    int cp_C = 0, cp_T = 0, cp_K = 0, cp_stride = 0, cp_chunk = 0;

    float* lut_f = nullptr;                  // mu-law decode tables (nvwn_get_audio): A floats, then 2 x A int16 (wrap / saturate)
    unsigned long long* trace = nullptr;     // debug timeline (nvwn_debug_trace)
    int trace_t = -1;

    WnLaunchInfo last{};
    unsigned long long launches = 0;

    template <typename T> T* at(size_t off) const { return reinterpret_cast<T*>(blob + off); }
};

namespace {

// dst (TD, device) <- src (fp32, host or device), n elements
int upload(nvwn_engine* e, void* dst, const float* src, size_t n, cudaStream_t stream = 0)
{
    if (n == 0) return 0;
    if (e->dtype != NVWN_FP16) {
        CK(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDefault, stream));
        return 0;
    }
    if (is_device_ptr(src)) {
        CK(wn_f32_to_f16(static_cast<__half*>(dst), src, n, stream));
        return 0;
    }
    // host source: bounce through the device staging buffer in chunks
    size_t done = 0;
    while (done < n) {
        const size_t m = (n - done < e->stage_elems) ? n - done : e->stage_elems;
        CK(cudaMemcpyAsync(e->stage_dev, src + done, m * sizeof(float), cudaMemcpyHostToDevice, stream));
        CK(wn_f32_to_f16(static_cast<__half*>(dst) + done, e->stage_dev, m, stream));
        done += m;
    }
    return 0;
}

// dst (fp32, host or device) <- src (fp32 device)
int download(float* dst, const float* src, size_t n)
{
    CK(cudaMemcpy(dst, src, n * sizeof(float), cudaMemcpyDefault));
    return 0;
}

// fp16 kernel choice, made ONCE per engine (the layouts of the conditioning store and of the history ring depend on it):
// 0 = stream, 1 = tensor-core (tcgen05, throughput mode), 2 = latency mode (mma.sync, register-resident chain).
// `impl` NVWN_KERNEL_* forces a kernel; the environment variable NVWN_FP16_KERNEL = stream | tc | lat overrides AUTO (tests).
int decide_fp16_kernel(int dtype, int impl, int R, int S, int A, int L, int B)
{
    if (dtype != NVWN_FP16) return 0;
    if (impl == NVWN_KERNEL_STREAM) return 0;
    const bool tc_ok = wn_tc_supported(R, S, A, L, B), lat_ok = wn_lat_supported(R, S, A, L);
    if (impl == NVWN_KERNEL_TENSORCORE) return tc_ok ? 1 : 0;
    if (impl == NVWN_KERNEL_LATENCY) return lat_ok ? 2 : 0;
    if (const char* env = getenv("NVWN_FP16_KERNEL")) {
        if (!strcmp(env, "stream")) return 0;
        if (!strcmp(env, "tc")) return tc_ok ? 1 : 0;
        if (!strcmp(env, "lat")) return lat_ok ? 2 : 0;
    }
    // one 16-utterance tile per SM: up to 148 x 16 utterances run as one wave of latency-mode CTAs
    int lat_max = 148 * 16;
    if (const char* env = getenv("NVWN_LAT_MAX_B")) lat_max = atoi(env);
    if (lat_ok && B <= lat_max) return 2;
    return tc_ok ? 1 : 0;
}

// `pitch` = yOut row stride (num_samples, or W on windowed engines); `origin` = the absolute sample held in slot 0 of the stores
void fill_params(const nvwn_engine* e, WnParams& p, int init_sample, int count, int pitch, int origin, int batch, int dump)
{
    memset(&p, 0, sizeof p);
    p.L = e->L; p.R = e->R; p.S = e->S; p.A = e->A; p.maxDil = e->maxDil;
    p.B = batch; p.N = pitch; p.init_sample = init_sample; p.count = count; p.origin = origin;
    p.tanhEmbed = e->tanhEmbed; p.dump = dump;
    p.embPrev = e->blob + e->o_embPrev; p.embCur = e->blob + e->o_embCur;
    p.Wprev = e->blob + e->o_Wprev; p.Wcur = e->blob + e->o_Wcur; p.Wres = e->blob + e->o_Wres; p.Wskip = e->blob + e->o_Wskip;
    p.Wzs = e->blob + e->o_Wzs; p.Wza = e->blob + e->o_Wza;
    p.Bh = e->blob + e->o_Bh; p.Bres = e->blob + e->o_Bres; p.Bskip = e->blob + e->o_Bskip; p.Bzs = e->blob + e->o_Bzs; p.Bza = e->blob + e->o_Bza;
    p.Lh = e->Lh; p.sel = e->sel; p.forced = e->use_forced ? e->forced : nullptr;
    p.yPrev = e->yPrev; p.yCur = e->yCur; p.ring = e->ring; p.yOut = e->yOut;
    p.xtOut = e->xtOut; p.skipOut = e->skipOut; p.Zs = e->Zs; p.Za = e->Za; p.P = e->P;
    p.trace = e->trace; p.trace_t = e->trace_t;
}

// Splits the absolute sample range [first, first + n) of a windowed engine's store at multiples of W: f(slot, offset into the
// range, length) per piece (one piece, or two where the range crosses the window edge).  On a full engine slot = first.
template <typename F>
int for_slots(const nvwn_engine* e, long long first, long long n, F f)
{
    if (!e->W) return n > 0 ? f((int)first, 0, (int)n) : 0;
    for (long long done = 0; done < n;) {
        const int slot = (int)((first + done) % e->W);
        const long long m = (n - done < e->W - slot) ? n - done : e->W - slot;
        const int rc = f(slot, (int)done, (int)m);
        if (rc) return rc;
        done += m;
    }
    return 0;
}

// the range check of the absolute-sample setters: a full engine holds [0, N); a windowed one takes any range of at most W samples
// with indices below 2^31
int check_range(const nvwn_engine* e, const char* fn, long long first, long long n)
{
    if (first < 0 || n < 0) return fail(NVWN_EINVAL, std::string(fn) + ": sample range out of bounds");
    if (!e->W) return first + n > e->N ? fail(NVWN_EINVAL, std::string(fn) + ": sample range out of bounds") : 0;
    if (n > e->W) return fail(NVWN_EINVAL, std::string(fn) + ": " + std::to_string(n) + " samples exceed the window of " + std::to_string(e->W));
    if (first + n > INT_MAX) return fail(NVWN_EINVAL, std::string(fn) + ": sample indices end at 2^31 - 1");
    return 0;
}

// the output getters of a windowed engine: the range must lie within the last W samples generated since nvwn_reset_history
int check_window_read(const nvwn_engine* e, const char* fn, long long offset, long long size)
{
    const long long lo = e->gen_hi - e->W > e->gen_lo ? e->gen_hi - e->W : e->gen_lo;
    if (offset < 0 || size < 0 || (size > 0 && (offset < lo || offset + size > e->gen_hi)))
        return fail(NVWN_EINVAL, std::string(fn) + ": samples [" + std::to_string(offset) + ", " + std::to_string(offset + size) +
                                     ") are not within the last window of generated samples [" + std::to_string(lo) + ", " +
                                     std::to_string(e->gen_hi < 0 ? 0 : e->gen_hi) + ")");
    return 0;
}

int windowed_unsupported(const nvwn_engine* e, const char* fn)
{
    return fail(NVWN_EUNSUPPORTED, std::string(fn) + ": a windowed engine (window " + std::to_string(e->W) +
                                       ") has no whole-utterance stores; use the range setters (nvwn_set_conditioning, "
                                       "nvwn_set_selectors_range, nvwn_set_selectors_random_range)");
}

int create_engine(nvwn_engine** out, const char* fn, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                  int batch_size, int num_samples, int window, int impl, int tanh_embed);

}  // namespace

extern "C" {

const char* nvwn_last_error(void) { return g_err.c_str(); }

int nvwn_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int nvwn_set_device(int device)
{
    CK(cudaSetDevice(device));
    return 0;
}

int nvwn_create(nvwn_engine** out, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                int batch_size, int num_samples, int impl, int tanh_embed)
{
    return create_engine(out, "nvwn_create", dtype, R, S, A, num_layers, max_dilation, batch_size, num_samples, 0, impl, tanh_embed);
}

int nvwn_create_windowed(nvwn_engine** out, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                         int batch_size, int window, int impl, int tanh_embed)
{
    return create_engine(out, "nvwn_create_windowed", dtype, R, S, A, num_layers, max_dilation, batch_size, window, window, impl, tanh_embed);
}

}  // extern "C"

namespace {

// num_samples = the length of every per-sample store: N of a full engine, W (= window) of a windowed one
int create_engine(nvwn_engine** out, const char* fn, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                  int batch_size, int num_samples, int window, int impl, int tanh_embed)
{
    const std::string f(fn);
    if (!out) return fail(NVWN_EINVAL, f + ": out is NULL");
    *out = nullptr;
    if (dtype != NVWN_FP32 && dtype != NVWN_FP16 && dtype != NVWN_FP32_FAST) return fail(NVWN_EINVAL, f + ": dtype must be NVWN_FP32, NVWN_FP16 or NVWN_FP32_FAST");
    if (num_layers < 1 || max_dilation < 1 || batch_size < 1 || num_samples < 1) return fail(NVWN_EINVAL, f + ": sizes must be positive");
    if (!wn_stream_supported(R, S, A, dtype == NVWN_FP16))
        return fail(NVWN_EUNSUPPORTED, f + ": unsupported channel counts (R,S) must be one of (32,128) (64,128) (64,256) (128,256); A a multiple of 32");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(NVWN_EUNSUPPORTED, f + ": no CUDA device (this engine has no CPU fallback)");
    }
    nvwn_engine* e = new nvwn_engine();
    e->dtype = dtype; e->R = R; e->S = S; e->A = A; e->L = num_layers; e->maxDil = max_dilation;
    e->B = batch_size; e->N = num_samples; e->W = window; e->impl = impl; e->tanhEmbed = tanh_embed ? 1 : 0;
    e->td = dtype == NVWN_FP16 ? 2 : 4;
    cudaGetDevice(&e->device);

    const size_t L = num_layers, td = e->td;
    size_t off = 0;
    auto take = [&](size_t elems) { size_t o = off; off = align_up(off + elems * td, 256); return o; };
    e->o_embPrev = take((size_t)A * R); e->o_embCur = take((size_t)A * R);
    e->o_Wprev = take(L * 2 * R * R); e->o_Wcur = take(L * 2 * R * R);
    e->o_Wres = take(L * R * R); e->o_Wskip = take(L * S * R);
    e->o_Wzs = take((size_t)A * S); e->o_Wza = take((size_t)A * A);
    e->o_Bh = take(L * 2 * R); e->o_Bres = take(L * R); e->o_Bskip = take(L * S);
    e->o_Bzs = take(A); e->o_Bza = take(A);
    e->blob_bytes = off;

    const size_t Bz = batch_size, Nz = num_samples;
    e->stage_elems = dtype == NVWN_FP16 ? ((size_t)16 << 20) : 0;      // 64 MB of fp32 staging
#define ALLOC(ptr, bytes)                                                                     \
    do {                                                                                      \
        cudaError_t _e = cudaMalloc((void**)&(ptr), (bytes));                                 \
        if (_e != cudaSuccess) {                                                              \
            int rc = fail((int)_e, std::string("cudaMalloc(" #ptr "): ") + cudaGetErrorString(_e)); \
            nvwn_destroy(e);                                                                  \
            return rc;                                                                        \
        }                                                                                     \
    } while (0)
    ALLOC(e->blob, e->blob_bytes);
    {
        const int k = decide_fp16_kernel(dtype, impl, R, S, A, num_layers, batch_size);
        e->tc_mode = k == 1; e->lat_mode = k == 2;
        if (const char* v = getenv("NVWN_LAT_CLUSTER")) e->lat_cluster = atoi(v) != 0;
        if (e->tc_mode) { e->tc_tile = wn_tc_tile_utt(batch_size, S); e->tc_fused = wn_tc_fused_default() || e->tc_tile == 32; }
    }
    ALLOC(e->Lh, e->tc_mode ? wn_tc_cond_bytes(e->tc_tile, num_layers, batch_size, num_samples)
                 : e->lat_mode ? wn_lat_cond_bytes(num_layers, batch_size, num_samples) : Nz * L * Bz * 2 * R * td);
    ALLOC(e->sel, Nz * Bz * sizeof(float));
    if (!window) ALLOC(e->forced, Nz * Bz * sizeof(int));           // teacher forcing is a whole-utterance operation
    ALLOC(e->yPrev, Bz * sizeof(int));
    ALLOC(e->yCur, Bz * sizeof(int));
    ALLOC(e->yOut, Nz * Bz * sizeof(int));
    size_t ring_bytes = (size_t)(max_dilation + 1) * L * Bz * R * td;
    if (e->tc_mode) {
        const size_t tcb = wn_tc_ring_bytes(e->tc_tile, num_layers, max_dilation, batch_size);     // tiled history layout of the tensor-core kernel
        if (tcb > ring_bytes) ring_bytes = tcb;
    }
    if (e->lat_mode) ring_bytes = wn_lat_ring_bytes(num_layers, max_dilation, batch_size);
    ALLOC(e->ring, ring_bytes);
    ALLOC(e->xtOut, L * Bz * R * sizeof(float));
    ALLOC(e->skipOut, L * Bz * S * sizeof(float));
    ALLOC(e->Zs, Bz * A * sizeof(float));
    ALLOC(e->Za, Bz * A * sizeof(float));
    ALLOC(e->P, Bz * A * sizeof(float));
    if (e->stage_elems) ALLOC(e->stage_dev, e->stage_elems * sizeof(float));
    if (e->tc_mode) ALLOC(e->tc_image, wn_tc_image_bytes(R, S, A, num_layers));
    if (e->lat_mode) ALLOC(e->tc_image, wn_lat_image_bytes(S, num_layers));
#undef ALLOC
    cudaMemsetAsync(e->blob, 0, e->blob_bytes, 0);
    cudaMemsetAsync(e->yOut, 0, Nz * Bz * sizeof(int), 0);
    cudaMemsetAsync(e->ring, 0, ring_bytes, 0);
    wn_fill_int(e->yPrev, 128, Bz, 0);
    wn_fill_int(e->yCur, 128, Bz, 0);
    cudaError_t se = cudaDeviceSynchronize();
    if (se != cudaSuccess) { int rc = fail((int)se, cudaGetErrorString(se)); nvwn_destroy(e); return rc; }
    *out = e;
    return 0;
}

}  // namespace

extern "C" {

int nvwn_destroy(nvwn_engine* e)
{
    if (!e) return 0;
    void* ptrs[] = {e->blob, e->Lh, e->sel, e->forced, e->yPrev, e->yCur, e->yOut, e->ring, e->xtOut, e->skipOut,
                    e->Zs, e->Za, e->P, e->stage_dev, e->tc_image, e->trace, e->lut_f, e->cp_scratch};
    for (void* p : ptrs) if (p) cudaFree(p);
    delete e;
    return 0;
}

int nvwn_set_embeddings(nvwn_engine* e, const float* embedPrev, const float* embedCur)
{
    if (!e || !embedPrev || !embedCur) return fail(NVWN_EINVAL, "nvwn_set_embeddings: NULL argument");
    int rc;
    if ((rc = upload(e, e->blob + e->o_embPrev, embedPrev, (size_t)e->A * e->R))) return rc;
    if ((rc = upload(e, e->blob + e->o_embCur, embedCur, (size_t)e->A * e->R))) return rc;
    e->tc_dirty = true;
    CK(cudaStreamSynchronize(0));
    return 0;
}

int nvwn_set_layer_weights(nvwn_engine* e, int layer, const float* Wprev, const float* Wcur, const float* Bh,
                           const float* Wres, const float* Bres, const float* Wskip, const float* Bskip)
{
    if (!e || !Wprev || !Wcur || !Bh || !Wres || !Bres || !Wskip || !Bskip) return fail(NVWN_EINVAL, "nvwn_set_layer_weights: NULL argument");
    if (layer < 0 || layer >= e->L) return fail(NVWN_EINVAL, "nvwn_set_layer_weights: layer out of range");
    const size_t R = e->R, S = e->S, l = layer, td = e->td;
    int rc;
    if ((rc = upload(e, e->blob + e->o_Wprev + l * 2 * R * R * td, Wprev, 2 * R * R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Wcur + l * 2 * R * R * td, Wcur, 2 * R * R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Bh + l * 2 * R * td, Bh, 2 * R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Wres + l * R * R * td, Wres, R * R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Bres + l * R * td, Bres, R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Wskip + l * S * R * td, Wskip, S * R))) return rc;
    if ((rc = upload(e, e->blob + e->o_Bskip + l * S * td, Bskip, S))) return rc;
    e->tc_dirty = true;
    CK(cudaStreamSynchronize(0));       // sources may be freed by the caller right after return
    return 0;
}

int nvwn_set_out_weights(nvwn_engine* e, const float* Wzs, const float* Bzs, const float* Wza, const float* Bza)
{
    if (!e || !Wzs || !Bzs || !Wza || !Bza) return fail(NVWN_EINVAL, "nvwn_set_out_weights: NULL argument");
    const size_t A = e->A, S = e->S;
    int rc;
    if ((rc = upload(e, e->blob + e->o_Wzs, Wzs, A * S))) return rc;
    if ((rc = upload(e, e->blob + e->o_Bzs, Bzs, A))) return rc;
    if ((rc = upload(e, e->blob + e->o_Wza, Wza, A * A))) return rc;
    if ((rc = upload(e, e->blob + e->o_Bza, Bza, A))) return rc;
    e->tc_dirty = true;
    CK(cudaStreamSynchronize(0));
    return 0;
}

int nvwn_cond_from_features_host(float* Lh, const float* features, int batch_size, int n_cond_channels, int num_frames,
                                 const float* upsample_weight, const float* upsample_bias, int window, int stride,
                                 const float* cond_weight, const float* cond_bias, int num_layers, int R)
{
    if (!Lh || !features || !upsample_weight || !upsample_bias || !cond_weight || !cond_bias) return fail(NVWN_EINVAL, "nvwn_cond_from_features_host: NULL argument");
    if (batch_size < 1 || n_cond_channels < 1 || num_frames < 1 || window < stride || stride < 1 || num_layers < 1 || R < 1)
        return fail(NVWN_EINVAL, "nvwn_cond_from_features_host: bad sizes (need window >= stride >= 1)");
    wn_cond_host(Lh, features, upsample_weight, upsample_bias, cond_weight, cond_bias, batch_size, n_cond_channels, num_frames, window, stride, num_layers, R);
    return 0;
}

int nvwn_cond_producer_load(nvwn_engine* e, const float* features, int n_cond_channels, int num_frames,
                            const float* upsample_weight, const float* upsample_bias, int window, int stride,
                            const float* cond_weight, const float* cond_bias, void* stream)
{
    if (!e || !features || !upsample_weight || !upsample_bias || !cond_weight || !cond_bias) return fail(NVWN_EINVAL, "nvwn_cond_producer_load: NULL argument");
    const int C = n_cond_channels, T = num_frames, K = window;
    if (C < 1 || T < 1 || stride < 1 || K < stride) return fail(NVWN_EINVAL, "nvwn_cond_producer_load: bad sizes (need window >= stride >= 1)");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t per = (size_t)e->L * e->B * 2 * e->R;                       // floats of conditioning per sample
    int chunk = (int)(((size_t)16 << 20) / per);                             // chunk of whole samples: ~64 MB of fp32 at a time
    if (chunk < 1) chunk = 1;
    const size_t n_feat = (size_t)e->B * C * T, n_wu = (size_t)C * C * K, n_wc = (size_t)e->L * 2 * e->R * C, n_bc = (size_t)e->L * 2 * e->R;
    const size_t floats = n_feat + 2 * n_wu + C + n_wc + n_bc + (size_t)e->B * chunk * C + (size_t)chunk * per + 16;
    if (floats > e->cp_floats) {
        if (e->cp_scratch) { CK(cudaDeviceSynchronize()); cudaFree(e->cp_scratch); e->cp_scratch = nullptr; e->cp_floats = 0; }
        CK(cudaMalloc((void**)&e->cp_scratch, floats * sizeof(float)));
        e->cp_floats = floats;
    }
    e->cp_C = C; e->cp_T = T; e->cp_K = K; e->cp_stride = stride; e->cp_chunk = chunk;
    float* d_feat = e->cp_scratch; float* d_wu = d_feat + n_feat; float* d_wut = d_wu + n_wu; float* d_bu = d_wut + n_wu;
    float* d_wc = d_bu + C; float* d_bc = d_wc + n_wc;
    cudaError_t ce = cudaSuccess;
    auto put = [&](float* dst, const float* src, size_t n) { if (ce == cudaSuccess) ce = cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDefault, st); };
    put(d_feat, features, n_feat); put(d_wu, upsample_weight, n_wu); put(d_bu, upsample_bias, C); put(d_wc, cond_weight, n_wc); put(d_bc, cond_bias, n_bc);
    if (ce == cudaSuccess) ce = wn_cond_transpose_wu(d_wut, d_wu, C, K, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);                   // host sources may be released by the caller now
    if (ce != cudaSuccess) return fail((int)ce, std::string("nvwn_cond_producer_load: ") + cudaGetErrorString(ce));
    return 0;
}

int nvwn_cond_producer_run(nvwn_engine* e, int first_sample, int sample_begin, int sample_count, void* stream)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_cond_producer_run: NULL engine");
    if (!e->cp_scratch || e->cp_T < 1) return fail(NVWN_EINVAL, "nvwn_cond_producer_run: nvwn_cond_producer_load has not been called");
    const int C = e->cp_C, T = e->cp_T, K = e->cp_K, stride = e->cp_stride, chunk = e->cp_chunk;
    const long long Nn = (long long)T * stride;
    if (sample_begin < 0 || sample_count < 0 || sample_begin + (long long)sample_count > Nn) return fail(NVWN_EINVAL, "nvwn_cond_producer_run: sample range outside num_frames * stride");
    if (e->W) {
        if (int rc = check_range(e, "nvwn_cond_producer_run", (long long)first_sample + sample_begin, sample_count)) return rc;
    } else if (first_sample < 0 || first_sample + (long long)sample_begin + sample_count > e->N) return fail(NVWN_EINVAL, "nvwn_cond_producer_run: samples do not fit the engine");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t per = (size_t)e->L * e->B * 2 * e->R;
    const size_t n_feat = (size_t)e->B * C * T, n_wu = (size_t)C * C * K, n_wc = (size_t)e->L * 2 * e->R * C, n_bc = (size_t)e->L * 2 * e->R;
    float* d_feat = e->cp_scratch; float* d_wut = d_feat + n_feat + n_wu; float* d_bu = d_wut + n_wu;
    float* d_wc = d_bu + C; float* d_bc = d_wc + n_wc; float* d_u = d_bc + n_bc;
    float* d_out = d_u + (size_t)e->B * chunk * C;
    d_out += (4 - ((size_t)(d_out - e->cp_scratch) & 3)) & 3;                 // 16-byte aligned rows for the tiled projection's float4 stores
    cudaError_t ce = cudaSuccess;
    int rc = 0;
    for (long long done = sample_begin; done < sample_begin + (long long)sample_count && ce == cudaSuccess && rc == 0; done += chunk) {
        const long long left = sample_begin + (long long)sample_count - done;
        const int m = (int)(left < chunk ? left : chunk);
        ce = wn_cond_produce(d_out, d_u, d_feat, d_wut, d_bu, d_wc, d_bc, e->B, C, T, K, stride, e->L, e->R, (int)done, m, st);
        if (ce == cudaSuccess) rc = nvwn_set_conditioning(e, d_out, first_sample + (int)done, m, stream);      // device source: converted in place, stream-ordered
    }
    if (ce != cudaSuccess) return fail((int)ce, std::string("nvwn_cond_producer_run: ") + cudaGetErrorString(ce));
    return rc;
}

int nvwn_set_conditioning_from_features(nvwn_engine* e, const float* features, int n_cond_channels, int num_frames,
                                        const float* upsample_weight, const float* upsample_bias, int window, int stride,
                                        const float* cond_weight, const float* cond_bias, int first_sample, void* stream)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_set_conditioning_from_features: NULL argument");
    const long long Nn = (long long)num_frames * stride;
    if (e->W && num_frames >= 1 && stride >= 1) {
        if (int rc = check_range(e, "nvwn_set_conditioning_from_features", first_sample, Nn)) return rc;
    } else if (first_sample < 0 || (num_frames >= 1 && stride >= 1 && first_sample + Nn > e->N)) return fail(NVWN_EINVAL, "nvwn_set_conditioning_from_features: num_frames * stride samples do not fit the engine");
    int rc = nvwn_cond_producer_load(e, features, n_cond_channels, num_frames, upsample_weight, upsample_bias, window, stride, cond_weight, cond_bias, stream);
    if (rc != 0) return rc;
    rc = nvwn_cond_producer_run(e, first_sample, 0, (int)Nn, stream);
    if (rc != 0) return rc;
    CK(cudaStreamSynchronize((cudaStream_t)stream));                        // "returns after the work has completed"
    return 0;
}

int nvwn_reset_history(nvwn_engine* e)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_reset_history: NULL engine");
    e->gen_lo = 0; e->gen_hi = -1;
    CK(wn_fill_int(e->yPrev, 128, e->B, 0));      // silenceInputs, nv_wavenet.cuh:213-218
    CK(wn_fill_int(e->yCur, 128, e->B, 0));
    return 0;
}

int nvwn_set_selectors(nvwn_engine* e, const float* selectors)
{
    if (!e || !selectors) return fail(NVWN_EINVAL, "nvwn_set_selectors: NULL argument");
    if (e->W) return windowed_unsupported(e, "nvwn_set_selectors");
    CK(cudaMemcpy(e->sel, selectors, (size_t)e->N * e->B * sizeof(float), cudaMemcpyDefault));
    return 0;
}

int nvwn_libc_selectors(float* selectors, int batch_size, int sample_count)
{
    if (!selectors || batch_size < 1 || sample_count < 1) return fail(NVWN_EINVAL, "nvwn_libc_selectors: bad argument");
    // Matrix outputSelectors(batch_size, sample_count); outputSelectors.randomize(0.5, 1.0)  (pytorch/wavenet_infer.cu:92-93,
    // matrix.cpp:38-56): rows = batch visited outermost, two rand() per element, column-major storage
    for (int b = 0; b < batch_size; b++) {
        for (int s = 0; s < sample_count; s++) {
            (void)(rand() % 100);                                   // sparsity draw (sparsity = 0)
            float r = static_cast<float>(rand()) / static_cast<float>(RAND_MAX);
            r -= 0.5;
            r = r * 1.0f + 0.5f;
            selectors[(size_t)s * batch_size + b] = r;
        }
    }
    return 0;
}

int nvwn_set_selectors_random(nvwn_engine* e, unsigned long long seed, void* stream)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_set_selectors_random: NULL engine");
    if (e->W) return windowed_unsupported(e, "nvwn_set_selectors_random");
    CK(wn_fill_selectors(e->sel, (size_t)e->N * e->B, 0, seed, (cudaStream_t)stream));
    return 0;
}

int nvwn_set_selectors_range(nvwn_engine* e, const float* selectors, int first_sample, int num_samples, void* stream)
{
    if (!e || !selectors) return fail(NVWN_EINVAL, "nvwn_set_selectors_range: NULL argument");
    if (int rc = check_range(e, "nvwn_set_selectors_range", first_sample, num_samples)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = e->B;
    int rc = for_slots(e, first_sample, num_samples, [&](int slot, int done, int m) {
        CK(cudaMemcpyAsync(e->sel + (size_t)slot * B, selectors + (size_t)done * B, (size_t)m * B * sizeof(float), cudaMemcpyDefault, st));
        return 0;
    });
    if (rc) return rc;
    if (!is_device_ptr(selectors)) CK(cudaStreamSynchronize(st));      // host source: copied before return
    return 0;
}

int nvwn_set_selectors_random_range(nvwn_engine* e, unsigned long long seed, int first_sample, int num_samples, void* stream)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_set_selectors_random_range: NULL engine");
    if (int rc = check_range(e, "nvwn_set_selectors_random_range", first_sample, num_samples)) return rc;
    const size_t B = e->B;
    return for_slots(e, first_sample, num_samples, [&](int slot, int done, int m) {
        CK(wn_fill_selectors(e->sel + (size_t)slot * B, (size_t)m * B, ((unsigned long long)first_sample + done) * B, seed, (cudaStream_t)stream));
        return 0;
    });
}

namespace {

// conditioning of store slots [first_sample, first_sample + num_samples) <- Lh (fp32 [num_samples][L][B][2R], host or device)
int put_conditioning(nvwn_engine* e, const float* Lh, int first_sample, int num_samples, void* stream)
{
    const size_t per = (size_t)e->L * e->B * 2 * e->R;
    if (!e->tc_mode && !e->lat_mode)
        return upload(e, static_cast<char*>(e->Lh) + (size_t)first_sample * per * e->td, Lh, per * num_samples, (cudaStream_t)stream);
    // tensor-core layout: fp16, tiled per 128 utterances, 128-byte rows pre-swizzled so that TMA drops them straight into
    // an MMA operand tile (wn_tc_kernel.cu).  Host sources bounce through the staging buffer in whole samples.
    cudaStream_t st = (cudaStream_t)stream;
    auto convert = [&](const float* src_dev, int first, int n) {
        return e->lat_mode ? wn_lat_cond_convert(e->Lh, src_dev, first, n, e->L, e->B, st)
                           : wn_tc_cond_convert(e->Lh, src_dev, first, n, e->tc_tile, e->L, e->B, st);
    };
    if (is_device_ptr(Lh)) {
        CK(convert(Lh, first_sample, num_samples));
        return 0;
    }
    const int chunk = (int)(e->stage_elems / per);
    if (chunk < 1) return fail(NVWN_ENOMEM, "nvwn_set_conditioning: staging buffer smaller than one sample of conditioning");
    for (int done = 0; done < num_samples; done += chunk) {
        const int m = (num_samples - done < chunk) ? num_samples - done : chunk;
        CK(cudaMemcpyAsync(e->stage_dev, Lh + (size_t)done * per, (size_t)m * per * sizeof(float), cudaMemcpyHostToDevice, st));
        CK(convert(e->stage_dev, first_sample + done, m));
    }
    CK(cudaStreamSynchronize(st));      // host source: the header promises the data is copied before return
    return 0;
}

}  // namespace

int nvwn_set_conditioning(nvwn_engine* e, const float* Lh, int first_sample, int num_samples, void* stream)
{
    if (!e || !Lh) return fail(NVWN_EINVAL, "nvwn_set_conditioning: NULL argument");
    if (int rc = check_range(e, "nvwn_set_conditioning", first_sample, num_samples)) return rc;
    const size_t per = (size_t)e->L * e->B * 2 * e->R;
    return for_slots(e, first_sample, num_samples, [&](int slot, int done, int m) {
        return put_conditioning(e, Lh + (size_t)done * per, slot, m, stream);
    });
}

int nvwn_set_inputs(nvwn_engine* e, const float* Lh, const float* selectors)
{
    if (!e || !Lh || !selectors) return fail(NVWN_EINVAL, "nvwn_set_inputs: NULL argument");
    if (e->W) return windowed_unsupported(e, "nvwn_set_inputs");
    int rc;
    if ((rc = nvwn_reset_history(e))) return rc;
    if ((rc = nvwn_set_conditioning(e, Lh, 0, e->N, nullptr))) return rc;
    if ((rc = nvwn_set_selectors(e, selectors))) return rc;
    CK(cudaStreamSynchronize(0));
    return 0;
}

int nvwn_set_forced(nvwn_engine* e, const int* forced)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_set_forced: NULL engine");
    if (e->W) return windowed_unsupported(e, "nvwn_set_forced");
    if (!forced) { e->use_forced = false; return 0; }
    CK(cudaMemcpy(e->forced, forced, (size_t)e->N * e->B * sizeof(int), cudaMemcpyDefault));
    e->use_forced = true;
    return 0;
}

int nvwn_weight_blob(nvwn_engine* e, void** dev_ptr, unsigned long long* bytes)
{
    if (!e || !dev_ptr || !bytes) return fail(NVWN_EINVAL, "nvwn_weight_blob: NULL argument");
    *dev_ptr = e->blob;
    *bytes = e->blob_bytes;
    return 0;
}

int nvwn_weights_updated(nvwn_engine* e)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_weights_updated: NULL engine");
    e->tc_dirty = true;
    return 0;
}

namespace {

// one kernel launch over samples [p.init_sample, p.init_sample + p.count), all in one window period of the stores
int launch(nvwn_engine* e, const WnParams& p, int batch_size, cudaStream_t stream)
{
    if (e->lat_mode) {
        // a smaller batch_size runs the first batch_size utterances of the engine's batch (conditioning was laid out per
        // 16-utterance tile for the engine's batch size at upload)
        if (e->tc_dirty) {
            CK(wn_lat_pack(e->tc_image, p, stream));
            e->tc_dirty = false;
        }
        CK(wn_launch_lat(p, e->tc_image, e->B, e->lat_cluster, stream, &e->last));
    } else if (e->tc_mode) {
        if (batch_size != e->B)
            return fail(NVWN_EINVAL, "nvwn_run_partial: the tensor-core path needs batch_size equal to the engine's batch size");
        if (e->tc_dirty) {
            CK(wn_tc_pack(e->tc_image, p, stream));
            e->tc_dirty = false;
        }
        CK(wn_launch_tc(p, e->tc_image, e->tc_tile, e->tc_fused, stream, &e->last));
    } else {
        CK(wn_launch_stream(p, e->dtype == NVWN_FP16 ? 1 : (e->dtype == NVWN_FP32_FAST ? 2 : 0), stream, &e->last));
    }
    e->launches++;
    return 0;
}

}  // namespace

int nvwn_run_partial(nvwn_engine* e, int init_sample, int count, int num_samples, int batch_size,
                     int* yOut, int dump_activations, void* stream_)
{
    if (!e) return fail(NVWN_EINVAL, "nvwn_run_partial: NULL engine");
    if (batch_size < 1 || batch_size > e->B || num_samples < 1 || (!e->W && num_samples > e->N))
        return fail(NVWN_EINVAL, "nvwn_run_partial: batch_size / num_samples exceed what the engine was created for");
    if (init_sample < 0 || count < 0 || (long long)init_sample + count > num_samples) return fail(NVWN_EINVAL, "nvwn_run_partial: sample range out of bounds");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int dump = dump_activations ? 1 : 0;
    WnParams p;
    if (!e->W) {
        fill_params(e, p, init_sample, count, num_samples, 0, batch_size, dump);
        if (count > 0)
            if (int rc = launch(e, p, batch_size, stream)) return rc;
        if (yOut) CK(cudaMemcpyAsync(yOut, e->yOut, (size_t)num_samples * batch_size * sizeof(int), cudaMemcpyDefault, stream));
        return 0;
    }
    // windowed: the stores hold samples [k W, (k + 1) W) at a time, so a run that crosses a multiple of W is two launches (the
    // history ring and the feedback indices carry over between them exactly as between any two run_partial calls)
    if (yOut) return fail(NVWN_EINVAL, "nvwn_run_partial: yOut must be NULL on a windowed engine (read results with nvwn_get_yout / nvwn_get_audio)");
    if (count > e->W) return fail(NVWN_EINVAL, "nvwn_run_partial: count " + std::to_string(count) + " exceeds the window of " + std::to_string(e->W));
    int rc = for_slots(e, init_sample, count, [&](int slot, int done, int m) {
        const int t0 = init_sample + done;
        fill_params(e, p, t0, m, e->W, t0 - slot, batch_size, dump && done + m == count);
        return launch(e, p, batch_size, stream);
    });
    if (rc) return rc;
    if (count > 0) {
        if (init_sample != e->gen_hi) e->gen_lo = init_sample;
        e->gen_hi = (long long)init_sample + count;
    }
    return 0;
}

int nvwn_run(nvwn_engine* e, int num_samples, int batch_size, int* yOut, int dump_activations, void* stream)
{
    return nvwn_run_partial(e, 0, num_samples, num_samples, batch_size, yOut, dump_activations, stream);
}

int nvwn_get_yout(nvwn_engine* e, int* yOut, int offset, int size, void* stream)
{
    if (!e || !yOut) return fail(NVWN_EINVAL, "nvwn_get_yout: NULL argument");
    if (e->W) {                                   // destination [B][size]; source rows of W slots, split at the window edge
        if (int rc = check_window_read(e, "nvwn_get_yout", offset, size)) return rc;
        return for_slots(e, offset, size, [&](int slot, int done, int m) {
            CK(cudaMemcpy2DAsync(yOut + done, (size_t)size * sizeof(int), e->yOut + slot, (size_t)e->W * sizeof(int), (size_t)m * sizeof(int),
                                 e->B, cudaMemcpyDefault, (cudaStream_t)stream));
            return 0;
        });
    }
    if (offset < 0 || size < 0 || offset + size > e->N) return fail(NVWN_EINVAL, "nvwn_get_yout: range out of bounds");
    if (size == 0) return 0;
    const size_t pitch = (size_t)e->N * sizeof(int);
    CK(cudaMemcpy2DAsync(yOut + offset, pitch, e->yOut + offset, pitch, (size_t)size * sizeof(int), e->B, cudaMemcpyDefault, (cudaStream_t)stream));
    return 0;
}

int nvwn_get_xt_out(nvwn_engine* e, int layer, float* out)
{
    if (!e || !out || layer < 0 || layer >= e->L) return fail(NVWN_EINVAL, "nvwn_get_xt_out: bad argument");
    return download(out, e->xtOut + (size_t)layer * e->B * e->R, (size_t)e->B * e->R);
}
int nvwn_get_skip_out(nvwn_engine* e, int layer, float* out)
{
    if (!e || !out || layer < 0 || layer >= e->L) return fail(NVWN_EINVAL, "nvwn_get_skip_out: bad argument");
    return download(out, e->skipOut + (size_t)layer * e->B * e->S, (size_t)e->B * e->S);
}
int nvwn_get_zs(nvwn_engine* e, float* out) { return (!e || !out) ? fail(NVWN_EINVAL, "nvwn_get_zs: NULL") : download(out, e->Zs, (size_t)e->B * e->A); }
int nvwn_get_za(nvwn_engine* e, float* out) { return (!e || !out) ? fail(NVWN_EINVAL, "nvwn_get_za: NULL") : download(out, e->Za, (size_t)e->B * e->A); }
int nvwn_get_p(nvwn_engine* e, float* out) { return (!e || !out) ? fail(NVWN_EINVAL, "nvwn_get_p: NULL") : download(out, e->P, (size_t)e->B * e->A); }

// mu-law expansion of one code, exactly as the reference's post-processing does it in double precision
// (pytorch/utils.py:62-70 mu_law_decode_numpy, called with mu_quantization = A by pytorch/nv_wavenet_inference.py:58):
//   mu = A - 1;  signal = 2 (x / mu) - 1;  audio = sign(signal) (1 / mu) ((1 + mu)^|signal| - 1)
static double mulaw_expand(int x, int A)
{
    const double mu = (double)A - 1.0;
    const double signal = 2.0 * ((double)x / mu) - 1.0;
    const double magnitude = (1.0 / mu) * (pow(1.0 + mu, fabs(signal)) - 1.0);
    return signal > 0.0 ? magnitude : (signal < 0.0 ? -magnitude : 0.0);
}

int nvwn_mulaw_table(int A, float* f32, short* i16_wrap, short* i16_saturate)
{
    if (A < 2) return fail(NVWN_EINVAL, "nvwn_mulaw_table: A must be at least 2");
    for (int x = 0; x < A; x++) {
        const double a = mulaw_expand(x, A);
        const long long iv = (long long)(32768.0 * a);                       // MAX_WAV_VALUE * audio, truncated (astype('int16'))
        if (f32) f32[x] = (float)a;
        if (i16_wrap) i16_wrap[x] = (short)(unsigned short)((unsigned long long)iv & 0xFFFFull);
        if (i16_saturate) i16_saturate[x] = (short)(iv > 32767 ? 32767 : (iv < -32768 ? -32768 : iv));
    }
    return 0;
}

int nvwn_get_audio(nvwn_engine* e, float* audio_f32, short* audio_i16, int offset, int size, int saturate, void* stream)
{
    if (!e || (!audio_f32 && !audio_i16)) return fail(NVWN_EINVAL, "nvwn_get_audio: NULL argument");
    if (e->W) {
        if (int rc = check_window_read(e, "nvwn_get_audio", offset, size)) return rc;
    } else if (offset < 0 || size < 0 || offset + size > e->N) return fail(NVWN_EINVAL, "nvwn_get_audio: range out of bounds");
    if (size == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int A = e->A;
    if (!e->lut_f) {
        // tables: float[A] | int16[A] (the reference's cast: trunc, code A-1 -> 32768 wraps to -32768) | int16[A] (clamped)
        std::vector<unsigned char> host((size_t)A * (sizeof(float) + 2 * sizeof(short)));
        float* hf = reinterpret_cast<float*>(host.data());
        short* hw = reinterpret_cast<short*>(host.data() + (size_t)A * sizeof(float));
        nvwn_mulaw_table(A, hf, hw, hw + A);
        CK(cudaMalloc((void**)&e->lut_f, host.size()));
        CK(cudaMemcpy(e->lut_f, host.data(), host.size(), cudaMemcpyHostToDevice));
    }
    const short* lut_s = reinterpret_cast<const short*>(e->lut_f + A) + (saturate ? A : 0);
    const size_t total = (size_t)e->B * size;
    const bool f_dev = !audio_f32 || is_device_ptr(audio_f32), s_dev = !audio_i16 || is_device_ptr(audio_i16);
    float* df = audio_f32;
    short* ds = audio_i16;
    void* tmp = nullptr;
    if (!f_dev || !s_dev) {                                                   // host destination(s): decode into a device scratch, copy out
        CK(cudaMalloc(&tmp, total * (sizeof(float) + sizeof(short))));
        if (!f_dev) df = static_cast<float*>(tmp);
        if (!s_dev) ds = reinterpret_cast<short*>(static_cast<char*>(tmp) + total * sizeof(float));
    }
    cudaError_t ce = cudaSuccess;
    for_slots(e, offset, size, [&](int slot, int done, int m) {       // windowed: split at the window edge
        if (ce == cudaSuccess) ce = wn_mulaw_decode(e->yOut, e->N, slot, m, e->B, A, e->lut_f, lut_s, df ? df + done : nullptr, ds ? ds + done : nullptr, (size_t)size, st);
        return 0;
    });
    if (ce == cudaSuccess && !f_dev) ce = cudaMemcpyAsync(audio_f32, df, total * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess && !s_dev) ce = cudaMemcpyAsync(audio_i16, ds, total * sizeof(short), cudaMemcpyDeviceToHost, st);
    if (tmp) {
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        cudaFree(tmp);
    }
    if (ce != cudaSuccess) return fail((int)ce, std::string("nvwn_get_audio: ") + cudaGetErrorString(ce));
    return 0;
}

// debug only (not part of the public ABI): the engine's conditioning store for samples [first_sample, first_sample + num_samples),
// converted back to fp32 [num_samples][L][B][2R] whatever the kernel-native layout (plain / tiled fp16 / fragment order) is
int nvwn_debug_get_conditioning(nvwn_engine* e, float* out, int first_sample, int num_samples)
{
    if (!e || !out) return fail(NVWN_EINVAL, "nvwn_debug_get_conditioning: NULL argument");
    if (first_sample < 0 || num_samples < 0 || first_sample + num_samples > e->N) return fail(NVWN_EINVAL, "nvwn_debug_get_conditioning: range out of bounds");
    const size_t per = (size_t)e->L * e->B * 2 * e->R, n = per * num_samples;
    if (n == 0) return 0;
    float* tmp = nullptr;
    CK(cudaMalloc((void**)&tmp, n * sizeof(float)));
    cudaError_t ce;
    if (e->lat_mode) ce = wn_lat_cond_readback(tmp, e->Lh, first_sample, num_samples, e->L, e->B, 0);
    else if (e->tc_mode) ce = wn_tc_cond_readback(tmp, e->Lh, first_sample, num_samples, e->tc_tile, e->L, e->B, 0);
    else if (e->dtype == NVWN_FP16) ce = wn_f16_to_f32(tmp, static_cast<const __half*>(e->Lh) + (size_t)first_sample * per, n, 0);
    else ce = cudaMemcpyAsync(tmp, static_cast<const float*>(e->Lh) + (size_t)first_sample * per, n * sizeof(float), cudaMemcpyDeviceToDevice, 0);
    if (ce == cudaSuccess) ce = cudaMemcpy(out, tmp, n * sizeof(float), cudaMemcpyDefault);
    cudaFree(tmp);
    if (ce != cudaSuccess) return fail((int)ce, std::string("nvwn_debug_get_conditioning: ") + cudaGetErrorString(ce));
    return 0;
}

// debug only (not part of the public ABI): record a clock64 timeline of sample `t` of block 0 into `out` (3 x 1024 words)
int nvwn_debug_trace(nvwn_engine* e, int t, unsigned long long* out_host, int fetch)
{
    if (!e) return NVWN_EINVAL;
    if (!fetch) {
        if (!e->trace) CK(cudaMalloc((void**)&e->trace, 3 * 1024 * sizeof(unsigned long long)));
        CK(cudaMemset(e->trace, 0, 3 * 1024 * sizeof(unsigned long long)));
        e->trace_t = t;
        return 0;
    }
    CK(cudaMemcpy(out_host, e->trace, 3 * 1024 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

// debug only: how many three-CTA clusters of the latency kernel the device runs at once (batches up to 16 x this use it)
int nvwn_debug_lat_max_clusters(int S) { return wn_lat_max_clusters(S); }

int nvwn_get_launch_info(nvwn_engine* e, nvwn_launch_info* info)
{
    if (!e || !info) return fail(NVWN_EINVAL, "nvwn_get_launch_info: NULL argument");
    info->kernel = e->last.kernel; info->grid = e->last.grid; info->block = e->last.block;
    info->smem_bytes = e->last.smem_bytes; info->batch_per_cta = e->last.batch_per_cta; info->cluster = e->last.cluster;
    info->launches = e->launches;
    const unsigned long long R = e->R, S = e->S, A = e->A, L = e->L;
    info->weight_bytes = e->td * (L * (2 * 2 * R * R + R * R + S * R + 3 * R + S) + A * S + A * A + 2 * A);
    return 0;
}

}  // extern "C"
