/*
 * nvwn_b200.h -- handle-based C-ABI of the B200 WaveNet inference engine.
 *
 * One entry point per public member of the reference's host class
 * nvWavenetInfer<T_weight,T_data,R,S,A> (nv_wavenet.cuh:220-640), so that the C++ facade
 * (include/nv_wavenet.hpp), the reference C-ABI (include/wavenet_infer.h) and any FFI
 * (ctypes, cgo, JNI ...) can drive the same engine.  Plain pointers and sizes only.
 *
 * Conventions
 *   - every function returns 0 on success, a cudaError_t (>0) or a negative NVWN_E* code on
 *     failure; nvwn_last_error() gives the message (thread-local).
 *   - every float* / int* data argument may be host or device memory (cudaMemcpyDefault),
 *     like the reference setters (nv_wavenet.cuh:285-308); data is copied before return.
 *   - matrices fp32 column-major M x K; embeddings [A][R]; Lh float[N][L][B][2R];
 *     selectors float[N][B]; yOut int[B][N]  (nv_wavenet.cuh:144, singleblock.cuh:232,245).
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).
 */
#ifndef NVWN_B200_H
#define NVWN_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nvwn_engine nvwn_engine;

enum { NVWN_FP32 = 0, NVWN_FP16 = 1,          /* T_data=float (bit-exact to the reference CPU model) / T_data=half of the reference */
       NVWN_FP32_FAST = 2 };                  /* fp32 in the reference GPU kernels' arithmetic: FMA, two interleaved partial sums per dot
                                                 product (matrix_math.cuh:80-117), float libm tanh/exp -- agrees with the CPU model like the
                                                 reference's own kernels do (nv_wavenet_test.cu:273-298), about twice as fast */
enum { NVWN_EINVAL = -1, NVWN_EUNSUPPORTED = -2, NVWN_ENOMEM = -3 };
/* kernel selection; the reference's Implementation enum values 0..4 are accepted and map to AUTO */
enum { NVWN_KERNEL_AUTO = 0, NVWN_KERNEL_STREAM = 16, NVWN_KERNEL_TENSORCORE = 17, NVWN_KERNEL_LATENCY = 18 };

/* nvWavenetInfer::nvWavenetInfer (nv_wavenet.cuh:311) */
int nvwn_create(nvwn_engine** out, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                int batch_size, int num_samples, int impl, int tanh_embed);
/* extension: a WINDOWED engine generates utterances of any length in device memory that does not depend on it.  Same dtypes,
 * shapes and kernel choice as nvwn_create; `window` (W) replaces num_samples.  Every per-sample store (conditioning, selectors,
 * yOut) holds W samples and sample t lives in slot t mod W; sample indices run from 0 to 2^31 - 1.  On a windowed engine:
 *   - nvwn_run_partial takes count <= W; num_samples (the utterance length) only bounds init_sample + count; yOut must be
 *     NULL (results are read with nvwn_get_yout / nvwn_get_audio).  A run that crosses a multiple of W is two launches.
 *   - nvwn_set_conditioning, nvwn_cond_producer_run, nvwn_set_conditioning_from_features, nvwn_set_selectors_range and
 *     nvwn_set_selectors_random_range take absolute sample ranges of at most W samples (a longer one is NVWN_EINVAL).
 *   - nvwn_get_yout / nvwn_get_audio take an absolute `offset`; the range must lie within the last W samples generated since
 *     nvwn_reset_history (else NVWN_EINVAL).
 *   - nvwn_set_inputs, nvwn_set_selectors, nvwn_set_selectors_random and nvwn_set_forced (whole-utterance operations) return
 *     NVWN_EUNSUPPORTED; there is no teacher forcing.
 * Writing samples t and t + W reuses one slot: a producer on another stream must wait (cudaStreamWaitEvent) for the run that
 * consumes t before it overwrites its slot with t + W, and a run must finish before get_yout / get_audio of its samples is
 * overtaken by the run W samples later -- the same event discipline as nvwn_cond_producer_run. */
int nvwn_create_windowed(nvwn_engine** out, int dtype, int R, int S, int A, int num_layers, int max_dilation,
                         int batch_size, int window, int impl, int tanh_embed);
/* nvWavenetInfer::~nvWavenetInfer (nv_wavenet.cuh:362-395) */
int nvwn_destroy(nvwn_engine* e);
const char* nvwn_last_error(void);

/* nv_wavenet.cuh:396-415 */
int nvwn_set_embeddings(nvwn_engine* e, const float* embedPrev, const float* embedCur);
int nvwn_set_layer_weights(nvwn_engine* e, int layer, const float* Wprev, const float* Wcur, const float* Bh,
                           const float* Wres, const float* Bres, const float* Wskip, const float* Bskip);
int nvwn_set_out_weights(nvwn_engine* e, const float* Wzs, const float* Bzs, const float* Wza, const float* Bza);
/* nv_wavenet.cuh:417-422: resets the feedback history to 128/128, copies Lh and selectors */
int nvwn_set_inputs(nvwn_engine* e, const float* Lh, const float* selectors);
/* extension: selectors only / conditioning only (conditioning may be uploaded in chunks of whole samples) */
int nvwn_set_selectors(nvwn_engine* e, const float* selectors);
int nvwn_set_conditioning(nvwn_engine* e, const float* Lh, int first_sample, int num_samples, void* stream);
/* extension (SURVEY.md 8f next-1): selectors drawn ON THE DEVICE, counter-based and stateless -- selector[i], i = sample *
 * batch_size + b, is the first output of Philox-4x32-10 with counter (i, 0) and key `seed`, as (x >> 8) * 2^-24 in [0, 1)
 * (the reference draws them on the host with libc rand(), pytorch/wavenet_infer.cu:92-93).  Asynchronous on `stream`. */
int nvwn_set_selectors_random(nvwn_engine* e, unsigned long long seed, void* stream);
/* extension, any engine: selectors of samples [first_sample, first_sample + num_samples) only -- from float[num_samples][B]
 * (host or device; a device source is read in order on `stream`), or drawn on the device with exactly the values
 * nvwn_set_selectors_random gives those samples (Philox counter sample * batch_size + b). */
int nvwn_set_selectors_range(nvwn_engine* e, const float* selectors, int first_sample, int num_samples, void* stream);
int nvwn_set_selectors_random_range(nvwn_engine* e, unsigned long long seed, int first_sample, int num_samples, void* stream);
/* host helper (needs no GPU): the selectors exactly as the reference wrapper draws them -- Matrix(batch, samples).randomize(0.5, 1.0)
 * on the caller's libc rand() stream (pytorch/wavenet_infer.cu:92-93, matrix.cpp:38-56) -- into selectors[sample * batch_size + b]. */
int nvwn_libc_selectors(float* selectors, int batch_size, int sample_count);
/* Conditioning producer on the device (SURVEY.md 8f next-2).  Replaces, for inference, WaveNet.get_cond_input
 * (pytorch/wavenet.py:190-202: ConvTranspose1d(C, C, window, stride) upsampling trimmed by window - stride, then the
 * 1x1 cond_layers convolution C -> L*2R) and the permutes to [N][L][B][2R] (pytorch/nv_wavenet.py:48-49,181):
 *   features [B][C][T] (mel frames), upsample_weight [C][C][window] (torch ConvTranspose1d layout), upsample_bias [C],
 *   cond_weight [L*2R][C] (Conv1d weight, kernel size 1), cond_bias [L*2R]; all fp32, host or device memory.
 * Produces conditioning for samples [first_sample, first_sample + T*stride) in chunks, directly in the engine's
 * conditioning store -- the [N][L][B][2R] fp32 tensor never exists.  Returns after the work has completed. */
int nvwn_set_conditioning_from_features(nvwn_engine* e, const float* features, int n_cond_channels, int num_frames,
                                        const float* upsample_weight, const float* upsample_bias, int window, int stride,
                                        const float* cond_weight, const float* cond_bias, int first_sample, void* stream);
/* The same in two steps, for producers that run concurrently with generation: _load copies the features and the two layers' weights
 * into engine-owned device memory (returns when the sources may be released); _run fills conditioning for samples
 * [sample_begin, sample_begin + sample_count) of the loaded sequence, stored from engine sample first_sample + sample_begin,
 * asynchronously on `stream` (order it before the nvwn_run_partial that consumes those samples with an event; successive _run
 * calls must be on one stream or ordered by the caller: they share scratch). */
int nvwn_cond_producer_load(nvwn_engine* e, const float* features, int n_cond_channels, int num_frames,
                            const float* upsample_weight, const float* upsample_bias, int window, int stride,
                            const float* cond_weight, const float* cond_bias, void* stream);
int nvwn_cond_producer_run(nvwn_engine* e, int first_sample, int sample_begin, int sample_count, void* stream);
/* The same arithmetic on the host (needs no GPU; test / reference use): Lh [T*stride][L][B][2R], host pointers. */
int nvwn_cond_from_features_host(float* Lh, const float* features, int batch_size, int n_cond_channels, int num_frames,
                                 const float* upsample_weight, const float* upsample_bias, int window, int stride,
                                 const float* cond_weight, const float* cond_bias, int num_layers, int R);
int nvwn_reset_history(nvwn_engine* e);
/* extension (teacher forcing): forced[b*num_samples + t] is fed back instead of the sampled index;
 * NULL switches it off.  Copied. */
int nvwn_set_forced(nvwn_engine* e, const int* forced);
/* extension: replicate rank `root`'s packed weights to every rank's engine is done by the caller
 * (NCCL broadcast of the blob below); these expose the packed device blob. */
int nvwn_weight_blob(nvwn_engine* e, void** dev_ptr, unsigned long long* bytes);
/* must be called after the blob was overwritten (e.g. by an NCCL broadcast) */
int nvwn_weights_updated(nvwn_engine* e);

/* nv_wavenet.cuh:499-639.  run_partial generates samples [init_sample, init_sample+count) of a
 * num_samples-long utterance batch; yOut (optional, host or device) receives the whole int[B][N]. */
int nvwn_run_partial(nvwn_engine* e, int init_sample, int count, int num_samples, int batch_size,
                     int* yOut, int dump_activations, void* stream);
int nvwn_run(nvwn_engine* e, int num_samples, int batch_size, int* yOut, int dump_activations, void* stream);
/* nv_wavenet.cuh:439-444: 2-D copy of yOut[b][offset .. offset+size) for every b.  On a full engine the destination is the
 * whole int[B][N] array and the samples land at column `offset` (like the reference); on a windowed engine it is int[B][size]. */
int nvwn_get_yout(nvwn_engine* e, int* yOut, int offset, int size, void* stream);
/* Output side (SURVEY.md 8f next-3): replaces the host post-processing of pytorch/nv_wavenet_inference.py:55-60 --
 * utils.mu_law_decode_numpy (pytorch/utils.py:62-70) with mu_quantization = A, then MAX_WAV_VALUE * audio and
 * astype('int16') -- on the device, straight from the engine's yOut: audio[b][j] for j in [0, size) decodes
 * yOut[b][offset + j].  audio_f32 (in [-1, 1]) and / or audio_i16 may be NULL; each is [B][size], host or device memory
 * (device destinations are filled asynchronously on `stream`).  Table-driven, the table computed on the host in double
 * exactly as numpy does, so values equal the reference's.  saturate = 0 keeps the reference's cast (code A-1 decodes to
 * +1.0 -> 32768 -> wraps to -32768), saturate = 1 clamps to 32767. */
int nvwn_get_audio(nvwn_engine* e, float* audio_f32, short* audio_i16, int offset, int size, int saturate, void* stream);
/* The decode table itself (host only, needs no GPU): entry x = decoded value of code x for mu_quantization = A; any of
 * the three outputs (A entries each) may be NULL. */
int nvwn_mulaw_table(int A, float* f32, short* i16_wrap, short* i16_saturate);

/* last-sample activations [B][dim] as fp32 (nv_wavenet.cuh:424-438); valid after a run with dump=1 */
int nvwn_get_xt_out(nvwn_engine* e, int layer, float* out);
int nvwn_get_skip_out(nvwn_engine* e, int layer, float* out);
int nvwn_get_zs(nvwn_engine* e, float* out);
int nvwn_get_za(nvwn_engine* e, float* out);
int nvwn_get_p(nvwn_engine* e, float* out);

/* introspection: what the last launch used */
typedef struct {
    int kernel;            /* NVWN_KERNEL_STREAM / NVWN_KERNEL_TENSORCORE / NVWN_KERNEL_LATENCY */
    int grid, block, smem_bytes, batch_per_cta, cluster;
    unsigned long long launches;        /* kernel launches issued by this engine so far */
    unsigned long long weight_bytes;    /* algorithmic weight+bias bytes per utterance-sample (BASELINE.md §2) */
} nvwn_launch_info;
int nvwn_get_launch_info(nvwn_engine* e, nvwn_launch_info* info);
int nvwn_device_count(void);
int nvwn_set_device(int device);

#ifdef __cplusplus
}
#endif
#endif
