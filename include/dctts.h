/*
 * dctts.h -- C-ABI of the B200-native DC-TTS synthesis path (libdctts_b200.so).
 *
 * The reference (Kyubyong/dc_tts) has no FFI layer: its operator API is the set of
 * Python signatures in modules.py / networks.py and the Graph attributes fetched by
 * synthesize.py.  Each entry point below states the reference interface it replaces
 * (file:line under /root/reference).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every tensor is float32, channels-last (B, time, C), dense unless an explicit
 *     leading dimension is passed; ids are int32, argmax outputs int64 (tf.argmax);
 *   - `x`/`out` pointers are DEVICE pointers on the handle's device, except in the
 *     `*_host` entry points, which take HOST pointers and do the copies themselves;
 *   - the caller owns all tensors; the handle owns weights, workspace and CUDA graphs;
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream);
 *   - every function returns 0 on success, non-zero on failure, never throws, and
 *     never falls back to a CPU implementation; dctts_last_error() describes the
 *     most recent failure on that handle (or the global one for create failures);
 *   - a handle is bound to one device and is not thread-safe.
 */
#ifndef DCTTS_H_
#define DCTTS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dctts_handle_s* dctts_handle;

/* Model hyper-parameters the kernels specialise on: reference hyperparams.py:19,27-32,38-40,14. */
typedef struct dctts_hparams {
    int32_t vocab_size;          /* len(hp.vocab) = 32 */
    int32_t e;                   /* hp.e = 128  */
    int32_t d;                   /* hp.d = 256  */
    int32_t c;                   /* hp.c = 512  */
    int32_t n_mels;              /* hp.n_mels = 80 */
    int32_t n_fft;               /* hp.n_fft = 2048 -> F = 1 + n_fft/2 */
    int32_t max_N;               /* hp.max_N = 180; at most 512 (see "key_capacity" below) */
    int32_t max_T;               /* hp.max_T = 210 */
    int32_t attention_win_size;  /* hp.attention_win_size = 3 */
    int32_t r;                   /* hp.r = 4 (SSRN upsampling = two stride-2 deconvs) */
} dctts_hparams;

/* ---- lifetime ------------------------------------------------------------------ */
/* Replaces Graph(mode="synthesize") construction + tf.Session() (train.py:22-80, synthesize.py:26-28).
 * The handle's key capacity -- the most characters (attention keys) any of its entry points takes -- is fixed here:
 * max(192, round_up(max_N, 64)).  max_N > 512 fails with an error that names the limit. */
int dctts_create(const dctts_hparams* hp, int device, dctts_handle* out);
int dctts_destroy(dctts_handle h);
const char* dctts_last_error(dctts_handle h);      /* h may be NULL: last create() error */
const char* dctts_version(void);

/* ---- parameters ---------------------------------------------------------------- */
/* Replaces Saver.restore into TF variables (synthesize.py:31-41).  `tf_name` is the TF
 * variable name (SURVEY.md App. C), `data` a HOST float32 array of `shape[0..rank)`.
 * dctts_commit_params() packs the staged variables into the kernels' layouts and
 * uploads them; it fails if any variable of the path is missing or mis-shaped. */
int dctts_set_param(dctts_handle h, const char* tf_name, const float* data,
                    const int64_t* shape, int32_t rank);
int dctts_commit_params(dctts_handle h);
int64_t dctts_num_params(dctts_handle h);           /* committed scalar count, -1 on error */

/* ---- building blocks (reference modules.py) ------------------------------------ */
/* `scope` is the full variable scope, e.g. "Text2Mel/AudioEnc/HC_4". */

/* embed (modules.py:13-42): ids (B,N) int32 -> out (B,N,e); row 0 of the table reads as zeros. */
int dctts_embed(dctts_handle h, const char* scope, const int32_t* ids, int32_t B, int32_t N,
                float* out, void* stream);
/* normalize (modules.py:45-64): LN over the last axis with `scope`/{gamma,beta}, eps 1e-12. */
int dctts_normalize(dctts_handle h, const char* scope, const float* x, int64_t rows, int32_t C,
                    float* out, void* stream);
/* conv1d (modules.py:91-141, training=False): conv(k, rate, SAME|CAUSAL) + bias -> LN -> act.
 * k, Cin, Cout come from the committed kernel; act: 0 none, 1 relu.  x (B,L,Cin) -> out (B,L,Cout). */
int dctts_conv1d(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L,
                 int32_t rate, int32_t causal, int32_t act, float* out, void* stream);
/* hc (modules.py:143-197): conv to 2C -> split -> LN(H1),LN(H2) -> sigmoid(H1) -> H1*H2+(1-H1)*x. */
int dctts_hc(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L,
             int32_t rate, int32_t causal, float* out, void* stream);
/* conv1d_transpose (modules.py:199-247): stride-2, k=3, 'same' -> LN.  x (B,L,C) -> out (B,2L,C). */
int dctts_conv1d_transpose(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L,
                           float* out, void* stream);

/* ---- networks (reference networks.py) ------------------------------------------ */
/* TextEnc (networks.py:14-71): L (B,N) int32 -> K,V (B,N,d) each. */
int dctts_textenc(dctts_handle h, const int32_t* L, int32_t B, float* K, float* V, void* stream);
/* AudioEnc (networks.py:73-124): S (B,T,n_mels) -> Q (B,T,d). */
int dctts_audioenc(dctts_handle h, const float* S, int32_t B, int32_t T, float* Q, void* stream);
/* Attention (networks.py:126-155): Q (B,T,d), K,V (B,N,d) -> R (B,T,2d), alignments (B,N,T),
 * max_attentions (B,T) int64.  prev_max_attentions (B) int32 selects the monotonic window
 * [p, p+win) when `monotonic` != 0 (ignored otherwise, may be NULL).  alignments and
 * max_attentions may be NULL. */
int dctts_attention(dctts_handle h, const float* Q, const float* K, const float* V,
                    int32_t B, int32_t T, int32_t N, int32_t monotonic,
                    const int32_t* prev_max_attentions,
                    float* R, float* alignments, int64_t* max_attentions, void* stream);
/* AudioDec (networks.py:157-212): R (B,T,2d) -> Y_logits, Y (B,T,n_mels). Y_logits may be NULL. */
int dctts_audiodec(dctts_handle h, const float* R, int32_t B, int32_t T,
                   float* Y_logits, float* Y, void* stream);
/* SSRN (networks.py:214-292): Y (B,T,n_mels) -> Z_logits, Z (B,4T,F). Z_logits may be NULL. */
int dctts_ssrn(dctts_handle h, const float* Y, int32_t B, int32_t T,
               float* Z_logits, float* Z, void* stream);

/* ---- graph-level (reference train.py Graph, synthesize.py loop) ------------------ */
/* One sess.run of the synthesize graph (train.py:48-68 fetched at synthesize.py:48-52):
 * L (B,max_N), mels (B,max_T,n_mels), prev_max_attentions (B) ->
 * Y (B,max_T,n_mels), max_attentions (B,max_T) int64, alignments (B,max_N,max_T).
 * alignments may be NULL.  All rows are recomputed, as the reference does. */
int dctts_text2mel_forward(dctts_handle h, const int32_t* L, const float* mels,
                           const int32_t* prev_max_attentions, int32_t B,
                           float* Y, int64_t* max_attentions, float* alignments, void* stream);
/* The whole autoregressive loop of synthesize.py:45-54 on the device: TextEnc once, then
 * `steps` (<= max_T; 0 means max_T) incremental steps replayed from a CUDA graph, each
 * reproducing exactly what the reference's full-graph pass yields for row j (including
 * the re-application of step j's attention window to the 85-row AudioDec history).
 * Outputs: Y (B,max_T,n_mels); optional prev_hist (B,max_T) int32 = the
 * prev_max_attentions value used at every step; optional final max_attentions /
 * alignments as the last sess.run would return them. */
int dctts_text2mel_generate(dctts_handle h, const int32_t* L, int32_t B, int32_t steps,
                            float* Y, int32_t* prev_hist,
                            int64_t* max_attentions, float* alignments, void* stream);
/* synthesize.py:45-57 end to end with HOST buffers: copies L_host in, runs
 * dctts_text2mel_generate + dctts_ssrn, copies Y_host (B,max_T,n_mels; may be NULL) and
 * Z_host (B,4*max_T,F) out, and synchronises.  Host buffers should be pinned for speed. */
int dctts_synthesize_host(dctts_handle h, const int32_t* L_host, int32_t B,
                          float* Y_host, float* Z_host);

/* ---- vocoder ("next" row after the path: reference utils.py:67-114) --------------------- */
/* Signal-processing constants of hyperparams.py:13-24 (defaults = the LJ values: hop 275, win 1102, power 1.5,
 * max_db 100, ref_db 20, preemphasis 0.97, n_iter 50; n_fft is fixed at 2048 = 2*(F-1)). */
int dctts_set_vocoder_params(dctts_handle h, int32_t hop_length, int32_t win_length, float power, float max_db,
                             float ref_db, float preemphasis, int32_t n_iter);
/* spectrogram2wav (utils.py:67-94) for a batch, entirely on the device: mag (B, T, F) normalised linear
 * magnitudes -> de-normalise, ^power, Griffin-Lim (n_iter x istft/stft with librosa's conventions), de-pre-emphasis.
 * wav (B, hop*(T-1)) DEVICE float32 receives the UNTRIMMED waveform; trim_host (B, 2) HOST int32 receives the
 * [start, end) sample range librosa.effects.trim (top_db 60) would keep.  n_iter < 0 means the configured value.
 * Synchronises `stream` before returning (trim_host is written by the host). */
int dctts_spectrogram2wav(dctts_handle h, const float* mag, int32_t B, int32_t T, int32_t n_iter, float* wav,
                          int32_t* trim_host, void* stream);

/* Feature extraction (next row, SURVEY 8f-4): get_spectrograms -- utils.py:20-65 -- for ONE utterance from the
 * loaded waveform on: trim (librosa.effects.trim), pre-emphasis, STFT, |.|, mel filterbank
 * (librosa.filters.mel(sample_rate, n_fft, n_mels)), 20 log10, normalisation with the constants of
 * dctts_set_vocoder_params.  `wav` DEVICE float32 [n_samples]; `mel` (t_capacity, n_mels) and `mag`
 * (t_capacity, 1 + n_fft/2) DEVICE outputs, rows [0, *t_out) written, t_capacity >= 1 + n_samples / hop_length;
 * `trim_host` (optional) receives the [start, end) sample range kept.  Synchronises the stream once. */
int dctts_get_spectrograms(dctts_handle h, const float* wav, int64_t n_samples, int32_t sample_rate, float* mel, float* mag,
                           int32_t t_capacity, int32_t* t_out, int32_t* trim_host, void* stream);

/* ---- training step (BASELINE config 5; SURVEY 8f-3) --------------------------------------
 * One optimiser step of the reference's Text2Mel trainer -- graph train.py:43-68 in mode "train" (dropout after
 * every block, full softmax attention), losses train.py:83-99 (L1 + sigmoid cross-entropy on the mels + guided
 * attention), elementwise clipping to [-1, 1] and tf.train.AdamOptimizer defaults with the Noam learning rate
 * (train.py:122-132, utils.py:141-145) -- for fixed-size batches L (B, max_N) int32, mels (B, max_T, n_mels), DEVICE
 * pointers.  All tensors are float32; the three GEMMs of every block (forward conv, data gradient, weight gradient) run on
 * tcgen05 as split-fp16 x3 with per-tensor power-of-two scales (option "train_tc", default 7; 0 = the float32 CUDA-core
 * kernels).  dctts_train_init allocates the saved activations and the gradient / Adam arenas and switches the handle's
 * SYNTHESIS entry points to the fp32 kernel set (the optimiser updates the fp32 weights only, the packed planes go stale).
 * Dropout uses a stateless hash of (element, block index, seed) -- TF's random stream cannot be reproduced.
 * losses_host (optional): {total, mels L1, binary divergence, guided attention}; reading them synchronises.
 * apply = 0 leaves the gradients in the arena (dctts_train_grads: one flat device buffer, what a data-parallel job
 * all-reduces) for dctts_train_apply.  dctts_train_tensor copies a variable (what = 0), its gradient (1) or Adam
 * moments (2, 3) to the host, in the TF variable's own layout. */
int dctts_train_init(dctts_handle h, int32_t B, float dropout_rate);
int dctts_train_step(dctts_handle h, const int32_t* L, const float* mels, int32_t B, int64_t global_step, uint32_t seed, float lr,
                     int32_t apply, float* losses_host, void* stream);
int dctts_train_apply(dctts_handle h, int64_t global_step, float lr, void* stream);
/* The SSRN trainer (train.py num = 2: SSRN on the GROUND-TRUTH mels :69-72, losses :100-108, same optimiser): mels
 * (B, T, n_mels), mags (B, 4T, 1 + n_fft/2) DEVICE pointers; losses_host = {total, mags L1, binary divergence, 0}.
 * A handle trains one of the two networks at a time (the init call selects which). */
int dctts_train_init_ssrn(dctts_handle h, int32_t B, int32_t T, float dropout_rate);
int dctts_train_step_ssrn(dctts_handle h, const float* mels, const float* mags, int32_t B, int64_t global_step, uint32_t seed, float lr,
                          int32_t apply, float* losses_host, void* stream);
/* Length-bucketed batches at their own shape, as the reference trains on them (data_load.py:122-129, dynamic_pad=True):
 * Text2Mel on L (B, N) int32 / mels (B, T, n_mels), SSRN on mels (B, T, n_mels) / mags (B, 4T, 1 + n_fft/2), DEVICE
 * pointers, B as given to the init call.  TextEnc and the attention keys run over N rows, the other networks over T
 * frames; the L1 / binary-divergence losses average over the batch's own extent.  The guided-attention term covers the
 * window n < min(N, max_N), t < min(T, max_T) of the (max_N, max_T) weight table, divided by B min(N, max_N) min(T, max_T)
 * (train.py:91-95 pads A with -1 and cuts it to (max_N, max_T)).  N <= the handle's key capacity (see dctts_create), T is
 * bounded by memory only.  The activation workspace grows on demand (the device is synchronised first);
 * dctts_train_reserve pre-sizes it for steps up to (N, T) (SSRN: N is ignored).  Growth keeps the variables, gradients,
 * Adam moments and everything dctts_train_tensor reads.  At (max_N, max_T) (SSRN: the init T) the shaped steps compute
 * what dctts_train_step / dctts_train_step_ssrn compute. */
int dctts_train_step_shaped(dctts_handle h, const int32_t* L, int32_t N, const float* mels, int32_t T, int32_t B,
                            int64_t global_step, uint32_t seed, float lr, int32_t apply, float* losses_host, void* stream);
int dctts_train_step_ssrn_shaped(dctts_handle h, const float* mels, const float* mags, int32_t B, int32_t T,
                                 int64_t global_step, uint32_t seed, float lr, int32_t apply, float* losses_host, void* stream);
int dctts_train_reserve(dctts_handle h, int32_t N, int32_t T);
int dctts_train_grads(dctts_handle h, float** grads, int64_t* count);
int dctts_train_tensor(dctts_handle h, const char* tf_name, int32_t what, float* host_out, int64_t count);
/* Inverse of dctts_train_tensor for what = 0 (variable), 2 (Adam m), 3 (Adam v): restores a training state (resume). */
int dctts_train_set_tensor(dctts_handle h, const char* tf_name, int32_t what, const float* host_in, int64_t count);

/* ---- utilities ----------------------------------------------------------------- */
/* Pre-size the workspace (otherwise grown lazily on first use) for batches up to B. */
int dctts_reserve(dctts_handle h, int32_t max_batch);
/* Number of kernels this library has launched on the handle since creation (graph
 * replays count their kernel nodes). */
int64_t dctts_launch_count(dctts_handle h);
/* Host utility for the checkpoint reader (dc_tts_b200/checkpoint.py): CRC-32C (Castagnoli) of `n` bytes,
 * continuing from `crc` (0 to start) -- the checksum TF's tensor bundle stores (masked) for every index
 * block and every tensor restored at synthesize.py:31-41.  No handle, no GPU. */
uint32_t dctts_crc32c(uint32_t crc, const void* data, int64_t n);
/* Selects the kernel set: 0 = one fp32 CUDA-core GEMM + one LN kernel per block (baseline),
 * 1 = default: tcgen05 split-fp16 (3-MMA, fp32-grade) fused blocks where they apply (whole
 * networks, full-sequence attention, and the wide AudioDec rows of the graph decode step when B >= 8). */
int dctts_set_tensor_path(dctts_handle h, int32_t mode);

/* Kernel-variant switches (every value is a parity-tested code path; defaults = measured best):
 *   "decode_mode"  1 = the whole AR loop (synthesize.py:45-54) as ONE persistent cluster kernel (default),
 *                  0 = one captured CUDA graph per mel frame (round-1 path)
 *   "tc_occ2" 0/1, "tc_cg2" 0/1/2, "tc_tile_pair" 0/1, "tc_mcast" 0/1, "tc_resid_tma" 0/1: tcgen05 block kernel variants
 *   "fused_ln" 0/1: graph decode, GEMM + LN in one launch;  "tc_debug" 0/1;  "decode_prof" 0/1;  "pdl" 0/1 (process-wide)
 *   "train_tc" 0..7: training GEMMs on tcgen05, bit mask 1 forward conv (+ tcgen05 attention), 2 data gradient, 4 weight gradient
 * dctts_get_option also answers "decode_available" (1 when this handle / device can run the persistent decode),
 * "key_capacity" (the most characters any entry point of this handle takes: max(192, round_up(max_N, 64)); dctts_attention,
 * dctts_train_step_shaped and dctts_train_reserve reject a larger N) and "decode_max_clusters" (16-CTA clusters of the
 * decode kernel that are co-resident on this device; 7 on a B200). */
int dctts_set_option(dctts_handle h, const char* name, int32_t value);
int dctts_get_option(dctts_handle h, const char* name, int32_t* value);
/* Of the last dctts_text2mel_generate on the persistent decode path: frames in which a cluster had to recompute the
 * AudioDec receptive field because an attention window moved (summed over clusters), utterance-frames recomputed,
 * clusters launched.  Synchronises the device. */
int dctts_decode_stats(dctts_handle h, int32_t* moved_frames, int32_t* moved_utterance_frames, int32_t* clusters);
/* SM-clock lap timers (cycles) of the last persistent decode run with option "decode_prof" = 1: cluster 0, CTA rank 0.
 * Buckets: 0 block start, 1 weight-stream wait, 2 GEMV, 3 slot release, 4 all-gather, 5 cluster barrier, 6 LayerNorm, 7 mix,
 * 8 attention, 9 recompute attention, 10 recompute GEMM, 11 recompute LayerNorm, 12 recompute barriers, 13 frame bookkeeping. */
int dctts_decode_profile(dctts_handle h, int64_t* cycles, int32_t n);
/* Measurement aid for bench.py's roofline leg: runs the block `scope` on a synthetic
 * (B,L,Cin) input `warmup`+`iters` times and returns the mean device time of each of its
 * kernels (CUDA events on `stream` around every launch), ms_per_kernel[0..*n_kernels), <= 8. */
int dctts_bench_block(dctts_handle h, const char* scope, int32_t B, int32_t L, int32_t iters,
                      int32_t warmup, float* ms_per_kernel, int32_t* n_kernels, void* stream);
/* Raw device memory helpers so that a host without torch can drive the library. */
int dctts_malloc(dctts_handle h, void** ptr, int64_t bytes);
int dctts_free(dctts_handle h, void* ptr);
int dctts_memcpy_h2d(dctts_handle h, void* dst, const void* src, int64_t bytes, void* stream);
int dctts_memcpy_d2h(dctts_handle h, void* dst, const void* src, int64_t bytes, void* stream);
int dctts_malloc_host(dctts_handle h, void** ptr, int64_t bytes);   /* pinned */
int dctts_free_host(dctts_handle h, void* ptr);
int dctts_stream_sync(dctts_handle h, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* DCTTS_H_ */
