// kernels.cuh -- argument blocks and launchers shared by the kernel files and the C-ABI.
//
// Row addressing (all kernels): an activation tensor is (B, L, C) float32 channels-last
// with leading dimension ld (floats).  A launch covers, for every batch element b, the
// time rows t in [t_end-R+1, t_end] where t_end = *jptr (device int, the AR step) when
// jptr != nullptr, else L-1.  Rows with t < 0 are skipped; a conv tap whose source row
// falls outside [0, L) contributes zeros (TF zero padding, reference modules.py:121-125).
// With R == L and jptr == nullptr this is the plain full-sequence case.
#pragma once
#include <vector>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdexcept>
#include <string>
#include <utility>

namespace dctts {

// Programmatic dependent launch (PDL): every kernel of the decode step starts with
// pdl_launch_dependents(); pdl_wait(); -- the next kernel's CTAs are scheduled while this one
// runs and only its main body waits for this grid's completion and memory flush.  That hides
// the kernel-to-kernel launch gap, which is what bounds the 50-kernel autoregressive step.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool& pdl_enabled();

template <typename... Params, typename... Args>
inline void launch_kernel(void (*kern)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
    if (e != cudaSuccess) throw std::runtime_error(std::string("kernel launch failed: ") + cudaGetErrorString(e));
}

struct RowWin {
    int B;            // batch
    int L;            // time length of the tensors
    int R;            // rows per batch element covered by this launch
    const int* jptr;  // device step index (window end), or nullptr -> L-1
};

struct ConvTap {
    const float* W;   // [K][ldw] row-major (output channel contiguous), zero padded to ldw
    int shift;        // source row = t + shift
};

// Y[orow][n] = bias[n] + sum_taps sum_k X[b, t+shift, k] * W_tap[k][n]
struct ConvArgs {
    const float* X; int ldx;
    float* Y; int ldy;             // pre-LN scratch, ldy == ldw (multiple of 4)
    const float* bias;             // [ldw], zero padded
    int K, N, ldw;
    int ntaps; ConvTap taps[3];
    RowWin win;
    int Lout, ostride, ooff;       // output row = b*Lout + t*ostride + ooff
    int accumulate = 0;            // tiled kernels only: Y += result (data gradient on top of the highway path)
};

// Dropout of the training step (modules.py:139 at training=True): a stateless hash of (dense element index, block index, seed) --
// TF's random stream cannot be reproduced, so the CPU checker and the kernels share this one (mix32).
struct DropArgs { uint32_t thresh = 0, layer = 0, seed = 0; float scale = 1.f; };   // keep iff mix32(i, layer, seed) >= thresh
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t mix32(uint32_t idx, uint32_t layer, uint32_t seed) {
    uint32_t x = idx * 0x9E3779B1u;
    x ^= layer * 0x85EBCA77u + seed;
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ float keep_mul(uint32_t idx, const DropArgs& d) {
    if (d.thresh == 0u) return 1.0f;
    return mix32(idx, d.layer, d.seed) >= d.thresh ? d.scale : 0.0f;
}
#endif

// Row-wise epilogue on the pre-LN scratch.
//  mode 0 (conv1d):  o = act(LN(y[0:C]) * g1 + b1);            out = o; out2 = sigmoid(o) if out2
//  mode 1 (hc):      H1 = sigmoid(LN(y[0:C])*g1+b1); H2 = LN(y[C:2C])*g2+b2;
//                    out = H1*H2 + (1-H1)*x
struct LnArgs {
    const float* Y; int ldy;       // scratch rows indexed like the output rows
    const float* g1; const float* b1; const float* g2; const float* b2;
    const float* X; int ldx;       // highway residual (mode 1), same row index as out
    float* out; int ldo;
    float* out2; int ldo2;         // optional sigmoid copy (mode 0)
    int C; int mode; int act;      // act: 0 none, 1 relu
    RowWin win;                    // rows are output rows: L here is the OUTPUT length
    int nparts = 1;                // split-K partials to sum (skinny GEMM), else 1
    int compact = 0;               // 1: scratch rows are indexed by b*R + r instead of the output row
    size_t part_stride = 0;        // floats between consecutive partials
    DropArgs drop;                 // training forward: dropout of the block output fused into this epilogue (thresh 0 = none)
};

struct GemmOut { int nparts; int compact; size_t part_stride; };

struct AttnArgs {
    const float* Q; int ldq;       // (B,T,d)
    const float* K; int ldk;       // (B,N,d)
    const float* V; int ldv;       // (B,N,d)
    float* Rout; int ldr;          // (B,T,2d) = [A.V ; Q]
    __half* r_hi; __half* r_lo; int ldr_h;   // optional split-plane copy of R for the tensor-core AudioDec
    float* align;                  // (B,N,T) or nullptr
    long long* maxatt;             // (B,T) or nullptr
    const int* pma;                // (B) window start, nullptr -> dense softmax over all keys
    int* p_next;                   // (B) or nullptr: argmax of row t_end
    int* p_hist;                   // (B,T) or nullptr: p_hist[b][t_end] = pma[b]
    int N, d, win_size;
    RowWin win;                    // rows = query rows (L = T)
};

// Griffin-Lim vocoder (kernels_vocoder.cu; reference utils.py:67-114)
struct VocoderArgs {
    const float* mag;          // (B, T, F) normalised linear magnitudes in [0, 1]
    float* S;                  // (B, T, F) amplitude target
    float2* X;                 // (B, T, F) complex spectrum estimate
    float* frames;             // (B, T, win) windowed time-domain frames
    float* wav;                // (B, hop*(T-1)) waveform (de-pre-emphasised at the end)
    float* mse;                // (B, 1 + Ly/512) frame energies for librosa.effects.trim
    const float2* tw; const float* window; const float* wss;
    double* deemph;                // (B, chunks) float64 states of the de-pre-emphasis recurrence
    int B, T, F, win, hop, n_iter;
    float max_db, ref_db, power, preemphasis;
};
void voc_make_tables(float2* tw_dev, float* window_dev, float* wss_dev, int T, int win, int hop, cudaStream_t s);
void voc_run(const VocoderArgs& a, cudaStream_t s);
int voc_launches_per_call(int n_iter);
size_t voc_deemph_scratch_bytes(int B, int T, int hop);
// feature extraction (reference utils.py:20-65)
void feat_make_mel_basis(int sr, int n_fft, int n_mels, std::vector<float>& w, std::vector<int>& range);
void feat_frame_mse(const float* y, float* mse, int n, int nfr, cudaStream_t s);
void feat_run(const float* y, int len, float preemph, float* mag, float* mel, const float* melw, const int* melrange,
              const float2* tw, const float* window, int T, int F, int n_mels, int win, int hop, float ref_db, float max_db,
              cudaStream_t s);


// ---- training step (kernels_train.cu; reference train.py mode "train") ----
struct BlockBwdArgs {
    const float* pre; int ldy;         // pre-LN conv output (rows, nconv)
    const float* gout; int ldg;        // gradient w.r.t. the block output (rows, C), leading dimension ldg (also of gin)
    const float* X; int ldx;           // block input (highway residual), mode 1
    const float* g1; const float* b1; const float* g2; const float* b2;
    float* dy;                         // out: gradient w.r.t. the conv output (rows, nconv), leading dimension ldy
    float* gin;                        // out, mode 1: highway part of the input gradient (rows, C)
    float* dg1; float* db1; float* dg2; float* db2; float* dbias;   // accumulated (+=)
    long long rows; int C; int mode; int act;
    DropArgs drop;
};
struct WgradArgs {
    const float* X; int ldx; const float* dy; int ldy; float* dW; int ldw;
    long long rows; int L, K, N, ntaps; int shifts[3];
    int nsplit = 1, rows_per_split = 0;
};
struct AttnBwdArgs {
    const float* gR;                   // (B,T,2d) gradient of [ctx ; Q]
    const float* Q; int ldq; const float* K; const float* V; int ldkv;
    const float* align;                // (B,N,T) probabilities of the forward pass
    const float* gts;                  // (max_N, max_T) guided-attention weights, leading dimension ld_gts
    float* dS;                         // (B,T,N) scratch
    float* gQ;                         // (B,T,d)
    float* gKV;                        // (B,N,2d)
    int B, T, N, d; float att_scale;   // att_scale = 1 / (B N_w T_w)
    int ld_gts, N_w, T_w;              // guided-attention window: keys n < N_w, frames t < T_w (train.py:91-95)
};
struct AdamEntry { float* p; float* g; float* m; float* v; long long n; };
void launch_train_dropout(float* x, long long rows, int C, int ld, const DropArgs& d, cudaStream_t s);
void launch_train_loss(const float* logits, int ldl, const float* target, float* dlogits, int ldg, double* sums, long long rows, int C,
                       cudaStream_t s);
void launch_train_block_bwd(const BlockBwdArgs& a, cudaStream_t s);
void launch_conv_wgrad(WgradArgs a, cudaStream_t s);
void launch_transpose_w(const float* W, float* WT, int ntaps, int K, int N, int ldw, int Kp, cudaStream_t s);
void launch_attn_bwd(const AttnBwdArgs& a, double* sums, cudaStream_t s);
void launch_guided_attention(float* W, int N, int T, cudaStream_t s);
void launch_embed_bwd(const int* ids, const float* g, float* dtable, int rows, int e, cudaStream_t s);
void launch_adam(const AdamEntry* entries_dev, int n_entries, float lr_t, float beta1, float beta2, float eps, cudaStream_t s);

// ---- the training GEMMs on tcgen05 (kernels_gemm_tc.cu): drop-ins for launch_conv_gemm (tiled path) / launch_conv_wgrad ----
struct GemmTcWs {
    __half* a_hi = nullptr; __half* a_lo = nullptr; size_t a_elems = 0;   // operand A planes (activations / gradients, plain or transposed)
    __half* b_hi = nullptr; __half* b_lo = nullptr; size_t b_elems = 0;   // operand B planes (weights / transposed gradients)
    unsigned* slots = nullptr; int n_slots = 0; int cursor = 0;           // per-tensor abs-max slots, cleared once per step
    int probe = 0;                                                        // measurement only: fetch the operands, issue no MMA, store nothing
};
void gemm_tc_begin_step(GemmTcWs& ws, cudaStream_t s);
bool conv_gemm_tc_ok(const ConvArgs& c, const GemmTcWs& ws);
struct GemmTcSlots { unsigned* x = nullptr; unsigned* w = nullptr; };   // in: abs-max already known (same tensor converted earlier this step); out: the slots used
int launch_conv_gemm_tc(const ConvArgs& c, GemmTcWs& ws, cudaStream_t s, GemmTcSlots* io = nullptr);
bool conv_wgrad_tc_ok(const WgradArgs& w, int B, const GemmTcWs& ws);
int launch_conv_wgrad_tc(const WgradArgs& w, int B, GemmTcWs& ws, cudaStream_t s, GemmTcSlots* io = nullptr);

// scratch_bytes bounds the split-K partial buffer of the skinny path
GemmOut launch_conv_gemm(const ConvArgs& a, cudaStream_t s, size_t scratch_bytes, bool allow_skinny = true);
void launch_ln_rows(const LnArgs& a, cudaStream_t s);
bool conv_gemm_ln_fusable(const ConvArgs& a, const LnArgs& n);
void launch_conv_gemm_ln(const ConvArgs& a, LnArgs n, int* tickets, cudaStream_t s, size_t scratch_bytes);
void launch_attention(const AttnArgs& a, cudaStream_t s);
void launch_embed(const int* ids, const float* table, float* out, int rows, int e, cudaStream_t s);
// p_cur = p_next; j += 1  (end of an AR step)
void launch_ar_advance(int* p_cur, const int* p_next, int* j, int B, cudaStream_t s);
void launch_fill_i32(int* p, int v, int n, cudaStream_t s);

}  // namespace dctts
