// kernels_tc.cuh -- interface of the tcgen05 fused conv + LayerNorm / highway kernels.
//
// Activation format on the tensor-core path ("split planes"): every fp32 activation x is
// held as two fp16 tensors hi = fp16(x), lo = fp16(x - hi) (22 significand bits together,
// 4 bytes per element like fp32).  A conv-GEMM is three tcgen05.mma passes per k-step:
// hi*Whi + hi*Wlo + lo*Whi accumulated in fp32 in TMEM -- fp32-grade results on the fp16
// tensor pipe.  Single-pass fp16/tf32 operands miss the 1e-3 parity budget (DESIGN.md).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"

namespace dctts {

struct Planes {
    __half* hi = nullptr;
    __half* lo = nullptr;
    int ld = 0;           // elements per row (multiple of 8 -> 16-byte rows for TMA)
};

struct TcArgs {
    // epilogue parameters
    const float* bias;             // [nconv] original (TF) column order
    const float* g1; const float* b1; const float* g2; const float* b2;
    int mode;                      // 0 conv1d (one LN), 1 hc (two LNs + gate + mix), 2 transposed conv (two LNs, two rows)
    int act;                       // mode 0: 0 none, 1 relu
    int C;                         // LN width (mode 0: cout; modes 1,2: cout of one half)
    int bn;                        // accumulator columns per CTA (modes 1,2: both halves)
    int half;                      // columns per LN half per CTA (mode 0: == bn)
    float inv_scale;               // 1 / (power-of-two weight scale)
    // reduction schedule
    int ntaps; int shifts[3]; int kb_per_tap; int stages;   // kb_per_tap in units of the kernel's BK (64 or 32)
    int mcast;                     // 1: the A tile is fetched once per cluster (each CTA loads 128/ncta rows, TMA multicast)
    int resid_tma;                 // 1 (hc): residual tile via TMA into a drained pipeline stage
    int out_tma;                   // 1 (hc, full sequences, needs resid_tma): output planes staged in that stage and TMA-stored
    // tiling: 128 rows = TT time rows x TB batch rows
    int TT, TB, tiles_t, ntiles;   // ntiles = batch groups x tiles_t (a CTA takes MT consecutive tiles)
    RowWin win;
    // residual (mode 1) and outputs
    Planes X;                      // highway residual, same row index as the output
    Planes out;                    // split-plane output (may be null)
    float* out_f32; int ld_f32;    // fp32 output (may be null)
    float* sig_f32; int ld_sig;    // fp32 sigmoid(output) (mode 0, may be null)
    Planes sig;                    // split planes of sigmoid(output) (mode 0, may be null)
    int* dbg;                      // optional host-mapped progress markers (debugging), else null
};

// Encodes the rank-3 (C, L, B) activation map with a {bk, TT, TB} box; bk = 64 -> 128-byte swizzle, 32 -> 64-byte.
void tc_make_act_map(CUtensorMap* m, const __half* base, int C, int ld, int L, int B, int TT, int TB, int bk);
// Encodes the rank-2 (Ktot, Nrows) K-major weight map with a {bk, bn} box, same swizzle rule.
void tc_make_w_map(CUtensorMap* m, const __half* base, int Ktot, int Nrows, int bn, int bk);

// Generic rank-3 fp16 map {d0 (contiguous), d1, d2} with byte strides and a {b0, b1, 1} box (b0 = 32 or 64 halfs).
void tc_make_map3(CUtensorMap* m, const __half* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                  uint64_t stride2_bytes, uint32_t b0, uint32_t b1);

// pipeline depth that fits the shared-memory budget for `bn` accumulator columns per CTA
int tc_stages_for(int bn, int bk, int mt);
// reduction slab per pipeline stage (fp16 elements): 64 (128B swizzle); DCTTS_TC_BK=32 selects 32 (64B swizzle, deeper pipeline)
int tc_bk();
// grid = (ncta, tiles); cluster (ncta,1,1)
void launch_conv_ln_tc(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi,
                       const CUtensorMap& w_lo, const CUtensorMap* io /* [4]: X hi, X lo, out hi, out lo ({64,128,1} boxes) or null */, const TcArgs& a, int ncta, int ctas_y, int bk, int mt, int cg, cudaStream_t s);

// ---- tcgen05 attention (kernels_attn_tc.cu) ----
struct AttnTcArgs {
    const float* Q; int ldq;       // fp32 queries (copied verbatim into R[:, d:2d])
    float* R; int ldr;             // (B,T,2d) = [A.V ; Q]
    Planes Rpl;                    // optional split-plane copy of R
    float* align;                  // (B,N,T) or nullptr
    long long* maxatt;             // (B,T) or nullptr
    const int* pma;                // (B) monotonic window start, nullptr -> dense softmax
    int T, N, d, win_size;
    float scale;                   // 1/sqrt(d)
};
// Keys the kernel pads N to: max(192, round_up(N, 64)); N <= attn_tc_max_keys() (512)
int attn_tc_padded_keys(int N);
int attn_tc_max_keys();
// K, V fp32 -> K planes (B,N,d) and transposed V planes (B,d,vtp.ld), keys in [N, attn_tc_padded_keys(N)) zero
void launch_attn_kv_planes(const float* K, int ldk, const float* V, int ldv, Planes kp, Planes vtp, int B, int N, int d,
                           cudaStream_t s);
void launch_attention_tc(const Planes& Q, const Planes& K, const Planes& Vt, const AttnTcArgs& a, int B, cudaStream_t s);

void launch_f32_to_planes(const float* x, int ldx, Planes p, long long rows, int C, cudaStream_t s);
void launch_planes_to_f32(Planes p, float* y, int ldy, long long rows, int C, cudaStream_t s);

}  // namespace dctts
