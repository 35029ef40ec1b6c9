// kernels_simt.cu -- fp32 CUDA-core kernels of the DC-TTS synthesis path (sm_100a).
//
// These are the exact-fp32 building blocks: an implicit-GEMM dilated/causal conv
// (reference modules.py:121-134,173-187 and the stride-2 transposed conv :232-239 as
// even/odd tap sets), the row-wise LayerNorm / highway epilogue (modules.py:135-137,
// 188-193, 241), the dot-product attention with the monotonic window
// (networks.py:140-153) and the embedding gather (modules.py:36-40).  They serve the
// small-M autoregressive decode (weight-bandwidth / latency bound) and are the
// reference the tensor-core kernels (kernels_tc.cu) are validated against.
#include "kernels.cuh"
#include <math.h>

namespace dctts {

bool& pdl_enabled() { static bool on = false; return on; }   // opt-in (dctts_set_option "pdl"): measured no gain inside CUDA graphs

__device__ __forceinline__ int win_t_end(const RowWin& w) {
    return w.jptr ? __ldg(w.jptr) : (w.L - 1);
}

// ------------------------------------------------------------------------------------
// Tiled implicit-GEMM conv: BMxBN output tile per CTA, BK-deep smem stages, register
// prefetch double buffering, TMxTN micro-tile per thread (float4 smem reads).
// ------------------------------------------------------------------------------------
template <int BM, int BN, int BK, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
conv_gemm_tiled(const ConvArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int NT = (BM / TM) * (BN / TN);
    constexpr int A_V = BM * BK / 4 / NT;      // float4 loads of A per thread per stage
    constexpr int B_V = BK * BN / 4 / NT;
    constexpr int KQ = BK / 4;
    constexpr int NQ = BN / 4;
    static_assert(A_V >= 1 && B_V >= 1, "tile too small for the thread count");
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Bs[2][BK][BN];

    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int L = a.win.L, R = a.win.R;
    const int t_end = win_t_end(a.win);
    const int Mtot = a.win.B * R;
    const bool vecA = ((a.ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.X) & 15) == 0);

    int a_b[A_V], a_t[A_V];
#pragma unroll
    for (int i = 0; i < A_V; ++i) {
        int idx = tid + i * NT;
        int m = m0 + idx / KQ;
        if (m < Mtot) {
            int b = m / R, r = m - b * R;
            a_b[i] = b;
            a_t[i] = t_end - (R - 1) + r;     // may be negative -> skipped row
        } else { a_b[i] = 0; a_t[i] = -1; }
    }

    const int KC = (a.K + BK - 1) / BK;
    const int iters = a.ntaps * KC;
    float4 ra[A_V], rb[B_V];

    auto gload = [&](int it) {
        const int tap = it / KC, k0 = (it - tap * KC) * BK;
        const float* __restrict__ W = a.taps[tap].W;
        const int shift = a.taps[tap].shift;
#pragma unroll
        for (int i = 0; i < A_V; ++i) {
            int idx = tid + i * NT;
            int k = k0 + (idx % KQ) * 4;
            int ts = a_t[i] + shift;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (a_t[i] >= 0 && ts >= 0 && ts < L && k < a.K) {
                const float* p = a.X + ((size_t)a_b[i] * L + ts) * a.ldx + k;
                if (vecA && k + 3 < a.K) {
                    v = __ldg(reinterpret_cast<const float4*>(p));
                } else {
                    v.x = __ldg(p);
                    if (k + 1 < a.K) v.y = __ldg(p + 1);
                    if (k + 2 < a.K) v.z = __ldg(p + 2);
                    if (k + 3 < a.K) v.w = __ldg(p + 3);
                }
            }
            ra[i] = v;
        }
#pragma unroll
        for (int i = 0; i < B_V; ++i) {
            int idx = tid + i * NT;
            int k = k0 + idx / NQ, n = n0 + (idx % NQ) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < a.K && n < a.ldw) v = __ldg(reinterpret_cast<const float4*>(W + (size_t)k * a.ldw + n));
            rb[i] = v;
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int i = 0; i < A_V; ++i) {
            int idx = tid + i * NT;
            int row = idx / KQ, kq = (idx % KQ) * 4;
            As[buf][kq + 0][row] = ra[i].x;
            As[buf][kq + 1][row] = ra[i].y;
            As[buf][kq + 2][row] = ra[i].z;
            As[buf][kq + 3][row] = ra[i].w;
        }
#pragma unroll
        for (int i = 0; i < B_V; ++i) {
            int idx = tid + i * NT;
            *reinterpret_cast<float4*>(&Bs[buf][idx / NQ][(idx % NQ) * 4]) = rb[i];
        }
    };

    constexpr int GM = TM / 4, GN = TN / 4;      // groups of 4 rows / cols per thread
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    gload(0);
    sstore(0);
    __syncthreads();
    for (int it = 0; it < iters; ++it) {
        const int buf = it & 1;
        if (it + 1 < iters) gload(it + 1);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float av[TM], bv[TN];
#pragma unroll
            for (int g = 0; g < GM; ++g) {
                float4 v = *reinterpret_cast<const float4*>(&As[buf][k][g * (BM / GM) + ty * 4]);
                av[g * 4 + 0] = v.x; av[g * 4 + 1] = v.y; av[g * 4 + 2] = v.z; av[g * 4 + 3] = v.w;
            }
#pragma unroll
            for (int g = 0; g < GN; ++g) {
                float4 v = *reinterpret_cast<const float4*>(&Bs[buf][k][g * (BN / GN) + tx * 4]);
                bv[g * 4 + 0] = v.x; bv[g * 4 + 1] = v.y; bv[g * 4 + 2] = v.z; bv[g * 4 + 3] = v.w;
            }
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (it + 1 < iters) {
            sstore(buf ^ 1);
            __syncthreads();
        }
    }

#pragma unroll
    for (int gi = 0; gi < GM; ++gi) {
#pragma unroll
        for (int ii = 0; ii < 4; ++ii) {
            int m = m0 + gi * (BM / GM) + ty * 4 + ii;
            if (m >= Mtot) continue;
            int b = m / R, r = m - b * R;
            int t = t_end - (R - 1) + r;
            if (t < 0) continue;
            float* yrow = a.Y + ((size_t)b * a.Lout + (size_t)t * a.ostride + a.ooff) * a.ldy;
#pragma unroll
            for (int gj = 0; gj < GN; ++gj) {
                int n = n0 + gj * (BN / GN) + tx * 4;
                if (n < a.ldw) {
                    float4 bsv = __ldg(reinterpret_cast<const float4*>(a.bias + n));
                    float4 o;
                    o.x = acc[gi * 4 + ii][gj * 4 + 0] + bsv.x;
                    o.y = acc[gi * 4 + ii][gj * 4 + 1] + bsv.y;
                    o.z = acc[gi * 4 + ii][gj * 4 + 2] + bsv.z;
                    o.w = acc[gi * 4 + ii][gj * 4 + 3] + bsv.w;
                    if (a.accumulate) {
                        const float4 prev = *reinterpret_cast<const float4*>(yrow + n);
                        o.x += prev.x; o.y += prev.y; o.z += prev.z; o.w += prev.w;
                    }
                    *reinterpret_cast<float4*>(yrow + n) = o;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------
// Skinny split-K conv-GEMM for the autoregressive decode (M = 1..256 rows in total, i.e.
// weight-bandwidth / latency bound): a CTA owns 16 rows x 64 columns x ONE 64-deep slice of
// the reduction (one tap, 64 input channels), so a 768x512 weight matrix is streamed once,
// coalesced, by 96 CTAs instead of 8.  Partial sums go to Y[ks][m][n] (compact row index
// m = b*R + r) and are reduced by the LN epilogue kernel, which needs whole rows anyway.
// ------------------------------------------------------------------------------------
__device__ void ln_row_256(const LnArgs& a, int rix, float* sm);

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// FUSED: the LayerNorm / highway epilogue runs in the same launch (one kernel boundary less per block of the
// decode step).  Every CTA of a 16-row block takes a ticket after its partial sums are visible; the LAST <= 16
// CTAs of the block in launch order are its finishers: they wait for the ticket count (they are dispatched after
// the CTAs they wait for, so the wait cannot starve them), then each normalises its share of the rows exactly
// like ln_row_cta_kernel (partials summed in ascending order).  The last finisher re-arms the counters.
template <bool FUSED>
__global__ void __launch_bounds__(256) conv_gemm_skinny(const ConvArgs a, const int chunks_per_cta,
                                                        const size_t part_stride, const LnArgs ln, int* tickets) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int BM = 16, BN = 64, BKS = 64, KG = 4, KPG = BKS / KG;
    __shared__ __align__(16) float As[BKS][BM];
    __shared__ float red[KG - 1][BM][BN];

    const int tid = threadIdx.x;
    const int c = tid % BN, kg = tid / BN;
    const int m0 = blockIdx.z * BM, n = blockIdx.x * BN + c;
    const int L = a.win.L, R = a.win.R;
    const int t_end = win_t_end(a.win);
    const int Mtot = a.win.B * R;
    const bool vecA = ((a.ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.X) & 15) == 0);
    const bool n_ok = n < a.ldw;

    // A-load role: row = tid % 16, k-quad = tid / 16
    const int lrow = tid % BM, lkq = (tid / BM) * 4;
    int lb = 0, lt = -1;
    {
        int m = m0 + lrow;
        if (m < Mtot) { lb = m / R; lt = t_end - (R - 1) + (m - lb * R); }
    }

    float acc[BM];
#pragma unroll
    for (int i = 0; i < BM; ++i) acc[i] = 0.f;

    const int KC = (a.K + BKS - 1) / BKS;
    const int nchunks = a.ntaps * KC;
    const int ch0 = blockIdx.y * chunks_per_cta;
    for (int ch = ch0; ch < min(ch0 + chunks_per_cta, nchunks); ++ch) {
        const int tap = ch / KC, k0 = (ch - tap * KC) * BKS;
        const float* __restrict__ W = a.taps[tap].W;
        const int ts = lt + a.taps[tap].shift;
        const bool row_ok = (lt >= 0 && ts >= 0 && ts < L);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        {
            int k = k0 + lkq;
            if (row_ok && k < a.K) {
                const float* p = a.X + ((size_t)lb * L + ts) * a.ldx + k;
                if (vecA && k + 3 < a.K) v = __ldg(reinterpret_cast<const float4*>(p));
                else {
                    v.x = __ldg(p);
                    if (k + 1 < a.K) v.y = __ldg(p + 1);
                    if (k + 2 < a.K) v.z = __ldg(p + 2);
                    if (k + 3 < a.K) v.w = __ldg(p + 3);
                }
            }
        }
        float w[KPG];
#pragma unroll
        for (int kk = 0; kk < KPG; ++kk) {
            int k = k0 + kg * KPG + kk;
            w[kk] = (n_ok && k < a.K) ? __ldg(W + (size_t)k * a.ldw + n) : 0.f;
        }
        __syncthreads();               // previous chunk fully consumed
        As[lkq + 0][lrow] = v.x; As[lkq + 1][lrow] = v.y;
        As[lkq + 2][lrow] = v.z; As[lkq + 3][lrow] = v.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < KPG; ++kk) {
            const float4* xr = reinterpret_cast<const float4*>(&As[kg * KPG + kk][0]);
            float4 x0 = xr[0], x1 = xr[1], x2 = xr[2], x3 = xr[3];
            float ww = w[kk];
            acc[0] = fmaf(x0.x, ww, acc[0]);   acc[1] = fmaf(x0.y, ww, acc[1]);
            acc[2] = fmaf(x0.z, ww, acc[2]);   acc[3] = fmaf(x0.w, ww, acc[3]);
            acc[4] = fmaf(x1.x, ww, acc[4]);   acc[5] = fmaf(x1.y, ww, acc[5]);
            acc[6] = fmaf(x1.z, ww, acc[6]);   acc[7] = fmaf(x1.w, ww, acc[7]);
            acc[8] = fmaf(x2.x, ww, acc[8]);   acc[9] = fmaf(x2.y, ww, acc[9]);
            acc[10] = fmaf(x2.z, ww, acc[10]); acc[11] = fmaf(x2.w, ww, acc[11]);
            acc[12] = fmaf(x3.x, ww, acc[12]); acc[13] = fmaf(x3.y, ww, acc[13]);
            acc[14] = fmaf(x3.z, ww, acc[14]); acc[15] = fmaf(x3.w, ww, acc[15]);
        }
    }
    if (kg > 0) {
#pragma unroll
        for (int i = 0; i < BM; ++i) red[kg - 1][i][c] = acc[i];
    }
    __syncthreads();
    if (kg == 0 && n_ok) {
        const float bsv = (blockIdx.y == 0) ? __ldg(a.bias + n) : 0.f;
        float* yp = a.Y + (size_t)blockIdx.y * part_stride;
#pragma unroll
        for (int i = 0; i < BM; ++i) {
            int m = m0 + i;
            if (m >= Mtot) break;
            float s = acc[i] + red[0][i][c] + red[1][i][c] + red[2][i][c] + bsv;
            yp[((size_t)m * a.ostride + a.ooff) * a.ldy + n] = s;
        }
    }
    if constexpr (FUSED) {
        __threadfence();                                   // partial sums visible device-wide before the ticket
        __syncthreads();
        const int tot = gridDim.x * gridDim.y, lin = blockIdx.y * gridDim.x + blockIdx.x;
        const int nfin = min(16, tot), f = lin - (tot - nfin);
        int* cnt = tickets + 2 * blockIdx.z;
        if (tid == 0) atomicAdd(cnt, 1);
        if (f < 0) return;
        if (tid == 0) {
            const long long t0 = clock64();
            while (ld_acquire_gpu(cnt) < tot)
                if (clock64() - t0 > 4000000000LL) __trap();   // ~2 s: fail loudly instead of hanging the device
        }
        __syncthreads();
        float* sm = &red[0][0][0];
        for (int i = f; i < BM; i += nfin) {
            const int m = m0 + i;
            if (m >= Mtot) break;
            ln_row_256(ln, m, sm);
        }
        if (tid == 0) {
            const int old = atomicAdd(cnt + 1, 1);
            if (old == nfin - 1) { cnt[1] = 0; __threadfence(); atomicExch(cnt, 0); }
        }
    }
}

GemmOut launch_conv_gemm(const ConvArgs& a, cudaStream_t s, size_t scratch_bytes, bool allow_skinny) {
    GemmOut out{1, 0, 0};
    const int M = a.win.B * a.win.R;
    if (M <= 0) return out;
    const int tiles128 = ((M + 127) / 128) * ((a.ldw + 127) / 128);
    if (M <= 256 && allow_skinny) {
        const size_t part = (size_t)M * a.ostride * a.ldy;            // floats per partial
        const int nchunks = a.ntaps * ((a.K + 63) / 64);
        int max_parts = (int)(scratch_bytes / sizeof(float) / (part ? part : 1));
        if (max_parts < 1) max_parts = 1;
        if (max_parts > 64) max_parts = 64;
        const int cpc = (nchunks + max_parts - 1) / max_parts;
        const int nparts = (nchunks + cpc - 1) / cpc;
        dim3 grid((a.ldw + 63) / 64, nparts, (M + 15) / 16);
        launch_kernel(conv_gemm_skinny<false>, grid, dim3(256), 0, s, a, cpc, part, LnArgs{}, (int*)nullptr);
        out.nparts = nparts; out.compact = 1; out.part_stride = part;
    } else if (tiles128 >= 120) {
        dim3 grid((a.ldw + 127) / 128, (M + 127) / 128);
        launch_kernel(conv_gemm_tiled<128, 128, 16, 8, 8>, grid, dim3(256), 0, s, a);
    } else {
        dim3 grid((a.ldw + 63) / 64, (M + 63) / 64);
        launch_kernel(conv_gemm_tiled<64, 64, 16, 4, 4>, grid, dim3(256), 0, s, a);
    }
    return out;
}

// Decode-step blocks (M <= 256 rows, C <= 256): split-K GEMM and LN epilogue in one launch.
bool conv_gemm_ln_fusable(const ConvArgs& a, const LnArgs& n) {
    const int M = a.win.B * a.win.R;
    return M > 0 && M <= 256 && n.C <= 256 && a.ostride == 1 && a.ooff == 0 && n.out != a.X && n.out2 != a.X;
}

void launch_conv_gemm_ln(const ConvArgs& a, LnArgs n, int* tickets, cudaStream_t s, size_t scratch_bytes) {
    const int M = a.win.B * a.win.R;
    const size_t part = (size_t)M * a.ldy;
    const int nchunks = a.ntaps * ((a.K + 63) / 64);
    int max_parts = (int)(scratch_bytes / sizeof(float) / (part ? part : 1));
    if (max_parts < 1) max_parts = 1;
    if (max_parts > 64) max_parts = 64;
    const int cpc = (nchunks + max_parts - 1) / max_parts;
    const int nparts = (nchunks + cpc - 1) / cpc;
    n.Y = a.Y; n.ldy = a.ldy; n.nparts = nparts; n.compact = 1; n.part_stride = part;
    dim3 grid((a.ldw + 63) / 64, nparts, (M + 15) / 16);
    launch_kernel(conv_gemm_skinny<true>, grid, dim3(256), 0, s, a, cpc, part, n, tickets);
}

// ------------------------------------------------------------------------------------
// Row-wise LayerNorm / highway epilogue: one warp per output row, values in registers,
// two-pass mean/variance (biased, eps 1e-12: tf.contrib.layers.layer_norm).
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

template <int MAXV>
__device__ __forceinline__ void ln_stats(const float (&v)[MAXV], int C, int lane, float& mean, float& inv) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) if (lane + 32 * i < C) s += v[i];
    mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) if (lane + 32 * i < C) { float d = v[i] - mean; q = fmaf(d, d, q); }
    float var = warp_sum(q) / (float)C;
    inv = 1.0f / sqrtf(var + 1e-12f);
}

// v[i] = sum_p y[p*stride + off + lane + 32 i]: the split-K partials of the skinny GEMM, summed
// in ascending p (deterministic).  Loads are issued G partials at a time so that their
// latencies overlap instead of forming a chain of nparts dependent round trips.
template <int MAXV>
__device__ __forceinline__ void ln_load_partials(const float* __restrict__ y, int off, int C, int lane, int nparts,
                                                 size_t stride, float (&v)[MAXV]) {
    constexpr int G = MAXV <= 8 ? 4 : (MAXV <= 16 ? 2 : 1);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) v[i] = 0.f;
#pragma unroll 1
    for (int p = 0; p < nparts; p += G) {
        float t[G][MAXV];
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                int c = lane + 32 * i;
                t[g][i] = (c < C && p + g < nparts) ? y[(size_t)(p + g) * stride + off + c] : 0.f;
            }
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
            for (int i = 0; i < MAXV; ++i) v[i] += t[g][i];
    }
}

template <int MAXV>
__global__ void __launch_bounds__(256) ln_rows_kernel(const LnArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int R = a.win.R, L = a.win.L;
    if (warp >= a.win.B * R) return;
    const int t_end = win_t_end(a.win);
    const int b = warp / R, r = warp - b * R;
    const int t = t_end - (R - 1) + r;
    if (t < 0) return;
    const size_t row = (size_t)b * L + t;
    // pre-LN rows: indexed like the output rows, or compactly by (b, r) with split-K partials
    const float* y = a.Y + (a.compact ? (size_t)warp : row) * a.ldy;
    const int C = a.C;

    float v1[MAXV];
    ln_load_partials<MAXV>(y, 0, C, lane, a.nparts, a.part_stride, v1);
    float mean1, inv1;
    ln_stats<MAXV>(v1, C, lane, mean1, inv1);

    if (a.mode == 0) {
        float* o = a.out + row * a.ldo;
        float* o2 = a.out2 ? a.out2 + row * a.ldo2 : nullptr;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            int c = lane + 32 * i;
            if (c < C) {
                float z = (v1[i] - mean1) * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c);
                if (a.act == 1) z = fmaxf(z, 0.f);
                o[c] = z * keep_mul((uint32_t)(row * C + c), a.drop);
                if (o2) o2[c] = sigmoidf_acc(z);
            }
        }
    } else {
        float v2[MAXV];
        ln_load_partials<MAXV>(y, C, C, lane, a.nparts, a.part_stride, v2);
        float mean2, inv2;
        ln_stats<MAXV>(v2, C, lane, mean2, inv2);
        const float* x = a.X + row * a.ldx;
        float* o = a.out + row * a.ldo;
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            int c = lane + 32 * i;
            if (c < C) {
                float h1 = sigmoidf_acc((v1[i] - mean1) * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c));
                float h2 = (v2[i] - mean2) * inv2 * __ldg(a.g2 + c) + __ldg(a.b2 + c);
                o[c] = (h1 * h2 + (1.0f - h1) * x[c]) * keep_mul((uint32_t)(row * C + c), a.drop);
            }
        }
    }
}

// Few rows (the decode step): one CTA of 128 threads per row, every thread owns <= 2 channels of
// each half, so all split-K partial loads of the row are in flight at once (a single warp per row
// needs nparts x C / 32 loads per lane in several dependent rounds -- it was the longest kernel of
// the step).  Statistics by two block reductions (mean, then centred second moment).
__device__ __forceinline__ float block_sum_128(float v, float* sm, int warp, int lane) {
    v = warp_sum(v);
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    const float t = sm[0] + sm[1] + sm[2] + sm[3];
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(128) ln_row_cta_kernel(const LnArgs a) {
    __shared__ float sm[4];
    pdl_launch_dependents();
    pdl_wait();
    const int R = a.win.R, L = a.win.L;
    const int rix = blockIdx.x;                                  // b * R + r
    const int t_end = win_t_end(a.win);
    const int b = rix / R, r = rix - b * R;
    const int t = t_end - (R - 1) + r;
    if (t < 0) return;                                           // whole CTA leaves together
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t row = (size_t)b * L + t;
    const float* y = a.Y + (a.compact ? (size_t)rix : row) * a.ldy;
    const int C = a.C;                                           // <= 256 on this path
    const int c0 = tid, c1 = tid + 128;
    const bool ok0 = c0 < C, ok1 = c1 < C;
    float v0 = 0.f, v1 = 0.f, w0 = 0.f, w1 = 0.f;                // first half (2 channels), second half (hc)
#pragma unroll 4
    for (int p = 0; p < a.nparts; ++p) {
        const float* yp = y + (size_t)p * a.part_stride;
        if (ok0) v0 += yp[c0];
        if (ok1) v1 += yp[c1];
        if (a.mode == 1) { if (ok0) w0 += yp[C + c0]; if (ok1) w1 += yp[C + c1]; }
    }
    const float fC = (float)C;      // divide, never multiply by 1/C: with eps = 1e-12 a constant row must give d == 0 exactly
    const float mean1 = block_sum_128((ok0 ? v0 : 0.f) + (ok1 ? v1 : 0.f), sm, warp, lane) / fC;
    float d0 = ok0 ? v0 - mean1 : 0.f, d1 = ok1 ? v1 - mean1 : 0.f;
    const float inv1 = 1.0f / sqrtf(block_sum_128(d0 * d0 + d1 * d1, sm, warp, lane) / fC + 1e-12f);
    if (a.mode == 0) {
        float* o = a.out + row * a.ldo;
        float* o2 = a.out2 ? a.out2 + row * a.ldo2 : nullptr;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int c = u ? c1 : c0;
            if (c < C) {
                float z = (u ? d1 : d0) * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c);
                if (a.act == 1) z = fmaxf(z, 0.f);
                o[c] = z * keep_mul((uint32_t)(row * C + c), a.drop);
                if (o2) o2[c] = sigmoidf_acc(z);
            }
        }
    } else {
        const float mean2 = block_sum_128((ok0 ? w0 : 0.f) + (ok1 ? w1 : 0.f), sm, warp, lane) / fC;
        float e0 = ok0 ? w0 - mean2 : 0.f, e1 = ok1 ? w1 - mean2 : 0.f;
        const float inv2 = 1.0f / sqrtf(block_sum_128(e0 * e0 + e1 * e1, sm, warp, lane) / fC + 1e-12f);
        const float* x = a.X + row * a.ldx;
        float* o = a.out + row * a.ldo;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int c = u ? c1 : c0;
            if (c < C) {
                const float h1 = sigmoidf_acc((u ? d1 : d0) * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c));
                const float h2 = (u ? e1 : e0) * inv2 * __ldg(a.g2 + c) + __ldg(a.b2 + c);
                o[c] = h1 * h2 + (1.0f - h1) * x[c];
            }
        }
    }
}

// The same epilogue for one row by a 256-thread CTA (the fused tail of conv_gemm_skinny<true>): one channel of
// each half per thread, partials read through L2 (they were written by other SMs in this launch).
__device__ __forceinline__ float block_sum_256(float v, float* sm, int warp, int lane) {
    v = warp_sum(v);
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    const float t = ((sm[0] + sm[1]) + (sm[2] + sm[3])) + ((sm[4] + sm[5]) + (sm[6] + sm[7]));
    __syncthreads();
    return t;
}

__device__ void ln_row_256(const LnArgs& a, int rix, float* sm) {
    const int R = a.win.R, L = a.win.L;
    const int t_end = win_t_end(a.win);
    const int b = rix / R, r = rix - b * R;
    const int t = t_end - (R - 1) + r;
    if (t < 0) return;                                           // uniform over the CTA
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t row = (size_t)b * L + t;
    const float* y = a.Y + (a.compact ? (size_t)rix : row) * a.ldy;
    const int C = a.C, c = tid;
    const bool ok = c < C;
    float v = 0.f, w = 0.f;
#pragma unroll 4
    for (int p = 0; p < a.nparts; ++p) {
        const float* yp = y + (size_t)p * a.part_stride;
        if (ok) { v += __ldcg(yp + c); if (a.mode == 1) w += __ldcg(yp + C + c); }
    }
    const float fC = (float)C;
    const float mean1 = block_sum_256(ok ? v : 0.f, sm, warp, lane) / fC;
    const float d = ok ? v - mean1 : 0.f;
    const float inv1 = 1.0f / sqrtf(block_sum_256(d * d, sm, warp, lane) / fC + 1e-12f);
    if (a.mode == 0) {
        if (ok) {
            float z = d * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c);
            if (a.act == 1) z = fmaxf(z, 0.f);
            a.out[row * a.ldo + c] = z;
            if (a.out2) a.out2[row * a.ldo2 + c] = sigmoidf_acc(z);
        }
    } else {
        const float mean2 = block_sum_256(ok ? w : 0.f, sm, warp, lane) / fC;
        const float e = ok ? w - mean2 : 0.f;
        const float inv2 = 1.0f / sqrtf(block_sum_256(e * e, sm, warp, lane) / fC + 1e-12f);
        if (ok) {
            const float h1 = sigmoidf_acc(d * inv1 * __ldg(a.g1 + c) + __ldg(a.b1 + c));
            const float h2 = e * inv2 * __ldg(a.g2 + c) + __ldg(a.b2 + c);
            a.out[row * a.ldo + c] = h1 * h2 + (1.0f - h1) * a.X[row * a.ldx + c];
        }
    }
}

void launch_ln_rows(const LnArgs& a, cudaStream_t s) {
    const int rows = a.win.B * a.win.R;
    if (rows <= 0) return;
    if (a.C <= 256 && rows <= 1024 && a.drop.thresh == 0u) {   // the decode step's blocks (no dropout there: only ln_rows_kernel applies the training mask)
        launch_kernel(ln_row_cta_kernel, dim3(rows), dim3(128), 0, s, a);
        return;
    }
    const int warps_per_cta = rows >= 2048 ? 8 : 2;     // small launches: spread over SMs
    const int threads = warps_per_cta * 32;
    const int grid = (rows + warps_per_cta - 1) / warps_per_cta;
    if (a.C <= 256)       launch_kernel(ln_rows_kernel<8>, dim3(grid), dim3(threads), 0, s, a);
    else if (a.C <= 512)  launch_kernel(ln_rows_kernel<16>, dim3(grid), dim3(threads), 0, s, a);
    else if (a.C <= 1024) launch_kernel(ln_rows_kernel<32>, dim3(grid), dim3(threads), 0, s, a);
    else                  launch_kernel(ln_rows_kernel<33>, dim3(grid), dim3(threads), 0, s, a);   // F = 1025
}

// ------------------------------------------------------------------------------------
// Attention (networks.py:140-153): one warp per query row.  With the monotonic window only
// keys p <= n < p+win are live -- every other softmax term is exactly 0 in the reference
// (mask value -2^32+1 underflows, SURVEY.md App. B) -- so only those are evaluated.
// Each warp keeps its row's scores in N floats of dynamic shared memory.
// ------------------------------------------------------------------------------------
constexpr int ATT_MAXN = 512;
constexpr int ATT_WARPS = 4;

__global__ void __launch_bounds__(ATT_WARPS * 32) attention_kernel(const AttnArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float probs[];           // [ATT_WARPS][N]
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = blockIdx.x * ATT_WARPS + wib;
    const int R = a.win.R, T = a.win.L;
    if (warp >= a.win.B * R) return;
    const int t_end = win_t_end(a.win);
    const int b = warp / R, r = warp - b * R;
    const int t = t_end - (R - 1) + r;
    if (t < 0) return;

    int n_lo = 0, n_hi = a.N;
    if (a.pma) {
        int p = __ldg(a.pma + b);
        n_lo = min(max(p, 0), a.N - 1);
        n_hi = min(n_lo + a.win_size, a.N);
        if (a.p_hist && t == t_end && lane == 0) a.p_hist[(size_t)b * T + t] = p;
    }
    const int d = a.d;                       // 256 = 32 lanes x 8
    const float* q = a.Q + ((size_t)b * T + t) * a.ldq;
    float qv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) qv[i] = (lane * 8 + i < d) ? q[lane * 8 + i] : 0.f;
    const float scale = rsqrtf((float)d);    // exact for d = 256
    float* pr = probs + (size_t)wib * a.N;

    // scores
    for (int n = n_lo; n < n_hi; ++n) {
        const float* k = a.K + ((size_t)b * a.N + n) * a.ldk;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) if (lane * 8 + i < d) s = fmaf(qv[i], __ldg(k + lane * 8 + i), s);
        s = warp_sum(s) * scale;
        if (lane == 0) pr[n - n_lo] = s;
    }
    __syncwarp();
    const int cnt = n_hi - n_lo;
    float mx = -INFINITY;
    for (int i = lane; i < cnt; i += 32) mx = fmaxf(mx, pr[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int i = lane; i < cnt; i += 32) { float e = expf(pr[i] - mx); pr[i] = e; sum += e; }
    sum = warp_sum(sum);
    __syncwarp();
    // probabilities, argmax (first index among equal maxima, like tf.argmax)
    float best = -1.f; int besti = 0x7fffffff;
    for (int i = lane; i < cnt; i += 32) {
        float p_ = pr[i] / sum;
        pr[i] = p_;
        if (p_ > best) { best = p_; besti = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ob = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
    }
    __syncwarp();
    const int amax = n_lo + besti;
    if (lane == 0) {
        if (a.maxatt) a.maxatt[(size_t)b * T + t] = (long long)amax;
        if (a.p_next && t == t_end) a.p_next[b] = amax;
    }
    // context = A . V ; R = [context ; Q]
    float ctx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) ctx[i] = 0.f;
    for (int n = n_lo; n < n_hi; ++n) {
        const float p_ = pr[n - n_lo];
        const float* v = a.V + ((size_t)b * a.N + n) * a.ldv;
#pragma unroll
        for (int i = 0; i < 8; ++i) if (lane * 8 + i < d) ctx[i] = fmaf(p_, __ldg(v + lane * 8 + i), ctx[i]);
    }
    float* ro = a.Rout + ((size_t)b * T + t) * a.ldr;
#pragma unroll
    for (int i = 0; i < 8; ++i) if (lane * 8 + i < d) { ro[lane * 8 + i] = ctx[i]; ro[d + lane * 8 + i] = qv[i]; }
    if (a.r_hi) {
        __half* rh = a.r_hi + ((size_t)b * T + t) * a.ldr_h;
        __half* rl = a.r_lo + ((size_t)b * T + t) * a.ldr_h;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (lane * 8 + i < d) {
                __half h = __float2half_rn(ctx[i]);
                rh[lane * 8 + i] = h; rl[lane * 8 + i] = __float2half_rn(ctx[i] - __half2float(h));
                h = __float2half_rn(qv[i]);
                rh[d + lane * 8 + i] = h; rl[d + lane * 8 + i] = __float2half_rn(qv[i] - __half2float(h));
            }
    }
    if (a.align) {
        for (int n = lane; n < a.N; n += 32) {
            float p_ = (n >= n_lo && n < n_hi) ? pr[n - n_lo] : 0.f;
            a.align[((size_t)b * a.N + n) * T + t] = p_;
        }
    }
}

void launch_attention(const AttnArgs& a, cudaStream_t s) {
    const int rows = a.win.B * a.win.R;
    if (rows <= 0) return;
    if (a.N < 1 || a.N > ATT_MAXN) throw std::runtime_error("attention: N must be in [1, 512]");
    launch_kernel(attention_kernel, dim3((rows + ATT_WARPS - 1) / ATT_WARPS), dim3(ATT_WARPS * 32),
                  (size_t)ATT_WARPS * a.N * sizeof(float), s, a);
}

// ------------------------------------------------------------------------------------
// Small helpers
// ------------------------------------------------------------------------------------
__global__ void embed_kernel(const int* __restrict__ ids, const float* __restrict__ table,
                             float* __restrict__ out, int rows, int e4) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * e4) return;
    int row = i / e4, c = i - row * e4;
    int id = __ldg(ids + row);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (id != 0) v = __ldg(reinterpret_cast<const float4*>(table) + (size_t)id * e4 + c);   // modules.py:36-38
    reinterpret_cast<float4*>(out)[i] = v;
}

void launch_embed(const int* ids, const float* table, float* out, int rows, int e, cudaStream_t s) {
    int n = rows * (e / 4);
    if (n <= 0) return;
    embed_kernel<<<(n + 255) / 256, 256, 0, s>>>(ids, table, out, rows, e / 4);
}

__global__ void ar_advance_kernel(int* p_cur, const int* p_next, int* j, int B) {
    pdl_launch_dependents();
    pdl_wait();
    int i = threadIdx.x + blockIdx.x * blockDim.x;
    if (i < B) p_cur[i] = p_next[i];
    if (i == 0) *j = *j + 1;
}
void launch_ar_advance(int* p_cur, const int* p_next, int* j, int B, cudaStream_t s) {
    launch_kernel(ar_advance_kernel, dim3((B + 127) / 128), dim3(128), 0, s, p_cur, p_next, j, B);
}

__global__ void fill_i32_kernel(int* p, int v, int n) {
    int i = threadIdx.x + blockIdx.x * blockDim.x;
    if (i < n) p[i] = v;
}
void launch_fill_i32(int* p, int v, int n, cudaStream_t s) {
    if (n > 0) fill_i32_kernel<<<(n + 255) / 256, 256, 0, s>>>(p, v, n);
}

}  // namespace dctts
