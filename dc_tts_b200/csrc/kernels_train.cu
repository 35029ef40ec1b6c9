// kernels_train.cu -- backward pass, losses and optimiser of ONE Text2Mel training step (reference train.py:43-68
// graph in mode "train", losses :83-99, Adam + clipping :122-132; BASELINE config 5, SURVEY.md 8(f)-3).
//
// First correct path: float32 CUDA-core kernels.  The forward pass reuses the fp32 block kernels of the synthesis
// path (conv_gemm_tiled + ln_rows_kernel) with every block's pre-LN tensor kept; this file adds
//   train_dropout_kernel     tf.layers.dropout with a stateless hash mask (the CPU checker restates the same hash)
//   train_loss_kernel        L1 + sigmoid cross-entropy on the mel logits, their gradient
//   train_block_bwd_kernel   dropout / activation / highway gate / LayerNorm backward of one block, one warp per
//                            row; gamma, beta and bias gradients reduced per CTA in shared memory
//   conv_wgrad_kernel        dW[tap] += X(shifted)^T . dy      (64x64 tiles, rows split over CTAs)
//   transpose_w_kernel       W[tap][cin][n] -> W^T so that the data gradient is the forward conv kernel with
//                            negated shifts (conv_gemm_tiled, accumulate flag for the highway residual)
//   attn_bwd_q_kernel / attn_bwd_kv_kernel   softmax attention backward incl. the guided-attention term
//   embed_bwd_kernel, adam_kernel
#include "kernels.cuh"

#include <cmath>

namespace dctts {

// ------------------------------------------------------------------------------------ dropout
// mix32 / keep_mul: kernels.cuh (shared with the LayerNorm epilogue, which applies the forward mask)

// x: (rows, C) with leading dimension ld; the mask index is the DENSE element index row * C + c
__global__ void train_dropout_kernel(float* __restrict__ x, long long n, int C, int ld, DropArgs d) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long row = i / C;
    const int c = (int)(i - row * C);
    x[row * ld + c] *= keep_mul((uint32_t)i, d);
}

void launch_train_dropout(float* x, long long rows, int C, int ld, const DropArgs& d, cudaStream_t s) {
    const long long n = rows * C;
    if (d.thresh == 0u || n <= 0) return;
    train_dropout_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, n, C, ld, d);
}

// ------------------------------------------------------------------------------------ losses
// sums[0] += sum |Y - m|, sums[1] += sum BCE(logit, m); dlogits = (sign(Y-m) Y (1-Y) + (Y - m)) / n.
// logits (rows, C) with leading dimension ldl, targets dense (rows, C), dlogits (rows, C) with leading dimension ldg.
__global__ void train_loss_kernel(const float* __restrict__ logits, int ldl, const float* __restrict__ target, float* __restrict__ dlogits,
                                  int ldg, double* __restrict__ sums, long long n, int C) {
    __shared__ double red[2][8];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double l1 = 0.0, bce = 0.0;
    if (i < n) {
        const long long row = i / C;
        const int c = (int)(i - row * C);
        const float x = logits[row * ldl + c], m = target[i];
        const float y = 1.0f / (1.0f + expf(-x));
        const float d = y - m;
        l1 = fabsf(d);
        bce = fmaxf(x, 0.f) - x * m + log1pf(expf(-fabsf(x)));
        const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
        dlogits[row * ldg + c] = (sg * y * (1.0f - y) + d) / (float)n;
    }
    for (int o = 16; o > 0; o >>= 1) { l1 += __shfl_xor_sync(0xffffffffu, l1, o); bce += __shfl_xor_sync(0xffffffffu, bce, o); }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { red[0][w] = l1; red[1][w] = bce; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int k = 0; k < 8; ++k) { a += red[0][k]; b += red[1][k]; }
        atomicAdd(&sums[0], a); atomicAdd(&sums[1], b);
    }
}

void launch_train_loss(const float* logits, int ldl, const float* target, float* dlogits, int ldg, double* sums, long long rows, int C,
                       cudaStream_t s) {
    const long long n = rows * C;
    train_loss_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(logits, ldl, target, dlogits, ldg, sums, n, C);
}

// ------------------------------------------------------------------------------------ block backward
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// LayerNorm backward for one half held in registers.  yhat = (y - mean) rstd, z = yhat g + b.
//   dy = rstd (dyh - mean(dyh) - yhat mean(dyh yhat)),  dyh = dz g
template <int MAXV>
__device__ __forceinline__ void ln_bwd_half(const float (&yhat)[MAXV], const float (&dz)[MAXV], const float* __restrict__ gam,
                                            int C, int lane, float rstd, float (&dy)[MAXV]) {
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = lane + 32 * i;
        if (c < C) { const float t = dz[i] * __ldg(gam + c); dy[i] = t; s1 += t; s2 = fmaf(t, yhat[i], s2); }
        else dy[i] = 0.f;
    }
    s1 = wsum(s1) / (float)C; s2 = wsum(s2) / (float)C;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) dy[i] = rstd * (dy[i] - s1 - yhat[i] * s2);
}

template <int MAXV>
__device__ __forceinline__ void ln_fwd_half(const float* __restrict__ y, int C, int lane, float (&yhat)[MAXV], float& rstd) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) { const int c = lane + 32 * i; yhat[i] = c < C ? y[c] : 0.f; s += yhat[i]; }
    const float mean = wsum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) { const int c = lane + 32 * i; const float d = c < C ? yhat[i] - mean : 0.f; yhat[i] = d; q = fmaf(d, d, q); }
    rstd = 1.0f / sqrtf(wsum(q) / (float)C + 1e-12f);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) yhat[i] *= rstd;
}

constexpr int BWD_WARPS = 8;
constexpr int BWD_ROWS_PER_WARP = 4;

// grid: ceil(rows / 32) CTAs of 8 warps; dynamic shared memory: (4 C + nconv) floats of column accumulators
template <int MAXV>
__global__ void __launch_bounds__(BWD_WARPS * 32) train_block_bwd_kernel(const BlockBwdArgs a) {
    extern __shared__ float acc[];                 // [dg1 C][db1 C][dg2 C][db2 C][dbias nconv]
    const int C = a.C, nconv = a.mode == 1 ? 2 * C : C;
    float* dg1 = acc; float* db1 = acc + C; float* dg2 = acc + 2 * C; float* db2 = acc + 3 * C; float* dbs = acc + 4 * C;
    for (int i = threadIdx.x; i < 4 * C + nconv; i += blockDim.x) acc[i] = 0.f;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int rr = 0; rr < BWD_ROWS_PER_WARP; ++rr) {
        const long long row = ((long long)blockIdx.x * BWD_WARPS + warp) * BWD_ROWS_PER_WARP + rr;
        if (row >= a.rows) break;                                                  // warp-uniform
        const float* y = a.pre + row * a.ldy;
        const float* go = a.gout + row * a.ldg;
        float* dyo = a.dy + row * a.ldy;
        float yh1[MAXV], dz1[MAXV], dy1[MAXV];
        float r1;
        ln_fwd_half<MAXV>(y, C, lane, yh1, r1);
        if (a.mode == 0) {
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = lane + 32 * i;
                float g = 0.f;
                if (c < C) {
                    g = go[c] * keep_mul((uint32_t)(row * C + c), a.drop);
                    const float z = yh1[i] * __ldg(a.g1 + c) + __ldg(a.b1 + c);
                    if (a.act == 1 && !(z > 0.f)) g = 0.f;
                    atomicAdd(&dg1[c], g * yh1[i]); atomicAdd(&db1[c], g);
                }
                dz1[i] = g;
            }
            ln_bwd_half<MAXV>(yh1, dz1, a.g1, C, lane, r1, dy1);
#pragma unroll
            for (int i = 0; i < MAXV; ++i) { const int c = lane + 32 * i; if (c < C) { dyo[c] = dy1[i]; atomicAdd(&dbs[c], dy1[i]); } }
        } else {
            float yh2[MAXV], dz2[MAXV], dy2[MAXV];
            float r2;
            ln_fwd_half<MAXV>(y + C, C, lane, yh2, r2);
            const float* x = a.X + row * a.ldx;
            float* gi = a.gin + row * a.ldg;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = lane + 32 * i;
                float d1 = 0.f, d2 = 0.f;
                if (c < C) {
                    const float g = go[c] * keep_mul((uint32_t)(row * C + c), a.drop);
                    const float h1 = 1.0f / (1.0f + expf(-(yh1[i] * __ldg(a.g1 + c) + __ldg(a.b1 + c))));
                    const float h2 = yh2[i] * __ldg(a.g2 + c) + __ldg(a.b2 + c);
                    d1 = g * (h2 - x[c]) * h1 * (1.0f - h1);
                    d2 = g * h1;
                    gi[c] = g * (1.0f - h1);                                       // highway path; the data gradient adds to it
                    atomicAdd(&dg1[c], d1 * yh1[i]); atomicAdd(&db1[c], d1);
                    atomicAdd(&dg2[c], d2 * yh2[i]); atomicAdd(&db2[c], d2);
                }
                dz1[i] = d1; dz2[i] = d2;
            }
            ln_bwd_half<MAXV>(yh1, dz1, a.g1, C, lane, r1, dy1);
            ln_bwd_half<MAXV>(yh2, dz2, a.g2, C, lane, r2, dy2);
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = lane + 32 * i;
                if (c < C) { dyo[c] = dy1[i]; dyo[C + c] = dy2[i]; atomicAdd(&dbs[c], dy1[i]); atomicAdd(&dbs[C + c], dy2[i]); }
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        atomicAdd(a.dg1 + i, dg1[i]); atomicAdd(a.db1 + i, db1[i]);
        if (a.mode == 1) { atomicAdd(a.dg2 + i, dg2[i]); atomicAdd(a.db2 + i, db2[i]); }
    }
    for (int i = threadIdx.x; i < nconv; i += blockDim.x) atomicAdd(a.dbias + i, dbs[i]);
}

void launch_train_block_bwd(const BlockBwdArgs& a, cudaStream_t s) {
    const int rows_per_cta = BWD_WARPS * BWD_ROWS_PER_WARP;
    const unsigned grid = (unsigned)((a.rows + rows_per_cta - 1) / rows_per_cta);
    const size_t smem = (size_t)(4 * a.C + (a.mode == 1 ? 2 * a.C : a.C)) * sizeof(float);
    if (a.C <= 128)      train_block_bwd_kernel<4><<<grid, BWD_WARPS * 32, smem, s>>>(a);
    else if (a.C <= 256) train_block_bwd_kernel<8><<<grid, BWD_WARPS * 32, smem, s>>>(a);
    else if (a.C <= 512) train_block_bwd_kernel<16><<<grid, BWD_WARPS * 32, smem, s>>>(a);
    else if (a.C <= 1024) train_block_bwd_kernel<32><<<grid, BWD_WARPS * 32, smem, s>>>(a);
    else if (a.C <= 1056) train_block_bwd_kernel<33><<<grid, BWD_WARPS * 32, smem, s>>>(a);     // F = 1025
    else throw std::runtime_error("train_block_bwd: C > 1056 is not on the path");
}

// ------------------------------------------------------------------------------------ weight gradient
// dW[tap][k][n] += sum_rows X[b, t + shift, k] dy[b, t, n].  grid (ceil(N/64), ceil(K/64), ntaps * nsplit), 256 threads.
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const WgradArgs a) {
    __shared__ __align__(16) float Xs[16][64 + 4];
    __shared__ __align__(16) float Ds[16][64 + 4];
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64;
    const int tap = blockIdx.z / a.nsplit, split = blockIdx.z - tap * a.nsplit;
    const int shift = a.shifts[tap];
    const long long r_begin = (long long)split * a.rows_per_split, r_end = min((long long)a.rows, r_begin + a.rows_per_split);
    const int tx = tid & 15, ty = tid >> 4;               // 16 x 16 threads, 4 x 4 outputs each
    const int lr = tid >> 4, lq = (tid & 15) * 4;         // loader: row lr (0..15), 4 consecutive columns at lq
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (long long r0 = r_begin; r0 < r_end; r0 += 16) {
        const long long row = r0 + lr;
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f), dv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < r_end) {
            const int b = (int)(row / a.L), t = (int)(row - (long long)b * a.L), ts = t + shift;
            const int k = k0 + lq, n = n0 + lq;
            if (ts >= 0 && ts < a.L && k < a.K) {
                const float* p = a.X + ((size_t)b * a.L + ts) * a.ldx + k;
                if (k + 3 < a.K) xv = __ldg(reinterpret_cast<const float4*>(p));
                else { xv.x = p[0]; if (k + 1 < a.K) xv.y = p[1]; if (k + 2 < a.K) xv.z = p[2]; }
            }
            if (n < a.N) dv = __ldg(reinterpret_cast<const float4*>(a.dy + row * a.ldy + n));     // N, ldy multiples of 4
        }
        __syncthreads();
        *reinterpret_cast<float4*>(&Xs[lr][lq]) = xv;
        *reinterpret_cast<float4*>(&Ds[lr][lq]) = dv;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const float4 xa = *reinterpret_cast<const float4*>(&Xs[r][ty * 4]);
            const float4 db = *reinterpret_cast<const float4*>(&Ds[r][tx * 4]);
            const float av[4] = {xa.x, xa.y, xa.z, xa.w}, bv[4] = {db.x, db.y, db.z, db.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
    }
    float* W = a.dW + (size_t)tap * a.K * a.ldw;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = k0 + ty * 4 + i;
        if (k >= a.K) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < a.N) atomicAdd(W + (size_t)k * a.ldw + n, acc[i][j]);
        }
    }
}

void launch_conv_wgrad(WgradArgs a, cudaStream_t s) {
    a.nsplit = (int)std::max<long long>(1, std::min<long long>(64, a.rows / 512));
    a.rows_per_split = (int)(((a.rows + a.nsplit - 1) / a.nsplit + 15) / 16 * 16);
    dim3 grid((a.N + 63) / 64, (a.K + 63) / 64, a.ntaps * a.nsplit);
    conv_wgrad_kernel<<<grid, 256, 0, s>>>(a);
}

// W[tap][K][ldw] -> WT[tap][N][Kp]   (N rows = columns of W taken, Kp >= K the padded row length; pad columns untouched)
__global__ void transpose_w_kernel(const float* __restrict__ W, float* __restrict__ WT, int K, int N, int ldw, int Kp) {
    __shared__ float tile[32][33];
    const int tap = blockIdx.z;
    const float* w = W + (size_t)tap * K * ldw;
    float* wt = WT + (size_t)tap * N * Kp;
    const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int k = k0 + i, n = n0 + threadIdx.x;
        tile[i][threadIdx.x] = (k < K && n < N) ? w[(size_t)k * ldw + n] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int n = n0 + i, k = k0 + threadIdx.x;
        if (n < N && k < K) wt[(size_t)n * Kp + k] = tile[threadIdx.x][i];
    }
}

void launch_transpose_w(const float* W, float* WT, int ntaps, int K, int N, int ldw, int Kp, cudaStream_t s) {
    dim3 grid((N + 31) / 32, (K + 31) / 32, ntaps);
    transpose_w_kernel<<<grid, dim3(32, 8), 0, s>>>(W, WT, K, N, ldw, Kp);
}

// ------------------------------------------------------------------------------------ attention backward
// Forward (networks.py:140-153, training: no window): S = Q K^T / sqrt(d), A = softmax_n(S), ctx = A V, R = [ctx ; Q];
// loss_att = sum_window |A gts| / (B N_w T_w) (train.py:91-95: A is padded with -1 and cut to (max_N, max_T), so only
// n < N_w = min(N, max_N), t < T_w = min(T, max_T) count; gts is the (max_N, max_T) table, leading dimension ld_gts).
// One warp per query row (b, t):
//   dA[n] = dctx . V[n] + [n < N_w, t < T_w] sign(A gts) gts[n,t] / (B N_w T_w);  dS[n] = A[n] (dA[n] - sum_m A[m] dA[m])
//   dQ = dR[d:2d] + sum_n dS[n] K[n] / sqrt(d);  dS is kept (B,T,N) for the key-side kernel.
// d = 256 = 32 lanes x 8; each warp keeps dA in N floats of dynamic shared memory.
constexpr int ATT_BWD_MAXN = 512;
__global__ void __launch_bounds__(128) attn_bwd_q_kernel(const AttnBwdArgs a) {
    extern __shared__ float sdA[];              // [4][N]
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + wib;
    if (row >= a.B * a.T) return;
    const int b = row / a.T, t = row - b * a.T;
    const float* gR = a.gR + (size_t)row * 2 * a.d;
    float dctx[8], dq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { dctx[i] = gR[lane * 8 + i]; dq[i] = gR[a.d + lane * 8 + i]; }
    float* da = sdA + (size_t)wib * a.N;
    float dot = 0.f;
    for (int n = 0; n < a.N; ++n) {
        const float* v = a.V + ((size_t)b * a.N + n) * a.ldkv;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s = fmaf(dctx[i], __ldg(v + lane * 8 + i), s);
        s = wsum(s);
        const float p = a.align[((size_t)b * a.N + n) * a.T + t];
        if (n < a.N_w && t < a.T_w) {
            const float g = a.gts[(size_t)n * a.ld_gts + t];
            const float pg = p * g;
            s += (pg > 0.f ? g : (pg < 0.f ? -g : 0.f)) * a.att_scale;
        }
        if (lane == 0) da[n] = s;
        dot = fmaf(p, s, dot);
    }
    __syncwarp();
    const float scale = rsqrtf((float)a.d);
    for (int n = 0; n < a.N; ++n) {
        const float p = a.align[((size_t)b * a.N + n) * a.T + t];
        const float ds = p * (da[n] - dot);
        if (lane == 0) a.dS[(size_t)row * a.N + n] = ds;
        const float* k = a.K + ((size_t)b * a.N + n) * a.ldkv;
        const float c = ds * scale;
#pragma unroll
        for (int i = 0; i < 8; ++i) dq[i] = fmaf(c, __ldg(k + lane * 8 + i), dq[i]);
    }
    float* o = a.gQ + (size_t)row * a.d;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[lane * 8 + i] = dq[i];
}

// One warp per key row (b, n): dK = sum_t dS[t,n] Q[t] / sqrt(d), dV = sum_t A[n,t] dctx[t]; gKV (B,N,2d) = [dK ; dV]
__global__ void __launch_bounds__(128) attn_bwd_kv_kernel(const AttnBwdArgs a) {
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 4 + wib;
    if (row >= a.B * a.N) return;
    const int b = row / a.N, n = row - b * a.N;
    float dk[8], dv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { dk[i] = 0.f; dv[i] = 0.f; }
    const float scale = rsqrtf((float)a.d);
    for (int t = 0; t < a.T; ++t) {
        const size_t qrow = (size_t)b * a.T + t;
        const float ds = a.dS[qrow * a.N + n] * scale;
        const float p = a.align[(size_t)row * a.T + t];
        const float* q = a.Q + qrow * a.ldq;
        const float* gc = a.gR + qrow * 2 * a.d;
#pragma unroll
        for (int i = 0; i < 8; ++i) { dk[i] = fmaf(ds, __ldg(q + lane * 8 + i), dk[i]); dv[i] = fmaf(p, __ldg(gc + lane * 8 + i), dv[i]); }
    }
    float* o = a.gKV + (size_t)row * 2 * a.d;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[lane * 8 + i] = dk[i]; o[a.d + lane * 8 + i] = dv[i]; }
}

// sums[2] += sum over the window n < N_w, t < T_w of |A gts|; align (B, N, T), gts leading dimension ld_gts
__global__ void attn_loss_kernel(const float* __restrict__ align, const float* __restrict__ gts, double* __restrict__ sums, int B, int N,
                                 int T, int ld_gts, int N_w, int T_w) {
    __shared__ double red[8];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double v = 0.0;
    if (i < (long long)B * N * T) {
        const int r = (int)(i % ((long long)N * T)), n = r / T, t = r - n * T;
        if (n < N_w && t < T_w) v = fabsf(align[i] * gts[(size_t)n * ld_gts + t]);
    }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) { double s = 0.0; for (int k = 0; k < 8; ++k) s += red[k]; atomicAdd(&sums[2], s); }
}

void launch_attn_bwd(const AttnBwdArgs& a, double* sums, cudaStream_t s) {
    if (a.d != 256 || a.N < 1 || a.N > ATT_BWD_MAXN) throw std::runtime_error("attention backward is built for d = 256, N <= 512");
    if (a.N_w > a.N || a.T_w > a.T || a.T_w > a.ld_gts) throw std::runtime_error("attention backward: guided-attention window exceeds the batch");
    const long long n = (long long)a.B * a.N * a.T;
    attn_loss_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a.align, a.gts, sums, a.B, a.N, a.T, a.ld_gts, a.N_w, a.T_w);
    attn_bwd_q_kernel<<<(a.B * a.T + 3) / 4, 128, (size_t)4 * a.N * sizeof(float), s>>>(a);
    attn_bwd_kv_kernel<<<(a.B * a.N + 3) / 4, 128, 0, s>>>(a);
}

// utils.py:134-140
__global__ void guided_attention_kernel(float* __restrict__ W, int N, int T, double g) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * T) return;
    const int n = i / T, t = i - n * T;
    const double d = (double)t / (double)T - (double)n / (double)N;
    W[i] = (float)(1.0 - exp(-(d * d) / (2.0 * g * g)));
}
void launch_guided_attention(float* W, int N, int T, cudaStream_t s) {
    guided_attention_kernel<<<(N * T + 255) / 256, 256, 0, s>>>(W, N, T, 0.2);
}

// ------------------------------------------------------------------------------------ embedding backward
// modules.py:36-40: row 0 of the table is replaced by zeros before the lookup, so it receives no gradient
__global__ void embed_bwd_kernel(const int* __restrict__ ids, const float* __restrict__ g, float* __restrict__ dtable, int rows, int e) {
    const int row = blockIdx.x, id = ids[row];
    if (id <= 0) return;
    for (int c = threadIdx.x; c < e; c += blockDim.x) atomicAdd(dtable + (size_t)id * e + c, g[(size_t)row * e + c]);
}
void launch_embed_bwd(const int* ids, const float* g, float* dtable, int rows, int e, cudaStream_t s) {
    embed_bwd_kernel<<<rows, 128, 0, s>>>(ids, g, dtable, rows, e);
}

// ------------------------------------------------------------------------------------ optimiser
// train.py:122-132: clip to [-1, 1], tf.train.AdamOptimizer (bias correction folded into lr_t by the host)
__global__ void adam_kernel(const AdamEntry* __restrict__ entries, int n_entries, float lr_t, float beta1, float beta2, float eps) {
    const AdamEntry e = entries[blockIdx.y];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < e.n; i += (long long)gridDim.x * blockDim.x) {
        const float g = fminf(fmaxf(e.g[i], -1.0f), 1.0f);
        const float m = beta1 * e.m[i] + (1.0f - beta1) * g;
        const float v = beta2 * e.v[i] + (1.0f - beta2) * g * g;
        e.m[i] = m; e.v[i] = v;
        e.p[i] -= lr_t * m / (sqrtf(v) + eps);
    }
}
void launch_adam(const AdamEntry* entries_dev, int n_entries, float lr_t, float beta1, float beta2, float eps, cudaStream_t s) {
    adam_kernel<<<dim3(64, n_entries), 256, 0, s>>>(entries_dev, n_entries, lr_t, beta1, beta2, eps);
}

}  // namespace dctts
