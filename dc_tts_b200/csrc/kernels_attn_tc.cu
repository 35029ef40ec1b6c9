// kernels_attn_tc.cu -- the dot-product attention (reference networks.py:126-155) as ONE
// tcgen05 kernel: S = Q K^T / sqrt(d) -> window mask -> softmax -> argmax -> A V -> [A V ; Q],
// alignments written transposed.  One CTA per (128 query rows, utterance).  The kernel is
// instantiated for NP padded keys, NP = max(192, round_up(N, 64)) <= 512 (keys >= N are
// zero-filled by TMA and masked).
//
//   GEMM 1  S[128 x NP]  = Q[128 x 256] . K^T        in chunks of up to 256 keys (one MMA's N),
//           chunk c into tensor-memory columns [256 c, ...)
//   softmax in the epilogue warps, one query row per thread, straight out of tensor memory;
//           the probabilities are written back to shared memory as split-fp16 planes in the
//           128B-swizzled K-major layout the tensor core reads (no global round trip)
//   GEMM 2  C[128 x 256]  = P[128 x NP] . V          (V pre-transposed to [d][keys] planes)
// Both GEMMs use the split-fp16 three-pass scheme (hi*hi + hi*lo + lo*hi, fp32 accumulate):
// the argmax of these probabilities is fed back into the next decode step, so the scores
// need fp32-grade accuracy.
//
// Tensor memory has 512 columns.  For NP <= 256, S sits at [0, NP) and the context at
// [256, 512).  For NP > 256, S fills [0, NP); the probabilities of keys [0, 256) are drained
// to shared memory first, GEMM 2 accumulates their share of the context into the freed
// columns [0, 256), and only then are the keys [256, NP) drained into the same P planes.
// Shared memory is reused: GEMM 1's two pipeline stages (one 64-channel k-block of Q and of
// one key chunk each; 80 KB at NP = 192, 96 KB above) become the P planes of one key chunk
// (96 / 128 KB) and one 64 KB V^T stage.
#include "kernels_tc.cuh"
#include "tc_ptx.cuh"

#include <algorithm>
#include <stdexcept>
#include <string>

namespace dctts {

using namespace ptx;

constexpr int AT_THREADS = 192;
constexpr int AT_NP_MIN = 192;                    // padded key count of every N <= 192 (3 x 64)
constexpr int AT_NP_MAX = 512;
constexpr int AT_D = 256;                         // head width (hp.d)
constexpr int AT_Q_PLANE = 128 * 64 * 2;          // 16 KB: 128 query rows x 64 channels fp16
constexpr int AT_VT_PLANE = AT_D * 64 * 2;        // 32 KB: 256 channels x 64 keys
constexpr int AT_TMEM_COLS = 512;

template <int NP>
struct AtShape {
    static_assert(NP % 64 == 0 && NP >= AT_NP_MIN && NP <= AT_NP_MAX, "attention_tc: NP must be a multiple of 64 in [192, 512]");
    static constexpr int KC = NP < 256 ? NP : 256;            // keys per GEMM-1 chunk
    static constexpr int NCH = (NP + 255) / 256;              // key chunks: 1 or 2
    static constexpr int K_PLANE = KC * 64 * 2;               // 24 / 32 KB
    static constexpr int STAGE1 = 2 * AT_Q_PLANE + 2 * K_PLANE;   // 80 / 96 KB
    static constexpr int P_PLANE = (KC / 64) * AT_Q_PLANE;    // one chunk of keys: KC/64 blocks of [128 x 64]
    static constexpr int SMEM_MAIN = (2 * STAGE1 > 2 * P_PLANE + 2 * AT_VT_PLANE) ? 2 * STAGE1 : 2 * P_PLANE + 2 * AT_VT_PLANE;
    static constexpr int CTX_COL = NCH == 1 ? 256 : 0;        // tensor-memory column of the context
    static constexpr int chunk_keys(int c) { return c + 1 < NCH ? 256 : NP - 256 * c; }
};

template <int NP>
__global__ void __launch_bounds__(AT_THREADS, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap mapQ_hi, const __grid_constant__ CUtensorMap mapQ_lo,
                    const __grid_constant__ CUtensorMap mapK_hi, const __grid_constant__ CUtensorMap mapK_lo,
                    const __grid_constant__ CUtensorMap mapV_hi, const __grid_constant__ CUtensorMap mapV_lo,
                    const AttnTcArgs a) {
    using Sh = AtShape<NP>;
    extern __shared__ uint8_t at_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(at_smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Sh::SMEM_MAIN);
    uint64_t* full_bar = bars;            // [2]
    uint64_t* empty_bar = bars + 2;       // [2]
    uint64_t* s_full = bars + 4;
    uint64_t* p_full = bars + 5;          // phase c: the probabilities of key chunk c are in shared memory
    uint64_t* vt_full = bars + 6;
    uint64_t* vt_empty = bars + 7;
    uint64_t* ctx_full = bars + 8;
    uint64_t* p_empty = bars + 9;         // GEMM 2 has consumed key chunk 0's planes (NP > 256)
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 10);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.y, t0 = blockIdx.x * 128;
    const int T = a.T, N = a.N;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&mapQ_hi); prefetch_tmap(&mapQ_lo); prefetch_tmap(&mapK_hi); prefetch_tmap(&mapK_lo);
        prefetch_tmap(&mapV_hi); prefetch_tmap(&mapV_lo);
        for (int s = 0; s < 2; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(s_full, 1); mbar_init(p_full, 128); mbar_init(vt_full, 1); mbar_init(vt_empty, 1); mbar_init(ctx_full, 1);
        mbar_init(p_empty, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<AT_TMEM_COLS>(tmem_ptr_smem);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    uint8_t* p_hi = smem;                          // [KC/64][128 rows][128 B]
    uint8_t* p_lo = smem + Sh::P_PLANE;
    uint8_t* vt_st = smem + 2 * Sh::P_PLANE;       // V^T hi (32 KB) | lo (32 KB)

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (lane == 0) {
            for (int it = 0; it < (AT_D / 64) * Sh::NCH; ++it) {      // k-block major, key chunk minor
                const int kb = it / Sh::NCH, ch = it % Sh::NCH, s = it & 1;
                mbar_wait(&empty_bar[s], ((uint32_t)(it >> 1) & 1u) ^ 1u);
                mbar_expect_tx(&full_bar[s], Sh::STAGE1);
                uint8_t* st = smem + (size_t)s * Sh::STAGE1;
                tma_load_3d(&mapQ_hi, &full_bar[s], st, kb * 64, t0, b);
                tma_load_3d(&mapQ_lo, &full_bar[s], st + AT_Q_PLANE, kb * 64, t0, b);
                tma_load_3d(&mapK_hi, &full_bar[s], st + 2 * AT_Q_PLANE, kb * 64, ch * 256, b);
                tma_load_3d(&mapK_lo, &full_bar[s], st + 2 * AT_Q_PLANE + Sh::K_PLANE, kb * 64, ch * 256, b);
            }
            mbar_wait(s_full, 0);                  // GEMM 1 has consumed its stages: the memory is free
            for (int kb = 0; kb < NP / 64; ++kb) {
                mbar_wait(vt_empty, ((uint32_t)kb & 1u) ^ 1u);
                mbar_expect_tx(vt_full, 2 * AT_VT_PLANE);
                tma_load_3d(&mapV_hi, vt_full, vt_st, kb * 64, 0, b);
                tma_load_3d(&mapV_lo, vt_full, vt_st + AT_VT_PLANE, kb * 64, 0, b);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // =========================== MMA issuer ===========================
        const uint32_t idesc2 = umma_idesc_f16(128, AT_D);
        for (int it = 0; it < (AT_D / 64) * Sh::NCH; ++it) {
            const int kb = it / Sh::NCH, ch = it % Sh::NCH, s = it & 1;
            mbar_wait(&full_bar[s], (uint32_t)(it >> 1) & 1u);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t idesc1 = umma_idesc_f16(128, Sh::chunk_keys(ch));
                const uint32_t dS = tmem_base + (uint32_t)(ch * 256);
                const uint32_t st = smem_u32(smem + (size_t)s * Sh::STAGE1);
                const uint64_t dQ_hi = umma_desc_kmajor<128>(st), dQ_lo = umma_desc_kmajor<128>(st + AT_Q_PLANE);
                const uint64_t dK_hi = umma_desc_kmajor<128>(st + 2 * AT_Q_PLANE);
                const uint64_t dK_lo = umma_desc_kmajor<128>(st + 2 * AT_Q_PLANE + Sh::K_PLANE);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint64_t adv = (uint64_t)(k * 2);
                    tc_mma_f16(dS, dQ_hi + adv, dK_hi + adv, idesc1, (kb | k) != 0);
                    tc_mma_f16(dS, dQ_hi + adv, dK_lo + adv, idesc1, 1u);
                    tc_mma_f16(dS, dQ_lo + adv, dK_hi + adv, idesc1, 1u);
                }
                tc_commit(&empty_bar[s]);
                if (it == (AT_D / 64) * Sh::NCH - 1) tc_commit(s_full);
            }
            __syncwarp();
        }
        for (int ch = 0; ch < Sh::NCH; ++ch) {
            mbar_wait(p_full, (uint32_t)ch & 1u);  // this chunk's probabilities are in shared memory (async-proxy visible)
            tc_fence_after();
            const int kb0 = ch * 4, kb1 = kb0 + Sh::chunk_keys(ch) / 64;
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(vt_full, (uint32_t)kb & 1u);
                tc_fence_after();
                if (lane == 0) {
                    const uint64_t dP_hi = umma_desc_kmajor<128>(smem_u32(p_hi + (kb - kb0) * AT_Q_PLANE));
                    const uint64_t dP_lo = umma_desc_kmajor<128>(smem_u32(p_lo + (kb - kb0) * AT_Q_PLANE));
                    const uint64_t dV_hi = umma_desc_kmajor<128>(smem_u32(vt_st));
                    const uint64_t dV_lo = umma_desc_kmajor<128>(smem_u32(vt_st + AT_VT_PLANE));
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t adv = (uint64_t)(k * 2);
                        tc_mma_f16(tmem_base + Sh::CTX_COL, dP_hi + adv, dV_hi + adv, idesc2, (kb | k) != 0);
                        tc_mma_f16(tmem_base + Sh::CTX_COL, dP_hi + adv, dV_lo + adv, idesc2, 1u);
                        tc_mma_f16(tmem_base + Sh::CTX_COL, dP_lo + adv, dV_hi + adv, idesc2, 1u);
                    }
                    tc_commit(vt_empty);
                    if (kb == kb1 - 1) tc_commit(ch + 1 < Sh::NCH ? p_empty : ctx_full);
                }
                __syncwarp();
            }
        }
    } else {
        // =========================== softmax / epilogue ===========================
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int t = t0 + r;
        const bool row_ok = t < T;
        int n_lo = 0, n_hi = N;
        if (a.pma) {                               // monotonic window [p, p + win) (networks.py:141-147)
            const int p = __ldg(a.pma + b);
            n_lo = min(max(p, 0), N - 1);
            n_hi = min(n_lo + a.win_size, N);
        }
        mbar_wait(s_full, 0);
        tc_fence_after();
        // pass 1: row maximum over the live keys
        float mx = -INFINITY;
        for (int c = 0; c < NP; c += 16) {
            float v[16];
            tmem_ld16(taddr + c, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) if (c + i >= n_lo && c + i < n_hi) mx = fmaxf(mx, v[i] * a.scale);
        }
        // pass 2: normaliser
        float sum = 0.f;
        for (int c = 0; c < NP; c += 16) {
            float v[16];
            tmem_ld16(taddr + c, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) if (c + i >= n_lo && c + i < n_hi) sum += expf(v[i] * a.scale - mx);
        }
        // pass 3, one key chunk at a time: probabilities -> split planes in shared memory (swizzled), alignments, argmax
        float best = -1.f; int besti = 0;
        float* al = a.align ? a.align + (size_t)b * N * T + t : nullptr;
        for (int ch = 0; ch < Sh::NCH; ++ch) {
            if (ch > 0) mbar_wait(p_empty, (uint32_t)(ch - 1) & 1u);   // GEMM 2 is done with the previous chunk's planes
            const int c0 = ch * 256;
            for (int c = c0; c < c0 + Sh::chunk_keys(ch); c += 16) {
                float v[16];
                tmem_ld16(taddr + c, v);
                __align__(16) __half ph[16];
                __align__(16) __half pl[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int n = c + i;
                    float p = 0.f;                 // masked keys are exactly 0 in the reference (exp underflow)
                    if (n >= n_lo && n < n_hi) p = expf(v[i] * a.scale - mx) / sum;
                    if (p > best) { best = p; besti = n; }
                    ph[i] = __float2half_rn(p);
                    pl[i] = __float2half_rn(p - __half2float(ph[i]));
                    if (al && row_ok && n < N) al[(size_t)n * T] = p;
                }
                const int kb = (c - c0) >> 6, c8 = (c & 63) >> 3;      // two 16-byte chunks: c8 and c8+1
                uint8_t* rowh = p_hi + kb * AT_Q_PLANE + r * 128;
                uint8_t* rowl = p_lo + kb * AT_Q_PLANE + r * 128;
                *reinterpret_cast<uint4*>(rowh + (((c8) ^ (r & 7)) << 4)) = reinterpret_cast<const uint4*>(ph)[0];
                *reinterpret_cast<uint4*>(rowh + (((c8 + 1) ^ (r & 7)) << 4)) = reinterpret_cast<const uint4*>(ph)[1];
                *reinterpret_cast<uint4*>(rowl + (((c8) ^ (r & 7)) << 4)) = reinterpret_cast<const uint4*>(pl)[0];
                *reinterpret_cast<uint4*>(rowl + (((c8 + 1) ^ (r & 7)) << 4)) = reinterpret_cast<const uint4*>(pl)[1];
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
            tc_fence_before();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(p_full)) : "memory");
        }
        if (row_ok && a.maxatt) a.maxatt[(size_t)b * T + t] = (long long)besti;

        // context rows out of tensor memory; R = [context ; Q]
        mbar_wait(ctx_full, 0);
        tc_fence_after();
        const size_t row = (size_t)b * T + t;
        for (int c = 0; c < AT_D; c += 16) {
            float v[16];
            tmem_ld16(taddr + Sh::CTX_COL + c, v);
            if (row_ok) {
                float* ro = a.R + row * a.ldr + c;
#pragma unroll
                for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(ro + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                const float* qs = a.Q + row * a.ldq + c;
                float qv[16];
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                    const float4 x = __ldg(reinterpret_cast<const float4*>(qs + i));
                    qv[i] = x.x; qv[i + 1] = x.y; qv[i + 2] = x.z; qv[i + 3] = x.w;
                    *reinterpret_cast<float4*>(ro + AT_D + i) = x;
                }
                if (a.Rpl.hi) {
                    __align__(16) __half h[16];
                    __align__(16) __half l[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) { h[i] = __float2half_rn(v[i]); l[i] = __float2half_rn(v[i] - __half2float(h[i])); }
                    uint4* dh = reinterpret_cast<uint4*>(a.Rpl.hi + row * a.Rpl.ld + c);
                    uint4* dl = reinterpret_cast<uint4*>(a.Rpl.lo + row * a.Rpl.ld + c);
                    dh[0] = reinterpret_cast<const uint4*>(h)[0]; dh[1] = reinterpret_cast<const uint4*>(h)[1];
                    dl[0] = reinterpret_cast<const uint4*>(l)[0]; dl[1] = reinterpret_cast<const uint4*>(l)[1];
#pragma unroll
                    for (int i = 0; i < 16; ++i) { h[i] = __float2half_rn(qv[i]); l[i] = __float2half_rn(qv[i] - __half2float(h[i])); }
                    dh = reinterpret_cast<uint4*>(a.Rpl.hi + row * a.Rpl.ld + AT_D + c);
                    dl = reinterpret_cast<uint4*>(a.Rpl.lo + row * a.Rpl.ld + AT_D + c);
                    dh[0] = reinterpret_cast<const uint4*>(h)[0]; dh[1] = reinterpret_cast<const uint4*>(h)[1];
                    dl[0] = reinterpret_cast<const uint4*>(l)[0]; dl[1] = reinterpret_cast<const uint4*>(l)[1];
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<AT_TMEM_COLS>(tmem_base);
    }
}

// K (B,N,d) and V (B,N,d) fp32 (leading dimension ld) -> K planes (B,N,d) and V^T planes (B,d,NP)
__global__ void attn_kv_planes_kernel(const float* __restrict__ K, int ldk, const float* __restrict__ V, int ldv,
                                      Planes kp, Planes vtp, int B, int N, int NP, int d) {
    const long long total = (long long)B * NP * d;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % d);
        const int n = (int)((i / d) % NP);
        const int b = (int)(i / ((long long)d * NP));
        float kv = 0.f, vv = 0.f;
        if (n < N) { kv = K[((size_t)b * N + n) * ldk + c]; vv = V[((size_t)b * N + n) * ldv + c]; }
        if (n < N) {
            __half h = __float2half_rn(kv);
            kp.hi[((size_t)b * N + n) * kp.ld + c] = h;
            kp.lo[((size_t)b * N + n) * kp.ld + c] = __float2half_rn(kv - __half2float(h));
        }
        __half h = __float2half_rn(vv);
        vtp.hi[((size_t)b * d + c) * vtp.ld + n] = h;                 // keys >= N are written as zeros
        vtp.lo[((size_t)b * d + c) * vtp.ld + n] = __float2half_rn(vv - __half2float(h));
    }
}

void launch_attn_kv_planes(const float* K, int ldk, const float* V, int ldv, Planes kp, Planes vtp, int B, int N, int d,
                           cudaStream_t s) {
    const int NP = attn_tc_padded_keys(N);
    if (vtp.ld < NP) throw std::runtime_error("attn_kv_planes: V^T planes narrower than the padded key count");
    const long long total = (long long)B * NP * d;
    const int grid = (int)std::min<long long>((total + 255) / 256, 4096);
    attn_kv_planes_kernel<<<grid, 256, 0, s>>>(K, ldk, V, ldv, kp, vtp, B, N, NP, d);
}

int attn_tc_padded_keys(int N) { return std::max(AT_NP_MIN, (N + 63) / 64 * 64); }

int attn_tc_max_keys() { return AT_NP_MAX; }

template <int NP>
void launch_attention_tc_np(const Planes& Q, const Planes& K, const Planes& Vt, const AttnTcArgs& a, int B, cudaStream_t s) {
    using Sh = AtShape<NP>;
    static bool attr_set_dev[64] = {};      // per device (the attribute is per device, not per process)
    int dev = 0;
    cudaGetDevice(&dev);
    bool& attr_set = attr_set_dev[dev & 63];
    const size_t smem = Sh::SMEM_MAIN + 128 + 1024;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) throw std::runtime_error(std::string("cudaFuncSetAttribute(attention_tc): ") + cudaGetErrorString(e));
        attr_set = true;
    }
    CUtensorMap mq_h, mq_l, mk_h, mk_l, mv_h, mv_l;
    tc_make_act_map(&mq_h, Q.hi, a.d, Q.ld, a.T, B, 128, 1, 64);
    tc_make_act_map(&mq_l, Q.lo, a.d, Q.ld, a.T, B, 128, 1, 64);
    tc_make_act_map(&mk_h, K.hi, a.d, K.ld, a.N, B, Sh::KC, 1, 64);   // one key chunk per box; rows >= N out of bounds -> zeros
    tc_make_act_map(&mk_l, K.lo, a.d, K.ld, a.N, B, Sh::KC, 1, 64);
    tc_make_act_map(&mv_h, Vt.hi, NP, Vt.ld, a.d, B, AT_D, 1, 64);    // (keys, channels, batch), box {64 keys, 256 channels}
    tc_make_act_map(&mv_l, Vt.lo, NP, Vt.ld, a.d, B, AT_D, 1, 64);
    dim3 grid((a.T + 127) / 128, B);
    attention_tc_kernel<NP><<<grid, AT_THREADS, smem, s>>>(mq_h, mq_l, mk_h, mk_l, mv_h, mv_l, a);
}

void launch_attention_tc(const Planes& Q, const Planes& K, const Planes& Vt, const AttnTcArgs& a, int B, cudaStream_t s) {
    if (a.d != AT_D || a.N < 1 || a.N > AT_NP_MAX) throw std::runtime_error("attention_tc: unsupported d / N");
    const int NP = attn_tc_padded_keys(a.N);
    if (Vt.ld < NP) throw std::runtime_error("attention_tc: V^T planes narrower than the padded key count");
    switch (NP) {
        case 192: launch_attention_tc_np<192>(Q, K, Vt, a, B, s); break;
        case 256: launch_attention_tc_np<256>(Q, K, Vt, a, B, s); break;
        case 320: launch_attention_tc_np<320>(Q, K, Vt, a, B, s); break;
        case 384: launch_attention_tc_np<384>(Q, K, Vt, a, B, s); break;
        case 448: launch_attention_tc_np<448>(Q, K, Vt, a, B, s); break;
        default:  launch_attention_tc_np<512>(Q, K, Vt, a, B, s); break;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw std::runtime_error(std::string("attention_tc launch: ") + cudaGetErrorString(e));
}

}  // namespace dctts
