// dctts_api.cu -- handle, parameter packing, network chains, AR decode engine and the
// C-ABI of include/dctts.h.
//
// Reference mapping (files under /root/reference):
//   layer tables ............ networks.py:23-68 (TextEnc), :81-124 (AudioEnc),
//                             :166-209 (AudioDec), :223-290 (SSRN)
//   block semantics ......... modules.py:91-141 (conv1d), :143-197 (hc), :199-247 (conv1d_transpose)
//   graph wiring / shift .... train.py:48-68, :74-77
//   autoregressive loop ..... synthesize.py:45-57
#include "../../include/dctts.h"
#include "kernels.cuh"
#include "kernels_tc.cuh"
#include "kernels_decode.cuh"

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

using namespace dctts;

#define CUDA_CHECK(expr)                                                                     \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            char _buf[512];                                                                  \
            snprintf(_buf, sizeof(_buf), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                                    \
            throw std::runtime_error(_buf);                                                  \
        }                                                                                    \
    } while (0)

#define REQUIRE(cond, msg)                                   \
    do {                                                     \
        if (!(cond)) throw std::runtime_error(std::string(msg)); \
    } while (0)

namespace {

std::string g_create_error;

inline int roundup(int x, int m) { return (x + m - 1) / m * m; }

enum Kind { K_C = 0, K_HC = 1, K_D = 2 };

struct LayerDev {
    std::string scope;   // full scope, e.g. "SSRN/HC_5"
    int kind = K_C;
    int cin = 0, cout = 0, size = 1, rate = 1;
    bool causal = false;
    int act = 0;
    int nconv = 0, ldw = 0;
    float* W = nullptr;      // [size][cin][ldw]
    std::vector<float> hostW;   // same, kept on the host until the decode stream is packed (AudioEnc / AudioDec only)
    float* bias = nullptr;   // [ldw]
    float *g1 = nullptr, *b1 = nullptr, *g2 = nullptr, *b2 = nullptr;
    // tensor-core path: split-fp16 K-major weight planes [ncta*bn][ntaps*cin_pad], pre-scaled
    struct TcPack {
        bool ok = false;
        int mode = 0, ntaps = 0, kb_per_tap = 0, Ktot = 0, ncta = 1, bn = 0, half = 0, nrows = 0;
        float inv_scale = 1.f;
        __half *Whi = nullptr, *Wlo = nullptr;
        CUtensorMap mWhi, mWlo;
    } tc;
};

struct HostParam {
    std::vector<float> data;
    std::vector<int64_t> shape;
};

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void ensure(size_t n) {
        if (n <= bytes) return;
        if (p) CUDA_CHECK(cudaFree(p));
        p = nullptr; bytes = 0;
        CUDA_CHECK(cudaMalloc(&p, n));
        bytes = n;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

}  // namespace

struct dctts_handle_s {
    dctts_hparams hp{};
    int device = 0;
    int F = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;      // device->host copies of finished spectrogram chunks (dctts_synthesize_host)
    cudaEvent_t chunk_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::string err;

    std::map<std::string, HostParam> staged;
    bool committed = false;
    int64_t n_params = 0;

    std::vector<LayerDev> textenc, audioenc, audiodec, ssrn;
    std::map<std::string, LayerDev*> by_scope;
    std::map<std::string, float*> dev_vec;    // every committed variable (flat copy) by TF name
    std::vector<void*> param_allocs;
    float* embed_table = nullptr;

    // workspace (sized for ws_B utterances)
    int ws_B = 0;
    DevBuf scratch, act0, act1;
    DevBuf tickets;               // arrival counters of the fused GEMM + LN launches (2 ints per 16-row block)
    DevBuf kv;                    // (B, N, 2d) TextEnc output
    DevBuf ybuf;                  // (B, T, n_mels) generated mels
    DevBuf rbuf;                  // (B, T, 2d)
    std::vector<DevBuf> ae_out;   // AudioEnc per-layer outputs (B, T, d)
    std::vector<DevBuf> ad_out;   // AudioDec per-layer outputs (B, T, d | n_mels)
    DevBuf ad_sig;                // scratch for sigmoid(logits) in full-graph mode
    DevBuf ibuf;                  // ints: j, p_cur[B], p_next[B], p_prev[B], p_hist[B*T]
    DevBuf lbuf;                  // (B, N) ids staging for the host entry point
    DevBuf zbuf;                  // (B, 4T, F) staging for the host entry point
    DevBuf plane[4];              // tensor-core path activations: {hi,lo} x ping-pong, rows x 1032 fp16
    DevBuf attpl[6];              // tcgen05 attention operands: Q, K planes and transposed V planes ({hi,lo} each)
    DevBuf arpl[10];              // AR decode planes: R (B,T,2d) and four AudioDec outputs (B,T,d), {hi,lo} each

    // training step (Text2Mel, reference train.py mode "train"): see the "training" section below
    struct TrainLayer {
        LayerDev* l = nullptr; int li = 0; long long rows = 0; int L = 0, L_in = 0, ld_out = 0; const float* in = nullptr; int ld_in = 0;
        float* pre = nullptr; float* out = nullptr; int extra_shift = 0; bool need_dgrad = true;
        float *dW = nullptr, *dbias = nullptr, *dg1 = nullptr, *db1 = nullptr, *dg2 = nullptr, *db2 = nullptr;
        GemmTcSlots tc_slots;      // abs-max slots of this block's input and weights, set by the forward GEMM of the current step
    };
    struct TrainTensor { float* p; float* g; float* m; float* v; long long n; int layout, d0, d1, d2, ld; };
    struct {
        bool ready = false; int B = 0, num = 1, T_in = 0; float rate = 0.f;
        int cap_N = 0, cap_T = 0;                               // the activation workspace holds steps up to (cap_N keys, cap_T frames)
        std::vector<TrainLayer> layers;
        std::map<std::string, TrainTensor> tensors;            // by TF variable name
        DevBuf pre, out, emb, R, align, dS, gbuf[4], dy, wT, zeros, gts, sums, ids, grads, mom, vel, entries;
        long long n_grad = 0; int n_entries = 0; float* d_table = nullptr;
        DevBuf tc_a_hi, tc_a_lo, tc_b_hi, tc_b_lo, tc_slots;    // operand planes of the tcgen05 training GEMMs (kernels_gemm_tc.cu)
        GemmTcWs tc;
        int first[3] = {0, 0, 0}, last[3] = {0, 0, 0};         // layer index ranges: TextEnc, AudioEnc, AudioDec
    } tr;

    // vocoder (Griffin-Lim) state
    struct { int hop = 275, win = 1102, n_iter = 50; float power = 1.5f, max_db = 100.f, ref_db = 20.f, preemph = 0.97f; } voc;
    DevBuf feat_melw, feat_range, feat_tw, feat_window, feat_wss;   // feature extraction tables (dctts_get_spectrograms)
    int feat_sr = 0, feat_win = 0;
    DevBuf voc_S, voc_X, voc_frames, voc_mse, voc_tw, voc_window, voc_wss, voc_deemph;
    int voc_tables_T = 0, voc_tables_win = 0, voc_tables_hop = 0;

    // AR decode graph
    cudaGraphExec_t ar_exec = nullptr;
    int ar_B = 0;
    int64_t ar_nodes = 0;

    int tensor_path = 1;          // tcgen05 blocks wherever they apply; 0 forces the fp32 CUDA-core kernels
    int key_cap = 192;            // longest text (keys) any entry point takes: max(192, round_up(max_N, 64)), fixed at create
    int64_t launches = 0;

    // kernel-variant switches (dctts_set_option); the defaults are the measured-best configuration
    struct {
        int tc_occ2 = 1;          // two tcgen05 CTAs per SM (32-wide slab, 2 stages) on launches that fill the machine
        int tc_cg2 = 0;           // CTA pairs (cta_group::2): 0 off, 1 wide (N = 512 per pair), 2 narrow (N = 256 per pair)
        int tc_tile_pair = 0;     // two 128-row tiles per CTA sharing one weight slab
        int tc_mcast = 1;         // TMA multicast of the activation tile across the cluster
        int tc_resid_tma = 1;     // hc: residual in / planes out through TMA
        int tc_debug = 0;         // progress markers + in-kernel cycle stamps (synchronising)
        int fused_ln = 0;         // graph decode: split-K GEMM and LN epilogue in one launch
        int decode_prof = 0;      // persistent decode: record SM-clock lap timers of cluster 0 / rank 0 (dctts_decode_profile)
        int decode_mode = 1;      // 1 = persistent cluster kernel (kernels_decode.cu), 0 = one CUDA graph per frame (round-1 path)
        int train_probe = 0;      // measurement only (tools/bench_train.py --probe): the training GEMMs fetch their operands but issue no MMA
        int train_tc = 7;         // training GEMMs on tcgen05, bit mask: 1 forward conv, 2 data gradient, 4 weight gradient; 0 = fp32 CUDA-core kernels
    } opt;

    // persistent decode (kernels_decode.cu)
    struct {
        bool ok = false;          // stream packed, geometry supported, 16-CTA clusters schedulable
        DecParams tab{};          // layer / chunk tables (+ parameter pointers); per-call fields filled by text2mel_generate
        DevBuf wstream, lnp, scr, stats, pfinal, prof;
        int max_clusters = 0;
        std::string why;          // why not ok
        int last_moved_frames = -1, last_moved_utt = -1, last_clusters = 0;
    } dec;

    ~dctts_handle_s() {
        if (ar_exec) cudaGraphExecDestroy(ar_exec);
        for (void* p : param_allocs) cudaFree(p);
        for (DevBuf* b : {&tr.pre, &tr.out, &tr.emb, &tr.R, &tr.align, &tr.dS, &tr.gbuf[0], &tr.gbuf[1], &tr.gbuf[2], &tr.gbuf[3], &tr.dy,
                          &tr.wT, &tr.zeros, &tr.gts, &tr.sums, &tr.ids, &tr.grads, &tr.mom, &tr.vel, &tr.entries, &tr.tc_a_hi, &tr.tc_a_lo, &tr.tc_b_hi,
                          &tr.tc_b_lo, &tr.tc_slots}) b->release();
        dec.prof.release(); dec.wstream.release(); dec.lnp.release(); dec.scr.release(); dec.stats.release(); dec.pfinal.release();
        tickets.release(); scratch.release(); act0.release(); act1.release(); kv.release(); ybuf.release();
        rbuf.release(); ad_sig.release(); ibuf.release(); lbuf.release(); zbuf.release();
        for (auto& b : plane) b.release();
        for (auto& b : arpl) b.release();
        for (auto& b : attpl) b.release();
        voc_S.release(); voc_X.release(); voc_frames.release(); voc_mse.release(); voc_tw.release(); voc_window.release(); voc_wss.release(); voc_deemph.release();
        feat_melw.release(); feat_range.release(); feat_tw.release(); feat_window.release(); feat_wss.release();
        for (auto& b : ae_out) b.release();
        for (auto& b : ad_out) b.release();
        if (copy_stream) { cudaStreamDestroy(copy_stream); for (auto e : chunk_done) if (e) cudaEventDestroy(e); }
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

using H = dctts_handle_s;

// ---------------------------------------------------------------------------- layer tables
void add_layer(std::vector<LayerDev>& v, const std::string& net, int kind, int idx, int cin, int cout,
               int size, int rate, bool causal, int act) {
    LayerDev l;
    const char* pre = kind == K_C ? "C_" : (kind == K_HC ? "HC_" : "D_");
    l.scope = net + "/" + pre + std::to_string(idx);
    l.kind = kind; l.cin = cin; l.cout = cout; l.size = size; l.rate = rate;
    l.causal = causal; l.act = act;
    l.nconv = (kind == K_HC) ? 2 * cout : cout;
    l.ldw = roundup(l.nconv, 4);
    v.push_back(l);
}

void build_tables(H* h) {
    const dctts_hparams& hp = h->hp;
    const int d = hp.d, d2 = 2 * hp.d, c = hp.c, F = h->F;
    int i;
    // TextEnc, networks.py:23-68
    {
        auto& v = h->textenc; const std::string n = "Text2Mel/TextEnc"; i = 2;
        add_layer(v, n, K_C, i++, hp.e, d2, 1, 1, false, 1);
        add_layer(v, n, K_C, i++, d2, d2, 1, 1, false, 0);
        for (int rep = 0; rep < 2; ++rep)
            for (int j = 0, r = 1; j < 4; ++j, r *= 3) add_layer(v, n, K_HC, i++, d2, d2, 3, r, false, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_HC, i++, d2, d2, 3, 1, false, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_HC, i++, d2, d2, 1, 1, false, 0);
    }
    // AudioEnc, networks.py:81-124
    {
        auto& v = h->audioenc; const std::string n = "Text2Mel/AudioEnc"; i = 1;
        add_layer(v, n, K_C, i++, hp.n_mels, d, 1, 1, true, 1);
        add_layer(v, n, K_C, i++, d, d, 1, 1, true, 1);
        add_layer(v, n, K_C, i++, d, d, 1, 1, true, 0);
        for (int rep = 0; rep < 2; ++rep)
            for (int j = 0, r = 1; j < 4; ++j, r *= 3) add_layer(v, n, K_HC, i++, d, d, 3, r, true, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_HC, i++, d, d, 3, 3, true, 0);
    }
    // AudioDec, networks.py:166-209
    {
        auto& v = h->audiodec; const std::string n = "Text2Mel/AudioDec"; i = 1;
        add_layer(v, n, K_C, i++, d2, d, 1, 1, true, 0);
        for (int j = 0, r = 1; j < 4; ++j, r *= 3) add_layer(v, n, K_HC, i++, d, d, 3, r, true, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_HC, i++, d, d, 3, 1, true, 0);
        for (int rep = 0; rep < 3; ++rep) add_layer(v, n, K_C, i++, d, d, 1, 1, true, 1);
        add_layer(v, n, K_C, i++, d, hp.n_mels, 1, 1, true, 0);
    }
    // SSRN, networks.py:223-290
    {
        auto& v = h->ssrn; const std::string n = "SSRN"; i = 1;
        add_layer(v, n, K_C, i++, hp.n_mels, c, 1, 1, false, 0);
        for (int j = 0, r = 1; j < 2; ++j, r *= 3) add_layer(v, n, K_HC, i++, c, c, 3, r, false, 0);
        for (int rep = 0; rep < 2; ++rep) {
            add_layer(v, n, K_D, i++, c, c, 3, 1, false, 0);
            for (int j = 0, r = 1; j < 2; ++j, r *= 3) add_layer(v, n, K_HC, i++, c, c, 3, r, false, 0);
        }
        add_layer(v, n, K_C, i++, c, 2 * c, 1, 1, false, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_HC, i++, 2 * c, 2 * c, 3, 1, false, 0);
        add_layer(v, n, K_C, i++, 2 * c, F, 1, 1, false, 0);
        for (int rep = 0; rep < 2; ++rep) add_layer(v, n, K_C, i++, F, F, 1, 1, false, 1);
        add_layer(v, n, K_C, i, F, F, 1, 1, false, 0);     // networks.py:285-290 (counter not advanced)
    }
    for (auto* vec : {&h->textenc, &h->audioenc, &h->audiodec, &h->ssrn})
        for (auto& l : *vec) h->by_scope[l.scope] = &l;
}

// ---------------------------------------------------------------------------- parameters
const HostParam& need(H* h, const std::string& name, std::vector<int64_t> shape) {
    auto it = h->staged.find(name);
    if (it == h->staged.end()) throw std::runtime_error("missing variable: " + name);
    if (it->second.shape != shape) throw std::runtime_error("bad shape for variable: " + name);
    return it->second;
}

float* upload(H* h, const std::vector<float>& v) {
    float* p = nullptr;
    CUDA_CHECK(cudaMalloc(&p, v.size() * sizeof(float)));
    h->param_allocs.push_back(p);
    CUDA_CHECK(cudaMemcpy(p, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
    return p;
}

float* upload_vec(H* h, const std::string& name, int n, int padded) {
    const HostParam& p = need(h, name, {n});
    std::vector<float> v(padded, 0.f);
    std::copy(p.data.begin(), p.data.end(), v.begin());
    float* d = upload(h, v);
    h->dev_vec[name] = d;
    h->n_params += n;
    return d;
}

// Split-fp16 packing for the tcgen05 kernel (kernels_tc.cu).  Rows are accumulator columns in
// cluster-slice order (CTA i owns rows [i*bn, (i+1)*bn); for hc / transposed conv its first
// `half` rows are the first LN half, the rest the second), columns are k = tap*cin_pad + ci.
// Weights are multiplied by a power of two that brings max|W| into [2^10, 2^11) so that the
// low plane stays in fp16's normal range; the kernel multiplies the accumulator back.
void pack_tc(H* h, LayerDev& l, const std::vector<float>& W /* [size][cin][ldw] */) {
    LayerDev::TcPack& p = l.tc;
    const int cin_pad = roundup(l.cin, 64);
    p.kb_per_tap = cin_pad / 64;
    if (l.kind == K_C) {
        p.mode = 0; p.ntaps = l.size;
        // small nets (<= 256 channels) are used on few rows (decode): prefer more, narrower CTAs
        const int maxbn = (l.cout <= 256 && l.cout % 64 == 0) ? 64 : 256;
        p.ncta = 1;
        while (roundup((l.cout + p.ncta - 1) / p.ncta, 16) > maxbn) p.ncta *= 2;
        p.bn = roundup((l.cout + p.ncta - 1) / p.ncta, 16); p.half = p.bn;
    } else {
        p.mode = (l.kind == K_HC) ? 1 : 2; p.ntaps = (l.kind == K_HC) ? l.size : 2;
        p.half = (l.cout <= 256) ? 32 : 128; p.bn = 2 * p.half; p.ncta = l.cout / p.half;   // decode nets: 8 narrow CTAs per tile
        if (l.cout % p.half) return;
    }
    if (p.ncta > 8) return;
    p.Ktot = p.ntaps * cin_pad; p.nrows = p.ncta * p.bn;
    auto wv = [&](int tap, int ci, int row) -> float {
        const int i = row / p.bn, a = row % p.bn;
        if (p.mode == 0) return row < l.cout ? W[((size_t)tap * l.cin + ci) * l.ldw + row] : 0.f;
        const bool second = a >= p.half;
        const int col = i * p.half + (a % p.half);
        if (p.mode == 1) return W[((size_t)tap * l.cin + ci) * l.ldw + (second ? l.cout + col : col)];
        // transposed conv: k-tap 0 reads x[t] (W0 -> even rows, W1 -> odd rows), k-tap 1 reads x[t-1] (W2 -> even rows)
        if (tap == 0) return W[((size_t)(second ? 1 : 0) * l.cin + ci) * l.ldw + col];
        return second ? 0.f : W[((size_t)2 * l.cin + ci) * l.ldw + col];
    };
    float maxabs = 0.f;
    for (int tap = 0; tap < p.ntaps; ++tap)
        for (int ci = 0; ci < l.cin; ++ci)
            for (int row = 0; row < p.nrows; ++row) maxabs = std::max(maxabs, std::fabs(wv(tap, ci, row)));
    float scale = 1.f;
    if (maxabs > 0.f) { int e; std::frexp(maxabs, &e); scale = std::ldexp(1.f, 11 - e); }   // maxabs*scale in [2^10, 2^11)
    p.inv_scale = 1.f / scale;
    std::vector<__half> hi((size_t)p.nrows * p.Ktot, __float2half_rn(0.f)), lo(hi);
    for (int row = 0; row < p.nrows; ++row)
        for (int tap = 0; tap < p.ntaps; ++tap)
            for (int ci = 0; ci < l.cin; ++ci) {
                const float v = wv(tap, ci, row) * scale;
                const __half hv = __float2half_rn(v);
                const size_t idx = (size_t)row * p.Ktot + (size_t)tap * cin_pad + ci;
                hi[idx] = hv;
                lo[idx] = __float2half_rn(v - __half2float(hv));
            }
    const size_t bytes = hi.size() * sizeof(__half);
    CUDA_CHECK(cudaMalloc(&p.Whi, bytes)); h->param_allocs.push_back(p.Whi);
    CUDA_CHECK(cudaMalloc(&p.Wlo, bytes)); h->param_allocs.push_back(p.Wlo);
    CUDA_CHECK(cudaMemcpy(p.Whi, hi.data(), bytes, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(p.Wlo, lo.data(), bytes, cudaMemcpyHostToDevice));
    tc_make_w_map(&p.mWhi, p.Whi, p.Ktot, p.nrows, p.bn, tc_bk());
    tc_make_w_map(&p.mWlo, p.Wlo, p.Ktot, p.nrows, p.bn, tc_bk());
    p.ok = true;
}

void commit_layer(H* h, LayerDev& l) {
    const int k = l.size, cin = l.cin, nconv = l.nconv, ldw = l.ldw;
    std::vector<float> W((size_t)k * cin * ldw, 0.f);
    if (l.kind == K_D) {
        // TF kernel [1, k, Cout, Cin] (modules.py:232-239) -> [tap][Cin][ldw]
        const HostParam& p = need(h, l.scope + "/conv2d_transpose/kernel", {1, k, l.cout, cin});
        for (int j = 0; j < k; ++j)
            for (int co = 0; co < l.cout; ++co)
                for (int ci = 0; ci < cin; ++ci)
                    W[((size_t)j * cin + ci) * ldw + co] = p.data[((size_t)j * l.cout + co) * cin + ci];
        l.bias = upload_vec(h, l.scope + "/conv2d_transpose/bias", l.cout, ldw);
        h->n_params += (int64_t)k * l.cout * cin;
    } else {
        // TF kernel [k, Cin, Nconv] (modules.py:134,187) -> same order, rows padded to ldw
        const HostParam& p = need(h, l.scope + "/conv1d/kernel", {k, cin, nconv});
        for (size_t row = 0; row < (size_t)k * cin; ++row)
            std::copy(p.data.begin() + row * nconv, p.data.begin() + (row + 1) * nconv, W.begin() + row * ldw);
        l.bias = upload_vec(h, l.scope + "/conv1d/bias", nconv, ldw);
        h->n_params += (int64_t)k * cin * nconv;
    }
    l.W = upload(h, W);
    if (l.scope.compare(0, 14, "Text2Mel/Audio") == 0) l.hostW = W;
    pack_tc(h, l, W);
    if (l.kind == K_HC) {
        l.g1 = upload_vec(h, l.scope + "/H1/gamma", l.cout, l.cout);
        l.b1 = upload_vec(h, l.scope + "/H1/beta", l.cout, l.cout);
        l.g2 = upload_vec(h, l.scope + "/H2/gamma", l.cout, l.cout);
        l.b2 = upload_vec(h, l.scope + "/H2/beta", l.cout, l.cout);
    } else {
        l.g1 = upload_vec(h, l.scope + "/normalize/gamma", l.cout, l.cout);
        l.b1 = upload_vec(h, l.scope + "/normalize/beta", l.cout, l.cout);
    }
}

std::vector<int> audiodec_rows(const std::vector<LayerDev>& net, int T);

// ---------------------------------------------------------------------------- persistent decode tables
// Layer / chunk tables and the per-rank weight streams of the cluster decode kernel (kernels_decode.cu).
// Stream of rank r = for every block of AudioEnc then AudioDec, for every tap, for every chunk of <= 4096 floats:
// the block's weight columns owned by rank r ([k/4][column][4]).  hc blocks: columns [0, cs) are the gate
// channels r*cs.., [cs, 2cs) the info channels of the same index (modules.py:188-193); conv blocks: cs columns
// (+ zero columns up to a multiple of 4).
void pack_decode(H* h) {
    auto& D = h->dec;
    D.ok = false;
    const dctts_hparams& hp = h->hp;
    const int d = hp.d;
    if (d != 256) { D.why = "persistent decode needs d = 256"; return; }
    if (hp.n_mels % DEC_NC || hp.n_mels > 128 || hp.attention_win_size > 4 || hp.attention_win_size < 1) { D.why = "persistent decode: unsupported n_mels / window"; return; }
    std::vector<LayerDev*> nets;
    for (auto& l : h->audioenc) nets.push_back(&l);
    for (auto& l : h->audiodec) nets.push_back(&l);
    if ((int)nets.size() > DEC_MAXL) { D.why = "persistent decode: too many blocks"; return; }
    DecParams& P = D.tab;
    memset(&P, 0, sizeof(P));
    P.nl = (int)nets.size(); P.n_enc = (int)h->audioenc.size();
    std::vector<int> prow = audiodec_rows(h->audiodec, hp.max_T);
    int nch = 0, off = 0;
    for (int li = 0; li < P.nl; ++li) {
        const LayerDev& l = *nets[li];
        DecLayer& L = P.L[li];
        if (l.kind == K_D || !l.causal || (l.cin % 4) || (l.kind == K_HC && (l.cin != d || l.cout != d)) || l.cout % DEC_NC ||
            (li != 0 && l.cin % 128)) { D.why = "persistent decode: unsupported block " + l.scope; return; }
        L.kind = l.kind == K_HC ? 1 : 0; L.cin = l.cin; L.cout = l.cout; L.ntaps = l.size; L.rate = l.rate; L.act = l.act;
        L.cs = l.cout / DEC_NC; L.ns = L.kind ? 2 * L.cs : (L.cs <= 8 ? 8 : roundup(L.cs, 4));
        if (L.ns != 8 && L.ns != 16 && L.ns != 32) { D.why = "persistent decode: unsupported slice width"; return; }
        L.prow = li >= P.n_enc ? prow[li - P.n_enc] : 1;
        if (L.prow > 1 && (L.cout != 256 || (L.ns != 32 && L.ns != 16) || L.prow > 85)) { D.why = "persistent decode: unsupported receptive field"; return; }
        L.ldin = l.cin;
        const int cinp = roundup(l.cin, 128);                     // AudioEnc C_1: 80 -> 128 zero rows
        if (l.size > 1 && cinp != 256) { D.why = "persistent decode: multi-tap blocks must have 256 input channels"; return; }
        const int K = l.size * cinp;
        L.krows = std::min(K, DEC_SLOT_F / L.ns);                 // k rows per chunk
        const int kr8 = L.krows / 8, sg = 32 / L.ns;
        if (K % L.krows || L.krows % 8 || kr8 * L.ns > DEC_REG_F || kr8 % (8 * sg) || (L.prow > 1 && kr8 % 16)) {
            D.why = "persistent decode: chunk geometry"; return;
        }
        if (L.prow > 1 && (L.prow - 1) + (l.size - 1) * l.rate > 96) { D.why = "persistent decode: receptive field too tall"; return; }
        L.ch0 = nch;
        for (int k0 = 0; k0 < K; k0 += L.krows) {
            if (nch >= DEC_MAXCH) { D.why = "persistent decode: too many weight chunks"; return; }
            DecChunk& c = P.C[nch++];
            c.off = off; c.nfl4 = (short)(L.krows * L.ns / 4); c.k0 = (short)k0; c.krows = (short)L.krows; c.layer = (short)li;
            off += L.krows * L.ns;
        }
        L.nch = nch - L.ch0;
        if (li == P.n_enc - 1) P.nch_enc = nch;
        if (L.prow > 1) { if (P.pyr_ch1 == 0) P.pyr_ch0 = L.ch0; P.pyr_ch1 = nch; }
    }
    if (P.L[P.nl - 1].prow != 1 || P.L[P.n_enc].ntaps != 1 || P.nch_enc <= DEC_NSLOT) { D.why = "persistent decode: unexpected AudioDec shape"; return; }
    for (int li = P.n_enc; li < P.nl; ++li)                        // the receptive-field blocks must be a prefix of AudioDec
        if (P.L[li].prow > 1 && li > P.n_enc && P.L[li - 1].prow <= 1) { D.why = "persistent decode: receptive-field blocks not contiguous"; return; }
    P.nch = nch;
    // the receptive-field blocks a second time, as split-fp16 MMA slabs (tcgen05 pre-pass): same chunk sizes, appended
    for (int li = 0; li < P.nl; ++li) {
        const DecLayer& L = P.L[li];
        if (L.prow <= 1) continue;
        if (L.krows % 128 || (L.ns != 32 && L.ns != 16)) { D.why = "persistent decode: tcgen05 pre-pass geometry"; return; }
        for (int c = L.ch0; c < L.ch0 + L.nch; ++c) { P.C[c].off16 = off; off += L.krows * L.ns; }
    }
    P.stream_len = off;
    // streams: chunk = 8 warp regions, region w = rows [w*kr8, (w+1)*kr8) as [k/4][column][4] (32-column slices: pair-split, below)
    std::vector<float> st((size_t)DEC_NC * off, 0.f);
    for (int li = 0; li < P.nl; ++li) {                              // power-of-two scale per receptive-field block (as pack_tc)
        const LayerDev& l = *nets[li]; const DecLayer& L = P.L[li];
        P.inv_scale[li] = 1.f;
        if (L.prow <= 1) continue;
        float maxabs = 0.f;
        for (size_t i = 0; i < l.hostW.size(); ++i) maxabs = std::max(maxabs, std::fabs(l.hostW[i]));
        float scale = 1.f;
        if (maxabs > 0.f) { int e; std::frexp(maxabs, &e); scale = std::ldexp(1.f, 11 - e); }
        P.inv_scale[li] = 1.f / scale;
    }
    for (int r = 0; r < DEC_NC; ++r)
        for (int li = 0; li < P.nl; ++li) {
            const LayerDev& l = *nets[li]; const DecLayer& L = P.L[li];
            REQUIRE(!l.hostW.empty(), "persistent decode: host weights missing");
            const int cinp = roundup(l.cin, 128), kr8 = L.krows / 8;
            auto column = [&](int n) -> int {
                if (L.kind) return n < L.cs ? r * L.cs + n : l.cout + r * L.cs + (n - L.cs);
                return n < L.cs ? r * L.cs + n : -1;
            };
            for (int c = L.ch0; c < L.ch0 + L.nch; ++c) {
                const DecChunk& ch = P.C[c];
                float* dst = st.data() + (size_t)r * off + ch.off;
                for (int kc = 0; kc < ch.krows; ++kc) {
                    const int k = ch.k0 + kc, tap = k / cinp, ci = k % cinp;
                    if (ci >= l.cin) continue;
                    const int w = kc / kr8, kk = kc % kr8;
                    const float* wrow = l.hostW.data() + ((size_t)tap * l.cin + ci) * l.ldw;
                    for (int n = 0; n < L.ns; ++n) {
                        const int col = column(n);
                        if (col < 0) continue;
                        // 32-column slices: pair-split layout per 8-k block [column parity][k-group][column pair][4 k]
                        // (gemv_warp32); narrower slices: [k/4][column][4]
                        const size_t idx = L.ns == 32 ? (size_t)(kk / 8) * 256 + ((size_t)((n & 1) * 2 + (kk / 4) % 2) * 16 + (n >> 1)) * 4 + (kk % 4)
                                                      : ((size_t)(kk / 4) * L.ns + n) * 4 + (kk % 4);
                        dst[(size_t)w * kr8 * L.ns + idx] = wrow[col];
                    }
                }
                if (L.prow <= 1) continue;
                // the same rows as MMA slabs of 16 k: [plane hi | lo][k8 group][column][8 halfs], 16*ns floats per slab, in k order
                // (slab s of the chunk sits at float offset s*16*ns: region w of the chunk = slabs [w*spr, (w+1)*spr))
                __half* d16 = reinterpret_cast<__half*>(st.data() + (size_t)r * off + ch.off16);
                const float scale = 1.f / P.inv_scale[li];
                for (int kc = 0; kc < ch.krows; ++kc) {
                    const int k = ch.k0 + kc, tap = k / cinp, ci = k % cinp;
                    const int slab = kc / 16, k16 = kc % 16, grp = k16 / 8, e8 = k16 % 8;
                    const float* wrow = l.hostW.data() + ((size_t)tap * l.cin + ci) * l.ldw;
                    for (int n = 0; n < L.ns; ++n) {
                        const int col = column(n);
                        const float v = (col >= 0 && ci < l.cin) ? wrow[col] * scale : 0.f;
                        const __half hv = __float2half_rn(v);
                        const size_t base = (size_t)slab * 32 * L.ns;                  // halfs per slab = 2 planes * 2 groups * ns * 8
                        const size_t idx = ((size_t)grp * L.ns + n) * 8 + e8;
                        d16[base + idx] = hv;
                        d16[base + (size_t)2 * L.ns * 8 + idx] = __float2half_rn(v - __half2float(hv));
                    }
                }
            }
        }
    D.wstream.ensure(st.size() * sizeof(float));
    CUDA_CHECK(cudaMemcpy(D.wstream.p, st.data(), st.size() * sizeof(float), cudaMemcpyHostToDevice));
    // LayerNorm parameters [layer][gamma1 | beta1 | gamma2 | beta2][256]
    D.lnp.ensure((size_t)P.nl * 1024 * sizeof(float));
    CUDA_CHECK(cudaMemset(D.lnp.p, 0, D.lnp.bytes));
    for (int li = 0; li < P.nl; ++li) {
        const LayerDev& l = *nets[li];
        float* base = D.lnp.as<float>() + (size_t)li * 1024;
        const float* src[4] = {l.g1, l.b1, l.kind == K_HC ? l.g2 : nullptr, l.kind == K_HC ? l.b2 : nullptr};
        for (int q = 0; q < 4; ++q)
            if (src[q]) CUDA_CHECK(cudaMemcpy(base + q * 256, src[q], (size_t)l.cout * sizeof(float), cudaMemcpyDeviceToDevice));
        P.lnp[li] = base; P.bias[li] = l.bias;
    }
    P.wstream = D.wstream.as<float>();
    for (auto* lp : nets) { lp->hostW.clear(); lp->hostW.shrink_to_fit(); }
    D.max_clusters = decode_max_active_clusters();
    if (D.max_clusters < 1) { D.why = "persistent decode: a 16-CTA cluster with " + std::to_string(decode_smem_bytes()) + " B of shared memory cannot be scheduled"; return; }
    D.ok = true; D.why.clear();
}

void commit_params(H* h) {
    REQUIRE(!h->committed, "parameters already committed on this handle");
    CUDA_CHECK(cudaSetDevice(h->device));
    h->n_params = 0;
    {
        const std::string name = "Text2Mel/TextEnc/embed_1/lookup_table";
        const HostParam& p = need(h, name, {h->hp.vocab_size, h->hp.e});
        h->embed_table = upload(h, p.data);
        h->dev_vec[name] = h->embed_table;
        h->n_params += (int64_t)h->hp.vocab_size * h->hp.e;
    }
    size_t expected = 1;
    for (auto* vec : {&h->textenc, &h->audioenc, &h->audiodec, &h->ssrn})
        for (auto& l : *vec) { commit_layer(h, l); expected += (l.kind == K_HC) ? 6 : 4; }
    if (h->staged.size() != expected) {
        for (auto& kvp : h->staged) {
            const std::string& n = kvp.first;
            bool known = h->dev_vec.count(n) || n.find("/kernel") != std::string::npos;
            if (!known) throw std::runtime_error("unknown variable staged: " + n);
        }
        throw std::runtime_error("staged variable count does not match the path's variable set");
    }
    pack_decode(h);
    h->staged.clear();
    h->committed = true;
}

// ---------------------------------------------------------------------------- workspace
void ensure_ws(H* h, int B) {
    if (B <= h->ws_B) return;
    const dctts_hparams& hp = h->hp;
    const int T = hp.max_T, N = hp.max_N, d = hp.d, F = h->F;
    const size_t rows_ssrn = (size_t)B * T * hp.r;
    // invalidate anything that baked pointers
    if (h->ar_exec) { CUDA_CHECK(cudaStreamSynchronize(h->stream)); cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; h->ar_B = 0; }
    CUDA_CHECK(cudaDeviceSynchronize());
    const size_t ld_scr = (size_t)roundup(std::max(std::max(4 * hp.c, F), 4 * d), 4);
    h->scratch.ensure(std::max(rows_ssrn * ld_scr * sizeof(float), (size_t)64 << 20));
    const size_t ld_act = (size_t)roundup(std::max(std::max(2 * hp.c, F), 2 * d), 4);
    h->act0.ensure(rows_ssrn * ld_act * sizeof(float));
    h->act1.ensure(rows_ssrn * ld_act * sizeof(float));
    h->kv.ensure((size_t)B * N * 2 * d * sizeof(float));
    h->ybuf.ensure((size_t)B * T * hp.n_mels * sizeof(float));
    h->rbuf.ensure((size_t)B * T * 2 * d * sizeof(float));
    h->ad_sig.ensure((size_t)B * T * hp.n_mels * sizeof(float));
    h->ae_out.resize(h->audioenc.size());
    for (size_t i = 0; i < h->audioenc.size(); ++i)
        h->ae_out[i].ensure((size_t)B * T * h->audioenc[i].cout * sizeof(float));
    h->ad_out.resize(h->audiodec.size());
    for (size_t i = 0; i < h->audiodec.size(); ++i)
        h->ad_out[i].ensure((size_t)B * T * h->audiodec[i].cout * sizeof(float));
    h->ibuf.ensure((size_t)(4 + 3 * B + (size_t)B * T) * sizeof(int));
    h->lbuf.ensure((size_t)B * N * sizeof(int));
    for (auto& pb : h->plane) pb.ensure(rows_ssrn * (size_t)roundup(std::max(std::max(2 * hp.c, F), 2 * d), 8) * sizeof(__half));
    for (int i = 0; i < 10; ++i) {
        const size_t bytes = (size_t)B * T * (i < 2 ? 2 * d : d) * sizeof(__half);
        h->arpl[i].ensure(bytes);
        CUDA_CHECK(cudaMemset(h->arpl[i].p, 0, h->arpl[i].bytes));
    }
    h->dec.scr.ensure((size_t)(B + DEC_GMAX) * 85 * 512 * sizeof(float));
    h->dec.stats.ensure((size_t)2 * B * sizeof(int));
    h->dec.pfinal.ensure((size_t)B * sizeof(int));
    h->ws_B = B;
}

void ensure_scratch(H* h, size_t bytes);
struct IntBufs { int *j, *p_cur, *p_next, *p_prev, *p_hist; };
IntBufs ints(H* h) {
    int* base = h->ibuf.as<int>();
    IntBufs r;
    r.j = base; r.p_cur = base + 4; r.p_next = r.p_cur + h->ws_B; r.p_prev = r.p_next + h->ws_B;
    r.p_hist = r.p_prev + h->ws_B;
    return r;
}

// ---------------------------------------------------------------------------- block runners
struct Launch {
    H* h; cudaStream_t s;
    std::vector<cudaEvent_t>* evs = nullptr;     // profile mode: one event after every kernel
    void count(int n = 1) {
        h->launches += n;
        if (evs) {
            cudaEvent_t e;
            CUDA_CHECK(cudaEventCreate(&e));
            CUDA_CHECK(cudaEventRecord(e, s));
            evs->push_back(e);
        }
    }
};

// conv (+bias) into scratch, then the LN / highway epilogue.  `extra_shift` moves every tap
// (AudioEnc's first block reads the mel buffer one frame back: train.py:51).
void run_block(Launch& lc, const LayerDev& l, int rate, bool causal, int act,
               const float* X, int ldx, RowWin win, float* out, int ldo, float* out2, int ldo2,
               int extra_shift = 0) {
    H* h = lc.h;
    REQUIRE(l.kind != K_D, "run_block: transposed conv must use run_deconv");
    ConvArgs c{};
    c.X = X; c.ldx = ldx; c.Y = h->scratch.as<float>(); c.ldy = l.ldw; c.bias = l.bias;
    c.K = l.cin; c.N = l.nconv; c.ldw = l.ldw;
    c.ntaps = l.size;
    const int tot = (l.size - 1) * rate;
    const int left = causal ? tot : tot / 2;
    for (int j = 0; j < l.size; ++j) {
        c.taps[j].W = l.W + (size_t)j * l.cin * l.ldw;
        c.taps[j].shift = j * rate - left + extra_shift;
    }
    c.win = win; c.Lout = win.L; c.ostride = 1; c.ooff = 0;
    LnArgs n{};
    n.Y = c.Y; n.ldy = l.ldw; n.g1 = l.g1; n.b1 = l.b1; n.g2 = l.g2; n.b2 = l.b2;
    n.X = X; n.ldx = ldx; n.out = out; n.ldo = ldo; n.out2 = out2; n.ldo2 = ldo2;
    n.C = l.cout; n.mode = (l.kind == K_HC) ? 1 : 0; n.act = act; n.win = win;
    // option fused_ln (experiment): GEMM and LN epilogue in one launch, the last CTAs of each 16-row block
    // waiting on an arrival counter.  Parity-green but SLOWER than two graph nodes (B=1: 220 vs 187 us per
    // decode step, B=32: 339 vs 303): a kernel boundary inside a CUDA graph costs less than the
    // ticket / spin / L2 round trips that replace it.
    if (h->opt.fused_ln && h->tickets.p && conv_gemm_ln_fusable(c, n)) {
        launch_conv_gemm_ln(c, n, h->tickets.as<int>(), lc.s, h->scratch.bytes); lc.count();
        return;
    }
    GemmOut go = launch_conv_gemm(c, lc.s, h->scratch.bytes); lc.count();
    n.nparts = go.nparts; n.compact = go.compact; n.part_stride = go.part_stride;
    launch_ln_rows(n, lc.s); lc.count();
}

// stride-2 transposed conv (modules.py:232-239): out[2t] = W0 x[t] + W2 x[t-1], out[2t+1] = W1 x[t].
void run_deconv(Launch& lc, const LayerDev& l, const float* X, int ldx, int B, int L, float* out, int ldo) {
    H* h = lc.h;
    ConvArgs c{};
    c.X = X; c.ldx = ldx; c.Y = h->scratch.as<float>(); c.ldy = l.ldw; c.bias = l.bias;
    c.K = l.cin; c.N = l.nconv; c.ldw = l.ldw;
    c.win = RowWin{B, L, L, nullptr}; c.Lout = 2 * L; c.ostride = 2;
    const size_t tapsz = (size_t)l.cin * l.ldw;
    c.ntaps = 2; c.taps[0] = ConvTap{l.W + 0 * tapsz, 0}; c.taps[1] = ConvTap{l.W + 2 * tapsz, -1}; c.ooff = 0;
    launch_conv_gemm(c, lc.s, h->scratch.bytes, false); lc.count();
    c.ntaps = 1; c.taps[0] = ConvTap{l.W + 1 * tapsz, 0}; c.ooff = 1;
    launch_conv_gemm(c, lc.s, h->scratch.bytes, false); lc.count();
    LnArgs n{};
    n.Y = c.Y; n.ldy = l.ldw; n.g1 = l.g1; n.b1 = l.b1; n.out = out; n.ldo = ldo;
    n.C = l.cout; n.mode = 0; n.act = 0; n.win = RowWin{B, 2 * L, 2 * L, nullptr};
    launch_ln_rows(n, lc.s); lc.count();
}

bool chain_tc_ok(H* h, const std::vector<LayerDev>& net);
void run_chain_tc_planes(Launch& lc, const std::vector<LayerDev>& net, Planes cur, int which, int B, int L,
                         float* out, float* out_sig, int first_extra_shift);
void run_chain_full_tc(Launch& lc, const std::vector<LayerDev>& net, const float* X, int ldx, int B, int L,
                       float* out, float* out_sig);

// A whole chain over full sequences, ping-ponging act0/act1; the last block writes
// `out` (dense, ld = its cout) and optionally sigmoid(out) into out_sig.
void run_chain_full(Launch& lc, const std::vector<LayerDev>& net, const float* X, int ldx, int B, int L,
                    float* out, float* out_sig) {
    H* h = lc.h;
    if (chain_tc_ok(h, net) && (out || out_sig)) { run_chain_full_tc(lc, net, X, ldx, B, L, out, out_sig); return; }
    const float* cur = X; int ld = ldx; int len = L;
    float* bufs[2] = {h->act0.as<float>(), h->act1.as<float>()};
    int which = 0;
    for (size_t i = 0; i < net.size(); ++i) {
        const LayerDev& l = net[i];
        const bool last = (i + 1 == net.size());
        float* dst = last ? out : bufs[which];
        const int ldo = last ? l.cout : roundup(l.cout, 4);
        if (last && !dst) { dst = bufs[which]; }            // logits not requested: park them
        if (l.kind == K_D) {
            run_deconv(lc, l, cur, ld, B, len, dst, ldo);
            len *= 2;
        } else {
            run_block(lc, l, l.rate, l.causal, l.act, cur, ld, RowWin{B, len, len, nullptr}, dst, ldo,
                      last ? out_sig : nullptr, l.cout);
        }
        cur = dst; ld = ldo; which ^= 1;
    }
}

Planes ws_planes(H* h, int which, int C) {
    Planes p; p.hi = h->plane[2 * which].as<__half>(); p.lo = h->plane[2 * which + 1].as<__half>(); p.ld = roundup(C, 8);
    return p;
}

// One reference block as ONE tcgen05 kernel (kernels_tc.cu).  X are the split planes of the
// (B, L, cin) input; the output goes to planes and/or fp32 tensors.
void run_block_tc(Launch& lc, const LayerDev& l, int rate, bool causal, int act, Planes X, RowWin win,
                  int TT, int TB, int tiles_t, Planes out, float* out_f32, int ld_f32, float* sig_f32, int ld_sig,
                  Planes sig, int extra_shift = 0) {
    const LayerDev::TcPack& p = l.tc;
    REQUIRE(p.ok, "tensor-core path not available for this block");
    TcArgs a{};
    a.bias = l.bias; a.g1 = l.g1; a.b1 = l.b1; a.g2 = (p.mode == 1) ? l.g2 : l.g1; a.b2 = (p.mode == 1) ? l.b2 : l.b1;
    a.mode = p.mode; a.act = act; a.C = l.cout; a.bn = p.bn; a.half = p.half; a.inv_scale = p.inv_scale;
    const int tiles = ((win.B + TB - 1) / TB) * tiles_t;
    // CTA pairs (tcgen05 cta_group::2): hc / transposed-conv blocks packed with 128-channel halves, on full
    // sequences.  Ranks (2s, 2s+1) of the cluster share channel slice s (256 channels), take consecutive tiles,
    // each stages half of the slice's weight slab; the accumulator is 512 columns (256 gate + 256 info).
    // Two CTAs per SM (default for launches that fill the machine): 32-wide slab, two pipeline stages -> ~105 KB of
    // shared memory and 256 TMEM columns per CTA, so one tile's epilogue runs under the other tile's main loop
    // (SSRN at B=32: 5.61 -> 4.66 ms).  Option tc_occ2 = 0 turns it off; tc_cg2 = 1 selects CTA pairs instead
    // (cta_group::2 needs all 512 TMEM columns, so the two cannot be combined).
    H* h = lc.h;
    const bool occ2_mode = h->opt.tc_occ2 != 0;
    // option tc_cg2: 1 = wide pairs (N = 512 per pair, all of TMEM, one CTA per SM), 2 = narrow pairs (N = 256 per pair,
    // 256 TMEM columns per CTA, so two CTAs per SM still overlap epilogue and main loop; the cluster doubles to
    // 2 x slices CTAs, 16 for the C = 1024 blocks)
    const int cg2_mode = h->opt.tc_cg2;
    const bool pairable = p.mode != 0 && p.half == 128 && p.bn == 256 && !win.jptr && TT == 128 && TB == 1;
    // Only when the paired grid still fills the machine: pairs halve the CTA count (B=1 SSRN: 1.09 vs 0.74 ms).
    const bool wide_pairs = cg2_mode == 1 && pairable && (p.ncta % 2) == 0 && tiles * p.ncta >= 4 * 148;
    const bool narrow_pairs = cg2_mode == 2 && pairable && 2 * p.ncta <= 16 && tiles * p.ncta >= 2 * 148;
    const int cg = (wide_pairs || narrow_pairs) ? 2 : 1;
    if (wide_pairs) { a.bn = 512; a.half = 256; }
    const int cluster = narrow_pairs ? 2 * p.ncta : p.ncta;
    // option tc_tile_pair: two 128-row tiles per CTA sharing one weight slab (a third fewer bytes per MMA).
    // Measured no gain (SSRN/HC_11: 1.27 vs 1.26 ms), like TMA multicast and a deeper pipeline.
    const bool pair = h->opt.tc_tile_pair != 0;
    const int mt = (cg == 1 && pair && !win.jptr && TT == 128 && TB == 1 && tiles * p.ncta >= 4 * 148) ? 2 : 1;
    const bool occ2 = occ2_mode && cg == 1 && mt == 1 && !win.jptr && TT == 128 && TB == 1 && tiles * p.ncta >= 148;
    const int bk = (mt == 2 || occ2 || narrow_pairs) ? 32 : (cg == 2 ? 64 : tc_bk());
    a.ntaps = p.ntaps; a.kb_per_tap = p.kb_per_tap * (64 / bk);
    if (p.mode == 2) { a.shifts[0] = 0; a.shifts[1] = -1; }
    else {
        const int tot = (l.size - 1) * rate, left = causal ? tot : tot / 2;
        for (int j = 0; j < l.size; ++j) a.shifts[j] = j * rate - left + extra_shift;
    }
    // decode-window launches: two stages keep the CTA under half an SM's shared memory, so two of them co-reside
    a.stages = std::min(narrow_pairs ? 3 : ((occ2 || win.jptr) ? 2 : tc_stages_for(p.bn, bk, mt)), std::max(1, a.ntaps * a.kb_per_tap));   // p.bn = weight rows staged per CTA
    a.TT = TT; a.TB = TB; a.tiles_t = tiles_t; a.ntiles = tiles; a.win = win;
    a.X = X; a.out = out; a.out_f32 = out_f32; a.ld_f32 = ld_f32; a.sig_f32 = sig_f32; a.ld_sig = ld_sig; a.sig = sig;
    // the A tile is identical in all CTAs of the cluster: fetch it once (TMA multicast) when the
    // tile is 128 consecutive time rows, each CTA contributing 128/ncta of them
    const bool no_mcast = h->opt.tc_mcast == 0;
    a.mcast = (!no_mcast && cg == 1 && p.ncta > 1 && TT == 128 && TB == 1) ? 1 : 0;
    const int box_rows = a.mcast ? TT / p.ncta : TT;
    CUtensorMap mAh, mAl;
    tc_make_act_map(&mAh, X.hi, l.cin, X.ld, win.L, win.B, box_rows, TB, bk);
    tc_make_act_map(&mAl, X.lo, l.cin, X.ld, win.L, win.B, box_rows, TB, bk);
    // option tc_debug: progress markers in host-mapped memory, dumped after a synchronising launch
    const bool debug = h->opt.tc_debug != 0;
    static int* dbg_host = nullptr;
    if (debug) {
        if (!dbg_host) CUDA_CHECK(cudaHostAlloc(&dbg_host, 16 * 64 * sizeof(int), cudaHostAllocMapped));
        memset(dbg_host, 0, 16 * 64 * sizeof(int));
        CUDA_CHECK(cudaHostGetDevicePointer(&a.dbg, dbg_host, 0));
        fprintf(stderr, "[tc] %s mode=%d ncta=%d bn=%d half=%d stages=%d nkb=%d tiles=%d TT=%d TB=%d L=%d B=%d\n", l.scope.c_str(),
                a.mode, p.ncta, a.bn, a.half, a.stages, a.ntaps * a.kb_per_tap, tiles, TT, TB, win.L, win.B);
    }
    CUtensorMap mWh = p.mWhi, mWl = p.mWlo;
    if (cg == 2) { tc_make_w_map(&mWh, p.Whi, p.Ktot, p.nrows, a.half / 2, bk); tc_make_w_map(&mWl, p.Wlo, p.Ktot, p.nrows, a.half / 2, bk); }   // gate / info boxes
    else if (bk != tc_bk()) { tc_make_w_map(&mWh, p.Whi, p.Ktot, p.nrows, p.bn, bk); tc_make_w_map(&mWl, p.Wlo, p.Ktot, p.nrows, p.bn, bk); }
    // hc on full sequences: the residual tile comes in by TMA and the output planes leave by TMA (staged in the
    // same drained pipeline stage), instead of row-scattered 32-byte loads / stores from the epilogue threads
    const bool no_rtma = h->opt.tc_resid_tma == 0;
    CUtensorMap io[4];
    a.resid_tma = 0;
    a.out_tma = 0;
    if (!no_rtma && p.mode == 1 && cg == 1 && mt == 1 && TT == 128 && TB == 1 && (a.half % 64) == 0 &&
        2 * a.half * 128 * 2 <= 2 * 128 * bk * 2 + 2 * a.bn * bk * 2) {
        a.resid_tma = 1;
        // TMA stores only on full sequences: in the decode window the tile starts at a negative time coordinate
        // (measured: the launch traps), and there the few output rows are cheap to store directly
        a.out_tma = (out.hi && !win.jptr) ? 1 : 0;
        tc_make_act_map(&io[0], X.hi, l.cin, X.ld, win.L, win.B, 128, 1, 64);
        tc_make_act_map(&io[1], X.lo, l.cin, X.ld, win.L, win.B, 128, 1, 64);
        if (a.out_tma) {
            tc_make_act_map(&io[2], out.hi, l.cout, out.ld, win.L, win.B, 128, 1, 64);
            tc_make_act_map(&io[3], out.lo, l.cout, out.ld, win.L, win.B, 128, 1, 64);
        } else { io[2] = io[0]; io[3] = io[1]; }
    }
    launch_conv_ln_tc(mAh, mAl, mWh, mWl, a.resid_tma ? io : nullptr, a, cluster, (tiles + mt * cg - 1) / (mt * cg), bk, mt, cg,
                      lc.s); lc.count();
    if (debug) {
        cudaError_t e = cudaStreamSynchronize(lc.s);
        for (int c = 0; c < std::min(16, p.ncta * tiles); ++c)
            fprintf(stderr, "[tc]  cta %2d: start=%d tmem=0x%x nkb=%d tma=%d mma=%d acc_ready=%d published=%d combined=%d\n", c,
                    dbg_host[64 * c], dbg_host[64 * c + 1], dbg_host[64 * c + 2], dbg_host[64 * c + 3], dbg_host[64 * c + 4],
                    dbg_host[64 * c + 5], dbg_host[64 * c + 6], dbg_host[64 * c + 7]);
        {
            const int* d0 = dbg_host;      // SM-clock deltas of CTA 0
            auto dt = [&](int a_, int b_) { return (d0[b_] - d0[a_]) & 0x7fffffff; };
            fprintf(stderr, "[tc]  cta 0 cycles: setup %d | main loop %d | sweeps1+2 %d | cluster barrier %d | sweep3+stores %d | teardown %d | total %d\n",
                    dt(8, 9), dt(9, 10), dt(10, 11), dt(11, 12), dt(12, 13), dt(13, 14), dt(8, 14));
        }
        if (e != cudaSuccess) throw std::runtime_error(std::string("conv_ln_tc failed: ") + cudaGetErrorString(e));
    }
}

bool chain_tc_ok(H* h, const std::vector<LayerDev>& net) {
    if (h->tensor_path != 1) return false;
    for (auto& l : net) if (!l.tc.ok) return false;
    return true;
}

// Whole chain on the tensor-core path, starting from split planes `cur` (buffer index `which`
// of the ping-pong pair, or -1 for an external buffer): ... -> fp32 out (+ sigmoid).
void run_chain_tc_planes(Launch& lc, const std::vector<LayerDev>& net, Planes cur, int which, int B, int L,
                         float* out, float* out_sig, int first_extra_shift) {
    H* h = lc.h;
    int len = L;
    int nxt = (which == 0) ? 1 : 0;
    for (size_t i = 0; i < net.size(); ++i) {
        const LayerDev& l = net[i];
        const bool last = (i + 1 == net.size());
        Planes dst = last ? Planes{} : ws_planes(h, nxt, l.cout);
        run_block_tc(lc, l, l.rate, l.causal, l.act, cur, RowWin{B, len, len, nullptr}, 128, 1, (len + 127) / 128,
                     dst, last ? out : nullptr, l.cout, last ? out_sig : nullptr, l.cout, Planes{},
                     i == 0 ? first_extra_shift : 0);
        if (l.kind == K_D) len *= 2;
        cur = dst; nxt ^= 1;
    }
}

// fp32 in -> planes -> chain
void run_chain_full_tc(Launch& lc, const std::vector<LayerDev>& net, const float* X, int ldx, int B, int L,
                       float* out, float* out_sig) {
    H* h = lc.h;
    Planes cur = ws_planes(h, 0, net[0].cin);
    launch_f32_to_planes(X, ldx, cur, (long long)B * L, net[0].cin, lc.s); lc.count();
    run_chain_tc_planes(lc, net, cur, 0, B, L, out, out_sig, 0);
}

void run_attention(Launch& lc, const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                   RowWin win, int N, const int* pma, float* R, float* align, long long* maxatt,
                   int* p_next, int* p_hist, Planes Rpl = Planes{}) {
    H* h = lc.h;
    REQUIRE(N <= h->key_cap, "attention: N = " + std::to_string(N) + " exceeds the handle's key capacity (" + std::to_string(h->key_cap) + ")");
    REQUIRE(h->hp.d <= 256, "attention: d exceeds 256");
    AttnArgs a{};
    a.Q = Q; a.ldq = ldq; a.K = K; a.ldk = ldk; a.V = V; a.ldv = ldv;
    a.r_hi = Rpl.hi; a.r_lo = Rpl.lo; a.ldr_h = Rpl.ld;
    a.Rout = R; a.ldr = 2 * h->hp.d; a.align = align; a.maxatt = maxatt; a.pma = pma;
    a.p_next = p_next; a.p_hist = p_hist; a.N = N; a.d = h->hp.d; a.win_size = h->hp.attention_win_size;
    a.win = win;
    launch_attention(a, lc.s); lc.count();
}

// Full-sequence attention on the tensor cores (kernels_attn_tc.cu): dense or with the monotonic
// window.  Q, K, V are fp32 device tensors; their split planes are built here.
bool attention_tc_ok(H* h, int N) { return h->tensor_path == 1 && h->hp.d == 256 && N <= h->key_cap; }

void run_attention_tc(Launch& lc, const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv, int B, int T,
                      int N, const int* pma, float* R, float* align, long long* maxatt, Planes Rpl) {
    H* h = lc.h;
    const int d = h->hp.d, NP = attn_tc_padded_keys(N);
    const size_t need[3] = {(size_t)B * T * d * sizeof(__half), (size_t)B * N * d * sizeof(__half), (size_t)B * d * NP * sizeof(__half)};
    for (int i = 0; i < 6; ++i)
        if (h->attpl[i].bytes < need[i / 2]) { CUDA_CHECK(cudaDeviceSynchronize()); h->attpl[i].ensure(need[i / 2]); }
    Planes qp, kp, vp;
    qp.hi = h->attpl[0].as<__half>(); qp.lo = h->attpl[1].as<__half>(); qp.ld = d;
    kp.hi = h->attpl[2].as<__half>(); kp.lo = h->attpl[3].as<__half>(); kp.ld = d;
    vp.hi = h->attpl[4].as<__half>(); vp.lo = h->attpl[5].as<__half>(); vp.ld = NP;
    launch_f32_to_planes(Q, ldq, qp, (long long)B * T, d, lc.s); lc.count();
    launch_attn_kv_planes(K, ldk, V, ldv, kp, vp, B, N, d, lc.s); lc.count();
    AttnTcArgs a{};
    a.Q = Q; a.ldq = ldq; a.R = R; a.ldr = 2 * d; a.Rpl = Rpl; a.align = align; a.maxatt = maxatt; a.pma = pma;
    a.T = T; a.N = N; a.d = d; a.win_size = h->hp.attention_win_size; a.scale = 1.0f / std::sqrt((float)d);
    launch_attention_tc(qp, kp, vp, a, B, lc.s); lc.count();
}

void run_textenc(Launch& lc, const int* L, int B, float* kv_out /* (B,N,2d) */) {
    H* h = lc.h;
    const int N = h->hp.max_N;
    float* emb = h->act1.as<float>();
    // park the embedding at the far end of act1 so the ping-pong (which starts on act0) never
    // overwrites it before the first block has consumed it
    launch_embed(L, h->embed_table, emb, B * N, h->hp.e, lc.s); lc.count();
    // first block reads act1 and writes act0, and so on
    run_chain_full(lc, h->textenc, emb, h->hp.e, B, N, kv_out, nullptr);
}

// Receptive-field pyramid of AudioDec for ONE new frame (SURVEY.md App. A / Q1): number of
// trailing rows each block must (re)compute at every AR step.
std::vector<int> audiodec_rows(const std::vector<LayerDev>& net, int T) {
    std::vector<int> rows(net.size(), 1);
    int need = 1;   // rows of this layer's OUTPUT needed
    for (int i = (int)net.size() - 1; i >= 0; --i) {
        rows[i] = std::min(need, T);
        need += (net[i].size - 1) * net[i].rate;    // rows of its input needed
    }
    return rows;
}

// One AR step (synthesize.py:48-54 restated incrementally, exact w.r.t. the reference's
// full recompute): AudioEnc row j, attention over the AudioDec receptive field under the
// CURRENT window, AudioDec pyramid, Y[j] = sigmoid(logits[j]), p <- argmax of row j, j <- j+1.
void run_ar_step(Launch& lc, int B) {
    H* h = lc.h;
    const dctts_hparams& hp = h->hp;
    const int T = hp.max_T, N = hp.max_N, d = hp.d;
    IntBufs ib = ints(h);
    // AudioEnc: one new row per utterance; first block reads Y[j-1] (train.py:51)
    const float* cur = h->ybuf.as<float>(); int ld = hp.n_mels;
    for (size_t i = 0; i < h->audioenc.size(); ++i) {
        const LayerDev& l = h->audioenc[i];
        float* dst = h->ae_out[i].as<float>();
        run_block(lc, l, l.rate, l.causal, l.act, cur, ld, RowWin{B, T, 1, ib.j}, dst, l.cout, nullptr, 0,
                  i == 0 ? -1 : 0);
        cur = dst; ld = l.cout;
    }
    const float* Q = cur;
    std::vector<int> rows = audiodec_rows(h->audiodec, T);
    const int att_rows = std::min(T, rows[0] + (h->audiodec[0].size - 1) * h->audiodec[0].rate);
    const float* K = h->kv.as<float>();
    // Large batches run the wide part of the AudioDec pyramid (85..59 rows per utterance) on the
    // tensor cores, one 128-row tile per utterance ending at row j; the narrow tail and the
    // one-row AudioEnc stay on the latency-oriented fp32 kernels.
    auto on_tc = [&](size_t i) { return h->tensor_path == 1 && B >= 8 && i < 4 && rows[i] >= 32 && h->audiodec[i].tc.ok; };
    auto ar_planes = [&](int idx, int C) {
        Planes p; p.hi = h->arpl[2 * idx].as<__half>(); p.lo = h->arpl[2 * idx + 1].as<__half>(); p.ld = C; return p;
    };
    Planes Rpl = on_tc(0) ? ar_planes(0, 2 * d) : Planes{};
    run_attention(lc, Q, d, K, 2 * d, K + d, 2 * d, RowWin{B, T, att_rows, ib.j}, N, ib.p_cur,
                  h->rbuf.as<float>(), nullptr, nullptr, ib.p_next, ib.p_hist, Rpl);
    cur = h->rbuf.as<float>(); ld = 2 * d;
    Planes cur_pl = Rpl;
    for (size_t i = 0; i < h->audiodec.size(); ++i) {
        const LayerDev& l = h->audiodec[i];
        const bool last = (i + 1 == h->audiodec.size());
        float* dst = h->ad_out[i].as<float>();
        if (on_tc(i)) {
            const bool next_tc = (i + 1 < h->audiodec.size()) && on_tc(i + 1);
            Planes outp = next_tc ? ar_planes((int)i + 1, l.cout) : Planes{};
            run_block_tc(lc, l, l.rate, l.causal, l.act, cur_pl, RowWin{B, T, rows[i], ib.j}, 128, 1, 1, outp,
                         next_tc ? nullptr : dst, l.cout, nullptr, 0, Planes{});
            cur_pl = outp;
        } else {
            run_block(lc, l, l.rate, l.causal, l.act, cur, ld, RowWin{B, T, rows[i], ib.j}, dst, l.cout,
                      last ? h->ybuf.as<float>() : nullptr, hp.n_mels);
        }
        cur = dst; ld = l.cout;
    }
    launch_ar_advance(ib.p_cur, ib.p_next, ib.j, B, lc.s); lc.count();
    // keep the window used by this step for the optional final alignment pass
}

void build_ar_graph(H* h, int B) {
    if (h->ar_exec && h->ar_B == B) return;
    if (h->ar_exec) { cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; }
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    cudaGraph_t graph = nullptr;
    int64_t before = h->launches;
    CUDA_CHECK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    try {
        Launch lc{h, h->stream};
        run_ar_step(lc, B);
    } catch (...) {
        cudaStreamEndCapture(h->stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        h->launches = before;
        throw;
    }
    CUDA_CHECK(cudaStreamEndCapture(h->stream, &graph));
    h->ar_nodes = h->launches - before;
    h->launches = before;
    cudaError_t e = cudaGraphInstantiate(&h->ar_exec, graph, 0);
    cudaGraphDestroy(graph);
    CUDA_CHECK(e);
    CUDA_CHECK(cudaGetLastError());
    h->ar_B = B;
}

// The whole AR loop as one persistent launch (kernels_decode.cu).  Returns false when this handle / device cannot run it.
bool decode_cluster(H* h, int B, int steps, cudaStream_t s) {
    auto& D = h->dec;
    if (!D.ok || h->opt.decode_mode != 1) return false;
    const dctts_hparams& hp = h->hp;
    IntBufs ib = ints(h);
    DecParams P = D.tab;
    for (int li = 0; li < P.nl; ++li) {
        const bool enc = li < P.n_enc;
        P.out_hist[li] = enc ? h->ae_out[li].as<float>() : h->ad_out[li - P.n_enc].as<float>();
        P.in_hist[li] = li == 0 ? nullptr : (li == P.n_enc ? h->rbuf.as<float>() : P.out_hist[li - 1]);
    }
    P.kv = h->kv.as<float>(); P.ybuf = h->ybuf.as<float>(); P.rbuf = h->rbuf.as<float>(); P.pre_scr = D.scr.as<float>();
    P.p_hist = ib.p_hist; P.p_final = D.pfinal.as<int>(); P.stats = D.stats.as<int>();
    P.prof = nullptr;
    if (h->opt.decode_prof) { D.prof.ensure(16 * sizeof(long long)); CUDA_CHECK(cudaMemsetAsync(D.prof.p, 0, 16 * sizeof(long long), s)); P.prof = D.prof.as<long long>(); }
    P.B = B;
    {   // utterances per cluster: the fewest that let every cluster be co-resident (a second wave doubles the time)
        const int mc = std::max(1, D.max_clusters);
        int G = 1;
        while (G < DEC_GMAX && (B + G - 1) / G > mc) ++G;
        P.G = G;
    }
    P.T = hp.max_T; P.N = hp.max_N; P.d = hp.d; P.n_mels = hp.n_mels;
    P.win_size = hp.attention_win_size; P.steps = steps;
    const int n_clusters = (B + P.G - 1) / P.G;
    cudaError_t e = launch_decode_cluster(P, n_clusters, s);
    if (e != cudaSuccess) {
        // a device on which the 16-CTA cluster cannot be placed after all: remember it and let the caller take the
        // graph-per-frame loop (another GPU path, not a CPU fallback)
        cudaGetLastError();
        D.ok = false; D.why = std::string("decode_cluster_kernel launch failed: ") + cudaGetErrorString(e);
        return false;
    }
    h->launches += 1;
    D.last_clusters = n_clusters; D.last_moved_frames = -1;
    return true;
}

void text2mel_generate(H* h, const int* L, int B, int steps, float* Y, int* prev_hist,
                       long long* maxatt, float* align, cudaStream_t s) {
    const dctts_hparams& hp = h->hp;
    const int T = hp.max_T, N = hp.max_N, d = hp.d;
    if (steps <= 0 || steps > T) steps = T;
    ensure_ws(h, B);
    const bool cluster = h->dec.ok && h->opt.decode_mode == 1;
    if (!cluster) build_ar_graph(h, B);
    IntBufs ib = ints(h);
    Launch lc{h, s};
    run_textenc(lc, L, B, h->kv.as<float>());
    CUDA_CHECK(cudaMemsetAsync(h->ybuf.p, 0, (size_t)B * T * hp.n_mels * sizeof(float), s));
    CUDA_CHECK(cudaMemsetAsync(h->ibuf.p, 0, (size_t)(4 + 3 * h->ws_B + (size_t)h->ws_B * T) * sizeof(int), s));
    if (cluster && decode_cluster(h, B, steps, s)) {
        // the whole loop ran as one launch
    } else {
        if (cluster) { CUDA_CHECK(cudaStreamSynchronize(s)); build_ar_graph(h, B); }
        for (int j = 0; j < steps; ++j) {
            CUDA_CHECK(cudaGraphLaunch(h->ar_exec, s));
            h->launches += h->ar_nodes;
        }
    }
    if (Y) CUDA_CHECK(cudaMemcpyAsync(Y, h->ybuf.p, (size_t)B * T * hp.n_mels * sizeof(float),
                                      cudaMemcpyDeviceToDevice, s));
    if (prev_hist) CUDA_CHECK(cudaMemcpy2DAsync(prev_hist, (size_t)T * sizeof(int), ib.p_hist,
                                                (size_t)T * sizeof(int), (size_t)T * sizeof(int), B,
                                                cudaMemcpyDeviceToDevice, s));
    if (maxatt || align) {
        // what the LAST sess.run (j = steps-1) returns: every row under that step's window.
        // p_hist[:, steps-1] is that window; gather it into p_prev.
        CUDA_CHECK(cudaMemcpy2DAsync(ib.p_prev, sizeof(int), ib.p_hist + (steps - 1), (size_t)T * sizeof(int),
                                     sizeof(int), B, cudaMemcpyDeviceToDevice, s));
        const float* K = h->kv.as<float>();
        run_attention(lc, h->ae_out.back().as<float>(), d, K, 2 * d, K + d, 2 * d, RowWin{B, T, T, nullptr}, N,
                      ib.p_prev, h->rbuf.as<float>(), align, maxatt, nullptr, nullptr);
    }
}

void text2mel_forward(H* h, const int* L, const float* mels, const int* pma, int B, float* Y,
                      long long* maxatt, float* align, cudaStream_t s) {
    const dctts_hparams& hp = h->hp;
    const int T = hp.max_T, N = hp.max_N, d = hp.d;
    ensure_ws(h, B);
    Launch lc{h, s};
    run_textenc(lc, L, B, h->kv.as<float>());
    const float* K = h->kv.as<float>();
    if (chain_tc_ok(h, h->audioenc) && chain_tc_ok(h, h->audiodec)) {
        // tensor-core path: every block over all B*T rows as one tcgen05 kernel
        Planes mp = ws_planes(h, 0, hp.n_mels);
        launch_f32_to_planes(mels, hp.n_mels, mp, (long long)B * T, hp.n_mels, lc.s); lc.count();
        float* Q = h->ae_out.back().as<float>();
        run_chain_tc_planes(lc, h->audioenc, mp, 0, B, T, Q, nullptr, -1);          // shift: train.py:51
        Planes Rpl; Rpl.hi = h->arpl[0].as<__half>(); Rpl.lo = h->arpl[1].as<__half>(); Rpl.ld = 2 * d;
        if (attention_tc_ok(h, N))
            run_attention_tc(lc, Q, d, K, 2 * d, K + d, 2 * d, B, T, N, pma, h->rbuf.as<float>(), align, maxatt, Rpl);
        else
            run_attention(lc, Q, d, K, 2 * d, K + d, 2 * d, RowWin{B, T, T, nullptr}, N, pma, h->rbuf.as<float>(),
                          align, maxatt, nullptr, nullptr, Rpl);
        run_chain_tc_planes(lc, h->audiodec, Rpl, -1, B, T, h->ad_out.back().as<float>(), Y, 0);
        return;
    }
    // AudioEnc over all rows, reading mels shifted by one frame (train.py:51)
    const float* cur = mels; int ld = hp.n_mels;
    for (size_t i = 0; i < h->audioenc.size(); ++i) {
        const LayerDev& l = h->audioenc[i];
        float* dst = h->ae_out[i].as<float>();
        run_block(lc, l, l.rate, l.causal, l.act, cur, ld, RowWin{B, T, T, nullptr}, dst, l.cout, nullptr, 0,
                  i == 0 ? -1 : 0);
        cur = dst; ld = l.cout;
    }
    run_attention(lc, cur, d, K, 2 * d, K + d, 2 * d, RowWin{B, T, T, nullptr}, N, pma, h->rbuf.as<float>(),
                  align, maxatt, nullptr, nullptr);
    cur = h->rbuf.as<float>(); ld = 2 * d;
    for (size_t i = 0; i < h->audiodec.size(); ++i) {
        const LayerDev& l = h->audiodec[i];
        const bool last = (i + 1 == h->audiodec.size());
        float* dst = h->ad_out[i].as<float>();
        run_block(lc, l, l.rate, l.causal, l.act, cur, ld, RowWin{B, T, T, nullptr}, dst, l.cout,
                  last ? Y : nullptr, hp.n_mels);
        cur = dst; ld = l.cout;
    }
}

// Op-level entry (modules.py signatures): fp32 in, fp32 out, on whichever path is selected.
void run_block_op(Launch& lc, const LayerDev& l, int rate, bool causal, int act, const float* x, int B, int L, float* out) {
    H* h = lc.h;
    const int Lout = (l.kind == K_D) ? 2 * L : L;
    if (h->tensor_path == 1 && l.tc.ok) {
        const size_t need = (size_t)B * L * roundup(l.cin, 8) * sizeof(__half);
        if (h->plane[0].bytes < need || h->plane[1].bytes < need) {
            CUDA_CHECK(cudaDeviceSynchronize());
            h->plane[0].ensure(need); h->plane[1].ensure(need);
        }
        Planes X = ws_planes(h, 0, l.cin);
        launch_f32_to_planes(x, l.cin, X, (long long)B * L, l.cin, lc.s); lc.count();
        run_block_tc(lc, l, rate, causal, act, X, RowWin{B, L, L, nullptr}, 128, 1, (L + 127) / 128, Planes{}, out, l.cout,
                     nullptr, 0, Planes{});
        return;
    }
    ensure_scratch(h, (size_t)B * Lout * l.ldw * sizeof(float));
    if (l.kind == K_D) run_deconv(lc, l, x, l.cin, B, L, out, l.cout);
    else run_block(lc, l, rate, causal, act, x, l.cin, RowWin{B, L, L, nullptr}, out, l.cout, nullptr, 0);
}

LayerDev* find_layer(H* h, const char* scope, int kind) {
    REQUIRE(h->committed, "parameters not committed");
    auto it = h->by_scope.find(scope ? scope : "");
    if (it == h->by_scope.end()) throw std::runtime_error(std::string("unknown scope: ") + (scope ? scope : "(null)"));
    if (it->second->kind != kind) throw std::runtime_error(std::string("scope has a different block kind: ") + scope);
    return it->second;
}

template <class Fn>
int guarded(dctts_handle h, Fn&& fn) {
    if (!h) { g_create_error = "null handle"; return 1; }
    try {
        CUDA_CHECK(cudaSetDevice(h->device));
        fn();
        CUDA_CHECK(cudaGetLastError());
        return 0;
    } catch (const std::exception& e) {
        h->err = e.what();
        cudaGetLastError();
        return 2;
    } catch (...) {
        h->err = "unknown failure";
        return 3;
    }
}

// NULL means the legacy default stream (what torch's default stream is), so calls made from a
// torch program are ordered with the surrounding torch work without extra synchronisation.
inline cudaStream_t S(dctts_handle, void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Grow the pre-LN scratch for an op-level call; a reallocation invalidates the AR graph,
// which has the old pointer baked in.
void ensure_scratch(H* h, size_t bytes) {
    bytes = std::max(bytes, (size_t)64 << 20);     // room for the skinny GEMM's split-K partials
    if (bytes <= h->scratch.bytes) return;
    CUDA_CHECK(cudaDeviceSynchronize());
    if (h->ar_exec) { cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; h->ar_B = 0; }
    h->scratch.ensure(bytes);
}

// ---------------------------------------------------------------------------- training
// One optimiser step of the reference's trainers (train.py mode "train"): num = 1 Text2Mel (graph :43-68, losses :83-99),
// num = 2 SSRN on ground-truth mels (:69-72, losses :100-108); Adam + clipping :122-132 -- fixed-size batches (BASELINE
// config 5) or length buckets at their own shape (data_load.py:122-129).  Forward = the fp32 block kernels with every pre-LN tensor kept; backward = kernels_train.cu.  Gradients, Adam
// moments and the pointers of all trained variables live in three arenas with identical offsets (the gradient arena is
// what a data-parallel all-reduce sums).  Activation / gradient rows use a leading dimension rounded to 4 floats (F = 1025).
// Per-step geometry: TextEnc runs over N rows, AudioEnc / AudioDec over T (Text2Mel), SSRN over T doubling at every
// transposed-conv block.  Only the row counts change from step to step; the buffers stay at their capacity offsets.
void train_set_geometry(H* h, int N, int T) {
    auto& tr = h->tr;
    const int nets = tr.num == 1 ? 3 : 1;
    for (int net = 0; net < nets; ++net) {
        int L = (tr.num == 1 && net == 0) ? N : T;
        for (int i = tr.first[net]; i <= tr.last[net]; ++i) {
            auto& t = tr.layers[i];
            t.L_in = L;
            if (t.l->kind == K_D) L *= 2;
            t.L = L; t.rows = (long long)tr.B * L;
        }
    }
}

// Activation workspace for steps of up to N keys (Text2Mel; ignored for SSRN) and T frames: the saved pre-LN tensors and
// block outputs, the gradient ping-pong buffers, the embedding, attention context / probabilities / score gradients and
// the tcgen05 operand planes.  Each layer's pre / out sits at the offset of the capacity shape.  Nothing here depends on
// the shape of the trained variables: the gradient / Adam / parameter arenas and the Adam entry table are untouched, so
// growing the workspace keeps the optimiser state.
void train_alloc_activations(H* h, int N, int T) {
    auto& tr = h->tr;
    const dctts_hparams& hp = h->hp;
    const int B = tr.B, d = hp.d;
    train_set_geometry(h, N, T);
    size_t pre_f = 0, out_f = 0, g_f = 0, dy_f = 0, tca_f = 0, tcb_f = 0;
    for (auto& t : tr.layers) {
        const LayerDev& l = *t.l;
        pre_f += (size_t)t.rows * l.ldw; out_f += (size_t)t.rows * t.ld_out;
        g_f = std::max(g_f, (size_t)t.rows * std::max(t.ld_out, roundup(l.cin, 4)));
        dy_f = std::max(dy_f, (size_t)t.rows * l.ldw);
        {   // operand planes of the tensor-core GEMMs: activations / gradients (plain and transposed), packed weights
            const size_t rows_in = (size_t)B * t.L_in, cmax = (size_t)roundup(std::max(l.cin, l.ldw), 8);
            tca_f = std::max(tca_f, std::max(rows_in * cmax, (size_t)l.size * B * roundup(l.cin, 8) * roundup(t.L_in, 8)));
            tcb_f = std::max(tcb_f, std::max((size_t)B * cmax * roundup(t.L_in, 8),
                                             (size_t)l.size * roundup(std::max(l.cin, l.ldw) + 255, 256) * roundup(std::max(l.cin, l.ldw), 32)));
        }
    }
    tr.pre.ensure(pre_f * sizeof(float)); tr.out.ensure(out_f * sizeof(float));
    if (tr.num == 1) {
        tr.emb.ensure((size_t)B * N * hp.e * sizeof(float)); tr.R.ensure((size_t)B * T * 2 * d * sizeof(float));
        tr.align.ensure((size_t)B * N * T * sizeof(float)); tr.dS.ensure((size_t)B * T * N * sizeof(float));
        g_f = std::max(g_f, (size_t)B * std::max(N, T) * (size_t)std::max(2 * d, hp.e));
    }
    for (auto& g : tr.gbuf) g.ensure(g_f * sizeof(float));
    tr.dy.ensure(dy_f * sizeof(float));
    tr.tc_a_hi.ensure(tca_f * sizeof(__half)); tr.tc_a_lo.ensure(tca_f * sizeof(__half));
    tr.tc_b_hi.ensure(tcb_f * sizeof(__half)); tr.tc_b_lo.ensure(tcb_f * sizeof(__half));
    tr.tc.a_hi = tr.tc_a_hi.as<__half>(); tr.tc.a_lo = tr.tc_a_lo.as<__half>(); tr.tc.a_elems = tca_f;
    tr.tc.b_hi = tr.tc_b_hi.as<__half>(); tr.tc.b_lo = tr.tc_b_lo.as<__half>(); tr.tc.b_elems = tcb_f;
    float* pre = tr.pre.as<float>(); float* out = tr.out.as<float>();
    for (auto& t : tr.layers) {
        t.pre = pre; pre += (size_t)t.rows * t.l->ldw;
        t.out = out; out += (size_t)t.rows * t.ld_out;
    }
    // inputs: each block reads the previous block's output; the first block of a network reads the embedding (TextEnc), the
    // mels shifted by one frame (AudioEnc, train.py:51; set per step), R (AudioDec) or the ground-truth mels (SSRN, per step)
    const int nets = tr.num == 1 ? 3 : 1;
    for (int net = 0; net < nets; ++net)
        for (int i = tr.first[net] + 1; i <= tr.last[net]; ++i) tr.layers[i].in = tr.layers[i - 1].out;
    if (tr.num == 1) {
        tr.layers[tr.first[0]].in = tr.emb.as<float>();
        tr.layers[tr.first[2]].in = tr.R.as<float>();
    }
    tr.cap_N = tr.num == 1 ? N : 0; tr.cap_T = T;
}

// Grows the activation workspace to hold (N, T) if it does not yet; waits for the device first (the old buffers may be
// in use by queued work).
void train_reserve(H* h, int N, int T) {
    auto& tr = h->tr;
    REQUIRE(tr.ready, "dctts_train_reserve: call dctts_train_init / dctts_train_init_ssrn first");
    if (tr.num == 2) N = 0;
    if (N <= tr.cap_N && T <= tr.cap_T) return;
    CUDA_CHECK(cudaDeviceSynchronize());
    train_alloc_activations(h, std::max(N, tr.cap_N), std::max(T, tr.cap_T));
}

void train_init(H* h, int B, float rate, int num, int T_in) {
    REQUIRE(h->committed, "dctts_train_init: parameters must be committed first");
    REQUIRE(B >= 1 && rate >= 0.f && rate < 1.f && (num == 1 || num == 2) && T_in >= 1, "dctts_train_init: bad arguments");
    auto& tr = h->tr;
    if (tr.ready && tr.B == B && tr.num == num && tr.T_in == T_in) { tr.rate = rate; return; }
    CUDA_CHECK(cudaDeviceSynchronize());
    if (h->ar_exec) { cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; h->ar_B = 0; }
    h->tensor_path = 0;            // the optimiser updates the fp32 weights only: this handle stops using the packed fp16 planes
    h->dec.ok = false; h->dec.why = "this handle has been trained: the packed decode stream is stale";
    tr.ready = false;
    const dctts_hparams& hp = h->hp;
    const int N = hp.max_N, T = T_in, d = hp.d;
    tr.layers.clear(); tr.tensors.clear();
    std::vector<std::vector<LayerDev>*> nets;
    if (num == 1) nets = {&h->textenc, &h->audioenc, &h->audiodec}; else nets = {&h->ssrn};
    size_t wt_f = 0;
    long long n_grad = 0;
    auto reserve = [&](long long n) { long long o = n_grad; n_grad += (n + 3) / 4 * 4; return o; };
    struct Off { long long W, bias, g1, b1, g2, b2; };
    std::vector<Off> offs;
    const long long table_off = num == 1 ? reserve((long long)hp.vocab_size * hp.e) : 0;
    int li = 0;
    for (size_t net = 0; net < nets.size(); ++net) {
        tr.first[net] = li;
        for (auto& l : *nets[net]) {
            H::TrainLayer t;
            t.l = &l; t.li = li++; t.ld_out = roundup(l.cout, 4);
            wt_f = std::max(wt_f, (size_t)l.size * l.ldw * roundup(l.cin, 4));
            Off o{};
            o.W = reserve((long long)l.size * l.cin * l.ldw); o.bias = reserve(l.ldw);
            o.g1 = reserve(l.cout); o.b1 = reserve(l.cout);
            if (l.kind == K_HC) { o.g2 = reserve(l.cout); o.b2 = reserve(l.cout); }
            offs.push_back(o);
            tr.layers.push_back(t);
        }
        tr.last[net] = li - 1;
    }
    tr.B = B; tr.num = num;
    tr.tc = GemmTcWs{};
    tr.cap_N = tr.cap_T = 0;
    train_alloc_activations(h, N, T);
    if (num == 1) { tr.gts.ensure((size_t)N * hp.max_T * sizeof(float)); launch_guided_attention(tr.gts.as<float>(), N, hp.max_T, h->stream); }
    tr.wT.ensure(wt_f * sizeof(float));
    tr.zeros.ensure(4096 * sizeof(float)); CUDA_CHECK(cudaMemset(tr.zeros.p, 0, 4096 * sizeof(float)));
    tr.tc_slots.ensure(2048 * sizeof(unsigned));
    tr.tc.slots = tr.tc_slots.as<unsigned>(); tr.tc.n_slots = 2048;
    tr.sums.ensure(4 * sizeof(double));
    tr.grads.ensure(n_grad * sizeof(float)); tr.mom.ensure(n_grad * sizeof(float)); tr.vel.ensure(n_grad * sizeof(float));
    CUDA_CHECK(cudaMemset(tr.grads.p, 0, n_grad * sizeof(float)));
    CUDA_CHECK(cudaMemset(tr.mom.p, 0, n_grad * sizeof(float))); CUDA_CHECK(cudaMemset(tr.vel.p, 0, n_grad * sizeof(float)));
    tr.n_grad = n_grad;
    float* G = tr.grads.as<float>(); float* M = tr.mom.as<float>(); float* V = tr.vel.as<float>();
    std::vector<AdamEntry> entries;
    // layout: 0 = the TF variable's own layout, 1 = [k][cin][ldw] with ldw > n columns, 2 = transposed conv [tap][cin][ldw] vs TF [1][k][cout][cin]
    auto reg = [&](const std::string& name, float* p, long long off, long long n, int layout = 0, int d0 = 0, int d1 = 0, int d2 = 0, int ld = 0) {
        tr.tensors[name] = H::TrainTensor{p, G + off, M + off, V + off, n, layout, d0, d1, d2, ld};
        entries.push_back(AdamEntry{p, G + off, M + off, V + off, n});
        return G + off;
    };
    if (num == 1) tr.d_table = reg("Text2Mel/TextEnc/embed_1/lookup_table", h->embed_table, table_off, (long long)hp.vocab_size * hp.e);
    for (size_t i = 0; i < tr.layers.size(); ++i) {
        auto& t = tr.layers[i]; LayerDev& l = *t.l; const Off& o = offs[i];
        const long long wn = (long long)l.size * l.cin * l.ldw;
        if (l.kind == K_D) {
            t.dW = reg(l.scope + "/conv2d_transpose/kernel", l.W, o.W, wn, 2, l.size, l.cin, l.cout, l.ldw);
            t.dbias = reg(l.scope + "/conv2d_transpose/bias", l.bias, o.bias, l.ldw, l.ldw != l.cout ? 1 : 0, 1, 1, l.cout, l.ldw);
        } else {
            t.dW = reg(l.scope + "/conv1d/kernel", l.W, o.W, wn, l.ldw != l.nconv ? 1 : 0, l.size, l.cin, l.nconv, l.ldw);
            t.dbias = reg(l.scope + "/conv1d/bias", l.bias, o.bias, l.ldw, l.ldw != l.nconv ? 1 : 0, 1, 1, l.nconv, l.ldw);
        }
        const std::string n1 = l.kind == K_HC ? "/H1" : "/normalize";
        t.dg1 = reg(l.scope + n1 + "/gamma", l.g1, o.g1, l.cout); t.db1 = reg(l.scope + n1 + "/beta", l.b1, o.b1, l.cout);
        if (l.kind == K_HC) { t.dg2 = reg(l.scope + "/H2/gamma", l.g2, o.g2, l.cout); t.db2 = reg(l.scope + "/H2/beta", l.b2, o.b2, l.cout); }
    }
    // leading dimensions of the blocks' inputs (the pointers are set by train_alloc_activations and, for the mels, per step)
    for (size_t net = 0; net < nets.size(); ++net)
        for (int i = tr.first[net] + 1; i <= tr.last[net]; ++i) tr.layers[i].ld_in = tr.layers[i - 1].ld_out;
    if (num == 1) {
        tr.layers[tr.first[0]].ld_in = hp.e;
        tr.layers[tr.first[1]].ld_in = hp.n_mels; tr.layers[tr.first[1]].extra_shift = -1; tr.layers[tr.first[1]].need_dgrad = false;
        tr.layers[tr.first[2]].ld_in = 2 * d;
    } else {
        tr.layers[0].ld_in = hp.n_mels; tr.layers[0].need_dgrad = false;
    }
    tr.entries.ensure(entries.size() * sizeof(AdamEntry));
    CUDA_CHECK(cudaMemcpy(tr.entries.p, entries.data(), entries.size() * sizeof(AdamEntry), cudaMemcpyHostToDevice));
    tr.n_entries = (int)entries.size();
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    tr.rate = rate; tr.T_in = T_in; tr.ready = true;
}

void layer_shifts(const LayerDev& l, int extra, int* shifts) {
    const int tot = (l.size - 1) * l.rate, left = l.causal ? tot : tot / 2;
    for (int j = 0; j < l.size; ++j) shifts[j] = j * l.rate - left + extra;
}

DropArgs drop_args(float rate, int li, uint32_t seed) {
    DropArgs d;
    if (rate > 0.f) {
        d.thresh = (uint32_t)std::min<double>((double)rate * 4294967296.0, 4294967295.0);
        d.scale = 1.0f / (1.0f - rate);
    }
    d.layer = (uint32_t)li; d.seed = seed;
    return d;
}

// forward of blocks [first, last], every pre-LN tensor and block output kept
void train_fwd(H* h, Launch& lc, int first, int last, int B, uint32_t seed) {
    auto& tr = h->tr;
    cudaStream_t s = lc.s;
    for (int i = first; i <= last; ++i) {
        auto& t = tr.layers[i]; const LayerDev& l = *t.l;
        ConvArgs c{};
        c.X = t.in; c.ldx = t.ld_in; c.Y = t.pre; c.ldy = l.ldw; c.bias = l.bias; c.K = l.cin; c.N = l.nconv; c.ldw = l.ldw;
        c.win = RowWin{B, t.L_in, t.L_in, nullptr};
        LnArgs n{};
        n.Y = t.pre; n.ldy = l.ldw; n.g1 = l.g1; n.b1 = l.b1; n.g2 = l.g2; n.b2 = l.b2; n.X = t.in; n.ldx = t.ld_in;
        n.out = t.out; n.ldo = t.ld_out; n.C = l.cout; n.mode = l.kind == K_HC ? 1 : 0; n.act = l.kind == K_D ? 0 : l.act;
        n.win = RowWin{B, t.L, t.L, nullptr};
        if (l.kind == K_D) {                                        // modules.py:232-239, like run_deconv
            const size_t tapsz = (size_t)l.cin * l.ldw;
            c.Lout = 2 * t.L_in; c.ostride = 2;
            c.ntaps = 2; c.taps[0] = ConvTap{l.W + 0 * tapsz, 0}; c.taps[1] = ConvTap{l.W + 2 * tapsz, -1}; c.ooff = 0;
            launch_conv_gemm(c, s, 0, false); lc.count();
            c.ntaps = 1; c.taps[0] = ConvTap{l.W + 1 * tapsz, 0}; c.ooff = 1;
            launch_conv_gemm(c, s, 0, false); lc.count();
        } else {
            c.ntaps = l.size;
            int sh[3]; layer_shifts(l, t.extra_shift, sh);
            for (int j = 0; j < l.size; ++j) { c.taps[j].W = l.W + (size_t)j * l.cin * l.ldw; c.taps[j].shift = sh[j]; }
            c.Lout = t.L; c.ostride = 1; c.ooff = 0;
            t.tc_slots = GemmTcSlots{};
            if ((h->opt.train_tc & 1) && conv_gemm_tc_ok(c, tr.tc)) lc.count(launch_conv_gemm_tc(c, tr.tc, s, &t.tc_slots));
            else { launch_conv_gemm(c, s, 0, false); lc.count(); }
        }
        if (tr.rate > 0.f) n.drop = drop_args(tr.rate, t.li, seed);      // the forward mask is applied by the LayerNorm epilogue
        launch_ln_rows(n, s); lc.count();
    }
}

// backward of blocks [first, last]: g_cur holds the gradient w.r.t. the last block's output; returns the buffer with the
// gradient w.r.t. the first block's input (g_cur and g_other alternate)
float* train_bwd(H* h, Launch& lc, int first, int last, int B, uint32_t seed, float* g_cur, float* g_other) {
    auto& tr = h->tr;
    cudaStream_t s = lc.s;
    float* dy = tr.dy.as<float>(); float* wT = tr.wT.as<float>();
    for (int i = last; i >= first; --i) {
        auto& t = tr.layers[i]; const LayerDev& l = *t.l;
        const int cin_p = roundup(l.cin, 4);
        BlockBwdArgs a{};
        a.pre = t.pre; a.ldy = l.ldw; a.gout = g_cur; a.ldg = t.ld_out; a.X = t.in; a.ldx = t.ld_in;
        a.g1 = l.g1; a.b1 = l.b1; a.g2 = l.g2; a.b2 = l.b2; a.dy = dy; a.gin = g_other;
        a.dg1 = t.dg1; a.db1 = t.db1; a.dg2 = t.dg2; a.db2 = t.db2; a.dbias = t.dbias;
        a.rows = t.rows; a.C = l.cout; a.mode = l.kind == K_HC ? 1 : 0; a.act = l.kind == K_D ? 0 : l.act;
        a.drop = drop_args(tr.rate, t.li, seed);
        launch_train_block_bwd(a, s); lc.count();
        if (t.need_dgrad) {
            if (cin_p != l.cin) CUDA_CHECK(cudaMemsetAsync(wT, 0, (size_t)l.size * l.ldw * cin_p * sizeof(float), s));   // zero pad columns
            launch_transpose_w(l.W, wT, l.size, l.cin, l.ldw, l.ldw, cin_p, s); lc.count();
        }
        ConvArgs c{};
        c.Y = g_other; c.ldy = cin_p; c.bias = tr.zeros.as<float>(); c.K = l.nconv; c.N = l.cin; c.ldw = cin_p;
        c.win = RowWin{B, t.L_in, t.L_in, nullptr}; c.Lout = t.L_in; c.ostride = 1; c.ooff = 0;
        const size_t tsz = (size_t)l.ldw * cin_p;                    // one transposed tap: [ldw rows (conv channels)][cin_p]
        WgradArgs w{};
        w.X = t.in; w.ldx = t.ld_in; w.ldw = l.ldw; w.L = t.L_in; w.K = l.cin;
        if (l.kind == K_D) {
            // rows of dy viewed as (B * L_in, 2 ldw): columns [0, C) belong to output row 2t, [ldw, ldw + C) to row 2t + 1.
            // forward: out[2t] = W0 x[t] + W2 x[t-1], out[2t+1] = W1 x[t]
            const size_t tapsz = (size_t)l.cin * l.ldw;
            w.rows = (long long)B * t.L_in; w.ldy = 2 * l.ldw; w.N = l.cout; w.ntaps = 1;
            w.dy = dy;         w.dW = t.dW + 0 * tapsz; w.shifts[0] = 0;  launch_conv_wgrad(w, s); lc.count();
            w.dy = dy;         w.dW = t.dW + 2 * tapsz; w.shifts[0] = -1; launch_conv_wgrad(w, s); lc.count();
            w.dy = dy + l.ldw; w.dW = t.dW + 1 * tapsz; w.shifts[0] = 0;  launch_conv_wgrad(w, s); lc.count();
            if (!t.need_dgrad) continue;
            // dx[u] = dyE[u] W0^T + dyE[u+1] W2^T + dyO[u] W1^T
            c.K = l.cout;
            c.X = dy; c.ldx = 2 * l.ldw; c.ntaps = 2; c.taps[0] = ConvTap{wT + 0 * tsz, 0}; c.taps[1] = ConvTap{wT + 2 * tsz, 1}; c.accumulate = 0;
            launch_conv_gemm(c, s, 0, false); lc.count();
            c.X = dy + l.ldw; c.ntaps = 1; c.taps[0] = ConvTap{wT + 1 * tsz, 0}; c.accumulate = 1;
            launch_conv_gemm(c, s, 0, false); lc.count();
        } else {
            w.rows = t.rows; w.dy = dy; w.ldy = l.ldw; w.dW = t.dW; w.N = l.nconv; w.ntaps = l.size;
            layer_shifts(l, t.extra_shift, w.shifts);
            GemmTcSlots gs{t.tc_slots.x, nullptr};                   // X's abs-max is known from the forward; dy's is computed once, for both gradients
            if ((h->opt.train_tc & 4) && conv_wgrad_tc_ok(w, B, tr.tc)) lc.count(launch_conv_wgrad_tc(w, B, tr.tc, s, &gs));
            else { launch_conv_wgrad(w, s); lc.count(); }
            if (!t.need_dgrad) continue;
            c.X = dy; c.ldx = l.ldw; c.ntaps = l.size;
            for (int j = 0; j < l.size; ++j) { c.taps[j].W = wT + (size_t)j * tsz; c.taps[j].shift = -w.shifts[j]; }
            c.accumulate = a.mode;
            GemmTcSlots gd{gs.w, t.tc_slots.w};                       // operands: dy and W^T (same magnitudes as W)
            if ((h->opt.train_tc & 2) && conv_gemm_tc_ok(c, tr.tc)) lc.count(launch_conv_gemm_tc(c, tr.tc, s, &gd));
            else { launch_conv_gemm(c, s, 0, false); lc.count(); }
        }
        std::swap(g_cur, g_other);
    }
    return g_cur;
}

void train_read_losses(H* h, float* losses_host, double n_el, double n_att, cudaStream_t s) {
    if (!losses_host) return;
    double sums[4];
    CUDA_CHECK(cudaMemcpyAsync(sums, h->tr.sums.p, sizeof(sums), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    losses_host[1] = (float)(sums[0] / n_el);
    losses_host[2] = (float)(sums[1] / n_el);
    losses_host[3] = n_att > 0 ? (float)(sums[2] / n_att) : 0.f;
    losses_host[0] = losses_host[1] + losses_host[2] + losses_host[3];
}

// Text2Mel on L (B, N) / mels (B, T, n_mels), any N <= the handle's key capacity and any T: the fixed-shape
// entry point passes (max_N, max_T), the shaped one the bucket's own extent (data_load.py:122-129, dynamic_pad=True).
void train_forward_backward(H* h, const int* L, const float* mels, int B, int N, int T, uint32_t seed, float* losses_host,
                            cudaStream_t s) {
    auto& tr = h->tr;
    REQUIRE(tr.ready && tr.num == 1 && tr.B == B, "dctts_train_step: call dctts_train_init with this batch size first");
    REQUIRE(N >= 1 && T >= 1, "dctts_train_step: bad batch shape");
    REQUIRE(N <= h->key_cap, "dctts_train_step: N = " + std::to_string(N) + " exceeds the handle's key capacity (" + std::to_string(h->key_cap) + ")");
    const dctts_hparams& hp = h->hp;
    const int d = hp.d;
    const int N_w = std::min(N, hp.max_N), T_w = std::min(T, hp.max_T);      // guided-attention window (train.py:91-95)
    train_reserve(h, N, T);
    train_set_geometry(h, N, T);
    Launch lc{h, s};
    CUDA_CHECK(cudaMemsetAsync(tr.grads.p, 0, tr.n_grad * sizeof(float), s));
    CUDA_CHECK(cudaMemsetAsync(tr.sums.p, 0, 4 * sizeof(double), s));
    gemm_tc_begin_step(tr.tc, s); tr.tc.probe = h->opt.train_probe;
    tr.layers[tr.first[1]].in = mels;
    launch_embed(L, h->embed_table, tr.emb.as<float>(), B * N, hp.e, s); lc.count();
    train_fwd(h, lc, tr.first[0], tr.last[0], B, seed);
    train_fwd(h, lc, tr.first[1], tr.last[1], B, seed);
    const float* KV = tr.layers[tr.last[0]].out;               // (B, N, 2d): K | V
    const float* Q = tr.layers[tr.last[1]].out;                // (B, T, d)
    // dense softmax attention (training: no window, networks.py:140-153): the tcgen05 kernel of the synthesis path when the
    // forward GEMMs are on the tensor cores (it does not touch the weights), else one warp per query row on CUDA cores
    if ((h->opt.train_tc & 1) && d == 256)
        run_attention_tc(lc, Q, d, KV, 2 * d, KV + d, 2 * d, B, T, N, nullptr, tr.R.as<float>(), tr.align.as<float>(), nullptr, Planes{});
    else
        run_attention(lc, Q, d, KV, 2 * d, KV + d, 2 * d, RowWin{B, T, T, nullptr}, N, nullptr, tr.R.as<float>(), tr.align.as<float>(),
                      nullptr, nullptr, nullptr);
    train_fwd(h, lc, tr.first[2], tr.last[2], B, seed);
    const auto& lastl = tr.layers[tr.last[2]];
    launch_train_loss(lastl.out, lastl.ld_out, mels, tr.gbuf[0].as<float>(), lastl.ld_out, tr.sums.as<double>(), (long long)B * T, hp.n_mels, s);
    lc.count();
    float* gR = train_bwd(h, lc, tr.first[2], tr.last[2], B, seed, tr.gbuf[0].as<float>(), tr.gbuf[1].as<float>());
    AttnBwdArgs ab{};
    ab.gR = gR; ab.Q = Q; ab.ldq = d; ab.K = KV; ab.V = KV + d; ab.ldkv = 2 * d; ab.align = tr.align.as<float>();
    ab.gts = tr.gts.as<float>(); ab.dS = tr.dS.as<float>(); ab.gQ = tr.gbuf[2].as<float>(); ab.gKV = tr.gbuf[3].as<float>();
    ab.B = B; ab.T = T; ab.N = N; ab.d = d; ab.att_scale = 1.0f / ((float)B * (float)N_w * (float)T_w);
    ab.ld_gts = hp.max_T; ab.N_w = N_w; ab.T_w = T_w;
    launch_attn_bwd(ab, tr.sums.as<double>(), s); lc.count(3);
    float* free_a = (gR == tr.gbuf[0].as<float>()) ? tr.gbuf[1].as<float>() : tr.gbuf[0].as<float>();
    train_bwd(h, lc, tr.first[1], tr.last[1], B, seed, tr.gbuf[2].as<float>(), free_a);
    float* gEmb = train_bwd(h, lc, tr.first[0], tr.last[0], B, seed, tr.gbuf[3].as<float>(), free_a);
    launch_embed_bwd(L, gEmb, tr.d_table, B * N, hp.e, s); lc.count();
    CUDA_CHECK(cudaGetLastError());
    train_read_losses(h, losses_host, (double)B * T * hp.n_mels, (double)B * N_w * T_w, s);
}

// SSRN (num = 2): ground-truth mels in, L1 + binary divergence against the linear magnitudes (train.py:100-108)
// mels (B, T, n_mels) -> mags (B, 4T, F); the fixed-shape entry point passes the T of dctts_train_init_ssrn
void train_forward_backward_ssrn(H* h, const float* mels, const float* mags, int B, int T, uint32_t seed, float* losses_host,
                                 cudaStream_t s) {
    auto& tr = h->tr;
    REQUIRE(tr.ready && tr.num == 2 && tr.B == B, "dctts_train_step_ssrn: call dctts_train_init_ssrn with this batch size first");
    REQUIRE(T >= 1, "dctts_train_step_ssrn: bad batch shape");
    train_reserve(h, 0, T);
    train_set_geometry(h, 0, T);
    Launch lc{h, s};
    CUDA_CHECK(cudaMemsetAsync(tr.grads.p, 0, tr.n_grad * sizeof(float), s));
    CUDA_CHECK(cudaMemsetAsync(tr.sums.p, 0, 4 * sizeof(double), s));
    gemm_tc_begin_step(tr.tc, s); tr.tc.probe = h->opt.train_probe;
    tr.layers[0].in = mels;
    const int last = (int)tr.layers.size() - 1;
    train_fwd(h, lc, 0, last, B, seed);
    const auto& ll = tr.layers[last];
    launch_train_loss(ll.out, ll.ld_out, mags, tr.gbuf[0].as<float>(), ll.ld_out, tr.sums.as<double>(), ll.rows, ll.l->cout, s); lc.count();
    train_bwd(h, lc, 0, last, B, seed, tr.gbuf[0].as<float>(), tr.gbuf[1].as<float>());
    CUDA_CHECK(cudaGetLastError());
    train_read_losses(h, losses_host, (double)ll.rows * ll.l->cout, 0.0, s);
}

void train_apply(H* h, long long global_step, float lr, cudaStream_t s) {
    auto& tr = h->tr;
    REQUIRE(tr.ready, "dctts_train_apply: no training state");
    const double beta1 = 0.9, beta2 = 0.999, warm = 4000.0;
    const double step = (double)(global_step + 1);
    const double lr_now = (double)(lr > 0.f ? lr : 0.001f) * std::sqrt(warm) * std::min(step * std::pow(warm, -1.5), 1.0 / std::sqrt(step));   // utils.py:141-145
    const double lr_t = lr_now * std::sqrt(1.0 - std::pow(beta2, step)) / (1.0 - std::pow(beta1, step));
    launch_adam(reinterpret_cast<const AdamEntry*>(tr.entries.p), tr.n_entries, (float)lr_t, (float)beta1, (float)beta2, 1e-8f, s);
    h->launches += 1;
    CUDA_CHECK(cudaGetLastError());
}

// librosa.effects.trim(y)[1] from the per-frame mean squares: frames within 60 dB of the loudest one
void trim_from_mse(const float* m, int nfr, int Ly, int32_t* out) {
    float mx = 0.f;
    for (int f = 0; f < nfr; ++f) mx = std::max(mx, m[f]);
    const double ref = 10.0 * std::log10(std::max(1e-10, (double)mx));
    int first = -1, last = -1;
    for (int f = 0; f < nfr; ++f) {
        const double db = 10.0 * std::log10(std::max(1e-10, (double)m[f])) - ref;
        if (db > -60.0) { if (first < 0) first = f; last = f; }
    }
    out[0] = first < 0 ? 0 : first * 512;
    out[1] = first < 0 ? 0 : std::min(Ly, (last + 1) * 512);
}

}  // namespace

// ==================================================================================== C-ABI
extern "C" {

const char* dctts_version(void) { return "dc_tts_b200 0.1.0 (sm_100a)"; }

const char* dctts_last_error(dctts_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int dctts_create(const dctts_hparams* hp, int device, dctts_handle* out) {
    if (!hp || !out) { g_create_error = "dctts_create: null argument"; return 1; }
    try {
        int ndev = 0;
        CUDA_CHECK(cudaGetDeviceCount(&ndev));
        if (device < 0 || device >= ndev) throw std::runtime_error("dctts_create: no such CUDA device (no CPU fallback exists)");
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) throw std::runtime_error("dctts_create: this library is built for sm_100a (B200) only");
        if (hp->d > 256 || hp->d % 8 || hp->e % 4 || hp->max_N < 1 || hp->max_T < 1 || hp->r != 4)
            throw std::runtime_error("dctts_create: unsupported hyper-parameters");
        if (hp->max_N > attn_tc_max_keys())
            throw std::runtime_error("dctts_create: max_N = " + std::to_string(hp->max_N) + " exceeds the attention kernels' limit of " +
                                     std::to_string(attn_tc_max_keys()) + " characters");
        std::unique_ptr<dctts_handle_s> h(new dctts_handle_s());
        h->hp = *hp; h->device = device; h->F = 1 + hp->n_fft / 2;
        h->key_cap = attn_tc_padded_keys(hp->max_N);
        CUDA_CHECK(cudaSetDevice(device));
        CUDA_CHECK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        build_tables(h.get());
        h->tickets.ensure(64 * sizeof(int));
        CUDA_CHECK(cudaMemset(h->tickets.p, 0, 64 * sizeof(int)));
        *out = h.release();
        return 0;
    } catch (const std::exception& e) {
        g_create_error = e.what();
        cudaGetLastError();
        return 2;
    }
}

int dctts_destroy(dctts_handle h) {
    if (!h) return 1;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    delete h;
    return 0;
}

int dctts_set_param(dctts_handle h, const char* tf_name, const float* data, const int64_t* shape, int32_t rank) {
    return guarded(h, [&] {
        REQUIRE(!h->committed, "parameters already committed");
        REQUIRE(tf_name && data && shape && rank >= 1 && rank <= 4, "dctts_set_param: bad arguments");
        HostParam p;
        size_t n = 1;
        for (int i = 0; i < rank; ++i) { REQUIRE(shape[i] > 0, "dctts_set_param: bad shape"); p.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
        p.data.assign(data, data + n);
        h->staged[tf_name] = std::move(p);
    });
}

int dctts_commit_params(dctts_handle h) { return guarded(h, [&] { commit_params(h); }); }

int64_t dctts_num_params(dctts_handle h) { return (h && h->committed) ? h->n_params : -1; }

int dctts_embed(dctts_handle h, const char* scope, const int32_t* ids, int32_t B, int32_t N, float* out, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        auto it = h->dev_vec.find(std::string(scope ? scope : "") + "/lookup_table");
        REQUIRE(it != h->dev_vec.end(), "dctts_embed: unknown scope");
        launch_embed(ids, it->second, out, B * N, h->hp.e, S(h, stream)); h->launches++;
    });
}

int dctts_normalize(dctts_handle h, const char* scope, const float* x, int64_t rows, int32_t C, float* out, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        auto g = h->dev_vec.find(std::string(scope ? scope : "") + "/gamma");
        auto b = h->dev_vec.find(std::string(scope ? scope : "") + "/beta");
        REQUIRE(g != h->dev_vec.end() && b != h->dev_vec.end(), "dctts_normalize: unknown scope");
        REQUIRE(C >= 1 && C <= 1056 && rows < (1ll << 31), "dctts_normalize: unsupported width");
        LnArgs n{};
        n.Y = x; n.ldy = C; n.g1 = g->second; n.b1 = b->second; n.out = out; n.ldo = C; n.C = C;
        n.mode = 0; n.act = 0; n.win = RowWin{1, (int)rows, (int)rows, nullptr};
        launch_ln_rows(n, S(h, stream)); h->launches++;
    });
}

int dctts_conv1d(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L, int32_t rate,
                 int32_t causal, int32_t act, float* out, void* stream) {
    return guarded(h, [&] {
        LayerDev* l = find_layer(h, scope, K_C);
        REQUIRE(B >= 1 && L >= 1 && rate >= 1, "dctts_conv1d: bad sizes");
        Launch lc{h, S(h, stream)};
        run_block_op(lc, *l, rate, causal != 0, act, x, B, L, out);
    });
}

int dctts_hc(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L, int32_t rate,
             int32_t causal, float* out, void* stream) {
    return guarded(h, [&] {
        LayerDev* l = find_layer(h, scope, K_HC);
        REQUIRE(B >= 1 && L >= 1 && rate >= 1, "dctts_hc: bad sizes");
        Launch lc{h, S(h, stream)};
        run_block_op(lc, *l, rate, causal != 0, 0, x, B, L, out);
    });
}

int dctts_conv1d_transpose(dctts_handle h, const char* scope, const float* x, int32_t B, int32_t L, float* out, void* stream) {
    return guarded(h, [&] {
        LayerDev* l = find_layer(h, scope, K_D);
        REQUIRE(B >= 1 && L >= 1, "dctts_conv1d_transpose: bad sizes");
        Launch lc{h, S(h, stream)};
        run_block_op(lc, *l, 1, false, 0, x, B, L, out);
    });
}

int dctts_textenc(dctts_handle h, const int32_t* L, int32_t B, float* K, float* V, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && L && K && V, "dctts_textenc: bad arguments");
        ensure_ws(h, B);
        cudaStream_t s = S(h, stream);
        Launch lc{h, s};
        run_textenc(lc, L, B, h->kv.as<float>());
        const int N = h->hp.max_N, d = h->hp.d;
        const size_t w = (size_t)d * sizeof(float);
        CUDA_CHECK(cudaMemcpy2DAsync(K, w, h->kv.as<float>(), 2 * w, w, (size_t)B * N, cudaMemcpyDeviceToDevice, s));
        CUDA_CHECK(cudaMemcpy2DAsync(V, w, h->kv.as<float>() + d, 2 * w, w, (size_t)B * N, cudaMemcpyDeviceToDevice, s));
    });
}

int dctts_audioenc(dctts_handle h, const float* Sin, int32_t B, int32_t T, float* Q, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && T >= 1 && T <= h->hp.max_T && Sin && Q, "dctts_audioenc: bad arguments (T must be <= max_T)");
        ensure_ws(h, B);
        Launch lc{h, S(h, stream)};
        run_chain_full(lc, h->audioenc, Sin, h->hp.n_mels, B, T, Q, nullptr);
    });
}

int dctts_attention(dctts_handle h, const float* Q, const float* K, const float* V, int32_t B, int32_t T, int32_t N,
                    int32_t monotonic, const int32_t* pma, float* R, float* alignments, int64_t* max_attentions,
                    void* stream) {
    return guarded(h, [&] {
        REQUIRE(B >= 1 && T >= 1 && N >= 1 && Q && K && V && R, "dctts_attention: bad arguments");
        REQUIRE(!monotonic || pma, "dctts_attention: monotonic attention needs prev_max_attentions");
        Launch lc{h, S(h, stream)};
        const int d = h->hp.d;
        if (attention_tc_ok(h, N))
            run_attention_tc(lc, Q, d, K, d, V, d, B, T, N, monotonic ? pma : nullptr, R, alignments,
                             reinterpret_cast<long long*>(max_attentions), Planes{});
        else
            run_attention(lc, Q, d, K, d, V, d, RowWin{B, T, T, nullptr}, N, monotonic ? pma : nullptr, R, alignments,
                          reinterpret_cast<long long*>(max_attentions), nullptr, nullptr);
    });
}

int dctts_audiodec(dctts_handle h, const float* R, int32_t B, int32_t T, float* Y_logits, float* Y, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && T >= 1 && T <= h->hp.max_T && R && Y, "dctts_audiodec: bad arguments (T must be <= max_T)");
        ensure_ws(h, B);
        Launch lc{h, S(h, stream)};
        run_chain_full(lc, h->audiodec, R, 2 * h->hp.d, B, T, Y_logits, Y);
    });
}

int dctts_ssrn(dctts_handle h, const float* Y, int32_t B, int32_t T, float* Z_logits, float* Z, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && T >= 1 && T <= h->hp.max_T && Y && Z, "dctts_ssrn: bad arguments (T must be <= max_T)");
        ensure_ws(h, B);
        Launch lc{h, S(h, stream)};
        run_chain_full(lc, h->ssrn, Y, h->hp.n_mels, B, T, Z_logits, Z);
    });
}

int dctts_text2mel_forward(dctts_handle h, const int32_t* L, const float* mels, const int32_t* pma, int32_t B,
                           float* Y, int64_t* max_attentions, float* alignments, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && L && mels && pma && Y, "dctts_text2mel_forward: bad arguments");
        text2mel_forward(h, L, mels, pma, B, Y, reinterpret_cast<long long*>(max_attentions), alignments, S(h, stream));
    });
}

int dctts_text2mel_generate(dctts_handle h, const int32_t* L, int32_t B, int32_t steps, float* Y, int32_t* prev_hist,
                            int64_t* max_attentions, float* alignments, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && L, "dctts_text2mel_generate: bad arguments");
        text2mel_generate(h, L, B, steps, Y, prev_hist, reinterpret_cast<long long*>(max_attentions), alignments,
                          S(h, stream));
    });
}

int dctts_synthesize_host(dctts_handle h, const int32_t* L_host, int32_t B, float* Y_host, float* Z_host) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(B >= 1 && L_host && Z_host, "dctts_synthesize_host: bad arguments");
        const dctts_hparams& hp = h->hp;
        const int T = hp.max_T, N = hp.max_N;
        ensure_ws(h, B);
        const size_t zbytes = (size_t)B * T * hp.r * h->F * sizeof(float);
        h->zbuf.ensure(zbytes);
        cudaStream_t s = h->stream;
        CUDA_CHECK(cudaMemcpyAsync(h->lbuf.p, L_host, (size_t)B * N * sizeof(int), cudaMemcpyHostToDevice, s));
        text2mel_generate(h, h->lbuf.as<int>(), B, T, nullptr, nullptr, nullptr, nullptr, s);
        if (Y_host) CUDA_CHECK(cudaMemcpyAsync(Y_host, h->ybuf.p, (size_t)B * T * hp.n_mels * sizeof(float), cudaMemcpyDeviceToHost, s));
        // SSRN in utterance chunks; the device->host copy of chunk i (copy stream) runs under the SSRN of chunk i+1.
        // Z is 3.5 MB per utterance: at PCIe rates the copy of a 32-utterance batch is as long as its SSRN.
        if (!h->copy_stream) {
            CUDA_CHECK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            for (auto& e : h->chunk_done) CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        // chunk ends: quarters of the batch (B >= 16) with the LAST quarter split again -- only the last chunk's copy is exposed,
        // and a chunk costs the SSRN a partly filled wave (measured ~0.55 ms per extra chunk at B = 32), so more, smaller chunks
        // at the front would cost more than they hide
        int ends[8], nchunk = 0;
        if (B >= 16) { for (int c = 1; c <= 3; ++c) ends[nchunk++] = (int)((long long)B * c / 4); ends[nchunk++] = (int)((long long)B * 7 / 8); ends[nchunk++] = B; }
        else if (B >= 4) { ends[nchunk++] = B / 2; ends[nchunk++] = B; }
        else ends[nchunk++] = B;
        const size_t zrow = (size_t)T * hp.r * h->F;
        Launch lc{h, s};
        int b0 = 0;
        for (int c = 0; c < nchunk; ++c) {
            const int b1 = ends[c];
            if (b1 <= b0) continue;
            float* zc = h->zbuf.as<float>() + (size_t)b0 * zrow;
            run_chain_full(lc, h->ssrn, h->ybuf.as<float>() + (size_t)b0 * T * hp.n_mels, hp.n_mels, b1 - b0, T, nullptr, zc);
            CUDA_CHECK(cudaEventRecord(h->chunk_done[c], s));
            CUDA_CHECK(cudaStreamWaitEvent(h->copy_stream, h->chunk_done[c], 0));
            CUDA_CHECK(cudaMemcpyAsync(Z_host + (size_t)b0 * zrow, zc, (size_t)(b1 - b0) * zrow * sizeof(float),
                                       cudaMemcpyDeviceToHost, h->copy_stream));
            b0 = b1;
        }
        CUDA_CHECK(cudaStreamSynchronize(h->copy_stream));
        CUDA_CHECK(cudaStreamSynchronize(s));
    });
}

int dctts_bench_block(dctts_handle h, const char* scope, int32_t B, int32_t L, int32_t iters, int32_t warmup,
                      float* ms_per_kernel, int32_t* n_kernels, void* stream) {
    return guarded(h, [&] {
        REQUIRE(h->committed, "parameters not committed");
        REQUIRE(scope && B >= 1 && L >= 1 && iters >= 1 && ms_per_kernel && n_kernels, "dctts_bench_block: bad arguments");
        auto it = h->by_scope.find(scope);
        REQUIRE(it != h->by_scope.end(), "dctts_bench_block: unknown scope");
        const LayerDev& l = *it->second;
        const int Lout = (l.kind == K_D) ? 2 * L : L;
        DevBuf x, y;
        x.ensure((size_t)B * L * l.cin * sizeof(float));
        y.ensure((size_t)B * Lout * l.cout * sizeof(float));
        cudaStream_t s = S(h, stream);
        CUDA_CHECK(cudaMemsetAsync(x.p, 0x3c, x.bytes, s));      // 0x3c3c3c3c = 0.0115 as float
        std::vector<cudaEvent_t> evs;
        std::vector<double> acc;
        int nk = 0;
        for (int i = 0; i < warmup + iters; ++i) {
            Launch lc{h, s};
            evs.clear();
            if (i >= warmup) {
                lc.evs = &evs;
                cudaEvent_t e0; CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventRecord(e0, s)); evs.push_back(e0);
            }
            run_block_op(lc, l, l.rate, l.causal, l.act, x.as<float>(), B, L, y.as<float>());
            if (i >= warmup) {
                CUDA_CHECK(cudaStreamSynchronize(s));
                nk = (int)evs.size() - 1;
                if (acc.empty()) acc.assign(nk, 0.0);
                for (int k = 0; k < nk; ++k) {
                    float ms = 0.f;
                    CUDA_CHECK(cudaEventElapsedTime(&ms, evs[k], evs[k + 1]));
                    acc[k] += ms;
                }
                for (auto e : evs) cudaEventDestroy(e);
            }
        }
        REQUIRE(nk <= 8, "dctts_bench_block: too many kernels");
        for (int k = 0; k < nk; ++k) ms_per_kernel[k] = (float)(acc[k] / iters);
        *n_kernels = nk;
        CUDA_CHECK(cudaStreamSynchronize(s));
        x.release(); y.release();
    });
}

int dctts_set_vocoder_params(dctts_handle h, int32_t hop_length, int32_t win_length, float power, float max_db,
                             float ref_db, float preemphasis, int32_t n_iter) {
    return guarded(h, [&] {
        REQUIRE(hop_length >= 1 && win_length >= 1 && win_length <= 2048 && n_iter >= 0, "dctts_set_vocoder_params: bad arguments");
        h->voc.hop = hop_length; h->voc.win = win_length; h->voc.power = power; h->voc.max_db = max_db;
        h->voc.ref_db = ref_db; h->voc.preemph = preemphasis; h->voc.n_iter = n_iter;
    });
}

int dctts_spectrogram2wav(dctts_handle h, const float* mag, int32_t B, int32_t T, int32_t n_iter, float* wav,
                          int32_t* trim_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(mag && wav && B >= 1 && T >= 2, "dctts_spectrogram2wav: bad arguments");
        REQUIRE(h->F == 1025, "dctts_spectrogram2wav: the FFT kernel is built for n_fft = 2048");
        cudaStream_t s = S(h, stream);
        const int F = h->F, win = h->voc.win, hop = h->voc.hop, Ly = hop * (T - 1), nfr = 1 + Ly / 512;
        const size_t n = (size_t)B * T * F;
        h->voc_S.ensure(n * sizeof(float)); h->voc_X.ensure(n * sizeof(float2));
        h->voc_frames.ensure((size_t)B * T * win * sizeof(float)); h->voc_mse.ensure((size_t)B * nfr * sizeof(float));
        h->voc_deemph.ensure(voc_deemph_scratch_bytes(B, T, hop));
        if (h->voc_tables_T != T || h->voc_tables_win != win || h->voc_tables_hop != hop) {
            h->voc_tw.ensure(2048 * sizeof(float2)); h->voc_window.ensure(win * sizeof(float));
            h->voc_wss.ensure((size_t)(2048 + hop * (T - 1)) * sizeof(float));
            voc_make_tables(h->voc_tw.as<float2>(), h->voc_window.as<float>(), h->voc_wss.as<float>(), T, win, hop, s);
            CUDA_CHECK(cudaGetLastError());
            h->voc_tables_T = T; h->voc_tables_win = win; h->voc_tables_hop = hop;
        }
        VocoderArgs a{};
        a.mag = mag; a.S = h->voc_S.as<float>(); a.X = h->voc_X.as<float2>(); a.frames = h->voc_frames.as<float>();
        a.wav = wav; a.mse = h->voc_mse.as<float>(); a.tw = h->voc_tw.as<float2>(); a.window = h->voc_window.as<float>();
        a.wss = h->voc_wss.as<float>(); a.deemph = h->voc_deemph.as<double>(); a.B = B; a.T = T; a.F = F; a.win = win; a.hop = hop;
        a.n_iter = n_iter < 0 ? h->voc.n_iter : n_iter;
        a.max_db = h->voc.max_db; a.ref_db = h->voc.ref_db; a.power = h->voc.power; a.preemphasis = h->voc.preemph;
        voc_run(a, s);
        h->launches += voc_launches_per_call(a.n_iter);
        CUDA_CHECK(cudaGetLastError());
        // librosa.effects.trim: frames whose energy is within 60 dB of the loudest
        std::vector<float> mse((size_t)B * nfr);
        CUDA_CHECK(cudaMemcpyAsync(mse.data(), a.mse, mse.size() * sizeof(float), cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        if (trim_host)
            for (int b = 0; b < B; ++b) trim_from_mse(mse.data() + (size_t)b * nfr, nfr, Ly, trim_host + 2 * b);
    });
}

int dctts_get_spectrograms(dctts_handle h, const float* wav, int64_t n_samples, int32_t sample_rate, float* mel, float* mag,
                           int32_t t_capacity, int32_t* t_out, int32_t* trim_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(wav && mel && mag && t_out && n_samples >= 2 && n_samples < (1ll << 30) && sample_rate > 0,
                "dctts_get_spectrograms: bad arguments");
        REQUIRE(h->F == 1025, "dctts_get_spectrograms: the FFT kernel is built for n_fft = 2048");
        cudaStream_t s = S(h, stream);
        const int n = (int)n_samples, F = h->F, win = h->voc.win, hop = h->voc.hop, n_mels = h->hp.n_mels;
        if (h->feat_sr != sample_rate || h->feat_win != win) {
            std::vector<float> w; std::vector<int> range;
            feat_make_mel_basis(sample_rate, h->hp.n_fft, n_mels, w, range);
            h->feat_melw.ensure(w.size() * sizeof(float)); h->feat_range.ensure(range.size() * sizeof(int));
            h->feat_tw.ensure(2048 * sizeof(float2)); h->feat_window.ensure(win * sizeof(float)); h->feat_wss.ensure(2048 * sizeof(float));
            CUDA_CHECK(cudaMemcpyAsync(h->feat_melw.p, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaMemcpyAsync(h->feat_range.p, range.data(), range.size() * sizeof(int), cudaMemcpyHostToDevice, s));
            voc_make_tables(h->feat_tw.as<float2>(), h->feat_window.as<float>(), h->feat_wss.as<float>(), 1, win, hop, s);   // synchronises
            h->feat_sr = sample_rate; h->feat_win = win;
        }
        // librosa.effects.trim (utils.py:36): frame energies on the device, threshold on the host
        const int nfr = 1 + n / 512;
        h->voc_mse.ensure((size_t)nfr * sizeof(float));
        feat_frame_mse(wav, h->voc_mse.as<float>(), n, nfr, s);
        std::vector<float> mse(nfr);
        CUDA_CHECK(cudaMemcpyAsync(mse.data(), h->voc_mse.p, mse.size() * sizeof(float), cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        int se[2];
        trim_from_mse(mse.data(), nfr, n, se);
        if (trim_host) { trim_host[0] = se[0]; trim_host[1] = se[1]; }
        const int len = se[1] - se[0];
        REQUIRE(len >= 2, "dctts_get_spectrograms: nothing left after trimming (silent input)");
        const int T = 1 + len / hop;
        *t_out = T;
        REQUIRE(T <= t_capacity, "dctts_get_spectrograms: output buffers too small (need 1 + n_samples / hop_length rows)");
        feat_run(wav + se[0], len, h->voc.preemph, mag, mel, h->feat_melw.as<float>(), h->feat_range.as<int>(), h->feat_tw.as<float2>(),
                 h->feat_window.as<float>(), T, F, n_mels, win, hop, h->voc.ref_db, h->voc.max_db, s);
        h->launches += 2;
        CUDA_CHECK(cudaGetLastError());
    });
}

int dctts_train_init(dctts_handle h, int32_t B, float dropout_rate) {
    return guarded(h, [&] { train_init(h, B, dropout_rate, 1, h->hp.max_T); });
}

int dctts_train_step(dctts_handle h, const int32_t* L, const float* mels, int32_t B, int64_t global_step, uint32_t seed, float lr,
                     int32_t apply, float* losses_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(L && mels && B >= 1 && global_step >= 0, "dctts_train_step: bad arguments");
        cudaStream_t s = S(h, stream);
        train_forward_backward(h, reinterpret_cast<const int*>(L), mels, B, h->hp.max_N, h->hp.max_T, seed, losses_host, s);
        if (apply) train_apply(h, global_step, lr, s);
    });
}

int dctts_train_step_shaped(dctts_handle h, const int32_t* L, int32_t N, const float* mels, int32_t T, int32_t B, int64_t global_step,
                            uint32_t seed, float lr, int32_t apply, float* losses_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(L && mels && B >= 1 && N >= 1 && T >= 1 && global_step >= 0, "dctts_train_step_shaped: bad arguments");
        cudaStream_t s = S(h, stream);
        train_forward_backward(h, reinterpret_cast<const int*>(L), mels, B, N, T, seed, losses_host, s);
        if (apply) train_apply(h, global_step, lr, s);
    });
}

int dctts_train_reserve(dctts_handle h, int32_t N, int32_t T) {
    return guarded(h, [&] {
        REQUIRE(N >= 0 && T >= 1, "dctts_train_reserve: bad arguments");
        REQUIRE(!(h->tr.ready && h->tr.num == 1 && N > h->key_cap),
                "dctts_train_reserve: N = " + std::to_string(N) + " exceeds the handle's key capacity (" + std::to_string(h->key_cap) + ")");
        train_reserve(h, N, T);
    });
}

int dctts_train_apply(dctts_handle h, int64_t global_step, float lr, void* stream) {
    return guarded(h, [&] { REQUIRE(global_step >= 0, "dctts_train_apply: bad step"); train_apply(h, global_step, lr, S(h, stream)); });
}

int dctts_train_grads(dctts_handle h, float** grads, int64_t* count) {
    return guarded(h, [&] {
        REQUIRE(h->tr.ready && grads && count, "dctts_train_grads: no training state");
        *grads = h->tr.grads.as<float>(); *count = h->tr.n_grad;
    });
}

int dctts_train_init_ssrn(dctts_handle h, int32_t B, int32_t T, float dropout_rate) {
    return guarded(h, [&] { train_init(h, B, dropout_rate, 2, T); });
}

int dctts_train_step_ssrn(dctts_handle h, const float* mels, const float* mags, int32_t B, int64_t global_step, uint32_t seed, float lr,
                          int32_t apply, float* losses_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(mels && mags && B >= 1 && global_step >= 0, "dctts_train_step_ssrn: bad arguments");
        cudaStream_t s = S(h, stream);
        train_forward_backward_ssrn(h, mels, mags, B, h->tr.T_in, seed, losses_host, s);
        if (apply) train_apply(h, global_step, lr, s);
    });
}

int dctts_train_step_ssrn_shaped(dctts_handle h, const float* mels, const float* mags, int32_t B, int32_t T, int64_t global_step, uint32_t seed,
                                 float lr, int32_t apply, float* losses_host, void* stream) {
    return guarded(h, [&] {
        REQUIRE(mels && mags && B >= 1 && T >= 1 && global_step >= 0, "dctts_train_step_ssrn_shaped: bad arguments");
        cudaStream_t s = S(h, stream);
        train_forward_backward_ssrn(h, mels, mags, B, T, seed, losses_host, s);
        if (apply) train_apply(h, global_step, lr, s);
    });
}

int dctts_train_tensor(dctts_handle h, const char* tf_name, int32_t what, float* host_out, int64_t count) {
    return guarded(h, [&] {
        REQUIRE(h->tr.ready && tf_name && host_out && what >= 0 && what <= 3, "dctts_train_tensor: bad arguments");
        auto it = h->tr.tensors.find(tf_name);
        REQUIRE(it != h->tr.tensors.end(), "dctts_train_tensor: not a variable of the network being trained");
        const auto& t = it->second;
        const long long logical = t.layout == 0 ? t.n : (long long)t.d0 * t.d1 * t.d2;
        REQUIRE(count == logical, "dctts_train_tensor: element count mismatch");
        const float* src = what == 0 ? t.p : what == 1 ? t.g : what == 2 ? t.m : t.v;
        CUDA_CHECK(cudaDeviceSynchronize());
        if (t.layout == 0) {
            CUDA_CHECK(cudaMemcpy(host_out, src, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost));
            return;
        }
        std::vector<float> tmp((size_t)t.n);
        CUDA_CHECK(cudaMemcpy(tmp.data(), src, tmp.size() * sizeof(float), cudaMemcpyDeviceToHost));
        if (t.layout == 1) {                                  // [d0][d1][ld] -> [d0][d1][d2]
            for (long long r = 0; r < (long long)t.d0 * t.d1; ++r)
                std::copy(tmp.begin() + r * t.ld, tmp.begin() + r * t.ld + t.d2, host_out + r * t.d2);
        } else {                                              // device [tap][cin][ld] -> TF [1][tap][cout][cin]
            for (int j = 0; j < t.d0; ++j)
                for (int co = 0; co < t.d2; ++co)
                    for (int ci = 0; ci < t.d1; ++ci)
                        host_out[((size_t)j * t.d2 + co) * t.d1 + ci] = tmp[((size_t)j * t.d1 + ci) * t.ld + co];
        }
    });
}

// Inverse of dctts_train_tensor: upload a variable (what = 0), its Adam first (2) or second (3) moment from the TF layout --
// what Supervisor's restore does for a resumed run (train.py:144; ADVICE r1: training could not resume).
int dctts_train_set_tensor(dctts_handle h, const char* tf_name, int32_t what, const float* host_in, int64_t count) {
    return guarded(h, [&] {
        REQUIRE(h->tr.ready && tf_name && host_in && (what == 0 || what == 2 || what == 3), "dctts_train_set_tensor: bad arguments");
        auto it = h->tr.tensors.find(tf_name);
        REQUIRE(it != h->tr.tensors.end(), "dctts_train_set_tensor: not a variable of the network being trained");
        const auto& t = it->second;
        const long long logical = t.layout == 0 ? t.n : (long long)t.d0 * t.d1 * t.d2;
        REQUIRE(count == logical, "dctts_train_set_tensor: element count mismatch");
        float* dst = what == 0 ? t.p : what == 2 ? t.m : t.v;
        CUDA_CHECK(cudaDeviceSynchronize());
        if (t.layout == 0) {
            CUDA_CHECK(cudaMemcpy(dst, host_in, (size_t)count * sizeof(float), cudaMemcpyHostToDevice));
            return;
        }
        std::vector<float> tmp((size_t)t.n, 0.f);
        if (t.layout == 1) {                                  // [d0][d1][d2] -> [d0][d1][ld]
            for (long long r = 0; r < (long long)t.d0 * t.d1; ++r)
                std::copy(host_in + r * t.d2, host_in + (r + 1) * t.d2, tmp.begin() + r * t.ld);
        } else {                                              // TF [1][tap][cout][cin] -> device [tap][cin][ld]
            for (int j = 0; j < t.d0; ++j)
                for (int co = 0; co < t.d2; ++co)
                    for (int ci = 0; ci < t.d1; ++ci)
                        tmp[((size_t)j * t.d1 + ci) * t.ld + co] = host_in[((size_t)j * t.d2 + co) * t.d1 + ci];
        }
        CUDA_CHECK(cudaMemcpy(dst, tmp.data(), tmp.size() * sizeof(float), cudaMemcpyHostToDevice));
    });
}

int dctts_reserve(dctts_handle h, int32_t max_batch) {
    return guarded(h, [&] { REQUIRE(max_batch >= 1, "dctts_reserve: bad batch"); ensure_ws(h, max_batch); });
}

int64_t dctts_launch_count(dctts_handle h) { return h ? h->launches : -1; }

// CRC-32C (polynomial 0x1EDC6F41, reflected 0x82F63B78), slicing-by-8 on the host.
uint32_t dctts_crc32c(uint32_t crc, const void* data, int64_t n) {
    struct Table {
        uint32_t T[8][256];
        Table() {
            for (uint32_t i = 0; i < 256; ++i) {
                uint32_t c = i;
                for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0x82F63B78u : (c >> 1);
                T[0][i] = c;
            }
            for (uint32_t i = 0; i < 256; ++i)
                for (int t = 1; t < 8; ++t) T[t][i] = (T[t - 1][i] >> 8) ^ T[0][T[t - 1][i] & 0xffu];
        }
    };
    static const Table tab;                 // C++11: initialised once, thread-safe
    const auto& T = tab.T;
    const uint8_t* p = static_cast<const uint8_t*>(data);
    uint32_t c = ~crc;
    while (n > 0 && (reinterpret_cast<uintptr_t>(p) & 7u)) { c = (c >> 8) ^ T[0][(c ^ *p++) & 0xffu]; --n; }
    while (n >= 8) {
        uint64_t v;
        memcpy(&v, p, 8);
        const uint32_t lo = (uint32_t)v ^ c, hi = (uint32_t)(v >> 32);
        c = T[7][lo & 0xffu] ^ T[6][(lo >> 8) & 0xffu] ^ T[5][(lo >> 16) & 0xffu] ^ T[4][lo >> 24] ^
            T[3][hi & 0xffu] ^ T[2][(hi >> 8) & 0xffu] ^ T[1][(hi >> 16) & 0xffu] ^ T[0][hi >> 24];
        p += 8; n -= 8;
    }
    while (n-- > 0) c = (c >> 8) ^ T[0][(c ^ *p++) & 0xffu];
    return ~c;
}

int dctts_set_tensor_path(dctts_handle h, int32_t mode) {
    return guarded(h, [&] {
        REQUIRE(mode == 0 || mode == 1, "dctts_set_tensor_path: mode must be 0 or 1");
        REQUIRE(!(h->tr.ready && mode == 1), "dctts_set_tensor_path: this handle has been trained -- its packed fp16 weight planes "
                "are stale; load the trained variables (dctts_train_tensor) into a new handle for the tcgen05 kernel set");
        if (mode != h->tensor_path && h->ar_exec) {      // the captured AR step depends on the mode
            CUDA_CHECK(cudaDeviceSynchronize());
            cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; h->ar_B = 0;
        }
        h->tensor_path = mode;
    });
}


// Kernel-variant switches: every value selects a parity-tested code path (tests/test_gpu_variants.py); the defaults are the
// measured-best configuration.  Replaces the environment variables of round 1, which froze at first use.
static int* option_slot(dctts_handle h, const char* name) {
    const std::string n = name ? name : "";
    if (n == "tc_occ2") return &h->opt.tc_occ2;
    if (n == "tc_cg2") return &h->opt.tc_cg2;
    if (n == "tc_tile_pair") return &h->opt.tc_tile_pair;
    if (n == "tc_mcast") return &h->opt.tc_mcast;
    if (n == "tc_resid_tma") return &h->opt.tc_resid_tma;
    if (n == "tc_debug") return &h->opt.tc_debug;
    if (n == "fused_ln") return &h->opt.fused_ln;
    if (n == "decode_mode") return &h->opt.decode_mode;
    if (n == "decode_prof") return &h->opt.decode_prof;
    if (n == "train_tc") return &h->opt.train_tc;
    if (n == "train_probe") return &h->opt.train_probe;
    return nullptr;
}

int dctts_set_option(dctts_handle h, const char* name, int32_t value) {
    return guarded(h, [&] {
        if (name && std::string(name) == "pdl") { pdl_enabled() = value != 0; return; }     // process-wide launch attribute
        int* slot = option_slot(h, name);
        REQUIRE(slot, "dctts_set_option: unknown option");
        REQUIRE(value >= 0 && value <= (std::string(name) == "train_tc" ? 7 : 2), "dctts_set_option: value out of range");
        if (std::string(name) == "decode_mode" && value == 1 && !h->dec.ok && h->committed)
            throw std::runtime_error("dctts_set_option: persistent decode unavailable: " + h->dec.why);
        if (*slot != value && h->ar_exec) {                  // the captured AR step bakes the variant in
            CUDA_CHECK(cudaDeviceSynchronize());
            cudaGraphExecDestroy(h->ar_exec); h->ar_exec = nullptr; h->ar_B = 0;
        }
        *slot = value;
    });
}

int dctts_get_option(dctts_handle h, const char* name, int32_t* value) {
    return guarded(h, [&] {
        REQUIRE(value, "dctts_get_option: null output");
        if (name && std::string(name) == "pdl") { *value = pdl_enabled() ? 1 : 0; return; }
        if (name && std::string(name) == "decode_available") { *value = h->dec.ok ? 1 : 0; return; }
        if (name && std::string(name) == "key_capacity") { *value = h->key_cap; return; }
        if (name && std::string(name) == "decode_max_clusters") { *value = h->dec.max_clusters; return; }   // co-resident 16-CTA clusters
        int* slot = option_slot(h, name);
        REQUIRE(slot, "dctts_get_option: unknown option");
        *value = *slot;
    });
}

// Of the last dctts_text2mel_generate on the persistent decode path: frames in which at least one utterance of a cluster
// moved its attention window (summed over clusters), utterance-frames whose receptive field was recomputed, clusters used.
int dctts_decode_stats(dctts_handle h, int32_t* moved_frames, int32_t* moved_utterance_frames, int32_t* clusters) {
    return guarded(h, [&] {
        auto& D = h->dec;
        REQUIRE(D.last_clusters > 0, "dctts_decode_stats: no persistent decode has run on this handle");
        if (D.last_moved_frames < 0) {
            std::vector<int> st(2 * (size_t)D.last_clusters);
            CUDA_CHECK(cudaDeviceSynchronize());
            CUDA_CHECK(cudaMemcpy(st.data(), D.stats.p, st.size() * sizeof(int), cudaMemcpyDeviceToHost));
            D.last_moved_frames = 0; D.last_moved_utt = 0;
            for (int c = 0; c < D.last_clusters; ++c) { D.last_moved_frames += st[2 * c]; D.last_moved_utt += st[2 * c + 1]; }
        }
        if (moved_frames) *moved_frames = D.last_moved_frames;
        if (moved_utterance_frames) *moved_utterance_frames = D.last_moved_utt;
        if (clusters) *clusters = D.last_clusters;
    });
}

// SM-clock lap timers of the last persistent decode run with option decode_prof = 1 (cluster 0, CTA rank 0, thread 0):
// cycles[0..13] = block start / stream wait / GEMV / slot release / gather / cluster barrier / LayerNorm / mix / attention /
// recompute attention / recompute GEMM / recompute LayerNorm / recompute barriers / frame bookkeeping.
int dctts_decode_profile(dctts_handle h, int64_t* cycles, int32_t n) {
    return guarded(h, [&] {
        REQUIRE(cycles && n >= 1 && n <= 16, "dctts_decode_profile: bad arguments");
        REQUIRE(h->dec.prof.p, "dctts_decode_profile: no profiled decode has run (set option decode_prof)");
        CUDA_CHECK(cudaDeviceSynchronize());
        long long v[16];
        CUDA_CHECK(cudaMemcpy(v, h->dec.prof.p, sizeof(v), cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; ++i) cycles[i] = v[i];
    });
}

int dctts_malloc(dctts_handle h, void** ptr, int64_t bytes) {
    return guarded(h, [&] { REQUIRE(ptr && bytes > 0, "dctts_malloc: bad arguments"); CUDA_CHECK(cudaMalloc(ptr, (size_t)bytes)); });
}
int dctts_free(dctts_handle h, void* ptr) { return guarded(h, [&] { CUDA_CHECK(cudaFree(ptr)); }); }
int dctts_memcpy_h2d(dctts_handle h, void* dst, const void* src, int64_t bytes, void* stream) {
    return guarded(h, [&] { CUDA_CHECK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, S(h, stream))); });
}
int dctts_memcpy_d2h(dctts_handle h, void* dst, const void* src, int64_t bytes, void* stream) {
    return guarded(h, [&] { CUDA_CHECK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, S(h, stream))); });
}
int dctts_malloc_host(dctts_handle h, void** ptr, int64_t bytes) {
    return guarded(h, [&] { REQUIRE(ptr && bytes > 0, "dctts_malloc_host: bad arguments"); CUDA_CHECK(cudaMallocHost(ptr, (size_t)bytes)); });
}
int dctts_free_host(dctts_handle h, void* ptr) { return guarded(h, [&] { CUDA_CHECK(cudaFreeHost(ptr)); }); }
int dctts_stream_sync(dctts_handle h, void* stream) { return guarded(h, [&] { CUDA_CHECK(cudaStreamSynchronize(S(h, stream))); }); }

}  // extern "C"
