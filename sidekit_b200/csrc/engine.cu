// Extraction engine: owns the packed weights, the per-batch geometry plan and the activation
// workspace, and sequences the kernels of one Xtractor.forward(x, is_eval=True) call
// (sidekit/nnet/xvector.py:876-907) for the "halfresnet34" and "xvector" (TDNN) architectures.
#include "sidekit_b200.h"
#include "conv_umma.cuh"
#include "layers.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <string>
#include <vector>

namespace skb {

// ----------------------------------------------------------------------------- errors / counters
static thread_local char g_err[512] = "";
void set_last_error(const char* file, int line, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s:%d: %s", file, line, msg);
}
std::atomic<long long> g_launches{0};
bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("SKB_NO_PDL"); return !(e && e[0] == '1'); }();
    return on;
}

bool sync_check_enabled() {
    static const bool on = [] { const char* e = getenv("SKB_SYNC_CHECK"); return e && e[0] == '1'; }();
    return on;
}

// Optional per-category device timing (CUDA events on the launching stream) used by bench.py for the
// roofline of the dominant kernel.  Off by default: events between launches cost a little.
enum { PROF_FRONTEND = 0, PROF_STEM = 1, PROF_CONV = 2, PROF_SE = 3, PROF_POOL = 4, PROF_HEAD = 5, PROF_NCAT = 8 };
struct ProfEv { int cat; cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::vector<ProfEv> g_prof;
struct ProfScope {
    cudaStream_t st; int idx = -1;
    ProfScope(int cat, cudaStream_t s) : st(s) {
        if (!g_prof_on) return;
        ProfEv e; e.cat = cat;
        cudaEventCreate(&e.a); cudaEventCreate(&e.b);
        cudaEventRecord(e.a, st);
        g_prof.push_back(e); idx = (int)g_prof.size() - 1;
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord(g_prof[idx].b, st); }
};


// ----------------------------------------------------------------------------- small host utilities
struct HostTensor {
    const float* p = nullptr;
    std::vector<int64_t> shape;
    int64_t numel() const {
        int64_t n = 1;
        for (auto d : shape) n *= d;
        return n;
    }
};
typedef std::map<std::string, HostTensor> WeightMap;

// SKB_TRACE_ALLOC=1: report every (re)allocation of a work buffer on stderr (they synchronise the device: none may
// happen in the steady state of a bulk extraction)
static bool trace_alloc() {
    static const bool on = [] { const char* e = getenv("SKB_TRACE_ALLOC"); return e && e[0] == '1'; }();
    return on;
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes, bool* grew = nullptr) {
        if (bytes <= cap) return SKB_OK;
        if (trace_alloc()) fprintf(stderr, "skb: device buffer grows %zu -> %zu bytes\n", cap, bytes);
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            set_last_error(__FILE__, __LINE__, cudaGetErrorString(e));
            return SKB_ERR_CUDA;
        }
        cap = want;
        if (grew) *grew = true;
        return SKB_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// Pinned host staging (table uploads must not block the host: the copy is enqueued and the host goes on planning)
struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return SKB_OK;
        if (trace_alloc()) fprintf(stderr, "skb: pinned buffer grows %zu -> %zu bytes\n", cap, bytes);
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 4 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) {
            set_last_error(__FILE__, __LINE__, cudaGetErrorString(e));
            return SKB_ERR_CUDA;
        }
        cap = want;
        return SKB_OK;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

template <typename T>
static int dev_upload(const std::vector<T>& v, T** out) {
    *out = nullptr;
    const size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
    SKB_CUDA_CHECK(cudaMalloc(out, bytes));
    if (!v.empty()) SKB_CUDA_CHECK(cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SKB_OK;
}

static uint16_t to16(float v, bool bf16) {
    if (bf16) {
        __nv_bfloat16 h = __float2bfloat16_rn(v);
        uint16_t u;
        memcpy(&u, &h, 2);
        return u;
    }
    __half h = __float2half_rn(v);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

static float from16(uint16_t u, bool bf16) {
    if (bf16) {
        __nv_bfloat16 h;
        memcpy(&h, &u, 2);
        return __bfloat162float(h);
    }
    __half h;
    memcpy(&h, &u, 2);
    return __half2float(h);
}

static const HostTensor* find(const WeightMap& w, const std::string& k) {
    auto it = w.find(k);
    if (it == w.end()) {
        set_last_error(__FILE__, __LINE__, ("missing weight tensor: " + k).c_str());
        return nullptr;
    }
    return &it->second;
}

// BatchNorm (eval) as y = s*x + t  (eps 1e-5, torch default)
static int bn_affine(const WeightMap& w, const std::string& prefix, std::vector<double>* s, std::vector<double>* t) {
    const HostTensor *g = find(w, prefix + ".weight"), *b = find(w, prefix + ".bias"),
                     *m = find(w, prefix + ".running_mean"), *v = find(w, prefix + ".running_var");
    if (!g || !b || !m || !v) return SKB_ERR_WEIGHTS;
    const int64_t n = g->numel();
    s->resize(n);
    t->resize(n);
    for (int64_t i = 0; i < n; ++i) {
        const double sc = (double)g->p[i] / std::sqrt((double)v->p[i] + 1e-5);
        (*s)[i] = sc;
        (*t)[i] = (double)b->p[i] - (double)m->p[i] * sc;
    }
    return SKB_OK;
}

// ----------------------------------------------------------------------------- packed conv weights
struct ConvW {
    uint16_t* w = nullptr;   // device, UMMA images
    uint16_t* w3 = nullptr;  // device, fused-tap images (3x3 convs with 32 or 64 output channels), else nullptr
    float* bias = nullptr;   // device [cout]
    int cin = 0, cout = 0, taps = 0, ncta = 0;
    bool phase_split = false;   // stride-2 3x3 conv packed for a phase-split input (cin = 4 * original channels)
};

// wf: folded weights [cout][cin_src][taps] (double), channels >= cin_src zero padded up to cin_pad.
static int pack_conv(const std::vector<double>& wf, const std::vector<double>& bias, int cout, int cin_src, int cin_pad,
                     int taps, bool bf16, ConvW* out) {
    const int ncta = conv_pick_ncta(cout);
    const int n_split = cout / ncta, n_kc = cin_pad / kConvKC;
    std::vector<uint16_t> img((size_t)n_split * n_kc * taps * 4 * ncta * 8);
    size_t o = 0;
    for (int ns = 0; ns < n_split; ++ns)
        for (int kc = 0; kc < n_kc; ++kc)
            for (int tap = 0; tap < taps; ++tap)
                for (int j = 0; j < 4; ++j)
                    for (int n = 0; n < ncta; ++n)
                        for (int e = 0; e < 8; ++e) {
                            const int co = ns * ncta + n, ci = kc * kConvKC + j * 8 + e;
                            const double v = ci < cin_src ? wf[((size_t)co * cin_src + ci) * taps + tap] : 0.0;
                            img[o++] = to16((float)v, bf16);
                        }
    std::vector<float> bf(bias.begin(), bias.end());
    out->cin = cin_pad; out->cout = cout; out->taps = taps; out->ncta = ncta;
    int rc = dev_upload(img, &out->w);
    if (rc) return rc;
    if (taps == 9 && (cout == 32 || cout == 64) && cin_pad == cin_src) {
        // fused-tap packing (conv3_umma.cuh): per (k-chunk, vertical tap r) one image [4 planes][3 * cout rows][8], row = s * cout + co
        std::vector<uint16_t> img3((size_t)n_kc * 3 * 4 * 3 * cout * 8);
        size_t o3 = 0;
        for (int kc = 0; kc < n_kc; ++kc)
            for (int r = 0; r < 3; ++r)
                for (int j = 0; j < 4; ++j)
                    for (int sc = 0; sc < 3 * cout; ++sc)
                        for (int e = 0; e < 8; ++e) {
                            const int s_tap = sc / cout, co = sc % cout, ci = kc * kConvKC + j * 8 + e;
                            img3[o3++] = to16((float)wf[((size_t)co * cin_src + ci) * 9 + r * 3 + s_tap], bf16);
                        }
        if ((rc = dev_upload(img3, &out->w3))) return rc;
    }
    return dev_upload(bf, &out->bias);
}

// Conv2d (no bias) followed by BatchNorm2d: w' = w*s[co], b' = t[co]
static int pack_conv_bn(const WeightMap& w, const std::string& conv_key, const std::string& bn_prefix, bool bf16, ConvW* out,
                        float** w_rounded_t = nullptr) {
    const HostTensor* cw = find(w, conv_key);
    if (!cw || cw->shape.size() != 4) return SKB_ERR_WEIGHTS;
    const int cout = (int)cw->shape[0], cin = (int)cw->shape[1], taps = (int)(cw->shape[2] * cw->shape[3]);
    std::vector<double> s, t;
    int rc = bn_affine(w, bn_prefix, &s, &t);
    if (rc) return rc;
    std::vector<double> wf((size_t)cout * cin * taps);
    for (int co = 0; co < cout; ++co)
        for (size_t i = 0; i < (size_t)cin * taps; ++i) wf[(size_t)co * cin * taps + i] = (double)cw->p[(size_t)co * cin * taps + i] * s[co];
    if (w_rounded_t) {
        std::vector<float> wt((size_t)cin * taps * cout);
        for (int co = 0; co < cout; ++co)
            for (size_t i = 0; i < (size_t)cin * taps; ++i)
                wt[i * cout + co] = from16(to16((float)wf[(size_t)co * cin * taps + i], bf16), bf16);
        rc = dev_upload(wt, w_rounded_t);
        if (rc) return rc;
    }
    return pack_conv(wf, t, cout, cin, cin, taps, bf16, out);
}

// Stride-2 3x3 conv + BN packed for a phase-split (space-to-depth) input: k-chunks run phase-major, phase (a, b) =
// (h & 1, w & 1); each phase is read by its own taps: (0,0): (1,1) | (0,1): (1,0) (1,2) | (1,0): (0,1) (2,1) |
// (1,1): (0,0) (0,2) (2,0) (2,2)   [(r, s) of the original kernel].
static const int kPhaseTaps[9][2] = {{1, 1}, {1, 0}, {1, 2}, {0, 1}, {2, 1}, {0, 0}, {0, 2}, {2, 0}, {2, 2}};
static const int kPhaseTapBegin[5] = {0, 1, 3, 5, 9};

// wf: folded weights [cout][cin][9] (double), bias [cout]
static int pack_conv_phase_split(const std::vector<double>& wf, const std::vector<double>& bias, int cout, int cin, bool bf16, ConvW* out) {
    if (cin % kConvKC != 0) {
        set_last_error(__FILE__, __LINE__, "phase-split conv needs input channels in multiples of 32");
        return SKB_ERR_WEIGHTS;
    }
    const int ncta = conv_pick_ncta(cout), n_split = cout / ncta, cpp = cin / kConvKC;   // chunks per phase
    std::vector<uint16_t> img((size_t)n_split * cpp * 9 * 4 * ncta * 8);
    size_t o = 0;
    for (int ns = 0; ns < n_split; ++ns)
        for (int ph = 0; ph < 4; ++ph)
            for (int ch = 0; ch < cpp; ++ch)
                for (int tp = kPhaseTapBegin[ph]; tp < kPhaseTapBegin[ph + 1]; ++tp) {
                    const int tap = kPhaseTaps[tp][0] * 3 + kPhaseTaps[tp][1];
                    for (int j = 0; j < 4; ++j)
                        for (int n = 0; n < ncta; ++n)
                            for (int e = 0; e < 8; ++e) {
                                const int co = ns * ncta + n, ci = ch * kConvKC + j * 8 + e;
                                img[o++] = to16((float)wf[((size_t)co * cin + ci) * 9 + tap], bf16);
                            }
                }
    std::vector<float> bf(bias.begin(), bias.end());
    out->cin = 4 * cin; out->cout = cout; out->taps = 9; out->ncta = ncta; out->phase_split = true;
    int rc;
    if ((rc = dev_upload(img, &out->w))) return rc;
    return dev_upload(bf, &out->bias);
}

static int pack_conv_bn_phase_split(const WeightMap& w, const std::string& conv_key, const std::string& bn_prefix, bool bf16,
                                    ConvW* out) {
    const HostTensor* cw = find(w, conv_key);
    if (!cw || cw->shape.size() != 4 || cw->shape[2] != 3 || cw->shape[3] != 3) return SKB_ERR_WEIGHTS;
    const int cout = (int)cw->shape[0], cin = (int)cw->shape[1];
    std::vector<double> s, t;
    int rc = bn_affine(w, bn_prefix, &s, &t);
    if (rc) return rc;
    std::vector<double> wf((size_t)cout * cin * 9);
    for (int co = 0; co < cout; ++co)
        for (size_t i = 0; i < (size_t)cin * 9; ++i) wf[(size_t)co * cin * 9 + i] = (double)cw->p[(size_t)co * cin * 9 + i] * s[co];
    return pack_conv_phase_split(wf, t, cout, cin, bf16, out);
}

static void free_conv(ConvW* c) {
    cudaFree(c->w);
    cudaFree(c->w3);
    cudaFree(c->bias);
    *c = ConvW();
}

// ----------------------------------------------------------------------------- models
struct BlockW {
    ConvW conv1, conv2, sc;
    bool has_sc = false;
    int stride = 1, C = 0;
    int layer = 1, index = 0;  // "layer<layer>.<index>" in the reference's module tree (debug stage names)
    bool level_up = false;     // first block of a layer that widens WITHOUT striding (fastresnet34 layer4): next level, same geometry
    float *se_w1 = nullptr, *se_w2 = nullptr;
    float* w2t = nullptr;      // conv2's folded weights as the tensor cores see them (16-bit rounded), fp32 [9*Cin][Cout]
};

struct Model {
    int archi = 0;
    bool bf16 = false;
    int emb = 0, n_spk = 0;
    float margin_s = 30.f;
    FrontendConsts fe;
    // halfresnet34
    StemConsts stem;            // folded stem conv + BN (host copy: passed to the kernel by value)
    int stem_c = 32;            // stem output channels: 32 (halfresnet34) or 128 (resnet34)
    int level_C[4] = {32, 64, 128, 256};   // channels of the four resolution levels (W = 80, 40, 20, 10)
    bool head_bn = true;        // before_speaker_embedding = Linear(no bias) + BatchNorm1d (halfresnet34) or a plain Linear (resnet34)
    int level_W[4] = {80, 40, 20, 10};     // width (frequency bins) of the four levels
    bool level_halves[4] = {false, true, true, true};   // does level l halve the time axis of level l-1
    bool global_context = true; // attentive pooling input = [x ; mean ; std] (halfresnet34 / resnet34) or x alone (fastresnet34)
    std::vector<BlockW> blocks;
    float *att_w1x = nullptr, *att_w1g = nullptr, *att_b1 = nullptr, *att_bn_s = nullptr, *att_bn_t = nullptr;
    float *att_w2 = nullptr, *att_b2 = nullptr;
    int att_A = 0, pool_D = 0;
    // head
    float *lin_w = nullptr, *lin_b = nullptr, *be_s = nullptr, *be_t = nullptr, *spk_wn = nullptr, *spk_b = nullptr;
    bool head_linear = false;   // loss='aps': logits = Linear(x) on the pre-normalisation embedding instead of s * cos(x, W)
    PackedOp p_w1x, p_w2;       // attention projections packed for the split-precision tcgen05 GEMM (M = frames)
    // tdnn
    std::vector<ConvW> tdnn;
    std::vector<int> tdnn_k, tdnn_d;
    float *pool_s = nullptr, *pool_t = nullptr;
};

static inline bool is_resnet(int archi) {
    return archi == SKB_ARCHI_HALFRESNET34 || archi == SKB_ARCHI_RESNET34 || archi == SKB_ARCHI_FASTRESNET34;
}

static int upload_f(const std::vector<double>& v, float** out) {
    std::vector<float> f(v.begin(), v.end());
    return dev_upload(f, out);
}
static int upload_raw(const HostTensor* t, float** out) {
    std::vector<float> f(t->p, t->p + t->numel());
    return dev_upload(f, out);
}

static int build_frontend(const WeightMap& w, Model* m) {
    // PreEmphasis.flipped_filter = [-coef, 1] (augmentation.py:59-62): a checkpoint trained with another coefficient is honoured
    auto pf = w.find("preprocessor.PreEmphasis.flipped_filter");
    if (pf != w.end() && pf->second.numel() == 2) {
        if (pf->second.p[1] != 1.f) {
            set_last_error(__FILE__, __LINE__, "unexpected PreEmphasis.flipped_filter (want [-coef, 1])");
            return SKB_ERR_WEIGHTS;
        }
        m->fe.preemph = -pf->second.p[0];
    }
    if (m->archi != SKB_ARCHI_XVECTOR) {
        const HostTensor *win = find(w, "preprocessor.MelSpec.spectrogram.window"), *fb = find(w, "preprocessor.MelSpec.mel_scale.fb");
        if (!win || !fb) return SKB_ERR_WEIGHTS;
        if (win->numel() != 400 || fb->shape.size() != 2 || fb->shape[0] != 513) {
            set_last_error(__FILE__, __LINE__, "unexpected log-Mel front-end buffers (want window 400, fb 513 x n_mels)");
            return SKB_ERR_WEIGHTS;
        }
        return frontend_consts_create(&m->fe, 1024, 400, 160, (int)fb->shape[1], (int)fb->shape[1], win->p, fb->p, nullptr);
    }
    const HostTensor *win = find(w, "preprocessor.MFCC.MelSpectrogram.spectrogram.window"),
                     *fb = find(w, "preprocessor.MFCC.MelSpectrogram.mel_scale.fb"), *dct = find(w, "preprocessor.MFCC.dct_mat");
    if (!win || !fb || !dct) return SKB_ERR_WEIGHTS;
    if (win->numel() != 1024 || fb->shape.size() != 2 || fb->shape[0] != 1025 || dct->shape.size() != 2 || dct->shape[0] != fb->shape[1]) {
        set_last_error(__FILE__, __LINE__, "unexpected MFCC front-end buffers");
        return SKB_ERR_WEIGHTS;
    }
    return frontend_consts_create(&m->fe, 2048, 1024, 512, (int)fb->shape[1], (int)dct->shape[1], win->p, fb->p, dct->p);
}

static int build_margin_head(const WeightMap& w, Model* m) {
    if (w.count("after_speaker_embedding.cce_backend.linear8.weight")) {
        // loss='aps' (SoftmaxAngularProto.forward(x, target=None), sidekit/nnet/loss.py:347-359): a plain Linear on the
        // (l2-normalised) embedding
        const HostTensor *lw = find(w, "after_speaker_embedding.cce_backend.linear8.weight"),
                         *lb = find(w, "after_speaker_embedding.cce_backend.linear8.bias");
        if (!lw || !lb || lw->shape.size() != 2 || lw->shape[1] != m->emb || lb->numel() != lw->shape[0]) return SKB_ERR_WEIGHTS;
        m->n_spk = (int)lw->shape[0];
        m->head_linear = true;
        int rc = upload_raw(lw, &m->spk_wn);
        if (rc) return rc;
        return upload_raw(lb, &m->spk_b);
    }
    if (!w.count("after_speaker_embedding.weight")) {   // loss='cce' / None: no head at inference time
        m->n_spk = 0;
        return SKB_OK;
    }
    const HostTensor* sw = find(w, "after_speaker_embedding.weight");
    if (!sw || sw->shape.size() != 2 || sw->shape[1] != m->emb) return SKB_ERR_WEIGHTS;
    m->n_spk = (int)sw->shape[0];
    std::vector<float> wn((size_t)m->n_spk * m->emb);
    for (int i = 0; i < m->n_spk; ++i) {   // F.normalize(weight): row / max(norm, 1e-12), loss.py:307
        double ss = 0;
        for (int k = 0; k < m->emb; ++k) ss += (double)sw->p[(size_t)i * m->emb + k] * sw->p[(size_t)i * m->emb + k];
        const double inv = 1.0 / std::max(std::sqrt(ss), 1e-12);
        for (int k = 0; k < m->emb; ++k) wn[(size_t)i * m->emb + k] = (float)(sw->p[(size_t)i * m->emb + k] * inv);
    }
    return dev_upload(wn, &m->spk_wn);
}

// fastresnet34 carries its 16-channel level with 32 channels (one K chunk of the tensor-core convolutions): the tensors of
// layer1 and the input side of layer2.0 are zero-padded here, so that the padded channels stay exactly 0 everywhere
// (zero weights, BN scale and shift 0 -> relu(0) = 0; zero SE rows) and the packing code sees ordinary 32-channel layers.
static void pad_tensor(WeightMap* w, std::deque<std::vector<float>>* store, const std::string& key, std::vector<int64_t> shape) {
    auto it = w->find(key);
    if (it == w->end()) return;
    const HostTensor src = it->second;
    if (src.shape.size() != shape.size()) return;
    int64_t n = 1;
    for (auto d : shape) n *= d;
    store->emplace_back((size_t)n, 0.f);
    std::vector<float>& dst = store->back();
    const size_t nd = shape.size();
    std::vector<int64_t> idx(nd, 0);
    for (int64_t i = 0; i < src.numel(); ++i) {
        int64_t o = 0;
        for (size_t d = 0; d < nd; ++d) o = o * shape[d] + idx[d];
        dst[(size_t)o] = src.p[i];
        for (int d = (int)nd - 1; d >= 0; --d) {
            if (++idx[d] < src.shape[d]) break;
            idx[d] = 0;
        }
    }
    HostTensor t;
    t.p = dst.data();
    t.shape = shape;
    (*w)[key] = t;
}

static void pad_fastresnet_weights(WeightMap* w, std::deque<std::vector<float>>* store) {
    const std::string sn = "sequence_network";
    for (int bi = 0; bi < 3; ++bi) {
        const std::string p = sn + ".layer1." + std::to_string(bi);
        for (const char* c : {".conv1.weight", ".conv2.weight"}) pad_tensor(w, store, p + c, {32, 32, 3, 3});
        for (const char* bn : {".bn1", ".bn2"})
            for (const char* f : {".weight", ".bias", ".running_mean", ".running_var"}) pad_tensor(w, store, p + bn + f, {32});
        pad_tensor(w, store, p + ".se.fc.0.weight", {2, 32});
        pad_tensor(w, store, p + ".se.fc.2.weight", {32, 2});
    }
    pad_tensor(w, store, sn + ".layer2.0.conv1.weight", {32, 32, 3, 3});
    pad_tensor(w, store, sn + ".layer2.0.shortcut.0.weight", {32, 32, 1, 1});
}

static int build_hr34(const WeightMap& w_in, Model* m) {
    int rc;
    WeightMap w = w_in;
    std::deque<std::vector<float>> padded;
    if (m->archi == SKB_ARCHI_FASTRESNET34) pad_fastresnet_weights(&w, &padded);
    const std::string sn = "sequence_network";
    // Trunk tables.  halfresnet34 (res_net.py:504-554): 4 layers (3,4,6,3) at 32/64/128/256 channels, strides 1,2,2,2 given
    // as TUPLES, so that `stride != 1` is true even for layer1.0 and it gets a 1x1 shortcut.  resnet34 (PreResNet34,
    // res_net.py:430-498): 7 layers (3,1,3,1,5,1,1 as built) at 128,128,128,256,256,256,256 channels with INT strides 1,2,1,2,1,2,1.
    // The shortcut of a block is simply whatever the state_dict holds.
    // fastresnet34 (PreFastResNet34, res_net.py:557-610): 7x7 stem with stride (1, 2) to 16 channels, 4 layers (3,4,6,3) at
    // 16/32/64/128 channels with strides 1 (int: no shortcut in layer1.0), (2,2), (2,2), (1,1) -- layer4 widens at the
    // resolution of layer3 (its first block has a 1x1 shortcut because the stride is the tuple (1,1)).
    const bool half = m->archi == SKB_ARCHI_HALFRESNET34, fast = m->archi == SKB_ARCHI_FASTRESNET34;
    const int n_layers = (half || fast) ? 4 : 7;
    const int planes_f[4] = {32 /* 16 padded */, 32, 64, 128}, strides_f[4] = {1, 2, 2, 1};
    const int nblocks_h[4] = {3, 4, 6, 3}, planes_h[4] = {32, 64, 128, 256}, strides_h[4] = {1, 2, 2, 2};
    const int nblocks_r[7] = {3, 1, 3, 1, 5, 1, 1} /* layer7 is built with num_blocks[5] (res_net.py:462) */, planes_r[7] = {128, 128, 128, 256, 256, 256, 256}, strides_r[7] = {1, 2, 1, 2, 1, 2, 1};
    const int* nblocks = (half || fast) ? nblocks_h : nblocks_r;
    const int* planes = half ? planes_h : (fast ? planes_f : planes_r);
    const int* lstrides = half ? strides_h : (fast ? strides_f : strides_r);
    m->stem_c = half ? 32 : (fast ? 16 : 128);
    const int stem_taps = fast ? 49 : 9;
    {   // stem: conv1 (C,1,k,k) + bn1 -> fp32 folded
        const HostTensor* cw = find(w, sn + ".conv1.weight");
        if (!cw || cw->numel() != m->stem_c * stem_taps) return SKB_ERR_WEIGHTS;
        std::vector<double> s, t;
        if ((rc = bn_affine(w, sn + ".bn1", &s, &t))) return rc;
        for (int c = 0; c < m->stem_c; ++c) {
            for (int k = 0; k < stem_taps; ++k) m->stem.w[c * stem_taps + k] = (float)((double)cw->p[c * stem_taps + k] * s[c]);
            m->stem.b[c] = (float)t[c];
        }
    }
    int level = 0;
    m->level_C[0] = fast ? 32 : m->stem_c;
    if (fast) {
        const int wf[4] = {40, 20, 10, 10};
        const bool hf[4] = {false, true, true, false};
        for (int l = 0; l < 4; ++l) { m->level_W[l] = wf[l]; m->level_halves[l] = hf[l]; }
    }
    m->global_context = !fast;
    for (int li = 0; li < n_layers; ++li)
        for (int bi = 0; bi < nblocks[li]; ++bi) {
            const std::string p = sn + ".layer" + std::to_string(li + 1) + "." + std::to_string(bi);
            BlockW b;
            b.C = planes[li];
            b.layer = li + 1;
            b.index = bi;
            b.stride = bi == 0 ? lstrides[li] : 1;
            b.level_up = bi == 0 && b.stride == 1 && b.C != m->level_C[level];
            if (b.stride == 2 || b.level_up) ++level;
            if (level > 3) return SKB_ERR_WEIGHTS;
            m->level_C[level] = b.C;
            if (b.stride == 2) {
                if ((rc = pack_conv_bn_phase_split(w, p + ".conv1.weight", p + ".bn1", m->bf16, &b.conv1))) return rc;
            } else if ((rc = pack_conv_bn(w, p + ".conv1.weight", p + ".bn1", m->bf16, &b.conv1))) return rc;
            if ((rc = pack_conv_bn(w, p + ".conv2.weight", p + ".bn2", m->bf16, &b.conv2, &b.w2t))) return rc;
            b.has_sc = w.count(p + ".shortcut.0.weight") > 0;
            if (b.has_sc && (rc = pack_conv_bn(w, p + ".shortcut.0.weight", p + ".shortcut.1", m->bf16, &b.sc))) return rc;
            const HostTensor *f0 = find(w, p + ".se.fc.0.weight"), *f2 = find(w, p + ".se.fc.2.weight");
            if (!f0 || !f2) return SKB_ERR_WEIGHTS;
            if ((rc = upload_raw(f0, &b.se_w1))) return rc;
            if ((rc = upload_raw(f2, &b.se_w2))) return rc;
            m->blocks.push_back(b);
        }
    // attentive pooling (num_channels*num_freqs = 2560, attention 128, global context)
    const HostTensor *a0w = find(w, "stat_pooling.attention.0.weight"), *a0b = find(w, "stat_pooling.attention.0.bias"),
                     *a4w = find(w, "stat_pooling.attention.4.weight"), *a4b = find(w, "stat_pooling.attention.4.bias");
    if (!a0w || !a0b || !a4w || !a4b) return SKB_ERR_WEIGHTS;
    const int A = (int)a0w->shape[0], D = (int)a4w->shape[0];
    const int in_factor = m->global_context ? 3 : 1;
    if (a0w->shape[1] != in_factor * D || D != m->level_C[3] * m->level_W[3]) {
        set_last_error(__FILE__, __LINE__, "stat_pooling.attention must be AttentivePooling(C, 10) over the trunk's C x 10 output "
                                           "(global_context=True for halfresnet34 / resnet34, False for fastresnet34)");
        return SKB_ERR_WEIGHTS;
    }
    m->att_A = A;
    m->pool_D = D;
    std::vector<float> w1x((size_t)A * D), w1g((size_t)A * 2 * D);
    for (int a = 0; a < A; ++a) {
        memcpy(&w1x[(size_t)a * D], a0w->p + (size_t)a * in_factor * D, D * sizeof(float));
        if (m->global_context) memcpy(&w1g[(size_t)a * 2 * D], a0w->p + (size_t)a * 3 * D + D, 2 * D * sizeof(float));
    }
    if ((rc = dev_upload(w1x, &m->att_w1x))) return rc;
    if (m->global_context && (rc = dev_upload(w1g, &m->att_w1g))) return rc;
    if ((rc = upload_raw(a0b, &m->att_b1))) return rc;
    std::vector<double> s, t;
    if ((rc = bn_affine(w, "stat_pooling.attention.2", &s, &t))) return rc;
    if ((rc = upload_f(s, &m->att_bn_s))) return rc;
    if ((rc = upload_f(t, &m->att_bn_t))) return rc;
    if ((rc = upload_raw(a4w, &m->att_w2))) return rc;
    if ((rc = upload_raw(a4b, &m->att_b2))) return rc;
    // embedding head: Linear(5120 -> E, no bias) + BatchNorm1d(E) (halfresnet34, xvector.py:578-581) or a plain
    // Linear(5120 -> E) with bias (resnet34, xvector.py:522-523)
    m->head_bn = half;
    const HostTensor* lw = find(w, half ? "before_speaker_embedding.lin_be.weight" : "before_speaker_embedding.weight");
    if (!lw || lw->shape.size() != 2 || lw->shape[1] != 2 * D) return SKB_ERR_WEIGHTS;
    m->emb = (int)lw->shape[0];
    if ((rc = upload_raw(lw, &m->lin_w))) return rc;
    if (half) {
        if ((rc = bn_affine(w, "before_speaker_embedding.bn_be", &s, &t))) return rc;
        if ((rc = upload_f(s, &m->be_s))) return rc;
        if ((rc = upload_f(t, &m->be_t))) return rc;
    } else {
        const HostTensor* lb = find(w, "before_speaker_embedding.bias");
        if (!lb || lb->numel() != m->emb) return SKB_ERR_WEIGHTS;
        if ((rc = upload_raw(lb, &m->lin_b))) return rc;
    }
    {
        // K permuted to k' = f * C + c (see gather_pack_kernel): column c * F + f of the Conv1d weight moves to f * C + c
        const int Cc = m->level_C[3], Ff = D / Cc;
        std::vector<float> w1p((size_t)A * D);
        for (int a = 0; a < A; ++a)
            for (int c = 0; c < Cc; ++c)
                for (int f = 0; f < Ff; ++f) w1p[(size_t)a * D + f * Cc + c] = w1x[(size_t)a * D + c * Ff + f];
        float* tmp = nullptr;
        if ((rc = dev_upload(w1p, &tmp))) return rc;
        rc = packed_create(tmp, A, D, &m->p_w1x, 0);
        cudaDeviceSynchronize();
        cudaFree(tmp);
        if (rc) return rc;
    }
    if ((rc = packed_create(m->att_w2, D, A, &m->p_w2, 0))) return rc;
    return build_margin_head(w, m);
}

static int build_tdnn(const WeightMap& w, Model* m) {
    // conv -> LeakyReLU(0.2) -> BatchNorm, x5 (xvector.py:467-483): BN_k folds FORWARD into conv_{k+1}
    // (exact: no padding), BN_5 folds into the statistics pooling.
    const int ks[5] = {5, 3, 3, 1, 1}, ds[5] = {1, 2, 3, 1, 1};
    std::vector<double> ps, pt;   // previous layer's BN affine
    int rc;
    for (int i = 0; i < 5; ++i) {
        const std::string c = "sequence_network.conv" + std::to_string(i + 1);
        const HostTensor *cw = find(w, c + ".weight"), *cb = find(w, c + ".bias");
        if (!cw || !cb || cw->shape.size() != 3 || cw->shape[2] != ks[i]) return SKB_ERR_WEIGHTS;
        const int cout = (int)cw->shape[0], cin = (int)cw->shape[1], K = ks[i];
        std::vector<double> wf((size_t)cout * cin * K), bf(cout);
        for (int co = 0; co < cout; ++co) {
            double b = cb->p[co];
            for (int ci = 0; ci < cin; ++ci)
                for (int k = 0; k < K; ++k) {
                    const double v = cw->p[((size_t)co * cin + ci) * K + k];
                    wf[((size_t)co * cin + ci) * K + k] = ps.empty() ? v : v * ps[ci];
                    if (!ps.empty()) b += v * pt[ci];
                }
            bf[co] = b;
        }
        const int cin_pad = (cin + kConvKC - 1) / kConvKC * kConvKC;
        ConvW cv;
        if ((rc = pack_conv(wf, bf, cout, cin, cin_pad, K, m->bf16, &cv))) return rc;
        m->tdnn.push_back(cv);
        m->tdnn_k.push_back(K);
        m->tdnn_d.push_back(ds[i]);
        if ((rc = bn_affine(w, "sequence_network.batch_norm" + std::to_string(i + 1), &ps, &pt))) return rc;
    }
    if ((rc = upload_f(ps, &m->pool_s))) return rc;
    if ((rc = upload_f(pt, &m->pool_t))) return rc;
    m->pool_D = (int)ps.size();
    const HostTensor *lw = find(w, "before_speaker_embedding.linear6.weight"), *lb = find(w, "before_speaker_embedding.linear6.bias");
    if (!lw || !lb || lw->shape[1] != 2 * m->pool_D) return SKB_ERR_WEIGHTS;
    m->emb = (int)lw->shape[0];
    if ((rc = upload_raw(lw, &m->lin_w))) return rc;
    if ((rc = upload_raw(lb, &m->lin_b))) return rc;
    return build_margin_head(w, m);
}

static void free_model(Model* m) {
    frontend_consts_destroy(&m->fe);
    for (auto& b : m->blocks) {
        free_conv(&b.conv1); free_conv(&b.conv2);
        if (b.has_sc) free_conv(&b.sc);
        cudaFree(b.se_w1); cudaFree(b.se_w2); cudaFree(b.w2t);
    }
    for (auto& c : m->tdnn) free_conv(&c);
    cudaFree(m->att_w1x); cudaFree(m->att_w1g); cudaFree(m->att_b1); cudaFree(m->att_bn_s); cudaFree(m->att_bn_t);
    cudaFree(m->att_w2); cudaFree(m->att_b2); cudaFree(m->lin_w); cudaFree(m->lin_b); cudaFree(m->be_s); cudaFree(m->be_t);
    cudaFree(m->spk_wn); cudaFree(m->spk_b); cudaFree(m->pool_s); cudaFree(m->pool_t);
    packed_free(&m->p_w1x); packed_free(&m->p_w2);
}

// ----------------------------------------------------------------------------- per-batch plan
struct Level {
    int W = 0, Wp = 0, C = 0;
    int n_rows = 0, G = 0, p_end = 0;
    long long plane = 0;           // pixels per chunk plane (incl. guards)
    std::vector<int> H;            // lines per utterance
    // offsets (in ints) into the device table buffer
    size_t o_row_b = 0, o_row_h = 0, o_utt_row0 = 0, o_utt_count = 0;
    size_t o_span = 0;             // per-256-pixel utterance table for plane_sum_kernel (halfresnet34 only)
    size_t o_pix_b = 0, o_pix_sub = 0;   // o_pix_sub: phase-split destination table (see pixmeta_kernel)   // offsets (ints) into the device pixel-meta buffer; o_pix_sub valid when has_sub
    bool has_sub = false;
};

struct Plan {
    int B = 0;
    std::vector<int64_t> lengths;
    std::vector<int> T;            // feature frames per utterance
    int t_max = 0;
    long long total_frames = 0, total_samples = 0;
    std::vector<Level> lv;         // 4 levels (halfresnet34) / 6 row-table variants (tdnn: input + 5 layers)
    int pool_frames = 0;           // frames entering the pooling
    size_t o_wave_len = 0, o_nframes = 0, o_frame_row = 0, o_frame_utt = 0, o_pool_nfr = 0, o_row_src = 0;
    size_t o_wave_off = 0, o_feat_off = 0, o_pool_off = 0;   // offsets (in long long) into the 64-bit table
    std::vector<int> tab32;
    std::vector<long long> tab64;
};

constexpr int kTailGuard = 640;    // >= largest CTA tile (512 pixels) + slack, so the last slab stays in bounds

static void plan_level(Plan* pl, Level* L, int W, int C, const std::vector<int>& H, bool pad_lines, int halo) {
    L->W = W; L->Wp = pad_lines ? W + 1 : W; L->C = C; L->H = H;
    const int B = (int)H.size();
    std::vector<int> row_b, row_h, utt_row0(B), utt_count(B);
    if (pad_lines) { row_b.push_back(-1); row_h.push_back(-1); }
    for (int b = 0; b < B; ++b) {
        utt_row0[b] = (int)row_b.size();
        utt_count[b] = H[b] * W;
        for (int h = 0; h < H[b]; ++h) { row_b.push_back(b); row_h.push_back(h); }
        if (pad_lines) { row_b.push_back(-1); row_h.push_back(-1); }
    }
    L->n_rows = (int)row_b.size();
    L->G = (halo + 7) / 8 * 8;
    if (L->G < 8) L->G = 8;
    L->p_end = L->G + L->n_rows * L->Wp;
    L->plane = (long long)L->p_end + kTailGuard + halo + 8;
    L->o_row_b = pl->tab32.size(); pl->tab32.insert(pl->tab32.end(), row_b.begin(), row_b.end());
    L->o_row_h = pl->tab32.size(); pl->tab32.insert(pl->tab32.end(), row_h.begin(), row_h.end());
    L->o_utt_row0 = pl->tab32.size(); pl->tab32.insert(pl->tab32.end(), utt_row0.begin(), utt_row0.end());
    L->o_utt_count = pl->tab32.size(); pl->tab32.insert(pl->tab32.end(), utt_count.begin(), utt_count.end());
}

}  // namespace skb

using namespace skb;

// ----------------------------------------------------------------------------- the handle
struct skb_xtractor {
    Model m;
    Plan plan;
    bool plan_valid = false;
    // Recently used plans (geometry tables live on the device): a bulk extraction cycles through a handful of length
    // buckets, and rebuilding a plan costs a host pass over every frame plus a synchronous table upload.
    // A plan's device tables, their pinned staging copies and the event that marks the upload as done travel together as
    // one SLOT.  A new geometry takes over the slot of the least recently used plan: no cudaFree / cudaMalloc (both
    // synchronise the device) and no host wait -- the tables are copied asynchronously from the pinned staging, in stream
    // order behind the kernels that may still be reading the slot's previous contents, so the host can plan the next
    // batches while the GPU works on this one.
    struct Slot {
        DevBuf tab32, tab64, pixmeta;
        PinnedBuf stage32, stage64;
        cudaEvent_t uploaded = nullptr;
        void release() {
            tab32.release(); tab64.release(); pixmeta.release(); stage32.release(); stage64.release();
            if (uploaded) cudaEventDestroy(uploaded);
            uploaded = nullptr;
        }
    };
    struct CachedPlan { Plan plan; Slot slot; unsigned long long stamp = 0; };
    std::vector<CachedPlan> cache;
    unsigned long long stamp = 0;
    Slot slot;                    // of the active plan
    cudaStream_t last_stream = nullptr;
    bool have_last_stream = false;
    DevBuf brd, cmvn, cmvn_part, skinny_ws;
    DevBuf ovf;                   // fp16 range guard: cumulative count of threads that stored a saturated activation (common.cuh)
    int device = 0;               // the CUDA device the weights and work buffers live on
    float slope_override = -1.f;  // >= 0: activation slope of the next run_conv (stand-alone operators)
    size_t hw_tab32 = 0, hw_tab64 = 0, hw_pixmeta = 0;   // high-water marks of the plan tables: every cache slot is sized for them
    DevBuf feats, sums, scale, poolX, poolH, poolL, gc, hb, pooled, lin, emb_pre, emb, logits, wave, dbg;
    std::vector<DevBuf> act;      // activation buffers
    std::vector<size_t> act_bytes;
    PackedOp poolA;               // frames x 2560 packed fp16 operand of the first attention projection
    int poolA_rows = 0;
    const int* d32 = nullptr;
    const long long* d64 = nullptr;
};

namespace skb {

static int build_pixmeta(skb_xtractor* h, cudaStream_t st);
static int num_frames(const Model& m, int64_t n) { return 1 + (int)(n / m.fe.hop); }

constexpr size_t kPlanCacheEntries = 8;
static int activate_plan(skb_xtractor* h, cudaStream_t st);

static int build_plan(skb_xtractor* h, const int64_t* lengths, int B, cudaStream_t st) {
    Plan& pl = h->plan;
    if (h->plan_valid && pl.B == B && std::equal(lengths, lengths + B, pl.lengths.begin())) return SKB_OK;
    // the slots are reused in stream order: a change of stream needs one device-wide join
    if (h->have_last_stream && h->last_stream != st) SKB_CUDA_CHECK(cudaDeviceSynchronize());
    h->last_stream = st;
    h->have_last_stream = true;
    // park the current plan (with its slot) in the cache, then look the requested one up
    if (h->plan_valid) {
        h->cache.emplace_back();
        skb_xtractor::CachedPlan& c = h->cache.back();
        std::swap(c.plan, h->plan);
        std::swap(c.slot, h->slot);
        c.stamp = ++h->stamp;
        h->plan_valid = false;
    }
    for (size_t i = 0; i < h->cache.size(); ++i) {
        skb_xtractor::CachedPlan& c = h->cache[i];
        if (c.plan.B == B && std::equal(lengths, lengths + B, c.plan.lengths.begin())) {
            std::swap(c.plan, h->plan);
            std::swap(c.slot, h->slot);
            h->cache.erase(h->cache.begin() + i);
            h->d32 = (const int*)h->slot.tab32.p;
            h->d64 = (const long long*)h->slot.tab64.p;
            return activate_plan(h, st);
        }
    }
    // a new geometry: take over the slot of the least recently used plan once the cache is full (h->slot is empty here
    // unless a previous build failed half-way, in which case it is simply reused)
    if (h->cache.size() > kPlanCacheEntries) {
        size_t oldest = 0;
        for (size_t i = 1; i < h->cache.size(); ++i)
            if (h->cache[i].stamp < h->cache[oldest].stamp) oldest = i;
        h->slot.release();
        std::swap(h->slot, h->cache[oldest].slot);
        h->cache.erase(h->cache.begin() + oldest);
    }
    pl = Plan();
    pl.B = B;
    pl.lengths.assign(lengths, lengths + B);
    const Model& m = h->m;
    std::vector<long long> wave_off(B), feat_off(B);
    std::vector<int> wave_len(B);
    for (int b = 0; b < B; ++b) {
        if (lengths[b] <= m.fe.n_fft / 2 || lengths[b] > 0x7fffffff) {
            set_last_error(__FILE__, __LINE__, "utterance too short for the reflect-padded STFT (needs > n_fft/2 samples) or too long");
            return SKB_ERR_ARG;
        }
        wave_off[b] = pl.total_samples;
        wave_len[b] = (int)lengths[b];
        pl.total_samples += lengths[b];
        const int T = num_frames(m, lengths[b]);
        pl.T.push_back(T);
        feat_off[b] = pl.total_frames;
        pl.total_frames += T;
        pl.t_max = std::max(pl.t_max, T);
    }
    pl.o_wave_len = pl.tab32.size(); pl.tab32.insert(pl.tab32.end(), wave_len.begin(), wave_len.end());
    pl.o_nframes = pl.tab32.size(); pl.tab32.insert(pl.tab32.end(), pl.T.begin(), pl.T.end());
    pl.o_wave_off = pl.tab64.size(); pl.tab64.insert(pl.tab64.end(), wave_off.begin(), wave_off.end());
    pl.o_feat_off = pl.tab64.size(); pl.tab64.insert(pl.tab64.end(), feat_off.begin(), feat_off.end());

    std::vector<int> pool_nfr(B);
    std::vector<long long> pool_off(B);
    std::vector<int> frame_row, frame_utt;
    if (is_resnet(m.archi)) {
        pl.lv.resize(4);
        std::vector<int> H = pl.T;
        for (int l = 0; l < 4; ++l) {
            if (l > 0 && m.level_halves[l]) for (auto& x : H) x = (x - 1) / 2 + 1;
            plan_level(&pl, &pl.lv[l], m.level_W[l], m.level_C[l], H, true, m.level_W[l] + 2);
        }
        const Level& L4 = pl.lv[3];
        long long off = 0;
        for (int b = 0; b < B; ++b) {
            pool_nfr[b] = L4.H[b];
            pool_off[b] = off;
            off += L4.H[b];
            const int r0 = pl.tab32[L4.o_utt_row0 + b];
            for (int t = 0; t < L4.H[b]; ++t) { frame_row.push_back(r0 + t); frame_utt.push_back(b); }
        }
        pl.pool_frames = (int)off;
    } else {
        // TDNN: one "line" per frame (W = 1, no pad lines); a row table per layer output marks the
        // frames that still exist after the unpadded dilated convolutions (T -> T-4 -> T-8 -> T-14).
        const int shrink[6] = {0, 4, 8, 14, 14, 14};
        const int Cs[6] = {96, 512, 512, 512, 512, 1536};
        pl.lv.resize(6);
        for (int l = 0; l < 6; ++l) {
            plan_level(&pl, &pl.lv[l], 1, Cs[l], pl.T, false, 8);
            // overwrite row_h with the validity of this layer's output
            size_t r = pl.lv[l].o_row_h;
            for (int b = 0; b < B; ++b)
                for (int t = 0; t < pl.T[b]; ++t, ++r) pl.tab32[r] = (t < pl.T[b] - shrink[l]) ? t : -1;
        }
        long long off = 0;
        for (int b = 0; b < B; ++b) {
            const int To = pl.T[b] - 14;
            if (To < 1) {
                set_last_error(__FILE__, __LINE__, "utterance shorter than the TDNN context (15 frames)");
                return SKB_ERR_ARG;
            }
            pool_nfr[b] = To;
            pool_off[b] = off;
            off += To;
            const int r0 = pl.tab32[pl.lv[5].o_utt_row0 + b];
            for (int t = 0; t < To; ++t) { frame_row.push_back(r0 + t); frame_utt.push_back(b); }
        }
        pl.pool_frames = (int)off;
        // source frame of every input row (identity here; kept explicit for the pack kernel)
        pl.o_row_src = pl.tab32.size();
        for (long long i = 0; i < pl.total_frames; ++i) pl.tab32.push_back((int)i);
    }
    pl.o_frame_row = pl.tab32.size(); pl.tab32.insert(pl.tab32.end(), frame_row.begin(), frame_row.end());
    pl.o_frame_utt = pl.tab32.size(); pl.tab32.insert(pl.tab32.end(), frame_utt.begin(), frame_utt.end());
    pl.o_pool_nfr = pl.tab32.size(); pl.tab32.insert(pl.tab32.end(), pool_nfr.begin(), pool_nfr.end());
    pl.o_pool_off = pl.tab64.size(); pl.tab64.insert(pl.tab64.end(), pool_off.begin(), pool_off.end());

    int rc;
    skb_xtractor::Slot& sl = h->slot;
    const size_t b32 = pl.tab32.size() * sizeof(int), b64 = pl.tab64.size() * sizeof(long long);
    h->hw_tab32 = std::max(h->hw_tab32, b32);
    h->hw_tab64 = std::max(h->hw_tab64, b64);
    if ((rc = sl.tab32.ensure(h->hw_tab32))) return rc;
    if ((rc = sl.tab64.ensure(h->hw_tab64))) return rc;
    // the staging copies of this slot's previous plan must have left the host before they are overwritten (they did,
    // unless the host is a whole cache of batches ahead of the device)
    if (sl.uploaded) SKB_CUDA_CHECK(cudaEventSynchronize(sl.uploaded));
    else SKB_CUDA_CHECK(cudaEventCreateWithFlags(&sl.uploaded, cudaEventDisableTiming));
    if ((rc = sl.stage32.ensure(h->hw_tab32))) return rc;
    if ((rc = sl.stage64.ensure(h->hw_tab64))) return rc;
    memcpy(sl.stage32.p, pl.tab32.data(), b32);
    memcpy(sl.stage64.p, pl.tab64.data(), b64);
    SKB_CUDA_CHECK(cudaMemcpyAsync(sl.tab32.p, sl.stage32.p, b32, cudaMemcpyHostToDevice, st));
    SKB_CUDA_CHECK(cudaMemcpyAsync(sl.tab64.p, sl.stage64.p, b64, cudaMemcpyHostToDevice, st));
    SKB_CUDA_CHECK(cudaEventRecord(sl.uploaded, st));
    h->d32 = (const int*)sl.tab32.p;
    h->d64 = (const long long*)sl.tab64.p;

    int rc2 = build_pixmeta(h, st);
    if (rc2) return rc2;
    return activate_plan(h, st);
}

// Everything a plan activation has to (re)establish in the shared work buffers, in ONE launch (it used to be up to 19
// cudaMemset2DAsync + 3 kernels + 1 memset per new batch geometry, ~0.3 ms of launch gaps per step of a bulk extraction):
//  * guards: the G pixels before the first computed pixel of every chunk plane of every activation buffer (tap (-1, -1)
//    of the first pixel reads pixel G - 1; the plane stride moves with the geometry);
//  * phase-split buffers: what the producing convolution never writes -- the pad pixels, and, when the source utterance
//    has an odd number of lines, the last line of the two odd-row phases (it has no source line and acts as the bottom
//    zero padding);
//  * the fixed-point SE channel totals.
struct ActGuard { uint16_t* p; long long plane; int n_planes, G; };
struct ActPs { uint16_t* buf; long long plane; int cpp, G, n, Wp, W, src_W, first_block; const int *row_b, *row_h, *src_utt_count; };
struct ActArgs {
    ActGuard g[20]; int n_guards;
    ActPs ps[3]; int n_ps;
    unsigned long long* sums; int n_sums, sums_first_block;
};
__global__ void __launch_bounds__(256) plan_activate_kernel(const __grid_constant__ ActArgs a) {
    const int blk = blockIdx.x;
    if (blk < a.n_guards) {
        const ActGuard& g = a.g[blk];
        const int per = g.G;                                    // 16-byte units per plane
        for (int i = threadIdx.x; i < g.n_planes * per; i += blockDim.x) {
            const int j = i / per, q = i - j * per;
            *reinterpret_cast<uint4*>(g.p + ((size_t)j * g.plane + q) * 8) = make_uint4(0u, 0u, 0u, 0u);
        }
        return;
    }
    if (blk >= a.sums_first_block) {
        const int i = (blk - a.sums_first_block) * blockDim.x + threadIdx.x;
        if (i < a.n_sums) a.sums[i] = 0ull;
        return;
    }
    int k = 0;
    while (k + 1 < a.n_ps && blk >= a.ps[k + 1].first_block) ++k;
    const ActPs& z = a.ps[k];
    // one thread per (line, chunk plane of the phase-split buffer): only the pad column, the pad lines and the odd-row phases
    // of an utterance's last line need zeros (walking every pixel cost 0.1 ms per batch: profiles/r02s_launches_hr34_step_summary.txt)
    const int idx = (blk - z.first_block) * blockDim.x + threadIdx.x;
    const int n_planes = 4 * z.cpp;
    const int n_lines = z.n / z.Wp;
    if (idx >= n_lines * n_planes) return;
    const int row = idx / n_planes, j = idx - row * n_planes;
    const int b = z.row_b[row], hh = z.row_h[row];
    uint16_t* line = z.buf + ((size_t)j * z.plane + z.G + (size_t)row * z.Wp) * 8;
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    if (b < 0 || hh < 0) {                                                           // pad line: every pixel, all four phases
        for (int w = 0; w < z.Wp; ++w) *reinterpret_cast<uint4*>(line + (size_t)w * 8) = zero;
        return;
    }
    for (int w = z.W; w < z.Wp; ++w) *reinterpret_cast<uint4*>(line + (size_t)w * 8) = zero;   // pad column(s)
    if (j >= 2 * z.cpp && 2 * hh + 1 >= z.src_utt_count[b] / z.src_W)               // no odd source line below: phases 2, 3
        for (int w = 0; w < z.W; ++w) *reinterpret_cast<uint4*>(line + (size_t)w * 8) = zero;
}

// Make `h->plan` current: size the shared work buffers for it and re-establish the few invariants that depend on the
// geometry.  Activation buffers are NOT cleared as a whole (5 GB of memset per plan change): every kernel writes all
// pixels of [G, p_end) of its output (zeros at the pads), and what lies after p_end only feeds accumulator rows that
// are discarded.
static int activate_plan(skb_xtractor* h, cudaStream_t st) {
    Plan& pl = h->plan;
    const Model& m = h->m;
    const int B = pl.B;
    int rc;
    std::vector<size_t> need;
    if (is_resnet(m.archi)) {
        for (int l = 0; l < 4; ++l) {
            const size_t bytes = (size_t)(pl.lv[l].C / 8) * pl.lv[l].plane * 16;
            // A, B (block in/out ping-pong), Y1, PS (phase-split copy of the previous level's output: 4 * C_prev/8 planes
            // = twice this level's plane count), SC (shortcut conv output)
            const size_t ps_bytes = (l == 0 || !m.level_halves[l]) ? 256 : (size_t)4 * (pl.lv[l - 1].C / 8) * pl.lv[l].plane * 16;
            for (int k = 0; k < 5; ++k) need.push_back(k == 3 ? ps_bytes : bytes);
        }
    } else {
        for (int l = 0; l < 6; ++l) need.push_back((size_t)(pl.lv[l].C / 8) * pl.lv[l].plane * 16);
    }
    h->act.resize(need.size());
    h->act_bytes = need;
    for (size_t i = 0; i < need.size(); ++i)
        if ((rc = h->act[i].ensure(need[i]))) return rc;
    const int Cmax = is_resnet(m.archi) ? 256 : 0;
    if (Cmax) {
        if ((rc = h->sums.ensure((size_t)B * Cmax * sizeof(unsigned long long)))) return rc;
        if ((rc = h->scale.ensure((size_t)B * Cmax * sizeof(float)))) return rc;
        if ((rc = h->brd.ensure((size_t)B * (8 + 36) * Cmax * sizeof(float)))) return rc;   // border sums + K-slice partial means

    }
    if (is_resnet(m.archi)) {
        // The one guard pixel that IS read into a kept accumulator row: tap (-1, -1) of the first pixel of the first
        // line reaches pixel G - 1.  Nothing ever writes below G, but the plane stride moves with the geometry, so the
        // guard of every chunk plane is cleared whenever the plan changes.
        ActArgs a;
        memset(&a, 0, sizeof(a));
        for (int l = 0; l < 4; ++l)
            for (int k = 0; k < 5; ++k) {
                if (k == 3 && (l == 0 || !m.level_halves[l])) continue;      // no phase-split buffer on this level
                const Level& L = pl.lv[l];
                ActGuard& g = a.g[a.n_guards++];
                g.p = (uint16_t*)h->act[l * 5 + k].p;
                g.plane = L.plane;
                g.n_planes = k == 3 ? 4 * (pl.lv[l - 1].C / 8) : L.C / 8;
                g.G = L.G;
            }
        int blocks = a.n_guards;
        for (int l = 1; l < 4; ++l) {
            if (!m.level_halves[l]) continue;
            const Level& Lo = pl.lv[l];
            const Level& Ls = pl.lv[l - 1];
            ActPs& z = a.ps[a.n_ps++];
            z.buf = (uint16_t*)h->act[l * 5 + 3].p; z.plane = Lo.plane; z.cpp = Ls.C / 8; z.G = Lo.G; z.n = Lo.p_end - Lo.G;
            z.Wp = Lo.Wp; z.W = Lo.W; z.src_W = Ls.W; z.first_block = blocks;
            z.row_b = h->d32 + Lo.o_row_b; z.row_h = h->d32 + Lo.o_row_h; z.src_utt_count = h->d32 + Ls.o_utt_count;
            blocks += ((z.n / z.Wp) * 4 * z.cpp + 255) / 256;
        }
        a.sums = (unsigned long long*)h->sums.p;
        a.n_sums = B * Cmax;
        a.sums_first_block = blocks;
        blocks += (a.n_sums + 255) / 256;
        SKB_CUDA_CHECK(launch_kernel(false, plan_activate_kernel, blocks, 256, 0, st, a));
    }
    if ((rc = h->feats.ensure((size_t)pl.total_frames * m.fe.n_out * sizeof(float)))) return rc;
    if ((rc = h->cmvn.ensure((size_t)B * m.fe.n_out * sizeof(float2)))) return rc;
    if ((rc = h->cmvn_part.ensure(frontend_cmvn_scratch_bytes(m.fe, B, pl.t_max)))) return rc;
    const int D = m.pool_D;
    if (is_resnet(m.archi)) {
        if ((rc = h->poolX.ensure((size_t)pl.pool_frames * D * sizeof(uint16_t)))) return rc;
        if ((rc = h->poolH.ensure((size_t)pl.pool_frames * m.att_A * sizeof(float)))) return rc;
        if ((rc = h->poolL.ensure((size_t)pl.pool_frames * D * sizeof(float)))) return rc;
        if ((rc = h->gc.ensure((size_t)B * 2 * D * sizeof(float)))) return rc;
        if ((rc = h->hb.ensure((size_t)B * m.att_A * sizeof(float)))) return rc;
    }
    if ((rc = h->pooled.ensure((size_t)B * 2 * D * sizeof(float)))) return rc;
    if ((rc = h->lin.ensure((size_t)B * m.emb * sizeof(float)))) return rc;
    if ((rc = h->emb_pre.ensure((size_t)B * m.emb * sizeof(float)))) return rc;
    h->plan_valid = true;
    return SKB_OK;
}

// Per-pixel tables for the conv epilogue (one coalesced read instead of a division and two dependent gathers), for ALL
// levels of a plan in one launch:
// pix_b[rel] = utterance of pixel G + rel or -1 for pad / invalid; pix_ps[rel] = destination of the pixel in the
// PHASE-SPLIT copy that feeds the next level's stride-2 block: four phase images (h & 1, w & 1) in the next level's
// geometry, stacked as groups of C/8 chunk planes:  dest = phase * (C/8) * plane' + G' + (row0'[b] + h/2) * Wp' + w/2;
// span_b[span] = the utterance of a 256-pixel span when every valid pixel belongs to one, -1 when it holds only pad
// pixels, -2 when it straddles utterances (plane_sum_kernel).  One warp per span.
struct MetaLevel {
    int n, Wp, W, out_G, out_Wp, first_block;
    const int *row_b, *row_h, *out_utt_row0;
    int *pix_b, *pix_ps, *span_b;
    long long phase_stride;
};
struct MetaArgs { MetaLevel lv[6]; int n_levels; };
__global__ void __launch_bounds__(256) planmeta_kernel(const __grid_constant__ MetaArgs a) {
    int k = 0;
    while (k + 1 < a.n_levels && (int)blockIdx.x >= a.lv[k + 1].first_block) ++k;
    const MetaLevel& L = a.lv[k];
    const int lane = threadIdx.x & 31;
    const int span = ((int)blockIdx.x - L.first_block) * 8 + (threadIdx.x >> 5);
    if (span * 256 >= L.n) return;
    int mn = 0x7fffffff, mx = -1;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int rel = span * 256 + q * 32 + lane;
        if (rel >= L.n) continue;
        const int row = rel / L.Wp, w = rel - row * L.Wp;
        const int b = L.row_b[row], hh = L.row_h[row];
        const bool valid = b >= 0 && hh >= 0 && w < L.W;
        L.pix_b[rel] = valid ? b : -1;
        if (L.pix_ps)
            L.pix_ps[rel] = valid ? (int)(((hh & 1) * 2 + (w & 1)) * L.phase_stride + L.out_G +
                                          (long long)(L.out_utt_row0[b] + (hh >> 1)) * L.out_Wp + (w >> 1))
                                  : -1;
        if (valid) { mn = min(mn, b); mx = max(mx, b); }
    }
    if (L.span_b) {
        mn = __reduce_min_sync(0xffffffffu, mn);
        mx = __reduce_max_sync(0xffffffffu, mx);
        if (lane == 0) L.span_b[span] = mx < 0 ? -1 : (mn == mx ? mn : -2);
    }
}

static int build_pixmeta(skb_xtractor* h, cudaStream_t st) {
    Plan& pl = h->plan;
    size_t total = 0;
    const bool hr = is_resnet(h->m.archi);
    if (pl.lv.size() > 6) {
        set_last_error(__FILE__, __LINE__, "internal: more than 6 geometry levels");
        return SKB_ERR_STATE;
    }
    for (size_t l = 0; l < pl.lv.size(); ++l) {
        Level& L = pl.lv[l];
        const size_t n = (size_t)(L.p_end - L.G);
        L.o_pix_b = total; total += n;
        L.has_sub = hr && l + 1 < pl.lv.size() && h->m.level_halves[l + 1];   // the next level strides: phase-split destinations
        if (L.has_sub) { L.o_pix_sub = total; total += n; }
        if (hr) { L.o_span = total; total += (size_t)span_table_size((int)n); }
    }
    // every slot of the plan cache is sized for the largest table set seen so far (a slot that had to grow would cost a
    // cudaFree / cudaMalloc pair, i.e. a device-wide synchronisation, in the middle of a bulk extraction)
    h->hw_pixmeta = std::max(h->hw_pixmeta, total * sizeof(int));
    int rc = h->slot.pixmeta.ensure(h->hw_pixmeta);
    if (rc) return rc;
    int* base = (int*)h->slot.pixmeta.p;
    MetaArgs a;
    memset(&a, 0, sizeof(a));
    a.n_levels = (int)pl.lv.size();
    int blocks = 0;
    for (size_t l = 0; l < pl.lv.size(); ++l) {
        const Level& L = pl.lv[l];
        const Level* Lo = L.has_sub ? &pl.lv[l + 1] : nullptr;
        MetaLevel& M = a.lv[l];
        M.n = L.p_end - L.G; M.Wp = L.Wp; M.W = L.W; M.first_block = blocks;
        M.row_b = h->d32 + L.o_row_b; M.row_h = h->d32 + L.o_row_h;
        M.pix_b = base + L.o_pix_b;
        M.pix_ps = Lo ? base + L.o_pix_sub : nullptr;
        M.span_b = hr ? base + L.o_span : nullptr;
        M.out_G = Lo ? Lo->G : 0; M.out_Wp = Lo ? Lo->Wp : 0;
        M.out_utt_row0 = Lo ? h->d32 + Lo->o_utt_row0 : nullptr;
        M.phase_stride = Lo ? (long long)(L.C / 8) * Lo->plane : 0;
        blocks += (span_table_size(M.n) + 7) / 8;
    }
    if (blocks > 0) SKB_CUDA_CHECK(launch_kernel(false, planmeta_kernel, blocks, 256, 0, st, a));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- conv launch helper
// kind: 0 = 1x1 / single tap, 1 = 3x3 pad 1, 2 = TDNN taps (tdnn_shifts), 3 = 3x3 stride 2 on a phase-split input.
// `Lg` is the geometry the kernel walks (= the input's pixel layout); `to_phase_split` redirects the stores into the
// phase-split buffer of the next level (`Lnext`).
static int run_conv(skb_xtractor* h, const ConvW& cw, int kind, const Level& Lg, const uint16_t* in, uint16_t* out, int act,
                    const int* tdnn_shifts, const float* se_scale, const uint16_t* res, const Level* pix_level,
                    const Level* Lnext, cudaStream_t st, unsigned long long* sums = nullptr, const ConvW* sc = nullptr,
                    const uint16_t* sc_in = nullptr) {
    ConvParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.in_plane = Lg.plane; p.w = cw.w; p.bias = cw.bias; p.out = out;
    p.out_plane = Lnext ? Lnext->plane : Lg.plane;
    p.cin = cw.cin; p.cout = cw.cout; p.taps = cw.taps;
    p.G = Lg.G; p.p_end = Lg.p_end;
    const int n_kc = cw.cin / kConvKC;
    p.kc_per_grp = n_kc;
    p.grp_tap[0] = 0;
    for (int g = 1; g < 5; ++g) p.grp_tap[g] = cw.taps;
    p.n_pairs = n_kc * cw.taps;
    int max_shift = 0;
    p.Wp = Lg.Wp;
    p.n_utt = h->plan.B;
    if (kind == 1) {
        p.w3 = cw.w3;
        p.halo = Lg.Wp + 1;
        for (int t = 0; t < 9; ++t) p.tap_shift[t] = (t / 3 - 1) * Lg.Wp + (t % 3 - 1);
        max_shift = Lg.Wp + 1;
    } else if (kind == 2) {
        p.halo = 0;
        for (int t = 0; t < cw.taps; ++t) { p.tap_shift[t] = tdnn_shifts[t]; max_shift = std::max(max_shift, tdnn_shifts[t]); }
    } else if (kind == 3) {
        // tap (r, s) of a stride-2 conv reads phase ((r-1) & 1, (s-1) & 1) at (h' + dh, w' + dw), dh/dw = -1 for r/s = 0 else 0
        p.halo = Lg.Wp + 1;
        for (int t = 0; t < 9; ++t) {
            const int dh = kPhaseTaps[t][0] == 0 ? -1 : 0, dw = kPhaseTaps[t][1] == 0 ? -1 : 0;
            p.tap_shift[t] = dh * Lg.Wp + dw;
        }
        p.kc_per_grp = n_kc / 4;
        for (int g = 0; g < 5; ++g) p.grp_tap[g] = kPhaseTapBegin[g];
        p.n_pairs = p.kc_per_grp * 9;
    } else {
        p.halo = 0;
        p.tap_shift[0] = 0;
    }
    const int tile_m = conv_tile_m(cw.ncta);
    p.rows_pad = (tile_m + p.halo + max_shift + 7) / 8 * 8;
    p.act_slope = act == 1 ? 0.f : (act == 2 ? 0.2f : 1.f);
    if (h->slope_override >= 0.f) p.act_slope = h->slope_override;
    const int* pm = (const int*)h->slot.pixmeta.p;
    // the validity table of `pix_level` decides what is stored as non-zero (TDNN: same geometry, fewer frames per layer)
    p.pix_b = pm + (pix_level ? pix_level->o_pix_b : Lg.o_pix_b);
    p.pix_sub = Lnext ? pm + Lg.o_pix_sub : nullptr;
    p.se_scale = se_scale;
    p.res = res;
    p.res_plane = Lg.plane;
    p.sums = sums;
    p.overflow = (unsigned*)h->ovf.p;
    if (sc) { p.sc_in = sc_in; p.sc_w = sc->w; p.sc_bias = sc->bias; p.sc_cin = sc->cin; }
    return launch_conv_umma(p, cw.ncta, h->m.bf16, st);
}

#define SKB_TRY(x)            \
    do {                      \
        int _rc = (x);        \
        if (_rc) return _rc;  \
    } while (0)

// planes -> dense (B, C, h_max, W) fp32 (test hook)
template <bool BF16>
__global__ void unpack_planes_kernel(const uint16_t* __restrict__ act, long long plane, int C, int W, int Wp, int G,
                                     const int* __restrict__ utt_row0, const int* __restrict__ utt_count, int h_max,
                                     float* __restrict__ out, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int w = (int)(idx % W);
    const int hh = (int)((idx / W) % h_max);
    const int c = (int)((idx / ((long long)W * h_max)) % C);
    const int b = (int)(idx / ((long long)W * h_max * C));
    const int H = utt_count[b] / W;
    float v = 0.f;
    if (hh < H) {
        const long long pix = (long long)G + (long long)(utt_row0[b] + hh) * Wp + w;
        const uint16_t u = act[((size_t)(c >> 3) * plane + pix) * 8 + (c & 7)];
        if (BF16) {
            __nv_bfloat16 t;
            memcpy(&t, &u, 2);
            v = __bfloat162float(t);
        } else {
            __half t;
            memcpy(&t, &u, 2);
            v = __half2float(t);
        }
    }
    out[idx] = v;
}

static int export_stage(skb_xtractor* h, const uint16_t* act, const Level& L, int h_max, float* out, int64_t* per_utt,
                        cudaStream_t st) {
    const long long total = (long long)h->plan.B * L.C * h_max * L.W;
    *per_utt = (int64_t)L.C * h_max * L.W;
    const int blocks = (int)((total + 255) / 256);
    SKB_CUDA_CHECK(launch_kernel(false, h->m.bf16 ? unpack_planes_kernel<true> : unpack_planes_kernel<false>, blocks, 256, 0, st, act, L.plane,
                                 L.C, L.W, L.Wp, L.G, h->d32 + L.o_utt_row0, h->d32 + L.o_utt_count, h_max, out, total));
    return SKB_OK;
}

// ----------------------------------------------------------------------------- forward passes
static int head_and_logits(skb_xtractor* h, int norm_embedding, float* emb_out, float* logits_out, cudaStream_t st) {
    const Model& m = h->m;
    const int B = h->plan.B, D = m.pool_D;
    // before_speaker_embedding: Linear (+ folded BatchNorm1d) (xvector.py:578-581 / :489-491)
    // M = batch size, K = 5120 / 3072: split-K fp32 GEMM (the packed tcgen05 GEMM would run on one or two CTAs)
    SKB_TRY(h->skinny_ws.ensure(std::max(skinny_gemm_ws_floats(B, m.emb, 2 * D), skinny_gemm_ws_floats(B, std::max(m.n_spk, 1), m.emb)) *
                                sizeof(float)));
    SKB_TRY(launch_skinny_gemm((const float*)h->pooled.p, B, 2 * D, m.lin_w, m.emb, m.lin_b, 1.f, (float*)h->lin.p, m.emb,
                               (float*)h->skinny_ws.p, st));
    SKB_TRY(launch_head_norm((const float*)h->lin.p, m.be_s, m.be_t, B, m.emb, norm_embedding, (float*)h->emb_pre.p, emb_out, st));
    if (logits_out && m.n_spk > 0) {   // ArcMarginProduct(target=None): s * cos (loss.py:299-310); 'aps': Linear(x) (loss.py:356-359)
        SKB_TRY(launch_skinny_gemm(m.head_linear ? (const float*)h->emb_pre.p : emb_out, B, m.emb, m.spk_wn, m.n_spk,
                                   m.head_linear ? m.spk_b : nullptr, m.head_linear ? 1.f : m.margin_s, logits_out, m.n_spk,
                                   (float*)h->skinny_ws.p, st));
    }
    return SKB_OK;
}

// SKB_NO_FUSED_SUMS=1: keep the separate plane_sum pass on every level (A/B knob, test reference)
static bool no_fused_sums() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SKB_NO_FUSED_SUMS");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

// SKB_UNFUSED_SHORTCUT=1: run the 1x1 shortcuts as stand-alone launches through a 16-bit buffer (A/B knob, test reference)
static bool unfused_shortcut() {
    static const bool v = [] { const char* e = getenv("SKB_UNFUSED_SHORTCUT"); return e && e[0] == '1'; }();
    return v;
}

static int forward_hr34(skb_xtractor* h, const float* wave, int norm_embedding, float* emb_out, float* logits_out,
                        const char* stop, int h_max, float* dbg_out, int64_t* per_utt, cudaStream_t st) {
    const Model& m = h->m;
    Plan& pl = h->plan;
    const int B = pl.B;
    const int* d32 = h->d32;
    const long long* d64 = h->d64;
    float* feats = (float*)h->feats.p;
    {
        ProfScope ps(PROF_FRONTEND, st);
        // raw log-Mel + CMVN statistics; the stem kernel normalises on the fly
        SKB_TRY(frontend_launch(m.fe, wave, d64 + pl.o_wave_off, d32 + pl.o_wave_len, d64 + pl.o_feat_off, d32 + pl.o_nframes, B,
                                pl.t_max, feats, (float2*)h->cmvn.p, h->cmvn_part.p, false, nullptr, st));
    }
    auto buf = [&](int level, int k) { return (uint16_t*)h->act[level * 5 + k].p; };
    const Level& L1 = pl.lv[0];
    {
        ProfScope ps(PROF_STEM, st);
        if (m.archi == SKB_ARCHI_FASTRESNET34)
            SKB_TRY(launch_stem7(m.bf16, feats, d64 + pl.o_feat_off, d32 + pl.o_nframes, (const float2*)h->cmvn.p, m.stem, buf(0, 0),
                                 L1.plane, L1.G, L1.p_end, L1.Wp, L1.W, m.fe.n_out, d32 + L1.o_row_b, d32 + L1.o_row_h, (unsigned*)h->ovf.p, st));
        else
            SKB_TRY(launch_stem(m.bf16, m.stem_c, feats, d64 + pl.o_feat_off, d32 + pl.o_nframes, (const float2*)h->cmvn.p, m.stem, buf(0, 0),
                                L1.plane, L1.G, L1.p_end, L1.Wp, L1.W, d32 + L1.o_row_b, d32 + L1.o_row_h, (unsigned*)h->ovf.p, st));
    }
    int level = 0, cur = 0;   // current activation = buf(level, cur), cur in {0, 1}
    if (stop && !strcmp(stop, "stem")) return export_stage(h, buf(0, 0), L1, h_max, dbg_out, per_utt, st);
    bool x_is_ps = false;     // the current activation lives phase-split in buf(level + 1, 3) instead of buf(level, cur)
    for (size_t i = 0; i < m.blocks.size(); ++i) {
        const BlockW& bw = m.blocks[i];
        char name[32];
        // a widening block without stride reads the previous level's buffer (same geometry) and writes the next level's
        const uint16_t* x_up = bw.level_up ? buf(level, cur) : nullptr;
        if (bw.stride == 2 || bw.level_up) { level++; cur = 1; }   // this block's output goes to buf(level, 0)
        snprintf(name, sizeof(name), "layer%d.%d", bw.layer, bw.index);
        const Level& L = pl.lv[level];
        // the block after this one strides: write this block's output phase-split in the next level's geometry
        const bool next_strides = i + 1 < m.blocks.size() && m.blocks[i + 1].stride == 2 && !(stop && !strcmp(stop, name));
        const uint16_t* x = bw.stride == 2 ? buf(level, 3) : (x_up ? x_up : buf(level, cur));
        if (bw.stride == 2 && !x_is_ps) {
            set_last_error(__FILE__, __LINE__, "internal: stride-2 block without a phase-split input");
            return SKB_ERR_STATE;
        }
        uint16_t *y1 = buf(level, 2), *scb = buf(level, 4), *nxt = buf(level, cur ^ 1);
        const bool sums_in_conv1 = conv_sums_supported(bw.conv1.ncta, bw.conv1.cout) && !no_fused_sums();
        const uint16_t* res = x;
        // narrow layers: conv2 computes the 1x1 shortcut itself, in a second TMEM accumulator (no launch, no round trip
        // of the shortcut through HBM); the <128, 2> tiles have no tensor memory left for it
        const bool fold_sc = bw.has_sc && bw.conv2.ncta <= 64 && bw.sc.ncta == bw.conv2.ncta && !unfused_shortcut();
        {
            ProfScope ps(PROF_CONV, st);
            // conv1's epilogue also accumulates the per-utterance channel totals of y1 (no plane_sum pass); they are complete
            // when conv1 is, which every kernel of the SE chain waits for (pdl_wait), and se_fc re-zeroes them for the next block
            SKB_TRY(run_conv(h, bw.conv1, bw.stride == 2 ? 3 : 1, L, x, y1, 1, nullptr, nullptr, nullptr, nullptr, nullptr, st,
                             sums_in_conv1 ? (unsigned long long*)h->sums.p : nullptr));
            if (bw.has_sc && !fold_sc) {
                // 1x1 shortcut; with stride 2 it reads phase (0, 0) = the first C_prev/8 planes of the phase-split input
                SKB_TRY(run_conv(h, bw.sc, 0, L, x, scb, 0, nullptr, nullptr, nullptr, nullptr, nullptr, st));
                res = scb;
            }
        }
        {
            // SE scales from conv2's INPUT (linearity of the convolution): one bandwidth-bound pass over y1 + small kernels
            ProfScope ps(PROF_SE, st);
            const int* pm = (const int*)h->slot.pixmeta.p;
            // Measured and rejected in round 2 (profiles/r02_se_merge.txt): border sums + channel totals in one launch, and the FC
            // layers done by the last-arriving partial-mean CTA -- fewer launches, but both variants were slower.
            // Kept from that experiment's lesson -- separate kernels with their own occupancy -- but OVERLAPPED: the border sums
            // go first and release the channel-total pass (when conv1 did not produce the totals) as soon as they have seen
            // conv1 complete (faster than one after the other: profiles/r02u_se_overlap_vs_serial.txt)
            const PlaneSumArgs totals = {L.p_end, pm + L.o_pix_b, pm + L.o_span};
            SKB_TRY(launch_se_scale(m.bf16, (unsigned long long*)h->sums.p, y1, L.plane, L.G, L.Wp, L.W, d32 + L.o_utt_row0,
                                    d32 + L.o_utt_count, B, bw.C, bw.C, bw.w2t, bw.conv2.bias, bw.se_w1, bw.se_w2,
                                    (float*)h->brd.p, (float*)h->scale.p, st, sums_in_conv1 ? nullptr : &totals));
        }
        {
            // conv2 with the fused SE tail: out = relu(bn2(conv2(y1)) * scale + residual)
            ProfScope ps(PROF_CONV, st);
            uint16_t* dst = next_strides ? buf(level + 1, 3) : nxt;
            SKB_TRY(run_conv(h, bw.conv2, 1, L, y1, dst, 1, nullptr, (const float*)h->scale.p, fold_sc ? nullptr : res, nullptr,
                             next_strides ? &pl.lv[level + 1] : nullptr, st, nullptr, fold_sc ? &bw.sc : nullptr, x));
        }
        x_is_ps = next_strides;
        cur ^= 1;
        if (stop && !strcmp(stop, name)) return export_stage(h, buf(level, cur), L, h_max, dbg_out, per_utt, st);
    }
    // attentive statistics pooling with global context (pooling.py:151-171)
    const Level& L4 = pl.lv[3];
    const int D = m.pool_D, A = m.att_A, F = pl.pool_frames;
    uint16_t* X = (uint16_t*)h->poolX.p;           // frames x D in the activations' 16-bit format
    float *Hh = (float*)h->poolH.p, *Lg = (float*)h->poolL.p;
    ProfScope pool_scope(PROF_POOL, st);
    SKB_TRY(launch_gather_frames(m.bf16, buf(level, cur), L4.plane, L4.C, L4.W, L4.Wp, L4.G, d32 + pl.o_frame_row, F, X, st));
    if (m.global_context) {
        SKB_TRY(launch_meanstd(m.bf16, X, d64 + pl.o_pool_off, d32 + pl.o_pool_nfr, B, D, nullptr, nullptr, (float*)h->gc.p, st));
        SKB_TRY(h->skinny_ws.ensure(skinny_gemm_ws_floats(B, A, 2 * D) * sizeof(float)));
        SKB_TRY(launch_skinny_gemm((const float*)h->gc.p, B, 2 * D, m.att_w1g, A, m.att_b1, 1.f, (float*)h->hb.p, A, (float*)h->skinny_ws.p, st));
    } else {
        SKB_TRY(launch_broadcast_rows(m.att_b1, B, A, (float*)h->hb.p, st));
    }
    if (F > h->poolA_rows) {
        if (trace_alloc()) fprintf(stderr, "skb: pooling operand grows %d -> %d frames\n", h->poolA_rows, F);
        packed_free(&h->poolA);
        h->poolA_rows = 0;
        SKB_TRY(packed_alloc_zero(&h->poolA, F + F / 8 + 128, D, st));
        h->poolA_rows = h->poolA.rows;
    }
    {
        PackedOp a = h->poolA;                     // view with this batch's frame count
        a.rows = F;
        a.rows_pad = (F + 127) / 128 * 128;
        SKB_TRY(launch_gather_pack(buf(level, cur), L4.plane, L4.C, L4.W, L4.Wp, L4.G, d32 + pl.o_frame_row, F, a.hi, st));
        SKB_TRY(gemm_packed_a(a, m.p_w1x, nullptr, 1.f, Hh, A, st));
    }
    SKB_TRY(launch_att_act(Hh, (const float*)h->hb.p, d32 + pl.o_frame_utt, m.att_bn_s, m.att_bn_t, F, A, st));
    SKB_TRY(gemm_nt_split(Hh, F, A, m.p_w2, m.att_b2, 1.f, Lg, D, st));
    SKB_TRY(launch_softmax_pool(m.bf16, X, Lg, d64 + pl.o_pool_off, d32 + pl.o_pool_nfr, B, D, (float*)h->pooled.p, st));
    if (stop && !strcmp(stop, "pooled")) {
        *per_utt = 2 * D;
        SKB_CUDA_CHECK(cudaMemcpyAsync(dbg_out, h->pooled.p, (size_t)B * 2 * D * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return SKB_OK;
    }
    if (stop) {
        set_last_error(__FILE__, __LINE__, "unknown debug stage");
        return SKB_ERR_ARG;
    }
    return head_and_logits(h, norm_embedding, emb_out, logits_out, st);
}

static int forward_tdnn(skb_xtractor* h, const float* wave, int norm_embedding, float* emb_out, float* logits_out,
                        const char* stop, int h_max, float* dbg_out, int64_t* per_utt, cudaStream_t st) {
    const Model& m = h->m;
    Plan& pl = h->plan;
    const int B = pl.B;
    const int* d32 = h->d32;
    const long long* d64 = h->d64;
    float* feats = (float*)h->feats.p;
    {
        ProfScope ps(PROF_FRONTEND, st);
        SKB_TRY(frontend_launch(m.fe, wave, d64 + pl.o_wave_off, d32 + pl.o_wave_len, d64 + pl.o_feat_off, d32 + pl.o_nframes, B,
                                pl.t_max, feats, (float2*)h->cmvn.p, h->cmvn_part.p, false, nullptr, st));
    }
    // raw MFCCs + CMVN statistics; the pack kernel normalises on the fly (no separate pass over the features)
    const Level& L0 = pl.lv[0];
    SKB_TRY(launch_pack_frames(m.bf16, feats, m.fe.n_out, L0.C, (int)pl.total_frames, d32 + pl.o_row_src, d32 + L0.o_row_b,
                               (const float2*)h->cmvn.p, (uint16_t*)h->act[0].p, L0.plane, L0.G, st));
    for (int i = 0; i < 5; ++i) {
        int shifts[10];
        for (int k = 0; k < m.tdnn_k[i]; ++k) shifts[k] = k * m.tdnn_d[i];
        const Level& Lin = pl.lv[i];
        const Level& Lout = pl.lv[i + 1];
        // validity (row_h) of the OUTPUT rows decides what gets stored as non-zero
        ProfScope ps(PROF_CONV, st);
        SKB_TRY(run_conv(h, m.tdnn[i], 2, Lin, (const uint16_t*)h->act[i].p, (uint16_t*)h->act[i + 1].p, 2, shifts, nullptr, nullptr,
                         &Lout, nullptr, st));
        if (stop) {
            char name[32];
            snprintf(name, sizeof(name), "tdnn%d", i + 1);
            if (!strcmp(stop, name)) return export_stage(h, (const uint16_t*)h->act[i + 1].p, Lout, h_max, dbg_out, per_utt, st);
        }
    }
    const Level& L5 = pl.lv[5];
    const int D = m.pool_D;
    ProfScope pool_scope(PROF_POOL, st);
    // mean / unbiased std over the valid frames of each utterance, read straight from the 16-bit planes (W == 1: a pixel is
    // a frame; the first T - 14 rows of an utterance are its valid output frames)
    SKB_TRY(launch_meanstd_planes(m.bf16, (const uint16_t*)h->act[5].p, L5.plane, L5.G, d32 + L5.o_utt_row0, d32 + pl.o_pool_nfr, B, D,
                                  m.pool_s, m.pool_t, (float*)h->pooled.p, st));
    if (stop && !strcmp(stop, "pooled")) {
        *per_utt = 2 * D;
        SKB_CUDA_CHECK(cudaMemcpyAsync(dbg_out, h->pooled.p, (size_t)B * 2 * D * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return SKB_OK;
    }
    if (stop) {
        set_last_error(__FILE__, __LINE__, "unknown debug stage");
        return SKB_ERR_ARG;
    }
    return head_and_logits(h, norm_embedding, emb_out, logits_out, st);
}

static int forward_any(skb_xtractor* h, const float* wave, const int64_t* lengths, int B, int norm_embedding, float* emb,
                       float* logits, const char* stop, int h_max, float* dbg, int64_t* per_utt, cudaStream_t st) {
    if (!h || !wave || !lengths || B <= 0) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    if (current_device() != h->device) {
        set_last_error(__FILE__, __LINE__, "this extractor handle lives on another CUDA device than the current one");
        return SKB_ERR_STATE;
    }
    SKB_TRY(build_plan(h, lengths, B, st));
    if (is_resnet(h->m.archi)) return forward_hr34(h, wave, norm_embedding, emb, logits, stop, h_max, dbg, per_utt, st);
    return forward_tdnn(h, wave, norm_embedding, emb, logits, stop, h_max, dbg, per_utt, st);
}

}  // namespace skb

// ----------------------------------------------------------------------------- C ABI
extern "C" {

int skb_version(void) { return 100; }
const char* skb_last_error(void) { return g_err; }
int64_t skb_kernel_launches(void) { return (int64_t)g_launches.load(); }

void skb_profile_enable(int on) {
    g_prof_on = on != 0;
}
int skb_profile_read(float* ms_by_category, int n_categories) {
    if (!ms_by_category || n_categories < PROF_NCAT) {
        set_last_error(__FILE__, __LINE__, "profile_read: need room for 8 categories");
        return SKB_ERR_ARG;
    }
    for (int i = 0; i < n_categories; ++i) ms_by_category[i] = 0.f;
    SKB_CUDA_CHECK(cudaDeviceSynchronize());
    for (auto& e : g_prof) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) ms_by_category[e.cat] += ms;
        cudaEventDestroy(e.a);
        cudaEventDestroy(e.b);
    }
    g_prof.clear();
    return SKB_OK;
}

int skb_xtractor_create(int archi, int n_tensors, const char* const* names, const float* const* data,
                        const int64_t* const* shapes, const int* ndims, int compute_dtype, float margin_s,
                        skb_xtractor_t** out) {
    if (!out || !names || !data || !shapes || !ndims || (archi != SKB_ARCHI_XVECTOR && !is_resnet(archi))) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    int dev_count = 0;
    if (cudaGetDeviceCount(&dev_count) != cudaSuccess || dev_count == 0) {
        set_last_error(__FILE__, __LINE__, "no CUDA device: sidekit_b200 has no CPU fallback");
        return SKB_ERR_CUDA;
    }
    WeightMap w;
    for (int i = 0; i < n_tensors; ++i) {
        HostTensor t;
        t.p = data[i];
        t.shape.assign(shapes[i], shapes[i] + ndims[i]);
        w[names[i]] = t;
    }
    skb_xtractor* h = new skb_xtractor();
    h->device = current_device();
    if (h->ovf.ensure(sizeof(unsigned)) != SKB_OK || cudaMemset(h->ovf.p, 0, sizeof(unsigned)) != cudaSuccess) {
        delete h;
        set_last_error(__FILE__, __LINE__, "cannot allocate the overflow counter");
        return SKB_ERR_CUDA;
    }
    h->m.archi = archi;
    h->m.bf16 = compute_dtype == 1;
    h->m.margin_s = margin_s;
    int rc = build_frontend(w, &h->m);
    if (!rc) rc = is_resnet(archi) ? build_hr34(w, &h->m) : build_tdnn(w, &h->m);
    if (rc) {
        skb_xtractor_destroy(h);
        return rc;
    }
    *out = h;
    return SKB_OK;
}

void skb_xtractor_destroy(skb_xtractor_t* h) {
    if (!h) return;
    free_model(&h->m);
    h->slot.release();
    DevBuf* bufs[] = {&h->feats, &h->sums, &h->scale, &h->poolX, &h->poolH, &h->poolL, &h->gc, &h->hb,
                      &h->pooled, &h->lin, &h->emb_pre, &h->emb, &h->logits, &h->wave, &h->dbg, &h->brd, &h->cmvn,
                      &h->cmvn_part, &h->skinny_ws, &h->ovf};
    for (auto* b : bufs) b->release();
    for (auto& b : h->act) b.release();
    for (auto& c : h->cache) c.slot.release();
    packed_free(&h->poolA);
    delete h;
}

int skb_xtractor_embedding_size(const skb_xtractor_t* h) { return h ? h->m.emb : 0; }
int skb_xtractor_speaker_number(const skb_xtractor_t* h) { return h ? h->m.n_spk : 0; }
int skb_xtractor_num_frames(const skb_xtractor_t* h, int64_t n_samples) { return h ? num_frames(h->m, n_samples) : 0; }

int skb_xtractor_forward(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt, int norm_embedding,
                         float* emb_dev, float* logits_dev, void* stream) {
    if (!emb_dev) {
        set_last_error(__FILE__, __LINE__, "emb_dev is NULL");
        return SKB_ERR_ARG;
    }
    return forward_any(h, wave_dev, lengths, n_utt, norm_embedding, emb_dev, logits_dev, nullptr, 0, nullptr, nullptr,
                       (cudaStream_t)stream);
}

int skb_xtractor_forward_host(skb_xtractor_t* h, const float* wave_host, const int64_t* lengths, int n_utt, int norm_embedding,
                              float* emb_host, float* logits_host, void* stream) {
    if (!h || !wave_host || !lengths || !emb_host || n_utt <= 0) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int64_t total = 0;
    for (int i = 0; i < n_utt; ++i) total += lengths[i];
    SKB_TRY(h->wave.ensure((size_t)total * sizeof(float)));
    SKB_TRY(h->emb.ensure((size_t)n_utt * h->m.emb * sizeof(float)));
    if (logits_host) SKB_TRY(h->logits.ensure((size_t)n_utt * h->m.n_spk * sizeof(float)));
    SKB_CUDA_CHECK(cudaMemcpyAsync(h->wave.p, wave_host, (size_t)total * sizeof(float), cudaMemcpyHostToDevice, st));
    SKB_TRY(forward_any(h, (const float*)h->wave.p, lengths, n_utt, norm_embedding, (float*)h->emb.p,
                        logits_host ? (float*)h->logits.p : nullptr, nullptr, 0, nullptr, nullptr, st));
    SKB_CUDA_CHECK(cudaMemcpyAsync(emb_host, h->emb.p, (size_t)n_utt * h->m.emb * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (logits_host)
        SKB_CUDA_CHECK(cudaMemcpyAsync(logits_host, h->logits.p, (size_t)n_utt * h->m.n_spk * sizeof(float), cudaMemcpyDeviceToHost, st));
    SKB_CUDA_CHECK(cudaStreamSynchronize(st));
    return SKB_OK;
}

int skb_xtractor_reserve(skb_xtractor_t* h, int max_utts, int64_t max_total_samples, void* stream) {
    if (!h || max_utts <= 0 || max_total_samples <= 0) {
        set_last_error(__FILE__, __LINE__, "reserve: bad arguments");
        return SKB_ERR_ARG;
    }
    if (current_device() != h->device) {
        set_last_error(__FILE__, __LINE__, "this extractor handle lives on another CUDA device than the current one");
        return SKB_ERR_STATE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // The largest tables / work buffers any batch within the budget can need: `max_utts` utterances sharing the audio
    // evenly (most lines, most pad lines, most pixels on every level), plus a few per cent for rounding.
    const int64_t min_len = h->m.fe.n_fft / 2 + 1 + 14 * (int64_t)h->m.fe.hop;
    const int64_t total = max_total_samples + max_total_samples / 20;
    const int64_t each = std::max<int64_t>(total / max_utts + 1, min_len);
    std::vector<int64_t> lengths((size_t)max_utts, each);
    SKB_TRY(build_plan(h, lengths.data(), max_utts, st));
    h->hw_tab32 += h->hw_tab32 / 16; h->hw_tab64 += h->hw_tab64 / 16; h->hw_pixmeta += h->hw_pixmeta / 16;
    {   // the buffers the forward pass itself sizes on demand (by pooled frames / batch size)
        const Model& m = h->m;
        const int B = max_utts, D = m.pool_D;
        size_t sk = std::max(skinny_gemm_ws_floats(B, m.emb, 2 * D), skinny_gemm_ws_floats(B, std::max(m.n_spk, 1), m.emb));
        if (is_resnet(m.archi)) {
            const int F = h->plan.pool_frames;
            sk = std::max(sk, skinny_gemm_ws_floats(B, m.att_A, 2 * D));
            if (F > h->poolA_rows) {
                packed_free(&h->poolA);
                h->poolA_rows = 0;
                SKB_TRY(packed_alloc_zero(&h->poolA, F + F / 8 + 128, D, st));
                h->poolA_rows = h->poolA.rows;
            }
            SKB_TRY(gemm_workspace_reserve(F + F / 8 + 128, std::max(m.att_A, 64)));
        }
        SKB_TRY(h->skinny_ws.ensure(sk * sizeof(float)));
    }
    // every slot of the plan cache now, at the high-water sizes: nothing is allocated once the bulk run has started
    while (h->cache.size() <= kPlanCacheEntries) {
        h->cache.emplace_back();
        skb_xtractor::CachedPlan& c = h->cache.back();       // an empty plan (B = 0) never matches a request; stamp 0 = recycled first
        SKB_TRY(c.slot.tab32.ensure(h->hw_tab32));
        SKB_TRY(c.slot.tab64.ensure(h->hw_tab64));
        SKB_TRY(c.slot.pixmeta.ensure(h->hw_pixmeta));
        SKB_TRY(c.slot.stage32.ensure(h->hw_tab32));
        SKB_TRY(c.slot.stage64.ensure(h->hw_tab64));
        SKB_CUDA_CHECK(cudaEventCreateWithFlags(&c.slot.uploaded, cudaEventDisableTiming));
        SKB_CUDA_CHECK(cudaEventRecord(c.slot.uploaded, st));
    }
    SKB_CUDA_CHECK(cudaStreamSynchronize(st));
    return SKB_OK;
}

int skb_xtractor_overflow_count(skb_xtractor_t* h, void* stream, int64_t* count) {
    if (!h || !count) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    unsigned v = 0;
    SKB_CUDA_CHECK(cudaMemcpyAsync(&v, h->ovf.p, sizeof(unsigned), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    SKB_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    *count = (int64_t)v;
    return SKB_OK;
}

int skb_xtractor_wait_tables(skb_xtractor_t* h, void* stream) {
    if (!h) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    // the geometry tables of the last forward call go over the same host-to-device copy engine as a caller's waveform
    // copies: a 67 MB waveform copy that becomes eligible at the same instant as the tables delays the forward by its
    // whole duration (profiles/r02u_e2e_timeline.txt), so the copy stream lets the tables go first
    if (h->slot.uploaded) SKB_CUDA_CHECK(cudaStreamWaitEvent((cudaStream_t)stream, h->slot.uploaded, 0));
    return SKB_OK;
}

int skb_xtractor_pre_embedding(skb_xtractor_t* h, int n_utt, float* out_dev, void* stream) {
    if (!h || !out_dev || !h->plan_valid || n_utt != h->plan.B) {
        set_last_error(__FILE__, __LINE__, "pre_embedding: no matching forward call");
        return SKB_ERR_STATE;
    }
    SKB_CUDA_CHECK(cudaMemcpyAsync(out_dev, h->emb_pre.p, (size_t)n_utt * h->m.emb * sizeof(float), cudaMemcpyDeviceToDevice,
                                   (cudaStream_t)stream));
    return SKB_OK;
}

int skb_xtractor_frontend(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt, int t_max,
                          float* feats_dev, void* stream) {
    if (!h || !wave_dev || !lengths || !feats_dev || n_utt <= 0) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (current_device() != h->device) {
        set_last_error(__FILE__, __LINE__, "this extractor handle lives on another CUDA device than the current one");
        return SKB_ERR_STATE;
    }
    SKB_TRY(build_plan(h, lengths, n_utt, st));
    Plan& pl = h->plan;
    if (t_max < pl.t_max) {
        set_last_error(__FILE__, __LINE__, "t_max smaller than the longest utterance's frame count");
        return SKB_ERR_ARG;
    }
    SKB_CUDA_CHECK(cudaMemsetAsync(feats_dev, 0, (size_t)n_utt * h->m.fe.n_out * t_max * sizeof(float), st));
    return frontend_launch(h->m.fe, wave_dev, h->d64 + pl.o_wave_off, h->d32 + pl.o_wave_len, h->d64 + pl.o_feat_off,
                           h->d32 + pl.o_nframes, n_utt, t_max, (float*)h->feats.p, (float2*)h->cmvn.p, h->cmvn_part.p, true,
                           feats_dev, st);
}

int skb_xtractor_debug_stage(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt, const char* stage,
                             int h_max, float* out_dev, int64_t* per_utt, void* stream) {
    if (!stage || !out_dev || !per_utt) {
        set_last_error(__FILE__, __LINE__, "bad arguments");
        return SKB_ERR_ARG;
    }
    return forward_any(h, wave_dev, lengths, n_utt, 1, nullptr, nullptr, stage, h_max, out_dev, per_utt, (cudaStream_t)stream);
}

}  // extern "C"

#include "module_ops.cuh"
