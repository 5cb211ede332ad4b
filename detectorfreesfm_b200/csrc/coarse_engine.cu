// HP-1: pairwise coarse matcher (LoFTR coarse_only path) on the B200 -- layer schedule and C ABI.
// Reference: third_party/LoFTR/src/loftr/loftr.py:29-73 (stage order), backbone/resnet_fpn.py:100-108 (coarse sub-graph),
// loftr_module/transformer.py:35-101, utils/coarse_matching.py:84-258.
#include <algorithm>
#include <map>
#include <memory>
#include <tuple>

#include "../../include/dfsfm_b200.h"
#include "engine_common.h"
#include "fine_kernels.cuh"
#include "refine_kernels.cuh"

namespace dfsfm {

namespace {

struct Geom {
    int H, W, Hp, Wp;
    long long rows;  // per image
    Geom() : H(0), W(0), Hp(0), Wp(0), rows(0) {}
    Geom(int h, int w) : H(h), W(w), Hp(h + 1), Wp(w + 1), rows(static_cast<long long>(h + 1) * (w + 1)) {}
    FlatGeom flat() const { return FlatGeom{Hp, Wp, H, W}; }
};

struct ParityBuf {  // [4 parity][2 hl][rows][C]
    __half* base = nullptr;
    long long rows = 0;
    int C = 0;
    HL plane(int k) const {
        HL b;
        b.hi = base + static_cast<long long>(k) * 2 * rows * C;
        b.rows = rows;
        b.C = C;
        return b;
    }
    long long plane_stride() const { return 2 * rows * C; }
};

struct FeatWs {  // backbone workspace for 1 or 2 images of one geometry: every flat buffer holds image 0, then image 1, each with its halo
    Geom g2, g4, g8;
    HL a2, b2, c2;
    ParityBuf p1, p2;
    HL a4, b4, a8, b8, c8;
    // fine FPN branch (allocated on first use)
    bool fine = false;
    HL x3o, t4a, t4b, x2o, t2a, t2b;
    float* f4 = nullptr;
    float* f2 = nullptr;
};

struct FineWs {  // fine-stage workspace for up to `cap` coarse matches
    int cap = 0;
    HL win, x, msg, m1, hid, cin, cwin;
    float *xf = nullptr, *qkv = nullptr, *u = nullptr, *kvstate = nullptr, *kvpart = nullptr, *d_query = nullptr;
    Seg* segs = nullptr;
    TrackRec* tracks = nullptr;
    ViewRec* views = nullptr;
};

struct TokWs {  // transformer / matcher workspace for up to `cap` tokens per side
    int cap = 0;
    HL x[2], msg[2], m1[2], hid[2];
    float* qkv[2] = {nullptr, nullptr};
    float* xf = nullptr;       // joint fp32 token array (residual stream)
    HL g;                      // [2 segments * 256][256] per-call folded attention-state x merge matrices (attn_fold_merge_kernel)
    float* ksum = nullptr;     // [2][256]
    float* kvp_part = nullptr;   // KvEpi per-CTA partial states [2 segments][2 column tiles][CTAs][4*32*33]
    unsigned* kvp_flags = nullptr;
    int L = 0, L1 = 0, S = 0;  // layout of the joint token array of the current transformer() call
    int kv_chunks = 0;
    float* kv_part = nullptr;
    float* kv_state = nullptr;
    Seg* seg_dev = nullptr;
    float2* part = nullptr;
    float* stat[2] = {nullptr, nullptr};  // log2-sum-exp2 per row / column
    unsigned long long* best[2] = {nullptr, nullptr};
};

}  // namespace

class CoarseEngine {
  public:
    explicit CoarseEngine(int device) : device_(device) {
        DFSFM_CUDA(cudaSetDevice(device));
        DFSFM_CUDA(cudaFuncSetAttribute(attn_apply_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_smem_bytes<32>()));
    }
    ~CoarseEngine() {
        for (auto& kv : feat_ws_) free_feat(kv.second);
        free_tok(tok_);
    }
    ParamStore params;

    // n_img = 1 or 2 images of the same size in one launch per layer; feat_f (the fine FPN branch) only with one image
    void features(const float* const* imgs, int n_img, int H, int W, const float* pe, float* const* tokens, float* feat_f, cudaStream_t st);
    void fine_match(const float* ff0, int Hf0, int Wf0, const float* ff1, int Hf1, int Wf1, const float* fc0, int w0c, const float* fc1, int w1c,
                    const int* i_ids, const int* j_ids, int M, float* coords_out, float* std_out, cudaStream_t st);
    void transformer(float* f0, int L, float* f1, int S, cudaStream_t st);
    void match(const float* f0, int h0c, int w0c, const float* f1, int h1c, int w1c, float thr, int border, float temperature, int* i_ids,
               int* j_ids, float* mconf, int* n_matches, int capacity, float* conf_out, cudaStream_t st);

  private:
    int device_;
    std::map<std::tuple<int, int, int>, FeatWs> feat_ws_;  // (H, W, n_img)
    TokWs tok_;
    unsigned kv_epoch_ = 0;
    FineWs fine_;
    void ensure_fine(int M);
    void fine_branch(FeatWs& w, float* feat_f, cudaStream_t st);
    void layer128(int li, bool self, int x0, int xn, int s0, int sn, const Seg* kv_segs, int n_kv, const Seg* apply_segs, int n_apply, cudaStream_t st);

    FeatWs& get_feat_ws(int H, int W, int n_img);
    void ensure_tok(int n);
    static void free_feat(FeatWs& w);
    static void free_tok(TokWs& w);

    template <int BN>
    void conv(const HL* ins, int n_in, GemmCore core, const std::string& wname, ConvEpiParams ep, cudaStream_t st, bool allow_slab = true);
    void conv_l3(int bn, const HL* ins, int n_in, const GemmCore& core, const std::string& wname, const ConvEpiParams& ep, cudaStream_t st);
    void layer_call(int li, bool self, int x0, int xn, int s0, int sn, int kv_seg0, int n_segs, int apply_seg0, int max_count, cudaStream_t st,
                    int seg_row0 = 0);
};

static int kv_tok() {  // tokens per KV-partial CTA (A/B: DFSFM_KV_TOK)
    static int v = 0;
    if (!v) {
        const char* e = getenv("DFSFM_KV_TOK");
        v = e ? atoi(e) : kKvTokPerCta;
        if (v < 16) v = 16;
    }
    return v;
}
// DFSFM_ATTN_FOLD=0: the round-1 schedule (fp32 q/k/v, attn_apply kernel, merge on the message) as an A/B reference.
static bool attn_fold() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFSFM_ATTN_FOLD");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v == 1 && engine_version() == 2;
}
// DFSFM_KV_EPI=0: k/v written as fp32 and reduced by kv_partial/kv_final (A/B reference for the fused-epilogue state reduction)
static bool kv_epi() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFSFM_KV_EPI");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v == 1;
}
// DFSFM_ENC_FUSED=0: q / merge / mlp.0 / mlp.2 as four GEMM launches (A/B reference for the fused encoder-layer kernel)
static bool enc_fused() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFSFM_ENC_FUSED");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v == 1;
}
static bool lin_bn128() {  // A/B switch: 128-wide N tiles for the wide linears (QKV, KV, mlp.0): twice the tiles, better last-round fill
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFSFM_LIN_BN128");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

static ParityBuf parity_alloc(long long rows, int C) {
    ParityBuf p;
    p.rows = rows;
    p.C = C;
    const size_t bytes = static_cast<size_t>(8) * rows * C * sizeof(__half);
    DFSFM_CUDA(cudaMalloc(&p.base, bytes));
    zero_device_sync(p.base, 0, bytes);
    return p;
}

FeatWs& CoarseEngine::get_feat_ws(int H, int W, int n_img) {
    const auto key = std::make_tuple(H, W, n_img);
    auto it = feat_ws_.find(key);
    if (it != feat_ws_.end()) return it->second;
    if (feat_ws_.size() >= 8) {  // bound the cache: drop everything (geometries repeat within a scene)
        for (auto& kv : feat_ws_) free_feat(kv.second);
        feat_ws_.clear();
    }
    FeatWs w;
    w.g2 = Geom(H / 2, W / 2);
    w.g4 = Geom(H / 4, W / 4);
    w.g8 = Geom(H / 8, W / 8);
    DFSFM_CHECK(n_img * w.g2.rows < (1ll << 31), "image too large for 32-bit row indices");
    w.a2 = hl_alloc(n_img * w.g2.rows, 128);
    w.b2 = hl_alloc(n_img * w.g2.rows, 128);
    w.c2 = hl_alloc(n_img * w.g2.rows, 128);
    w.p1 = parity_alloc(n_img * w.g4.rows, 128);
    w.a4 = hl_alloc(n_img * w.g4.rows, 208);
    w.b4 = hl_alloc(n_img * w.g4.rows, 208);
    w.p2 = parity_alloc(n_img * w.g8.rows, 208);
    w.a8 = hl_alloc(n_img * w.g8.rows, 256);
    w.b8 = hl_alloc(n_img * w.g8.rows, 256);
    w.c8 = hl_alloc(n_img * w.g8.rows, 256);
    return feat_ws_.emplace(key, w).first->second;
}
void CoarseEngine::free_feat(FeatWs& w) {
    hl_free(w.a2); hl_free(w.b2); hl_free(w.c2); hl_free(w.a4); hl_free(w.b4); hl_free(w.a8); hl_free(w.b8); hl_free(w.c8);
    if (w.p1.base) cudaFree(w.p1.base);
    if (w.p2.base) cudaFree(w.p2.base);
    if (w.fine) {
        hl_free(w.x3o); hl_free(w.t4a); hl_free(w.t4b); hl_free(w.x2o); hl_free(w.t2a); hl_free(w.t2b);
        cudaFree(w.f4); cudaFree(w.f2);
    }
}

template <int BN>
void CoarseEngine::conv(const HL* ins, int n_in, GemmCore core, const std::string& wname, ConvEpiParams ep, cudaStream_t st, bool allow_slab) {
    const HL& w = params.mat(wname + ".w");
    const bool slab = BN <= 128 && allow_slab && slab_applicable(core, n_in);
    TmapPack maps;
    for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = make_tmap(ins[i < n_in ? i : 0], slab ? kSlabRows : kBM);
    maps.b = make_tmap(w, bbox(BN));
    core.b_row0 = 0;
    DFSFM_CHECK(static_cast<long long>(core.num_taps) * core.cpad == w.C, "weight K does not match taps*cpad for " + wname);
    ep.M = core.M;
    ep.bias = params.has_vec(wname + ".b") ? params.vec(wname + ".b") : nullptr;
    if constexpr (BN <= 128) {
        if (slab) {
            launch_gemm_slab_counted<BN, ConvEpi>(maps, core, ep, ep.N, st, "conv");
            return;
        }
    }
    launch_gemm_counted<BN, true, ConvEpi>(maps, core, ep, ep.N, st, "conv");
}

// Column tile width of the 256-channel layer-3 convs: 256, or two 128-wide tiles per row tile when that takes fewer SM-pair rounds
// counted in half-tile time (a 128-wide tile does half the MMAs of a 256-wide one).  Two 832x832 images: 87 row tiles are 2 full
// rounds on 74 SM pairs, 174 half tiles are 3 half rounds.  A tie keeps 256 (half the operand traffic per output).
static int layer3_bn(int M) {
    const int pairs = sm_count() / 2;
    const int row_tiles = (M + 2 * kBM - 1) / (2 * kBM);
    const int full_rounds = (row_tiles + pairs - 1) / pairs;
    const int half_rounds = (2 * row_tiles + pairs - 1) / pairs;
    return half_rounds < 2 * full_rounds ? 128 : 256;
}
// The 128-wide variant runs without tap slabs: the slab kernel orders a row's K steps kchunk-major within a group of three taps, the
// plain one tap-major, so only the plain kernel accumulates in the 256-wide kernel's order and the outputs do not depend on the width.
// (Slabs bought nothing here: 51.7 ms of conv per 28-pair step with or without them, B200 at 1000 W.)
void CoarseEngine::conv_l3(int bn, const HL* ins, int n_in, const GemmCore& core, const std::string& wname, const ConvEpiParams& ep,
                           cudaStream_t st) {
    if (bn == 128) conv<128>(ins, n_in, core, wname, ep, st, false);
    else conv<256>(ins, n_in, core, wname, ep, st);
}

static ConvEpiParams epi_flat(const Geom& g, int N, const HL& out, bool relu, const HL* res) {
    ConvEpiParams e;
    memset(&e, 0, sizeof(e));
    e.N = N;
    e.g = g.flat();
    e.relu = relu ? 1 : 0;
    if (res) { e.res_hi = res->hi; e.res_lo = res->lo(); e.res_ld = res->C; }
    e.out_mode = OUT_FLAT;
    e.out_hi = out.hi;
    e.out_lo = out.lo();
    e.out_ld = out.C;
    return e;
}
static ConvEpiParams epi_parity(const Geom& g, int N, const ParityBuf& out, bool relu, const HL* res) {
    ConvEpiParams e = epi_flat(g, N, out.plane(0), relu, res);
    e.out_mode = OUT_PARITY;
    e.plane_stride = out.plane_stride();
    return e;
}

// The images of a pair are independent until the transformer, so two images of one size share every launch: each conv runs over the
// rows of both flat buffers (a tap of an interior output row never leaves its own image's block, and the epilogue maps every row to its
// image), which gives the launches twice the tiles to spread over the SMs.  Every output row accumulates in the same order as in a
// one-image call, so the tokens are bitwise the same.
void CoarseEngine::features(const float* const* imgs, int n_img, int H, int W, const float* pe, float* const* tokens, float* feat_f,
                            cudaStream_t st) {
    DFSFM_CHECK(H % 8 == 0 && W % 8 == 0 && H >= 16 && W >= 16, "image size must be a multiple of 8 (CoarseMatchingDataset df=8)");
    DFSFM_CHECK(n_img == 1 || (n_img == 2 && !feat_f), "one image, or two without the fine branch");
    FeatWs& w = get_feat_ws(H, W, n_img);
    // conv1 + bn1 + relu (resnet_fpn.py:102)
    {
        dim3 grid((w.g2.W + kStemTW - 1) / kStemTW, (w.g2.H + kStemTH - 1) / kStemTH, n_img);
        { LaunchScope ls("stem", st);
          stem_conv_kernel<<<grid, 128, 0, st>>>(imgs[0], imgs[n_img - 1], H, W, params.vec("stem.w"), params.vec("stem.b"), w.a2.hi, w.a2.lo()); }
        DFSFM_CUDA(cudaGetLastError());
    }
    GemmCore c;
    memset(&c, 0, sizeof(c));
    // layer1 (two BasicBlocks, stride 1, 128 ch) -- resnet_fpn.py:32-40,103
    c.M = static_cast<int>(n_img * w.g2.rows);
    set_k(c, 128);
    conv_taps_s1(c, 3, w.g2.Wp);
    { const HL in[1] = {w.a2}; conv<128>(in, 1, c, "l1.0.c1", epi_flat(w.g2, 128, w.b2, true, nullptr), st); }
    { const HL in[1] = {w.b2}; conv<128>(in, 1, c, "l1.0.c2", epi_flat(w.g2, 128, w.c2, true, &w.a2), st); }
    { const HL in[1] = {w.c2}; conv<128>(in, 1, c, "l1.1.c1", epi_flat(w.g2, 128, w.b2, true, nullptr), st); }
    { const HL in[1] = {w.b2}; conv<128>(in, 1, c, "l1.1.c2", epi_parity(w.g2, 128, w.p1, true, &w.c2), st); }
    // layer2 (stride 2, 196 -> 208 padded channels) -- the 1x1 stride-2 downsample rides as a 10th tap of conv2
    c.M = static_cast<int>(n_img * w.g4.rows);
    set_k(c, 128);
    conv_taps_s2(c, w.g4.Wp);
    { const HL in[4] = {w.p1.plane(0), w.p1.plane(1), w.p1.plane(2), w.p1.plane(3)};
      conv<208>(in, 4, c, "l2.0.c1", epi_flat(w.g4, 208, w.a4, true, nullptr), st); }
    set_k(c, 208);
    conv_taps_s1(c, 3, w.g4.Wp);
    c.num_taps = 10; c.tap_map[9] = 1; c.tap_shift[9] = 0;
    { const HL in[2] = {w.a4, w.p1.plane(0)}; conv<208>(in, 2, c, "l2.0.c2", epi_flat(w.g4, 208, w.b4, true, nullptr), st); }
    conv_taps_s1(c, 3, w.g4.Wp);
    { const HL in[1] = {w.b4}; conv<208>(in, 1, c, "l2.1.c1", epi_flat(w.g4, 208, w.a4, true, nullptr), st); }
    { const HL in[1] = {w.a4}; conv<208>(in, 1, c, "l2.1.c2", epi_parity(w.g4, 208, w.p2, true, &w.b4), st); }
    // layer3 (stride 2, 256 ch)
    c.M = static_cast<int>(n_img * w.g8.rows);
    const int bn3 = layer3_bn(c.M);
    set_k(c, 208);
    conv_taps_s2(c, w.g8.Wp);
    { const HL in[4] = {w.p2.plane(0), w.p2.plane(1), w.p2.plane(2), w.p2.plane(3)};
      conv_l3(bn3, in, 4, c, "l3.0.c1", epi_flat(w.g8, 256, w.a8, true, nullptr), st); }
    set_k(c, 256);
    conv_taps_s1(c, 3, w.g8.Wp);
    c.num_taps = 10; c.tap_map[9] = 1; c.tap_shift[9] = 0;
    { const HL in[2] = {w.a8, w.p2.plane(0)}; conv_l3(bn3, in, 2, c, "l3.0.c2", epi_flat(w.g8, 256, w.b8, true, nullptr), st); }
    conv_taps_s1(c, 3, w.g8.Wp);
    { const HL in[1] = {w.b8}; conv_l3(bn3, in, 1, c, "l3.1.c1", epi_flat(w.g8, 256, w.a8, true, nullptr), st); }
    { const HL in[1] = {w.a8}; conv_l3(bn3, in, 1, c, "l3.1.c2", epi_flat(w.g8, 256, w.c8, true, &w.b8), st); }
    // layer3_outconv (1x1) + position encoding + flatten to tokens (resnet_fpn.py:108, loftr.py:58)
    conv_taps_s1(c, 1, w.g8.Wp);
    {
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.N = 256;
        e.g = w.g8.flat();
        e.addend = pe;
        e.out_mode = OUT_DENSE;
        e.out_f32 = tokens[0];
        e.out_f32_1 = n_img == 2 ? tokens[1] : nullptr;
        e.out_f32_ld = 256;
        if (feat_f) {
            if (!w.fine) {
                w.x3o = hl_alloc(w.g8.rows, 256);
                w.t4a = hl_alloc(w.g4.rows, 256); w.t4b = hl_alloc(w.g4.rows, 256); w.x2o = hl_alloc(w.g4.rows, 208);
                w.t2a = hl_alloc(w.g2.rows, 208); w.t2b = hl_alloc(w.g2.rows, 208);
                DFSFM_CUDA(cudaMalloc(&w.f4, static_cast<size_t>(w.g4.rows) * 256 * sizeof(float)));
                DFSFM_CUDA(cudaMalloc(&w.f2, static_cast<size_t>(w.g2.rows) * 208 * sizeof(float)));
                w.fine = true;
            }
            // tokens get x3_out + PE; the raw x3_out planes (same flat geometry, no PE) feed the FPN top-down path.
            // OUT_DENSE and OUT_FLAT differ only in the row mapping, so the planes come from a second epilogue pass below.
        }
        const HL in[1] = {w.c8};
        conv_l3(bn3, in, 1, c, "out3", e, st);
        if (feat_f) {
            ConvEpiParams e2 = epi_flat(w.g8, 256, w.x3o, false, nullptr);
            conv_l3(bn3, in, 1, c, "out3", e2, st);
            fine_branch(w, feat_f, st);
        }
    }
}

// FPN top-down path to the 1/2-resolution fine feature map (resnet_fpn.py:110-118), only for match type 'coarse_fine'.
void CoarseEngine::fine_branch(FeatWs& w, float* feat_f, cudaStream_t st) {
    GemmCore c;
    memset(&c, 0, sizeof(c));
    auto up_add = [&](const HL& low, const Geom& gl, int C, const float* lateral, const HL& out) {
        const long long total = static_cast<long long>(2 * gl.H) * (2 * gl.W) * (C / 8);
        LaunchScope ls("upsample", st);
        upsample2x_add_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(low.hi, low.lo(), gl.H, gl.W, C, lateral, out.hi, out.lo(), total);
        DFSFM_CUDA(cudaGetLastError());
    };
    // x2_out = layer2_outconv(x2) [1x1 on the four parity planes of x2] + up(x3_out)
    c.M = static_cast<int>(w.g8.rows);
    set_k(c, 208);
    conv_taps_s1(c, 1, w.g8.Wp);
    for (int k = 0; k < 4; ++k) {
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.N = 256; e.g = w.g8.flat(); e.out_mode = OUT_UNPARITY; e.upy = k >> 1; e.upx = k & 1; e.ohp = w.g4.Hp; e.owp = w.g4.Wp;
        e.out_f32 = w.f4; e.out_f32_ld = 256;
        const HL in[1] = {w.p2.plane(k)};
        conv<256>(in, 1, c, "fpn.l2o", e, st);
    }
    up_add(w.x3o, w.g8, 256, w.f4, w.t4a);
    c.M = static_cast<int>(w.g4.rows);
    set_k(c, 256);
    conv_taps_s1(c, 3, w.g4.Wp);
    { ConvEpiParams e = epi_flat(w.g4, 256, w.t4b, false, nullptr); e.relu = 2; const HL in[1] = {w.t4a}; conv<256>(in, 1, c, "fpn.l2o2a", e, st); }
    { ConvEpiParams e = epi_flat(w.g4, 208, w.x2o, false, nullptr); const HL in[1] = {w.t4b}; conv<208>(in, 1, c, "fpn.l2o2b", e, st); }
    // x1_out = layer1_outconv(x1) [1x1 on the parity planes of x1] + up(x2_out)
    set_k(c, 128);
    conv_taps_s1(c, 1, w.g4.Wp);
    for (int k = 0; k < 4; ++k) {
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.N = 208; e.g = w.g4.flat(); e.out_mode = OUT_UNPARITY; e.upy = k >> 1; e.upx = k & 1; e.ohp = w.g2.Hp; e.owp = w.g2.Wp;
        e.out_f32 = w.f2; e.out_f32_ld = 208;
        const HL in[1] = {w.p1.plane(k)};
        conv<208>(in, 1, c, "fpn.l1o", e, st);
    }
    up_add(w.x2o, w.g4, 208, w.f2, w.t2a);
    c.M = static_cast<int>(w.g2.rows);
    set_k(c, 208);
    conv_taps_s1(c, 3, w.g2.Wp);
    { ConvEpiParams e = epi_flat(w.g2, 208, w.t2b, false, nullptr); e.relu = 2; const HL in[1] = {w.t2a}; conv<208>(in, 1, c, "fpn.l1o2a", e, st); }
    {
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.N = 128; e.g = w.g2.flat(); e.out_mode = OUT_DENSE; e.out_f32 = feat_f; e.out_f32_ld = 128;
        const HL in[1] = {w.t2b};
        conv<128>(in, 1, c, "fpn.l1o2b", e, st);
    }
}

// -------------------------------------------------------------------------------------------- transformer
void CoarseEngine::free_tok(TokWs& w) {
    for (int s = 0; s < 2; ++s) {
        hl_free(w.x[s]); hl_free(w.msg[s]); hl_free(w.m1[s]); hl_free(w.hid[s]);
        if (w.qkv[s]) cudaFree(w.qkv[s]);
        if (w.stat[s]) cudaFree(w.stat[s]);
        if (w.best[s]) cudaFree(w.best[s]);
        w.qkv[s] = nullptr; w.stat[s] = nullptr; w.best[s] = nullptr;
    }
    if (w.xf) cudaFree(w.xf);
    w.xf = nullptr;
    hl_free(w.g);
    if (w.ksum) cudaFree(w.ksum);
    if (w.kvp_part) cudaFree(w.kvp_part);
    if (w.kvp_flags) cudaFree(w.kvp_flags);
    w.ksum = nullptr; w.kvp_part = nullptr; w.kvp_flags = nullptr;
    if (w.kv_part) cudaFree(w.kv_part);
    if (w.kv_state) cudaFree(w.kv_state);
    if (w.seg_dev) cudaFree(w.seg_dev);
    if (w.part) cudaFree(w.part);
    w.kv_part = w.kv_state = nullptr; w.seg_dev = nullptr; w.part = nullptr;
    w.cap = 0;
}
void CoarseEngine::ensure_tok(int n) {
    if (n <= tok_.cap) return;
    free_tok(tok_);
    const int cap = ((n + 1023) / 1024) * 1024;
    tok_.cap = cap;
    for (int s = 0; s < 2; ++s) {
        tok_.x[s] = hl_alloc(cap, 256);
        tok_.msg[s] = hl_alloc(cap, 256);
        tok_.m1[s] = hl_alloc(cap, 256);
        tok_.hid[s] = hl_alloc(cap, 512);
        DFSFM_CUDA(cudaMalloc(&tok_.qkv[s], static_cast<size_t>(cap) * 768 * sizeof(float)));
        DFSFM_CUDA(cudaMalloc(&tok_.stat[s], static_cast<size_t>(cap) * sizeof(float)));
        DFSFM_CUDA(cudaMalloc(&tok_.best[s], static_cast<size_t>(cap) * sizeof(unsigned long long)));
    }
    tok_.kv_chunks = (cap + kv_tok() - 1) / kv_tok();
    DFSFM_CUDA(cudaMalloc(&tok_.xf, static_cast<size_t>(cap) * 256 * sizeof(float)));
    tok_.g = hl_alloc(512, 256);
    DFSFM_CUDA(cudaMalloc(&tok_.ksum, 512 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&tok_.kvp_part, static_cast<size_t>(4) * sm_count() * kKvPartFloats * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&tok_.kvp_flags, static_cast<size_t>(4) * sm_count() * sizeof(unsigned)));
    zero_device_sync(tok_.kvp_flags, 0, static_cast<size_t>(4) * sm_count() * sizeof(unsigned));
    DFSFM_CUDA(cudaMalloc(&tok_.kv_part, static_cast<size_t>(2) * tok_.kv_chunks * 256 * 33 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&tok_.kv_state, static_cast<size_t>(2) * 256 * 33 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&tok_.seg_dev, 8 * sizeof(Seg)));
    const int tiles = 2 * ((cap + 255) / 256);  // engine 2 writes one partial per half tile
    DFSFM_CUDA(cudaMalloc(&tok_.part, static_cast<size_t>(tiles) * cap * sizeof(float2)));
}

// One LoFTREncoderLayer.forward (transformer.py:35-58) on the token rows [x0, x0+xn) of the joint token array (image 0 at rows
// [0,L), image 1 at [L,L+S)).  `self`: source == x (both images in one call, two attention segments); otherwise the source
// rows are [s0, s0+sn).  kv_segs / apply_segs index the 6-entry device table built in transformer().
// DFSFM_RES_HL=0: keep a separate fp32 residual stream (A/B switch; engine 1 always does)
static bool res_hl() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DFSFM_RES_HL");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v == 1 && engine_version() == 2;
}

void CoarseEngine::layer_call(int li, bool self, int x0, int xn, int s0, int sn, int kv_seg0, int n_segs, int apply_seg0, int max_count,
                              cudaStream_t st, int seg_row0) {
    const std::string p = "tr." + std::to_string(li);
    GemmCore c;
    memset(&c, 0, sizeof(c));
    set_k(c, 256);
    conv_taps_s1(c, 1, 0);
    LinEpiParams e;
    float* qkv = tok_.qkv[0];
    float* xf = tok_.xf;
    auto rows_map = [&](const HL& b, int r0, int n) { return make_tmap(b.hi + static_cast<long long>(r0) * b.C, b.C, n, b.plane_elems(), kBM); };
    const bool fold = attn_fold();
    // v_length of each source segment of this call (self: image 0 / image 1 themselves; cross: the one source image)
    const float qz_len[2] = {static_cast<float>(seg_row0 > 0 ? tok_.L : sn), static_cast<float>(tok_.S)};
    if (fold && kv_epi()) {
        // (1+2) k, v projection of the source rows with the linear-attention state reduced in the GEMM epilogue (KvEpi)
        TmapPack maps;
        maps.b = make_tmap(params.mat(p + ".kvp"), bbox(256));
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], s0, sn);
        KvEpiParams ke;
        memset(&ke, 0, sizeof(ke));
        ke.M = sn;
        ke.seg_row0 = seg_row0;
        if (seg_row0 > 0) {  // both images: rows [0,L) and [L1, L1+S)
            ke.row_begin[0] = 0; ke.row_end[0] = tok_.L; ke.row_begin[1] = tok_.L1; ke.row_end[1] = tok_.L1 + tok_.S;
        } else {
            ke.row_begin[0] = 0; ke.row_end[0] = sn;
        }
        ke.part = tok_.kvp_part; ke.flags = tok_.kvp_flags; ke.epoch = ++kv_epoch_;
        c.M = sn; c.b_row0 = 0;
        const int tiles = ((sn + 2 * kBM - 1) / (2 * kBM)) * 2;
        const int n_ctas = 2 * std::min(tiles, sm_count() / 2);
        { LaunchScope ls("kvproj", st);
          launch_gemm2<256, true, KvEpi>(maps, c, ke, 512, st); }
        // (3) partial states -> V/len -> G = KV . Wm^T and Ksum, in one kernel
        { const HL& wm = params.mat(p + ".merge");
          LaunchScope ls("fold", st);
          kvp_fold_kernel<<<dim3(8, 8, n_segs), 1024, 0, st>>>(tok_.kvp_part, tok_.kvp_flags, ke.epoch, n_ctas, tok_.seg_dev + kv_seg0, wm.hi, wm.lo(),
                                                         tok_.g.hi, tok_.g.lo(), tok_.ksum); }
        DFSFM_CUDA(cudaGetLastError());
    }
    if (fold && !kv_epi()) {
        // (1) k, v of the source rows (elu+1 on k) -> fp32 for the state reduction
        {
            TmapPack maps;
            maps.b = make_tmap(params.mat(p + ".qkv"), bbox(256));
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], s0, sn);
            memset(&e, 0, sizeof(e));
            e.mode = LIN_F32_ELU; e.out_f32_ld = 768;
            c.M = sn; c.b_row0 = 256;
            e.M = sn; e.N = 512; e.elu_cols = 256; e.out_f32 = qkv + static_cast<long long>(s0) * 768; e.out_col0 = 256;
            launch_gemm_counted<256, true, LinEpi>(maps, c, e, 512, st, "lin");
        }
        // (2) KV state(s) of the source segment(s)
        const int chunks = (max_count + kv_tok() - 1) / kv_tok();
        { LaunchScope ls("kv", st);
          kv_partial_kernel<32><<<dim3(chunks, n_segs), 256, 0, st>>>(qkv + 256, qkv + 512, 768, tok_.seg_dev + kv_seg0, tok_.kv_chunks, tok_.kv_part,
                                                                      kv_tok()); }
        { LaunchScope ls("kv_final", st);
          kv_final_kernel<32><<<dim3((256 * 33 + 63) / 64, n_segs), kKvFinalThreads, 0, st>>>(tok_.kv_part, tok_.seg_dev + kv_seg0, tok_.kv_chunks,
                                                                                   tok_.kv_state, kv_tok()); }
    }
    if (fold) {
        // (3) fold the state into the merge projection: G = KV . Wm^T per segment, Ksum as a dense vector
        if (!kv_epi()) {
          const HL& wm = params.mat(p + ".merge");
          LaunchScope ls("fold", st);
          attn_fold_merge_kernel<32><<<dim3(8, n_segs), 256, 0, st>>>(tok_.kv_state, tok_.seg_dev + kv_seg0, wm.hi, wm.lo(), tok_.g.hi, tok_.g.lo(),
                                                                  tok_.ksum); }
        DFSFM_CUDA(cudaGetLastError());
        if (enc_fused() && res_hl()) {
            // (4-7) everything on the attending rows in ONE kernel: q + normaliser, attention/merge, norm1, mlp, norm2 + residual
            EncParams ep;
            memset(&ep, 0, sizeof(ep));
            ep.seg_tile0 = seg_row0 / (2 * kBM);
            ep.ksum = tok_.ksum;
            ep.qz_scale[0] = qz_len[0]; ep.qz_scale[1] = qz_len[1];
            ep.ln1_g = params.vec(p + ".ln1.g"); ep.ln1_b = params.vec(p + ".ln1.b");
            LinEpiParams& e4 = ep.e4;
            e4.M = xn; e4.N = 256; e4.mode = LIN_LN;
            e4.gamma = params.vec(p + ".ln2.g"); e4.beta = params.vec(p + ".ln2.b");
            e4.res_hi = tok_.x[0].hi + static_cast<long long>(x0) * 256; e4.res_lo = tok_.x[0].lo() + static_cast<long long>(x0) * 256; e4.res_ld = 256;
            e4.out_hi = tok_.x[0].hi + static_cast<long long>(x0) * 256; e4.out_lo = tok_.x[0].lo() + static_cast<long long>(x0) * 256; e4.out_ld = 256;
            if (li == 7) { e4.out_f32 = xf + static_cast<long long>(x0) * 256; e4.out_f32_ld = 256; }
            launch_enc256_fused(tok_.x[0], x0, xn, params.mat(p + ".qkv"), tok_.g, params.mat(p + ".mlp0"), params.mat(p + ".mlp2"), ep, st);
            return;
        }
        // (4) q of the attending rows with the normaliser folded in: Q*Z -> split planes (the msg buffer)
        {
            TmapPack maps;
            maps.b = make_tmap(params.mat(p + ".qkv"), bbox(256));
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], x0, xn);
            memset(&e, 0, sizeof(e));
            e.mode = LIN_QZ; e.ksum = tok_.ksum; e.seg_row0 = seg_row0;
            e.qz_scale[0] = qz_len[0]; e.qz_scale[1] = qz_len[1];
            c.M = xn; c.b_row0 = 0;
            e.M = xn; e.N = 256;
            e.out_hi = tok_.msg[0].hi + static_cast<long long>(x0) * 256; e.out_lo = tok_.msg[0].lo() + static_cast<long long>(x0) * 256; e.out_ld = 256;
            launch_gemm_counted<256, true, LinEpi>(maps, c, e, 256, st, "lin");
        }
        // (5) attention + merge + norm1 in one GEMM against the folded matrix of the row's segment
        {
            TmapPack maps;
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.msg[0], x0, xn);
            maps.b = make_tmap(tok_.g, bbox(256));
            GemmCore cg = c;
            cg.seg_mp0 = seg_row0 / (2 * kBM); cg.seg_b_rows = 256;
            memset(&e, 0, sizeof(e));
            e.M = xn; e.N = 256; e.mode = LIN_LN;
            e.gamma = params.vec(p + ".ln1.g"); e.beta = params.vec(p + ".ln1.b");
            e.out_hi = tok_.m1[0].hi + static_cast<long long>(x0) * 256; e.out_lo = tok_.m1[0].lo() + static_cast<long long>(x0) * 256; e.out_ld = 256;
            launch_gemm_counted<256, true, LinEpi>(maps, cg, e, 256, st, "lin");
        }
    }
    // q/k/v projections (+ elu+1 feature map on q,k)
    if (!fold) {
        TmapPack maps;
        maps.b = make_tmap(params.mat(p + ".qkv"), bbox(256));
        memset(&e, 0, sizeof(e));
        e.mode = LIN_F32_ELU;
        e.out_f32_ld = 768;
        if (self) {
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], x0, xn);
            c.M = xn; c.b_row0 = 0;
            e.M = xn; e.N = 768; e.elu_cols = 512; e.out_f32 = qkv + static_cast<long long>(x0) * 768; e.out_col0 = 0;
            if (lin_bn128()) { maps.b = make_tmap(params.mat(p + ".qkv"), bbox(128)); launch_gemm_counted<128, true, LinEpi>(maps, c, e, 768, st, "lin"); }
            else launch_gemm_counted<256, true, LinEpi>(maps, c, e, 768, st, "lin");
        } else {
            {   // q of the attending tokens
                for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], x0, xn);
                c.M = xn; c.b_row0 = 0;
                e.M = xn; e.N = 256; e.elu_cols = 256; e.out_f32 = qkv + static_cast<long long>(x0) * 768; e.out_col0 = 0;
                launch_gemm_counted<256, true, LinEpi>(maps, c, e, 256, st, "lin");
            }
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.x[0], s0, sn);
            c.M = sn;
            e.M = sn; e.out_f32 = qkv + static_cast<long long>(s0) * 768;
            c.b_row0 = 256; e.N = 512; e.elu_cols = 256; e.out_col0 = 256;
            if (lin_bn128()) { maps.b = make_tmap(params.mat(p + ".qkv"), bbox(128)); launch_gemm_counted<128, true, LinEpi>(maps, c, e, 512, st, "lin"); }
            else launch_gemm_counted<256, true, LinEpi>(maps, c, e, 512, st, "lin");
        }
    }
    if (!fold) {   // KV state(s): K = qkv[:,256:512] (already elu+1), V = qkv[:,512:768]
        const int chunks = (max_count + kv_tok() - 1) / kv_tok();
        { LaunchScope ls("kv", st);
          kv_partial_kernel<32><<<dim3(chunks, n_segs), 256, 0, st>>>(qkv + 256, qkv + 512, 768, tok_.seg_dev + kv_seg0, tok_.kv_chunks, tok_.kv_part,
                                                                      kv_tok()); }
        { LaunchScope ls("kv_final", st);
          kv_final_kernel<32><<<dim3((256 * 33 + 63) / 64, n_segs), kKvFinalThreads, 0, st>>>(tok_.kv_part, tok_.seg_dev + kv_seg0, tok_.kv_chunks,
                                                                                   tok_.kv_state, kv_tok()); }
        { LaunchScope ls("attn", st);
          attn_apply_kernel<32><<<dim3((max_count + kAttnTokCoarse - 1) / kAttnTokCoarse, n_segs), 256, attn_smem_bytes<32>(), st>>>(
              qkv, 768, tok_.seg_dev + apply_seg0, tok_.kv_state, tok_.msg[0].hi, tok_.msg[0].lo(), 256, kAttnTokCoarse); }
        DFSFM_CUDA(cudaGetLastError());
    }
    c.M = xn; c.b_row0 = 0;
    // merge + norm1
    if (!fold) {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.msg[0], x0, xn);
        maps.b = make_tmap(params.mat(p + ".merge"), bbox(256));
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 256; e.mode = LIN_LN;
        e.gamma = params.vec(p + ".ln1.g"); e.beta = params.vec(p + ".ln1.b");
        e.out_hi = tok_.m1[0].hi + static_cast<long long>(x0) * 256; e.out_lo = tok_.m1[0].lo() + static_cast<long long>(x0) * 256; e.out_ld = 256;
        launch_gemm_counted<256, true, LinEpi>(maps, c, e, 256, st, "lin");
    }
    // mlp.0 on cat[x, message] + relu
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(i == 1 ? tok_.m1[0] : tok_.x[0], x0, xn);
        maps.b = make_tmap(params.mat(p + ".mlp0"), bbox(256));
        GemmCore c2 = c;
        c2.num_taps = 2; c2.tap_map[0] = 0; c2.tap_map[1] = 1; c2.tap_shift[0] = c2.tap_shift[1] = 0;
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 512; e.mode = LIN_RELU_HL;
        e.out_hi = tok_.hid[0].hi + static_cast<long long>(x0) * 512; e.out_lo = tok_.hid[0].lo() + static_cast<long long>(x0) * 512; e.out_ld = 512;
        if (lin_bn128()) { maps.b = make_tmap(params.mat(p + ".mlp0"), bbox(128)); launch_gemm_counted<128, true, LinEpi>(maps, c2, e, 512, st, "lin"); }
        else launch_gemm_counted<256, true, LinEpi>(maps, c2, e, 512, st, "lin");
    }
    // mlp.2 + norm2 + residual
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(tok_.hid[0], x0, xn);
        maps.b = make_tmap(params.mat(p + ".mlp2"), bbox(256));
        GemmCore c3 = c;
        set_k(c3, 512);
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 256; e.mode = LIN_LN;
        e.gamma = params.vec(p + ".ln2.g"); e.beta = params.vec(p + ".ln2.b");
        if (res_hl()) {
            // the residual stream lives in the split planes (x = hi + lo carries 22 mantissa bits); the fp32 copy is only
            // written by the last layer, for the matcher and the fine stage
            e.res_hi = tok_.x[0].hi + static_cast<long long>(x0) * 256; e.res_lo = tok_.x[0].lo() + static_cast<long long>(x0) * 256; e.res_ld = 256;
            if (li == 7) { e.out_f32 = xf + static_cast<long long>(x0) * 256; e.out_f32_ld = 256; }
        } else {
            e.resid = xf + static_cast<long long>(x0) * 256; e.resid_ld = 256;
            e.out_f32 = xf + static_cast<long long>(x0) * 256; e.out_f32_ld = 256;
        }
        e.out_hi = tok_.x[0].hi + static_cast<long long>(x0) * 256; e.out_lo = tok_.x[0].lo() + static_cast<long long>(x0) * 256; e.out_ld = 256;
        launch_gemm_counted<256, true, LinEpi>(maps, c3, e, 256, st, "lin");
    }
}

static void split_rows(const float* in, long long rows, int C, __half* hi, __half* lo, cudaStream_t st) {
    const long long n4 = rows * C / 4;
    LaunchScope ls("split", st);
    split_rows_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, st>>>(in, n4, hi, lo);
    DFSFM_CUDA(cudaGetLastError());
}

void CoarseEngine::transformer(float* f0, int L, float* f1, int S, cudaStream_t st) {
    // joint token array: image 0 rows [0,L), image 1 rows [L1,L1+S).  With the folded schedule image 1 starts on a 256-row tile
    // boundary (rows [L,L1) are zero padding that no attention segment covers), so that every row tile of a launch over both
    // images belongs to ONE image and can pick that image's folded merge matrix.  Attention segments / KV-state slots:
    //   [0],[1]: self (own state 0 / 1);  [2]: image 0 reading state 1;  [3]: image 1 reading state 0
    const bool fold = attn_fold();
    const int L1 = fold ? ((L + 2 * kBM - 1) / (2 * kBM)) * (2 * kBM) : L;
    const int T = L1 + S;
    ensure_tok(T);
    tok_.L = L; tok_.L1 = L1; tok_.S = S;
    const Seg segs[4] = {{0, L, L, 0}, {L1, S, S, 1}, {0, L, L, 1}, {L1, S, S, 0}};
    DFSFM_CUDA(cudaMemcpyAsync(tok_.seg_dev, segs, sizeof(segs), cudaMemcpyHostToDevice, st));
    DFSFM_CUDA(cudaMemcpyAsync(tok_.xf, f0, static_cast<size_t>(L) * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (L1 > L) DFSFM_CUDA(cudaMemsetAsync(tok_.xf + static_cast<long long>(L) * 256, 0, static_cast<size_t>(L1 - L) * 256 * sizeof(float), st));
    DFSFM_CUDA(cudaMemcpyAsync(tok_.xf + static_cast<long long>(L1) * 256, f1, static_cast<size_t>(S) * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    split_rows(tok_.xf, T, 256, tok_.x[0].hi, tok_.x[0].lo(), st);
    const int mx = L > S ? L : S;
    for (int li = 0; li < 8; ++li) {
        if ((li % 2) == 0) {  // layer_names = ['self','cross'] * 4 (default.py:22): both images in one pass
            layer_call(li, true, 0, T, 0, T, 0, 2, 0, mx, st, fold ? L1 : 0);
        } else {
            layer_call(li, false, 0, L, L1, S, 1, 1, 2, mx, st);  // feat0 attends feat1
            layer_call(li, false, L1, S, 0, L, 0, 1, 3, mx, st);  // feat1 attends the UPDATED feat0 (transformer.py:96-97)
        }
    }
    DFSFM_CUDA(cudaMemcpyAsync(f0, tok_.xf, static_cast<size_t>(L) * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    DFSFM_CUDA(cudaMemcpyAsync(f1, tok_.xf + static_cast<long long>(L1) * 256, static_cast<size_t>(S) * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st));
}

// ------------------------------------------------------------------------------------------------ matching
void CoarseEngine::match(const float* f0, int h0c, int w0c, const float* f1, int h1c, int w1c, float thr, int border, float temperature,
                         int* i_ids, int* j_ids, float* mconf, int* n_matches, int capacity, float* conf_out, cudaStream_t st) {
    const int L = h0c * w0c, S = h1c * w1c;
    ensure_tok(L > S ? L : S);
    split_rows(f0, L, 256, tok_.x[0].hi, tok_.x[0].lo(), st);
    split_rows(f1, S, 256, tok_.x[1].hi, tok_.x[1].lo(), st);
    GemmCore c;
    memset(&c, 0, sizeof(c));
    set_k(c, 256);
    conv_taps_s1(c, 1, 0);
    SimEpiParams e;
    memset(&e, 0, sizeof(e));
    // sim = (f0 / sqrt(256)) . (f1 / sqrt(256)) / temperature (coarse_matching.py:103-107), carried in the log2 domain
    e.c2 = static_cast<float>(1.4426950408889634 / (256.0 * static_cast<double>(temperature)));
    const int n[2] = {L, S};
    // softmax statistics along both axes: rows of sim (dim=2) and rows of sim^T (dim=1)
    for (int side = 0; side < 2; ++side) {
        const int o = 1 - side;
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = make_tmap(tok_.x[side].hi, 256, n[side], tok_.x[side].plane_elems(), kBM);
        maps.b = make_tmap(tok_.x[o].hi, 256, n[o], tok_.x[o].plane_elems(), bbox(256));
        c.M = n[side];
        e.M = n[side]; e.N = n[o]; e.mode = SIM_STATS; e.part = tok_.part;
        launch_gemm_counted<256, true, SimEpi>(maps, c, e, n[o], st, "sim");
        const int tiles = ((n[o] + 255) / 256) * (engine_version() == 2 ? 2 : 1);
        { LaunchScope ls("stats_merge", st);
          stats_merge_kernel<<<(n[side] + 255) / 256, 256, 0, st>>>(tok_.part, tiles, n[side], tok_.stat[side]); }
    }
    DFSFM_CUDA(cudaMemsetAsync(tok_.best[0], 0, static_cast<size_t>(L) * 8, st));
    DFSFM_CUDA(cudaMemsetAsync(tok_.best[1], 0, static_cast<size_t>(S) * 8, st));
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = make_tmap(tok_.x[0].hi, 256, L, tok_.x[0].plane_elems(), kBM);
        maps.b = make_tmap(tok_.x[1].hi, 256, S, tok_.x[1].plane_elems(), bbox(256));
        c.M = L;
        e.M = L; e.N = S; e.mode = SIM_CONF;
        e.row_lse = tok_.stat[0]; e.col_lse = tok_.stat[1]; e.thr = thr;
        // conf = 2^(...) > thr: thr > 0 -> exponent > log2(thr); thr == 0 -> any non-zero (subnormal included) result, exponent >= -150
        e.lthr = thr > 0.f ? log2f(thr) - 0.01f : (thr == 0.f ? -152.f : -INFINITY);
        e.row_best = tok_.best[0]; e.col_best = tok_.best[1]; e.conf_out = conf_out;
        launch_gemm_counted<256, true, SimEpi>(maps, c, e, S, st, "sim");
    }
    { LaunchScope ls("select", st);
      match_select_kernel<<<1, 1024, 0, st>>>(tok_.best[0], tok_.best[1], L, w0c, w1c, border, capacity, i_ids, j_ids, mconf, n_matches); }
    DFSFM_CUDA(cudaGetLastError());
}


// ------------------------------------------------------------------------------------------------ fine stage
void CoarseEngine::ensure_fine(int M) {
    FineWs& f = fine_;
    if (M <= f.cap) return;
    hl_free(f.win); hl_free(f.x); hl_free(f.msg); hl_free(f.m1); hl_free(f.hid); hl_free(f.cin); hl_free(f.cwin);
    for (float* q : {f.xf, f.qkv, f.u, f.kvstate, f.kvpart, f.d_query}) if (q) cudaFree(q);
    if (f.segs) cudaFree(f.segs);
    if (f.tracks) cudaFree(f.tracks);
    if (f.views) cudaFree(f.views);
    const int cap = ((M + 1023) / 1024) * 1024;
    f.cap = cap;
    const long long R = 2ll * cap * 25;
    f.win = hl_alloc(R, 128); f.x = hl_alloc(R, 128); f.msg = hl_alloc(R, 128); f.m1 = hl_alloc(R, 128); f.hid = hl_alloc(R, 256);
    f.cin = hl_alloc(2ll * cap, 256); f.cwin = hl_alloc(2ll * cap, 128);
    DFSFM_CUDA(cudaMalloc(&f.xf, static_cast<size_t>(R) * 128 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.qkv, static_cast<size_t>(R) * 384 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.u, static_cast<size_t>(2) * cap * 128 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.kvstate, static_cast<size_t>(2) * cap * 2176 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.kvpart, static_cast<size_t>(2) * cap * 2176 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.d_query, static_cast<size_t>(cap) * 2 * sizeof(float)));
    DFSFM_CUDA(cudaMalloc(&f.segs, static_cast<size_t>(4) * cap * sizeof(Seg)));
    DFSFM_CUDA(cudaMalloc(&f.tracks, static_cast<size_t>(cap) * sizeof(TrackRec)));
    DFSFM_CUDA(cudaMalloc(&f.views, static_cast<size_t>(cap) * sizeof(ViewRec)));
}

// One LoFTREncoderLayer of loftr_fine (d_model 128, 8 heads) on token rows [x0, x0+xn) of the window-token array; source rows
// [s0, s0+sn) when not self.  Same structure as layer_call, 128-wide.
void CoarseEngine::layer128(int li, bool self, int x0, int xn, int s0, int sn, const Seg* kv_segs, int n_kv, const Seg* apply_segs, int n_apply,
                            cudaStream_t st) {
    FineWs& f = fine_;
    const std::string p = "fine.tr." + std::to_string(li);
    GemmCore c;
    memset(&c, 0, sizeof(c));
    set_k(c, 128);
    conv_taps_s1(c, 1, 0);
    LinEpiParams e;
    auto rows_map = [&](const HL& b, int r0, int n) { return make_tmap(b.hi + static_cast<long long>(r0) * b.C, b.C, n, b.plane_elems(), kBM); };
    {
        TmapPack maps;
        maps.b = make_tmap(params.mat(p + ".qkv"), bbox(128));
        memset(&e, 0, sizeof(e));
        e.mode = LIN_F32_ELU;
        e.out_f32_ld = 384;
        if (self) {
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.x, x0, xn);
            c.M = xn; c.b_row0 = 0;
            e.M = xn; e.N = 384; e.elu_cols = 256; e.out_f32 = f.qkv + static_cast<long long>(x0) * 384; e.out_col0 = 0;
            launch_gemm_counted<128, true, LinEpi>(maps, c, e, 384, st, "fine_lin");
        } else {
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.x, x0, xn);
            c.M = xn; c.b_row0 = 0;
            e.M = xn; e.N = 128; e.elu_cols = 128; e.out_f32 = f.qkv + static_cast<long long>(x0) * 384; e.out_col0 = 0;
            launch_gemm_counted<128, true, LinEpi>(maps, c, e, 128, st, "fine_lin");
            for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.x, s0, sn);
            c.M = sn; c.b_row0 = 128;
            e.M = sn; e.N = 256; e.elu_cols = 128; e.out_f32 = f.qkv + static_cast<long long>(s0) * 384; e.out_col0 = 128;
            launch_gemm_counted<128, true, LinEpi>(maps, c, e, 256, st, "fine_lin");
        }
    }
    { LaunchScope ls("fine_kv", st);
      kv_partial_kernel<16><<<dim3(1, n_kv), 128, 0, st>>>(f.qkv + 128, f.qkv + 256, 384, kv_segs, 1, f.kvpart, 32); }
    { LaunchScope ls("fine_kv", st);
      kv_final_kernel<16><<<dim3((8 * 16 * 17 + 63) / 64, n_kv), kKvFinalThreads, 0, st>>>(f.kvpart, kv_segs, 1, f.kvstate, 32); }
    { LaunchScope ls("fine_attn", st);
      attn_apply_kernel<16><<<dim3(1, n_apply), 256, attn_smem_bytes<16>(), st>>>(f.qkv, 384, apply_segs, f.kvstate, f.msg.hi, f.msg.lo(), 128, 32); }
    DFSFM_CUDA(cudaGetLastError());
    c.M = xn; c.b_row0 = 0;
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.msg, x0, xn);
        maps.b = make_tmap(params.mat(p + ".merge"), bbox(128));
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 128; e.mode = LIN_LN; e.gamma = params.vec(p + ".ln1.g"); e.beta = params.vec(p + ".ln1.b");
        e.out_hi = f.m1.hi + static_cast<long long>(x0) * 128; e.out_lo = f.m1.lo() + static_cast<long long>(x0) * 128; e.out_ld = 128;
        launch_gemm_counted<128, true, LinEpi>(maps, c, e, 128, st, "fine_lin");
    }
    if (fused_mlp_enabled()) {
        launch_mlp128_fused(f.x, f.m1, x0, xn, params.mat(p + ".mlp0"), params.mat(p + ".mlp2"), params.vec(p + ".ln2.g"), params.vec(p + ".ln2.b"),
                            f.xf, st);
        return;
    }
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(i == 1 ? f.m1 : f.x, x0, xn);
        maps.b = make_tmap(params.mat(p + ".mlp0"), bbox(256));
        GemmCore c2 = c;
        c2.num_taps = 2; c2.tap_map[0] = 0; c2.tap_map[1] = 1; c2.tap_shift[0] = c2.tap_shift[1] = 0;
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 256; e.mode = LIN_RELU_HL;
        e.out_hi = f.hid.hi + static_cast<long long>(x0) * 256; e.out_lo = f.hid.lo() + static_cast<long long>(x0) * 256; e.out_ld = 256;
        launch_gemm_counted<256, true, LinEpi>(maps, c2, e, 256, st, "fine_lin");
    }
    {
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.hid, x0, xn);
        maps.b = make_tmap(params.mat(p + ".mlp2"), bbox(128));
        GemmCore c3 = c;
        set_k(c3, 256);
        memset(&e, 0, sizeof(e));
        e.M = xn; e.N = 128; e.mode = LIN_LN; e.gamma = params.vec(p + ".ln2.g"); e.beta = params.vec(p + ".ln2.b");
        e.resid = f.xf + static_cast<long long>(x0) * 128; e.resid_ld = 128;
        e.out_f32 = f.xf + static_cast<long long>(x0) * 128; e.out_f32_ld = 128;
        e.out_hi = f.x.hi + static_cast<long long>(x0) * 128; e.out_lo = f.x.lo() + static_cast<long long>(x0) * 128; e.out_ld = 128;
        launch_gemm_counted<128, true, LinEpi>(maps, c3, e, 128, st, "fine_lin");
    }
}

// FinePreprocess.forward + loftr_fine + FineMatching.forward (fine_preprocess.py:29-59, transformer.py:80-101,
// utils/fine_matching.py:15-61) for M coarse matches.  coords_out [M][2] = coords_normed * (W // 2); std_out [M].
void CoarseEngine::fine_match(const float* ff0, int Hf0, int Wf0, const float* ff1, int Hf1, int Wf1, const float* fc0, int w0c, const float* fc1,
                              int w1c, const int* i_ids, const int* j_ids, int M, float* coords_out, float* std_out, cudaStream_t st) {
    if (M <= 0) return;
    ensure_fine(M);
    FineWs& f = fine_;
    const int stride = Wf0 / w0c;  // hw0_f // hw0_c (fine_preprocess.py:31)
    const int MW = M * 25, R = 2 * MW;
    // host tables: attention segments (window = 25 tokens) and the per-match records of the matching kernel
    std::vector<Seg> segs(static_cast<size_t>(4) * M);
    std::vector<TrackRec> tracks(M);
    std::vector<ViewRec> views(M);
    for (int w = 0; w < 2 * M; ++w) segs[w] = Seg{w * 25, 25, 25, w};
    for (int m = 0; m < M; ++m) {
        segs[static_cast<size_t>(2) * M + m] = Seg{m * 25, 25, 25, M + m};        // feat0 windows read the feat1 states
        segs[static_cast<size_t>(3) * M + m] = Seg{(M + m) * 25, 25, 25, m};      // feat1 windows read the (updated) feat0 states
        TrackRec& t = tracks[m];
        t.tok0 = m * 25; t.qtok0 = (M + m) * 25; t.n_views = 1; t.movable = 0; t.qx = t.qy = 0.f; t.sqx = t.sqy = 1.f;
        views[m] = ViewRec{0.f, 0.f, 1.f, 1.f};
    }
    DFSFM_CUDA(cudaMemcpyAsync(f.segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, st));
    DFSFM_CUDA(cudaMemcpyAsync(f.tracks, tracks.data(), tracks.size() * sizeof(TrackRec), cudaMemcpyHostToDevice, st));
    DFSFM_CUDA(cudaMemcpyAsync(f.views, views.data(), views.size() * sizeof(ViewRec), cudaMemcpyHostToDevice, st));
    { LaunchScope ls("fine_gather", st);
      gather_windows_kernel<<<2 * M, 128, 0, st>>>(ff0, Hf0, Wf0, w0c, ff1, Hf1, Wf1, w1c, stride, i_ids, j_ids, M, f.win.hi, f.win.lo()); }
    { LaunchScope ls("fine_gather", st);
      gather_coarse_kernel<<<2 * M, 256, 0, st>>>(fc0, fc1, i_ids, j_ids, M, f.cin.hi, f.cin.lo()); }
    DFSFM_CUDA(cudaGetLastError());
    GemmCore c;
    memset(&c, 0, sizeof(c));
    conv_taps_s1(c, 1, 0);
    auto rows_map = [&](const HL& b, int n) { return make_tmap(b.hi, b.C, n, b.plane_elems(), kBM); };
    {   // c_win = down_proj(cat[feat_c0[i], feat_c1[j]])                      (fine_preprocess.py:50-51)
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.cin, 2 * M);
        maps.b = make_tmap(params.mat("fine.down.w"), bbox(128));
        set_k(c, 256);
        c.M = 2 * M;
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.M = 2 * M; e.N = 128; e.bias = params.vec("fine.down.b"); e.out_mode = OUT_FLAT;
        e.out_hi = f.cwin.hi; e.out_lo = f.cwin.lo(); e.out_ld = 128;
        launch_gemm_counted<128, true, ConvEpi>(maps, c, e, 128, st, "fine_lin");
    }
    {   // u = merge_feat.weight[:, 128:] . c_win + merge_feat.bias   (the coarse half of the concat, constant over a window)
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.cwin, 2 * M);
        maps.b = make_tmap(params.mat("fine.merge_c.w"), bbox(128));
        set_k(c, 128);
        c.M = 2 * M;
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.M = 2 * M; e.N = 128; e.bias = params.vec("fine.merge.b"); e.out_mode = OUT_FLAT; e.out_f32 = f.u; e.out_f32_ld = 128;
        launch_gemm_counted<128, true, ConvEpi>(maps, c, e, 128, st, "fine_lin");
    }
    {   // tokens = merge_feat.weight[:, :128] . window + u[window]          (fine_preprocess.py:52-56)
        TmapPack maps;
        for (int i = 0; i < kMaxAMaps; ++i) maps.a[i] = rows_map(f.win, R);
        maps.b = make_tmap(params.mat("fine.merge_f.w"), bbox(128));
        set_k(c, 128);
        c.M = R;
        ConvEpiParams e;
        memset(&e, 0, sizeof(e));
        e.M = R; e.N = 128; e.g = FlatGeom{25, 1, 25, 1};  // "image" = window, 25 rows: n_img indexes u
        e.addend = f.u; e.addend_mode = 1; e.out_mode = OUT_FLAT;
        e.out_f32 = f.xf; e.out_f32_ld = 128; e.out_hi = f.x.hi; e.out_lo = f.x.lo(); e.out_ld = 128;
        launch_gemm_counted<128, true, ConvEpi>(maps, c, e, 128, st, "fine_lin");
    }
    // loftr_fine: ['self', 'cross'] (default.py:44), cross = feat0 first, then feat1 against the updated feat0
    layer128(0, true, 0, R, 0, R, f.segs, 2 * M, f.segs, 2 * M, st);
    layer128(1, false, 0, MW, MW, MW, f.segs + M, M, f.segs + 2 * M, M, st);
    layer128(1, false, MW, MW, 0, MW, f.segs, M, f.segs + 3 * M, M, st);
    {   // FineMatching: centre token of window 0 against the 25 tokens of window 1, soft-argmax + std
        const size_t smem = fine_match_smem_bytes(5, 1);
        DFSFM_CUDA(cudaMemsetAsync(coords_out, 0, static_cast<size_t>(M) * 2 * sizeof(float), st));
        LaunchScope ls("fine_match", st);
        fine_match_kernel<<<M, kFmThreads, smem, st>>>(f.xf, f.tracks, f.views, 1, 5, 1, f.d_query, coords_out, std_out, M);
        DFSFM_CUDA(cudaGetLastError());
    }
}

}  // namespace dfsfm

// ================================================================================================ C ABI
using dfsfm::CoarseEngine;
struct dfsfm_coarse { std::unique_ptr<CoarseEngine> e; };

extern "C" {

int dfsfm_coarse_create(dfsfm_coarse_t** out, int device) {
    return dfsfm::guard([&] {
        auto* h = new dfsfm_coarse;
        h->e.reset(new CoarseEngine(device));
        *out = h;
    });
}
void dfsfm_coarse_destroy(dfsfm_coarse_t* h) { delete h; }

int dfsfm_coarse_set_param(dfsfm_coarse_t* h, const char* name, const float* host, int64_t rows, int64_t cols, int kind) {
    return dfsfm::guard([&] { h->e->params.set(name, host, rows, cols, kind); });
}
int dfsfm_coarse_features(dfsfm_coarse_t* h, const float* image_dev, int H, int W, const float* pe_dev, float* tokens_out_dev, void* stream) {
    return dfsfm::guard([&] { h->e->features(&image_dev, 1, H, W, pe_dev, &tokens_out_dev, nullptr, static_cast<cudaStream_t>(stream)); });
}
int dfsfm_coarse_features_pair(dfsfm_coarse_t* h, const float* image0_dev, const float* image1_dev, int H, int W, const float* pe_dev,
                               float* tokens0_out_dev, float* tokens1_out_dev, void* stream) {
    return dfsfm::guard([&] {
        const float* imgs[2] = {image0_dev, image1_dev};
        float* tokens[2] = {tokens0_out_dev, tokens1_out_dev};
        h->e->features(imgs, 2, H, W, pe_dev, tokens, nullptr, static_cast<cudaStream_t>(stream));
    });
}
int dfsfm_coarse_features_fine(dfsfm_coarse_t* h, const float* image_dev, int H, int W, const float* pe_dev, float* tokens_out_dev,
                               float* feat_f_out_dev, void* stream) {
    return dfsfm::guard([&] { h->e->features(&image_dev, 1, H, W, pe_dev, &tokens_out_dev, feat_f_out_dev, static_cast<cudaStream_t>(stream)); });
}
int dfsfm_coarse_fine_match(dfsfm_coarse_t* h, const float* feat_f0_dev, int Hf0, int Wf0, const float* feat_f1_dev, int Hf1, int Wf1,
                            const float* feat_c0_dev, int w0c, const float* feat_c1_dev, int w1c, const int32_t* i_ids_dev,
                            const int32_t* j_ids_dev, int M, float* coords_out_dev, float* std_out_dev, void* stream) {
    return dfsfm::guard([&] {
        h->e->fine_match(feat_f0_dev, Hf0, Wf0, feat_f1_dev, Hf1, Wf1, feat_c0_dev, w0c, feat_c1_dev, w1c, i_ids_dev, j_ids_dev, M, coords_out_dev,
                         std_out_dev, static_cast<cudaStream_t>(stream));
    });
}
int dfsfm_coarse_transformer(dfsfm_coarse_t* h, float* feat0_dev, int L, float* feat1_dev, int S, void* stream) {
    return dfsfm::guard([&] { h->e->transformer(feat0_dev, L, feat1_dev, S, static_cast<cudaStream_t>(stream)); });
}
int dfsfm_coarse_match(dfsfm_coarse_t* h, const float* feat0_dev, int h0c, int w0c, const float* feat1_dev, int h1c, int w1c, float thr,
                       int border_rm, float temperature, int32_t* i_ids_dev, int32_t* j_ids_dev, float* mconf_dev, int32_t* n_matches_dev,
                       int capacity, float* conf_out_dev, void* stream) {
    return dfsfm::guard([&] {
        h->e->match(feat0_dev, h0c, w0c, feat1_dev, h1c, w1c, thr, border_rm, temperature, i_ids_dev, j_ids_dev, mconf_dev, n_matches_dev,
                    capacity, conf_out_dev, static_cast<cudaStream_t>(stream));
    });
}

}  // extern "C"
