// MSG-CHN ProxyTTA engine: the whole per-frame adaptation step (src/tta_main.py:583-633 of the
// reference) as a fixed sequence of sm_100a kernels over an engine-owned activation arena.
//
// Graph restated from external_src/MSG_CHN/workspace/exp_msg_chn/network_exp_msg_chn_adapt.py
// (RGBEncoder :214-264, DepthEncoder :166-211, DepthDecoder :267-311, Res_Conv :28-36,
// _rgbd_meta_contrast :463-557, heads :1022-1098).  The backward pass is hand-derived and only
// visits what the adapted ("meta") tensors need (SURVEY.md section 8 a16): the proxy head on the real
// rows, decoder3/encoder3/decoder2/encoder2, decoder1's prediction layers and the meta layer.
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>
#include <atomic>

#include "common.cuh"
#include "conv_mma.cuh"
#include "gemm_mma.cuh"
#include "small_kernels.cuh"
#include "conv_tc.cuh"
#include "conv_tc_s2.cuh"
#include "conv_tc_t2.cuh"
#include "stem_tc.cuh"
#include "gemm_tc.cuh"
#include "gemm_tn_tc.cuh"
#include "nlspn_prop.cuh"
#include "augment.cuh"
#include "../../include/ptta_b200.h"

namespace ptta {

static thread_local std::string g_error;
static std::atomic<long long> g_launches(0);

bool pdl_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("PTTA_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
    return v != 0;
}

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
}

// timing experiments: when a trace is active every launch is followed by an event on the stream it went to
struct LaunchTrace { std::vector<std::string> names; std::vector<int> streams; std::vector<cudaEvent_t> events; cudaStream_t* cur; cudaStream_t main; };
static LaunchTrace* g_trace = nullptr;

int check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_trace) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        cudaEventRecord(ev, *g_trace->cur);
        g_trace->names.push_back(what); g_trace->streams.push_back(*g_trace->cur == g_trace->main ? 0 : 1); g_trace->events.push_back(ev);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("kernel launch %s failed: %s", what, cudaGetErrorString(e));
        return 3;
    }
    return 0;
}

// -------------------------------------------------------------------------------------------------
struct Map32 { bf16* p = nullptr; int n = 0, h = 0, w = 0, c = 32; size_t numel() const { return (size_t)n * h * w * c; } };
struct Map1 { float* p = nullptr; int n = 0, h = 0, w = 0; size_t numel() const { return (size_t)n * h * w; } };
struct TensorInfo { void* p; int dtype; long long d[4]; };

struct Arena {
    char* base = nullptr;
    size_t off = 0;
    void* take(size_t bytes) {
        size_t o = (off + 255) & ~(size_t)255;
        off = o + bytes;
        return base ? base + o : nullptr;
    }
};

struct ConvLayer {
    std::string name;
    int cin = 32, cout = 32;
    bool transposed = false, has_bias = true;
    const float* w = nullptr; const float* b = nullptr;
    bf16* pack_fwd = nullptr; bf16* pack_dgrad = nullptr;
    bf16* img_fwd = nullptr; bf16* img_dgrad = nullptr;     // tcgen05 weight images (32->32 stride-1 roles only)
    int mode_fwd = MODE_S1, mode_dgrad = MODE_S1;
};
struct StemLayer {   // init.0: {1,2,3} -> 32
    std::string name; int cin = 1;
    const float* w = nullptr; const float* b = nullptr;
    float* dgrad_ch1 = nullptr;   // [9][32] flipped weights of input plane 1 (cascade encoders)
    std::vector<float> raw_host;  // host copy of w taken at pack time ...
    float wk[3 * 9 * 32];         // ... re-ordered [ci][tap][co]: passed by value to stem_convc_kernel (constant-bank operands)
    float bk[32];
    float dk[9 * 32];             // host copy of dgrad_ch1 ([9][32]) for head_convc_kernel
    bf16* img_dgrad1 = nullptr;   // tcgen05 weight image of dgrad_ch1 (conv3x3_tc_head_kernel)
    bf16* img_tc = nullptr;       // tcgen05 weight image of w (stem_tc_kernel: B_hi | B_lo)
};
struct HeadLayer {   // prdct.3: 32 -> 1
    std::string name;
    const float* w = nullptr; const float* b = nullptr;
    float* w_fwd = nullptr;       // [9][32]
    float* w_dgrad = nullptr;     // [32][1][3][3] flipped, stem-shaped
    float bias_host = 0.f;
    std::vector<float> raw_host;  // host copy of w_dgrad ([32][1][3][3], flipped) ...
    float wdk[9 * 32];            // ... re-ordered [tap][co] for stem_convc_kernel<1>
    float wfk[9 * 32];            // host copy of w_fwd ([9][32]) for head_convc_kernel
    bf16* img_fwd = nullptr;      // tcgen05 weight image of w_fwd (conv3x3_tc_head_kernel)
    bf16* img_dgrad_tc = nullptr; // tcgen05 weight image of w_dgrad (stem_tc_kernel<1>)
};
struct BnState {     // per call-site statistics
    float *mean = nullptr, *invstd = nullptr, *scale = nullptr, *shift = nullptr, *uvar = nullptr;
};
struct BnLayer {
    std::string name; int c = 0;
    float *gamma = nullptr, *beta = nullptr, *rm = nullptr, *rv = nullptr; long long* nbt = nullptr;
};
struct LinearLayer {
    std::string name; int in = 0, out = 0;
    const float* w = nullptr; const float* b = nullptr;
    bf16* pack = nullptr;     // [out][in]
    bf16* pack_t = nullptr;   // [in][out]  (data gradient)
};

struct EncW { StemLayer init0; ConvLayer init2, e1a, e1b, e2a, e2b, e3a, e3b, e4a, e4b; int nenc = 2; };
struct DecW { ConvLayer d2a, d2b, d1a, d1b, p1; HeadLayer p3; };

struct EncAct { Map32 a0, x0, t1, x1, t2, x2; Map32 x0r, x1r; };    // x0r / x1r = ReLU(x0) / ReLU(x1): inputs of the stride-2 convs
struct DecAct { Map32 x2, x1, x0, u2, x3, s1, u1, x4, s0, h; Map32 x2r; Map1 out; };   // x2r = ReLU(x2): input of the transposed conv dec2.1
struct Branch {
    Map32 c[5];            // rgb features (c[2] after the meta layer)
    Map32 cr[4];           // ReLU of the rgb encoder's own x0..x3 (inputs of its stride-2 convs)
    Map32 c2raw;           // rgb x2 before the meta layer
    Map32 mh, mg;          // meta: conv1 output (128 ch), conv2 output (32 ch), both pre-BN
    BnState bn1, bn2;
    EncAct e1, e2, e3;
    DecAct d1, d2, d3;
    Map1 p12, p11;
    Map1 output;
};

}  // namespace ptta

using namespace ptta;

struct ptta_msgchn {
    int N, H, W;                    // shape the network runs at (multiples of 16; 2 x the user batch when `padded`)
    int Nu, Hu, Wu;                 // shape of the caller's tensors
    bool padded = false;            // pad + flip-pad ensembling active (src/msg_chn_model_adapt.py:58-125)
    float *pimg = nullptr, *psp = nullptr;   // padded image [N,3,H,W] / sparse depth [N,1,H,W]
    Map1 out_u, g_out_u;            // un-padded mean prediction and its gradient
    bool two_layers, has_heads;
    std::string prepare_mode;
    cudaStream_t st = nullptr;      // stream of the call in flight (helpers launch on `st`)
    cudaStream_t st2 = nullptr;     // side stream: the zero-image branch runs concurrently with the real branch
    cudaStream_t st3 = nullptr;     // second side stream: proxy head of the real rows (forward + backward) and the meta layer's second
                                    // weight gradient run beside decoder 3 / the data-gradient chain
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_projbn = nullptr, ev_enc1 = nullptr, ev_zmeta = nullptr;
    cudaEvent_t ev_e3 = nullptr, ev_mlp = nullptr, ev_lossg = nullptr, ev_headb = nullptr, ev_gmg = nullptr, ev_wg2 = nullptr;
    bool two_streams = true;
    bool mlp_on_st3 = false;        // set by forward_impl for the duration of the real cascade
    bool tc_enabled = true; long long tc_min_pixels = 6000, tc_s2_min_pixels = 6000, tc_t2_min_pixels = 1500, tc_head_min_pixels = 20000, tc_stem_min_pixels = 20000;
    Arena arena;
    size_t ws_bytes = 0;
    bool bound = false, packed = false;
    std::map<std::string, std::pair<void*, long long>> ext;   // façade-owned tensors by key
    std::vector<std::string> keys;                            // required keys
    std::map<std::string, TensorInfo> named;
    std::vector<std::string> named_order;

    // weights
    EncW rgbW, enc1W, enc2W, enc3W;
    DecW dec1W, dec2W, dec3W;
    ConvLayer meta1, meta2;          // 2layers: 32->128 (no bias), 128->32 ; 1layer: meta1 = 32->32
    BnLayer metaBn1, metaBn2;
    LinearLayer proj0, proj3, pred0, pred3;
    bf16* projpred_pack = nullptr; float* projpred_bias = nullptr;   // pred.0 o proj.3 as one Linear layer (zero-image rows: emb = pred(proj(z)))
    bool fuse_projpred = true;
    // shared-model mode (ptta_msgchn_set_comm): SyncBatchNorm sums and the gradient all-reduce go through peer memory (peer_comm.cuh)
    PeerComm comm;
    int next_xid = 0;                // exchange slots are handed out in call order; every rank runs the same sequence
    BnLayer projBn, predBn;
    std::vector<std::string> adapt_names;
    // source-domain preparation (SURVEY section 8 f3): stage 1 = supervised fit of the meta layer (src/init_main.py:448-572, no proxy branch),
    // stage 2 = fit of the predictor head `pred` on the frozen network (src/head_main.py:415-541)
    bool train_head = false;         // option "trainable_head": the trained tensors are pred.{0,1,3}.{weight,bias}, not the meta layer
    bool skip_dec3 = false;          // stage 2 never looks at the prediction: decoder 3 of the real branch is not run
    bool proxy_in_backward = true;   // false after a stage-1 forward: no gradient arrives through the proxy head
    float* gw_part = nullptr;        // split-K partial tiles of the Linear weight gradients (gemm_tn_tc.cuh)
    bf16 *g_q0 = nullptr;            // stage 2: gradient wrt pred.0's output
    const float* l_gt = nullptr; float l_maxd = 0.f;

    // activations
    Branch real, zero;
    Map32 rgbT[5];                   // rgb encoder temporaries (a0 / t_k), per resolution
    Map32 zc[5];                     // cached rgb_encoder(0) features
    Map32 zcr[4];                    // scratch ReLU copies while rgb_encoder(0) is (re)computed
    Map1 fd, fv, dcl, d12, d14;      // filtered depth / validity, clamped depth, pyramid
    float *stage_img = nullptr, *stage_sp = nullptr;   // engine-owned copies of the caller's frame: what a captured step reads
    // heads
    long long R = 0;
    bf16 *h_an2 = nullptr; double* partial2 = nullptr;
    bf16 *h_a0z = nullptr, *h_a0r = nullptr, *h_an = nullptr, *h_pz = nullptr, *h_q0 = nullptr, *emb = nullptr, *ref = nullptr;
    bf16 *g_ref = nullptr, *g_a3 = nullptr, *g_a0 = nullptr;
    BnState bnProjZ, bnProjR, bnPred;
    float* rowstat = nullptr;
    // backward scratch
    Map32 T1a, T1b, T2a, T2b, D2, G4a, G4b, D4, GC2, GZ, D8, E8, M128a, M128b;
    Map1 g_out, g_p11, g_q, g_p12, g_o14;
    float *k0 = nullptr, *k1 = nullptr, *k2 = nullptr;
    double* partial = nullptr; size_t partial_doubles = 0;
    float* wgrad_ws = nullptr; float* wgrad_ws2 = nullptr;
    double* partial3 = nullptr;
    LossScalars* losses = nullptr;
    double *loss_map_partial = nullptr, *loss_cos_partial = nullptr;
    int loss_map_blocks = 0, loss_cos_blocks = 0;
    AdamHyper* adam_hyper = nullptr;
    AdamChunk* adam_chunks = nullptr; int n_adam_chunks = 0;
    const float* adam_g_base = nullptr; size_t adam_g_floats = 0;   // extent of the gradient pointers in the chunk table
    float* zero_bias = nullptr;
    // loss inputs remembered for backward
    const float *l_img = nullptr, *l_d = nullptr, *l_v = nullptr; float l_cap = 0, l_wsd = 0, l_wsm = 0;
    // graph
    cudaGraphExec_t graph_exec = nullptr;
    struct GraphKey { float isc[3], ish[3], cap, w_sd, w_sm, w_cos; } graph_key;   // everything a capture bakes in (inputs are staged)
    cudaGraphExec_t prep_graph_exec = nullptr;      // captured stage-1 / stage-2 step (an engine runs one of the two)
    GraphKey prep_graph_key;
    float* stage_gt = nullptr;                      // engine-owned copy of the ground truth the captured stage-1 step reads
    void drop_graphs() {
        if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
        if (prep_graph_exec) { cudaGraphExecDestroy(prep_graph_exec); prep_graph_exec = nullptr; }
    }

    // ---------------------------------------------------------------------------------------------
    Map32 alloc32(const char* name, int h, int w, int c = 32) {
        Map32 m; m.n = N; m.h = h; m.w = w; m.c = c;
        m.p = (bf16*)arena.take(m.numel() * sizeof(bf16));
        if (name) reg(name, m.p, 1, N, h, w, c);
        return m;
    }
    Map1 alloc1(const char* name, int h, int w) {
        Map1 m; m.n = N; m.h = h; m.w = w;
        m.p = (float*)arena.take(m.numel() * sizeof(float));
        if (name) reg(name, m.p, 0, N, h, w, 1);
        return m;
    }
    template <typename T> T* allocv(size_t count) { return (T*)arena.take(count * sizeof(T)); }
    void reg(const std::string& name, void* p, int dtype, long long a, long long b, long long c, long long d) {
        if (!named.count(name)) named_order.push_back(name);
        TensorInfo t; t.p = p; t.dtype = dtype; t.d[0] = a; t.d[1] = b; t.d[2] = c; t.d[3] = d;
        named[name] = t;
    }
    BnState alloc_bn(int c) {
        BnState s; s.mean = allocv<float>(c); s.invstd = allocv<float>(c); s.scale = allocv<float>(c); s.shift = allocv<float>(c);
        s.uvar = allocv<float>(c);
        return s;
    }
    void need(const std::string& k) { keys.push_back(k); }

    void def_conv(ConvLayer& L, const std::string& name, int cin, int cout, bool transposed, bool bias) {
        L.name = name; L.cin = cin; L.cout = cout; L.transposed = transposed; L.has_bias = bias;
        need(name + ".weight");
        if (bias) need(name + ".bias");
    }
    void def_enc(EncW& E, const std::string& prefix, int cin, int nenc) {
        E.nenc = nenc;
        E.init0.name = prefix + ".init.0"; E.init0.cin = cin;
        need(E.init0.name + ".weight"); need(E.init0.name + ".bias");
        def_conv(E.init2, prefix + ".init.2", 32, 32, false, true);
        ConvLayer* ls[8] = {&E.e1a, &E.e1b, &E.e2a, &E.e2b, &E.e3a, &E.e3b, &E.e4a, &E.e4b};
        for (int k = 0; k < nenc; ++k) {
            def_conv(*ls[2 * k], prefix + ".enc" + std::to_string(k + 1) + ".1", 32, 32, false, true);
            ls[2 * k]->mode_fwd = MODE_S2; ls[2 * k]->mode_dgrad = MODE_T2;
            def_conv(*ls[2 * k + 1], prefix + ".enc" + std::to_string(k + 1) + ".3", 32, 32, false, true);
        }
    }
    void def_dec(DecW& D, const std::string& prefix) {
        def_conv(D.d2a, prefix + ".dec2.1", 32, 32, true, true); D.d2a.mode_fwd = MODE_T2; D.d2a.mode_dgrad = MODE_S2;
        def_conv(D.d2b, prefix + ".dec2.3", 32, 32, false, true);
        def_conv(D.d1a, prefix + ".dec1.1", 32, 32, true, true); D.d1a.mode_fwd = MODE_T2; D.d1a.mode_dgrad = MODE_S2;
        def_conv(D.d1b, prefix + ".dec1.3", 32, 32, false, true);
        def_conv(D.p1, prefix + ".prdct.1", 32, 32, false, true);
        D.p3.name = prefix + ".prdct.3";
        need(D.p3.name + ".weight"); need(D.p3.name + ".bias");
    }
    void def_bn(BnLayer& B, const std::string& name, int c) {
        B.name = name; B.c = c;
        need(name + ".weight"); need(name + ".bias"); need(name + ".running_mean"); need(name + ".running_var");
        need(name + ".num_batches_tracked");
    }
    void def_linear(LinearLayer& L, const std::string& name, int in, int out) {
        L.name = name; L.in = in; L.out = out;
        need(name + ".weight"); need(name + ".bias");
    }

    int define_model() {
        def_enc(rgbW, "rgb_encoder", 3, 4);
        def_enc(enc1W, "depth_encoder1", 1, 2); def_dec(dec1W, "depth_decoder1");
        def_enc(enc2W, "depth_encoder2", 2, 2); def_dec(dec2W, "depth_decoder2");
        def_enc(enc3W, "depth_encoder3", 2, 2); def_dec(dec3W, "depth_decoder3");
        if (two_layers) {
            const std::string p = "conv1_rgb_meta.conv1_meta";
            def_conv(meta1, p + ".0.0", 32, 128, false, false);
            def_bn(metaBn1, p + ".0.1", 128);
            def_conv(meta2, p + ".1", 128, 32, false, true);
            def_bn(metaBn2, p + ".2", 32);
            adapt_names = {p + ".0.0.weight", p + ".0.1.weight", p + ".0.1.bias", p + ".1.weight", p + ".1.bias",
                           p + ".2.weight", p + ".2.bias"};
        } else {
            def_conv(meta1, "conv1_rgb_meta", 32, 32, false, true);
            adapt_names = {"conv1_rgb_meta.weight", "conv1_rgb_meta.bias"};
        }
        if (has_heads) {
            def_linear(proj0, "proj.0", 32, 512); def_bn(projBn, "proj.1", 512); def_linear(proj3, "proj.3", 512, 512);
            def_linear(pred0, "pred.0", 512, 512); def_bn(predBn, "pred.1", 512); def_linear(pred3, "pred.3", 512, 512);
            if (prepare_mode.find("ema") != std::string::npos)      // EMA copy of proj (network_exp_msg_chn_adapt.py:1052-1060): stage 2 updates it
                for (const char* t : {"0.weight", "0.bias", "1.weight", "1.bias", "3.weight", "3.bias"}) need(std::string("proj_t.") + t);
        }
        return 0;
    }

    // stage 2 of the source-domain preparation: the trained tensors are the predictor head's
    int select_trainable_head() {
        PTTA_CHECK(has_heads, "option trainable_head needs the proxy heads ('selfsup' prepare mode)");
        PTTA_CHECK(!bound, "option trainable_head must be set before the workspace is bound");
        // head_main.py:268 hands proj.* and pred.* to Adam, but proj's output is detached on the trained path
        // (network_exp_msg_chn_adapt.py:692): only pred ever receives a gradient, torch.optim.Adam skips the rest
        train_head = true;
        adapt_names = {"pred.0.weight", "pred.0.bias", "pred.1.weight", "pred.1.bias", "pred.3.weight", "pred.3.bias"};
        fuse_projpred = false;       // pred.0 is trained: it cannot be pre-multiplied with proj.3
        plan();                      // sizing pass again: the weight-gradient workspace joins the arena
        return 0;
    }

    // ---- arena plan (run twice: sizing pass with base == nullptr, then with the bound workspace) ----
    void plan_conv(ConvLayer& L) {
        L.pack_fwd = allocv<bf16>((size_t)9 * L.cin * L.cout);
        L.pack_dgrad = allocv<bf16>((size_t)9 * L.cin * L.cout);
        if (L.cin == 32 && L.cout == 32) {
            L.img_fwd = allocv<bf16>(9 * 32 * 32);
            L.img_dgrad = allocv<bf16>(9 * 32 * 32);
        }
    }
    void plan_enc_w(EncW& E) {
        E.init0.dgrad_ch1 = allocv<float>(288);
        E.init0.img_dgrad1 = allocv<bf16>(9 * 16 * 32);
        E.init0.img_tc = allocv<bf16>(2 * 32 * 32);
        plan_conv(E.init2);
        ConvLayer* ls[8] = {&E.e1a, &E.e1b, &E.e2a, &E.e2b, &E.e3a, &E.e3b, &E.e4a, &E.e4b};
        for (int k = 0; k < 2 * E.nenc; ++k) plan_conv(*ls[k]);
    }
    void plan_dec_w(DecW& D) {
        plan_conv(D.d2a); plan_conv(D.d2b); plan_conv(D.d1a); plan_conv(D.d1b); plan_conv(D.p1);
        D.p3.w_fwd = allocv<float>(288); D.p3.w_dgrad = allocv<float>(288);
        D.p3.img_fwd = allocv<bf16>(9 * 16 * 32);
        D.p3.img_dgrad_tc = allocv<bf16>(2 * 32 * 32);
    }
    void plan_enc_act(EncAct& A, const std::string& tag, int h, int w) {
        A.a0 = alloc32((tag + ".a0").c_str(), h, w); A.x0 = alloc32((tag + ".x0").c_str(), h, w);
        A.t1 = alloc32((tag + ".t1").c_str(), h / 2, w / 2); A.x1 = alloc32((tag + ".x1").c_str(), h / 2, w / 2);
        A.t2 = alloc32((tag + ".t2").c_str(), h / 4, w / 4); A.x2 = alloc32((tag + ".x2").c_str(), h / 4, w / 4);
        A.x0r = alloc32((tag + ".x0r").c_str(), h, w); A.x1r = alloc32((tag + ".x1r").c_str(), h / 2, w / 2);
    }
    void plan_dec_act(DecAct& A, const std::string& tag, int h, int w) {   // h,w = resolution of x0 / out
        A.x2 = alloc32((tag + ".x2").c_str(), h / 4, w / 4); A.x1 = alloc32((tag + ".x1").c_str(), h / 2, w / 2);
        A.x0 = alloc32((tag + ".x0").c_str(), h, w);
        A.x2r = alloc32(nullptr, h / 4, w / 4);
        A.u2 = alloc32((tag + ".u2").c_str(), h / 2, w / 2); A.x3 = alloc32((tag + ".x3").c_str(), h / 2, w / 2);
        A.s1 = alloc32((tag + ".s1").c_str(), h / 2, w / 2);
        A.u1 = alloc32((tag + ".u1").c_str(), h, w); A.x4 = alloc32((tag + ".x4").c_str(), h, w);
        A.s0 = alloc32((tag + ".s0").c_str(), h, w); A.h = alloc32((tag + ".h").c_str(), h, w);
        A.out = alloc1((tag + ".out").c_str(), h, w);
    }
    void plan_branch(Branch& B, const std::string& tag, bool is_real) {
        if (is_real) {
            for (int k = 0; k < 5; ++k) B.c[k] = alloc32((tag + ".c" + std::to_string(k)).c_str(), H >> k, W >> k);
            for (int k = 0; k < 4; ++k) B.cr[k] = alloc32(nullptr, H >> k, W >> k);
            B.c2raw = alloc32((tag + ".c2raw").c_str(), H / 4, W / 4);
        } else {
            // zero-image branch: rgb features are the cached rgb_encoder(0) maps; only the meta output is its own
            for (int k = 0; k < 5; ++k) B.c[k] = zc[k];
            B.c2raw = zc[2];
            B.c[2] = alloc32((tag + ".c2").c_str(), H / 4, W / 4);
        }
        if (two_layers) {
            B.mh = alloc32((tag + ".mh").c_str(), H / 4, W / 4, 128);
            B.mg = alloc32((tag + ".mg").c_str(), H / 4, W / 4);
            B.bn1 = alloc_bn(128); B.bn2 = alloc_bn(32);
        }
        if (is_real) plan_enc_act(B.e1, tag + ".e1", H / 4, W / 4); else B.e1 = real.e1;   // identical input -> shared
        plan_dec_act(B.d1, tag + ".d1", H / 4, W / 4);
        B.p12 = alloc1((tag + ".p12").c_str(), H / 2, W / 2);
        plan_enc_act(B.e2, tag + ".e2", H / 2, W / 2);
        plan_dec_act(B.d2, tag + ".d2", H / 2, W / 2);
        B.p11 = alloc1((tag + ".p11").c_str(), H, W);
        plan_enc_act(B.e3, tag + ".e3", H, W);
        if (is_real) {
            plan_dec_act(B.d3, tag + ".d3", H, W);
            B.output = alloc1((tag + ".output").c_str(), H, W);
        }
    }
    void plan() {
        arena.off = 0;
        named.clear(); named_order.clear();
        plan_enc_w(rgbW); plan_enc_w(enc1W); plan_enc_w(enc2W); plan_enc_w(enc3W);
        plan_dec_w(dec1W); plan_dec_w(dec2W); plan_dec_w(dec3W);
        plan_conv(meta1);
        if (two_layers) plan_conv(meta2);
        zero_bias = allocv<float>(512);
        auto alloc_user = [&](const char* name) {
            Map1 m; m.n = Nu; m.h = Hu; m.w = Wu;
            m.p = (float*)arena.take(m.numel() * sizeof(float));
            reg(name, m.p, 0, Nu, Hu, Wu, 1);
            return m;
        };
        fd = alloc_user("filtered_depth"); fv = alloc_user("filtered_validity");
        stage_img = allocv<float>((size_t)Nu * 3 * Hu * Wu); reg("stage_image", stage_img, 0, Nu, 3, Hu, Wu);
        stage_sp = allocv<float>((size_t)Nu * Hu * Wu); reg("stage_sparse", stage_sp, 0, Nu, 1, Hu, Wu);
        stage_gt = allocv<float>((size_t)Nu * Hu * Wu); reg("stage_ground_truth", stage_gt, 0, Nu, 1, Hu, Wu);
        if (padded) {
            pimg = allocv<float>((size_t)N * 3 * H * W);
            psp = allocv<float>((size_t)N * H * W);
            out_u = alloc_user("output_mean"); g_out_u = alloc_user("g_output_mean");
        }
        dcl = alloc1("depth_clamped", H, W); d12 = alloc1("d12", H / 2, W / 2); d14 = alloc1("d14", H / 4, W / 4);
        for (int k = 0; k < 5; ++k) rgbT[k] = alloc32(("rgbT" + std::to_string(k)).c_str(), H >> k, W >> k);
        plan_branch(real, "real", true);
        if (padded) {
            reg("output", out_u.p, 0, Nu, Hu, Wu, 1); reg("output_padded", real.output.p, 0, N, H, W, 1);
        } else {
            reg("output", real.output.p, 0, N, H, W, 1);
        }
        R = (long long)N * (H / 4) * (W / 4);
        if (has_heads) {
            for (int k = 0; k < 5; ++k) zc[k] = alloc32(("zc" + std::to_string(k)).c_str(), H >> k, W >> k);
            for (int k = 0; k < 4; ++k) zcr[k] = real.cr[k];      // rgb_encoder(0) runs at pack time only: borrow the real branch's copies
            plan_branch(zero, "zero", false);
            auto lin = [&](LinearLayer& L) { L.pack = allocv<bf16>((size_t)L.in * L.out); L.pack_t = allocv<bf16>((size_t)L.in * L.out); };
            lin(proj0); lin(proj3); lin(pred0); lin(pred3);
            projpred_pack = allocv<bf16>((size_t)512 * 512); projpred_bias = allocv<float>(512);
            size_t rm = (size_t)R * 512;
            h_an2 = allocv<bf16>(rm);
            h_a0z = allocv<bf16>(rm); h_a0r = allocv<bf16>(rm); h_an = allocv<bf16>(rm); h_pz = allocv<bf16>(rm); h_q0 = allocv<bf16>(rm);
            emb = allocv<bf16>(rm); ref = allocv<bf16>(rm);
            reg("emb", emb, 1, R, 512, 1, 1); reg("ref", ref, 1, R, 512, 1, 1);
            reg("heads.a0_real", h_a0r, 1, R, 512, 1, 1);
            g_ref = allocv<bf16>(rm); g_a3 = allocv<bf16>(rm); g_a0 = allocv<bf16>(rm);
            reg("g_ref", g_ref, 1, R, 512, 1, 1); reg("g_emb", g_a3, 1, R, 512, 1, 1);
            bnProjZ = alloc_bn(512); bnProjR = alloc_bn(512); bnPred = alloc_bn(512);
            rowstat = allocv<float>((size_t)R * 3);
        }
        // backward scratch
        T1a = alloc32("T1a", H, W); T1b = alloc32("T1b", H, W);
        T2a = alloc32("T2a", H / 2, W / 2); T2b = alloc32("T2b", H / 2, W / 2); D2 = alloc32("D2", H / 2, W / 2);
        G4a = alloc32("G4a", H / 4, W / 4); G4b = alloc32("G4b", H / 4, W / 4); D4 = alloc32("D4", H / 4, W / 4);
        GC2 = alloc32("g_c2", H / 4, W / 4); GZ = alloc32("g_z", H / 4, W / 4);
        D8 = alloc32("D8", H / 8, W / 8); E8 = alloc32("E8", H / 8, W / 8);
        if (two_layers) { M128a = alloc32("M128a", H / 4, W / 4, 128); M128b = alloc32("M128b", H / 4, W / 4, 128); }
        g_out = alloc1(padded ? "g_output_padded" : "g_output", H, W); g_p11 = alloc1("g_p11", H, W);
        if (padded) reg("g_output", g_out_u.p, 0, Nu, Hu, Wu, 1);
        g_q = alloc1("g_q", H / 2, W / 2); g_p12 = alloc1("g_p12", H / 2, W / 2); g_o14 = alloc1("g_out14", H / 4, W / 4);
        k0 = allocv<float>(512); k1 = allocv<float>(512); k2 = allocv<float>(512);
        long long max_rows = std::max<long long>(R, 1);
        partial_doubles = (size_t)cdiv(max_rows, STATS_ROWS_PER_BLOCK) * 2 * 512;
        partial = allocv<double>(partial_doubles);
        partial2 = allocv<double>(partial_doubles);
        size_t wg = std::max(wgrad_partial_bytes(N, H / 4, W / 4, 32, 128), wgrad_partial_bytes(N, H / 4, W / 4, 128, 32));
        wgrad_ws = (float*)arena.take(wg);
        wgrad_ws2 = (float*)arena.take(wg);
        partial3 = allocv<double>(partial_doubles);
        losses = (LossScalars*)arena.take(sizeof(LossScalars));
        reg("losses", losses, 0, 5, 1, 1, 1);
        loss_map_blocks = std::min(cdiv((long long)H * W, LOSS_BLOCK * 4), 1184);
        loss_cos_blocks = (int)std::min<long long>(std::max<long long>(cdiv(R, 8), 1), 1184);
        loss_map_partial = allocv<double>((size_t)N * loss_map_blocks * 4);
        loss_cos_partial = allocv<double>(loss_cos_blocks);
        adam_hyper = (AdamHyper*)arena.take(sizeof(AdamHyper));
        adam_chunks = (AdamChunk*)arena.take(sizeof(AdamChunk) * ADAM_MAX_CHUNKS);
        if (train_head) { gw_part = (float*)arena.take(gemm_tn_workspace_bytes(R, 512, 512)); g_q0 = allocv<bf16>((size_t)R * 512); }
        ws_bytes = arena.off + 256;
    }

    // ---- tensor lookup ------------------------------------------------------------------------------
    template <typename T> int get(const std::string& key, T*& out, long long numel) {
        auto it = ext.find(key);
        PTTA_CHECK(it != ext.end(), "state-dict entry '%s' was not bound (ptta_msgchn_set_tensor)", key.c_str());
        PTTA_CHECK(numel < 0 || it->second.second == numel, "state-dict entry '%s' has %lld elements, expected %lld", key.c_str(),
                   it->second.second, numel);
        out = (T*)it->second.first;
        return 0;
    }
    int bind_conv(ConvLayer& L) {
        float* w; PTTA_TRY(get(L.name + ".weight", w, (long long)9 * L.cin * L.cout)); L.w = w;
        if (L.has_bias) { float* b; PTTA_TRY(get(L.name + ".bias", b, L.cout)); L.b = b; }
        return 0;
    }
    int bind_enc(EncW& E) {
        float* w; PTTA_TRY(get(E.init0.name + ".weight", w, 32LL * E.init0.cin * 9)); E.init0.w = w;
        float* b; PTTA_TRY(get(E.init0.name + ".bias", b, 32)); E.init0.b = b;
        PTTA_TRY(bind_conv(E.init2));
        ConvLayer* ls[8] = {&E.e1a, &E.e1b, &E.e2a, &E.e2b, &E.e3a, &E.e3b, &E.e4a, &E.e4b};
        for (int k = 0; k < 2 * E.nenc; ++k) PTTA_TRY(bind_conv(*ls[k]));
        return 0;
    }
    int bind_dec(DecW& D) {
        PTTA_TRY(bind_conv(D.d2a)); PTTA_TRY(bind_conv(D.d2b)); PTTA_TRY(bind_conv(D.d1a)); PTTA_TRY(bind_conv(D.d1b));
        PTTA_TRY(bind_conv(D.p1));
        float* w; PTTA_TRY(get(D.p3.name + ".weight", w, 288)); D.p3.w = w;
        float* b; PTTA_TRY(get(D.p3.name + ".bias", b, 1)); D.p3.b = b;
        return 0;
    }
    int bind_bn(BnLayer& B) {
        PTTA_TRY(get(B.name + ".weight", B.gamma, B.c)); PTTA_TRY(get(B.name + ".bias", B.beta, B.c));
        PTTA_TRY(get(B.name + ".running_mean", B.rm, B.c)); PTTA_TRY(get(B.name + ".running_var", B.rv, B.c));
        PTTA_TRY(get(B.name + ".num_batches_tracked", B.nbt, 1));
        return 0;
    }
    int bind_linear(LinearLayer& L) {
        float* w; PTTA_TRY(get(L.name + ".weight", w, (long long)L.in * L.out)); L.w = w;
        float* b; PTTA_TRY(get(L.name + ".bias", b, L.out)); L.b = b;
        return 0;
    }
    int bind_all() {
        PTTA_TRY(bind_enc(rgbW)); PTTA_TRY(bind_enc(enc1W)); PTTA_TRY(bind_enc(enc2W)); PTTA_TRY(bind_enc(enc3W));
        PTTA_TRY(bind_dec(dec1W)); PTTA_TRY(bind_dec(dec2W)); PTTA_TRY(bind_dec(dec3W));
        PTTA_TRY(bind_conv(meta1));
        if (two_layers) { PTTA_TRY(bind_conv(meta2)); PTTA_TRY(bind_bn(metaBn1)); PTTA_TRY(bind_bn(metaBn2)); }
        if (has_heads) {
            PTTA_TRY(bind_linear(proj0)); PTTA_TRY(bind_linear(proj3)); PTTA_TRY(bind_linear(pred0)); PTTA_TRY(bind_linear(pred3));
            PTTA_TRY(bind_bn(projBn)); PTTA_TRY(bind_bn(predBn));
        }
        return 0;
    }

    // ---- weight packing -------------------------------------------------------------------------------
    int pack_conv(const ConvLayer& L) {
        const int tot = 9 * L.cin * L.cout;
        const int blocks = cdiv(tot, 256);
        if (!L.transposed) {
            // Conv2d weight [cout][cin][3][3]
            launch_k(pack_conv_weight_kernel, blocks, 256, 0, st, L.w, L.pack_fwd, L.cout, L.cin, L.cin * 9, 9, 0);
            PTTA_TRY(check_launch("pack_fwd"));
            // data gradient: output channel = cin, input channel = cout; stride-1 layers flip the taps,
            // stride-2 layers run as a transposed conv with the taps as they are
            launch_k(pack_conv_weight_kernel, blocks, 256, 0, st, L.w, L.pack_dgrad, L.cin, L.cout, 9, L.cin * 9, L.mode_fwd == MODE_S1 ? 1 : 0);
            PTTA_TRY(check_launch("pack_dgrad"));
        } else {
            // ConvTranspose2d weight [cin][cout][3][3]
            launch_k(pack_conv_weight_kernel, blocks, 256, 0, st, L.w, L.pack_fwd, L.cout, L.cin, 9, L.cout * 9, 0);
            PTTA_TRY(check_launch("pack_fwd_t"));
            launch_k(pack_conv_weight_kernel, blocks, 256, 0, st, L.w, L.pack_dgrad, L.cin, L.cout, L.cout * 9, 9, 0);
            PTTA_TRY(check_launch("pack_dgrad_t"));
        }
        if (L.img_fwd) {
            if (L.mode_fwd == MODE_S1) launch_k(pack_conv_weight_tc_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_fwd, L.img_fwd);
            else if (L.mode_fwd == MODE_S2) launch_k(pack_conv_weight_tc_s2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_fwd, L.img_fwd);
            else launch_k(pack_conv_weight_tc_t2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_fwd, L.img_fwd);
            PTTA_TRY(check_launch("pack_fwd_tc"));
        }
        if (L.img_dgrad) {
            if (L.mode_dgrad == MODE_S1) launch_k(pack_conv_weight_tc_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_dgrad, L.img_dgrad);
            else if (L.mode_dgrad == MODE_S2) launch_k(pack_conv_weight_tc_s2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_dgrad, L.img_dgrad);
            else launch_k(pack_conv_weight_tc_t2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, st, L.pack_dgrad, L.img_dgrad);
            PTTA_TRY(check_launch("pack_dgrad_tc"));
        }
        return 0;
    }
    int pack_enc(EncW& E) {
        if (E.init0.cin == 2) {
            launch_k(pack_head_weight_kernel, 2, 256, 0, st, E.init0.w + 9, E.init0.dgrad_ch1, 18, 1);
            PTTA_TRY(check_launch("pack_stem_dgrad"));
            launch_k(pack_conv_weight_tc_head_kernel, cdiv(9 * 16 * 4, 256), 256, 0, st, E.init0.dgrad_ch1, E.init0.img_dgrad1);
            PTTA_TRY(check_launch("pack_stem_dgrad_tc"));
        }
        launch_k(pack_stem_weight_tc_kernel, 1, 256, 0, st, E.init0.w, E.init0.img_tc, E.init0.cin);
        PTTA_TRY(check_launch("pack_stem_tc"));
        PTTA_TRY(pack_conv(E.init2));
        ConvLayer* ls[8] = {&E.e1a, &E.e1b, &E.e2a, &E.e2b, &E.e3a, &E.e3b, &E.e4a, &E.e4b};
        for (int k = 0; k < 2 * E.nenc; ++k) PTTA_TRY(pack_conv(*ls[k]));
        if (E.init0.cin == 2) PTTA_CUDA(cudaMemcpyAsync(E.init0.dk, E.init0.dgrad_ch1, sizeof(E.init0.dk), cudaMemcpyDeviceToHost, st));
        E.init0.raw_host.resize(32 * E.init0.cin * 9 + 32);
        PTTA_CUDA(cudaMemcpyAsync(E.init0.raw_host.data(), E.init0.w, sizeof(float) * 32 * E.init0.cin * 9, cudaMemcpyDeviceToHost, st));
        PTTA_CUDA(cudaMemcpyAsync(E.init0.raw_host.data() + 32 * E.init0.cin * 9, E.init0.b, sizeof(float) * 32, cudaMemcpyDeviceToHost, st));
        return 0;
    }
    // after the stream has been synchronised: [co][ci][tap] -> [ci][tap][co]
    void finish_host_weights(EncW& E) {
        StemLayer& S = E.init0;
        for (int co = 0; co < 32; ++co)
            for (int r = 0; r < S.cin * 9; ++r) S.wk[r * 32 + co] = S.raw_host[(size_t)co * S.cin * 9 + r];
        for (int c = 0; c < 32; ++c) S.bk[c] = S.raw_host[32 * S.cin * 9 + c];
    }
    void finish_host_weights(DecW& D) {
        for (int co = 0; co < 32; ++co)
            for (int t = 0; t < 9; ++t) D.p3.wdk[t * 32 + co] = D.p3.raw_host[co * 9 + t];
    }
    int pack_dec(DecW& D) {
        PTTA_TRY(pack_conv(D.d2a)); PTTA_TRY(pack_conv(D.d2b)); PTTA_TRY(pack_conv(D.d1a)); PTTA_TRY(pack_conv(D.d1b));
        PTTA_TRY(pack_conv(D.p1));
        launch_k(pack_head_weight_kernel, 2, 256, 0, st, D.p3.w, D.p3.w_fwd, 9, 0);
        PTTA_TRY(check_launch("pack_head"));
        launch_k(pack_conv_weight_tc_head_kernel, cdiv(9 * 16 * 4, 256), 256, 0, st, D.p3.w_fwd, D.p3.img_fwd);
        PTTA_TRY(check_launch("pack_head_tc"));
        launch_k(pack_flip9_kernel, 2, 256, 0, st, D.p3.w, D.p3.w_dgrad, 32);
        PTTA_TRY(check_launch("pack_head_dgrad"));
        launch_k(pack_stem_weight_tc_kernel, 1, 256, 0, st, D.p3.w_dgrad, D.p3.img_dgrad_tc, 1);
        PTTA_TRY(check_launch("pack_head_dgrad_tc"));
        PTTA_CUDA(cudaMemcpyAsync(&D.p3.bias_host, D.p3.b, sizeof(float), cudaMemcpyDeviceToHost, st));
        PTTA_CUDA(cudaMemcpyAsync(D.p3.wfk, D.p3.w_fwd, sizeof(D.p3.wfk), cudaMemcpyDeviceToHost, st));
        D.p3.raw_host.resize(288);
        PTTA_CUDA(cudaMemcpyAsync(D.p3.raw_host.data(), D.p3.w_dgrad, sizeof(float) * 288, cudaMemcpyDeviceToHost, st));
        return 0;
    }
    int pack_linear(LinearLayer& L) {
        int tot = L.in * L.out;
        launch_k(pack_matrix_kernel, cdiv(tot, 256), 256, 0, st, L.w, L.pack, L.out, L.in, L.in, 1);
        PTTA_TRY(check_launch("pack_linear"));
        launch_k(pack_matrix_kernel, cdiv(tot, 256), 256, 0, st, L.w, L.pack_t, L.in, L.out, 1, L.in);
        PTTA_TRY(check_launch("pack_linear_t"));
        return 0;
    }
    int pack_adapted() {
        if (train_head) { PTTA_TRY(pack_linear(pred0)); return pack_linear(pred3); }
        PTTA_TRY(pack_conv(meta1));
        if (two_layers) PTTA_TRY(pack_conv(meta2));
        return 0;
    }
    int pack_all() {
        PTTA_TRY(bind_all());
        PTTA_CUDA(cudaMemsetAsync(zero_bias, 0, 512 * sizeof(float), st));
        PTTA_TRY(pack_enc(rgbW)); PTTA_TRY(pack_enc(enc1W)); PTTA_TRY(pack_enc(enc2W)); PTTA_TRY(pack_enc(enc3W));
        PTTA_TRY(pack_dec(dec1W)); PTTA_TRY(pack_dec(dec2W)); PTTA_TRY(pack_dec(dec3W));
        PTTA_TRY(pack_conv(meta1));
        if (two_layers) PTTA_TRY(pack_conv(meta2));
        if (has_heads) {
            PTTA_TRY(pack_linear(proj0)); PTTA_TRY(pack_linear(proj3)); PTTA_TRY(pack_linear(pred0)); PTTA_TRY(pack_linear(pred3));
            launch_k(fuse_linear_kernel, dim3(cdiv(proj3.in, 256), pred0.out), 256, 0, st, pred0.w, pred0.b, proj3.w, proj3.b, projpred_pack,
                     projpred_bias, pred0.out, proj3.out, proj3.in);
            PTTA_TRY(check_launch("fuse_linear"));
        }
        PTTA_CUDA(cudaStreamSynchronize(st));   // bias_host / host weight copies
        finish_host_weights(rgbW); finish_host_weights(enc1W); finish_host_weights(enc2W); finish_host_weights(enc3W);
        finish_host_weights(dec1W); finish_host_weights(dec2W); finish_host_weights(dec3W);
        // Adam chunk table over the adapted tensors
        std::vector<AdamChunk> chunks;
        for (const std::string& k : adapt_names) {
            auto it = ext.find(k);
            PTTA_CHECK(it != ext.end(), "adapted tensor '%s' not bound", k.c_str());
            long long n = it->second.second;
            float *p = (float*)it->second.first, *g = nullptr, *m = nullptr, *v = nullptr;
            if (ext.count("grad/" + k)) g = (float*)ext["grad/" + k].first;
            if (ext.count("adam_m/" + k)) m = (float*)ext["adam_m/" + k].first;
            if (ext.count("adam_v/" + k)) v = (float*)ext["adam_v/" + k].first;
            if (!g || !m || !v) { chunks.clear(); break; }
            for (long long o = 0; o < n; o += ADAM_CHUNK) {
                AdamChunk c; c.p = p + o; c.g = g + o; c.m = m + o; c.v = v + o; c.n = (int)std::min<long long>(ADAM_CHUNK, n - o);
                chunks.push_back(c);
            }
        }
        if (ext.count("adam/hyper")) {
            // one step counter / hyper-parameter block per WRAPPER, shared by its engines of all shapes (a second shape must not
            // restart the bias correction at step 0 on warm moments)
            PTTA_CHECK(ext["adam/hyper"].second >= (long long)sizeof(AdamHyper), "'adam/hyper' needs %zu bytes", sizeof(AdamHyper));
            adam_hyper = (AdamHyper*)ext["adam/hyper"].first;
        }
        adam_g_base = nullptr; adam_g_floats = 0;
        if (!chunks.empty()) {
            const float *lo = chunks[0].g, *hi = chunks[0].g + chunks[0].n;
            for (const AdamChunk& c : chunks) { if (c.g < lo) lo = c.g; if (c.g + c.n > hi) hi = c.g + c.n; }
            adam_g_base = lo; adam_g_floats = (size_t)(hi - lo);
        }
        PTTA_CHECK(chunks.size() <= ADAM_MAX_CHUNKS, "too many Adam chunks (%zu)", chunks.size());
        n_adam_chunks = (int)chunks.size();
        if (n_adam_chunks) PTTA_CUDA(cudaMemcpyAsync(adam_chunks, chunks.data(), sizeof(AdamChunk) * chunks.size(), cudaMemcpyHostToDevice, st));
        if (has_heads) {
            // rgb_encoder(0): constant while the encoder is frozen ('meta' adapt mode never touches it)
            PTTA_TRY(run_rgb_encoder(nullptr, nullptr, nullptr, zc, zcr));
        }
        PTTA_CUDA(cudaStreamSynchronize(st));
        packed = true;
        drop_graphs();
        return 0;
    }

    // ---- layer helpers ----------------------------------------------------------------------------------
    // the tcgen05 kernel takes the big 32->32 stride-1 maps; small maps (where any kernel is launch-bound) stay on mma.sync
    bool use_tc(const Map32& m) const { return tc_enabled && conv_tc_supported(m.n, m.h, m.w) && (long long)m.n * m.h * m.w >= tc_min_pixels; }
    bool use_tc_s2(const Map32& m) const {
        return tc_enabled && conv_tc_s2_supported(m.n, m.h, m.w) && (long long)m.n * m.h * m.w >= tc_s2_min_pixels;
    }
    bool use_tc_t2(const Map32& m) const {       // m: the INPUT map of the transposed conv
        return tc_enabled && conv_tc_t2_supported(m.n, m.h, m.w) && (long long)m.n * m.h * m.w >= tc_t2_min_pixels;
    }
    int conv_tc_t2(const bf16* image, const float* bias, const Map32& in, const Map32& out, int relu_out, const bf16* mask, const bf16* add) {
        ConvTcParams p; memset(&p, 0, sizeof(p));
        p.w = image; p.bias = bias; p.out = out.p; p.mask = mask; p.add = add; p.N = in.n; p.H = in.h; p.W = in.w; p.relu_out = relu_out;
        return launch_conv_tc_t2(in.p, p, st);
    }
    int conv_tc(const bf16* image, const float* bias, const Map32& in, const Map32& out, int relu_out, const bf16* mask, const bf16* add,
                bf16* out2 = nullptr, bool stride2 = false, const bf16* add2 = nullptr, const bf16* up2 = nullptr) {
        ConvTcParams p; memset(&p, 0, sizeof(p));
        p.w = image; p.bias = bias; p.out = out.p; p.out2 = out2; p.add2 = add2; p.mask = mask; p.add = add; p.N = in.n; p.H = in.h; p.W = in.w;
        p.up2 = up2;
        p.relu_out = relu_out;
        return stride2 ? launch_conv_tc_s2(in.p, p, st) : launch_conv_tc(in.p, p, st);
    }
    // relu_out: the output is only ever read through a ReLU (or as a ReLU mask), so ReLU(x) is what gets stored
    // out2 (optional): a second copy holding ReLU(out), for outputs that are read both raw and through a tensor-core conv
    // add2 (with out2): out2 = ReLU(out + add2) -- the decoder sums s = ReLU(conv(..) + skip) without a separate pass
    // true when conv_fwd(L, in, ...) runs on the stride-1 tcgen05 kernel, whose epilogue can add a x2-upsampled half-resolution map
    bool up2_in_epilogue(const ConvLayer& L, const Map32& in) const {
        return L.img_fwd && L.mode_fwd == MODE_S1 && use_tc(in) && (in.h & 1) == 0 && (in.w & 1) == 0;
    }
    int conv_fwd(const ConvLayer& L, const Map32& in, const Map32& out, int pro, const BnState* probn = nullptr, int relu_out = 0,
                 bf16* out2 = nullptr, const bf16* add2 = nullptr, const bf16* up2 = nullptr) {
        if (L.img_fwd && pro == PRO_NONE) {
            if (L.mode_fwd == MODE_S1 && use_tc(in))
                return conv_tc(L.img_fwd, L.has_bias ? L.b : nullptr, in, out, relu_out, nullptr, nullptr, out2, false, add2, up2);
            PTTA_CHECK(up2 == nullptr, "conv_fwd: the upsampled addend is fused by the stride-1 tcgen05 kernel only");
            if (L.mode_fwd == MODE_S2 && use_tc_s2(in) && !add2)
                return conv_tc(L.img_fwd, L.has_bias ? L.b : nullptr, in, out, relu_out, nullptr, nullptr, out2, true);
            if (L.mode_fwd == MODE_T2 && use_tc_t2(in) && !add2 && !out2)
                return conv_tc_t2(L.img_fwd, L.has_bias ? L.b : nullptr, in, out, relu_out, nullptr, nullptr);
        }
        ConvParams p; memset(&p, 0, sizeof(p));
        p.relu_out = relu_out; p.out2 = out2; p.add2 = add2;
        p.in = in.p; p.out = out.p; p.w = L.pack_fwd; p.bias = L.has_bias ? L.b : nullptr;
        p.N = in.n; p.Hin = in.h; p.Win = in.w; p.pro = pro; p.slope = 0.2f;
        if (probn) { p.pro_scale = probn->scale; p.pro_shift = probn->shift; }
        return launch_conv3x3(p, L.cin, L.cout, L.mode_fwd, st);
    }
    // gin = [add +] mask * dgrad(gout)
    int conv_dgrad(const ConvLayer& L, const Map32& gout, const Map32& gin, const bf16* mask, const bf16* add,
                   int mask_mode = MASK_RELU, const BnState* maskbn = nullptr) {
        if (L.img_dgrad && (!mask || mask_mode == MASK_RELU)) {
            if (L.mode_dgrad == MODE_S1 && use_tc(gout)) return conv_tc(L.img_dgrad, nullptr, gout, gin, 0, mask, add);
            if (L.mode_dgrad == MODE_S2 && use_tc_s2(gout)) return conv_tc(L.img_dgrad, nullptr, gout, gin, 0, mask, add, nullptr, true);
            if (L.mode_dgrad == MODE_T2 && use_tc_t2(gout)) return conv_tc_t2(L.img_dgrad, nullptr, gout, gin, 0, mask, add);
        }
        ConvParams p; memset(&p, 0, sizeof(p));
        p.in = gout.p; p.out = gin.p; p.w = L.pack_dgrad; p.bias = nullptr;
        p.N = gout.n; p.Hin = gout.h; p.Win = gout.w; p.pro = PRO_NONE; p.slope = 0.2f;
        p.mask = mask; p.mask_mode = mask ? mask_mode : MASK_NONE; p.add = add;
        if (maskbn) { p.mask_scale = maskbn->scale; p.mask_shift = maskbn->shift; }
        return launch_conv3x3(p, L.cout, L.cin, L.mode_dgrad, st);
    }
    int add32(const Map32& a, const Map32& b, const Map32& out, int relu = 0) {
        long long n8 = (long long)a.numel() / 8;
        launch_k(ew_add_kernel, cdiv(n8, 256), 256, 0, st, a.p, b.p, out.p, n8, relu);
        return check_launch("ew_add");
    }
    int add_up2(const Map32& x, const Map32& half, bf16* relu_copy = nullptr) {   // x += up2(half) [; relu_copy = ReLU(x)]
        long long tot = (long long)x.n * x.h * x.w * 4;
        launch_k(add_up2_c32_kernel, cdiv(tot, 256), 256, 0, st, x.p, half.p, x.p, x.n, half.h, half.w, relu_copy);
        return check_launch("add_up2_c32");
    }
    int up2_adj32(const Map32& ghi, const Map32& glo, int accumulate) {
        long long tot = (long long)glo.n * glo.h * glo.w * 4;
        launch_k(up2_c32_adj_kernel, cdiv(tot, 256), 256, 0, st, ghi.p, glo.p, glo.n, glo.h, glo.w, accumulate);
        return check_launch("up2_c32_adj");
    }
    int up2_1(const Map1& a, const float* b, const float* c, const Map1& out) {
        long long tot = (long long)out.numel();
        launch_k(up2_1ch_kernel, cdiv(tot, 256), 256, 0, st, a.p, b, c, out.p, a.n, a.h, a.w);
        return check_launch("up2_1ch");
    }
    int up2_adj1(const Map1& ghi, const Map1& glo) {
        long long tot = (long long)glo.numel();
        launch_k(up2_1ch_adj_kernel, cdiv(tot, 256), 256, 0, st, ghi.p, glo.p, glo.n, glo.h, glo.w, 0);
        return check_launch("up2_1ch_adj");
    }
    int stem(const StemLayer& S, const float* p0, long long s0, float sc0, float sh0, const float* p1, long long s1, float sc1,
             float sh1, const float* p2, long long s2, float sc2, float sh2, const Map32& out) {
        if (use_tc_stem(out)) {         // contraction on the tensor cores (stem_tc.cuh)
            StemTcParams t; memset(&t, 0, sizeof(t));
            t.relu_out = 1;
            t.plane[0] = p0; t.plane[1] = p1; t.plane[2] = p2;
            t.batch_stride[0] = s0; t.batch_stride[1] = s1; t.batch_stride[2] = s2;
            t.scale[0] = sc0; t.scale[1] = sc1; t.scale[2] = sc2; t.shift[0] = sh0; t.shift[1] = sh1; t.shift[2] = sh2;
            t.w = S.img_tc; t.bias = S.b; t.out = out.p; t.N = out.n; t.H = out.h; t.W = out.w;
            return launch_stem_tc(t, S.cin, st);
        }
        if ((out.w & 1) == 0) {         // weights by value (constant bank): the FMA-only kernel
            StemCParams c; memset(&c, 0, sizeof(c));
            c.relu_out = 1;
            c.plane[0] = p0; c.plane[1] = p1; c.plane[2] = p2;
            c.batch_stride[0] = s0; c.batch_stride[1] = s1; c.batch_stride[2] = s2;
            c.scale[0] = sc0; c.scale[1] = sc1; c.scale[2] = sc2; c.shift[0] = sh0; c.shift[1] = sh1; c.shift[2] = sh2;
            c.out = out.p; c.N = out.n; c.H = out.h; c.W = out.w;
            memcpy(c.w, S.wk, sizeof(float) * S.cin * 9 * 32); memcpy(c.bias, S.bk, sizeof(c.bias));
            launch_stem_const(c, S.cin, st);
            return check_launch("stem_conv");
        }
        StemParams p; memset(&p, 0, sizeof(p));
        p.relu_out = 1;                 // init.0 outputs are consumed through ReLU only (and as ReLU masks in backward)
        p.plane[0] = p0; p.plane[1] = p1; p.plane[2] = p2;
        p.batch_stride[0] = s0; p.batch_stride[1] = s1; p.batch_stride[2] = s2;
        p.scale[0] = sc0; p.scale[1] = sc1; p.scale[2] = sc2; p.shift[0] = sh0; p.shift[1] = sh1; p.shift[2] = sh2;
        p.w = S.w; p.bias = S.b; p.mask = nullptr; p.out = out.p; p.N = out.n; p.H = out.h; p.W = out.w;
        launch_stem(p, S.cin, st);
        return check_launch("stem_conv");
    }
    bool use_tc_stem(const Map32& m) const { return tc_enabled && (long long)m.n * m.h * m.w >= tc_stem_min_pixels; }
    bool use_tc_head(const Map1& m) const {
        return tc_enabled && conv_tc_supported(m.n, m.h, m.w) && (long long)m.n * m.h * m.w >= tc_head_min_pixels;
    }
    // the 32 -> 1 convolution on the tensor cores (the input already holds ReLU(.) where the layer reads it through one)
    int head_conv_tc(const bf16* in, const bf16* image, float bias, const float* add, const Map1& out) {
        ConvTcParams p; memset(&p, 0, sizeof(p));
        p.w = image; p.N = out.n; p.H = out.h; p.W = out.w; p.out_f32 = out.p; p.add_f32 = add; p.bias0 = bias;
        return launch_conv_tc_head(in, p, st);
    }
    // prediction layer: out = conv32->1(relu(h)) + bias [+ add]
    int head_convv(const bf16* in, const float* wk, float bias, const float* add, const Map1& out, int relu_in) {
        HeadCParams c; memset(&c, 0, sizeof(c));
        c.in = in; c.add = add; c.out = out.p; c.N = out.n; c.H = out.h; c.W = out.w; c.relu_in = relu_in; c.bias = bias;
        memcpy(c.w, wk, sizeof(c.w));
        launch_k(head_convc_kernel, dim3(cdiv(out.w, HEADC_TW), cdiv(out.h, HEADC_TH), out.n), dim3(HEADC_TW, HEADC_TH), 0, st, c);
        return 0;
    }
    int head_fwd(const HeadLayer& Hd, const Map32& h, const float* add, const Map1& out) {
        if (use_tc_head(out)) return head_conv_tc(h.p, Hd.img_fwd, Hd.bias_host, add, out);      // h is stored as ReLU(h) by prdct.1
        PTTA_TRY(head_convv(h.p, Hd.wfk, Hd.bias_host, add, out, 1));
        return check_launch("head_conv");
    }
    // g_h = dgrad_{1->32}(g_out) * [h > 0]
    int head_dgrad(const HeadLayer& Hd, const Map1& gout, const Map32& hmask, const Map32& gh) {
        if (use_tc_stem(gh)) {
            StemTcParams t; memset(&t, 0, sizeof(t));
            t.plane[0] = gout.p; t.batch_stride[0] = (long long)gout.h * gout.w; t.scale[0] = 1.f;
            t.w = Hd.img_dgrad_tc; t.mask = hmask.p; t.out = gh.p; t.N = gh.n; t.H = gh.h; t.W = gh.w;
            return launch_stem_tc(t, 1, st);
        }
        if ((gh.w & 1) == 0) {
            StemCParams c; memset(&c, 0, sizeof(c));
            c.plane[0] = gout.p; c.batch_stride[0] = (long long)gout.h * gout.w; c.scale[0] = 1.f;
            c.mask = hmask.p; c.out = gh.p; c.N = gh.n; c.H = gh.h; c.W = gh.w;
            memcpy(c.w, Hd.wdk, sizeof(Hd.wdk));
            launch_stem_const(c, 1, st);
            return check_launch("head_dgrad");
        }
        StemParams p; memset(&p, 0, sizeof(p));
        p.plane[0] = gout.p; p.batch_stride[0] = (long long)gout.h * gout.w; p.scale[0] = 1.f;
        p.w = Hd.w_dgrad; p.bias = nullptr; p.mask = hmask.p; p.out = gh.p; p.N = gh.n; p.H = gh.h; p.W = gh.w; p.relu_out = 0;
        launch_stem(p, 1, st);
        return check_launch("head_dgrad");
    }
    // gradient wrt input plane 1 of a 2-plane stem: out = conv32->1(g_a0; flipped plane-1 weights) + add
    int stem_dgrad_ch1(const StemLayer& S, const Map32& ga0, const float* add, const Map1& out) {
        if (use_tc_head(out)) return head_conv_tc(ga0.p, S.img_dgrad1, 0.f, add, out);
        PTTA_TRY(head_convv(ga0.p, S.dk, 0.f, add, out, 0));
        return check_launch("stem_dgrad");
    }
    int take_xid() {
        if (next_xid >= PTTA_COMM_MAX_XID) { set_error("shared-model mode: more than %d peer exchanges in one step", PTTA_COMM_MAX_XID); return -1; }
        return next_xid++;
    }
    int stats(const bf16* x, const bf16* dy, long long rows, int C, int mode, const BnState* s, int relu_mask, int& nblk) {
        nblk = cdiv(rows, STATS_ROWS_PER_BLOCK);
        PTTA_CHECK((size_t)nblk * 2 * C <= partial_doubles, "stats partial buffer too small");
        launch_k(col_stats_kernel, nblk, 256, 2 * 2048 * sizeof(double), st, x, dy, partial, rows, C, mode, s ? s->mean : nullptr,
                                                                      s ? s->invstd : nullptr, s ? s->scale : nullptr,
                                                                      s ? s->shift : nullptr, relu_mask);
        return check_launch("col_stats");
    }
    // defer_running: compute the batch statistics now, leave the running-statistics update to bn_running_update (ordering)
    int bn_forward_stats(const BnLayer& L, const BnState& s, const bf16* x, long long rows, bool training, bool defer_running = false) {
        int nblk = 0;
        BnParams p; p.gamma = L.gamma; p.beta = L.beta; p.running_mean = L.rm; p.running_var = L.rv; p.num_batches_tracked = L.nbt;
        if (defer_running) { p.running_mean = nullptr; p.running_var = nullptr; p.num_batches_tracked = nullptr; }
        p.uvar = s.uvar;
        p.mean = s.mean; p.invstd = s.invstd; p.scale = s.scale; p.shift = s.shift; p.momentum = 0.1f; p.eps = 1e-5f;
        if (training) PTTA_TRY(stats(x, nullptr, rows, L.c, 0, nullptr, 0, nblk));
        const int xid = (training && comm.world > 1) ? take_xid() : 0;
        if (xid < 0) return 1;
        launch_k(bn_finalize_kernel, cdiv(L.c, 32), FIN_THREADS, 0, st, partial, nblk, rows, L.c, p, training ? 1 : 0, comm, xid);
        return check_launch("bn_finalize");
    }
    int bn_running_update(const BnLayer& L, const BnState& s) {
        launch_k(bn_running_update_kernel, cdiv(L.c, 128), 128, 0, st, s.mean, s.uvar, L.rm, L.rv, L.nbt, L.c, 0.1f);
        return check_launch("bn_running_update");
    }
    int bn_apply(const bf16* x, const bf16* res, bf16* y, long long rows, int C, const BnState& s, int act) {
        launch_k(bn_apply_kernel, cdiv(rows, (256 / (C / 8)) * EW_ROWS), 256, 0, st, x, res, y, rows, C, s.scale, s.shift, act);
        return check_launch("bn_apply");
    }
    // dx = BN-backward(dy [* relu mask]); optionally writes dgamma / dbeta
    int bn_backward(const BnLayer& L, const BnState& s, const bf16* dy, const bf16* x, bf16* dx, long long rows, int relu_mask,
                    float* dgamma, float* dbeta) {
        int nblk = 0;
        PTTA_TRY(stats(x, dy, rows, L.c, 1, &s, relu_mask, nblk));
        const int xid = comm.world > 1 ? take_xid() : 0;
        if (xid < 0) return 1;
        launch_k(bn_bwd_finalize_kernel, cdiv(L.c, 32), FIN_THREADS, 0, st, partial, nblk, rows, L.c, L.gamma, s.invstd, dgamma, dbeta, k0, k1, k2, comm, xid);
        PTTA_TRY(check_launch("bn_bwd_finalize"));
        launch_k(bn_bwd_apply_kernel, cdiv(rows, (256 / (L.c / 8)) * EW_ROWS), 256, 0, st, dy, x, dx, rows, L.c, s.mean, s.invstd, k0, k1, k2, s.scale, s.shift, relu_mask);
        return check_launch("bn_bwd_apply");
    }
    int gemm(const bf16* A, const bf16* B, bf16* C, const float* bias, long long M, int Nn, int K) {
        if (gemm_tc_supported(M, Nn, K)) return launch_gemm_tc(A, B, C, bias, M, Nn, K, st);
        GemmParams p; p.A = A; p.B = B; p.C = C; p.bias = bias; p.M = M; p.N = Nn; p.K = K;
        return launch_gemm(p, st);
    }

    // ---- network pieces -------------------------------------------------------------------------------
    // image == nullptr -> zero image (constant planes: scale 0, shift 0)
    int run_rgb_encoder(const float* image, const float* isc, const float* ish, Map32* c, Map32* cr) {
        const long long hw = (long long)H * W;
        const float* base = image ? image : fd.p;   // any valid pointer; scale 0 makes the value irrelevant
        float s[3], b[3];
        for (int k = 0; k < 3; ++k) { s[k] = image ? isc[k] : 0.f; b[k] = image ? ish[k] : 0.f; }
        if (image)
            PTTA_TRY(stem(rgbW.init0, base, 3 * hw, s[0], b[0], base + hw, 3 * hw, s[1], b[1], base + 2 * hw, 3 * hw, s[2], b[2], rgbT[0]));
        else
            PTTA_TRY(stem(rgbW.init0, base, hw, 0.f, 0.f, base, hw, 0.f, 0.f, base, hw, 0.f, 0.f, rgbT[0]));
        PTTA_TRY(conv_fwd(rgbW.init2, rgbT[0], c[0], PRO_NONE, nullptr, 0, cr[0].p));
        const ConvLayer* ls[8] = {&rgbW.e1a, &rgbW.e1b, &rgbW.e2a, &rgbW.e2b, &rgbW.e3a, &rgbW.e3b, &rgbW.e4a, &rgbW.e4b};
        for (int k = 1; k <= 4; ++k) {
            PTTA_TRY(conv_fwd(*ls[2 * (k - 1)], cr[k - 1], rgbT[k], PRO_NONE, nullptr, 1));      // stride 2 on ReLU(x_{k-1})
            PTTA_TRY(conv_fwd(*ls[2 * (k - 1) + 1], rgbT[k], c[k], PRO_NONE, nullptr, 0, k < 4 ? cr[k].p : nullptr));
        }
        return 0;
    }
    // c2 = meta(c2raw)
    int run_meta(Branch& B, bool training, bool defer_running = false) {
        if (!two_layers) return conv_fwd(meta1, B.c2raw, B.c[2], PRO_NONE);
        const long long rows = (long long)N * (H / 4) * (W / 4);
        PTTA_TRY(conv_fwd(meta1, B.c2raw, B.mh, PRO_NONE));
        PTTA_TRY(bn_forward_stats(metaBn1, B.bn1, B.mh.p, rows, training, defer_running));
        PTTA_TRY(conv_fwd(meta2, B.mh, B.mg, PRO_BN_LEAKY, &B.bn1));
        PTTA_TRY(bn_forward_stats(metaBn2, B.bn2, B.mg.p, rows, training, defer_running));
        return bn_apply(B.mg.p, B.c2raw.p, B.c[2].p, rows, 32, B.bn2, 0);
    }
    int run_encoder(const EncW& Wt, EncAct& A, const float* p0, const float* p1, const Map32* pre_x4, const Map32* pre_x3,
                    const Map32* pre_x2) {
        const long long hw = (long long)A.a0.h * A.a0.w;
        PTTA_TRY(stem(Wt.init0, p0, hw, 1.f, 0.f, p1 ? p1 : p0, hw, 1.f, 0.f, p0, hw, 0.f, 0.f, A.a0));
        // a0, t1, t2 hold ReLU(.) (stored by their producers): the stride-1 convs need no prologue
        // x0 / x1 are needed through ReLU by the stride-2 convs (and as ReLU masks in backward): whoever writes them last also writes the ReLU copy
        // x_k = conv(.) + up2(pre_x): the upsampled addend rides in the epilogue of the tcgen05 conv (no pass of its own); maps too small
        // for that kernel keep the separate add_up2 pass
        if (pre_x4 && up2_in_epilogue(Wt.init2, A.a0)) {
            PTTA_TRY(conv_fwd(Wt.init2, A.a0, A.x0, PRO_NONE, nullptr, 0, A.x0r.p, nullptr, pre_x4->p));
        } else {
            PTTA_TRY(conv_fwd(Wt.init2, A.a0, A.x0, PRO_NONE, nullptr, 0, pre_x4 ? nullptr : A.x0r.p));
            if (pre_x4) PTTA_TRY(add_up2(A.x0, *pre_x4, A.x0r.p));
        }
        PTTA_TRY(conv_fwd(Wt.e1a, A.x0r, A.t1, PRO_NONE, nullptr, 1));
        if (pre_x3 && up2_in_epilogue(Wt.e1b, A.t1)) {
            PTTA_TRY(conv_fwd(Wt.e1b, A.t1, A.x1, PRO_NONE, nullptr, 0, A.x1r.p, nullptr, pre_x3->p));
        } else {
            PTTA_TRY(conv_fwd(Wt.e1b, A.t1, A.x1, PRO_NONE, nullptr, 0, pre_x3 ? nullptr : A.x1r.p));
            if (pre_x3) PTTA_TRY(add_up2(A.x1, *pre_x3, A.x1r.p));
        }
        PTTA_TRY(conv_fwd(Wt.e2a, A.x1r, A.t2, PRO_NONE, nullptr, 1));
        if (pre_x2 && up2_in_epilogue(Wt.e2b, A.t2)) {
            PTTA_TRY(conv_fwd(Wt.e2b, A.t2, A.x2, PRO_NONE, nullptr, 0, nullptr, nullptr, pre_x2->p));
        } else {
            PTTA_TRY(conv_fwd(Wt.e2b, A.t2, A.x2, PRO_NONE));
            if (pre_x2) PTTA_TRY(add_up2(A.x2, *pre_x2));
        }
        return 0;
    }
    // cx0/cx1/cx2: rgb features at the resolutions of x0/x1/x2; out = prediction [+ add]
    int run_decoder(const DecW& Wt, DecAct& A, const EncAct& E, const Map32& cx0, const Map32& cx1, const Map32& cx2,
                    const float* add, const Map1& out) {
        {   // x2 = dx2 + cx2 (and ReLU(x2)), x1 = dx1 + cx1, x0 = dx0 + cx0 in one launch
            DecSumsParams dp;
            dp.a[0] = E.x2.p; dp.b[0] = cx2.p; dp.out[0] = A.x2.p; dp.n8[0] = (long long)A.x2.numel() / 8;
            dp.a[1] = E.x1.p; dp.b[1] = cx1.p; dp.out[1] = A.x1.p; dp.n8[1] = (long long)A.x1.numel() / 8;
            dp.a[2] = E.x0.p; dp.b[2] = cx0.p; dp.out[2] = A.x0.p; dp.n8[2] = (long long)A.x0.numel() / 8;
            dp.out0_relu = A.x2r.p;
            launch_k(dec_sums_kernel, cdiv(dp.n8[0] + dp.n8[1] + dp.n8[2], 256), 256, 0, st, dp);
            PTTA_TRY(check_launch("dec_sums"));
        }
        // x2r, u2, s1, u1, s0, h hold ReLU(.): each is read through a ReLU only (forward) or as a ReLU mask (backward)
        PTTA_TRY(conv_fwd(Wt.d2a, A.x2r, A.u2, PRO_NONE, nullptr, 1));
        PTTA_TRY(conv_fwd(Wt.d2b, A.u2, A.x3, PRO_NONE, nullptr, 0, A.s1.p, A.x1.p));      // x3, and s1 = ReLU(x1 + x3) from the same epilogue
        PTTA_TRY(conv_fwd(Wt.d1a, A.s1, A.u1, PRO_NONE, nullptr, 1));
        PTTA_TRY(conv_fwd(Wt.d1b, A.u1, A.x4, PRO_NONE, nullptr, 0, A.s0.p, A.x0.p));      // x4, and s0 = ReLU(x4 + x0)
        PTTA_TRY(conv_fwd(Wt.p1, A.s0, A.h, PRO_NONE, nullptr, 1));
        return head_fwd(Wt.p3, A.h, add, out);
    }
    int run_cascade(Branch& B, bool is_real, bool enc1_done = false) {
        if (is_real && !enc1_done) PTTA_TRY(run_encoder(enc1W, B.e1, d14.p, nullptr, nullptr, nullptr, nullptr));
        PTTA_TRY(run_decoder(dec1W, B.d1, B.e1, B.c[2], B.c[3], B.c[4], nullptr, B.d1.out));
        PTTA_TRY(up2_1(B.d1.out, nullptr, nullptr, B.p12));                        // p12 = up2(out14)
        PTTA_TRY(run_encoder(enc2W, B.e2, d12.p, B.p12.p, &B.d1.x4, &B.d1.x3, &B.d1.x2));
        PTTA_TRY(run_decoder(dec2W, B.d2, B.e2, B.c[1], B.c[2], B.c[3], nullptr, B.d2.out));
        PTTA_TRY(up2_1(B.d2.out, B.p12.p, nullptr, B.p11));                        // p11 = up2(out12 + p12)
        PTTA_TRY(run_encoder(enc3W, B.e3, dcl.p, B.p11.p, &B.d2.x4, &B.d2.x3, &B.d2.x2));
        if (!is_real) return 0;                                                    // zero branch stops after encoder 3
        if (mlp_on_st3) {
            // ref = proj(z_real) needs e3.x2 only: it runs on the second side stream while decoder 3 runs here
            PTTA_CUDA(cudaEventRecord(ev_e3, st));
            PTTA_CUDA(cudaStreamWaitEvent(st3, ev_e3, 0));
            cudaStream_t main = st; double* main_partial = partial;
            st = st3; partial = partial3;
            int rc3 = mlp(proj0, projBn, bnProjR, proj3, real.e3.x2.p, 32, h_a0r, ref, true, h_an, nullptr, ev_projbn);
            if (!rc3 && cudaEventRecord(ev_mlp, st3) != cudaSuccess) { set_error("cudaEventRecord failed"); rc3 = 2; }
            st = main; partial = main_partial;
            if (rc3) return rc3;
        }
        if (skip_dec3) return 0;
        return run_decoder(dec3W, B.d3, B.e3, B.c[0], B.c[1], B.c[2], B.p11.p, B.output);   // output = out11 + p11
    }
    int mlp(const LinearLayer& L0, const BnLayer& bn, const BnState& s, const LinearLayer& L3, const bf16* x, int in_dim, bf16* a0, bf16* out,
            bool training, bf16* scratch, cudaEvent_t after_bn = nullptr, cudaEvent_t before_bn = nullptr) {
        PTTA_TRY(gemm(x, L0.pack, a0, L0.b, R, L0.out, in_dim));
        if (before_bn) PTTA_CUDA(cudaStreamWaitEvent(st, before_bn, 0));      // running statistics are updated in the reference's order
        PTTA_TRY(bn_forward_stats(bn, s, a0, R, training));
        if (after_bn) PTTA_CUDA(cudaEventRecord(after_bn, st));
        PTTA_TRY(bn_apply(a0, nullptr, scratch, R, L0.out, s, 1));
        return gemm(scratch, L3.pack, out, L3.b, R, L3.out, L3.in);
    }

    // image / sparse are the caller's (Nu, Hu, Wu) tensors; with `padded` the network runs on the flip-padded pair
    // mode: 0 = eval, 1 = train with the proxy branch (TTA and the stage-2 head trainer), 2 = train WITHOUT it (stage 1:
    // network_exp_msg_chn_adapt.py:559-607 `_rgbd_meta_contrast_init` -- real branch only, meta-layer BatchNorm in train mode)
    int forward(const float* image, const float* isc, const float* ish, const float* sparse, float cap, int mode) {
        PTTA_CHECK(bound && packed, "engine not ready: bind a workspace and pack weights first");
        PTTA_CHECK(mode >= 0 && mode <= 2, "forward: mode %d", mode);
        PTTA_CHECK(mode != 1 || has_heads, "training forward needs the proxy heads ('selfsup' prepare mode)");
        PTTA_CHECK(mode != 2 || !skip_dec3, "stage-1 forward needs decoder 3 (option skip_dec3 is set)");
        proxy_in_backward = mode != 2;
        next_xid = 0;                   // a step's peer exchanges are numbered from its forward pass on
        if (!padded) return forward_impl(image, isc, ish, sparse, cap, mode);
        {
            // the reference pads the NORMALISED image with zeros (msg_chn_model_adapt.py:79-101): fill with the raw value that
            // normalises to zero, so that the affine folded into the stem reproduces it
            float f[3];
            for (int c = 0; c < 3; ++c) f[c] = isc[c] != 0.f ? -ish[c] / isc[c] : 0.f;
            long long tot = (long long)N * 3 * H * W;
            launch_k(pad_pair_kernel, cdiv(tot, 256), 256, 0, st, image, pimg, Nu, 3, Hu, Wu, H, W, 1.f, f[0], f[1], f[2]);
            PTTA_TRY(check_launch("pad_pair(image)"));
            tot = (long long)N * H * W;
            launch_k(pad_pair_kernel, cdiv(tot, 256), 256, 0, st, sparse, psp, Nu, 1, Hu, Wu, H, W, 1.f, 0.f, 0.f, 0.f);
            PTTA_TRY(check_launch("pad_pair(sparse)"));
        }
        PTTA_TRY(forward_impl(pimg, isc, ish, psp, cap, mode));
        long long tot = (long long)Nu * Hu * Wu;
        launch_k(unpad_mean_kernel, cdiv(tot, 256), 256, 0, st, real.output.p, out_u.p, Nu, Hu, Wu, H, W);
        return check_launch("unpad_mean");
    }
    int forward_impl(const float* image, const float* isc, const float* ish, const float* sparse, float cap, int mode) {
        const bool training = mode == 1;
        {
            long long tot = (long long)N * (H / 4) * (W / 4);
            launch_k(pyramid_kernel, cdiv(tot, 128), 128, 0, st, sparse, dcl.p, d12.p, d14.p, N, H, W, cap, cap > 0.f ? 1 : 0);
            PTTA_TRY(check_launch("pyramid"));
        }
        Map32 rc[5] = {real.c[0], real.c[1], real.c2raw, real.c[3], real.c[4]};
        const bool fork = training && two_streams && st2 != nullptr;
        if (!fork) {
            PTTA_TRY(run_rgb_encoder(image, isc, ish, rc, real.cr));
            PTTA_TRY(run_meta(real, mode != 0));
            PTTA_TRY(run_cascade(real, true));
            if (!training) return 0;
            PTTA_TRY(zero_side(false));
            return mlp(proj0, projBn, bnProjR, proj3, real.e3.x2.p, 32, h_a0r, ref, true, h_an);
        }
        // Two streams.  The zero-image branch depends on the sparse depth and the weights only -- not on the image -- so it
        // starts right after the pyramid, together with encoder 1 (shared by both branches), while the main stream runs the RGB
        // encoder.  What the reference's execution order fixes (real branch first, zero branch second) are the in-place
        // BatchNorm running-statistics updates: the zero branch defers its meta-layer updates (they are applied on the main
        // stream after the real ones) and the proxy-head BatchNorm keeps zero rows -> real rows through ev_projbn.
        PTTA_CUDA(cudaEventRecord(ev_fork, st));
        {
            cudaStream_t main = st;
            double* main_partial = partial;
            PTTA_CUDA(cudaStreamWaitEvent(st2, ev_fork, 0));
            st = st2; partial = partial2;
            int rc2 = run_encoder(enc1W, real.e1, d14.p, nullptr, nullptr, nullptr, nullptr);
            if (!rc2 && cudaEventRecord(ev_enc1, st2) != cudaSuccess) { set_error("cudaEventRecord failed"); rc2 = 2; }
            if (!rc2) rc2 = zero_side(true);
            if (!rc2 && cudaEventRecord(ev_join, st2) != cudaSuccess) { set_error("cudaEventRecord failed"); rc2 = 2; }
            st = main; partial = main_partial;
            if (rc2) return rc2;
        }
        PTTA_TRY(run_rgb_encoder(image, isc, ish, rc, real.cr));
        PTTA_TRY(run_meta(real, true));
        if (two_layers) {
            PTTA_CUDA(cudaStreamWaitEvent(st, ev_zmeta, 0));
            PTTA_TRY(bn_running_update(metaBn1, zero.bn1));
            PTTA_TRY(bn_running_update(metaBn2, zero.bn2));
        }
        PTTA_CUDA(cudaStreamWaitEvent(st, ev_enc1, 0));
        mlp_on_st3 = true;
        int rcc = run_cascade(real, true, true);
        mlp_on_st3 = false;
        PTTA_TRY(rcc);
        PTTA_CUDA(cudaStreamWaitEvent(st, ev_mlp, 0));
        PTTA_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
        return 0;
    }
    // zero-image branch (no_grad in the reference, network_exp_msg_chn_adapt.py:508-532; BN running statistics are updated a second
    // time here, exactly as the reference does) and emb = pred(proj(z_zero)) (:553); rows = pixels of the /4 map (NHWC)
    int zero_side(bool defer_meta_running) {
        PTTA_TRY(run_meta(zero, true, defer_meta_running));
        if (defer_meta_running && two_layers) PTTA_CUDA(cudaEventRecord(ev_zmeta, st));
        PTTA_TRY(run_cascade(zero, false));
        if (!fuse_projpred) {
            PTTA_TRY(mlp(proj0, projBn, bnProjZ, proj3, zero.e3.x2.p, 32, h_a0z, h_pz, true, h_an2, ev_projbn));
            return mlp(pred0, predBn, bnPred, pred3, h_pz, 512, h_q0, emb, true, h_an2);
        }
        // proj.3 and pred.0 are two Linear layers with nothing between them: one GEMM with W = W_pred0 W_proj3 (pack time, fp32)
        PTTA_TRY(gemm(zero.e3.x2.p, proj0.pack, h_a0z, proj0.b, R, proj0.out, 32));
        PTTA_TRY(bn_forward_stats(projBn, bnProjZ, h_a0z, R, true));
        PTTA_CUDA(cudaEventRecord(ev_projbn, st));
        PTTA_TRY(bn_apply(h_a0z, nullptr, h_an2, R, proj0.out, bnProjZ, 1));
        PTTA_TRY(gemm(h_an2, projpred_pack, h_q0, projpred_bias, R, pred0.out, proj3.in));
        PTTA_TRY(bn_forward_stats(predBn, bnPred, h_q0, R, true));
        PTTA_TRY(bn_apply(h_q0, nullptr, h_an2, R, pred0.out, bnPred, 1));
        return gemm(h_an2, pred3.pack, emb, pred3.b, R, pred3.out, pred3.in);
    }

    // ---- losses (src/external_model_adapt.py:371-441) ----------------------------------------------------
    int loss(const float* image_raw, const float* sparse, const float* validity, float cap, float w_sd, float w_sm, float w_cos) {
        PTTA_CHECK(Nu <= 64, "loss: batch size %d > 64 not supported", Nu);
        l_img = image_raw; l_d = sparse; l_v = validity; l_cap = cap; l_wsd = w_sd; l_wsm = w_sm;
        // the map losses are taken on the caller-shaped prediction (the un-padded mean when `padded`); the cosine loss on all R rows
        const float* pred = padded ? out_u.p : real.output.p;
        dim3 grid(loss_map_blocks, Nu);
        launch_k(loss_map_reduce_kernel, grid, LOSS_BLOCK, 0, st, pred, sparse, validity, image_raw, loss_map_partial, Hu, Wu, cap,
                                                           cap > 0.f ? 1 : 0);
        PTTA_TRY(check_launch("loss_map_reduce"));
        launch_k(loss_cos_rows_kernel, loss_cos_blocks, 256, 0, st, emb, ref, rowstat, loss_cos_partial, R, 512);
        PTTA_TRY(check_launch("loss_cos_rows"));
        launch_k(loss_finalize_kernel, 1, 256, 0, st, loss_map_partial, loss_map_blocks, loss_cos_partial, loss_cos_blocks, Nu, Hu, Wu, R, w_sd, w_sm,
                                              w_cos, 0.3f, losses);
        return check_launch("loss_finalize");
    }

    // ---- backward -----------------------------------------------------------------------------------------
    float* grad_of(const std::string& key) {
        auto it = ext.find("grad/" + key);
        return it == ext.end() ? nullptr : (float*)it->second.first;
    }
    // prediction layers of a decoder: gs0 = [add +] dgrad(prdct.1)(dgrad(prdct.3)(gout) * [h>0]) * [s0>0]
    int dec_pred_backward(const DecW& Wt, const DecAct& A, const Map1& gout, const Map32& tmp, const Map32& gs0, const bf16* add) {
        PTTA_TRY(head_dgrad(Wt.p3, gout, A.h, tmp));
        return conv_dgrad(Wt.p1, tmp, gs0, A.s0.p, add);
    }
    // d loss / d output (g_out) and d loss / d ref (g_ref)
    int loss_backward(float gscale) {
        PTTA_CHECK(l_img != nullptr, "backward called before loss");
        const Branch& B = real;
        {
            long long tot = (long long)Nu * Hu * Wu;
            launch_k(loss_map_grad_kernel, cdiv(tot, 256), 256, 0, st, padded ? out_u.p : B.output.p, l_d, l_v, l_img, padded ? g_out_u.p : g_out.p, losses,
                                                               Nu, Hu, Wu, l_cap, l_cap > 0.f ? 1 : 0, l_wsd, l_wsm, gscale);
            PTTA_TRY(check_launch("loss_map_grad"));
            launch_k(loss_cos_grad_kernel, loss_cos_blocks, 256, 0, st, emb, ref, rowstat, losses, g_ref, R, 512, gscale, 0);
            PTTA_TRY(check_launch("loss_cos_grad"));
        }
        return 0;
    }
    // from (g_out, g_ref) to the gradients of the adapted tensors
    int network_backward() {
        PTTA_CHECK(!train_head, "network_backward: this engine trains the predictor head (option trainable_head); use head_backward");
        for (const std::string& k : adapt_names) PTTA_CHECK(grad_of(k) != nullptr, "gradient buffer 'grad/%s' not bound", k.c_str());
        const Branch& B = real;
        if (padded) {   // adjoint of the crop + mean: each copy receives half of the gradient at its crop, zero elsewhere
            long long tot = (long long)N * H * W;
            launch_k(pad_pair_kernel, cdiv(tot, 256), 256, 0, st, g_out_u.p, g_out.p, Nu, 1, Hu, Wu, H, W, 0.5f, 0.f, 0.f, 0.f);
            PTTA_TRY(check_launch("pad_pair(g_output)"));
        }
        // proxy head on the real rows: ref = L3(relu(bn(L0(z)))).  Its data gradient g_z joins the decoder-3 chain only at "G4b = GC2 + g_z":
        // with the side streams available it runs on st3 beside the full-resolution data gradients of decoder 3.
        const bool side = two_streams && st3 != nullptr;
        {
            cudaStream_t main = st; double* main_partial = partial;
            if (side) {
                PTTA_CUDA(cudaEventRecord(ev_lossg, st));
                PTTA_CUDA(cudaStreamWaitEvent(st3, ev_lossg, 0));
                st = st3; partial = partial3;
            }
            int rc3 = 0;
            if (!proxy_in_backward) {      // stage 1 (supervised): nothing arrives through ref = proj(z_real)
                if (cudaMemsetAsync(GZ.p, 0, GZ.numel() * sizeof(bf16), st) != cudaSuccess) { set_error("cudaMemsetAsync(g_z) failed"); rc3 = 2; }
            } else {
                rc3 = gemm(g_ref, proj3.pack_t, g_a3, nullptr, R, 512, 512);
                if (!rc3) rc3 = bn_backward(projBn, bnProjR, g_a3, h_a0r, g_a0, R, 1, nullptr, nullptr);
                if (!rc3) rc3 = gemm(g_a0, proj0.pack_t, GZ.p, nullptr, R, 32, 512);     // g_z (grad wrt e3.x2 from the heads)
            }
            if (side && !rc3 && cudaEventRecord(ev_headb, st3) != cudaSuccess) { set_error("cudaEventRecord failed"); rc3 = 2; }
            st = main; partial = main_partial;
            if (rc3) return rc3;
        }

        // ---- decoder 3 ----
        PTTA_TRY(dec_pred_backward(dec3W, B.d3, g_out, T1a, T1b, nullptr));                 // T1b = g_s0 (= g_x4 = g_e3x0)
        PTTA_TRY(conv_dgrad(dec3W.d1b, T1b, T1a, B.d3.u1.p, nullptr));                      // T1a = g_u1
        PTTA_TRY(conv_dgrad(dec3W.d1a, T1a, T2a, B.d3.s1.p, nullptr));                      // T2a = g_s1 (= g_e3x1 = g_x3)
        PTTA_TRY(conv_dgrad(dec3W.d2b, T2a, T2b, B.d3.u2.p, nullptr));                      // T2b = g_u2
        PTTA_TRY(conv_dgrad(dec3W.d2a, T2b, GC2, B.d3.x2.p, nullptr));                      // GC2 = grad of d3.x2 (meta contribution #1)
        if (side) PTTA_CUDA(cudaStreamWaitEvent(st, ev_headb, 0));
        PTTA_TRY(add32(GC2, GZ, G4b));                                                      // G4b = g_e3x2 = GC2 + g_z
        // ---- encoder 3 ----
        PTTA_TRY(up2_adj32(G4b, D8, 0));                                                    // D8 = grad of d2.x2 (skip)
        PTTA_TRY(conv_dgrad(enc3W.e2b, G4b, G4a, B.e3.t2.p, nullptr));                      // G4a = g_t2
        PTTA_TRY(conv_dgrad(enc3W.e2a, G4a, T2b, B.e3.x1r.p, T2a.p));                        // T2b = g_x1 total
        PTTA_TRY(up2_adj32(T2b, D4, 0));                                                    // D4 = grad of d2.x3 (skip)
        PTTA_TRY(conv_dgrad(enc3W.e1b, T2b, T2a, B.e3.t1.p, nullptr));                      // T2a = g_t1
        PTTA_TRY(conv_dgrad(enc3W.e1a, T2a, T1a, B.e3.x0r.p, T1b.p));                        // T1a = g_x0 total
        PTTA_TRY(up2_adj32(T1a, D2, 0));                                                    // D2 = grad of d2.x4 (skip)
        PTTA_TRY(conv_dgrad(enc3W.init2, T1a, T1b, B.e3.a0.p, nullptr));                    // T1b = g_a0
        PTTA_TRY(stem_dgrad_ch1(enc3W.init0, T1b, g_out.p, g_p11));                         // g_p11 = g_output + stem grad
        PTTA_TRY(up2_adj1(g_p11, g_q));                                                     // g_q = g_out12 = g_p12 (part)
        // ---- decoder 2 ----
        PTTA_TRY(dec_pred_backward(dec2W, B.d2, g_q, T2a, T2b, nullptr));                   // T2b = g_s0 (= g_e2x0)
        PTTA_TRY(add32(D2, T2b, T2a));                                                      // T2a = g_x4 total
        PTTA_TRY(conv_dgrad(dec2W.d1b, T2a, D2, B.d2.u1.p, nullptr));                       // D2 = g_u1
        PTTA_TRY(conv_dgrad(dec2W.d1a, D2, G4a, B.d2.s1.p, nullptr));                       // G4a = g_s1 (= g_e2x1; meta contribution #2)
        PTTA_TRY(add32(GC2, G4a, GC2));
        PTTA_TRY(add32(D4, G4a, D4));                                                       // D4 = g_x3 total
        PTTA_TRY(conv_dgrad(dec2W.d2b, D4, G4b, B.d2.u2.p, nullptr));                       // G4b = g_u2
        PTTA_TRY(conv_dgrad(dec2W.d2a, G4b, E8, B.d2.x2.p, D8.p));                          // E8 = g_e2x2
        // ---- encoder 2 ----
        PTTA_TRY(conv_dgrad(enc2W.e2b, E8, D8, B.e2.t2.p, nullptr));                        // D8 = g_t2
        PTTA_TRY(conv_dgrad(enc2W.e2a, D8, G4b, B.e2.x1r.p, G4a.p));                         // G4b = g_x1 total
        PTTA_TRY(conv_dgrad(enc2W.e1b, G4b, D4, B.e2.t1.p, nullptr));                       // D4 = g_t1
        PTTA_TRY(conv_dgrad(enc2W.e1a, D4, T2a, B.e2.x0r.p, T2b.p));                         // T2a = g_x0 total
        PTTA_TRY(conv_dgrad(enc2W.init2, T2a, D2, B.e2.a0.p, nullptr));                     // D2 = g_a0
        PTTA_TRY(stem_dgrad_ch1(enc2W.init0, D2, g_q.p, g_p12));                            // g_p12 = g_q + stem grad
        PTTA_TRY(up2_adj1(g_p12, g_o14));                                                   // g_out14
        // ---- decoder 1 (prediction layers only) ----
        PTTA_TRY(dec_pred_backward(dec1W, B.d1, g_o14, G4a, GC2, GC2.p));                   // GC2 += g_s0 (meta contribution #3)

        // ---- meta layer ----
        const long long rows = (long long)N * (H / 4) * (W / 4);
        if (!two_layers) {
            WgradParams wp; memset(&wp, 0, sizeof(wp));
            wp.in = B.c2raw.p; wp.gout = GC2.p; wp.partial = wgrad_ws; wp.N = N; wp.H = H / 4; wp.W = W / 4; wp.pro = PRO_NONE;
            PTTA_TRY(launch_wgrad(wp, grad_of("conv1_rgb_meta.weight"), 32, 32, st));
            int nblk = 0;
            PTTA_TRY(stats(GC2.p, nullptr, rows, 32, 0, nullptr, 0, nblk));
            launch_k(colsum_finalize_kernel, 1, FIN_THREADS, 0, st, partial, nblk, 32, grad_of("conv1_rgb_meta.bias"));
            return check_launch("colsum_finalize");
        }
        const std::string p = "conv1_rgb_meta.conv1_meta";
        // BN2: c2 = bn2(mg) + c2raw
        PTTA_TRY(bn_backward(metaBn2, B.bn2, GC2.p, B.mg.p, G4a.p, rows, 0, grad_of(p + ".2.weight"), grad_of(p + ".2.bias")));   // G4a = g_mg
        {   // conv2's bias and weight gradients need g_mg only: on st3, beside the data gradient of conv2 and everything upstream of it
            cudaStream_t main = st; double* main_partial = partial; float* main_ws = wgrad_ws;
            if (side) {
                PTTA_CUDA(cudaEventRecord(ev_gmg, st));
                PTTA_CUDA(cudaStreamWaitEvent(st3, ev_gmg, 0));
                st = st3; partial = partial3; wgrad_ws = wgrad_ws2;
            }
            int nblk = 0;
            int rc3 = stats(G4a.p, nullptr, rows, 32, 0, nullptr, 0, nblk);
            if (!rc3) {
                launch_k(colsum_finalize_kernel, 1, FIN_THREADS, 0, st, partial, nblk, 32, grad_of(p + ".1.bias"));
                rc3 = check_launch("colsum_finalize");
            }
            if (!rc3) {   // conv2 wgrad: input = leaky(bn1(mh))
                WgradParams wp; memset(&wp, 0, sizeof(wp));
                wp.in = B.mh.p; wp.gout = G4a.p; wp.partial = wgrad_ws; wp.N = N; wp.H = H / 4; wp.W = W / 4;
                wp.pro = PRO_BN_LEAKY; wp.pro_scale = B.bn1.scale; wp.pro_shift = B.bn1.shift; wp.slope = 0.2f;
                rc3 = launch_wgrad(wp, grad_of(p + ".1.weight"), 128, 32, st);
            }
            if (side && !rc3 && cudaEventRecord(ev_wg2, st3) != cudaSuccess) { set_error("cudaEventRecord failed"); rc3 = 2; }
            st = main; partial = main_partial; wgrad_ws = main_ws;
            if (rc3) return rc3;
        }
        PTTA_TRY(conv_dgrad(meta2, G4a, M128a, B.mh.p, nullptr, MASK_BN_LEAKY, &B.bn1));    // M128a = grad wrt bn1 output
        PTTA_TRY(bn_backward(metaBn1, B.bn1, M128a.p, B.mh.p, M128b.p, rows, 0, grad_of(p + ".0.1.weight"), grad_of(p + ".0.1.bias")));
        {   // conv1 wgrad: input = c2raw
            WgradParams wp; memset(&wp, 0, sizeof(wp));
            wp.in = B.c2raw.p; wp.gout = M128b.p; wp.partial = wgrad_ws; wp.N = N; wp.H = H / 4; wp.W = W / 4; wp.pro = PRO_NONE;
            PTTA_TRY(launch_wgrad(wp, grad_of(p + ".0.0.weight"), 32, 128, st));
        }
        if (side) PTTA_CUDA(cudaStreamWaitEvent(st, ev_wg2, 0));
        return 0;
    }

    int backward(float gscale) {
        PTTA_TRY(loss_backward(gscale));
        return network_backward();
    }

    // ---- source-domain preparation (SURVEY section 8 f3) -------------------------------------------------------
    // stage 1 loss (src/init_main.py:510-517 -> src/msg_chn_model_adapt.py:224-264 -> src/loss_utils.py:266-287): ground truth clamped to
    // [0, max_predict_depth], v = [gt > 0], loss = mean_n( sum v (pred - gt)^2 / sum v )
    int l2_loss(const float* gt, float max_predict) {
        PTTA_CHECK(Nu <= 64, "l2_loss: batch size %d > 64 not supported", Nu);
        PTTA_CHECK(!padded, "stage-1 / stage-2 training needs H and W that are multiples of 16 (the reference pads in 'adapt' mode only: "
                            "src/msg_chn_model_adapt.py:54-55)");
        l_gt = gt; l_maxd = max_predict;
        dim3 grid(loss_map_blocks, Nu);
        launch_k(l2_loss_reduce_kernel, grid, LOSS_BLOCK, 0, st, real.output.p, gt, loss_map_partial, Hu * Wu, max_predict);
        PTTA_TRY(check_launch("l2_loss_reduce"));
        launch_k(l2_loss_finalize_kernel, 1, 256, 0, st, loss_map_partial, loss_map_blocks, Nu, losses);
        return check_launch("l2_loss_finalize");
    }
    int l2_loss_backward(float gscale) {
        PTTA_CHECK(l_gt != nullptr, "l2_loss_backward called before l2_loss");
        const long long tot = (long long)Nu * Hu * Wu;
        launch_k(l2_loss_grad_kernel, cdiv(tot, 256), 256, 0, st, real.output.p, l_gt, g_out.p, losses, Nu, Hu * Wu, l_maxd, gscale);
        return check_launch("l2_loss_grad");
    }
    // one supervised step on the meta layer: forward without the proxy branch, L2 loss, backward, Adam (src/init_main.py:482-522)
    int init_step(const float* image_raw, const float* isc, const float* ish, const float* sparse, const float* gt, float cap, float max_predict) {
        PTTA_CHECK(!train_head, "init_step: this engine trains the predictor head (option trainable_head)");
        PTTA_TRY(forward(image_raw, isc, ish, sparse, cap, 2));
        PTTA_TRY(l2_loss(gt, max_predict));
        PTTA_TRY(l2_loss_backward(1.f));
        PTTA_TRY(network_backward());
        return adam_step();
    }

    // stage 2 loss (src/head_main.py:469-475 -> src/external_model_adapt.py:524-540): mean_r(2 - 2 cos(emb_r, ref_r)), no gate
    int cos_loss() {
        launch_k(loss_cos_rows_kernel, loss_cos_blocks, 256, 0, st, emb, ref, rowstat, loss_cos_partial, R, 512);
        PTTA_TRY(check_launch("loss_cos_rows"));
        launch_k(cos_loss_finalize_kernel, 1, 256, 0, st, loss_cos_partial, loss_cos_blocks, R, losses);
        return check_launch("cos_loss_finalize");
    }
    // proj_t <- tau proj_t + (1 - tau) proj over the PARAMETERS of proj (network_exp_msg_chn_adapt.py:701-703, called once per stage-2
    // forward at :689); skipped when the checkpoint has no EMA copy
    int ema_update_head(double tau) {     // tau as the reference's Python float: 1 - tau is formed in double, then both factors are rounded to fp32
        static const char* names[6] = {"0.weight", "0.bias", "1.weight", "1.bias", "3.weight", "3.bias"};
        EmaParams ep; memset(&ep, 0, sizeof(ep));
        long long maxn = 0;
        for (int i = 0; i < 6; ++i) {
            auto t = ext.find(std::string("proj_t.") + names[i]);
            auto sidx = ext.find(std::string("proj.") + names[i]);
            if (t == ext.end()) continue;
            PTTA_CHECK(sidx != ext.end() && sidx->second.second == t->second.second, "ema_update: proj.%s / proj_t.%s mismatch", names[i], names[i]);
            ep.t[ep.count] = (float*)t->second.first; ep.s[ep.count] = (const float*)sidx->second.first; ep.n[ep.count] = t->second.second;
            maxn = std::max(maxn, t->second.second);
            ++ep.count;
        }
        if (!ep.count) return 0;
        ep.tau = (float)tau; ep.one_minus_tau = (float)(1.0 - tau);
        launch_k(ema_update_kernel, dim3(cdiv(maxn, 256), ep.count), 256, 0, st, ep);
        return check_launch("ema_update");
    }
    // gradients of pred.{0,1,3}: emb = pred(proj(z_zero).detach()) (network_exp_msg_chn_adapt.py:692)
    //   emb = a1 W3^T + b3,  a1 = relu(bn(q0)),  q0 = pz W0^T + b0,  pz = proj(z_zero)
    // d loss / d emb of the stage-2 loss into "g_emb"
    int cos_loss_backward(float gscale) {
        launch_k(loss_cos_grad_kernel, loss_cos_blocks, 256, 0, st, emb, ref, rowstat, losses, g_a3, R, 512, gscale, 1);
        return check_launch("loss_cos_grad(emb)");
    }
    int head_backward() {
        PTTA_CHECK(train_head, "head_backward: engine was not created with option trainable_head");
        for (const std::string& k : adapt_names) PTTA_CHECK(grad_of(k) != nullptr, "gradient buffer 'grad/%s' not bound", k.c_str());
        bf16* g_emb = g_a3; bf16* g_a1 = g_a0;
        int nblk = 0;
        // pred.3
        PTTA_TRY(launch_gemm_tn_tc(g_emb, h_an2, grad_of("pred.3.weight"), gw_part, R, 512, 512, st));
        PTTA_TRY(stats(g_emb, nullptr, R, 512, 0, nullptr, 0, nblk));
        launch_k(colsum_finalize_kernel, cdiv(512, 32), FIN_THREADS, 0, st, partial, nblk, 512, grad_of("pred.3.bias"));
        PTTA_TRY(check_launch("colsum_finalize"));
        PTTA_TRY(gemm(g_emb, pred3.pack_t, g_a1, nullptr, R, 512, 512));
        // pred.1 (BatchNorm1d, train mode) behind the ReLU
        PTTA_TRY(bn_backward(predBn, bnPred, g_a1, h_q0, g_q0, R, 1, grad_of("pred.1.weight"), grad_of("pred.1.bias")));
        // pred.0
        PTTA_TRY(launch_gemm_tn_tc(g_q0, h_pz, grad_of("pred.0.weight"), gw_part, R, 512, 512, st));
        PTTA_TRY(stats(g_q0, nullptr, R, 512, 0, nullptr, 0, nblk));
        launch_k(colsum_finalize_kernel, cdiv(512, 32), FIN_THREADS, 0, st, partial, nblk, 512, grad_of("pred.0.bias"));
        return check_launch("colsum_finalize");
    }
    // one stage-2 step (src/head_main.py:437-480): frozen network on the frame and on the zero image, EMA copy of proj, cosine loss
    // between pred(proj(z_zero)) and proj(z_real), gradients of pred, Adam
    int head_step(const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap) {
        PTTA_CHECK(train_head, "head_step: engine was not created with option trainable_head");
        PTTA_CHECK(!padded, "stage-2 training needs H and W that are multiples of 16");
        PTTA_TRY(forward(image_raw, isc, ish, sparse, cap, 1));
        PTTA_TRY(ema_update_head(0.999));
        PTTA_TRY(cos_loss());
        PTTA_TRY(cos_loss_backward(1.f));
        PTTA_TRY(head_backward());
        return adam_step();
    }

    // captured stage-1 / stage-2 steps (same scheme as ptta_msgchn_tta_step_graph: inputs staged into engine-owned buffers, one eager step to
    // set the function attributes and validate, then capture-without-execute and replay)
    template <class Body>
    int prep_step_graphed(const GraphKey& key, cudaStream_t stream_, Body body) {
        ptta_msgchn* e = this; cudaStream_t st = stream_;
        if (e->prep_graph_exec && memcmp(&key, &e->prep_graph_key, sizeof(key)) != 0) { cudaGraphExecDestroy(e->prep_graph_exec); e->prep_graph_exec = nullptr; }
        if (!e->prep_graph_exec) {
            e->st = st;
            PTTA_TRY(body());
            PTTA_CUDA(cudaStreamSynchronize(st));
            cudaGraph_t graph = nullptr;
            PTTA_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            int rc = body();
            cudaError_t ce = cudaStreamEndCapture(st, &graph);
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            PTTA_CHECK(ce == cudaSuccess, "graph capture failed: %s", cudaGetErrorString(ce));
            ce = cudaGraphInstantiate(&e->prep_graph_exec, graph, 0);
            cudaGraphDestroy(graph);
            PTTA_CHECK(ce == cudaSuccess, "graph instantiate failed: %s", cudaGetErrorString(ce));
            memcpy(&e->prep_graph_key, &key, sizeof(key));
            return 0;   // the eager step above WAS this call's step
        }
        PTTA_CUDA(cudaGraphLaunch(e->prep_graph_exec, st));
        return 0;
    }


    int adam_step() {
        PTTA_CHECK(n_adam_chunks > 0, "Adam state not bound (grad/, adam_m/, adam_v/ entries for every adapted tensor)");
        if (comm.world > 1) {
            // shared model: one-shot mean all-reduce of the flat gradient buffer fused with the Adam update (identical on every rank)
            const int xid = take_xid();
            if (xid < 0) return 1;
            const float* g_base = nullptr;      // lowest gradient pointer of the chunk table = start of the flat buffer the chunks index into
            PTTA_CHECK(adam_g_base != nullptr && adam_g_floats <= comm.grad_floats, "shared-model mode: gradient buffer (%zu floats) exceeds the communicator's slot (%zu)",
                       adam_g_floats, comm.grad_floats);
            g_base = adam_g_base;
            launch_k(adam_allreduce_kernel, n_adam_chunks, 256, 0, st, adam_chunks, adam_hyper, comm, xid, g_base);
            PTTA_TRY(check_launch("adam_allreduce"));
            launch_k(adam_advance_kernel, 1, 1, 0, st, adam_hyper);
            PTTA_TRY(check_launch("adam_advance"));
            launch_k(comm_advance_kernel, 1, 32, 0, st, comm);
            PTTA_TRY(check_launch("comm_advance"));
            return pack_adapted();
        }
        launch_k(adam_kernel, n_adam_chunks, 256, 0, st, adam_chunks, adam_hyper);
        PTTA_TRY(check_launch("adam"));
        launch_k(adam_advance_kernel, 1, 1, 0, st, adam_hyper);
        PTTA_TRY(check_launch("adam_advance"));
        return pack_adapted();
    }

    int outlier(const float* sparse) {
        dim3 grid(cdiv(Wu, OR_TX), cdiv(Hu, OR_TY), Nu), block(OR_TX, OR_TY);
        size_t sm = (size_t)(OR_TX + 6) * (OR_TY + 6) * sizeof(float);
        launch_k(outlier_removal_kernel, grid, block, sm, st, sparse, fd.p, fv.p, Hu, Wu, 7, 1.5f);
        return check_launch("outlier_removal");
    }

    int tta_step(const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap, float w_sd, float w_sm,
                 float w_cos) {
        PTTA_TRY(outlier(sparse));                                               // src/tta_main.py:583-590
        PTTA_TRY(forward(image_raw, isc, ish, fd.p, cap, 1));                    // :610-614
        PTTA_TRY(loss(image_raw, fd.p, fv.p, cap, w_sd, w_sm, w_cos));           // :619-629
        PTTA_TRY(backward(1.f));                                                 // :631-632
        return adam_step();                                                      // :633
    }
};

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* ptta_last_error(void) { return g_error.c_str(); }
int ptta_version(void) { return 100; }

int ptta_outlier_removal(const float* d, float* d_out, float* v_out, int n, int h, int w, int ksize, float thr, ptta_stream_t stream) {
    PTTA_CHECK(ksize >= 1 && ksize <= 15 && (ksize & 1), "outlier_removal: kernel_size %d must be odd and <= 15", ksize);
    int pad = ksize / 2;
    dim3 grid(cdiv(w, OR_TX), cdiv(h, OR_TY), n), block(OR_TX, OR_TY);
    size_t sm = (size_t)(OR_TX + 2 * pad) * (OR_TY + 2 * pad) * sizeof(float);
    launch_k(outlier_removal_kernel, grid, block, sm, (cudaStream_t)stream, d, d_out, v_out, h, w, ksize, thr);
    return check_launch("outlier_removal");
}

int ptta_pyramid(const float* d, float* dc, float* d2, float* d4, int n, int h, int w, float cap, int do_clamp, ptta_stream_t stream) {
    PTTA_CHECK(h % 4 == 0 && w % 4 == 0, "pyramid: %dx%d must be multiples of 4", h, w);
    long long tot = (long long)n * (h / 4) * (w / 4);
    launch_k(pyramid_kernel, cdiv(tot, 128), 128, 0, (cudaStream_t)stream, d, dc, d2, d4, n, h, w, cap, do_clamp);
    return check_launch("pyramid");
}

int ptta_pack_conv_weight(const float* src, void* dst, int o, int i, int s_o, int s_i, int flip, ptta_stream_t stream) {
    launch_k(pack_conv_weight_kernel, cdiv(9 * o * i, 256), 256, 0, (cudaStream_t)stream, src, (bf16*)dst, o, i, s_o, s_i, flip);
    return check_launch("pack_conv_weight");
}

int ptta_conv3x3(const void* in, void* out, const void* wpack, const float* bias, int n, int hin, int win, int cin, int cout, int mode,
                 int prologue, const float* pro_scale, const float* pro_shift, float slope, const void* mask, int mask_mode,
                 const float* mask_scale, const float* mask_shift, const void* add, ptta_stream_t stream) {
    ConvParams p; memset(&p, 0, sizeof(p));
    p.in = (const bf16*)in; p.out = (bf16*)out; p.w = (const bf16*)wpack; p.bias = bias;
    p.N = n; p.Hin = hin; p.Win = win; p.pro = prologue; p.pro_scale = pro_scale; p.pro_shift = pro_shift; p.slope = slope;
    p.mask = (const bf16*)mask; p.mask_mode = mask ? mask_mode : MASK_NONE; p.mask_scale = mask_scale; p.mask_shift = mask_shift;
    p.add = (const bf16*)add;
    PTTA_CHECK(prologue != PRO_BN_LEAKY || (pro_scale && pro_shift), "conv3x3: BN prologue needs scale and shift");
    PTTA_CHECK(p.mask_mode != MASK_BN_LEAKY || (mask_scale && mask_shift), "conv3x3: BN mask needs scale and shift");
    return launch_conv3x3(p, cin, cout, mode, (cudaStream_t)stream);
}

int ptta_conv3x3_tc(const void* in, void* out, const void* wimage, const float* bias, int n, int h, int w, int relu_in, int relu_out,
                    const void* mask, const void* add, ptta_stream_t stream) {
    PTTA_CHECK(in && out && wimage, "conv3x3_tc: null argument");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.bias = bias; p.out = (bf16*)out; p.mask = (const bf16*)mask; p.add = (const bf16*)add;
    p.N = n; p.H = h; p.W = w; p.relu_in = relu_in; p.relu_out = relu_out;
    return launch_conv_tc((const bf16*)in, p, (cudaStream_t)stream);
}

int ptta_conv3x3_tc_ex(const void* in, void* out, void* out2, const void* wimage, const float* bias, int n, int h, int w, int relu_out,
                       const void* mask, const void* add, const void* add2, ptta_stream_t stream) {
    PTTA_CHECK(in && out && wimage, "conv3x3_tc_ex: null argument");
    PTTA_CHECK(!(add && add2), "conv3x3_tc_ex: add and add2 are mutually exclusive");
    PTTA_CHECK(!add2 || out2, "conv3x3_tc_ex: add2 needs out2");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.bias = bias; p.out = (bf16*)out; p.out2 = (bf16*)out2; p.mask = (const bf16*)mask; p.add = (const bf16*)add;
    p.add2 = (const bf16*)add2; p.N = n; p.H = h; p.W = w; p.relu_out = relu_out;
    return launch_conv_tc((const bf16*)in, p, (cudaStream_t)stream);
}

int ptta_conv3x3_tc_up2(const void* in, void* out, void* out_relu, const void* wimage, const float* bias, const void* half, int n, int h, int w,
                        ptta_stream_t stream) {
    PTTA_CHECK(in && out && wimage && half, "conv3x3_tc_up2: null argument");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.bias = bias; p.out = (bf16*)out; p.out2 = (bf16*)out_relu; p.up2 = (const bf16*)half; p.N = n; p.H = h; p.W = w;
    return launch_conv_tc((const bf16*)in, p, (cudaStream_t)stream);
}

int ptta_pack_conv_weight_tc(const void* wpack, void* image, ptta_stream_t stream) {
    PTTA_CHECK(wpack && image, "pack_conv_weight_tc: null argument");
    launch_k(pack_conv_weight_tc_kernel, cdiv(9 * 32 * 4, 256), 256, 0, (cudaStream_t)stream, (const bf16*)wpack, (bf16*)image);
    return check_launch("pack_conv_weight_tc");
}

int ptta_pack_conv_weight_tc_t2(const void* wpack, void* image, ptta_stream_t stream) {
    PTTA_CHECK(wpack && image, "pack_conv_weight_tc_t2: null argument");
    launch_k(pack_conv_weight_tc_t2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, (cudaStream_t)stream, (const bf16*)wpack, (bf16*)image);
    return check_launch("pack_conv_weight_tc_t2");
}
int ptta_conv3x3_tc_t2(const void* in, void* out, const void* wimage, const float* bias, int n, int h, int w, int relu_out, const void* mask,
                       const void* add, ptta_stream_t stream) {
    PTTA_CHECK(in && out && wimage, "conv3x3_tc_t2: null argument");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.bias = bias; p.out = (bf16*)out; p.mask = (const bf16*)mask; p.add = (const bf16*)add;
    p.N = n; p.H = h; p.W = w; p.relu_out = relu_out;
    return launch_conv_tc_t2((const bf16*)in, p, (cudaStream_t)stream);
}

int ptta_pack_conv_weight_tc_s2(const void* wpack, void* image, ptta_stream_t stream) {
    PTTA_CHECK(wpack && image, "pack_conv_weight_tc_s2: null argument");
    launch_k(pack_conv_weight_tc_s2_kernel, cdiv(9 * 32 * 4, 256), 256, 0, (cudaStream_t)stream, (const bf16*)wpack, (bf16*)image);
    return check_launch("pack_conv_weight_tc_s2");
}
int ptta_conv3x3_tc_s2(const void* in, void* out, void* out_relu, const void* wimage, const float* bias, int n, int h, int w, int relu_out,
                       const void* mask, const void* add, ptta_stream_t stream) {
    PTTA_CHECK(in && out && wimage, "conv3x3_tc_s2: null argument");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.bias = bias; p.out = (bf16*)out; p.out2 = (bf16*)out_relu; p.mask = (const bf16*)mask; p.add = (const bf16*)add;
    p.N = n; p.H = h; p.W = w; p.relu_out = relu_out;
    return launch_conv_tc_s2((const bf16*)in, p, (cudaStream_t)stream);
}

#ifdef PTTA_STAMPS
extern "C" int ptta_stamps_reset(void) {
    unsigned int z = 0;
    PTTA_CUDA(cudaMemcpyToSymbol(g_stamp_count, &z, sizeof(z)));
    return 0;
}
extern "C" int ptta_stamps_read(unsigned long long* out, int capacity) {
    unsigned int n = 0;
    PTTA_CUDA(cudaMemcpyFromSymbol(&n, g_stamp_count, sizeof(n)));
    if ((int)n > capacity) n = capacity;
    if (n > 8192u) n = 8192u;
    PTTA_CUDA(cudaMemcpyFromSymbol(out, g_stamps, sizeof(unsigned long long) * n));
    return (int)n + 1000000;      // count + 1e6 (so that 0 stays "ok" for the usual status convention)
}
#endif

size_t ptta_conv3x3_wgrad_workspace_bytes(int n, int h, int w, int cin, int cout) { return wgrad_partial_bytes(n, h, w, cin, cout); }

int ptta_conv3x3_wgrad(const void* in, const void* gout, float* dw, void* workspace, int n, int h, int w, int cin, int cout, int prologue,
                       const float* pro_scale, const float* pro_shift, float slope, ptta_stream_t stream) {
    WgradParams p; memset(&p, 0, sizeof(p));
    p.in = (const bf16*)in; p.gout = (const bf16*)gout; p.partial = (float*)workspace; p.N = n; p.H = h; p.W = w;
    p.pro = prologue; p.pro_scale = pro_scale; p.pro_shift = pro_shift; p.slope = slope;
    return launch_wgrad(p, dw, cin, cout, (cudaStream_t)stream);
}

int ptta_stem_conv(const float* const* planes, const long long* strides, const float* scale, const float* shift, int cin,
                   const float* weight, const float* bias, const void* mask, void* out, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(cin >= 1 && cin <= 3, "stem_conv: cin=%d", cin);
    StemParams p; memset(&p, 0, sizeof(p));
    for (int k = 0; k < 3; ++k) {
        int s = k < cin ? k : 0;
        p.plane[k] = planes[s]; p.batch_stride[k] = strides[s]; p.scale[k] = scale[s]; p.shift[k] = shift[s];
    }
    p.w = weight; p.bias = bias; p.mask = (const bf16*)mask; p.out = (bf16*)out; p.N = n; p.H = h; p.W = w;
    launch_stem(p, cin, (cudaStream_t)stream);
    return check_launch("stem_conv");
}

int ptta_stem_conv_const(const float* const* planes, const long long* strides, const float* scale, const float* shift, int cin,
                         const float* weight_host, const float* bias_host, const void* mask, void* out, int relu_out, int n, int h, int w,
                         ptta_stream_t stream) {
    PTTA_CHECK(cin >= 1 && cin <= 3 && (w & 1) == 0, "stem_conv_const: cin=%d (1..3), W=%d (even)", cin, w);
    PTTA_CHECK(weight_host && out, "stem_conv_const: null argument");
    StemCParams c; memset(&c, 0, sizeof(c));
    for (int k = 0; k < 3; ++k) {
        int s = k < cin ? k : 0;
        c.plane[k] = planes[s]; c.batch_stride[k] = strides[s]; c.scale[k] = scale[s]; c.shift[k] = shift[s];
    }
    for (int co = 0; co < 32; ++co)
        for (int r = 0; r < cin * 9; ++r) c.w[r * 32 + co] = weight_host[(size_t)co * cin * 9 + r];
    if (bias_host) memcpy(c.bias, bias_host, sizeof(c.bias));
    c.mask = (const bf16*)mask; c.out = (bf16*)out; c.N = n; c.H = h; c.W = w; c.relu_out = relu_out;
    launch_stem_const(c, cin, (cudaStream_t)stream);
    return check_launch("stem_conv_const");
}

int ptta_head_conv(const void* in, const float* w, float bias, const float* add, float* out, int n, int h, int ww, int relu_in,
                   int accumulate, ptta_stream_t stream) {
    long long tot = (long long)n * h * ww;
    launch_k(head_conv_kernel, dim3(cdiv(ww, HEADC_TW), cdiv(h, HEADC_TH), n), dim3(HEADC_TW, HEADC_TH), 0, (cudaStream_t)stream, (const bf16*)in, w, bias, add, out, n, h, ww, relu_in, accumulate);
    return check_launch("head_conv");
}

int ptta_head_conv_const(const void* in, const float* weight_host_9x32, float bias, const float* add, float* out, int n, int h, int ww,
                         int relu_in, int accumulate, ptta_stream_t stream) {
    PTTA_CHECK(in && weight_host_9x32 && out, "head_conv_const: null argument");
    HeadCParams c; memset(&c, 0, sizeof(c));
    c.in = (const bf16*)in; c.add = add; c.out = out; c.N = n; c.H = h; c.W = ww; c.relu_in = relu_in; c.accumulate = accumulate; c.bias = bias;
    memcpy(c.w, weight_host_9x32, sizeof(c.w));
    launch_k(head_convc_kernel, dim3(cdiv(ww, HEADC_TW), cdiv(h, HEADC_TH), n), dim3(HEADC_TW, HEADC_TH), 0, (cudaStream_t)stream, c);
    return check_launch("head_conv_const");
}

int ptta_stem_conv_tc(const float* const* planes, const long long* strides, const float* scale, const float* shift, int cin,
                      const float* weight, const float* bias, const void* mask, void* out, void* image_scratch, int relu_out, int n, int h, int w,
                      ptta_stream_t stream) {
    PTTA_CHECK(cin >= 1 && cin <= 3 && planes && out && image_scratch, "stem_conv_tc: bad arguments");
    if (weight) {                        // null: image_scratch already holds the packed weights of an earlier call
        launch_k(pack_stem_weight_tc_kernel, 1, 256, 0, (cudaStream_t)stream, weight, (bf16*)image_scratch, cin);
        PTTA_TRY(check_launch("pack_stem_tc"));
    }
    StemTcParams t; memset(&t, 0, sizeof(t));
    for (int k = 0; k < 3; ++k) {
        const int s = k < cin ? k : 0;
        t.plane[k] = planes[s]; t.batch_stride[k] = strides[s]; t.scale[k] = scale ? scale[s] : 1.f; t.shift[k] = shift ? shift[s] : 0.f;
    }
    t.w = (const bf16*)image_scratch; t.bias = bias; t.mask = (const bf16*)mask; t.out = (bf16*)out; t.N = n; t.H = h; t.W = w; t.relu_out = relu_out;
    return launch_stem_tc(t, cin, (cudaStream_t)stream);
}

int ptta_pack_head_weight_tc(const float* weight_9x32, void* image, ptta_stream_t stream) {
    PTTA_CHECK(weight_9x32 && image, "pack_head_weight_tc: null argument");
    launch_k(pack_conv_weight_tc_head_kernel, cdiv(9 * 16 * 4, 256), 256, 0, (cudaStream_t)stream, weight_9x32, (bf16*)image);
    return check_launch("pack_head_weight_tc");
}

int ptta_head_conv_tc(const void* in, const void* wimage, float bias, const float* add, float* out, int n, int h, int ww, ptta_stream_t stream) {
    PTTA_CHECK(in && wimage && out, "head_conv_tc: null argument");
    ConvTcParams p; memset(&p, 0, sizeof(p));
    p.w = (const bf16*)wimage; p.N = n; p.H = h; p.W = ww; p.out_f32 = out; p.add_f32 = add; p.bias0 = bias;
    return launch_conv_tc_head((const bf16*)in, p, (cudaStream_t)stream);
}

int ptta_up2_1ch(const float* a, const float* b, const float* c, float* out, int n, int h, int w, ptta_stream_t stream) {
    long long tot = (long long)n * h * w * 4;
    launch_k(up2_1ch_kernel, cdiv(tot, 256), 256, 0, (cudaStream_t)stream, a, b, c, out, n, h, w);
    return check_launch("up2_1ch");
}
int ptta_up2_1ch_adjoint(const float* ghi, float* glo, int n, int h, int w, int accumulate, ptta_stream_t stream) {
    long long tot = (long long)n * h * w;
    launch_k(up2_1ch_adj_kernel, cdiv(tot, 256), 256, 0, (cudaStream_t)stream, ghi, glo, n, h, w, accumulate);
    return check_launch("up2_1ch_adj");
}
int ptta_add_up2_c32(const void* x, const void* half, void* out, int n, int h, int w, ptta_stream_t stream) {
    long long tot = (long long)n * h * w * 4 * 4;
    launch_k(add_up2_c32_kernel, cdiv(tot, 256), 256, 0, (cudaStream_t)stream, (const bf16*)x, (const bf16*)half, (bf16*)out, n, h, w, nullptr);
    return check_launch("add_up2_c32");
}
int ptta_up2_c32_adjoint(const void* ghi, void* glo, int n, int h, int w, int accumulate, ptta_stream_t stream) {
    long long tot = (long long)n * h * w * 4;
    launch_k(up2_c32_adj_kernel, cdiv(tot, 256), 256, 0, (cudaStream_t)stream, (const bf16*)ghi, (bf16*)glo, n, h, w, accumulate);
    return check_launch("up2_c32_adj");
}

int ptta_gemm_bf16(const void* a, const void* b, void* c, const float* bias, long long m, int n, int k, ptta_stream_t stream) {
    GemmParams p; p.A = (const bf16*)a; p.B = (const bf16*)b; p.C = (bf16*)c; p.bias = bias; p.M = m; p.N = n; p.K = k;
    return launch_gemm(p, (cudaStream_t)stream);
}

int ptta_gemm_bf16_tc(const void* a, const void* b, void* c, const float* bias, long long m, int n, int k, ptta_stream_t stream) {
    PTTA_CHECK(a && b && c, "gemm_bf16_tc: null argument");
    return launch_gemm_tc((const bf16*)a, (const bf16*)b, (bf16*)c, bias, m, n, k, (cudaStream_t)stream);
}

__global__ void adam_flat_kernel(float* p, const float* g, float* m, float* v, long long n, double lr, double b1, double b2, float eps,
                                 float wd, int step) {
    PDL_SYNC();
    const double bc1 = 1.0 - pow(b1, (double)step);
    const double bc2 = 1.0 - pow(b2, (double)step);
    const float step_size = (float)(lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float fb2 = (float)b2, omb1 = (float)(1.0 - b1), omb2 = (float)(1.0 - b2);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float pp = p[i], mm = m[i], vv = v[i];
        adam_update(pp, g[i], mm, vv, fb2, omb1, omb2, eps, wd, step_size, bc2_sqrt);
        p[i] = pp; m[i] = mm; v[i] = vv;
    }
}
// CUDA-graph friendly variant: step counter and hyper-parameters (lr, beta1, beta2, eps, weight_decay as doubles) live on the device
__global__ void adam_tick_kernel(int* step) {
    PDL_SYNC(); *step += 1; }
__global__ void adam_flat_dev_kernel(float* p, const float* g, float* m, float* v, long long n, const double* __restrict__ hy, const int* __restrict__ step) {
    PDL_SYNC();
    const double b1 = hy[1], b2 = hy[2];
    const int t = *step;
    const double bc1 = 1.0 - pow(b1, (double)t);
    const double bc2 = 1.0 - pow(b2, (double)t);
    const float step_size = (float)(hy[0] / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float fb2 = (float)b2, omb1 = (float)(1.0 - b1), omb2 = (float)(1.0 - b2), eps = (float)hy[3], wd = (float)hy[4];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float pp = p[i], mm = m[i], vv = v[i];
        adam_update(pp, g[i], mm, vv, fb2, omb1, omb2, eps, wd, step_size, bc2_sqrt);
        p[i] = pp; m[i] = mm; v[i] = vv;
    }
}
// shared-model mode of the flat-buffer Adam (the NLSPN back-end): mean all-reduce of the gradient buffer FUSED with the update, one-shot
// over peer memory like adam_allreduce_kernel.  Block = one ADAM_CHUNK slice of the buffer: it copies its slice of the local gradient into
// the rank's slot, the ranks rendezvous (peer_comm.cuh), then it sums the W copies in rank order (bit-identical on all ranks), scales by
// 1/W, writes the averaged gradient back to g (what DDP leaves in .grad) and applies the update of adam_flat_dev_kernel
__global__ void __launch_bounds__(256) adam_flat_allreduce_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                                  long long n, const double* __restrict__ hy, const int* __restrict__ step,
                                                                  const PeerComm comm, int xid) {
    PDL_SYNC();
    const long long i0 = (long long)blockIdx.x * ADAM_CHUNK;
    const int cnt = n - i0 < ADAM_CHUNK ? (int)(n - i0) : ADAM_CHUNK;
    const uint32_t tag = comm_tag(comm);
    const size_t off = comm_grad_off((int)(tag & 1u), comm.grad_floats);
    float* mine = reinterpret_cast<float*>(comm.base[comm.rank] + off) + i0;
    for (int i = threadIdx.x; i < cnt; i += 256) mine[i] = g[i0 + i];
    comm_publish_and_wait(comm, xid, tag);
    const double b1 = hy[1], b2 = hy[2];
    const int t = *step;
    const double bc1 = 1.0 - pow(b1, (double)t);
    const double bc2 = 1.0 - pow(b2, (double)t);
    const float step_size = (float)(hy[0] / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float fb2 = (float)b2, omb1 = (float)(1.0 - b1), omb2 = (float)(1.0 - b2), eps = (float)hy[3], wd = (float)hy[4];
    const float inv_w = 1.f / (float)comm.world;
    for (int i = threadIdx.x; i < cnt; i += 256) {
        float gs = 0.f;
        for (int r = 0; r < comm.world; ++r) gs += ld_volatile_f32(reinterpret_cast<const float*>(comm.base[r] + off) + i0 + i);
        gs *= inv_w;
        g[i0 + i] = gs;
        float pp = p[i0 + i], mm = m[i0 + i], vv = v[i0 + i];
        adam_update(pp, gs, mm, vv, fb2, omb1, omb2, eps, wd, step_size, bc2_sqrt);
        p[i0 + i] = pp; m[i0 + i] = mm; v[i0 + i] = vv;
    }
}
// ---- stand-alone fused TTA loss (used by the NLSPN back-end, whose graph is driven from Python) -------------------------------------
struct TtaLossLayout { size_t scalars, map_partial, cos_partial, rowstat, total; int map_blocks, cos_blocks; };
static TtaLossLayout tta_loss_layout(int n, int h, int w, long long rows) {
    TtaLossLayout L;
    L.map_blocks = std::min(cdiv((long long)h * w, LOSS_BLOCK * 4), 1184);
    L.cos_blocks = (int)std::min<long long>(std::max<long long>(cdiv(rows, 8), 1), 1184);
    size_t o = 0;
    L.scalars = o; o += 512;
    L.map_partial = o; o += (size_t)n * L.map_blocks * 4 * sizeof(double);
    L.cos_partial = o; o += (size_t)L.cos_blocks * sizeof(double);
    L.rowstat = o; o += (size_t)rows * 3 * sizeof(float);
    L.total = (o + 255) / 256 * 256;
    return L;
}
size_t ptta_tta_loss_workspace_bytes(int n, int h, int w, long long rows) { return tta_loss_layout(n, h, w, rows).total; }

int ptta_tta_loss_forward(const float* pred, const float* image_raw, const float* sparse, const float* validity, float cap, const void* emb,
                          const void* ref, long long rows, int dim, float w_sd, float w_sm, float w_cos, void* workspace, int n, int h, int w,
                          ptta_stream_t stream) {
    PTTA_CHECK(pred && image_raw && sparse && validity && emb && ref && workspace, "tta_loss_forward: null pointer");
    PTTA_CHECK(n <= 64 && dim % 256 == 0, "tta_loss_forward: batch %d > 64 or row length %d not a multiple of 256", n, dim);
    const TtaLossLayout L = tta_loss_layout(n, h, w, rows);
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(L.map_blocks, n);
    launch_k(loss_map_reduce_kernel, grid, LOSS_BLOCK, 0, st, pred, sparse, validity, image_raw, (double*)(ws + L.map_partial), h, w, cap, cap > 0.f ? 1 : 0);
    PTTA_TRY(check_launch("loss_map_reduce"));
    launch_k(loss_cos_rows_kernel, L.cos_blocks, 256, 0, st, (const bf16*)emb, (const bf16*)ref, (float*)(ws + L.rowstat), (double*)(ws + L.cos_partial), rows, dim);
    PTTA_TRY(check_launch("loss_cos_rows"));
    launch_k(loss_finalize_kernel, 1, 256, 0, st, (const double*)(ws + L.map_partial), L.map_blocks, (const double*)(ws + L.cos_partial), L.cos_blocks, n, h, w,
                                          rows, w_sd, w_sm, w_cos, 0.3f, (LossScalars*)(ws + L.scalars));
    return check_launch("loss_finalize");
}

int ptta_tta_loss_backward(const float* pred, const float* image_raw, const float* sparse, const float* validity, float cap, const void* emb,
                           const void* ref, long long rows, int dim, float w_sd, float w_sm, void* workspace, float gscale, float* g_pred,
                           void* g_ref, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(pred && image_raw && sparse && validity && emb && ref && workspace && g_pred && g_ref, "tta_loss_backward: null pointer");
    const TtaLossLayout L = tta_loss_layout(n, h, w, rows);
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    const long long tot = (long long)n * h * w;
    launch_k(loss_map_grad_kernel, cdiv(tot, 256), 256, 0, st, pred, sparse, validity, image_raw, g_pred, (const LossScalars*)(ws + L.scalars), n, h, w, cap,
                                                       cap > 0.f ? 1 : 0, w_sd, w_sm, gscale);
    PTTA_TRY(check_launch("loss_map_grad"));
    launch_k(loss_cos_grad_kernel, L.cos_blocks, 256, 0, st, (const bf16*)emb, (const bf16*)ref, (const float*)(ws + L.rowstat),
                                                      (const LossScalars*)(ws + L.scalars), (bf16*)g_ref, rows, dim, gscale, 0);
    return check_launch("loss_cos_grad");
}

int ptta_tta_loss_backward_emb(const void* emb, const void* ref, long long rows, int dim, void* workspace, float gscale, void* g_emb, int n, int h,
                               int w, ptta_stream_t stream) {
    PTTA_CHECK(emb && ref && workspace && g_emb, "tta_loss_backward_emb: null pointer");
    const TtaLossLayout L = tta_loss_layout(n, h, w, rows);
    char* ws = (char*)workspace;
    launch_k(loss_cos_grad_kernel, L.cos_blocks, 256, 0, (cudaStream_t)stream, (const bf16*)emb, (const bf16*)ref, (const float*)(ws + L.rowstat),
                                                      (const LossScalars*)(ws + L.scalars), (bf16*)g_emb, rows, dim, gscale, 1);
    return check_launch("loss_cos_grad(emb)");
}

// stage-2 loss on stand-alone buffers (the NLSPN head trainer, driven from Python): mean(2 - 2 cos(emb, ref)) with no gate
// (src/external_model_adapt.py:524-540); same workspace layout as ptta_tta_loss_forward, so ptta_tta_loss_backward_emb follows it
int ptta_cos_loss_forward(const void* emb, const void* ref, long long rows, int dim, void* workspace, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(emb && ref && workspace && rows >= 1, "cos_loss_forward: bad argument");
    PTTA_CHECK(dim % 256 == 0, "cos_loss_forward: row length %d not a multiple of 256", dim);
    const TtaLossLayout L = tta_loss_layout(n, h, w, rows);
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    launch_k(loss_cos_rows_kernel, L.cos_blocks, 256, 0, st, (const bf16*)emb, (const bf16*)ref, (float*)(ws + L.rowstat), (double*)(ws + L.cos_partial), rows, dim);
    PTTA_TRY(check_launch("loss_cos_rows"));
    launch_k(cos_loss_finalize_kernel, 1, 256, 0, st, (const double*)(ws + L.cos_partial), L.cos_blocks, rows, (LossScalars*)(ws + L.scalars));
    return check_launch("cos_loss_finalize");
}

// target <- target * tau + source * (1 - tau), two products and one sum (no FMA) like the reference's tensor expression
// (nlspnmodel_adapt.py:1314-1316, network_exp_msg_chn_adapt.py:701-703); 1 - tau is formed in double like the Python float
int ptta_ema_update(float* target, const float* source, long long count, double tau, ptta_stream_t stream) {
    PTTA_CHECK(target && source && count >= 1, "ema_update: bad argument");
    EmaParams ep; memset(&ep, 0, sizeof(ep));
    ep.t[0] = target; ep.s[0] = source; ep.n[0] = count; ep.count = 1;
    ep.tau = (float)tau; ep.one_minus_tau = (float)(1.0 - tau);
    launch_k(ema_update_kernel, dim3(cdiv(count, 256), 1), 256, 0, (cudaStream_t)stream, ep);
    return check_launch("ema_update");
}

// ---- on-device augmentations (augment.cuh; SURVEY section 8 f2) ----------------------------------------------------------------------
int ptta_augment_photometric(const float* image, float* out, int n, int h, int w, const unsigned char* do_brightness, const float* f_brightness,
                             const unsigned char* do_contrast, const float* f_contrast, const unsigned char* do_saturation,
                             const float* f_saturation, const unsigned char* do_gamma, const float* f_gamma, const unsigned char* do_hue,
                             const float* f_hue, const unsigned char* do_noise, const float* noise, float noise_spread, int noise_uniform,
                             int quantize, int norm_mode, const float* mean3, const float* std3, void* workspace, ptta_stream_t stream) {
    PTTA_CHECK(image && out && n >= 1 && h >= 1 && w >= 1, "augment_photometric: bad argument");
    PTTA_CHECK(norm_mode >= 0 && norm_mode <= 3, "augment_photometric: normalisation mode %d", norm_mode);
    PTTA_CHECK(norm_mode != 3 || (mean3 && std3), "augment_photometric: standard normalisation needs mean and std");
    PTTA_CHECK((!do_brightness || f_brightness) && (!do_contrast || f_contrast) && (!do_saturation || f_saturation) && (!do_gamma || f_gamma),
               "augment_photometric: a flag array without its factor array");
    PTTA_CHECK(!do_contrast || workspace, "augment_photometric: the contrast transform needs a workspace of 8 * n bytes");
    PTTA_CHECK(quantize || !(do_brightness || do_contrast || do_saturation || do_gamma || do_hue), "augment_photometric: the photometric transforms work on the uint8 image");
    PTTA_CHECK((!do_hue || f_hue) && (!do_noise || noise), "augment_photometric: a flag array without its factor / noise array");
    PTTA_CHECK((long long)h * w < (1ll << 31) / 3 && n <= 65535, "augment_photometric: image too large");
    cudaStream_t st = (cudaStream_t)stream;
    PhotoParams p; memset(&p, 0, sizeof(p));
    p.in = image; p.out = out; p.do_b = do_brightness; p.do_c = do_contrast; p.do_s = do_saturation;
    p.f_b = f_brightness; p.f_c = f_contrast; p.f_s = f_saturation; p.gray_sum = (unsigned long long*)workspace;
    p.do_g = do_gamma; p.f_g = f_gamma; p.do_h = do_hue; p.f_h = f_hue;
    p.do_n = do_noise; p.noise = noise; p.noise_spread = noise_spread; p.noise_uniform = noise_uniform;
    p.N = n; p.HW = h * w; p.quantize = quantize; p.norm_mode = norm_mode;
    for (int k = 0; k < 3; ++k) { p.mean[k] = mean3 ? mean3[k] : 0.f; p.std[k] = std3 ? std3[k] : 1.f; }
    // 16-byte accesses when every colour plane starts on a 16-byte boundary; ~2 waves of blocks over the whole batch
    const bool vec = (p.HW % 4 == 0) && (((uintptr_t)image | (uintptr_t)out) & 15) == 0;
    const int per_block = 256 * (vec ? 4 : 1) * 2;
    const int bx = std::max(1, std::min(cdiv(p.HW, per_block), cdiv(2368, n)));
    if (do_contrast) {
        PTTA_CUDA(cudaMemsetAsync(workspace, 0, sizeof(unsigned long long) * n, st));
        if (vec) launch_k(photo_gray_sum_kernel<4>, dim3(bx, n), 256, 0, st, p);
        else launch_k(photo_gray_sum_kernel<1>, dim3(bx, n), 256, 0, st, p);
        PTTA_TRY(check_launch("photo_gray_sum"));
    }
    if (vec) launch_k(photo_apply_kernel<4>, dim3(bx, n), 256, 0, st, p);
    else launch_k(photo_apply_kernel<1>, dim3(bx, n), 256, 0, st, p);
    return check_launch("photo_apply");
}

int ptta_augment_flip(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_hflip, const unsigned char* do_vflip,
                      ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && n >= 1 && c >= 1 && h >= 1 && w >= 1, "augment_flip: bad argument (in-place is not supported)");
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_flip: map too large");
    const bool vec = (w % 4 == 0) && (((uintptr_t)in | (uintptr_t)out) & 15) == 0;
    const int bx = std::max(1, std::min(cdiv((long long)c * h * w, 256 * (vec ? 4 : 1) * 2), cdiv(2368, n)));
    if (vec) launch_k(flip_kernel<4>, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_hflip, do_vflip);
    else launch_k(flip_kernel<1>, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_hflip, do_vflip);
    return check_launch("flip");
}

int ptta_augment_crop(const float* in, float* out, int n, int c, int h, int w, int crop_h, int crop_w, const int* start_y, const int* start_x,
                      ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && start_y && start_x && n >= 1 && c >= 1, "augment_crop: bad argument");
    PTTA_CHECK(crop_h >= 1 && crop_w >= 1 && crop_h <= h && crop_w <= w, "augment_crop: window %dx%d does not fit %dx%d", crop_h, crop_w, h, w);
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_crop: map too large");
    const int bx = std::max(1, std::min(cdiv((long long)c * crop_h * crop_w, 256 * 4), cdiv(2368, n)));
    launch_k(crop_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, crop_h, crop_w, start_y, start_x);
    return check_launch("crop");
}

int ptta_augment_crop_pad(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_crop_pad, const int* window_n_x_6,
                          ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && do_crop_pad && window_n_x_6 && n >= 1 && c >= 1 && h >= 1 && w >= 1, "augment_crop_pad: bad argument");
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_crop_pad: map too large");
    const int bx = std::max(1, std::min(cdiv((long long)c * h * w, 256 * 4), cdiv(2368, n)));
    launch_k(crop_pad_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_crop_pad, window_n_x_6);
    return check_launch("crop_pad");
}

int ptta_augment_remove_patches(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_remove, const unsigned char* selected,
                                const int* patch_n_x_2, ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && do_remove && selected && patch_n_x_2 && n >= 1 && c >= 1 && h >= 1 && w >= 1, "augment_remove_patches: bad argument");
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_remove_patches: map too large");
    const int bx = std::max(1, std::min(cdiv((long long)h * w, 256 * 2), cdiv(2368, n)));
    launch_k(remove_patches_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_remove, selected, patch_n_x_2);
    return check_launch("remove_patches");
}

int ptta_augment_resize_pad(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_resize_pad, const int* geometry_n_x_4,
                            int mode, ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && do_resize_pad && geometry_n_x_4 && n >= 1 && c >= 1 && h >= 1 && w >= 1, "augment_resize_pad: bad argument");
    PTTA_CHECK(mode == 0 || mode == 1, "augment_resize_pad: interpolation mode %d (0 nearest, 1 bilinear)", mode);
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_resize_pad: map too large");
    const int bx = std::max(1, std::min(cdiv((long long)h * w, 256 * 2), cdiv(2368, n)));
    launch_k(resize_pad_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_resize_pad, geometry_n_x_4, mode);
    return check_launch("resize_pad");
}

int ptta_augment_divide_samples(float* data, int n, long long per_sample, const unsigned char* do_divide, const float* divisor_n, ptta_stream_t stream) {
    PTTA_CHECK(data && do_divide && divisor_n && n >= 1 && n <= 65535 && per_sample >= 1, "augment_divide_samples: bad argument");
    const int bx = (int)std::max(1ll, std::min((per_sample + 511) / 512, (long long)cdiv(2368, n)));
    launch_k(divide_samples_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, data, per_sample, do_divide, divisor_n);
    return check_launch("divide_samples");
}

int ptta_augment_rotate(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_rotate, const float* theta_n_x_6,
                        int mode, ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && do_rotate && theta_n_x_6 && n >= 1 && c >= 1 && h >= 1 && w >= 1, "augment_rotate: bad argument");
    PTTA_CHECK(mode == 0 || mode == 1, "augment_rotate: interpolation mode %d (0 nearest, 1 bilinear)", mode);
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_rotate: map too large");
    const int bx = std::min(cdiv((long long)h * w, 256 * 2), 2368);
    launch_k(rotate_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_rotate, theta_n_x_6, mode);
    return check_launch("rotate");
}

int ptta_augment_resize_crop(const float* in, float* out, int n, int c, int h, int w, const unsigned char* do_resize, const int* resize_h,
                             const int* resize_w, const int* start_y, const int* start_x, int mode, ptta_stream_t stream) {
    PTTA_CHECK(in && out && in != out && do_resize && resize_h && resize_w && start_y && start_x && n >= 1 && c >= 1 && h >= 1 && w >= 1,
               "augment_resize_crop: bad argument");
    PTTA_CHECK(mode == 0 || mode == 1, "augment_resize_crop: interpolation mode %d (0 nearest, 1 bilinear)", mode);
    PTTA_CHECK((long long)c * h * w < (1ll << 31) && n <= 65535, "augment_resize_crop: map too large");
    const int bx = std::min(cdiv((long long)h * w, 256 * 2), 2368);
    launch_k(resize_crop_kernel, dim3(bx, n), 256, 0, (cudaStream_t)stream, in, out, c, h, w, do_resize, resize_h, resize_w, start_y, start_x, mode);
    return check_launch("resize_crop");
}

int ptta_adam_flat(float* p, const float* g, float* m, float* v, long long n, double lr, double b1, double b2, double eps, double wd, int step,
                   ptta_stream_t stream) {
    PTTA_CHECK(step >= 1, "adam: step must be >= 1");
    if (n <= 0) return 0;
    int blocks = (int)std::min<long long>(cdiv(n, 256), 1184);
    launch_k(adam_flat_kernel, blocks, 256, 0, (cudaStream_t)stream, p, g, m, v, n, lr, b1, b2, (float)eps, (float)wd, step);
    return check_launch("adam_flat");
}

int ptta_adam_flat_dev(float* p, const float* g, float* m, float* v, long long n, const double* hyper_dev, int* step_dev, ptta_stream_t stream) {
    PTTA_CHECK(p && g && m && v && hyper_dev && step_dev, "adam_flat_dev: null pointer");
    if (n <= 0) return 0;
    launch_k(adam_tick_kernel, 1, 1, 0, (cudaStream_t)stream, step_dev);
    PTTA_TRY(check_launch("adam_tick"));
    int blocks = (int)std::min<long long>(cdiv(n, 256), 1184);
    launch_k(adam_flat_dev_kernel, blocks, 256, 0, (cudaStream_t)stream, p, g, m, v, n, hyper_dev, step_dev);
    return check_launch("adam_flat_dev");
}

int ptta_adam_flat_dev_comm(float* p, float* g, float* m, float* v, long long n, const double* hyper_dev, int* step_dev, ptta_comm* comm, int xid,
                            ptta_stream_t stream) {
    PTTA_CHECK(p && g && m && v && hyper_dev && step_dev && comm, "adam_flat_dev_comm: null pointer");
    PTTA_CHECK(xid >= 0 && xid < PTTA_COMM_MAX_XID, "adam_flat_dev_comm: exchange id %d outside [0, %d)", xid, PTTA_COMM_MAX_XID);
    PTTA_CHECK(n > 0 && (size_t)n <= comm->dev.grad_floats, "adam_flat_dev_comm: %lld floats, the communicator's gradient slot holds %zu", n,
               comm->dev.grad_floats);
    // every block spins in the rendezvous: all of them must be resident at once (peer_comm.cuh: a spinning kernel has at most
    // PTTA_COMM_MAX_SPIN_BLOCKS blocks; the NLSPN buffer needs 23)
    const long long blocks = cdiv(n, (long long)ADAM_CHUNK);
    PTTA_CHECK(blocks <= PTTA_COMM_MAX_SPIN_BLOCKS, "adam_flat_dev_comm: %lld floats need %lld blocks (at most %d spin at once)", n, blocks,
               PTTA_COMM_MAX_SPIN_BLOCKS);
    for (int r = 0; r < comm->dev.world; ++r) PTTA_CHECK(comm->dev.base[r] != nullptr, "adam_flat_dev_comm: peer %d not opened (ptta_comm_open_peers)", r);
    launch_k(adam_tick_kernel, 1, 1, 0, (cudaStream_t)stream, step_dev);
    PTTA_TRY(check_launch("adam_tick"));
    launch_k(adam_flat_allreduce_kernel, (int)blocks, 256, 0, (cudaStream_t)stream, p, g, m, v, n, hyper_dev, step_dev, comm->dev, xid);
    return check_launch("adam_flat_allreduce");
}

// ---- NLSPN propagation path (SURVEY.md section 8 a20-a21) ------------------------------------------------------
static int mdconv_check(int c_in, int c_out, int kh, int kw, int stride, int pad, int dil, int groups, int dgroups) {
    PTTA_CHECK(c_in == 1 && c_out == 1 && groups == 1 && dgroups == 1,
               "mdconv: only the single-channel configuration of NLSPN is implemented (got C_in=%d C_out=%d groups=%d deformable_groups=%d)",
               c_in, c_out, groups, dgroups);
    PTTA_CHECK(kh == kw && (kh & 1) && kh <= 7, "mdconv: kernel %dx%d must be square, odd and <= 7", kh, kw);
    PTTA_CHECK(stride == 1 && dil == 1, "mdconv: stride %d / dilation %d not implemented (NLSPN uses 1 / 1)", stride, dil);
    PTTA_CHECK(pad >= 0 && 2 * pad <= kh - 1, "mdconv: padding %d larger than (k-1)/2", pad);
    return 0;
}

int ptta_mdconv_forward(const float* input, const float* weight, const float* bias, const float* offset, const float* mask, float* output,
                        int n, int c_in, int h, int w, int c_out, int kh, int kw, int stride, int pad, int dil, int groups, int dgroups,
                        ptta_stream_t stream) {
    PTTA_CHECK(input && weight && offset && mask && output, "mdconv_forward: null argument");
    PTTA_TRY(mdconv_check(c_in, c_out, kh, kw, stride, pad, dil, groups, dgroups));
    const int ho = h + 2 * pad - (kh - 1), wo = w + 2 * pad - (kw - 1);
    PTTA_CHECK(ho >= 1 && wo >= 1 && n >= 1, "mdconv_forward: empty output");
    dim3 grid(cdiv(wo, PROP_TX), cdiv(ho, PROP_TY), n), block(PROP_TX, PROP_TY);
    launch_k(mdconv1_forward_kernel, grid, block, 0, (cudaStream_t)stream, input, weight, bias, offset, mask, output, h, w, ho, wo, kh, pad);
    return check_launch("mdconv1_forward");
}

int ptta_mdconv_backward(const float* input, const float* weight, const float* offset, const float* mask, const float* grad_output,
                         float* grad_input, float* grad_offset, float* grad_mask, float* grad_weight, float* grad_bias,
                         int n, int c_in, int h, int w, int c_out, int kh, int kw, int stride, int pad, int dil, int groups, int dgroups,
                         ptta_stream_t stream) {
    PTTA_CHECK(input && weight && offset && mask && grad_output, "mdconv_backward: null argument");
    PTTA_TRY(mdconv_check(c_in, c_out, kh, kw, stride, pad, dil, groups, dgroups));
    const int ho = h + 2 * pad - (kh - 1), wo = w + 2 * pad - (kw - 1);
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_input) PTTA_CUDA(cudaMemsetAsync(grad_input, 0, sizeof(float) * (size_t)n * h * w, st));
    if (grad_weight) PTTA_CUDA(cudaMemsetAsync(grad_weight, 0, sizeof(float) * kh * kw, st));
    if (grad_bias) PTTA_CUDA(cudaMemsetAsync(grad_bias, 0, sizeof(float), st));
    dim3 grid(cdiv(wo, PROP_TX), cdiv(ho, PROP_TY), n), block(PROP_TX, PROP_TY);
    launch_k(mdconv1_backward_kernel, grid, block, 0, st, input, weight, offset, mask, grad_output, grad_input, grad_offset, grad_mask, grad_weight,
                                                   grad_bias, h, w, ho, wo, kh, pad);
    return check_launch("mdconv1_backward");
}

int ptta_nlspn_offset_affinity_forward(const float* offset_aff, const float* confidence, float aff_scale_const, int legacy, float* offset,
                                       float* aff, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(offset_aff && offset && aff, "nlspn_offset_affinity_forward: null argument");
    PTTA_CHECK(n >= 1 && h >= 1 && w >= 1, "nlspn_offset_affinity_forward: bad shape %dx%dx%d", n, h, w);
    dim3 grid(cdiv(w, PROP_TX), cdiv(h, PROP_TY), n), block(PROP_TX, PROP_TY);
    launch_k(offset_affinity_forward_kernel, grid, block, 0, (cudaStream_t)stream, offset_aff, confidence, 1.f / (aff_scale_const + 1e-8f), legacy, offset, aff,
                                                                             h, w);
    return check_launch("offset_affinity_forward");
}
int ptta_nlspn_offset_affinity_backward(const float* offset_aff, const float* confidence, float aff_scale_const, int legacy,
                                        const float* grad_offset, const float* grad_aff, float* grad_offset_aff, float* grad_confidence,
                                        int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(offset_aff && grad_offset && grad_aff && grad_offset_aff, "nlspn_offset_affinity_backward: null argument");
    PTTA_CHECK(!confidence == !grad_confidence || !grad_confidence, "nlspn_offset_affinity_backward: grad_confidence without confidence");
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_confidence) PTTA_CUDA(cudaMemsetAsync(grad_confidence, 0, sizeof(float) * (size_t)n * h * w, st));
    dim3 grid(cdiv(w, PROP_TX), cdiv(h, PROP_TY), n), block(PROP_TX, PROP_TY);
    launch_k(offset_affinity_backward_kernel, grid, block, 0, st, offset_aff, confidence, 1.f / (aff_scale_const + 1e-8f), legacy, grad_offset, grad_aff,
                                                           grad_offset_aff, grad_confidence, h, w);
    return check_launch("offset_affinity_backward");
}

size_t ptta_nlspn_saved_bytes(int n, int h, int w, int prop_time) { return sizeof(float) * (size_t)n * h * w * (size_t)(prop_time > 0 ? prop_time : 0); }
size_t ptta_nlspn_backward_scratch_bytes(int n, int h, int w) { return sizeof(float) * 2 * (size_t)n * h * w; }

int ptta_nlspn_propagate_forward(const float* feat_init, const float* offset, const float* aff, const float* feat_fix, float* feat_out,
                                 float* saved, float* list_feat, int n, int h, int w, int prop_time, ptta_stream_t stream) {
    PTTA_CHECK(feat_init && offset && aff && feat_out && saved, "nlspn_propagate_forward: null argument");
    PTTA_CHECK(n >= 1 && h >= 1 && w >= 1 && prop_time >= 1, "nlspn_propagate_forward: bad shape %dx%dx%d, prop_time %d", n, h, w, prop_time);
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)n * h * w;
    launch_k(prop_blend_kernel, cdiv(total, 256), 256, 0, st, feat_init, feat_fix, saved, total);
    PTTA_TRY(check_launch("prop_blend"));
    dim3 grid(cdiv(w, PROP_TX), cdiv(h, PROP_TY), n), block(PROP_TX, PROP_TY);
    for (int k = 0; k < prop_time; ++k) {
        const bool last = k == prop_time - 1;
        float* raw = last ? feat_out : (list_feat ? list_feat + (size_t)k * total : nullptr);
        launch_k(prop_step_kernel, grid, block, 0, st, saved + (size_t)k * total, offset, aff, feat_fix, raw, last ? nullptr : saved + (size_t)(k + 1) * total,
                                                h, w);
        PTTA_TRY(check_launch("prop_step"));
        if (last && list_feat) PTTA_CUDA(cudaMemcpyAsync(list_feat + (size_t)k * total, feat_out, sizeof(float) * total, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

int ptta_nlspn_propagate_backward(const float* grad_out, const float* offset, const float* aff, const float* feat_fix, const float* saved,
                                  float* grad_feat_init, float* grad_offset, float* grad_aff, float* scratch, int n, int h, int w, int prop_time,
                                  ptta_stream_t stream) {
    PTTA_CHECK(grad_out && offset && aff && saved && grad_feat_init && grad_offset && grad_aff && scratch, "nlspn_propagate_backward: null argument");
    PTTA_CHECK(n >= 1 && h >= 1 && w >= 1 && prop_time >= 1, "nlspn_propagate_backward: bad shape %dx%dx%d, prop_time %d", n, h, w, prop_time);
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)n * h * w;
    float* a = scratch;
    float* b = scratch + total;
    PTTA_CUDA(cudaMemcpyAsync(a, grad_out, sizeof(float) * total, cudaMemcpyDeviceToDevice, st));
    PTTA_CUDA(cudaMemsetAsync(b, 0, sizeof(float) * total, st));
    dim3 grid(cdiv(w, PROP_TX), cdiv(h, PROP_TY), n), block(PROP_TX, PROP_TY);
    for (int k = prop_time - 1; k >= 0; --k) {
        const bool first = k == prop_time - 1;
        launch_k(prop_step_backward_kernel, grid, block, 0, st, saved + (size_t)k * total, offset, aff, feat_fix, a, b, grad_offset, grad_aff, h, w,
                                                         first ? 0 : 1, first ? 0 : 1);
        PTTA_TRY(check_launch("prop_step_backward"));
        float* t = a; a = b; b = t;          // `a` now holds the gradient wrt this step's blended input; `b` has been cleared
    }
    launch_k(prop_mask_grad_kernel, cdiv(total, 256), 256, 0, st, a, feat_fix, grad_feat_init, total);
    return check_launch("prop_mask_grad");
}

// ---- engine ---------------------------------------------------------------------------------------
int ptta_msgchn_create(ptta_msgchn** out, int n, int h, int w, const char* prepare_mode) {
    PTTA_CHECK(out != nullptr, "create: null out pointer");
    PTTA_CHECK(n >= 1 && h >= 1 && w >= 1, "create: bad shape %dx%dx%d", n, h, w);
    std::string mode = prepare_mode ? prepare_mode : "";
    PTTA_CHECK(mode.find("meta") != std::string::npos && mode.find("seq") != std::string::npos,
               "create: prepare_mode '%s' has no sequential meta layer (network_exp_msg_chn_adapt.py:1063-1077)", mode.c_str());
    bool two = mode.find("2layers") != std::string::npos, one = mode.find("1layer") != std::string::npos;
    PTTA_CHECK(two || one, "create: prepare_mode '%s' must contain '1layer' or '2layers'", mode.c_str());
    ptta_msgchn* e = new ptta_msgchn();
    e->Nu = n; e->Hu = h; e->Wu = w;
    e->padded = (h % 16 != 0) || (w % 16 != 0);          // pad to /16 + flip-pad pair (src/msg_chn_model_adapt.py:58-102)
    e->N = e->padded ? 2 * n : n; e->H = (h + 15) / 16 * 16; e->W = (w + 15) / 16 * 16;
    e->two_layers = two; e->prepare_mode = mode;
    e->has_heads = mode.find("selfsup") != std::string::npos;
    e->define_model();
    e->plan();
    *out = e;
    return 0;
}
// ---- peer communicator of the shared-model mode (peer_comm.cuh) ---------------------------------------------------------
// struct ptta_comm: peer_comm.cuh (the NLSPN entry points of nlspn_net.cu read its device view too)
int ptta_comm_create(ptta_comm** out, int rank, int world, long long grad_floats) {
    PTTA_CHECK(out && world >= 1 && world <= PTTA_COMM_MAX_RANKS && rank >= 0 && rank < world && grad_floats > 0, "comm_create: bad arguments (rank %d of %d)", rank, world);
    ptta_comm* c = new ptta_comm();
    c->dev.world = world; c->dev.rank = rank; c->dev.grad_floats = (size_t)grad_floats;
    c->bytes = comm_block_bytes((size_t)grad_floats);
    if (cudaMalloc(&c->local, c->bytes) != cudaSuccess) { delete c; set_error("comm_create: cudaMalloc(%zu) failed", c->bytes); return 2; }
    PTTA_CUDA(cudaMemset(c->local, 0, c->bytes));
    PTTA_CUDA(cudaDeviceSynchronize());
    c->dev.base[rank] = (unsigned char*)c->local;
    *out = c;
    return 0;
}
int ptta_comm_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }
int ptta_comm_local_handle(ptta_comm* c, void* handle_out) {
    PTTA_CHECK(c && handle_out, "comm_local_handle: null argument");
    cudaIpcMemHandle_t h;
    PTTA_CUDA(cudaIpcGetMemHandle(&h, c->local));
    memcpy(handle_out, &h, sizeof(h));
    return 0;
}
/* handles: world x ptta_comm_handle_bytes() bytes, rank order (this rank's own entry is ignored) */
int ptta_comm_open_peers(ptta_comm* c, const void* handles) {
    PTTA_CHECK(c && handles, "comm_open_peers: null argument");
    for (int r = 0; r < c->dev.world; ++r) {
        if (r == c->dev.rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * sizeof(h), sizeof(h));
        void* p = nullptr;
        cudaError_t err = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        PTTA_CHECK(err == cudaSuccess, "comm_open_peers: cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(err));
        c->opened[r] = p;
        c->dev.base[r] = (unsigned char*)p;
    }
    return 0;
}
/* 0: no exchange ever timed out; k > 0: exchange k-1 of some step gave up waiting for a peer (results since then are void) */
int ptta_comm_error(ptta_comm* c) {
    if (!c || !c->local) return -1;
    uint32_t v = 0;
    if (cudaMemcpy(&v, (const char*)c->local + comm_error_off(), sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int)v;
}
void ptta_comm_destroy(ptta_comm* c) {
    if (!c) return;
    for (int r = 0; r < PTTA_COMM_MAX_RANKS; ++r) if (c->opened[r]) cudaIpcCloseMemHandle(c->opened[r]);
    if (c->local) cudaFree(c->local);
    delete c;
}
int ptta_comm_max_exchanges(void) { return PTTA_COMM_MAX_XID; }
int ptta_comm_advance(ptta_comm* c, ptta_stream_t stream) {
    PTTA_CHECK(c && c->local, "comm_advance: null communicator");
    launch_k(comm_advance_kernel, 1, 32, 0, (cudaStream_t)stream, c->dev);
    return check_launch("comm_advance");
}
/* shared-model mode on: SyncBatchNorm statistics over all ranks + gradient all-reduce fused with Adam (comm = NULL: off).  Exchange slots
 * are numbered in host call order, which is the same on every rank; kernels of different streams may reach their exchanges in any
 * order (each exchange has its own flags, and the spinning kernels are a few blocks that never fill the machine).  Option two_streams = 0
 * puts the whole step on one stream. */
int ptta_msgchn_set_comm(ptta_msgchn* e, ptta_comm* c) {
    PTTA_CHECK(e, "set_comm: null engine");
    if (c) {
        for (int r = 0; r < c->dev.world; ++r) PTTA_CHECK(c->dev.base[r] != nullptr, "set_comm: peer %d not opened (ptta_comm_open_peers)", r);
        e->comm = c->dev;
    } else {
        e->comm = PeerComm();
    }
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    return 0;
}

int ptta_msgchn_set_option(ptta_msgchn* e, const char* name, long long value) {
    PTTA_CHECK(e && name, "set_option: null argument");
    const std::string k = name;
    if (k == "tc_min_pixels") e->tc_min_pixels = value;                 // smallest map (pixels) the stride-1 tcgen05 conv takes
    else if (k == "tc_s2_min_pixels") e->tc_s2_min_pixels = value;      // same for the stride-2 tcgen05 conv
    else if (k == "tc_t2_min_pixels") e->tc_t2_min_pixels = value;      // same for the transposed stride-2 tcgen05 conv (INPUT pixels)
    else if (k == "tc_head_min_pixels") e->tc_head_min_pixels = value;  // same for the 32 -> 1 tcgen05 conv (prediction layers, stem data gradients)
    else if (k == "tc_stem_min_pixels") e->tc_stem_min_pixels = value;  // same for the {1,2,3} -> 32 tcgen05 stem (and the prediction layers' data gradient)
    else if (k == "tc_enabled") e->tc_enabled = value != 0;
    else if (k == "two_streams") e->two_streams = value != 0;
    else if (k == "fuse_projpred") e->fuse_projpred = value != 0;
    else if (k == "trainable_head") { if (value) PTTA_TRY(e->select_trainable_head()); }   // stage-2 trainer: Adam steps pred.*, not the meta layer
    else if (k == "skip_dec3") e->skip_dec3 = value != 0;                  // stage 2 never reads the prediction of the real branch
    else PTTA_CHECK(false, "set_option: unknown option '%s'", name);
    e->drop_graphs();   // a captured step bakes the dispatch in
    return 0;
}
void ptta_msgchn_destroy(ptta_msgchn* e) {
    if (!e) return;
    e->drop_graphs();
    if (e->st2) { cudaStreamDestroy(e->st2); cudaEventDestroy(e->ev_fork); cudaEventDestroy(e->ev_join); cudaEventDestroy(e->ev_projbn);
                 cudaEventDestroy(e->ev_enc1); cudaEventDestroy(e->ev_zmeta); }
    if (e->st3) { cudaStreamDestroy(e->st3); cudaEventDestroy(e->ev_e3); cudaEventDestroy(e->ev_mlp); cudaEventDestroy(e->ev_lossg);
                 cudaEventDestroy(e->ev_headb); cudaEventDestroy(e->ev_gmg); cudaEventDestroy(e->ev_wg2); }
    delete e;
}
size_t ptta_msgchn_workspace_bytes(const ptta_msgchn* e) { return e ? e->ws_bytes : 0; }

int ptta_msgchn_bind_workspace(ptta_msgchn* e, void* ws, size_t bytes, ptta_stream_t stream) {
    PTTA_CHECK(e && ws, "bind_workspace: null argument");
    PTTA_CHECK(bytes >= e->ws_bytes, "bind_workspace: %zu bytes given, %zu needed", bytes, e->ws_bytes);
    PTTA_CHECK(((uintptr_t)ws & 255) == 0, "bind_workspace: pointer must be 256-byte aligned");
    e->arena.base = (char*)ws;
    e->plan();
    e->bound = true; e->packed = false;
    if (!e->st2) {
        PTTA_CUDA(cudaStreamCreateWithFlags(&e->st2, cudaStreamNonBlocking));
        PTTA_CUDA(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
        PTTA_CUDA(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
        PTTA_CUDA(cudaEventCreateWithFlags(&e->ev_projbn, cudaEventDisableTiming));
        PTTA_CUDA(cudaEventCreateWithFlags(&e->ev_enc1, cudaEventDisableTiming));
        PTTA_CUDA(cudaEventCreateWithFlags(&e->ev_zmeta, cudaEventDisableTiming));
        PTTA_CUDA(cudaStreamCreateWithFlags(&e->st3, cudaStreamNonBlocking));
        cudaEvent_t* evs[6] = {&e->ev_e3, &e->ev_mlp, &e->ev_lossg, &e->ev_headb, &e->ev_gmg, &e->ev_wg2};
        for (cudaEvent_t* ev : evs) PTTA_CUDA(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    }
    PTTA_CUDA(cudaMemsetAsync(ws, 0, e->ws_bytes, (cudaStream_t)stream));
    AdamHyper hy;
    {
        hy.lr = 1e-4f; hy.beta1 = 0.9f; hy.beta2 = 0.999f; hy.eps = 1e-8f; hy.weight_decay = 0.f;
        hy.one_minus_beta1 = (float)(1.0 - 0.9); hy.one_minus_beta2 = (float)(1.0 - 0.999);
        hy.step = 0; hy.beta1_d = 0.9; hy.beta2_d = 0.999; hy.lr_d = 1e-4;
    }
    PTTA_CUDA(cudaMemcpyAsync(e->adam_hyper, &hy, sizeof(hy), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    PTTA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

int ptta_msgchn_set_tensor(ptta_msgchn* e, const char* key, void* ptr, long long numel) {
    PTTA_CHECK(e && key && ptr, "set_tensor: null argument");
    e->ext[key] = std::make_pair(ptr, numel);
    e->packed = false;
    return 0;
}
int ptta_msgchn_num_keys(const ptta_msgchn* e) { return e ? (int)e->keys.size() : 0; }
const char* ptta_msgchn_key(const ptta_msgchn* e, int i) { return (e && i >= 0 && i < (int)e->keys.size()) ? e->keys[i].c_str() : nullptr; }

int ptta_msgchn_pack_weights(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e && e->bound, "pack_weights: bind a workspace first");
    e->st = (cudaStream_t)stream;
    return e->pack_all();
}
int ptta_msgchn_pack_adapted(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e && e->bound && e->packed, "pack_adapted: engine not ready");
    e->st = (cudaStream_t)stream;
    return e->pack_adapted();
}

int ptta_msgchn_forward(ptta_msgchn* e, const float* image, const float* isc, const float* ish, const float* sparse, float cap,
                        int training, ptta_stream_t stream) {
    PTTA_CHECK(e && image && sparse && isc && ish, "forward: null argument");
    e->st = (cudaStream_t)stream;
    return e->forward(image, isc, ish, sparse, cap, training);
}
// ---- source-domain preparation steps (SURVEY section 8 f3) -----------------------------------------------------------------------------
int ptta_msgchn_l2_loss(ptta_msgchn* e, const float* ground_truth, float max_predict_depth, ptta_stream_t stream) {
    PTTA_CHECK(e && ground_truth, "l2_loss: null argument");
    e->st = (cudaStream_t)stream;
    return e->l2_loss(ground_truth, max_predict_depth);
}
int ptta_msgchn_l2_loss_backward(ptta_msgchn* e, float gscale, ptta_stream_t stream) {
    PTTA_CHECK(e, "l2_loss_backward: null engine");
    e->st = (cudaStream_t)stream;
    return e->l2_loss_backward(gscale);
}
int ptta_msgchn_init_step(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, const float* ground_truth,
                          float cap, float max_predict_depth, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && ground_truth && isc && ish, "init_step: null argument");
    e->st = (cudaStream_t)stream;
    return e->init_step(image_raw, isc, ish, sparse, ground_truth, cap, max_predict_depth);
}
int ptta_msgchn_cos_loss(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e && e->has_heads, "cos_loss: engine has no proxy heads");
    e->st = (cudaStream_t)stream;
    return e->cos_loss();
}
int ptta_msgchn_ema_update_head(ptta_msgchn* e, double tau, ptta_stream_t stream) {
    PTTA_CHECK(e && e->has_heads, "ema_update_head: engine has no proxy heads");
    e->st = (cudaStream_t)stream;
    return e->ema_update_head(tau);
}
int ptta_msgchn_cos_loss_backward(ptta_msgchn* e, float gscale, ptta_stream_t stream) {
    PTTA_CHECK(e && e->has_heads, "cos_loss_backward: engine has no proxy heads");
    e->st = (cudaStream_t)stream;
    return e->cos_loss_backward(gscale);
}
int ptta_msgchn_head_backward(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e, "head_backward: null engine");
    e->st = (cudaStream_t)stream;
    return e->head_backward();
}
int ptta_msgchn_head_step(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap,
                          ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && isc && ish, "head_step: null argument");
    e->st = (cudaStream_t)stream;
    return e->head_step(image_raw, isc, ish, sparse, cap);
}
size_t ptta_gemm_tn_workspace_bytes(long long rows, int m, int n) { return gemm_tn_supported(rows, m, n) ? gemm_tn_workspace_bytes(rows, m, n) : 0; }
int ptta_gemm_tn_bf16_tc(const void* a, const void* b, float* c, void* workspace, long long rows, int m, int n, ptta_stream_t stream) {
    PTTA_CHECK(a && b && c && workspace, "gemm_tn_bf16_tc: null argument");
    return launch_gemm_tn_tc((const bf16*)a, (const bf16*)b, c, (float*)workspace, rows, m, n, (cudaStream_t)stream);
}

int ptta_msgchn_loss(ptta_msgchn* e, const float* image_raw, const float* sparse, const float* validity, float cap, float w_sd, float w_sm,
                     float w_cos, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && validity, "loss: null argument");
    PTTA_CHECK(e->has_heads, "loss: engine has no proxy heads");
    e->st = (cudaStream_t)stream;
    return e->loss(image_raw, sparse, validity, cap, w_sd, w_sm, w_cos);
}
int ptta_msgchn_read_losses(ptta_msgchn* e, float* out5, ptta_stream_t stream) {
    PTTA_CHECK(e && out5, "read_losses: null argument");
    PTTA_CUDA(cudaMemcpyAsync(out5, e->losses, 5 * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    PTTA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}
int ptta_msgchn_backward(ptta_msgchn* e, float gscale, ptta_stream_t stream) {
    PTTA_CHECK(e, "backward: null engine");
    e->st = (cudaStream_t)stream;
    return e->backward(gscale);
}
int ptta_msgchn_loss_backward(ptta_msgchn* e, float gscale, ptta_stream_t stream) {
    PTTA_CHECK(e, "loss_backward: null engine");
    e->st = (cudaStream_t)stream;
    return e->loss_backward(gscale);
}
int ptta_msgchn_network_backward(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e && e->bound && e->packed, "network_backward: engine not ready");
    e->st = (cudaStream_t)stream;
    return e->network_backward();
}
static AdamHyper make_hyper(double lr, double b1, double b2, double eps, double wd, int step) {
    AdamHyper hy;
    hy.lr = (float)lr; hy.beta1 = (float)b1; hy.beta2 = (float)b2; hy.eps = (float)eps; hy.weight_decay = (float)wd;
    hy.one_minus_beta1 = (float)(1.0 - b1); hy.one_minus_beta2 = (float)(1.0 - b2);
    hy.step = step; hy.beta1_d = b1; hy.beta2_d = b2; hy.lr_d = lr;
    return hy;
}
int ptta_msgchn_set_adam(ptta_msgchn* e, double lr, double b1, double b2, double eps, double wd, int step_count, ptta_stream_t stream) {
    PTTA_CHECK(e && e->bound, "set_adam: engine not bound");
    cudaStream_t st = (cudaStream_t)stream;
    AdamHyper hy = make_hyper(lr, b1, b2, eps, wd, step_count);
    if (step_count < 0) {   // keep the device-side step count, update the rest
        PTTA_CUDA(cudaMemcpyAsync(e->adam_hyper, &hy, offsetof(AdamHyper, step), cudaMemcpyHostToDevice, st));
        PTTA_CUDA(cudaMemcpyAsync(&e->adam_hyper->beta1_d, &hy.beta1_d, 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    } else {
        PTTA_CUDA(cudaMemcpyAsync(e->adam_hyper, &hy, sizeof(hy), cudaMemcpyHostToDevice, st));
    }
    PTTA_CUDA(cudaStreamSynchronize(st));   // hy is a stack object
    return 0;
}
int ptta_msgchn_adam_step(ptta_msgchn* e, ptta_stream_t stream) {
    PTTA_CHECK(e && e->bound && e->packed, "adam_step: engine not ready");
    e->st = (cudaStream_t)stream;
    return e->adam_step();
}
int ptta_msgchn_tta_step(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap,
                         float w_sd, float w_sm, float w_cos, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && isc && ish, "tta_step: null argument");
    e->st = (cudaStream_t)stream;
    return e->tta_step(image_raw, isc, ish, sparse, cap, w_sd, w_sm, w_cos);
}
int ptta_msgchn_tta_step_graph(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap,
                               float w_sd, float w_sm, float w_cos, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && isc && ish, "tta_step_graph: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    PTTA_CHECK(st != nullptr, "tta_step_graph: needs a non-default stream (legacy stream 0 cannot be captured)");
    ptta_msgchn::GraphKey key;
    memset(&key, 0, sizeof(key));
    key.cap = cap; key.w_sd = w_sd; key.w_sm = w_sm; key.w_cos = w_cos;
    for (int c = 0; c < 3; ++c) { key.isc[c] = isc[c]; key.ish[c] = ish[c]; }
    // The captured step reads engine-owned staging buffers, so a caller may pass a fresh tensor every frame (the usual
    // `.to(device)` of a data loader) without re-capturing; a caller that writes its frames straight into "stage_image" /
    // "stage_sparse" (ptta_msgchn_get_tensor) and passes those pointers skips the copies.
    const size_t px = (size_t)e->Nu * e->Hu * e->Wu;
    if (image_raw != e->stage_img) PTTA_CUDA(cudaMemcpyAsync(e->stage_img, image_raw, 3 * px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (sparse != e->stage_sp) PTTA_CUDA(cudaMemcpyAsync(e->stage_sp, sparse, px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    image_raw = e->stage_img; sparse = e->stage_sp;
    if (e->graph_exec && memcmp(&key, &e->graph_key, sizeof(key)) != 0) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    if (!e->graph_exec) {
        // one eager step first: sets every cudaFuncAttribute (not capturable) and validates the arguments
        e->st = st;
        PTTA_TRY(e->tta_step(image_raw, isc, ish, sparse, cap, w_sd, w_sm, w_cos));
        PTTA_CUDA(cudaStreamSynchronize(st));
        // capture a second pass WITHOUT executing it
        cudaGraph_t graph = nullptr;
        PTTA_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        int rc = e->tta_step(image_raw, isc, ish, sparse, cap, w_sd, w_sm, w_cos);
        cudaError_t ce = cudaStreamEndCapture(st, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        PTTA_CHECK(ce == cudaSuccess, "graph capture failed: %s", cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&e->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        PTTA_CHECK(ce == cudaSuccess, "graph instantiate failed: %s", cudaGetErrorString(ce));
        memcpy(&e->graph_key, &key, sizeof(key));
        return 0;   // the eager step above WAS this call's step
    }
    PTTA_CUDA(cudaGraphLaunch(e->graph_exec, st));
    return 0;
}

int ptta_msgchn_init_step_graph(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse,
                                const float* ground_truth, float cap, float max_predict_depth, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && ground_truth && isc && ish, "init_step_graph: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    PTTA_CHECK(st != nullptr, "init_step_graph: needs a non-default stream (legacy stream 0 cannot be captured)");
    ptta_msgchn::GraphKey key; memset(&key, 0, sizeof(key));
    key.cap = cap; key.w_sd = max_predict_depth; key.w_sm = 1.f;        // w_sm = 1: stage 1
    for (int c = 0; c < 3; ++c) { key.isc[c] = isc[c]; key.ish[c] = ish[c]; }
    const size_t px = (size_t)e->Nu * e->Hu * e->Wu;
    if (image_raw != e->stage_img) PTTA_CUDA(cudaMemcpyAsync(e->stage_img, image_raw, 3 * px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (sparse != e->stage_sp) PTTA_CUDA(cudaMemcpyAsync(e->stage_sp, sparse, px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (ground_truth != e->stage_gt) PTTA_CUDA(cudaMemcpyAsync(e->stage_gt, ground_truth, px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return e->prep_step_graphed(key, st, [&]() { return e->init_step(e->stage_img, isc, ish, e->stage_sp, e->stage_gt, cap, max_predict_depth); });
}

int ptta_msgchn_head_step_graph(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap,
                                ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && isc && ish, "head_step_graph: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    PTTA_CHECK(st != nullptr, "head_step_graph: needs a non-default stream (legacy stream 0 cannot be captured)");
    ptta_msgchn::GraphKey key; memset(&key, 0, sizeof(key));
    key.cap = cap; key.w_sm = 2.f;                                       // w_sm = 2: stage 2
    for (int c = 0; c < 3; ++c) { key.isc[c] = isc[c]; key.ish[c] = ish[c]; }
    const size_t px = (size_t)e->Nu * e->Hu * e->Wu;
    if (image_raw != e->stage_img) PTTA_CUDA(cudaMemcpyAsync(e->stage_img, image_raw, 3 * px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (sparse != e->stage_sp) PTTA_CUDA(cudaMemcpyAsync(e->stage_sp, sparse, px * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return e->prep_step_graphed(key, st, [&]() { return e->head_step(e->stage_img, isc, ish, e->stage_sp, cap); });
}

int ptta_msgchn_get_tensor(ptta_msgchn* e, const char* name, void** ptr, int* dtype, long long* dims4) {
    PTTA_CHECK(e && name && ptr, "get_tensor: null argument");
    PTTA_CHECK(e->bound, "get_tensor: no workspace bound");
    auto it = e->named.find(name);
    PTTA_CHECK(it != e->named.end(), "get_tensor: unknown tensor '%s'", name);
    *ptr = it->second.p;
    if (dtype) *dtype = it->second.dtype;
    if (dims4) for (int k = 0; k < 4; ++k) dims4[k] = it->second.d[k];
    return 0;
}
int ptta_msgchn_num_tensors(const ptta_msgchn* e) { return e ? (int)e->named_order.size() : 0; }
const char* ptta_msgchn_tensor_name(const ptta_msgchn* e, int i) {
    return (e && i >= 0 && i < (int)e->named_order.size()) ? e->named_order[i].c_str() : nullptr;
}
long long ptta_msgchn_launch_count(const ptta_msgchn*) { return g_launches.load(); }

/* timing experiments only: one eager step with an event after every launch; prints "end_us stream kernel" lines to stdout */
int ptta_msgchn_trace_step(ptta_msgchn* e, const float* image_raw, const float* isc, const float* ish, const float* sparse, float cap,
                           float w_sd, float w_sm, float w_cos, ptta_stream_t stream) {
    PTTA_CHECK(e && image_raw && sparse && isc && ish, "trace_step: null argument");
    e->st = (cudaStream_t)stream;
    LaunchTrace tr; tr.cur = &e->st; tr.main = e->st;
    cudaEvent_t t0;
    PTTA_CUDA(cudaEventCreate(&t0));
    PTTA_CUDA(cudaStreamSynchronize(e->st));
    PTTA_CUDA(cudaEventRecord(t0, e->st));
    g_trace = &tr;
    int rc = e->tta_step(image_raw, isc, ish, sparse, cap, w_sd, w_sm, w_cos);
    g_trace = nullptr;
    PTTA_CUDA(cudaDeviceSynchronize());
    float prev[2] = {0.f, 0.f};
    for (size_t i = 0; i < tr.events.size(); ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t0, tr.events[i]);
        printf("%9.1f  s%d  +%7.1f  %s\n", ms * 1e3f, tr.streams[i], ms * 1e3f - prev[tr.streams[i]], tr.names[i].c_str());
        prev[tr.streams[i]] = ms * 1e3f;
        cudaEventDestroy(tr.events[i]);
    }
    fflush(stdout);
    cudaEventDestroy(t0);
    return rc;
}

}  // extern "C"
