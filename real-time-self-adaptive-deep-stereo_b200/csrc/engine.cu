// MADNet engine: forward, MAD / FULL backward and momentum update (see engine.h).
//
// Graph restated from the reference (never copied): pyramid encoder Nets/MadNet.py:173-249, per-level
// warp -> correlation -> 6-conv estimator loop :251-351, context network :122-171, outputs :68-71,:362-364;
// train-op structure Stereo_Online_Adaptation.py:87-128 (MAD: one module per step with gradients cut between
// levels by `bulkhead`; FULL: everything, gradients also flow through the up-sampled disparities).
#include <nvtx3/nvToolsExt.h>

#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace ms {

static const int PYR_CH[13] = {3, 16, 16, 32, 32, 64, 64, 96, 96, 128, 128, 192, 192};
static const int EST_CH[6] = {128, 128, 96, 64, 32, 1};
static const int CTX_CH[7] = {128, 128, 128, 96, 64, 32, 1};
static const int CTX_RATE[7] = {1, 2, 4, 8, 16, 1, 1};
static const float MAD_ALPHA = 0.2f;

static inline int pad4(int c) { return (c + 3) / 4 * 4; }
static inline int feat_of(int k) { return 2 * k; }
static inline int est_layer(int k, int j) { return 12 + (6 - k) * 6 + (j - 1); }
static inline int ctx_layer(int j) { return 42 + (j - 1); }

static void same_pad(int in, int k, int s, int d, int& out, int& before) {
    int keff = (k - 1) * d + 1;
    out = (in + s - 1) / s;
    int total = std::max((out - 1) * s + keff - in, 0);
    before = total / 2;
}

Engine::Engine()
    : net(0), B(1), H(0), W(0), Hp(0), Wp(0), radius_d(2), corr_stride(1), warping(1), n_groups(0), n_params(0),
      Wt(nullptr), Gr(nullptr), Mo(nullptr), ws(nullptr), ws_floats(0), bound(false), wT(nullptr), wT_floats(0),
      wg_ws(nullptr), wg_ws_floats(0), rs_tmp(nullptr), rs_tmp_floats(0), loss_ws(nullptr), loss_ws_floats(0),
      scalars(nullptr), gt(nullptr), proxy(nullptr), loss_kind(0), proxy_w_full(0.01f), proxy_w_module(0.1f), profiling(0), prof_capturing(false), prof_event_overhead_ms(0.f) {
    prof_reset();
    weights_dirty = true;
    gstream = nullptr; ev_in = nullptr; ev_out = nullptr;
    wstream = nullptr; ev_fork = nullptr; ev_join = nullptr; wstream_dirty = false;
    { const char* e8 = getenv("MS_WGRAD_OVERLAP"); use_overlap = (e8 && e8[0] == '0') ? 0 : 1; }
    { const char* e2 = getenv("MS_GRAPHS"); use_graphs = (e2 && e2[0] == '0') ? 0 : 1; }
    { const char* e5 = getenv("MS_HEADS"); use_heads = (e5 && e5[0] == '0') ? 0 : 1; }
    { const char* e7 = getenv("MS_STEM"); use_stem = (e7 && e7[0] == '0') ? 0 : 1; }
    { const char* e6 = getenv("MS_BF_WGRAD"); use_bf_wgrad = (e6 && e6[0] == '0') ? 0 : 1; }
    wg_xp.hi = wg_xp.lo = nullptr; wg_xp.cs = 0; wg_xp.fmt = 0; wg_xp.scale = 1.f; wg_xp_halfs = 0;
    act_scale = 0.f;
    bf_jobs_dev = nullptr; bf_max_total = 0; bf_part = nullptr; bf_tickets = nullptr; gemm_part = nullptr;
    dp_rank = 0; dp_world = 1; dp_connected = false; dp_xbuf = nullptr; dp_state = nullptr; dp_cap_floats = 0;
}

void Engine::add_planes(Bump& A, const TView& v, int fmt) {
    const bool sizing = A.base == nullptr;         // (sizing pass: pointers are null or null + a slice offset -- never dedupe)
    if (!sizing && planes.count(v.p)) return;
    ActPlanes pl;
    pl.fmt = fmt;
    pl.scale = fmt == 1 ? act_scale : 1.f;
    pl.cs = (v.c + 7) / 8 * 8;
    const size_t floats = (v.pixels() * pl.cs + 1) / 2;     // bf16 elements -> floats
    pl.hi = A.alloc(floats);
    pl.lo = A.alloc(floats);
    if (!sizing) planes[v.p] = pl;
}
const ActPlanes* Engine::planes_of(const TView& v) const {
    auto it = planes.find(v.p);
    if (it == planes.end() || !it->second.hi || it->second.cs < v.c) return nullptr;
    return &it->second;
}
int Engine::ensure_planes(const TView& v, cudaStream_t st) {
    if (fresh.count(v.p)) return 0;
    const ActPlanes* pl = planes_of(v);
    MS_REQUIRE(pl != nullptr, "ensure_planes: tensor has no bf16 planes");
    if (split_planes(v, *pl, st)) return -1;
    fresh.insert(v.p);
    return 0;
}

void Engine::prof_reset() {
    for (int i = 0; i < N_CAT; ++i) { cat_ms[i] = 0; cat_macs[i] = 0; cat_bytes[i] = 0; cat_calls[i] = 0; }
    for (int d = 0; d < 3; ++d) { layer_ms[d].assign(layers.size(), 0.0); layer_calls[d].assign(layers.size(), 0); }
}
void Engine::prof_begin(int cat, cudaStream_t st, int layer) {
    if (!profiling || (profiling == 2 && !prof_capturing)) return;
    Span s; s.cat = cat; s.layer = layer; s.macs = 0; s.bytes = 0;
    for (cudaEvent_t* e : {&s.a, &s.b}) {
        if (!event_pool.empty()) { *e = event_pool.back(); event_pool.pop_back(); }
        else cudaEventCreate(e);
    }
    // inside a stream capture the record becomes an EXTERNAL event node: it fires at every replay of the graph
    if (prof_capturing) cudaEventRecordWithFlags(s.a, st, cudaEventRecordExternal);
    else cudaEventRecord(s.a, st);
    spans.push_back(s);
}
void Engine::prof_end(cudaStream_t st) {
    if (!profiling || spans.empty() || (profiling == 2 && !prof_capturing)) return;
    if (prof_capturing) cudaEventRecordWithFlags(spans.back().b, st, cudaEventRecordExternal);
    else cudaEventRecord(spans.back().b, st);
}
void Engine::prof_note(double macs, double bytes) {
    if (!profiling || spans.empty() || (profiling == 2 && !prof_capturing)) return;
    spans.back().macs += macs; spans.back().bytes += bytes;
}
int Engine::prof_fold(std::vector<Span>& v, bool recycle) {
    // an EMPTY span (two back-to-back event records, cat < 0) calibrates what the event nodes themselves cost inside a
    // graph; it is subtracted from every span of the same replay
    float t0 = 0.f;
    for (auto& s : v)
        if (s.cat < 0) {
            MS_CHECK_CUDA(cudaEventSynchronize(s.b));
            MS_CHECK_CUDA(cudaEventElapsedTime(&t0, s.a, s.b));
            prof_event_overhead_ms = t0;
        }
    for (auto& s : v) {
        if (s.cat < 0) { if (recycle) { event_pool.push_back(s.a); event_pool.push_back(s.b); } continue; }
        MS_CHECK_CUDA(cudaEventSynchronize(s.b));
        float ms = 0.f;
        MS_CHECK_CUDA(cudaEventElapsedTime(&ms, s.a, s.b));
        ms = ms > t0 ? ms - t0 : 0.f;
        cat_ms[s.cat] += ms; cat_calls[s.cat] += 1; cat_macs[s.cat] += s.macs; cat_bytes[s.cat] += s.bytes;
        if (s.layer >= 0 && s.cat <= CAT_CONV_WGRAD && s.layer < (int)layer_ms[s.cat].size()) {
            layer_ms[s.cat][s.layer] += ms; layer_calls[s.cat][s.layer] += 1;
        }
        if (recycle) { event_pool.push_back(s.a); event_pool.push_back(s.b); }
    }
    if (recycle) v.clear();
    return 0;
}
int Engine::prof_collect() { return prof_fold(spans, true); }

int Engine::build_madnet() {
    layers.clear();
    char buf[128];
    for (int i = 1; i <= 12; ++i) {
        ConvLayer L;
        snprintf(buf, sizeof buf, "left/conv%d", i); L.name = buf;
        snprintf(buf, sizeof buf, "model/gc-read-pyramid/conv%d", i); L.scope = buf;
        L.bname = "biases";
        L.kh = L.kw = 3; L.cin = PYR_CH[i - 1]; L.cout = PYR_CH[i]; L.stride = (i % 2) ? 2 : 1; L.dil = 1;
        L.alpha = MAD_ALPHA; L.transposed = 0; L.group = -1; L.w_off = L.b_off = 0;
        layers.push_back(L);
    }
    const int nd = (2 * radius_d) / corr_stride + 1;
    for (int k = 6; k >= 2; --k) {
        int cin = PYR_CH[feat_of(k)] + nd + (k < 6 ? 1 : 0);
        for (int j = 1; j <= 6; ++j) {
            ConvLayer L;
            snprintf(buf, sizeof buf, "fgc-volume-filtering-%d/disp%d", k, j); L.name = buf;
            snprintf(buf, sizeof buf, "model/G%d/fgc-volume-filtering-%d/disp-%d", k, k, j); L.scope = buf;
            L.bname = "biases";
            L.kh = L.kw = 3; L.cin = cin; L.cout = EST_CH[j - 1]; L.stride = 1; L.dil = 1;
            L.alpha = j < 6 ? MAD_ALPHA : 1.f; L.transposed = 0; L.group = -1; L.w_off = L.b_off = 0;
            layers.push_back(L);
            cin = L.cout;
        }
    }
    int cin = PYR_CH[4] + 1;
    for (int j = 1; j <= 7; ++j) {
        ConvLayer L;
        snprintf(buf, sizeof buf, "context%d", j); L.name = buf;
        snprintf(buf, sizeof buf, "model/context-%d", j); L.scope = buf;
        L.bname = "biases";
        L.kh = L.kw = 3; L.cin = cin; L.cout = CTX_CH[j - 1]; L.stride = 1; L.dil = CTX_RATE[j - 1];
        L.alpha = j < 7 ? MAD_ALPHA : 1.f; L.transposed = 0; L.group = -1; L.w_off = L.b_off = 0;
        layers.push_back(L);
        cin = L.cout;
    }
    return 0;
}

int Engine::finalize_groups(const int* group_of_layer, int ng) {
    n_groups = ng;
    for (size_t i = 0; i < layers.size(); ++i) {
        int g = group_of_layer ? group_of_layer[i] : -1;
        MS_REQUIRE(g >= -1 && g < ng, "finalize_groups: group index out of range");
        layers[i].group = g;
    }
    group_begin.assign(ng, 0);
    group_end.assign(ng, 0);
    size_t off = 0;
    auto place = [&](ConvLayer& L) {
        L.w_off = off; off += (size_t)L.kh * L.kw * L.cin * L.cout; off = (off + 3) / 4 * 4;
        L.b_off = off; off += (size_t)L.cout; off = (off + 3) / 4 * 4;
    };
    for (int g = 0; g < ng; ++g) {
        group_begin[g] = off;
        for (auto& L : layers) if (L.group == g) place(L);
        group_end[g] = off;
    }
    for (auto& L : layers) if (L.group < 0) place(L);
    n_params = off;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// workspace layout
// ---------------------------------------------------------------------------------------------
size_t Engine::layout(float* base) {
    Bump A{base, 0};
    auto alloc = [&](size_t n) -> float* { return A.alloc(n); };
    auto tens = [&](int n, int h, int w, int c, int cs = 0) { return A.tens(n, h, w, c, cs); };
    tensors.clear();
    planes.clear(); fresh.clear();
    char nm[128];
    const int nd = (2 * radius_d) / corr_stride + 1;
    TView raw_l = tens(B, H, W, 3), raw_r = tens(B, H, W, 3);
    tensors["raw_left"] = raw_l; tensors["raw_right"] = raw_r;
    img = tens(2 * B, Hp, Wp, 3, 4);
    tensors["img"] = img;
    if (net == 1) add_planes(A, img, 1);           // DispNet's 7x7 stem runs on the tensor cores
    size_t max_wg = 0, max_wt = 0;
    auto track = [&](const ConvLayer& L, size_t pixels) {
        max_wg = std::max(max_wg, conv_wgrad_workspace_floats(L.kh * L.kw, L.cin, L.cout, pixels));
        if (L.stride == 1 && L.cout <= 192)   // tcgen05 wgrad: NCHW copy of dY + <=64 split partials + bias partials
            max_wg = std::max(max_wg, pixels * L.cout + 64 * (size_t)L.kh * L.kw * L.cin * L.cout + 128 * (size_t)L.cout + 8192);
        max_wt = std::max(max_wt, (size_t)L.kh * L.kw * L.cin * L.cout);
        if (L.cout == 1) max_wg = std::max(max_wg, (size_t)2 * 148 * ((size_t)L.kh * L.kw * L.cin + 1));    // conv_head_wgrad partials
        if (!L.transposed && L.cin >= 3 && L.cout >= 16) {
            max_wg = std::max(max_wg, std::min<size_t>(wgrad_bf_workspace_floats(L.kh, L.kw, L.cin, L.cout), (size_t)48 << 20));
            wg_xp_halfs = std::max(wg_xp_halfs, pixels * L.stride * L.stride * (size_t)((L.cin + 7) / 8 * 8));
        }
    };
    wg_xp_halfs = 0;
    if (net == 1) {
        layout_dispnet(A, max_wg, max_wt);
    } else {
    int h = Hp, w = Wp;
    for (int i = 1; i <= 12; ++i) {
        if (i % 2) { h = (h + 1) / 2; w = (w + 1) / 2; }
        pyr[i] = tens(2 * B, h, w, PYR_CH[i]);
        g_pyr[i] = tens(2 * B, h, w, PYR_CH[i]);
        add_planes(A, pyr[i], 1); add_planes(A, g_pyr[i], 0);
        track(layers[i - 1], (size_t)2 * B * h * w);
        snprintf(nm, sizeof nm, "left/conv%d", i); tensors[nm] = batch(pyr[i], 0, B);
        snprintf(nm, sizeof nm, "right/conv%d", i); tensors[nm] = batch(pyr[i], B, B);
        snprintf(nm, sizeof nm, "grad/left/conv%d", i); tensors[nm] = batch(g_pyr[i], 0, B);
        snprintf(nm, sizeof nm, "grad/right/conv%d", i); tensors[nm] = batch(g_pyr[i], B, B);
    }
    ctxin = tens(B, pyr[4].h, pyr[4].w, PYR_CH[4] + 1, pad4(PYR_CH[4] + 1));
    g_ctxin = tens(B, pyr[4].h, pyr[4].w, PYR_CH[4] + 1, pad4(PYR_CH[4] + 1));
    tensors["ctxin"] = ctxin; tensors["grad/ctxin"] = g_ctxin;
    add_planes(A, ctxin, 1);
    for (int k = 6; k >= 2; --k) {
        const int f = feat_of(k), C = PYR_CH[f];
        const int hh = pyr[f].h, ww = pyr[f].w;
        const int ct = C + nd + (k < 6 ? 1 : 0);
        cost[k] = tens(B, hh, ww, ct, pad4(ct));
        g_cost[k] = tens(B, hh, ww, ct, pad4(ct));
        add_planes(A, cost[k], 1);
        snprintf(nm, sizeof nm, "cost%d", k); tensors[nm] = cost[k];
        snprintf(nm, sizeof nm, "grad/cost%d", k); tensors[nm] = g_cost[k];
        for (int j = 1; j <= 5; ++j) {
            est[k][j] = tens(B, hh, ww, EST_CH[j - 1]);
            g_est[k][j] = tens(B, hh, ww, EST_CH[j - 1]);
            add_planes(A, est[k][j], 1); add_planes(A, g_est[k][j], 0);
            snprintf(nm, sizeof nm, "fgc-volume-filtering-%d/disp%d", k, j); tensors[nm] = est[k][j];
            snprintf(nm, sizeof nm, "grad/fgc-volume-filtering-%d/disp%d", k, j); tensors[nm] = g_est[k][j];
        }
        if (k == 2) V[k] = slice(ctxin, PYR_CH[4], 1);
        else V[k] = tens(B, hh, ww, 1);
        g_V[k] = tens(B, hh, ww, 1);
        g_u[k] = tens(B, hh, ww, 1);
        snprintf(nm, sizeof nm, "fgc-volume-filtering-%d/disp6", k); tensors[nm] = V[k];
        snprintf(nm, sizeof nm, "grad/fgc-volume-filtering-%d/disp6", k); tensors[nm] = g_V[k];
        snprintf(nm, sizeof nm, "grad/u%d", k); tensors[nm] = g_u[k];
        for (int j = 1; j <= 6; ++j) track(layers[est_layer(k, j)], (size_t)B * hh * ww);
    }
    for (int j = 1; j <= 6; ++j) {
        ctx[j] = tens(B, pyr[4].h, pyr[4].w, CTX_CH[j - 1]);
        g_ctx[j] = tens(B, pyr[4].h, pyr[4].w, CTX_CH[j - 1]);
        add_planes(A, ctx[j], 1); add_planes(A, g_ctx[j], 0);
        snprintf(nm, sizeof nm, "context%d", j); tensors[nm] = ctx[j];
        snprintf(nm, sizeof nm, "grad/context%d", j); tensors[nm] = g_ctx[j];
    }
    for (int j = 1; j <= 7; ++j) track(layers[ctx_layer(j)], (size_t)B * pyr[4].h * pyr[4].w);
    final_ = tens(B, pyr[4].h, pyr[4].w, 1);
    g_final = tens(B, pyr[4].h, pyr[4].w, 1);
    tensors["final_disp"] = final_; tensors["grad/final_disp"] = g_final;
    }   // net == 0
    n_disp = net == 1 ? 7 : 6;
    for (int i = 0; i < n_disp; ++i) {
        disp[i] = tens(B, H, W, 1);
        snprintf(nm, sizeof nm, "disp%d", i); tensors[nm] = disp[i];
    }
    tensors["rescaled_prediction"] = disp[n_disp - 1];
    g_disp = tens(B, H, W, 1);
    tensors["grad/disp"] = g_disp;
    wT_floats = max_wt; wT = alloc(max_wt);
    wg_ws_floats = max_wg; wg_ws = alloc(max_wg);
    // split 16-bit weight tiles per layer and orientation (forward: fp16, dgrad: bf16) + their batched prep job table
    bfw[0].assign(layers.size(), BfW{nullptr, false});
    bfw[1].assign(layers.size(), BfW{nullptr, false});
    bf_jobs.clear(); bf_job_begin.assign(n_groups + 1, 0); bf_job_end.assign(n_groups + 1, 0);
    bf_max_total = 0;
    for (int gidx = 0; gidx <= n_groups; ++gidx) {
        bf_job_begin[gidx] = (int)bf_jobs.size();
        for (size_t li = 0; li < layers.size(); ++li) {
            const ConvLayer& L = layers[li];
            const int lg = L.group < 0 ? n_groups : L.group;
            // (MADNet's 3 -> 16 conv1 stays on its direct kernel; a 3-channel stem with a large filter -- DispNet conv1, 7x7 --
            //  is 2.3 GMAC and goes to the tensor cores with its K block zero-padded)
            const bool stem = L.cin >= 3 && L.cin < 8 && L.kh * L.kw >= 25 && L.cout >= 16;
            if (lg != gidx || (L.cin < 8 && !stem) || L.cout < 8 || L.kh * L.kw > 49 || L.stride > 2) continue;
            if (L.transposed) {
                // conv2d_transpose forward = fractionally strided gather: M = cout, K = cin, canonical W is already
                // [tap][cout][cin] = [tap][M][K]
                int Mpad, Kpad; conv_bf_weight_dims(L.cout, L.cin, Mpad, Kpad);
                const size_t halfs = conv_bf_weight_halfs(L.kh * L.kw, L.cout, L.cin);
                BfW t; t.ok = true;
                t.tiles = alloc((halfs + 1) / 2);
                bfw[0][li] = t;
                BfPrepJob j{base ? Wt + L.w_off : nullptr, t.tiles, L.kh * L.kw, L.cout, L.cin, Mpad, Kpad, 0, 1};
                bf_jobs.push_back(j);
                bf_max_total = std::max(bf_max_total, halfs);
                // its input gradient = the stride-2 conv of dY with the same filter read as HWIO [.,.,cout,cin]:
                // M = cin, K = cout, canonical W = [tap][K][M]; bf16 (gradient planes)
                conv_bf_weight_dims(L.cin, L.cout, Mpad, Kpad);
                const size_t halfs_d = conv_bf_weight_halfs(L.kh * L.kw, L.cin, L.cout);
                BfW td; td.ok = true;
                td.tiles = alloc((halfs_d + 1) / 2);
                bfw[1][li] = td;
                BfPrepJob jd{base ? Wt + L.w_off : nullptr, td.tiles, L.kh * L.kw, L.cin, L.cout, Mpad, Kpad, 1, 0};
                bf_jobs.push_back(jd);
                bf_max_total = std::max(bf_max_total, halfs_d);
                continue;
            }
            for (int dir = 0; dir < 2; ++dir) {
                if (dir == 1 && stem) continue;                  // no input gradient for the image
                const int M = dir == 0 ? L.cout : L.cin, K = dir == 0 ? L.cin : L.cout;
                int Mpad, Kpad; conv_bf_weight_dims(M, K, Mpad, Kpad);
                const size_t halfs = conv_bf_weight_halfs(L.kh * L.kw, M, K);
                BfW t; t.ok = true;
                t.tiles = alloc((halfs + 1) / 2);
                bfw[dir][li] = t;
                BfPrepJob j{base ? Wt + L.w_off : nullptr, t.tiles, L.kh * L.kw, M, K, Mpad, Kpad, dir == 0 ? 1 : 0, dir == 0 ? 1 : 0};
                bf_jobs.push_back(j);
                bf_max_total = std::max(bf_max_total, halfs);
            }
        }
        bf_job_end[gidx] = (int)bf_jobs.size();
    }
    if (wg_xp_halfs) {
        wg_xp.hi = alloc((wg_xp_halfs + 1) / 2); wg_xp.lo = alloc((wg_xp_halfs + 1) / 2); wg_xp.fmt = 0;
    }
    bf_part = alloc(conv_bf_part_floats());
    bf_tickets = reinterpret_cast<unsigned int*>(alloc(conv_bf_ticket_words()));
    bf_jobs_dev = reinterpret_cast<BfPrepJob*>(alloc((bf_jobs.size() + 1) * sizeof(BfPrepJob) / sizeof(float) + 16));
    gemm_part = alloc(conv_gemm_part_floats());
    rs_tmp_floats = (size_t)B * H * Wp; rs_tmp = alloc(rs_tmp_floats);
    loss_ws_floats = loss_workspace_floats(B, H, W); loss_ws = alloc(loss_ws_floats);
    scalars = alloc(64);
    u8_stage = reinterpret_cast<unsigned char*>(alloc(((size_t)2 * B * H * W * 3 + 3) / 4 + 64));
    gt = alloc((size_t)B * H * W);
    proxy = alloc((size_t)B * H * W);
    return A.off;
}

// ---------------------------------------------------------------------------------------------
// conv helpers
// ---------------------------------------------------------------------------------------------
int Engine::conv_fwd(const ConvLayer& L, const TView& x, const TView& y, const float* res, int res_cs,
                     cudaStream_t st) {
    ConvGemm p{};
    p.x = x; p.y = y; p.kh = L.kh; p.kw = L.kw;
    p.bias = Wt + L.b_off;
    p.alpha = L.alpha;
    p.res = res; p.res_cs = res_cs;
    p.mask = nullptr; p.mask_cs = 0; p.mask_alpha = 1.f; p.accumulate = 0;
    p.part = gemm_part; p.part_floats = conv_gemm_part_floats();
    int oh, ow, pt, pl;
    if (!L.transposed) {
        same_pad(x.h, L.kh, L.stride, L.dil, oh, pt);
        same_pad(x.w, L.kw, L.stride, L.dil, ow, pl);
        MS_REQUIRE(oh == y.h && ow == y.w && x.c == L.cin && y.c == L.cout, "conv_fwd: shape mismatch");
        p.wmat = Wt + L.w_off;
        p.mul = L.stride; p.off_y = -pt; p.off_x = -pl; p.step = L.dil; p.div = 1;
    } else {
        same_pad(y.h, L.kh, L.stride, 1, oh, pt);
        same_pad(y.w, L.kw, L.stride, 1, ow, pl);
        MS_REQUIRE(oh == x.h && ow == x.w && x.c == L.cin && y.c == L.cout, "conv_fwd(T): shape mismatch");
        p.wmat = wT;
        p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -1; p.div = L.stride;
        const int li_t = (int)(&L - &layers[0]);
        const bool bf_t = bfw[0][li_t].ok && conv_bf_supported(p) && planes_of(x);
        // canonical W is [tap][cout][cin]; the gather GEMM wants [tap][K=cin][N=cout] (the tensor-core path has its own tiles)
        if (!bf_t && transpose_taps(Wt + L.w_off, wT, L.kh * L.kw, L.cout, L.cin, st)) return -1;
    }
    const int li = (int)(&L - &layers[0]);
    prof_begin(CAT_CONV_FWD, st, li);
    int rc;
    const ActPlanes* xpl = (bfw[0][li].ok && conv_bf_supported(p)) ? planes_of(x) : nullptr;
    if (use_heads && conv_head_kind(p) == 1) {
        fresh.erase(y.p);
        rc = conv_head(p, st);
    } else if (use_heads && L.cin == 1 && L.cout == 1 && conv_one_channel_supported(p)) {
        fresh.erase(y.p);
        p.wmat = Wt + L.w_off;                       // [tap][1][1]: canonical weights serve either orientation
        rc = conv_one_channel(p, st);
    } else if (use_stem && !L.transposed && (p.wmat = Wt + L.w_off, conv_stem_fwd_supported(p))) {
        // DispNet conv1: 3 real channels per 32-wide K block on the tensor-core path; the CUDA cores do it in a third of the time
        const ActPlanes* ypl = planes_of(y);
        rc = conv_stem_fwd(p, ypl, st);
        if (ypl) fresh.insert(y.p); else fresh.erase(y.p);
    } else if (!L.transposed && L.cout <= 16 && conv_small_fwd_supported(p)) {
        // full-resolution 16-channel layers (conv2: 2 x 192 x 640 x 16): M = cout = 16 would waste 7/8 of the swap-AB
        // tile's TMEM lanes and epilogue threads (183 us on the split-16-bit path); the shared-memory tiled direct
        // kernel is bandwidth-shaped
        fresh.erase(y.p);
        rc = conv_small_fwd(p, st);
    } else if (xpl) {
        if (ensure_planes(x, st)) return -1;
        const ActPlanes* ypl = planes_of(y);
        rc = conv_bf(p, *xpl, bfw[0][li].tiles, ypl, bf_part, bf_tickets, st);
        if (ypl) fresh.insert(y.p);
    } else {
        fresh.erase(y.p);
        rc = conv_gemm(p, st);
    }
    prof_end(st);
    prof_note((double)y.pixels() * L.kh * L.kw * L.cin * L.cout / (L.transposed ? L.stride * L.stride : 1), 0);
    return rc;
}

// x: forward input of the layer; dpre: grad wrt pre-activation output; dx: where to write grad wrt x
int Engine::conv_bwd(const ConvLayer& L, const TView& x, const TView& dpre, const TView* dx, const TView* dx_mask,
                     float mask_alpha, int dx_acc, int want_wgrad, cudaStream_t st) {
    int oh, ow, pt, pl;
    MS_REQUIRE(!L.transposed, "conv_bwd: transposed layers use deconv_bwd");
    same_pad(x.h, L.kh, L.stride, L.dil, oh, pt);
    same_pad(x.w, L.kw, L.stride, L.dil, ow, pl);
    MS_REQUIRE(oh == dpre.h && ow == dpre.w && x.c == L.cin && dpre.c == L.cout, "conv_bwd: shape mismatch");
    if (net == 1) fresh.clear();    // DispNet's backward mutates gradient tensors in place between convs: always re-split
    if (want_wgrad) {
        ConvWgrad q{};
        q.x = x; q.dy = dpre; q.dw = Gr + L.w_off; q.db = Gr + L.b_off;
        q.kh = L.kh; q.kw = L.kw; q.stride = L.stride; q.dil = L.dil; q.pad_t = pt; q.pad_l = pl;
        q.workspace = wg_ws; q.workspace_floats = wg_ws_floats; q.accumulate = 0;
        prof_begin(CAT_CONV_WGRAD, st, (int)(&L - &layers[0]));
        int rc = 0;
        const bool stem_w = use_stem && conv_stem_wgrad_supported(q);
        const ActPlanes* wxp = (!stem_w && use_bf_wgrad && wgrad_bf_supported(q)) ? planes_of(x) : nullptr;
        const ActPlanes* wdp = wxp ? planes_of(dpre) : nullptr;
        // the planes of dpre also feed the dgrad below: they are produced on `st` BEFORE the fork
        if (wxp && wdp) rc = ensure_planes(dpre, st);
        cudaStream_t ws = st;
        if (!rc) rc = fork_wgrad(st, &ws);
        if (!rc && wxp && wdp) {
            // bf16 copy of the forward activation in scratch planes: kind::f16 MMAs reject f16 x bf16 operand pairs
            // (probed on sm_100a: illegal instruction), so the fp16 forward planes cannot serve here
            ActPlanes xb = wg_xp; xb.cs = (x.c + 7) / 8 * 8;
            MS_REQUIRE(xb.hi && x.pixels() * (size_t)xb.cs <= wg_xp_halfs, "conv_bwd: wgrad scratch planes too small");
            rc = split_planes(x, xb, ws);
            if (!rc) rc = wgrad_bf(q, xb, *wdp, ws);
        } else if (!rc && stem_w) {
            rc = conv_stem_wgrad(q, ws);                 // DispNet conv1
        } else if (!rc && use_heads && conv_head_wgrad_supported(q)) {
            rc = conv_head_wgrad(q, ws);                 // single-channel disparity heads
        } else if (!rc) {
            rc = wgrad_tc_supported(q) ? wgrad_tc(q, ws) : conv_wgrad(q, ws);
        }
        prof_end(st);
        prof_note((double)dpre.pixels() * L.kh * L.kw * L.cin * L.cout, 0);
        if (rc) return -1;
    }
    if (dx) {
        ConvGemm p{};
        p.x = dpre; p.wmat = wT; p.bias = nullptr; p.y = *dx; p.kh = L.kh; p.kw = L.kw;
        p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -L.dil; p.div = L.stride;
        p.alpha = 1.f;
        p.mask = dx_mask ? dx_mask->p : nullptr; p.mask_cs = dx_mask ? dx_mask->cs : 0; p.mask_alpha = mask_alpha;
        p.res = nullptr; p.res_cs = 0; p.accumulate = dx_acc;
        p.part = gemm_part; p.part_floats = conv_gemm_part_floats();
        const int li = (int)(&L - &layers[0]);
        prof_begin(CAT_CONV_DGRAD, st, li);
        int rc;
        const ActPlanes* xpl = (bfw[1][li].ok && conv_bf_supported(p)) ? planes_of(dpre) : nullptr;
        if (use_heads && L.cout == 1 && (p.wmat = Wt + L.w_off, conv_head_kind(p) == 2)) {
            fresh.erase(dx->p);
            rc = conv_head(p, st);          // [tap][cin][1] == [tap][1][cin]: the canonical weights serve directly
        } else if (xpl) {
            p.wmat = wT;
            rc = ensure_planes(dpre, st);
            const ActPlanes* ypl = planes_of(*dx);
            if (!rc) rc = conv_bf(p, *xpl, bfw[1][li].tiles, ypl, bf_part, bf_tickets, st);
            if (ypl) fresh.insert(dx->p);
        } else {
            p.wmat = wT;
            fresh.erase(dx->p);
            rc = transpose_taps(Wt + L.w_off, wT, L.kh * L.kw, L.cin, L.cout, st);   // -> [tap][cout][cin]
            if (!rc) rc = conv_gemm(p, st);
        }
        prof_end(st);
        prof_note((double)dpre.pixels() * L.kh * L.kw * L.cin * L.cout, 0);
        if (rc) return -1;
    }
    return 0;
}

bool Engine::trainable(int layer, int mode, int group) const {
    if (mode == 2) return true;
    if (mode == 1) return layers[layer].group == group;
    return false;
}

// ---------------------------------------------------------------------------------------------
// input / forward
// ---------------------------------------------------------------------------------------------
int Engine::set_input(const float* left, const float* right, cudaStream_t st) {
    MS_REQUIRE(bound, "engine not bound");
    TView rl = tensors["raw_left"], rr = tensors["raw_right"];
    size_t bytes = (size_t)B * H * W * 3 * sizeof(float);
    MS_CHECK_CUDA(cudaMemcpyAsync(rl.p, left, bytes, cudaMemcpyDefault, st));
    MS_CHECK_CUDA(cudaMemcpyAsync(rr.p, right, bytes, cudaMemcpyDefault, st));
    return 0;
}

// uint8 frames (host or device): 4x fewer bytes over PCIe than fp32; converted on the device
int Engine::set_input_u8(const unsigned char* left, const unsigned char* right, cudaStream_t st) {
    MS_REQUIRE(bound, "engine not bound");
    TView rl = tensors["raw_left"], rr = tensors["raw_right"];
    const size_t n = (size_t)B * H * W * 3;
    MS_REQUIRE((n & 3) == 0, "set_input_u8: B*H*W*3 must be a multiple of 4");
    MS_CHECK_CUDA(cudaMemcpyAsync(u8_stage, left, n, cudaMemcpyDefault, st));
    MS_CHECK_CUDA(cudaMemcpyAsync(u8_stage + n, right, n, cudaMemcpyDefault, st));
    if (u8_to_f32(u8_stage, rl.p, n, st)) return -1;
    return u8_to_f32(u8_stage + n, rr.p, n, st);
}

int Engine::prep_layers(int group, cudaStream_t st) {
    if (bf_jobs.empty()) return 0;
    int b, e;
    if (group < 0) { b = 0; e = (int)bf_jobs.size(); }
    else { b = bf_job_begin[group]; e = bf_job_end[group]; }
    return bf_prep_weights(bf_jobs_dev + b, e - b, bf_max_total, st);
}

int Engine::forward(int disp_mask, cudaStream_t st) {
    MS_REQUIRE(bound, "engine not bound");
    fresh.clear();
    const int nd = (2 * radius_d) / corr_stride + 1;
    {
        TView rl = tensors["raw_left"], rr = tensors["raw_right"];
        TView il = batch(img, 0, B), ir = batch(img, B, B);
        // DispNet normalises (x/255 - 100/255, Nets/DispNet.py:59-73); MADNet feeds raw 0..255 (Nets/MadNet.py:56-66)
        const float sc = net == 1 ? 1.f / 255.f : 1.f, bi = net == 1 ? -100.f / 255.f : 0.f;
        if (pad_reflect(rl.p, B, H, W, 3, il.p, Hp, Wp, img.cs, sc, bi, st)) return -1;
        if (pad_reflect(rr.p, B, H, W, 3, ir.p, Hp, Wp, img.cs, sc, bi, st)) return -1;
    }
    if (weights_dirty) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(st, &cs);
        MS_REQUIRE(cs == cudaStreamCaptureStatusNone, "forward: weights changed while capturing a graph");
        if (prep_layers(-1, st)) return -1;
        weights_dirty = false;
    }
    if (net == 1) return forward_dispnet(disp_mask, st);
    TView x = img;
    for (int i = 1; i <= 12; ++i) {
        if (conv_fwd(layers[i - 1], x, pyr[i], nullptr, 0, st)) return -1;
        x = pyr[i];
    }
    for (int k = 6; k >= 2; --k) {
        const int f = feat_of(k), C = PYR_CH[f];
        TView Lf = batch(pyr[f], 0, B), Rf = batch(pyr[f], B, B);
        const float* u = nullptr;
        if (k < 6) {
            TView us = slice(cost[k], C + nd, 1);
            if (resize_bilinear(V[k + 1].p, V[k + 1].cs, B, V[k + 1].h, V[k + 1].w, us.p, us.cs, cost[k].h, cost[k].w,
                                cost[k].h, cost[k].w, 1.f, 0, 20.f / (float)(1 << k), 0, st)) return -1;
            if (warping) u = us.p;
        }
        CorrFwd cf{};
        cf.left = Lf.p; cf.lcs = Lf.cs; cf.right = Rf.p; cf.rcs = Rf.cs;
        cf.u = u; cf.ucs = cost[k].cs;
        cf.out = cost[k].p; cf.ocs = cost[k].cs;
        cf.out2 = (k == 2) ? ctxin.p : nullptr; cf.o2cs = ctxin.cs;
        cf.B = B; cf.h = cost[k].h; cf.w = cost[k].w; cf.C = C; cf.max_disp = radius_d; cf.stride = corr_stride;
        cf.copy_left = 1; cf.u_chan = (k < 6) ? 1 : 0;
        prof_begin(CAT_CORR_FWD, st);
        int crc = corr_fwd(cf, st);
        prof_end(st);
        prof_note(0, (double)B * cf.h * cf.w * (3.0 * C + nd + (cf.u_chan ? 1 : 0) + (cf.out2 ? C : 0)) * 4.0);   // reads L, R(, u); writes corr + the left copy (fused concat)
        if (crc) return -1;
        TView xin = cost[k];
        for (int j = 1; j <= 6; ++j) {
            TView y = (j < 6) ? est[k][j] : V[k];
            if (conv_fwd(layers[est_layer(k, j)], xin, y, nullptr, 0, st)) return -1;
            xin = y;
        }
    }
    {
        TView xin = ctxin;
        for (int j = 1; j <= 7; ++j) {
            TView y = (j < 7) ? ctx[j] : final_;
            if (conv_fwd(layers[ctx_layer(j)], xin, y, j == 7 ? V[2].p : nullptr, V[2].cs, st)) return -1;
            xin = y;
        }
    }
    for (int i = 0; i < 6; ++i) {
        if (!(disp_mask & (1 << i))) continue;
        const TView& src = (i < 4) ? V[6 - i] : final_;
        if (i < 5) {
            if (resize_bilinear(src.p, src.cs, B, src.h, src.w, disp[i].p, 1, Hp, Wp, H, W, -20.f, 1, 1.f, 0, st)) return -1;
        } else {
            if (resize_bilinear(src.p, src.cs, B, src.h, src.w, disp[i].p, 1, Hp, Wp, H, W, 1.f, 0, -20.f, 1, st)) return -1;
        }
    }
    return 0;
}

int Engine::loss(int which, int with_grad, int slot, float grad_scale, cudaStream_t st) {
    MS_REQUIRE(bound && which >= 0 && which < n_disp && slot >= 0 && slot < 2, "loss: bad arguments");
    if (loss_kind == 1) {
        // Stereo_Continual_Adaptation.py:75 (full-resolution loss, weight 0.01; also the FULL train op :133) and :112
        // (module losses, weight 0.1)
        const float wgt = slot == 0 ? proxy_w_full : proxy_w_module;
        prof_begin(CAT_LOSS, st);
        int rc = proxy_loss(disp[which].p, proxy, B * H * W, wgt, grad_scale, scalars + slot, with_grad ? g_disp.p : nullptr, loss_ws, st);
        prof_end(st);
        return rc;
    }
    ReprojLoss p{};
    p.left = tensors["raw_left"].p; p.right = tensors["raw_right"].p;
    p.disp = disp[which].p; p.loss = scalars + slot;
    p.ddisp = with_grad ? g_disp.p : nullptr;
    p.workspace = loss_ws; p.B = B; p.H = H; p.W = W; p.grad_scale = grad_scale;
    prof_begin(CAT_LOSS, st);
    int rc = reproj_loss(p, st);
    prof_end(st);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// every weight-gradient launch of the backward pass goes to `wstream`, ordered after the point of `st` that produced its
// operands; they share one workspace, so they serialise among themselves while the dgrad chain proceeds on `st`
int Engine::fork_wgrad(cudaStream_t st, cudaStream_t* ws) {
    *ws = st;
    if (!use_overlap || profiling || net != 0) return 0;
    if (!wstream) {
        MS_CHECK_CUDA(cudaStreamCreateWithFlags(&wstream, cudaStreamNonBlocking));
        MS_CHECK_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        MS_CHECK_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    }
    MS_CHECK_CUDA(cudaEventRecord(ev_fork, st));
    MS_CHECK_CUDA(cudaStreamWaitEvent(wstream, ev_fork, 0));
    wstream_dirty = true;
    *ws = wstream;
    return 0;
}
int Engine::join_wgrad(cudaStream_t st) {
    if (!wstream_dirty) return 0;
    wstream_dirty = false;
    MS_CHECK_CUDA(cudaEventRecord(ev_join, wstream));
    MS_CHECK_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
    return 0;
}

int Engine::backward(int mode, int group, cudaStream_t st) {
    const int rc = backward_impl(mode, group, st);
    const int rj = join_wgrad(st);            // always: a captured side branch must be joined before the capture ends
    return rc ? rc : rj;
}

int Engine::backward_impl(int mode, int group, cudaStream_t st) {
    MS_REQUIRE(bound, "backward: engine not bound");
    if (net == 1) {
        // the reference cannot run MAD on DispNet either: 6 side predictions vs 5 groups trips the assert at
        // Stereo_Online_Adaptation.py:97
        MS_REQUIRE(mode == 2, "backward: DispNet supports FULL adaptation only");
        return backward_dispnet(st);
    }
    MS_REQUIRE(mode == 2 || (mode == 1 && group >= 0 && group < n_groups), "backward: bad mode/group");
    const int nd = (2 * radius_d) / corr_stride + 1;
    for (int i = 1; i <= 12; ++i) fresh.erase(g_pyr[i].p);     // gradient planes never survive from an earlier pass
    for (int k = 2; k <= 6; ++k) for (int j = 1; j <= 5; ++j) fresh.erase(g_est[k][j].p);
    for (int j = 1; j <= 6; ++j) fresh.erase(g_ctx[j].p);

    // lowest-index trainable pyramid conv (13 = none)
    int lo_pyr = 13;
    for (int i = 1; i <= 12; ++i) if (trainable(i - 1, mode, group)) { lo_pyr = i; break; }
    auto any_trainable = [&](int first, int last) {
        for (int i = first; i <= last; ++i) if (trainable(i, mode, group)) return true;
        return false;
    };

    // ---- estimator chain of level k: dpre(V_k) in g_V[k] -> (optionally) g_cost[k]
    auto est_bwd = [&](int k, bool need_cost_grad) -> int {
        TView dpre = g_V[k];
        for (int j = 6; j >= 1; --j) {
            const int li = est_layer(k, j);
            TView xin = (j == 1) ? cost[k] : est[k][j - 1];
            bool need_dx = (j > 1) ? (need_cost_grad || any_trainable(est_layer(k, 1), li - 1)) : need_cost_grad;
            TView dx = (j > 1) ? g_est[k][j - 1] : g_cost[k];
            TView mask = (j > 1) ? est[k][j - 1] : cost[k];
            if (conv_bwd(layers[li], xin, dpre, need_dx ? &dx : nullptr, (j > 1) ? &mask : nullptr, MAD_ALPHA, 0,
                         trainable(li, mode, group), st)) return -1;
            if (!need_dx) break;
            dpre = dx;
        }
        return 0;
    };
    // ---- context chain: g_final -> g_ctxin
    auto ctx_bwd = [&](bool need_in_grad) -> int {
        TView dpre = g_final;
        for (int j = 7; j >= 1; --j) {
            const int li = ctx_layer(j);
            TView xin = (j == 1) ? ctxin : ctx[j - 1];
            bool need_dx = (j > 1) ? (need_in_grad || any_trainable(ctx_layer(1), li - 1)) : need_in_grad;
            TView dx = (j > 1) ? g_ctx[j - 1] : g_ctxin;
            TView mask = (j > 1) ? ctx[j - 1] : ctxin;
            if (conv_bwd(layers[li], xin, dpre, need_dx ? &dx : nullptr, (j > 1) ? &mask : nullptr, MAD_ALPHA, 0,
                         trainable(li, mode, group), st)) return -1;
            if (!need_dx) break;
            dpre = dx;
        }
        return 0;
    };
    // ---- correlation + warp backward of level k -> g_pyr[f] (left|right halves), optional g_u[k]
    auto corr_level_bwd = [&](int k, bool want_du) -> int {
        const int f = feat_of(k), C = PYR_CH[f];
        TView Lf = batch(pyr[f], 0, B), Rf = batch(pyr[f], B, B);
        TView dL = batch(g_pyr[f], 0, B), dR = batch(g_pyr[f], B, B);
        CorrBwd cb{};
        cb.left = Lf.p; cb.lcs = Lf.cs; cb.right = Rf.p; cb.rcs = Rf.cs;
        cb.u = (k < 6 && warping) ? slice(cost[k], C + nd, 1).p : nullptr; cb.ucs = cost[k].cs;
        cb.dcost = g_cost[k].p; cb.dcs = g_cost[k].cs;
        cb.dleft = dL.p; cb.dlcs = dL.cs; cb.dright = dR.p; cb.drcs = dR.cs;
        cb.du = (want_du && cb.u) ? g_u[k].p : nullptr; cb.ducs = 1;
        cb.B = B; cb.h = cost[k].h; cb.w = cost[k].w; cb.C = C; cb.max_disp = radius_d; cb.stride = corr_stride;
        cb.add_left_slice = 1; cb.acc_left = 0; cb.acc_right = 0; cb.gcoff = -1;
        fresh.erase(g_pyr[f].p);
        prof_begin(CAT_CORR_BWD, st);
        int crc = corr_bwd(cb, st);
        prof_end(st);
        prof_note(0, (double)B * cb.h * cb.w * (4.0 * C + nd) * 4.0);
        return crc;
    };
    // ---- pyramid: g_pyr[top] holds d(post-activation output of conv `top`), complete
    auto pyr_bwd = [&](int top, int lo, bool accumulate_feats) -> int {
        if (lo > top) return 0;
        fresh.erase(g_pyr[top].p);
        if (leaky_bwd(g_pyr[top].p, g_pyr[top].cs, pyr[top].p, pyr[top].cs, g_pyr[top].pixels(), g_pyr[top].c,
                      MAD_ALPHA, st)) return -1;
        for (int i = top; i >= lo; --i) {
            TView xin = (i > 1) ? pyr[i - 1] : img;
            bool need_dx = i > lo;
            int acc = 0;
            if (need_dx && accumulate_feats && (i - 1) >= 4 && ((i - 1) % 2 == 0)) acc = 1;
            TView dx = g_pyr[i > 1 ? i - 1 : 1];
            TView mask = pyr[i > 1 ? i - 1 : 1];
            if (conv_bwd(layers[i - 1], xin, g_pyr[i], need_dx ? &dx : nullptr, need_dx ? &mask : nullptr, MAD_ALPHA,
                         acc, trainable(i - 1, mode, group), st)) return -1;
        }
        return 0;
    };
    auto ctx_tail = [&]() -> int {   // g_V[2] = g_final + g_ctxin[...,32]
        if (add_channels(g_V[2].p, 1, g_final.p, 1, g_final.pixels(), 1, 1.f, 0, st)) return -1;
        return add_channels(g_V[2].p, 1, g_ctxin.p + PYR_CH[4], g_ctxin.cs, g_final.pixels(), 1, 1.f, 1, st);
    };
    auto ctx_feat = [&]() -> int {   // g_pyr[4].left += g_ctxin[..., :32]
        TView dL = batch(g_pyr[4], 0, B);
        fresh.erase(g_pyr[4].p);
        return add_channels(dL.p, dL.cs, g_ctxin.p, g_ctxin.cs, dL.pixels(), PYR_CH[4], 1.f, 1, st);
    };

    if (mode == 1) {
        const int k = 6 - group;   // seed: disparity `group` of get_disparities() (D6,D5,D4,D3,D2ctx)
        MS_REQUIRE(k >= 2 && k <= 6, "backward(MAD): group has no disparity head");
        const int f = feat_of(k);
        const bool need_feat = lo_pyr <= f;
        const TView& head = (k == 2) ? final_ : V[k];
        TView& ghead = (k == 2) ? g_final : g_V[k];
        if (resize_bilinear_bwd(g_disp.p, 1, head.p, head.cs, B, head.h, head.w, ghead.p, 1, Hp, Wp, H, W, -20.f, 1,
                                1.f, 0, 0, rs_tmp, st)) return -1;
        if (k == 2) {
            bool est_train = any_trainable(est_layer(2, 1), est_layer(2, 6));
            if (ctx_bwd(need_feat || est_train)) return -1;
            if (need_feat || est_train) { if (ctx_tail()) return -1; }
            else return 0;
        }
        if (est_bwd(k, need_feat)) return -1;
        if (!need_feat) return 0;
        if (corr_level_bwd(k, false)) return -1;
        if (k == 2 && ctx_feat()) return -1;
        return pyr_bwd(f, lo_pyr, false);
    }

    // ---- FULL: loss on disp[5] = relu(resize(final)*-20)
    if (resize_bilinear_bwd(g_disp.p, 1, final_.p, final_.cs, B, final_.h, final_.w, g_final.p, 1, Hp, Wp, H, W, 1.f, 0,
                            -20.f, 1, 0, rs_tmp, st)) return -1;
    if (ctx_bwd(true)) return -1;
    if (ctx_tail()) return -1;
    for (int k = 2; k <= 6; ++k) {
        const int f = feat_of(k), C = PYR_CH[f];
        if (est_bwd(k, true)) return -1;
        if (corr_level_bwd(k, true)) return -1;
        if (k == 2 && ctx_feat()) return -1;
        if (k < 6) {
            // d u_k = warp-coordinate grad (if warping) + estimator-input slice
            const int acc = warping ? 1 : 0;
            if (add_channels(g_u[k].p, 1, g_cost[k].p + C + nd, g_cost[k].cs, g_u[k].pixels(), 1, 1.f, acc, st)) return -1;
            if (resize_bilinear_bwd(g_u[k].p, 1, V[k + 1].p, V[k + 1].cs, B, V[k + 1].h, V[k + 1].w, g_V[k + 1].p, 1,
                                    cost[k].h, cost[k].w, cost[k].h, cost[k].w, 1.f, 0, 20.f / (float)(1 << k), 0, 0,
                                    rs_tmp, st)) return -1;
        }
    }
    return pyr_bwd(12, 1, true);
}

int Engine::update(int group, float lr, float mu, float gscale, cudaStream_t st) {
    MS_REQUIRE(bound, "engine not bound");
    size_t b = 0, e = n_params;
    if (group >= 0) { MS_REQUIRE(group < n_groups, "update: bad group"); b = group_begin[group]; e = group_end[group]; }
    if (momentum_update(Wt + b, Gr + b, Mo + b, e - b, lr, mu, gscale, st)) return -1;
    return prep_layers(group, st);      // refresh the 16-bit weight tiles of exactly the weights that moved
}

// forward + losses + backward (+ update) as one sequence; replayed as a CUDA graph after the first call
int Engine::run_eager(int mode, int group, int disp_mask, int with_update, float lr, float mu, float gscale,
                      cudaStream_t st) {
    const int full = n_disp - 1;
    int mask = disp_mask | (1 << full);
    if (mode == 1) mask |= 1 << group;
    // NVTX ranges (SURVEY section 5: tracing): visible in nsys / ncu timelines, free when no tool is attached
    struct Range { explicit Range(const char* n) { nvtxRangePushA(n); } ~Range() { nvtxRangePop(); } };
    { Range r("madstereo/forward"); if (forward(mask, st)) return -1; }
    { Range r("madstereo/loss_full"); if (loss(full, mode == 2, 0, 1.f, st)) return -1; }
    if (mode == 1) {
        { Range r("madstereo/loss_module"); if (loss(group, 1, 1, 1.f, st)) return -1; }
        { Range r("madstereo/backward_mad"); if (backward(1, group, st)) return -1; }
        Range r("madstereo/update");
        if (with_update == 1 && update(group, lr, mu, gscale, st)) return -1;
        if (with_update == 2 && dp_update(group, lr, mu, st)) return -1;       // all-reduce over peer memory + update
    } else if (mode == 2) {
        { Range r("madstereo/backward_full"); if (backward(2, 0, st)) return -1; }
        Range r("madstereo/update");
        if (with_update == 1 && update(-1, lr, mu, gscale, st)) return -1;
        if (with_update == 2 && dp_update(-1, lr, mu, st)) return -1;
    }
    return 0;
}

int Engine::run(int mode, int group, int disp_mask, int with_update, float lr, float mu, float gscale, cudaStream_t st) {
    MS_REQUIRE(bound, "engine not bound");
    MS_REQUIRE(mode == 0 || mode == 2 || (mode == 1 && group >= 0 && group < n_groups), "run: bad mode/group");
    if (!use_graphs || profiling == 1) return run_eager(mode, group, disp_mask, with_update, lr, mu, gscale, st);
    if (weights_dirty) {                    // load / restore happened: refresh every weight tile outside the graph
        if (prep_layers(-1, st)) return -1;
        weights_dirty = false;
    }
    if (!gstream) {
        MS_CHECK_CUDA(cudaStreamCreateWithFlags(&gstream, cudaStreamNonBlocking));
        MS_CHECK_CUDA(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
        MS_CHECK_CUDA(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
    }
    GraphKey key;
    memset(&key, 0, sizeof key);
    key.mode = mode; key.group = mode == 1 ? group : 0; key.mask = disp_mask; key.with_update = with_update;
    key.lr = lr; key.mu = mu; key.gs = gscale; key.prof = profiling == 2 ? 1 : 0;
    auto it = graphs.find(key);
    if (it == graphs.end()) {
        if (conv_bf_init() || wgrad_bf_init() || corr_init() || wgrad_tc_init()) return -1;
        cudaGraph_t graph = nullptr;
        const long long l0 = launch_count();
        if (profiling == 2) { if (prof_collect()) return -1; }
        MS_CHECK_CUDA(cudaStreamBeginCapture(gstream, cudaStreamCaptureModeThreadLocal));
        prof_capturing = profiling == 2;
        pdl_set_suppressed(prof_capturing);
        if (prof_capturing) { prof_begin(-1, gstream); prof_end(gstream); }      // calibration span (see prof_fold)
        int rc = run_eager(mode, group, disp_mask, with_update, lr, mu, gscale, gstream);
        prof_capturing = false;
        pdl_set_suppressed(false);
        cudaError_t ce = cudaStreamEndCapture(gstream, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); spans.clear(); return rc; }
        MS_CHECK_CUDA(ce);
        cudaGraphExec_t exec = nullptr;
        MS_CHECK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
        cudaGraphDestroy(graph);
        GraphRec rec{exec, launch_count() - l0, nullptr};
        if (profiling == 2) { rec.spans = new std::vector<Span>(spans); spans.clear(); }
        add_launches(-rec.kernels);            // counted again at every replay below
        it = graphs.emplace(key, rec).first;
    }
    // order: caller's stream -> private stream (graph) -> caller's stream
    MS_CHECK_CUDA(cudaEventRecord(ev_in, st));
    MS_CHECK_CUDA(cudaStreamWaitEvent(gstream, ev_in, 0));
    MS_CHECK_CUDA(cudaGraphLaunch(it->second.exec, gstream));
    add_launches(it->second.kernels);
    MS_CHECK_CUDA(cudaEventRecord(ev_out, gstream));
    MS_CHECK_CUDA(cudaStreamWaitEvent(st, ev_out, 0));
    if (profiling == 2 && it->second.spans) {        // in-graph timing: read the event nodes of THIS replay
        MS_CHECK_CUDA(cudaStreamSynchronize(gstream));
        if (prof_fold(*it->second.spans, false)) return -1;
    }
    return 0;
}

}  // namespace ms
