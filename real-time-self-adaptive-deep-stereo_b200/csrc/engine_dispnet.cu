// DispNet-C schedule for the engine: forward and FULL backward (see engine.h).
//
// Graph restated from the reference (never copied): Nets/DispNet.py:75-152 (_build_network, correlation=True),
// :45-57 (_upsampling_block: deconv 4x4 s2, predict 3x3 -> 1, up_predict 4x4 s2 1 -> 1, concat 3x3 linear),
// :39-43 (_make_disp), :59-73 (input normalisation), MAX_DISP=40 (:7).  conv2d default activation = leaky 0.1
// (Nets/sharedLayers.py:54).  MAD is not defined for DispNet in the reference (assert at
// Stereo_Online_Adaptation.py:97), so only NONE / FULL exist here.
#include <algorithm>

#include "engine.h"

namespace ms {

static const float DN_ALPHA = 0.1f;
static const int DN_MAXD = 40;
struct EncSpec { const char* scope; const char* name; int k, cin, cout, stride; };
static const EncSpec DN_ENC[11] = {
    {"conv1", "conv1a", 7, 3, 64, 2},        {"conv2", "conv2a", 5, 64, 128, 2},     {"conv_redir", "conv_redir", 1, 128, 64, 1},
    {"conv3", "conv3", 5, 145, 256, 2},      {"conv3/1", "conv3/1", 3, 256, 256, 1}, {"conv4", "conv4", 3, 256, 512, 2},
    {"conv4/1", "conv4/1", 3, 512, 512, 1},  {"conv5", "conv5", 3, 512, 512, 2},     {"conv5/1", "conv5/1", 3, 512, 512, 1},
    {"conv6", "conv6", 3, 512, 1024, 2},     {"conv6/1", "conv6/1", 3, 1024, 1024, 1}};
struct UpSpec { const char* name; int cin, cout, skip; };
static const UpSpec DN_UP[5] = {{"up5", 1024, 512, 512}, {"up4", 512, 256, 512}, {"up3", 256, 128, 256},
                                {"up2", 128, 64, 128},   {"up1", 64, 32, 64}};
static inline int up_layer(int u, int j) { return 11 + 4 * u + j; }   // j: 0 deconv, 1 predict, 2 up_predict, 3 concat
static const int DN_PRED = 31;
static inline int pad4i(int c) { return (c + 3) / 4 * 4; }

int Engine::build_dispnet() {
    layers.clear();
    auto add = [&](const std::string& name, const std::string& scope, int k, int cin, int cout, int stride, float alpha,
                   int transposed) {
        ConvLayer L;
        L.name = name; L.scope = "model/" + scope; L.bname = "bias";
        L.kh = L.kw = k; L.cin = cin; L.cout = cout; L.stride = stride; L.dil = 1; L.alpha = alpha;
        L.transposed = transposed; L.group = -1; L.w_off = L.b_off = 0;
        layers.push_back(L);
    };
    for (const auto& e : DN_ENC) add(e.name, e.scope, e.k, e.cin, e.cout, e.stride, DN_ALPHA, 0);
    for (const auto& u : DN_UP) {
        std::string n(u.name);
        add(n + "/deconv", n + "/deconv", 4, u.cin, u.cout, 2, DN_ALPHA, 1);
        add(n + "/predict", n + "/predict", 3, u.cin, 1, 1, 1.f, 0);
        add(n + "/up_predict", n + "/up_predict", 4, 1, 1, 2, 1.f, 1);
        add(n + "/concat", n + "/concat", 3, u.cout + u.skip + 1, u.cout, 1, 1.f, 0);
    }
    add("prediction", "prediction", 3, 32, 1, 1, 1.f, 0);
    radius_d = DN_MAXD; corr_stride = 1; warping = 0;
    return 0;
}

void Engine::layout_dispnet(Bump& A, size_t& max_wg, size_t& max_wt) {
    auto track = [&](const ConvLayer& L, size_t pixels) {
        max_wg = std::max(max_wg, conv_wgrad_workspace_floats(L.kh * L.kw, L.cin, L.cout, pixels));
        max_wg = std::max(max_wg, conv_wgrad_workspace_floats(L.kh * L.kw, L.cout, L.cin, pixels));
        max_wt = std::max(max_wt, (size_t)L.kh * L.kw * L.cin * L.cout);
        if (L.cout == 1) max_wg = std::max(max_wg, (size_t)2 * 148 * ((size_t)L.kh * L.kw * L.cin + 1));    // conv_head_wgrad partials
        if (L.kh == 7 && L.cin == 3 && L.cout == 64) max_wg = std::max(max_wg, (size_t)2 * 148 * (147 * 64 + 64));   // conv_stem_wgrad partials
        if (!L.transposed && L.cin >= 3 && L.cout >= 16) {
            max_wg = std::max(max_wg, std::min<size_t>(wgrad_bf_workspace_floats(L.kh, L.kw, L.cin, L.cout), (size_t)48 << 20));
            wg_xp_halfs = std::max(wg_xp_halfs, pixels * L.stride * L.stride * (size_t)((L.cin + 7) / 8 * 8));
        }
        if (L.transposed && L.cin >= 16 && L.cout >= 8) {
            // conv2d_transpose: its weight gradient is the wgrad of the stride-2 conv big map (cout) -> small map (cin);
            // `pixels` counts the big map, the bf16 scratch copy is of the small one (the layer's forward input)
            max_wg = std::max(max_wg, std::min<size_t>(wgrad_bf_workspace_floats(L.kh, L.kw, L.cout, L.cin), (size_t)48 << 20));
            wg_xp_halfs = std::max(wg_xp_halfs, pixels / (L.stride * L.stride) * (size_t)((L.cin + 7) / 8 * 8));
        }
        if (L.stride == 1 && !L.transposed && L.cout <= 192)
            max_wg = std::max(max_wg, pixels * L.cout + 64 * (size_t)L.kh * L.kw * L.cin * L.cout + 128 * (size_t)L.cout + 8192);
    };
    const int h2 = Hp / 2, w2 = Wp / 2, h4 = Hp / 4, w4 = Wp / 4;
    d_c1 = A.tens(2 * B, h2, w2, 64); gd_c1 = A.tens(2 * B, h2, w2, 64);
    d_c2 = A.tens(2 * B, h4, w4, 128); gd_c2 = A.tens(2 * B, h4, w4, 128);
    d_cat3 = A.tens(B, h4, w4, 145, 148); gd_cat3 = A.tens(B, h4, w4, 145, 148);
    add_planes(A, d_c1, 1); add_planes(A, d_c2, 1); add_planes(A, d_cat3, 1);
    add_planes(A, gd_c1, 0); add_planes(A, gd_c2, 0); add_planes(A, gd_cat3, 0);
    track(layers[0], (size_t)2 * B * h2 * w2); track(layers[1], (size_t)2 * B * h4 * w4); track(layers[2], (size_t)B * h4 * w4);
    int hh = h4, ww = w4;
    for (int i = 0; i < 8; ++i) {
        const ConvLayer& L = layers[3 + i];
        if (L.stride == 2) { hh /= 2; ww /= 2; }
        d_enc[i] = A.tens(B, hh, ww, L.cout); gd_enc[i] = A.tens(B, hh, ww, L.cout);
        add_planes(A, d_enc[i], 1); add_planes(A, gd_enc[i], 0);
        track(L, (size_t)B * hh * ww);
        tensors[L.name] = d_enc[i]; tensors["grad/" + L.name] = gd_enc[i];
    }
    tensors["conv1a"] = batch(d_c1, 0, B); tensors["conv1b"] = batch(d_c1, B, B);
    tensors["conv2a"] = batch(d_c2, 0, B); tensors["conv2b"] = batch(d_c2, B, B);
    tensors["corr"] = slice(d_cat3, 0, 2 * DN_MAXD + 1);
    tensors["conv_redir"] = slice(d_cat3, 2 * DN_MAXD + 1, 64);
    tensors["grad/conv1"] = gd_c1; tensors["grad/conv2"] = gd_c2; tensors["grad/cat3"] = gd_cat3;
    // decoder: bottom of up5 is conv6/1 at Hp/64
    int bh = Hp / 64, bw = Wp / 64;
    for (int u = 0; u < 5; ++u) {
        const UpSpec& S = DN_UP[u];
        const int ct = S.skip + S.cout + 1;
        d_pr[u] = A.tens(B, bh, bw, 1); gd_pr[u] = A.tens(B, bh, bw, 1);
        d_cat[u] = A.tens(B, 2 * bh, 2 * bw, ct, pad4i(ct)); gd_cat[u] = A.tens(B, 2 * bh, 2 * bw, ct, pad4i(ct));
        d_cc[u] = A.tens(B, 2 * bh, 2 * bw, S.cout); gd_cc[u] = A.tens(B, 2 * bh, 2 * bw, S.cout);
        add_planes(A, d_cat[u], 1); add_planes(A, d_cc[u], 1); add_planes(A, gd_cc[u], 0);
        // compact bf16 planes of the deconv output's gradient (a channel slice of gd_cat[u], keyed by the slice pointer)
        add_planes(A, slice(gd_cat[u], S.skip, S.cout), 0);
        for (int j = 0; j < 4; ++j) track(layers[up_layer(u, j)], (size_t)B * 4 * bh * bw);
        std::string n(S.name);
        tensors[n + "/predict"] = d_pr[u];
        tensors[n + "/deconv"] = slice(d_cat[u], S.skip, S.cout);
        tensors[n + "/up_predict"] = slice(d_cat[u], S.skip + S.cout, 1);
        tensors[n + "/concat"] = d_cc[u];
        tensors["grad/" + n + "/concat"] = gd_cc[u];
        bh *= 2; bw *= 2;
    }
    d_pred = A.tens(B, h2, w2, 1); gd_pred = A.tens(B, h2, w2, 1);
    track(layers[DN_PRED], (size_t)B * h2 * w2);
    tensors["prediction"] = d_pred;
}

int Engine::forward_dispnet(int disp_mask, cudaStream_t st) {
    const int nd = 2 * DN_MAXD + 1;
    if (conv_fwd(layers[0], img, d_c1, nullptr, 0, st)) return -1;
    if (conv_fwd(layers[1], d_c1, d_c2, nullptr, 0, st)) return -1;
    TView c2a = batch(d_c2, 0, B), c2b = batch(d_c2, B, B);
    if (conv_fwd(layers[2], c2a, slice(d_cat3, nd, 64), nullptr, 0, st)) return -1;
    {
        CorrFwd cf{};
        cf.left = c2a.p; cf.lcs = c2a.cs; cf.right = c2b.p; cf.rcs = c2b.cs; cf.u = nullptr; cf.ucs = 0;
        cf.out = d_cat3.p; cf.ocs = d_cat3.cs; cf.out2 = nullptr; cf.o2cs = 0;
        cf.B = B; cf.h = d_c2.h; cf.w = d_c2.w; cf.C = 128; cf.max_disp = DN_MAXD; cf.stride = 1; cf.copy_left = 0; cf.u_chan = 0;
        cf.plane_scale = act_scale;   // same fp16 hi/lo arithmetic as the forward convs
        prof_begin(CAT_CORR_FWD, st);
        int rc = corr_fwd(cf, st);
        prof_end(st);
        prof_note(0, (double)B * cf.h * cf.w * (2.0 * 128 + nd) * 4.0);
        if (rc) return -1;
    }
    TView x = d_cat3;
    for (int i = 0; i < 8; ++i) {
        if (conv_fwd(layers[3 + i], x, d_enc[i], nullptr, 0, st)) return -1;
        x = d_enc[i];
    }
    const TView skips[5] = {d_enc[5], d_enc[3], d_enc[1], c2a, batch(d_c1, 0, B)};
    TView bottom = d_enc[7];
    for (int u = 0; u < 5; ++u) {
        const UpSpec& S = DN_UP[u];
        TView cat = d_cat[u];
        if (add_channels(cat.p, cat.cs, skips[u].p, skips[u].cs, cat.pixels(), S.skip, 1.f, 0, st)) return -1;   // tf.concat copy
        if (conv_fwd(layers[up_layer(u, 0)], bottom, slice(cat, S.skip, S.cout), nullptr, 0, st)) return -1;
        if (conv_fwd(layers[up_layer(u, 1)], bottom, d_pr[u], nullptr, 0, st)) return -1;
        if (conv_fwd(layers[up_layer(u, 2)], d_pr[u], slice(cat, S.skip + S.cout, 1), nullptr, 0, st)) return -1;
        if (conv_fwd(layers[up_layer(u, 3)], cat, d_cc[u], nullptr, 0, st)) return -1;
        bottom = d_cc[u];
    }
    if (conv_fwd(layers[DN_PRED], d_cc[4], d_pred, nullptr, 0, st)) return -1;
    for (int i = 0; i < 7; ++i) {
        if (!(disp_mask & (1 << i))) continue;
        const TView& src = i < 5 ? d_pr[i] : d_pred;
        if (i < 6) {   // _make_disp: resize(relu(op * Wp/w_op))
            if (resize_bilinear(src.p, src.cs, B, src.h, src.w, disp[i].p, 1, Hp, Wp, H, W, (float)Wp / (float)src.w, 1, 1.f, 0, st)) return -1;
        } else {       // rescaled_prediction = resize(prediction) * 2, no relu (DispNet.py:149)
            if (resize_bilinear(src.p, src.cs, B, src.h, src.w, disp[i].p, 1, Hp, Wp, H, W, 1.f, 0, 2.f, 0, st)) return -1;
        }
    }
    return 0;
}

// conv2d_transpose backward.  x: its input [n,h,w,cin]; dpre: grad wrt pre-activation output [n,2h,2w,cout].
//   dW[kh,kw,cout,cin] = wgrad of the stride-2 conv that maps the big map (channels cout) to the small one (channels cin)
//   dx                 = that stride-2 conv applied to dpre with the same (canonical) weights as HWIO [.,.,cout,cin]
int Engine::deconv_bwd(const ConvLayer& L, const TView& x, const TView& dpre, const TView* dx, int dx_acc, cudaStream_t st) {
    MS_REQUIRE(L.transposed && dpre.h == x.h * L.stride && dpre.w == x.w * L.stride, "deconv_bwd: shape mismatch");
    int keff = L.kh, oh = x.h;
    int total = std::max((oh - 1) * L.stride + keff - dpre.h, 0);
    const int pt = total / 2;
    total = std::max((x.w - 1) * L.stride + L.kw - dpre.w, 0);
    const int pl = total / 2;
    const int li = (int)(&L - &layers[0]);
    const ActPlanes* dpl = planes_of(dpre);       // bf16 planes of the big map's gradient
    if (dpl) { fresh.erase(dpre.p); if (ensure_planes(dpre, st)) return -1; }
    {
        ConvWgrad q{};
        q.x = dpre; q.dy = x; q.dw = Gr + L.w_off; q.db = nullptr;
        q.kh = L.kh; q.kw = L.kw; q.stride = L.stride; q.dil = 1; q.pad_t = pt; q.pad_l = pl;
        q.workspace = wg_ws; q.workspace_floats = wg_ws_floats; q.accumulate = 0;
        prof_begin(CAT_CONV_WGRAD, st, li);
        int rc;
        if (dpl && use_bf_wgrad && wg_xp.hi && wgrad_bf_supported(q)) {
            // tcgen05: "x" = dY planes, "dy" = a bf16 re-split of the layer's forward input (kind::f16 rejects f16 x bf16)
            ActPlanes xb = wg_xp; xb.cs = (x.c + 7) / 8 * 8;
            MS_REQUIRE(x.pixels() * (size_t)xb.cs <= wg_xp_halfs, "deconv_bwd: wgrad scratch planes too small");
            rc = split_planes(x, xb, st);
            if (!rc) rc = wgrad_bf(q, *dpl, xb, st);
        } else if (use_heads && conv_head_wgrad_supported(q)) {
            rc = conv_head_wgrad(q, st);                 // up_predict: 1 -> 1 channel
        } else {
            rc = conv_wgrad(q, st);
        }
        if (!rc) rc = bias_grad(dpre, Gr + L.b_off, wg_ws, wg_ws_floats, st);
        prof_end(st);
        prof_note((double)x.pixels() * L.kh * L.kw * L.cin * L.cout, 0);
        if (rc) return -1;
    }
    if (dx) {
        ConvGemm p{};
        p.x = dpre; p.wmat = Wt + L.w_off; p.bias = nullptr; p.y = *dx; p.kh = L.kh; p.kw = L.kw;
        p.mul = L.stride; p.off_y = -pt; p.off_x = -pl; p.step = 1; p.div = 1;
        p.alpha = 1.f; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = dx_acc;
        p.part = gemm_part; p.part_floats = conv_gemm_part_floats();
        prof_begin(CAT_CONV_DGRAD, st, li);
        int rc;
        if (dpl && bfw[1][li].ok && conv_bf_supported(p)) {
            fresh.erase(dx->p);                         // (accumulating launches leave dx's own planes stale)
            rc = conv_bf(p, *dpl, bfw[1][li].tiles, nullptr, bf_part, bf_tickets, st);
        } else {
            rc = conv_gemm(p, st);
        }
        prof_end(st);
        prof_note((double)x.pixels() * L.kh * L.kw * L.cin * L.cout, 0);
        if (rc) return -1;
    }
    return 0;
}

int Engine::backward_dispnet(cudaStream_t st) {
    const int nd = 2 * DN_MAXD + 1;
    // loss on disp[6] = crop(resize(prediction) * 2)
    if (resize_bilinear_bwd(g_disp.p, 1, d_pred.p, d_pred.cs, B, d_pred.h, d_pred.w, gd_pred.p, 1, Hp, Wp, H, W, 1.f, 0, 2.f, 0,
                            0, rs_tmp, st)) return -1;
    // prediction conv (linear): -> grad of up1/concat output
    if (conv_bwd(layers[DN_PRED], d_cc[4], gd_pred, &gd_cc[4], nullptr, 1.f, 0, 1, st)) return -1;

    TView c2a = batch(d_c2, 0, B);
    const TView skips[5] = {d_enc[5], d_enc[3], d_enc[1], c2a, batch(d_c1, 0, B)};
    TView gskip[5] = {gd_enc[5], gd_enc[3], gd_enc[1], batch(gd_c2, 0, B), batch(gd_c1, 0, B)};
    for (int u = 4; u >= 0; --u) {
        const UpSpec& S = DN_UP[u];
        const TView bottom = u == 0 ? d_enc[7] : d_cc[u - 1];
        TView gbottom = u == 0 ? gd_enc[7] : gd_cc[u - 1];
        // concat conv (linear): dpre = gd_cc[u] ; input = d_cat[u]
        if (conv_bwd(layers[up_layer(u, 3)], d_cat[u], gd_cc[u], &gd_cat[u], nullptr, 1.f, 0, 1, st)) return -1;
        TView g_dec = slice(gd_cat[u], S.skip, S.cout), g_up = slice(gd_cat[u], S.skip + S.cout, 1);
        TView dec_act = slice(d_cat[u], S.skip, S.cout);
        if (leaky_bwd(g_dec.p, g_dec.cs, dec_act.p, dec_act.cs, g_dec.pixels(), S.cout, DN_ALPHA, st)) return -1;
        // up_predict (transposed, linear): input = predict output
        if (deconv_bwd(layers[up_layer(u, 2)], d_pr[u], g_up, &gd_pr[u], 0, st)) return -1;
        // predict conv (linear): dpre = gd_pr[u] -> gbottom (write)
        if (conv_bwd(layers[up_layer(u, 1)], bottom, gd_pr[u], &gbottom, nullptr, 1.f, 0, 1, st)) return -1;
        // deconv (transposed, leaky already applied): -> gbottom (accumulate)
        if (deconv_bwd(layers[up_layer(u, 0)], bottom, g_dec, &gbottom, 1, st)) return -1;
        (void)skips;
    }
    // ---- encoder, top down.  gd_enc[7] = d(conv6/1 output) complete.
    // feature grads that also receive a skip-slice contribution: enc[5] (up5), enc[3] (up4), enc[1] (up3)
    auto skip_slice = [&](int u) { return slice(gd_cat[u], 0, DN_UP[u].skip); };
    if (leaky_bwd(gd_enc[7].p, gd_enc[7].cs, d_enc[7].p, d_enc[7].cs, gd_enc[7].pixels(), gd_enc[7].c, DN_ALPHA, st)) return -1;
    for (int i = 7; i >= 0; --i) {
        const TView xin = i == 0 ? d_cat3 : d_enc[i - 1];
        TView dx = i == 0 ? gd_cat3 : gd_enc[i - 1];
        int acc = 0;
        const int below = i - 1;              // index of the feature receiving dx
        int skip_u = below == 5 ? 0 : (below == 3 ? 1 : (below == 1 ? 2 : -1));
        if (skip_u >= 0) {                    // seed with the skip-connection gradient, then accumulate the dgrad
            TView sl = skip_slice(skip_u);
            if (add_channels(dx.p, dx.cs, sl.p, sl.cs, dx.pixels(), dx.c, 1.f, 0, st)) return -1;
            acc = 1;
        }
        TView mask = i == 0 ? d_cat3 : d_enc[i - 1];
        if (conv_bwd(layers[3 + i], xin, gd_enc[i], &dx, i == 0 ? nullptr : &mask, DN_ALPHA, acc, 1, st)) return -1;
    }
    // gd_cat3: [0,81) corr grads (linear), [81,145) conv_redir output grads (leaky)
    {
        TView g_red = slice(gd_cat3, nd, 64), red_act = slice(d_cat3, nd, 64);
        if (leaky_bwd(g_red.p, g_red.cs, red_act.p, red_act.cs, g_red.pixels(), 64, DN_ALPHA, st)) return -1;
        TView gc2a = batch(gd_c2, 0, B), gc2b = batch(gd_c2, B, B);
        if (conv_bwd(layers[2], c2a, g_red, &gc2a, nullptr, 1.f, 0, 1, st)) return -1;           // writes d(conv2a)
        CorrBwd cb{};
        TView c2b = batch(d_c2, B, B);
        cb.left = c2a.p; cb.lcs = c2a.cs; cb.right = c2b.p; cb.rcs = c2b.cs; cb.u = nullptr; cb.ucs = 0;
        cb.dcost = gd_cat3.p; cb.dcs = gd_cat3.cs; cb.dleft = gc2a.p; cb.dlcs = gc2a.cs; cb.dright = gc2b.p; cb.drcs = gc2b.cs;
        cb.du = nullptr; cb.ducs = 0;
        cb.B = B; cb.h = d_c2.h; cb.w = d_c2.w; cb.C = 128; cb.max_disp = DN_MAXD; cb.stride = 1;
        cb.add_left_slice = 0; cb.acc_left = 1; cb.acc_right = 0; cb.gcoff = 0;
        prof_begin(CAT_CORR_BWD, st);
        int rc = corr_bwd(cb, st);
        prof_end(st);
        prof_note(0, (double)B * cb.h * cb.w * (4.0 * 128 + nd) * 4.0);
        if (rc) return -1;
        TView sl = skip_slice(3);                                                                   // up2 skip = conv2a
        if (add_channels(gc2a.p, gc2a.cs, sl.p, sl.cs, gc2a.pixels(), 128, 1.f, 1, st)) return -1;
    }
    if (leaky_bwd(gd_c2.p, gd_c2.cs, d_c2.p, d_c2.cs, gd_c2.pixels(), 128, DN_ALPHA, st)) return -1;
    // conv2 (shared, batch 2B): wgrad + dgrad -> gd_c1 ; then the up1 skip (conv1a) ; then leaky
    if (conv_bwd(layers[1], d_c1, gd_c2, &gd_c1, nullptr, 1.f, 0, 1, st)) return -1;
    {
        TView gc1a = batch(gd_c1, 0, B), sl = skip_slice(4);
        if (add_channels(gc1a.p, gc1a.cs, sl.p, sl.cs, gc1a.pixels(), 64, 1.f, 1, st)) return -1;
    }
    if (leaky_bwd(gd_c1.p, gd_c1.cs, d_c1.p, d_c1.cs, gd_c1.pixels(), 64, DN_ALPHA, st)) return -1;
    return conv_bwd(layers[0], img, gd_c1, nullptr, nullptr, 1.f, 0, 1, st);
}

}  // namespace ms
