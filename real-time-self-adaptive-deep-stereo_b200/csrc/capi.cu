// extern "C" surface of libmadstereo (declared in include/madstereo.h).
#include <cstring>

#pragma GCC visibility push(default)
#include "../../include/madstereo.h"
#pragma GCC visibility pop
#include "engine.h"

namespace ms { const char* last_error_cstr(); }
using namespace ms;

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static void same_pad_c(int in, int k, int s, int d, int& out, int& before) {
    int keff = (k - 1) * d + 1;
    out = (in + s - 1) / s;
    int total = (out - 1) * s + keff - in;
    if (total < 0) total = 0;
    before = total / 2;
}
static void copy_str(char* dst, int cap, const std::string& s) {
    if (!dst || cap <= 0) return;
    size_t n = std::min((size_t)cap - 1, s.size());
    memcpy(dst, s.data(), n);
    dst[n] = 0;
}

extern "C" {

int ms_version(void) { return 101; }
const char* ms_last_error(void) { return ms::last_error_cstr(); }

int ms_corr_fwd(const float* left, int left_cs, const float* right, int right_cs, const float* u, int u_cs,
                float* out, int out_cs, int B, int h, int w, int C, int max_disp, int stride, int copy_left,
                int u_chan, void* stream) {
    CorrFwd p{};
    p.left = left; p.lcs = left_cs; p.right = right; p.rcs = right_cs; p.u = u; p.ucs = u_cs;
    p.out = out; p.ocs = out_cs; p.out2 = nullptr; p.o2cs = 0;
    p.B = B; p.h = h; p.w = w; p.C = C; p.max_disp = max_disp; p.stride = stride; p.copy_left = copy_left;
    p.u_chan = u_chan;
    return corr_fwd(p, S(stream));
}

int ms_debug_mma_probe(int a_mn, int b_mn, int n, int n_acc, int rot, int iters, int uni, int ctas, long long* out_dev, void* stream) {
    return mma_probe(a_mn, b_mn, n, n_acc, rot, iters, uni, ctas, out_dev, S(stream));
}
int ms_corr_fwd_wide(const float* left, int left_cs, const float* right, int right_cs, float* out, int out_cs, int B, int h,
                     int w, int C, int max_disp, float act_scale, void* stream) {
    CorrFwd p{};
    p.left = left; p.lcs = left_cs; p.right = right; p.rcs = right_cs; p.u = nullptr; p.ucs = 0;
    p.out = out; p.ocs = out_cs; p.out2 = nullptr; p.o2cs = 0;
    p.B = B; p.h = h; p.w = w; p.C = C; p.max_disp = max_disp; p.stride = 1; p.copy_left = 0; p.u_chan = 0;
    p.plane_scale = act_scale;
    if (!corr_mma_supported(p)) { set_error("ms_corr_fwd_wide: needs >= 17 displacements (max_disp 8..40), C % 16 == 0, 16-byte aligned rows, act_scale > 0"); return -3; }
    return corr_mma(p, S(stream));
}

int ms_corr_bwd(const float* left, int left_cs, const float* right, int right_cs, const float* u, int u_cs,
                const float* dcost, int dcost_cs, float* dleft, int dleft_cs, float* dright, int dright_cs,
                float* du, int du_cs, int B, int h, int w, int C, int max_disp, int stride, int add_left_slice,
                void* stream) {
    CorrBwd p{};
    p.left = left; p.lcs = left_cs; p.right = right; p.rcs = right_cs; p.u = u; p.ucs = u_cs;
    p.dcost = dcost; p.dcs = dcost_cs; p.dleft = dleft; p.dlcs = dleft_cs; p.dright = dright; p.drcs = dright_cs;
    p.du = du; p.ducs = du_cs;
    p.B = B; p.h = h; p.w = w; p.C = C; p.max_disp = max_disp; p.stride = stride;
    p.add_left_slice = add_left_slice; p.acc_left = 0; p.acc_right = 0; p.gcoff = -1;
    return corr_bwd(p, S(stream));
}

int ms_conv2d_fwd(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights, const float* bias,
                  float* y, int cout, int y_cs, int kh, int kw, int stride, int dilation, float alpha, void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh, pt);
    same_pad_c(w, kw, stride, dilation, ow, pl);
    ConvGemm p{};
    p.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    p.y = view(y, n, oh, ow, cout, y_cs);
    p.wmat = weights; p.bias = bias; p.kh = kh; p.kw = kw;
    p.mul = stride; p.off_y = -pt; p.off_x = -pl; p.step = dilation; p.div = 1;
    p.alpha = alpha; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    return conv_gemm(p, S(stream));
}

int ms_conv2d_dgrad(const float* dy, int n, int oh, int ow, int cout, int dy_cs, const float* weights, float* dx,
                    int h, int w, int cin, int dx_cs, int kh, int kw, int stride, int dilation, float* scratch,
                    void* stream) {
    int oh2, ow2, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh2, pt);
    same_pad_c(w, kw, stride, dilation, ow2, pl);
    if (oh2 != oh || ow2 != ow) { set_error("ms_conv2d_dgrad: shape mismatch"); return -2; }
    if (transpose_taps(weights, scratch, kh * kw, cin, cout, S(stream))) return -1;
    ConvGemm p{};
    p.x = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);
    p.y = view(dx, n, h, w, cin, dx_cs);
    p.wmat = scratch; p.bias = nullptr; p.kh = kh; p.kw = kw;
    p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -dilation; p.div = stride;
    p.alpha = 1.f; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    return conv_gemm(p, S(stream));
}

int ms_conv2d_fwd_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights, const float* bias,
                     float* y, int cout, int y_cs, int kh, int kw, int stride, int dilation, float alpha, float act_scale,
                     void* scratch, size_t scratch_bytes, void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh, pt);
    same_pad_c(w, kw, stride, dilation, ow, pl);
    ConvGemm p{};
    p.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    p.y = view(y, n, oh, ow, cout, y_cs);
    p.wmat = weights; p.bias = bias; p.kh = kh; p.kw = kw;
    p.mul = stride; p.off_y = -pt; p.off_x = -pl; p.step = dilation; p.div = 1;
    p.alpha = alpha; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    if (!conv_bf_supported(p)) { set_error("ms_conv2d_fwd_bf: shape not supported by the split-bf16 tcgen05 path"); return -3; }
    return conv_bf_oneshot(p, 0, 1, act_scale, scratch, scratch_bytes, S(stream));      // forward: fp16 planes of x * act_scale
}
int ms_conv2d_dgrad_bf(const float* dy, int n, int oh, int ow, int cout, int dy_cs, const float* weights, float* dx,
                       int h, int w, int cin, int dx_cs, int kh, int kw, int stride, int dilation, void* scratch,
                       size_t scratch_bytes, void* stream) {
    int oh2, ow2, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh2, pt);
    same_pad_c(w, kw, stride, dilation, ow2, pl);
    if (oh2 != oh || ow2 != ow) { set_error("ms_conv2d_dgrad_bf: shape mismatch"); return -2; }
    ConvGemm p{};
    p.x = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);
    p.y = view(dx, n, h, w, cin, dx_cs);
    p.wmat = weights; p.bias = nullptr; p.kh = kh; p.kw = kw;
    p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -dilation; p.div = stride;
    p.alpha = 1.f; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    if (!conv_bf_supported(p)) { set_error("ms_conv2d_dgrad_bf: shape not supported by the split-bf16 tcgen05 path"); return -3; }
    return conv_bf_oneshot(p, 1, 0, 1.f, scratch, scratch_bytes, S(stream));      // gradients: bf16 planes
}
size_t ms_conv2d_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout) {
    ConvGemm a{}, b{};
    a.x = view(nullptr, n, h, w, cin, cin); a.y = view(nullptr, n, h, w, cout, cout); a.kh = kh; a.kw = kw;
    b.x = view(nullptr, n, h, w, cout, cout); b.y = view(nullptr, n, h, w, cin, cin); b.kh = kh; b.kw = kw;
    size_t sa = conv_bf_oneshot_scratch_bytes(a), sb = conv_bf_oneshot_scratch_bytes(b);
    return sa > sb ? sa : sb;
}
int ms_conv2d_wgrad_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int oh, int ow, int cout,
                       int dy_cs, float* dw, float* db, int kh, int kw, int stride, int dilation, void* scratch,
                       size_t scratch_bytes, void* stream) {
    int oh2, ow2, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh2, pt);
    same_pad_c(w, kw, stride, dilation, ow2, pl);
    if (oh2 != oh || ow2 != ow) { set_error("ms_conv2d_wgrad_bf: shape mismatch"); return -2; }
    ConvWgrad q{};
    q.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    q.dy = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);
    q.dw = dw; q.db = db; q.kh = kh; q.kw = kw; q.stride = stride; q.dil = dilation; q.pad_t = pt; q.pad_l = pl;
    q.accumulate = 0;
    if (!wgrad_bf_supported(q)) { set_error("ms_conv2d_wgrad_bf: shape not supported by the split-bf16 tcgen05 path"); return -3; }
    return wgrad_bf_oneshot(q, scratch, scratch_bytes, S(stream));
}
size_t ms_conv2d_wgrad_bf_scratch(int n, int h, int w, int oh, int ow, int kh, int kw, int cin, int cout) {
    ConvWgrad q{};
    q.x = view(nullptr, n, h, w, cin, cin); q.dy = view(nullptr, n, oh, ow, cout, cout); q.kh = kh; q.kw = kw;
    return wgrad_bf_oneshot_scratch_bytes(q);
}
// ---- DispNet conv1 (7x7 stride 2, 3 -> 64; Nets/DispNet.py:82-86) on the direct CUDA-core kernels (csrc/conv_stem.cu).
//      x: [n,h,w,3] stored with a channel stride of 4 floats (the engine's padded image layout)
int ms_conv2d_stem_fwd(const float* x4, int n, int h, int w, const float* weights, const float* bias, float* y, int y_cs,
                       float alpha, void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, 7, 2, 1, oh, pt);
    same_pad_c(w, 7, 2, 1, ow, pl);
    ConvGemm p{};
    p.x = view(const_cast<float*>(x4), n, h, w, 3, 4);
    p.y = view(y, n, oh, ow, 64, y_cs);
    p.wmat = weights; p.bias = bias; p.kh = 7; p.kw = 7;
    p.mul = 2; p.off_y = -pt; p.off_x = -pl; p.step = 1; p.div = 1;
    p.alpha = alpha; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    if (!conv_stem_fwd_supported(p)) { set_error("ms_conv2d_stem_fwd: unsupported layout"); return -3; }
    return conv_stem_fwd(p, nullptr, S(stream));
}
size_t ms_conv2d_stem_wgrad_workspace(int n, int h, int w) {
    ConvWgrad q{};
    q.x = view(nullptr, n, h, w, 3, 4); q.dy = view(nullptr, n, (h + 1) / 2, (w + 1) / 2, 64, 64); q.kh = q.kw = 7; q.stride = 2; q.dil = 1;
    return conv_stem_wgrad_workspace_floats(q);
}
int ms_conv2d_stem_wgrad(const float* x4, int n, int h, int w, const float* dy, int dy_cs, float* dw, float* db, float* workspace,
                         size_t workspace_floats, void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, 7, 2, 1, oh, pt);
    same_pad_c(w, 7, 2, 1, ow, pl);
    ConvWgrad q{};
    q.x = view(const_cast<float*>(x4), n, h, w, 3, 4);
    q.dy = view(const_cast<float*>(dy), n, oh, ow, 64, dy_cs);
    q.dw = dw; q.db = db; q.kh = q.kw = 7; q.stride = 2; q.dil = 1; q.pad_t = pt; q.pad_l = pl;
    q.workspace = workspace; q.workspace_floats = workspace_floats; q.accumulate = 0;
    if (!conv_stem_wgrad_supported(q)) { set_error("ms_conv2d_stem_wgrad: unsupported layout"); return -3; }
    return conv_stem_wgrad(q, S(stream));
}

// ---- conv2d_transpose (Nets/sharedLayers.py:80-92) and its two gradients on the split-16-bit tcgen05 path.
//      weights [kh,kw,cout,cin] (TF layout); x [n,h,w,cin]; y / dy [n,h*stride,w*stride,cout]
static void transpose_geom(int h, int w, int kh, int kw, int stride, int& oh, int& ow, int& pt, int& pl) {
    oh = h * stride; ow = w * stride;
    int t0, t1;
    same_pad_c(oh, kh, stride, 1, t0, pt);
    same_pad_c(ow, kw, stride, 1, t1, pl);
}
int ms_conv2d_transpose_fwd_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights, const float* bias,
                               float* y, int cout, int y_cs, int kh, int kw, int stride, float alpha, float act_scale,
                               void* scratch, size_t scratch_bytes, void* stream) {
    int oh, ow, pt, pl;
    transpose_geom(h, w, kh, kw, stride, oh, ow, pt, pl);
    ConvGemm p{};
    p.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    p.y = view(y, n, oh, ow, cout, y_cs);
    p.wmat = weights; p.bias = bias; p.kh = kh; p.kw = kw;
    p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -1; p.div = stride;
    p.alpha = alpha; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    if (!conv_bf_supported(p)) { set_error("ms_conv2d_transpose_fwd_bf: shape not supported by the tcgen05 path"); return -3; }
    return conv_bf_oneshot(p, 1, 1, act_scale, scratch, scratch_bytes, S(stream));     // [tap][M = cout][K = cin], fp16 planes
}
int ms_conv2d_transpose_dgrad_bf(const float* dy, int n, int h, int w, int cout, int dy_cs, const float* weights, float* dx,
                                 int cin, int dx_cs, int kh, int kw, int stride, void* scratch, size_t scratch_bytes,
                                 void* stream) {
    int oh, ow, pt, pl;
    transpose_geom(h, w, kh, kw, stride, oh, ow, pt, pl);
    ConvGemm p{};
    p.x = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);
    p.y = view(dx, n, h, w, cin, dx_cs);
    p.wmat = weights; p.bias = nullptr; p.kh = kh; p.kw = kw;
    p.mul = stride; p.off_y = -pt; p.off_x = -pl; p.step = 1; p.div = 1;      // = the strided conv of dy with HWIO [.,.,cout,cin]
    p.alpha = 1.f; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    if (!conv_bf_supported(p)) { set_error("ms_conv2d_transpose_dgrad_bf: shape not supported by the tcgen05 path"); return -3; }
    return conv_bf_oneshot(p, 0, 0, 1.f, scratch, scratch_bytes, S(stream));           // [tap][K = cout][M = cin], bf16 planes
}
size_t ms_conv2d_transpose_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout, int stride) {
    ConvGemm a{}, b{};
    a.x = view(nullptr, n, h, w, cin, cin); a.y = view(nullptr, n, h * stride, w * stride, cout, cout); a.kh = kh; a.kw = kw;
    b.x = view(nullptr, n, h * stride, w * stride, cout, cout); b.y = view(nullptr, n, h, w, cin, cin); b.kh = kh; b.kw = kw;
    size_t sa = conv_bf_oneshot_scratch_bytes(a), sb = conv_bf_oneshot_scratch_bytes(b);
    return sa > sb ? sa : sb;
}
static ConvWgrad transpose_wgrad_geom(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int cout, int dy_cs,
                                      int kh, int kw, int stride) {
    int oh, ow, pt, pl;
    transpose_geom(h, w, kh, kw, stride, oh, ow, pt, pl);
    ConvWgrad q{};
    q.x = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);      // the strided conv's input is the big map ...
    q.dy = view(const_cast<float*>(x), n, h, w, cin, x_cs);          // ... and its "output gradient" the layer's input
    q.kh = kh; q.kw = kw; q.stride = stride; q.dil = 1; q.pad_t = pt; q.pad_l = pl; q.accumulate = 0;
    return q;
}
size_t ms_conv2d_transpose_wgrad_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout, int stride) {
    ConvWgrad q = transpose_wgrad_geom(nullptr, n, h, w, cin, cin, nullptr, cout, cout, kh, kw, stride);
    return wgrad_bf_oneshot_scratch_bytes(q);
}
int ms_conv2d_transpose_wgrad_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int cout, int dy_cs,
                                 float* dw, float* db, int kh, int kw, int stride, void* scratch, size_t scratch_bytes,
                                 void* stream) {
    ConvWgrad q = transpose_wgrad_geom(x, n, h, w, cin, x_cs, dy, cout, dy_cs, kh, kw, stride);
    q.dw = dw; q.db = nullptr;                                        // dw [kh,kw,cout,cin]
    if (!wgrad_bf_supported(q)) { set_error("ms_conv2d_transpose_wgrad_bf: shape not supported by the tcgen05 path"); return -3; }
    if (wgrad_bf_oneshot(q, scratch, scratch_bytes, S(stream))) return -1;
    if (!db) return 0;
    // bias gradient = per-channel sum of dy; the partial-sum region of the scratch is free again after the reduction
    return bias_grad(q.x, db, static_cast<float*>(scratch), scratch_bytes / sizeof(float), S(stream));
}
// ---- plane-level entry points of the split-bf16 path: what the engine calls per layer in steady state (operands
//      already split: activations by the producing epilogue, weights once per update)
int ms_bf_split(const float* x, int n, int h, int w, int c, int x_cs, void* hi, void* lo, int plane_cs, int fmt, float scale,
                void* stream) {
    ActPlanes pl; pl.hi = hi; pl.lo = lo; pl.cs = plane_cs; pl.fmt = fmt; pl.scale = fmt == 1 ? scale : 1.f;
    return split_planes(view(const_cast<float*>(x), n, h, w, c, x_cs), pl, S(stream));
}
size_t ms_bf_weight_halfs(int taps, int m, int k) { return conv_bf_weight_halfs(taps, m, k); }
int ms_bf_prep_weights(const float* weights_hwio, int taps, int cin, int cout, int for_dgrad, int fmt, void* tiles,
                       void* job_dev, void* stream) {
    const int M = for_dgrad ? cin : cout, K = for_dgrad ? cout : cin;
    int Mpad, Kpad; conv_bf_weight_dims(M, K, Mpad, Kpad);
    BfPrepJob job{weights_hwio, tiles, taps, M, K, Mpad, Kpad, for_dgrad ? 0 : 1, fmt};
    MS_CHECK_CUDA(cudaMemcpyAsync(job_dev, &job, sizeof job, cudaMemcpyHostToDevice, S(stream)));
    MS_CHECK_CUDA(cudaStreamSynchronize(S(stream)));
    return bf_prep_weights(static_cast<const BfPrepJob*>(job_dev), 1, conv_bf_weight_halfs(taps, M, K), S(stream));
}
int ms_conv2d_fwd_bf_planes(const void* xhi, const void* xlo, int x_pcs, int fmt, float scale, int n, int h, int w, int cin,
                            const void* wtiles, const float* bias, float* y, int cout, int y_cs, void* yhi, void* ylo,
                            int y_pcs, int kh, int kw, int stride, int dilation, float alpha, float* part,
                            unsigned int* tickets, void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh, pt);
    same_pad_c(w, kw, stride, dilation, ow, pl);
    ConvGemm p{};
    p.x = view(nullptr, n, h, w, cin, cin);
    p.y = view(y, n, oh, ow, cout, y_cs);
    p.bias = bias; p.kh = kh; p.kw = kw;
    p.mul = stride; p.off_y = -pt; p.off_x = -pl; p.step = dilation; p.div = 1;
    p.alpha = alpha; p.mask_alpha = 1.f;
    if (!conv_bf_supported(p)) { set_error("ms_conv2d_fwd_bf_planes: shape not supported"); return -3; }
    ActPlanes xp; xp.hi = const_cast<void*>(xhi); xp.lo = const_cast<void*>(xlo); xp.cs = x_pcs; xp.fmt = fmt; xp.scale = fmt == 1 ? scale : 1.f;
    ActPlanes yp; yp.hi = yhi; yp.lo = ylo; yp.cs = y_pcs; yp.fmt = fmt; yp.scale = xp.scale;
    return conv_bf(p, xp, wtiles, yhi ? &yp : nullptr, part, tickets, S(stream));
}
size_t ms_conv2d_bf_part_floats() { return conv_bf_part_floats(); }
size_t ms_conv2d_bf_ticket_words() { return conv_bf_ticket_words(); }
int ms_conv2d_wgrad_bf_planes(const void* xhi, const void* xlo, int x_pcs, int n, int h, int w, int cin,
                              const void* dhi, const void* dlo, int d_pcs, int oh, int ow, int cout, float* dw, float* db,
                              int kh, int kw, int stride, int dilation, float* workspace, size_t workspace_floats, void* stream) {
    int oh2, ow2, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh2, pt);
    same_pad_c(w, kw, stride, dilation, ow2, pl);
    if (oh2 != oh || ow2 != ow) { set_error("ms_conv2d_wgrad_bf_planes: shape mismatch"); return -2; }
    ConvWgrad q{};
    q.x = view(nullptr, n, h, w, cin, cin); q.dy = view(nullptr, n, oh, ow, cout, cout);
    q.dw = dw; q.db = db; q.kh = kh; q.kw = kw; q.stride = stride; q.dil = dilation; q.pad_t = pt; q.pad_l = pl;
    q.workspace = workspace; q.workspace_floats = workspace_floats;
    if (!wgrad_bf_supported(q)) { set_error("ms_conv2d_wgrad_bf_planes: shape not supported"); return -3; }
    ActPlanes xp; xp.hi = const_cast<void*>(xhi); xp.lo = const_cast<void*>(xlo); xp.cs = x_pcs; xp.fmt = 0; xp.scale = 1.f;
    ActPlanes dp; dp.hi = const_cast<void*>(dhi); dp.lo = const_cast<void*>(dlo); dp.cs = d_pcs; dp.fmt = 0; dp.scale = 1.f;
    return wgrad_bf(q, xp, dp, S(stream));
}
size_t ms_conv2d_wgrad_bf_workspace(int kh, int kw, int cin, int cout) { return wgrad_bf_workspace_floats(kh, kw, cin, cout); }

size_t ms_conv2d_wgrad_workspace(int kh, int kw, int cin, int cout, size_t out_pixels) {
    return conv_wgrad_workspace_floats(kh * kw, cin, cout, out_pixels);
}

int ms_conv2d_wgrad(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int oh, int ow, int cout,
                    int dy_cs, float* dw, float* db, int kh, int kw, int stride, int dilation, float* workspace,
                    size_t workspace_floats, void* stream) {
    int oh2, ow2, pt, pl;
    same_pad_c(h, kh, stride, dilation, oh2, pt);
    same_pad_c(w, kw, stride, dilation, ow2, pl);
    if (oh2 != oh || ow2 != ow) { set_error("ms_conv2d_wgrad: shape mismatch"); return -2; }
    ConvWgrad q{};
    q.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    q.dy = view(const_cast<float*>(dy), n, oh, ow, cout, dy_cs);
    q.dw = dw; q.db = db; q.kh = kh; q.kw = kw; q.stride = stride; q.dil = dilation; q.pad_t = pt; q.pad_l = pl;
    q.workspace = workspace; q.workspace_floats = workspace_floats; q.accumulate = 0;
    return conv_wgrad(q, S(stream));
}

int ms_conv2d_wgrad_tc(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int cout, int dy_cs,
                       float* dw, float* db, int kh, int kw, int dilation, float* workspace, size_t workspace_floats,
                       void* stream) {
    int oh, ow, pt, pl;
    same_pad_c(h, kh, 1, dilation, oh, pt);
    same_pad_c(w, kw, 1, dilation, ow, pl);
    ConvWgrad q{};
    q.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    q.dy = view(const_cast<float*>(dy), n, h, w, cout, dy_cs);
    q.dw = dw; q.db = db; q.kh = kh; q.kw = kw; q.stride = 1; q.dil = dilation; q.pad_t = pt; q.pad_l = pl;
    q.workspace = workspace; q.workspace_floats = workspace_floats; q.accumulate = 0;
    if (!wgrad_tc_supported(q)) { set_error("ms_conv2d_wgrad_tc: shape not supported by the tcgen05 path"); return -3; }
    return wgrad_tc(q, S(stream));
}
size_t ms_conv2d_wgrad_tc_workspace(int kh, int kw, int cin, int cout, int n, int h, int w) {
    return wgrad_tc_workspace_floats(kh * kw, cin, cout, n, h, w);
}

int ms_conv2d_transpose_fwd(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights,
                            const float* bias, float* y, int cout, int y_cs, int kh, int kw, int stride, float alpha,
                            float* scratch, void* stream) {
    const int oh = h * stride, ow = w * stride;
    int t0, t1, pt, pl;
    same_pad_c(oh, kh, stride, 1, t0, pt);
    same_pad_c(ow, kw, stride, 1, t1, pl);
    if (transpose_taps(weights, scratch, kh * kw, cout, cin, S(stream))) return -1;   // [tap][cout][cin] -> [tap][cin][cout]
    ConvGemm p{};
    p.x = view(const_cast<float*>(x), n, h, w, cin, x_cs);
    p.y = view(y, n, oh, ow, cout, y_cs);
    p.wmat = scratch; p.bias = bias; p.kh = kh; p.kw = kw;
    p.mul = 1; p.off_y = pt; p.off_x = pl; p.step = -1; p.div = stride;
    p.alpha = alpha; p.mask = nullptr; p.mask_alpha = 1.f; p.res = nullptr; p.accumulate = 0;
    return conv_gemm(p, S(stream));
}

int ms_resize_bilinear(const float* src, int src_cs, int B, int ih, int iw, float* dst, int dst_cs, int rh, int rw,
                       int oh, int ow, float pre_scale, int pre_relu, float post_scale, int post_relu, void* stream) {
    return resize_bilinear(src, src_cs, B, ih, iw, dst, dst_cs, rh, rw, oh, ow, pre_scale, pre_relu, post_scale,
                           post_relu, S(stream));
}
int ms_resize_bilinear_bwd(const float* dout, int dout_cs, const float* src, int src_cs, int B, int ih, int iw,
                           float* dsrc, int dsrc_cs, int rh, int rw, int oh, int ow, float pre_scale, int pre_relu,
                           float post_scale, int post_relu, int accumulate, float* tmp, void* stream) {
    return resize_bilinear_bwd(dout, dout_cs, src, src_cs, B, ih, iw, dsrc, dsrc_cs, rh, rw, oh, ow, pre_scale,
                               pre_relu, post_scale, post_relu, accumulate, tmp, S(stream));
}

size_t ms_reproj_loss_workspace(int B, int H, int W) { return loss_workspace_floats(B, H, W); }
int ms_reproj_loss(const float* left, const float* right, const float* disp, int B, int H, int W, float* loss_out,
                   float* ddisp, float* workspace, float grad_scale, void* stream) {
    ReprojLoss p{};
    p.left = left; p.right = right; p.disp = disp; p.loss = loss_out; p.ddisp = ddisp; p.workspace = workspace;
    p.B = B; p.H = H; p.W = W; p.grad_scale = grad_scale;
    return reproj_loss(p, S(stream));
}

int ms_momentum_update(float* w, const float* g, float* m, size_t n, float lr, float mu, float grad_scale,
                       void* stream) {
    return momentum_update(w, g, m, n, lr, mu, grad_scale, S(stream));
}

int ms_pad_reflect(const float* src, int B, int H, int W, int C, float* dst, int Hp, int Wp, int dst_cs, float scale,
                   float bias, void* stream) {
    return pad_reflect(src, B, H, W, C, dst, Hp, Wp, dst_cs, scale, bias, S(stream));
}

// ---- engine --------------------------------------------------------------------------------------
void* ms_engine_create(const char* net_name, int B, int H, int W, int radius_d, int corr_stride, int warping) {
    if (!net_name || B < 1 || H < 8 || W < 8 || radius_d < 0 || corr_stride < 1) {
        set_error("ms_engine_create: bad arguments");
        return nullptr;
    }
    Engine* e = new Engine();
    e->B = B; e->H = H; e->W = W;
    e->Hp = (H + 63) / 64 * 64; e->Wp = (W + 63) / 64 * 64;
    e->radius_d = radius_d; e->corr_stride = corr_stride; e->warping = warping;
    if (!strcmp(net_name, "MADNet")) { e->net = 0; e->build_madnet(); }
    else if (!strcmp(net_name, "Dispnet")) { e->net = 1; e->build_dispnet(); }
    else { set_error(std::string("Unrecognized network name: ") + net_name); delete e; return nullptr; }
    // scale of the fp16 forward planes (stored value = activation * scale, a power of two): MADNet consumes raw 0..255
    // images (Nets/MadNet.py:56-66) -> activations up to ~1e4, 1/16 keeps |x| <= 1e6 finite; DispNet normalises its input
    // to [-0.4, 0.6] (Nets/DispNet.py:59-73) -> activations O(1e-3 .. 10), 64 lifts them out of fp16's subnormal range
    e->act_scale = e->net == 1 ? 64.f : 0.0625f;
    if (const char* as = getenv("MS_ACT_SCALE")) { const float v = (float)atof(as); if (v > 0.f) e->act_scale = v; }
    e->finalize_groups(nullptr, 0);
    return e;
}
int ms_engine_destroy(void* h) { delete static_cast<Engine*>(h); return 0; }
int ms_engine_num_layers(void* h) { return (int)static_cast<Engine*>(h)->layers.size(); }
int ms_engine_layer_info(void* h, int i, char* name, int name_cap, char* scope, int scope_cap, char* bias_name,
                         int bias_cap, int* dims7, float* alpha_out) {
    Engine* e = static_cast<Engine*>(h);
    if (i < 0 || i >= (int)e->layers.size()) { set_error("layer index out of range"); return -2; }
    const ConvLayer& L = e->layers[i];
    copy_str(name, name_cap, L.name); copy_str(scope, scope_cap, L.scope); copy_str(bias_name, bias_cap, L.bname);
    if (dims7) { dims7[0] = L.kh; dims7[1] = L.kw; dims7[2] = L.cin; dims7[3] = L.cout; dims7[4] = L.stride; dims7[5] = L.dil; dims7[6] = L.transposed; }
    if (alpha_out) *alpha_out = L.alpha;
    return 0;
}
int ms_engine_set_groups(void* h, const int* group_of_layer, int n_layers, int n_groups) {
    Engine* e = static_cast<Engine*>(h);
    if (e->bound) { set_error("ms_engine_set_groups: engine already bound"); return -2; }
    if (n_layers != (int)e->layers.size()) { set_error("ms_engine_set_groups: layer count mismatch"); return -2; }
    return e->finalize_groups(group_of_layer, n_groups);
}
int ms_engine_sizes(void* h, size_t* n_param_floats, size_t* workspace_floats) {
    Engine* e = static_cast<Engine*>(h);
    if (n_param_floats) *n_param_floats = e->n_params;
    if (workspace_floats) *workspace_floats = e->layout(nullptr);
    return 0;
}
int ms_engine_param_offsets(void* h, int i, size_t* w_off, size_t* b_off) {
    Engine* e = static_cast<Engine*>(h);
    if (i < 0 || i >= (int)e->layers.size()) { set_error("layer index out of range"); return -2; }
    *w_off = e->layers[i].w_off; *b_off = e->layers[i].b_off;
    return 0;
}
int ms_engine_group_range(void* h, int g, size_t* begin, size_t* end) {
    Engine* e = static_cast<Engine*>(h);
    if (g < 0 || g >= e->n_groups) { set_error("group index out of range"); return -2; }
    *begin = e->group_begin[g]; *end = e->group_end[g];
    return 0;
}
int ms_engine_bind(void* h, float* weights, float* grads, float* momentum, float* workspace, size_t workspace_floats,
                   void* stream) {
    Engine* e = static_cast<Engine*>(h);
    size_t need = e->layout(nullptr);
    if (workspace_floats < need) { set_error("ms_engine_bind: workspace too small"); return -2; }
    if (((uintptr_t)weights | (uintptr_t)grads | (uintptr_t)momentum | (uintptr_t)workspace) & 255) {
        set_error("ms_engine_bind: arenas must be 256-byte aligned"); return -2;
    }
    e->Wt = weights; e->Gr = grads; e->Mo = momentum; e->ws = workspace; e->ws_floats = workspace_floats;
    if (e->layout(workspace) > need) { set_error("ms_engine_bind: layout exceeds the size reported by ms_engine_sizes"); return -2; }
    MS_CHECK_CUDA(cudaMemsetAsync(workspace, 0, need * sizeof(float), S(stream)));
    MS_CHECK_CUDA(cudaMemsetAsync(grads, 0, e->n_params * sizeof(float), S(stream)));
    if (!e->bf_jobs.empty())
        MS_CHECK_CUDA(cudaMemcpyAsync(e->bf_jobs_dev, e->bf_jobs.data(), e->bf_jobs.size() * sizeof(BfPrepJob),
                                      cudaMemcpyHostToDevice, S(stream)));
    MS_CHECK_CUDA(cudaStreamSynchronize(S(stream)));   // the host job table must outlive the copy
    e->weights_dirty = true;
    e->bound = true;
    return 0;
}
int ms_engine_set_input(void* h, const float* left, const float* right, void* stream) {
    return static_cast<Engine*>(h)->set_input(left, right, S(stream));
}
int ms_engine_set_input_u8(void* h, const unsigned char* left, const unsigned char* right, void* stream) {
    return static_cast<Engine*>(h)->set_input_u8(left, right, S(stream));
}
int ms_engine_set_gt(void* h, const float* gt, void* stream) {
    Engine* e = static_cast<Engine*>(h);
    if (!e->bound) { set_error("engine not bound"); return -2; }
    MS_CHECK_CUDA(cudaMemcpyAsync(e->gt, gt, (size_t)e->B * e->H * e->W * sizeof(float), cudaMemcpyDefault, S(stream)));
    return 0;
}
int ms_engine_set_proxy(void* h, const float* proxy, void* stream) {
    Engine* e = static_cast<Engine*>(h);
    if (!e->bound) { set_error("engine not bound"); return -2; }
    MS_CHECK_CUDA(cudaMemcpyAsync(e->proxy, proxy, (size_t)e->B * e->H * e->W * sizeof(float), cudaMemcpyDefault, S(stream)));
    return 0;
}
int ms_engine_set_loss(void* h, int kind, float weight_full, float weight_module) {
    Engine* e = static_cast<Engine*>(h);
    if (kind != 0 && kind != 1) { set_error("ms_engine_set_loss: kind must be 0 (reprojection) or 1 (proxy L1)"); return -2; }
    if (kind != e->loss_kind || weight_full != e->proxy_w_full || weight_module != e->proxy_w_module) {
        for (auto& g : e->graphs) cudaGraphExecDestroy(g.second.exec);       // the loss kernels are baked into the step graphs
        e->graphs.clear();
    }
    e->loss_kind = kind; e->proxy_w_full = weight_full; e->proxy_w_module = weight_module;
    return 0;
}
int ms_engine_forward(void* h, int disp_mask, void* stream) { return static_cast<Engine*>(h)->forward(disp_mask, S(stream)); }
int ms_engine_loss(void* h, int which, int with_grad, int slot, float grad_scale, void* stream) {
    return static_cast<Engine*>(h)->loss(which, with_grad, slot, grad_scale, S(stream));
}
int ms_engine_backward(void* h, int mode, int group, void* stream) {
    return static_cast<Engine*>(h)->backward(mode, group, S(stream));
}
int ms_engine_update(void* h, int group, float lr, float mu, float grad_scale, void* stream) {
    return static_cast<Engine*>(h)->update(group, lr, mu, grad_scale, S(stream));
}
int ms_engine_dp_create(void* h, int rank, int world, unsigned char* handles_out128) {
    return static_cast<Engine*>(h)->dp_create(rank, world, handles_out128);
}
int ms_engine_dp_connect(void* h, const unsigned char* all_handles) { return static_cast<Engine*>(h)->dp_connect(all_handles); }
int ms_engine_dp_error(void* h, unsigned int* out) { return static_cast<Engine*>(h)->dp_error(out); }
int ms_engine_run(void* h, int mode, int group, int disp_mask, int with_update, float lr, float mu, float grad_scale,
                  void* stream) {
    return static_cast<Engine*>(h)->run(mode, group, disp_mask, with_update, lr, mu, grad_scale, S(stream));
}
int ms_engine_weights_changed(void* h) {
    static_cast<Engine*>(h)->weights_dirty = true;
    return 0;
}
int ms_engine_metrics(void* h, void* stream) {
    Engine* e = static_cast<Engine*>(h);
    if (!e->bound) { set_error("engine not bound"); return -2; }
    return epe_bad3(e->disp[e->n_disp - 1].p, e->gt, e->B * e->H * e->W, e->scalars + 2, e->loss_ws, S(stream));
}
int ms_engine_read_scalars(void* h, float* host4, void* stream) {
    Engine* e = static_cast<Engine*>(h);
    if (!e->bound) { set_error("engine not bound"); return -2; }
    MS_CHECK_CUDA(cudaMemcpyAsync(host4, e->scalars, 4 * sizeof(float), cudaMemcpyDeviceToHost, S(stream)));
    MS_CHECK_CUDA(cudaStreamSynchronize(S(stream)));
    return 0;
}
int ms_engine_profile(void* h, int enable) {
    Engine* e = static_cast<Engine*>(h);
    e->profiling = enable < 0 ? 0 : (enable > 2 ? 2 : enable);     // 1 = eager events, 2 = event nodes inside the replayed graph
    if (enable) e->prof_reset();
    return 0;
}
int ms_engine_profile_read(void* h, double* ms7, double* macs7, double* bytes7, long long* calls7) {
    Engine* e = static_cast<Engine*>(h);
    if (e->prof_collect()) return -1;
    for (int i = 0; i < Engine::N_CAT; ++i) {
        if (ms7) ms7[i] = e->cat_ms[i];
        if (macs7) macs7[i] = e->cat_macs[i];
        if (bytes7) bytes7[i] = e->cat_bytes[i];
        if (calls7) calls7[i] = e->cat_calls[i];
    }
    return 0;
}
int ms_engine_profile_layers(void* h, double* ms3n, long long* calls3n) {
    Engine* e = static_cast<Engine*>(h);
    if (e->prof_collect()) return -1;
    const size_t n = e->layers.size();
    for (int d = 0; d < 3; ++d)
        for (size_t i = 0; i < n; ++i) {
            ms3n[d * n + i] = i < e->layer_ms[d].size() ? e->layer_ms[d][i] : 0.0;
            calls3n[d * n + i] = i < e->layer_calls[d].size() ? e->layer_calls[d][i] : 0;
        }
    return 0;
}
float ms_engine_profile_event_overhead_ms(void* h) { return static_cast<Engine*>(h)->prof_event_overhead_ms; }
long long ms_launch_count(void) { return ms::launch_count(); }
int ms_debug_bf_prof(unsigned long long* out, int max_ctas) { return ms::conv_bf_read_prof(out, max_ctas); }
int ms_engine_num_tensors(void* h) { return (int)static_cast<Engine*>(h)->tensors.size(); }
int ms_engine_tensor_name(void* h, int i, char* name, int cap) {
    Engine* e = static_cast<Engine*>(h);
    if (i < 0 || i >= (int)e->tensors.size()) { set_error("tensor index out of range"); return -2; }
    auto it = e->tensors.begin();
    std::advance(it, i);
    copy_str(name, cap, it->first);
    return 0;
}
int ms_engine_tensor(void* h, const char* name, float** ptr, int* dims5) {
    Engine* e = static_cast<Engine*>(h);
    auto it = e->tensors.find(name);
    if (it == e->tensors.end()) { set_error(std::string("unknown tensor: ") + name); return -2; }
    if (ptr) *ptr = it->second.p;
    if (dims5) { dims5[0] = it->second.n; dims5[1] = it->second.h; dims5[2] = it->second.w; dims5[3] = it->second.c; dims5[4] = it->second.cs; }
    return 0;
}

}  // extern "C"
