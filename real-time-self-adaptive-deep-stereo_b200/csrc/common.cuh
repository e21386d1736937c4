// Shared declarations for libmadstereo (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

namespace ms {

// NHWC fp32 view: `cs` = floats between consecutive pixels (>= c), so that a tensor can live as a
// channel slice of a wider concat buffer (zero-copy tf.concat).
struct TView {
    float* p;
    int n, h, w, c, cs;
    __host__ __device__ size_t pixels() const { return (size_t)n * h * w; }
};

inline TView view(float* p, int n, int h, int w, int c, int cs = 0) {
    TView v; v.p = p; v.n = n; v.h = h; v.w = w; v.c = c; v.cs = cs ? cs : c; return v;
}
inline TView slice(const TView& t, int c0, int c) { TView v = t; v.p = t.p + c0; v.c = c; return v; }
inline TView batch(const TView& t, int n0, int n) {
    TView v = t; v.p = t.p + (size_t)n0 * t.h * t.w * t.cs; v.n = n; return v;
}

void set_error(const std::string& s);
int check_launch(const char* what, int n_kernels = 1);
long long launch_count();
void add_launches(long long n);

#define MS_CHECK_CUDA(expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            ms::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                \
            return -1;                                                                        \
        }                                                                                     \
    } while (0)

#define MS_REQUIRE(cond, msg)                                                                 \
    do {                                                                                      \
        if (!(cond)) { ms::set_error(std::string("requirement failed: ") + msg); return -2; } \
    } while (0)

// ---------------------------------------------------------------------------------------------
// programmatic dependent launch (PDL): every kernel of the step starts with pdl_prologue() and is launched through
// launch_k(), which sets cudaLaunchAttributeProgrammaticStreamSerialization (MS_PDL=0 disables).  A kernel's CTAs may
// then become resident while the previous kernel of the stream is still draining; nothing of the kernel body runs before
// that kernel has completed and flushed (griddepcontrol.wait), so the data dependences of the stream order are intact --
// what overlaps is launch latency and, in the tcgen05 kernels, barrier / TMEM set-up.  Inside the captured step graph the
// attribute becomes a programmatic edge.  Measured on the conv -> conv edges alone: 551 -> 561 FPS.
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_trigger(); pdl_wait(); }
#endif
bool pdl_enabled();
// MS_CARVEOUT=1: every kernel launched through launch_k() asks for the maximum shared-memory carve-out, so consecutive
// kernels of the step never make an SM re-partition L1 / shared memory (experiment; off by default)
void carveout_once(const void* kernel);
void pdl_set_suppressed(bool s);      // the instrumented (event-node) graphs of ms_engine_profile(2) are captured without PDL edges
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    carveout_once(reinterpret_cast<const void*>(kernel));
    (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);      // errors surface in check_launch()
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t cdivz(size_t a, size_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// conv geometry: generic "gather GEMM".  For output pixel (oy,ox) and tap (r,s) the gathered
// input coordinate is   t = o*mul + off + tap*step ;  if (div>1) { require t % div == 0; t /= div }.
//   forward conv      : mul=stride, off=-pad_before, step=+dilation, div=1
//   dgrad / conv_transpose : mul=1, off=+pad_before, step=-dilation, div=stride
// ---------------------------------------------------------------------------------------------
struct ConvGemm {
    TView x;              // gathered operand  [n, xh, xw, K-channels]
    const float* wmat;    // [taps][x.c][y.c] row-major
    const float* bias;    // [y.c] or nullptr
    TView y;              // output [n, yh, yw, N-channels]
    int kh, kw;
    int mul, off_y, off_x, step, div;
    float alpha;          // epilogue leaky slope (1 = linear)
    const float* mask; int mask_cs; float mask_alpha;   // optional: y *= (mask>0 ? 1 : mask_alpha)
    const float* res;  int res_cs;                      // optional: y += res (same channel index)
    int accumulate;       // y += existing y (applied before mask)
    float* part; size_t part_floats;   // optional split-K scratch (small grids): partial sums, then a reduce+epilogue pass
    int ksplit;           // set by conv_gemm()
};
int conv_gemm(const ConvGemm& p, cudaStream_t st);
size_t conv_gemm_part_floats();      // size of the split-K scratch the engine passes as ConvGemm::part

struct ConvWgrad {
    TView x;              // forward-conv input   [n, xh, xw, ci]
    TView dy;             // grad wrt conv pre-activation output [n, yh, yw, co]
    float* dw;            // [taps][ci][co]
    float* db;            // [co] or nullptr
    int kh, kw, stride, dil, pad_t, pad_l;
    float* workspace; size_t workspace_floats;   // split-K partials
    int accumulate;       // dw += (shared weights called twice); normally 0
};
int conv_wgrad(const ConvWgrad& p, cudaStream_t st);
// conv_stem.cu: DispNet conv1 (7x7 stride 2, 3 -> 64) on the CUDA cores, forward and weight gradient
bool conv_stem_fwd_supported(const ConvGemm& g);
struct ActPlanes;
int conv_stem_fwd(const ConvGemm& g, const ActPlanes* yp, cudaStream_t st);
bool conv_stem_wgrad_supported(const ConvWgrad& q);
size_t conv_stem_wgrad_workspace_floats(const ConvWgrad& q);
int conv_stem_wgrad(const ConvWgrad& q, cudaStream_t st);
// conv_head.cu: weight gradient of a single-output-channel conv (disparity heads, DispNet up_predict)
bool conv_head_wgrad_supported(const ConvWgrad& q);
size_t conv_head_wgrad_workspace_floats(const ConvWgrad& q);
int conv_head_wgrad(const ConvWgrad& q, cudaStream_t st);
size_t conv_wgrad_workspace_floats(int taps, int ci, int co, size_t pixels);

// conv_small.cu: direct kernels for the full-resolution 3->16 / 16->16 pyramid layers
bool conv_small_fwd_supported(const ConvGemm& p);
int conv_small_fwd(const ConvGemm& p, cudaStream_t st);
bool conv_small_wgrad_shape(int taps, int ci, int co);
bool conv_small_wgrad_supported(const ConvWgrad& p);
size_t conv_small_wgrad_workspace_floats(int taps, int ci, int co, size_t pixels);
int conv_small_wgrad(const ConvWgrad& p, int* split_out, cudaStream_t st);

int bias_grad(const TView& dy, float* db, float* workspace, size_t workspace_floats, cudaStream_t st);
int transpose_taps(const float* w, float* wt, int taps, int ci, int co, cudaStream_t st);

// correlation / warp (corr.cu)
struct CorrFwd {
    const float* left;  int lcs;     // [B,h,w,C] view
    const float* right; int rcs;     // [B,h,w,C] view (un-warped)
    const float* u;     int ucs;     // optional [B,h,w,1] horizontal offsets (nullptr = no warp)
    float* out; int ocs;             // cost buffer: channels [0,C)=left (if copy_left), [C,C+nd)=corr
    float* out2; int o2cs;           // optional 2nd destination for the left copy (context input)
    int B, h, w, C, max_disp, stride, copy_left;
    int u_chan;                      // 1 if the concat buffer keeps a `u` channel right after the corr channels
    float plane_scale;               // > 0: power-of-two scale s with |feature * s| < 65504 -- enables the fp16 hi/lo banded
                                     // tensor-core kernel for wide windows (corr_mma.cu); 0: CUDA-core kernels only
};
int corr_fwd(const CorrFwd& p, cudaStream_t st);
int corr_init();
int mma_probe(int a_mn, int b_mn, int n, int n_acc, int rot, int iters, int uni, int ctas, long long* out_dev, cudaStream_t st);   // wgrad_bf.cu (diagnosis)
bool corr_mma_supported(const CorrFwd& p);          // corr_mma.cu: wide window (>= 17 displacements), no warp, stride 1
int corr_mma(const CorrFwd& p, cudaStream_t st);
int corr_fwd4(const CorrFwd& p, cudaStream_t st);   // corr_tma.cu: 0 launched, 1 shape not handled, -1 error

struct CorrBwd {
    const float* left;  int lcs;
    const float* right; int rcs;
    const float* u;     int ucs;     // nullptr = no warp
    const float* dcost; int dcs;     // grad of cost buffer; corr grads at channel offset C
    float* dleft;  int dlcs;         // out: d(left feature)  = dcost[:, :C]*add_left_slice + corr term
    float* dright; int drcs;         // out: d(right feature) (scatter through the warp)
    float* du;     int ducs;         // optional out: d(u) from the warp coordinates (FULL mode)
    int B, h, w, C, max_disp, stride, add_left_slice, acc_left, acc_right;
    int gcoff;                       // channel offset of the corr grads inside dcost (-1 => C, the concat layout)
};
int corr_bwd(const CorrBwd& p, cudaStream_t st);
bool corr_mma_bwd_supported(const CorrBwd& p);       // corr_mma.cu: wide window, no warp, stride 1, C in {32, 64, 96, 128}
int corr_mma_bwd(const CorrBwd& p, cudaStream_t st);

// elementwise / resampling (elementwise.cu)
int pad_reflect(const float* src, int B, int H, int W, int C, float* dst, int Hp, int Wp, int dcs,
                float scale, float bias, cudaStream_t st);
// dst = post( resize_bilinear_legacy( pre(src) ) ) cropped (centre) to [oh,ow] from [rh,rw]
//   pre(v)  = pre_relu ? max(v*pre_scale,0) : v*pre_scale ;  post(v) = post_relu ? max(v*post_scale,0) : v*post_scale
int resize_bilinear(const float* src, int scs, int B, int ih, int iw, float* dst, int dcs, int rh, int rw,
                    int oh, int ow, float pre_scale, int pre_relu, float post_scale, int post_relu,
                    cudaStream_t st);
// gradient of the above wrt src (gather form, deterministic). needs src for the relu masks.
int resize_bilinear_bwd(const float* dout, int docs, const float* src, int scs, int B, int ih, int iw,
                        float* dsrc, int dscs, int rh, int rw, int oh, int ow, float pre_scale, int pre_relu,
                        float post_scale, int post_relu, int accumulate, float* tmp /* B*oh*iw floats */,
                        cudaStream_t st);
int leaky_bwd(float* g, int gcs, const float* act, int acs, size_t pixels, int c, float alpha, cudaStream_t st);
int add_channels(float* dst, int dcs, const float* src, int scs, size_t pixels, int c, float scale,
                 int accumulate, cudaStream_t st);
int fill(float* p, size_t n, float v, cudaStream_t st);
int u8_to_f32(const unsigned char* src, float* dst, size_t n, cudaStream_t st);

// loss (loss.cu)
struct ReprojLoss {
    const float* left; const float* right;   // [B,H,W,3], 0..255
    const float* disp;                        // [B,H,W,1]
    float* loss;                              // device scalar out
    float* ddisp;                             // optional [B,H,W,1] gradient out (nullptr = forward only)
    float* workspace;                         // >= loss_workspace_floats(B,H,W)
    int B, H, W;
    float grad_scale;                         // multiplies the gradient (1 for a single rank)
};
size_t loss_workspace_floats(int B, int H, int W);
int reproj_loss(const ReprojLoss& p, cudaStream_t st);
int epe_bad3(const float* disp, const float* gt, int n, float* out2, float* workspace, cudaStream_t st);
// masked mean-L1 against proxy disparities (loss_factory.get_proxy_loss('mean_l1')); workspace >= 2 * ceil(n/256) + 2 floats
int proxy_loss(const float* disp, const float* proxy, int n, float weight, float grad_scale, float* loss, float* ddisp,
               float* workspace, cudaStream_t st);

// optimizer (optim.cu)
int momentum_update(float* w, const float* g, float* m, size_t n, float lr, float mu, float gscale,
                    cudaStream_t st);

}  // namespace ms

namespace ms {
// 3xTF32 tcgen05 weight gradient of stride-1 convolutions (wgrad_tc.cu): the engine's weight gradient for the shapes the
// split-bf16 kernel does not take (DispNet's conv_redir, whose output gradient is a channel slice without bf16 planes)
bool wgrad_tc_supported(const ConvWgrad& q);
size_t wgrad_tc_workspace_floats(int taps, int ci, int co, int n, int h, int w);
int wgrad_tc_init();
int wgrad_tc(const ConvWgrad& q, cudaStream_t st);
}  // namespace ms

namespace ms {
// split-bf16 tcgen05 path (conv_bf.cu): every activation that feeds a convolution also lives as two bf16 planes
// (hi = bf16(x), lo = bf16(x - hi)), NHWC with channel stride `cs` (bf16 elements, multiple of 8).
struct ActPlanes { void* hi; void* lo; int cs; int fmt; float scale; };   // fmt 0 = bf16 (gradients), 1 = fp16 of x * scale (forward activations; scale a power of two)
struct BfPrepJob {
    const float* src; void* tiles;           // tiles: [M block][tap][K block][hi tile | lo tile], swizzled smem images
    int taps, M, K, Mpad, Kpad, transposed_src, fmt;
};
int conv_head_kind(const ConvGemm& g);      // conv_head.cu: 1 = forward 3x3 -> 1 head, 2 = its dgrad, 0 = no
int conv_head(const ConvGemm& g, cudaStream_t st);
bool conv_one_channel_supported(const ConvGemm& g);   // conv_head.cu: 1 -> 1 channel gather (any geometry)
int conv_one_channel(const ConvGemm& g, cudaStream_t st);
bool conv_bf_supported(const ConvGemm& g);
void conv_bf_weight_dims(int M, int K, int& Mpad, int& Kpad);
size_t conv_bf_weight_halfs(int taps, int M, int K);
size_t conv_bf_part_floats();
size_t conv_bf_ticket_words();
int conv_bf_init();
int conv_bf_read_prof(unsigned long long* out, int max_ctas);
int bf_prep_weights(const BfPrepJob* jobs_dev, int njobs, size_t max_total, cudaStream_t st);
int split_planes(const TView& x, const ActPlanes& pl, cudaStream_t st);
int conv_bf(const ConvGemm& g, const ActPlanes& xp, const void* wtiles, const ActPlanes* yp, float* part,
            unsigned int* tickets, cudaStream_t st);
// wgrad_bf.cu: weight + bias gradient on the same planes (MN-major UMMA operands, no transposes)
bool wgrad_bf_supported(const ConvWgrad& q);
size_t wgrad_bf_workspace_floats(int kh, int kw, int ci, int co);
int wgrad_bf_init();
int wgrad_bf(const ConvWgrad& q, const ActPlanes& xp, const ActPlanes& dp, cudaStream_t st);
size_t wgrad_bf_oneshot_scratch_bytes(const ConvWgrad& q);
int wgrad_bf_oneshot(const ConvWgrad& q, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t conv_bf_oneshot_scratch_bytes(const ConvGemm& g);
int conv_bf_oneshot(const ConvGemm& g, int wmat_is_mk, int fmt, float act_scale, void* scratch, size_t scratch_bytes, cudaStream_t st);
}  // namespace ms
