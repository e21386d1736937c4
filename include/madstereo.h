/* libmadstereo — C ABI of the B200-native real-time self-adaptive stereo engine.
 *
 * Drop-in boundary for ONE hot path of CVLAB-Unibo/Real-time-self-adaptive-deep-stereo: the per-frame
 * MADNet/DispNet forward + (MAD | FULL) backward + momentum update.  Every entry point names the reference
 * interface it replaces (paths relative to the reference checkout).
 *
 * Conventions: all tensors are NHWC fp32 in DEVICE memory owned by the caller; `cs` arguments are channel
 * strides in floats (>= channels) so tensors can live inside concat buffers; `stream` is a cudaStream_t
 * passed as void*; every function returns 0 on success and a negative code on failure, with the message
 * available from ms_last_error().  Nothing allocates on the step path.  One host thread per GPU.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef MADSTEREO_H
#define MADSTEREO_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

int ms_version(void);
const char* ms_last_error(void);

/* ---- operator level ------------------------------------------------------------------------------ */

/* Replaces ShiftCorrKernelLauncher (Nets/Native/shift_corr.cu.cc:193-233), the TF op "ShiftCorr"
 * (Nets/Native/shift_corr.cc:5-9,25-56) and sharedLayers.correlation / correlation_tf
 * (Nets/sharedLayers.py:23-51).  Unlike the native op the inputs are NOT pre-padded and the output is NHWC.
 *   out[b,y,x,out_coff+i] = mean_c left[b,y,x,c] * RW[b,y,x+(-max_disp+i*stride),c]
 * `u` (optional, may be NULL) fuses MadNet._linear_warping (Nets/MadNet.py:400-436) of `right` by the
 * horizontal offsets u[b,y,x].  copy_left != 0 additionally writes left into out[...,0:C] (the tf.concat of
 * MadNet._stereo_cost_volume_correlation, Nets/MadNet.py:370-375) and the corr channels start at C. */
int ms_corr_fwd(const float* left, int left_cs, const float* right, int right_cs, const float* u, int u_cs,
                float* out, int out_cs, int B, int h, int w, int C, int max_disp, int stride, int copy_left,
                int u_chan, void* stream);

/* Wide-window variant for DispNet-C (Nets/DispNet.py:92-101 -> Nets/sharedLayers.py:23-51 with max_disp = 40): the band
 * |x' - x| <= max_disp of L R^T per image row on mma.sync tensor-core tiles, fp16 hi/lo operands split on the fly
 * (x * act_scale = hi + lo, three MMAs per product, fp32 accumulation).  out channels [0, 2*max_disp+1) of a buffer with
 * channel stride out_cs.  act_scale: power of two with |feature * act_scale| < 65504 (the engine passes its activation
 * scale).  csrc/corr_mma.cu. */
int ms_corr_fwd_wide(const float* left, int left_cs, const float* right, int right_cs, float* out, int out_cs, int B, int h,
                     int w, int C, int max_disp, float act_scale, void* stream);

/* Replaces ShiftCorrGradKernelLauncher (Nets/Native/shift_corr.cu.cc:235-289) / TF op "ShiftCorrGrad"
 * (Nets/Native/shift_corr.cc:11-17,62-93) with the mathematical gradient of correlation_tf (the native
 * backward is defective: wrong input wiring shift_corr.cc:76, CHW/NHWC mix-up and out-of-bounds writes
 * shift_corr.cu.cc:80,129,143,187).  dcost holds corr grads at channel offset C (and, if add_left_slice,
 * the concat-slice grads of `left` at [0,C)).  du (optional) receives the warp-coordinate gradient. */
int ms_corr_bwd(const float* left, int left_cs, const float* right, int right_cs, const float* u, int u_cs,
                const float* dcost, int dcost_cs, float* dleft, int dleft_cs, float* dright, int dright_cs,
                float* du, int du_cs, int B, int h, int w, int C, int max_disp, int stride, int add_left_slice,
                void* stream);

/* Replaces sharedLayers.conv2d / dilated_conv2d (Nets/sharedLayers.py:54-77): act(conv2d_SAME(x,W)+b),
 * W in HWIO, act = max(alpha*v, v) (alpha = 1 -> linear). */
int ms_conv2d_fwd(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights /*HWIO*/,
                  const float* bias, float* y, int cout, int y_cs, int kh, int kw, int stride, int dilation,
                  float alpha, void* stream);
/* Gradients tf.gradients derives for the op above.  dy = grad wrt the PRE-activation output.
 * scratch: >= kh*kw*cin*cout floats (dgrad) / ms_conv2d_wgrad_workspace() floats (wgrad). */
int ms_conv2d_dgrad(const float* dy, int n, int oh, int ow, int cout, int dy_cs, const float* weights,
                    float* dx, int h, int w, int cin, int dx_cs, int kh, int kw, int stride, int dilation,
                    float* scratch, void* stream);
/* Split-16-bit tcgen05 path (csrc/conv_bf.cu; the engine's implementation of every eligible layer): operands as two
 * 16-bit planes (x ~= hi + lo), three kind::f16 MMAs per K step at the bf16/fp16 tensor rate.  Forward operands are
 * fp16 planes of x * act_scale and of w (22 mantissa bits, ~2^-22 relative
 * product error; the power-of-two scale is undone exactly in the epilogue); gradient operands are bf16 planes (16 bits, fp32 exponent
 * range).  GEMM transposed so that M = output channels and N = up to 256 pixels, halo patches by TMA (64-channel K
 * blocks), pre-tiled weights by 1-D bulk copies, stride 1 or 2 (TMA element strides), any dilation, split-K reduced by
 * the last-arriving CTA.  Same semantics as ms_conv2d_fwd / ms_conv2d_dgrad (a stride-2 dgrad runs as four dense
 * parity-class launches).  scratch: ms_conv2d_bf_scratch() BYTES, 256-byte aligned.  -3 = not eligible. */
int ms_conv2d_fwd_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights /*HWIO*/,
                     const float* bias, float* y, int cout, int y_cs, int kh, int kw, int stride, int dilation,
                     float alpha, float act_scale /* power of two: the fp16 planes hold x * act_scale */, void* scratch,
                     size_t scratch_bytes, void* stream);
int ms_conv2d_dgrad_bf(const float* dy, int n, int oh, int ow, int cout, int dy_cs, const float* weights /*HWIO*/,
                       float* dx, int h, int w, int cin, int dx_cs, int kh, int kw, int stride, int dilation,
                       void* scratch, size_t scratch_bytes, void* stream);
size_t ms_conv2d_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout);
/* tcgen05 weight + bias gradient on the same planes (csrc/wgrad_bf.cu; the engine's default for eligible layers):
 * replaces the filter / bias gradient sub-graphs of tf.nn.conv2d / atrous_conv2d / bias_add (reference
 * Nets/sharedLayers.py:58-59,72-73 under the train ops of Stereo_Online_Adaptation.py:118,128).  x and dy planes feed
 * the UMMA as MN-major operands straight from NHWC; stride 1 or 2, any dilation.  Same outputs as ms_conv2d_wgrad.
 * Both plane sets are bf16 (tcgen05 kind::f16 rejects an f16 x bf16 operand pair: probed, illegal instruction; the engine
 * therefore re-splits the forward activation into bf16 scratch planes for this kernel).
 * scratch: ms_conv2d_wgrad_bf_scratch() BYTES, 256-byte aligned.  -3 = not eligible. */
int ms_conv2d_wgrad_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int oh, int ow, int cout,
                       int dy_cs, float* dw /*HWIO*/, float* db, int kh, int kw, int stride, int dilation,
                       void* scratch, size_t scratch_bytes, void* stream);
size_t ms_conv2d_wgrad_bf_scratch(int n, int h, int w, int oh, int ow, int kh, int kw, int cin, int cout);
/* Plane-level entry points of the same path (what the engine issues per layer in steady state: activations are split
 * by the producing kernel's epilogue, weights once per update).  hi / lo planes: 16-bit NHWC, channel stride `*_pcs`
 * (multiple of 8), fmt 0 = bf16, 1 = fp16 of value * scale (scale a power of two); weight tiles: ms_bf_weight_halfs() 16-bit elements (both planes,
 * pre-tiled shared-memory images); job_dev: >= 64 bytes of device scratch; part / tickets:
 * ms_conv2d_bf_part_floats() floats / ms_conv2d_bf_ticket_words() zeroed words (split-K). */
int ms_bf_split(const float* x, int n, int h, int w, int c, int x_cs, void* hi, void* lo, int plane_cs, int fmt, float scale,
                void* stream);
size_t ms_bf_weight_halfs(int taps, int m, int k);
int ms_bf_prep_weights(const float* weights_hwio, int taps, int cin, int cout, int for_dgrad, int fmt, void* tiles,
                       void* job_dev, void* stream);
int ms_conv2d_fwd_bf_planes(const void* xhi, const void* xlo, int x_pcs, int fmt, float scale, int n, int h, int w, int cin,
                            const void* wtiles, const float* bias, float* y, int cout, int y_cs, void* yhi, void* ylo,
                            int y_pcs, int kh, int kw, int stride, int dilation, float alpha, float* part,
                            unsigned int* tickets, void* stream);
size_t ms_conv2d_bf_part_floats(void);
size_t ms_conv2d_bf_ticket_words(void);
int ms_conv2d_wgrad_bf_planes(const void* xhi, const void* xlo, int x_pcs, int n, int h, int w, int cin,
                              const void* dhi, const void* dlo, int d_pcs, int oh, int ow, int cout, float* dw, float* db,
                              int kh, int kw, int stride, int dilation, float* workspace, size_t workspace_floats, void* stream);
size_t ms_conv2d_wgrad_bf_workspace(int kh, int kw, int cin, int cout);
/* 3xTF32 tcgen05 weight gradient of a stride-1 conv (same outputs as ms_conv2d_wgrad); the engine uses it for the layers
 * whose output gradient has no bf16 planes.  workspace from ..._workspace().  -3 = not eligible. */
int ms_conv2d_wgrad_tc(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int cout, int dy_cs,
                       float* dw /*HWIO*/, float* db, int kh, int kw, int dilation, float* workspace,
                       size_t workspace_floats, void* stream);
size_t ms_conv2d_wgrad_tc_workspace(int kh, int kw, int cin, int cout, int n, int h, int w);
size_t ms_conv2d_wgrad_workspace(int kh, int kw, int cin, int cout, size_t out_pixels);
int ms_conv2d_wgrad(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int oh, int ow,
                    int cout, int dy_cs, float* dw /*HWIO*/, float* db, int kh, int kw, int stride,
                    int dilation, float* workspace, size_t workspace_floats, void* stream);
/* Replaces sharedLayers.conv2d_transpose (Nets/sharedLayers.py:80-92); weights [kh,kw,cout,cin]. */
int ms_conv2d_transpose_fwd(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights,
                            const float* bias, float* y, int cout, int y_cs, int kh, int kw, int stride,
                            float alpha, float* scratch, void* stream);

/* DispNet conv1 -- sharedLayers.conv2d 7x7 stride 2, 3 -> 64 (Nets/DispNet.py:82-86; Nets/sharedLayers.py:54-63) -- and its
 * filter / bias gradient on direct CUDA-core kernels (csrc/conv_stem.cu): with 3 input channels the tensor-core tiles are
 * 90 % padding.  x4: [n,h,w,3] stored with a channel stride of 4 floats; weights HWIO [7,7,3,64]; y / dy [n,ceil(h/2),
 * ceil(w/2),64]; workspace: ms_conv2d_stem_wgrad_workspace floats. */
int ms_conv2d_stem_fwd(const float* x4, int n, int h, int w, const float* weights, const float* bias, float* y, int y_cs,
                       float alpha, void* stream);
size_t ms_conv2d_stem_wgrad_workspace(int n, int h, int w);
int ms_conv2d_stem_wgrad(const float* x4, int n, int h, int w, const float* dy, int dy_cs, float* dw, float* db, float* workspace,
                         size_t workspace_floats, void* stream);

/* The same layer and its two gradients on the split-16-bit tcgen05 path (csrc/conv_bf.cu, csrc/wgrad_bf.cu): forward as a
 * fractionally strided gather in four output-parity launches (fp16 planes of x*act_scale), input gradient as the
 * stride-`stride` conv of dy with the filter read as HWIO [kh,kw,cout,cin], weight gradient as that conv's wgrad with the
 * big map in the activation role (both bf16 planes).  dy [n,h*stride,w*stride,cout]; dw [kh,kw,cout,cin]; db [cout] or NULL.
 * Backward of Nets/sharedLayers.py:80-92 as tf.gradients derives it (Stereo_Online_Adaptation.py:143-151).
 * scratch: 256-byte aligned, ms_conv2d_transpose_bf_scratch / ms_conv2d_transpose_wgrad_bf_scratch bytes. */
int ms_conv2d_transpose_fwd_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* weights, const float* bias,
                               float* y, int cout, int y_cs, int kh, int kw, int stride, float alpha, float act_scale,
                               void* scratch, size_t scratch_bytes, void* stream);
int ms_conv2d_transpose_dgrad_bf(const float* dy, int n, int h, int w, int cout, int dy_cs, const float* weights, float* dx,
                                 int cin, int dx_cs, int kh, int kw, int stride, void* scratch, size_t scratch_bytes,
                                 void* stream);
size_t ms_conv2d_transpose_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout, int stride);
int ms_conv2d_transpose_wgrad_bf(const float* x, int n, int h, int w, int cin, int x_cs, const float* dy, int cout, int dy_cs,
                                 float* dw, float* db, int kh, int kw, int stride, void* scratch, size_t scratch_bytes,
                                 void* stream);
size_t ms_conv2d_transpose_wgrad_bf_scratch(int n, int h, int w, int kh, int kw, int cin, int cout, int stride);


/* Replaces tf.image.resize_images (legacy bilinear) + resize_image_with_crop_or_pad + the relu/scale
 * of MadNet._make_disp (Nets/MadNet.py:68-71,274,362-364): dst = post(resize(pre(src)))[centre crop]. */
int ms_resize_bilinear(const float* src, int src_cs, int B, int ih, int iw, float* dst, int dst_cs, int rh,
                       int rw, int oh, int ow, float pre_scale, int pre_relu, float post_scale, int post_relu,
                       void* stream);
int ms_resize_bilinear_bwd(const float* dout, int dout_cs, const float* src, int src_cs, int B, int ih, int iw,
                           float* dsrc, int dsrc_cs, int rh, int rw, int oh, int ow, float pre_scale,
                           int pre_relu, float post_scale, int post_relu, int accumulate,
                           float* tmp /* B*oh*iw floats */, void* stream);

/* Replaces loss_factory.get_reprojection_loss('mean_SSIM_l1') (Losses/loss_factory.py:353-395) with
 * preprocessing.warp_image (Data_utils/preprocessing.py:121-230); ddisp may be NULL (forward only). */
size_t ms_reproj_loss_workspace(int B, int H, int W);
int ms_reproj_loss(const float* left, const float* right, const float* disp, int B, int H, int W,
                   float* loss_out /*device scalar*/, float* ddisp, float* workspace, float grad_scale,
                   void* stream);

/* Replaces tf.train.MomentumOptimizer(lr,0.9) apply ops (Stereo_Online_Adaptation.py:85,118,128). */
int ms_momentum_update(float* w, const float* g, float* m, size_t n, float lr, float mu, float grad_scale,
                       void* stream);

/* Replaces preprocessing.pad_image REFLECT padding (Data_utils/preprocessing.py:7-29). */
int ms_pad_reflect(const float* src, int B, int H, int W, int C, float* dst, int Hp, int Wp, int dst_cs,
                   float scale, float bias, void* stream);

/* ---- engine level: what one sess.run(fetches) does (Stereo_Online_Adaptation.py:194-208) ---------- */

/* Replaces Nets.get_stereo_net(name,args) graph construction (Nets/__init__.py:9-13, Nets/MadNet.py:251-364).
 * net_name: "MADNet" | "Dispnet".  Returns NULL on failure. */
void* ms_engine_create(const char* net_name, int B, int H, int W, int radius_d, int corr_stride, int warping);
int ms_engine_destroy(void* e);
int ms_engine_num_layers(void* e);
/* dims: kh,kw,cin,cout,stride,dilation,transposed ; alpha_out: leaky slope (1 = linear) */
int ms_engine_layer_info(void* e, int i, char* name, int name_cap, char* scope, int scope_cap, char* bias_name,
                         int bias_cap, int* dims7, float* alpha_out);
/* Replaces the per-module var_list construction from block_config JSON (Stereo_Online_Adaptation.py:110-118,
 * Nets/Stereo_net.py:213-222): group_of_layer[i] = MAD module index of layer i, or -1. Fixes the arena order. */
int ms_engine_set_groups(void* e, const int* group_of_layer, int n_layers, int n_groups);
int ms_engine_sizes(void* e, size_t* n_param_floats, size_t* workspace_floats);
int ms_engine_param_offsets(void* e, int i, size_t* w_off, size_t* b_off);
int ms_engine_group_range(void* e, int g, size_t* begin, size_t* end);
int ms_engine_bind(void* e, float* weights, float* grads, float* momentum, float* workspace,
                   size_t workspace_floats, void* stream);
/* left/right: [B,H,W,3] fp32 0..255, host (pinned recommended) or device pointers. */
int ms_engine_set_input(void* e, const float* left, const float* right, void* stream);
/* the same with uint8 frames [B,H,W,3] (host or device): what the reference's decode ops deliver before tf.cast
 * (Data_utils/data_reader.py); converted to fp32 on the device. */
int ms_engine_set_input_u8(void* e, const unsigned char* left, const unsigned char* right, void* stream);
int ms_engine_set_gt(void* e, const float* gt, void* stream);
/* Continual-adaptation variant (reference Stereo_Continual_Adaptation.py:75,112,133; Losses/loss_factory.py:304-351
 * get_proxy_loss('mean_l1')): proxy disparities [B,H,W,1] (host or device) and the loss selector.  kind 0 = reprojection
 * SSIM + L1 (default), 1 = weight * sum(valid * |d - proxy|) / sum(valid) with valid = !(proxy <= 0 || proxy >= 192);
 * weight_full (reference 0.01) for the full-resolution loss / FULL train op, weight_module (0.1) for the MAD module losses.
 * Changing the loss drops the captured step graphs. */
int ms_engine_set_proxy(void* e, const float* proxy, void* stream);
int ms_engine_set_loss(void* e, int kind, float weight_full, float weight_module);
/* disp_mask bit i => materialise get_disparities()[i] (MADNet: D6,D5,D4,D3,D2ctx,full). */
int ms_engine_forward(void* e, int disp_mask, void* stream);
/* slot 0 = full-res loss fetched every frame (Stereo_Online_Adaptation.py:70,209), slot 1 = train loss */
int ms_engine_loss(void* e, int which_disp, int with_grad, int slot, float grad_scale, void* stream);
/* mode 1 = MAD (train op `group`, Stereo_Online_Adaptation.py:87-121), 2 = FULL (:126-128) */
int ms_engine_backward(void* e, int mode, int group, void* stream);
int ms_engine_update(void* e, int group /* -1 = all */, float lr, float mu, float grad_scale, void* stream);
/* One whole frame = what a single sess.run(tf_fetches) executes (Stereo_Online_Adaptation.py:194-208):
 * forward, full-res loss (slot 0), and for mode 1/2 the train op (module loss in slot 1, backward,
 * momentum update if with_update).  After the first call per (mode, group, ...) the sequence is replayed as
 * ONE CUDA graph launch.  with_update=0 leaves the gradients in the arena for an external all-reduce
 * followed by ms_engine_update; with_update=2 (after ms_engine_dp_connect) appends the data-parallel exchange to the
 * same graph: one kernel all-reduces the module's gradient range + the loss scalars over NVLink peer memory and
 * applies the momentum update with the 1/N mean folded in (csrc/dp.cu). */
/* Data parallel (new functionality, SURVEY 8e; the reference is single-GPU): one process per GPU.  dp_create allocates
 * this rank's exchange buffer + flag block and returns their two 64-byte CUDA IPC handles; the caller all-gathers the
 * 128 bytes of every rank (any transport) and passes world x 128 bytes to dp_connect.  dp_error: 0 ok, 1 peer
 * timeout, 2 ranks disagreed on the module being adapted. */
int ms_engine_dp_create(void* e, int rank, int world, unsigned char* handles_out128);
int ms_engine_dp_connect(void* e, const unsigned char* all_handles);
int ms_engine_dp_error(void* e, unsigned int* out);
int ms_engine_run(void* e, int mode, int group, int disp_mask, int with_update, float lr, float mu,
                  float grad_scale, void* stream);
/* Tell the engine that the weight arena was written from outside (checkpoint load / divergence reset). */
int ms_engine_weights_changed(void* e);
/* scalars: [0]=slot-0 loss, [1]=slot-1 loss, [2]=EPE, [3]=bad3. Synchronises `stream`. */
int ms_engine_read_scalars(void* e, float* host4, void* stream);
int ms_engine_metrics(void* e, void* stream);
/* Profiling aid for bench.py (no reference counterpart): CUDA events around kernel groups on the launching
 * stream.  Categories: 0 conv fwd, 1 conv dgrad, 2 conv wgrad, 3 corr fwd, 4 corr bwd, 5 loss, 6 other.
 * Arrays have 7 entries: summed device ms, algorithmic MACs, algorithmic bytes, number of timed calls. */
/* enable: 0 off; 1 eager steps with CUDA events between launches; 2 = the step still replays as ONE CUDA graph, with
 * external event-record nodes around every kernel group inside the graph (per-kernel times under the same launch
 * conditions as the timed replay; ms_engine_run then synchronises once per step to read them). */
int ms_engine_profile(void* e, int enable);
/* per layer and direction (0 fwd, 1 dgrad, 2 wgrad): accumulated milliseconds and call counts, arrays of 3 * num_layers */
int ms_engine_profile_layers(void* e, double* ms3n, long long* calls3n);
/* mode 2: the event-to-event latency of an EMPTY span inside the graph (already subtracted from every reported span) */
float ms_engine_profile_event_overhead_ms(void* e);
int ms_engine_profile_read(void* e, double* ms7, double* macs7, double* bytes7, long long* calls7);
/* Kernels launched by this library in this process so far. */
long long ms_launch_count(void);
/* Diagnosis: cycles per tcgen05.mma.kind::f16 (M = 128, K = 16, bf16) issued back to back by one thread per CTA on zeroed
 * shared memory, for K-major / MN-major operand layouts, MMA N, number of accumulators visited round-robin, and the
 * issue scheme (uni = 0: loop on lane 0 only; 1: warp-uniform loop, elected lane issues).  out_dev:
 * 2 * ctas int64 (issue-loop cycles, cycles until the last MMA retired).  scripts/mma_probe.py prints the table. */
int ms_debug_mma_probe(int a_mn, int b_mn, int n, int n_acc, int rot, int iters, int uni, int ctas, long long* out_dev, void* stream);

/* MS_BF_PROF=1: clock64 stamps of the last conv_bf launch, 8 per CTA (entry, setup done, first data, MMAs issued,
 * accumulator seen, epilogue done, exit, MMA-thread wait cycles); returns the number of CTAs copied */
int ms_debug_bf_prof(unsigned long long* out, int max_ctas);
int ms_engine_num_tensors(void* e);
int ms_engine_tensor_name(void* e, int i, char* name, int cap);
/* dims: n,h,w,c,cs */
int ms_engine_tensor(void* e, const char* name, float** ptr, int* dims5);

#ifdef __cplusplus
}
#endif
#endif
