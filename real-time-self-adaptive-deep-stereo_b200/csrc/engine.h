// Engine: per-frame MADNet / DispNet forward + (MAD | FULL) backward + momentum update, orchestrated in C++
// over caller-owned device memory.  Replaces what one `sess.run(fetches)` executes in the reference's inner
// loop (Stereo_Online_Adaptation.py:208) for the graphs built by Nets/MadNet.py and Nets/DispNet.py.
#pragma once
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "common.cuh"

namespace ms {

struct ConvLayer {
    std::string name;     // reference layer name as used in block_config JSON ("left/conv1", "context3", ...)
    std::string scope;    // TF variable scope ("model/gc-read-pyramid/conv1")
    std::string bname;    // "biases" (MADNet) or "bias" (DispNet)
    int kh, kw, cin, cout, stride, dil;
    float alpha;          // leaky slope, 1 = linear
    int transposed;       // conv2d_transpose (weights [kh,kw,cout,cin])
    size_t w_off, b_off;  // float offsets in the parameter arena
    int group;            // MAD module index or -1
};

constexpr int DP_MAX_WORLD = 8;
struct DpState {               // device-resident exchange state of one rank (IPC-mapped into every peer), csrc/dp.cu
    unsigned int ready[DP_MAX_WORLD];   // ready[src] = (epoch << 8) | module tag, written by rank src
    unsigned int done[DP_MAX_WORLD];    // done[src]  = last epoch rank src finished reading this rank's buffer
    unsigned int epoch, blocks_done, error, pad;
};

struct Bump {            // workspace bump allocator (sizes only when base == nullptr)
    float* base; size_t off;
    float* alloc(size_t n) { float* p = base ? base + off : nullptr; off += (n + 63) / 64 * 64; return p; }
    TView tens(int n, int h, int w, int c, int cs = 0) { cs = cs ? cs : c; return view(alloc((size_t)n * h * w * cs), n, h, w, c, cs); }
};

struct Engine {
    // configuration
    int net;              // 0 = MADNet, 1 = DispNet
    int B, H, W, Hp, Wp;
    int radius_d, corr_stride, warping;
    std::vector<ConvLayer> layers;
    int n_groups;
    std::vector<size_t> group_begin, group_end;   // float ranges in the arena
    size_t n_params;      // arena floats (incl. alignment pads)

    // bound memory
    float *Wt, *Gr, *Mo;  // weights / grads / momentum arenas
    float* ws; size_t ws_floats;
    bool bound;

    // tensors (valid after bind)
    std::map<std::string, TView> tensors;
    std::string last_plan_error;

    // ---- MADNet buffers
    TView img;                       // [2B,Hp,Wp,3] cs=4
    TView pyr[13], g_pyr[13];        // 1..12
    TView cost[7], g_cost[7];        // levels 2..6
    TView est[7][7], g_est[7][7];    // [level][1..5]
    TView V[7], g_V[7];              // [level] (V[2] is a slice of ctxin)
    TView g_u[7];
    TView ctxin, g_ctxin, ctx[8], g_ctx[8], final_, g_final;
    TView disp[7];                   // MADNet: D6,D5,D4,D3,D2ctx,full ; DispNet: up5..up1 predict, prediction, full
    int n_disp;
    TView g_disp;
    float* wT; size_t wT_floats;     // transposed-weight scratch
    float* gemm_part;                            // split-K partial sums of the fp32 conv_gemm on small maps
    bool weights_dirty;
    int prep_layers(int group, cudaStream_t st); // -1 = all
    // whole-step CUDA graphs keyed by (mode, group, disp_mask, with_update, lr, mu, gscale)
    struct GraphKey { int mode, group, mask, with_update, prof; float lr, mu, gs;
                      bool operator<(const GraphKey& o) const { return memcmp(this, &o, sizeof(GraphKey)) < 0; } };
    struct Span;
    struct GraphRec { cudaGraphExec_t exec; long long kernels; std::vector<Span>* spans; };
    std::map<GraphKey, GraphRec> graphs;
    int use_graphs;
    cudaStream_t gstream; cudaEvent_t ev_in, ev_out;   // graphs run on a private stream (the legacy default stream cannot be captured)
    // weight gradients on a side stream: wgrad(layer j) only needs dpre_j and the forward activation, so it runs concurrently
    // with the dgrad chain (fork / join through events; inside the captured step this becomes a parallel graph branch)
    int use_overlap;                                   // MS_WGRAD_OVERLAP (default 1; MADNet only, off while profiling)
    cudaStream_t wstream; cudaEvent_t ev_fork, ev_join; bool wstream_dirty;
    int fork_wgrad(cudaStream_t st, cudaStream_t* ws);
    int join_wgrad(cudaStream_t st);
    int backward_impl(int mode, int group, cudaStream_t st);
    int run(int mode, int group, int disp_mask, int with_update, float lr, float mu, float gscale, cudaStream_t st);
    int run_eager(int mode, int group, int disp_mask, int with_update, float lr, float mu, float gscale, cudaStream_t st);
    // ---- split-bf16 tcgen05 path (conv_bf.cu), the implementation of every eligible conv / dgrad
    int use_stem;                                  // direct CUDA-core kernels for DispNet conv1 (MS_STEM=0: tensor-core path)
    int use_bf_wgrad;                              // split-bf16 weight gradients (MS_BF_WGRAD=0: the 3xTF32 / fp32 kernels)
    int use_heads;                                 // direct kernels for the 3x3 -> 1 heads (MS_HEADS=0: generic path)
    std::map<const float*, ActPlanes> planes;      // bf16 hi/lo planes of tensors that feed convolutions (key: base pointer)
    std::set<const float*> fresh;                  // planes already written by a conv_bf epilogue in the current pass
    struct BfW { void* tiles; bool ok; };
    std::vector<BfW> bfw[2];                       // prepared weights per layer and orientation (0 = forward, 1 = dgrad)
    std::vector<BfPrepJob> bf_jobs; std::vector<int> bf_job_begin, bf_job_end;
    BfPrepJob* bf_jobs_dev; size_t bf_max_total;
    float* bf_part; unsigned int* bf_tickets;
    void add_planes(Bump& A, const TView& v, int fmt);      // fmt 1 = forward activation (fp16 of x/16), 0 = gradient (bf16)
    ActPlanes wg_xp; size_t wg_xp_halfs;              // bf16 scratch planes: forward activations re-split for the weight gradient
    float act_scale;                                  // power-of-two scale of the fp16 forward planes (per network, MS_ACT_SCALE overrides)
    const ActPlanes* planes_of(const TView& v) const;
    int ensure_planes(const TView& v, cudaStream_t st);
    // ---- data-parallel exchange over NVLink peer memory (csrc/dp.cu)
    int dp_rank, dp_world; bool dp_connected;
    float* dp_xbuf; DpState* dp_state; size_t dp_cap_floats;
    float* dp_peer_xbuf[DP_MAX_WORLD]; DpState* dp_peer_state[DP_MAX_WORLD];
    int dp_create(int rank, int world, unsigned char* handles_out /* 128 bytes */);
    int dp_connect(const unsigned char* all_handles /* world x 128 bytes */);
    int dp_update(int group, float lr, float mu, cudaStream_t st);
    int dp_error(unsigned int* out);
    float* wg_ws; size_t wg_ws_floats;
    float* rs_tmp; size_t rs_tmp_floats;
    float* loss_ws; size_t loss_ws_floats;
    unsigned char* u8_stage;         // 2 x B*H*W*3 bytes: uint8 input staging (set_input_u8)
    float* scalars;                  // [0]=full loss, [1]=train loss, [2]=epe, [3]=bad3
    float* gt;                       // optional ground truth [B,H,W,1]
    float* proxy;                    // proxy disparities [B,H,W,1] of the continual-adaptation variant (loss_kind 1)
    int loss_kind;                   // 0 = reprojection SSIM+L1 (Stereo_Online_Adaptation.py), 1 = masked L1 to proxy labels (Stereo_Continual_Adaptation.py)
    float proxy_w_full, proxy_w_module;   // loss weights of the reference: 0.01 (full-resolution loss / FULL train op), 0.1 (MAD module losses)

    // ---- profiling (off by default): CUDA events around kernel groups on the launching stream
    enum Cat { CAT_CONV_FWD = 0, CAT_CONV_DGRAD, CAT_CONV_WGRAD, CAT_CORR_FWD, CAT_CORR_BWD, CAT_LOSS, CAT_OTHER, N_CAT };
    struct Span { int cat, layer; cudaEvent_t a, b; double macs, bytes; };
    int profiling;                   // 0 off, 1 eager (events between launches), 2 in-graph (external event nodes inside the replayed graph)
    bool prof_capturing;
    float prof_event_overhead_ms;    // in-graph event-to-event latency with nothing in between (calibration)
    std::vector<Span> spans;
    std::vector<cudaEvent_t> event_pool;
    double cat_ms[N_CAT]; double cat_macs[N_CAT]; double cat_bytes[N_CAT]; long long cat_calls[N_CAT];
    void prof_begin(int cat, cudaStream_t st, int layer = -1);
    void prof_end(cudaStream_t st);
    void prof_note(double macs, double bytes);   // work of the span just closed
    int prof_fold(std::vector<Span>& v, bool recycle);
    std::vector<double> layer_ms[3]; std::vector<long long> layer_calls[3];   // per layer: fwd / dgrad / wgrad
    int prof_collect();      // synchronises; folds spans into cat_ms
    void prof_reset();

    // ---- DispNet buffers (engine_dispnet.cu)
    TView d_c1, d_c2, d_cat3, d_enc[8], d_cat[5], d_pr[5], d_cc[5], d_pred;
    TView gd_c1, gd_c2, gd_cat3, gd_enc[8], gd_cat[5], gd_pr[5], gd_cc[5], gd_pred;
    int build_dispnet();
    void layout_dispnet(Bump& A, size_t& max_wg, size_t& max_wt);
    int forward_dispnet(int disp_mask, cudaStream_t st);
    int backward_dispnet(cudaStream_t st);
    int deconv_bwd(const ConvLayer& L, const TView& x, const TView& dpre, const TView* dx, int dx_acc, cudaStream_t st);

    Engine();
    size_t layout(float* base);      // returns floats needed; assigns views when base != nullptr
    int build_madnet();
    int finalize_groups(const int* group_of_layer, int n_groups);

    int set_input(const float* left, const float* right, cudaStream_t st);
    int set_input_u8(const unsigned char* left, const unsigned char* right, cudaStream_t st);
    int forward(int disp_mask, cudaStream_t st);
    int loss(int which, int with_grad, int slot, float grad_scale, cudaStream_t st);
    int backward(int mode, int group, cudaStream_t st);     // mode 1 = MAD(group), 2 = FULL
    int update(int group, float lr, float mu, float gscale, cudaStream_t st);

    // helpers
    int conv_fwd(const ConvLayer& L, const TView& x, const TView& y, const float* res, int res_cs, cudaStream_t st);
    int conv_bwd(const ConvLayer& L, const TView& x, const TView& dpre, const TView* dx, const TView* dx_mask,
                 float mask_alpha, int dx_acc, int want_wgrad, cudaStream_t st);
    bool trainable(int layer, int mode, int group) const;
};

}  // namespace ms
