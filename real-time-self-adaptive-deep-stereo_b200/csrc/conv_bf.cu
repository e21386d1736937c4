// conv_bf: tcgen05 implicit-GEMM convolution on split 16-bit operands -- the tensor-core path of the conv stacks.
//
// Replaces the cuDNN calls behind tf.nn.conv2d / tf.nn.atrous_conv2d (reference Nets/sharedLayers.py:58,72) and their
// input gradients for the estimator / context / pyramid layers of MADNet (Nets/MadNet.py:73-171,173-249) and the
// DispNet encoder / refinement convs (Nets/DispNet.py:77-140).
//
// Why this tensor-core generation (round-2 findings, DESIGN.md section 4): round 1's 3xTF32 kernels (since removed) split
// fp32 activations inside the main loop (splitter warps, three-party mbarrier hand-shakes) and every 128-pixel CTA
// re-streams the whole weight set: 10x L2->SM amplification, tensor pipe < 50 %.  Here
//   * operands are PRE-SPLIT: every tensor that feeds a convolution also exists as two 16-bit planes (x ~= hi + lo),
//     written by the producing kernel's epilogue; weights are split once per update.  The main loop is the canonical
//     TMA -> tcgen05.mma -> epilogue pipeline, no splitter.
//       forward operands : fp16 planes of x/16 and of w  (hi = fp16, lo = fp16 of the remainder: 22 mantissa bits,
//                          ~2^-22 relative product error -- fp32-grade, so no extra relu / floor / |.| kink flips; the
//                          1/16 pre-scale keeps |x| <= 1e6 inside the fp16 range, undone exactly in the epilogue)
//       gradient operands: bf16 planes (hi + lo: 16 mantissa bits, ~2^-16, full fp32 exponent range for 1e-9 gradients)
//   * three kind::f16 MMAs per K step (w_lo*x_hi + w_hi*x_lo into one accumulator, w_hi*x_hi into another) at the
//     bf16/fp16 tensor rate (twice the tf32 rate).
//   * the GEMM is transposed ("swap AB"): M = output channels (128 TMEM lanes), N = up to 256 output pixels per CTA.
//     One weight tile serves 256 pixels, per-MMA shared-memory reads drop from 128 to 96 B/clk, and the epilogue
//     thread <-> channel mapping makes every NHWC store a coalesced 128-byte line.
//   * K blocks of 64 channels (128-byte rows, SWIZZLE_128B) whenever cin > 32: the first version used 32-channel
//     blocks = 64-byte TMA rows and was bound by the TMA request rate (15.7 k requests per CTA on the dominant layer,
//     ncu: tensor pipe 35 %, epilogue warps idle on the accumulator barrier for 80 % of the kernel).
//   * weights are stored PRE-TILED in their shared-memory image (per (M block, tap, K block): hi tile | lo tile,
//     swizzle applied by the prep kernel) and arrive as ONE 1-D bulk copy per tap instead of 2 x 128 TMA rows.
//   * A tile's pixels are `TW` wide and N/TW high.  For each filter column the kernel loads ONE halo patch
//     (N/TW + (kh-1)*dilation rows) per K block; the kh taps of that column are row offsets into the patch
//     (patch rows are whole swizzle atoms, so a tap is just a different UMMA descriptor start address).
//     Stride-2 convolutions use TMA element strides {1,2,2,1}: a patch then holds every second pixel / row.
//   * split-K over (K block, patch) units for small maps; the last-arriving CTA of a tile reduces the partial
//     sums in fixed order (deterministic) and runs the epilogue -- no separate reduce launch.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-9 = epilogue.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace ms {

constexpr int BF_THREADS = 320;
constexpr int BF_MAX_PATCH = 16;
constexpr int BF_MAX_TAPS = 49;

struct BfPatch { short dx, dy, ntaps, tap0; };
struct BfTap { short row_off, widx; };

struct ConvBfParams {
    int H, W, NB;                 // output lattice handled by this launch (tile validity)
    int Hout, Wout, os, oy0, ox0; // output tensor; lattice point (j) is output pixel j * os + o0
    int TW, tw_shift, N;          // pixel tile: TW wide (power of two), N pixels
    int tiles_x, tiles_y;
    int sx;                       // input coordinate = out * sx + patch.d
    int kblocks, n_patches;
    int kch;                      // channels per K block: 32 (64-byte rows, SWIZZLE_64B) or 64 (128-byte rows, SWIZZLE_128B)
    int taps_total;
    uint32_t slot_bytes;          // bytes of one patch plane in shared memory
    uint32_t wtile_bytes;         // bytes of one weight tile plane (128 rows x kch x 2)
    int NP, NW;
    int nacc;                     // accumulators: 2 = cross terms and hi*hi separately, 1 = everything in one
    int nprod;                    // 3 = split x3, 1 = hi*hi only (accuracy experiments)
    int fmt;                      // operand format: 0 = bf16 planes, 1 = fp16 planes (activation planes hold x * scale)
    float acc_scale;              // multiplies the accumulator (1 / scale of the input planes, a power of two: exact)
    int tmem_cols;
    int cout;
    int ksplit;
    unsigned long long* prof;     // MS_BF_PROF=1: per-CTA clock64 stamps [8] (entry, setup done, first data, MMAs issued, accumulator seen, epilogue done, exit, MMA-thread wait cycles)
    int debug;                    // MS_BF_DEBUG kill switches (measurement only): 1 = no MMAs, 2 = no weight loads, 4 = no patch loads, 8 = no epilogue stores
    const unsigned char* wtiles;  // pre-tiled weights [M block][tap][K block][hi tile | lo tile]
    float* part; unsigned int* tickets;
    float* y; int ycs;
    const float* bias; float alpha;
    const float* res; int res_cs;
    const float* mask; int mask_cs; float mask_alpha;
    int accumulate;
    void* ohi; void* olo; int ocs; int ofmt; float oscale;   // optional output planes (format, stored value = t * oscale)
    BfPatch patch[BF_MAX_PATCH];
    BfTap tap[BF_MAX_TAPS];
};

__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// K-major shared-memory matrix descriptors (cute::UMMA::SmemDescriptor), version 1:
//   SWIZZLE_64B : rows of 64 bytes, 8-row atoms of 512 bytes (SBO), layout_type 4
//   SWIZZLE_128B: rows of 128 bytes, 8-row atoms of 1024 bytes (SBO), layout_type 2
__device__ __forceinline__ uint64_t umma_desc_k(uint32_t smem_byte_addr, bool sw128) {
    const uint64_t lo = (uint64_t)((smem_byte_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (1ull << 46);
    return sw128 ? (lo | (64ull << 32) | (2ull << 61)) : (lo | (32ull << 32) | (4ull << 61));
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(s_addr(dst)), "l"(src), "r"(bytes), "r"(s_addr(bar)) : "memory");
}

// 16-bit split of a float: fmt 0 -> bf16 hi/lo of v (any magnitude), fmt 1 -> fp16 hi/lo of v * scale (22 mantissa bits while
// |v * scale| stays inside fp16's normal range; saturating, so an out-of-range value degrades instead of becoming inf)
__device__ __forceinline__ void split16(float v, int fmt, float scale, unsigned short& hi, unsigned short& lo) {
    if (fmt == 0) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
        hi = __bfloat16_as_ushort(h); lo = __bfloat16_as_ushort(l);
    } else {
        const float s = v * scale;
        asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(hi) : "f"(s));
        const float r = s - __half2float(__ushort_as_half(hi));
        asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(lo) : "f"(r));
    }
}

__global__ void __launch_bounds__(BF_THREADS, 1)
conv_bf_kernel(const __grid_constant__ CUtensorMap mapXh, const __grid_constant__ CUtensorMap mapXl,
               const __grid_constant__ ConvBfParams p) {
    extern __shared__ unsigned char smem_dyn[];
    __shared__ __align__(8) uint64_t pfull[4], pempty[4], wfull[8], wempty[8], accum_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ int last_flag;

    const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
    const uint32_t base = (s_addr(smem_dyn) + 1023u) & ~1023u;
    unsigned char* gbase = smem_dyn + (base - s_addr(smem_dyn));
    const uint32_t pslot = 2u * p.slot_bytes;                 // hi plane | lo plane
    const uint32_t w_off = (uint32_t)p.NP * pslot;
    const uint32_t wslot = 2u * p.wtile_bytes;                // hi tile | lo tile

    int bid = blockIdx.x;
    const int tx = bid % p.tiles_x; bid /= p.tiles_x;
    const int ty = bid % p.tiles_y;
    const int img = bid / p.tiles_y;
    const int TH = p.N >> p.tw_shift;
    const int x0 = tx * p.TW, y0 = ty * TH;
    const int units = p.kblocks * p.n_patches;
    const int u0 = (int)(((long)blockIdx.z * units) / p.ksplit), u1 = (int)(((long)(blockIdx.z + 1) * units) / p.ksplit);
    unsigned long long* prof = p.prof ? p.prof + ((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 : nullptr;
    if (prof && threadIdx.x == 0) prof[0] = clock64();
    // programmatic dependent launch (common.cuh): the next kernel's CTAs may become resident as soon as every CTA of this
    // grid has started; this kernel's own global traffic starts only after pdl_wait() below
    pdl_trigger();

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.NP; ++i) { mb_init(&pfull[i], 1); mb_init(&pempty[i], 1); }
        for (int i = 0; i < p.NW; ++i) { mb_init(&wfull[i], 1); mb_init(&wempty[i], 1); }
        mb_init(&accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_addr(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();                                               // everything above (barriers, TMEM) overlapped the previous kernel's tail
    if (prof && threadIdx.x == 0) prof[1] = clock64();

    if (warp == 0) {
        // ================= producer: halo patches by TMA (per K block x filter column) + weight tiles by bulk copy (per tap) ===
        const bool leader = elect_one();               // warp-uniform loop, elected lane issues (tc_ptx.cuh:elect_one)
        {
            int ps = 0, ws = 0;
            uint32_t pph = 0, wph = 0;
            const unsigned char* wbase = p.wtiles + (size_t)blockIdx.y * p.taps_total * p.kblocks * wslot;
            int kb = u0 / p.n_patches, pi = u0 - kb * p.n_patches;
            for (int u = u0; u < u1; ++u) {
                const BfPatch pt = p.patch[pi];
                mb_wait(&pempty[ps], pph ^ 1u);
                unsigned char* dst = gbase + (size_t)ps * pslot;
                if (p.debug & 4) { if (leader) mb_arrive(&pfull[ps]); }
                else if (leader) {
                    mb_expect_tx(&pfull[ps], pslot);
                    tma_load_4d(dst, &mapXh, &pfull[ps], kb * p.kch, x0 * p.sx + pt.dx, y0 * p.sx + pt.dy, img);
                    tma_load_4d(dst + p.slot_bytes, &mapXl, &pfull[ps], kb * p.kch, x0 * p.sx + pt.dx, y0 * p.sx + pt.dy, img);
                }
                if (++ps == p.NP) { ps = 0; pph ^= 1u; }
                for (int t = pt.tap0; t < pt.tap0 + pt.ntaps; ++t) {
                    mb_wait(&wempty[ws], wph ^ 1u);
                    if (p.debug & 2) { if (leader) mb_arrive(&wfull[ws]); }
                    else if (leader) {
                        mb_expect_tx(&wfull[ws], wslot);
                        bulk_load(gbase + w_off + (size_t)ws * wslot, wbase + ((size_t)p.tap[t].widx * p.kblocks + kb) * wslot, wslot, &wfull[ws]);
                    }
                    if (++ws == p.NW) { ws = 0; wph ^= 1u; }
                }
                if (++pi == p.n_patches) { pi = 0; ++kb; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: the whole warp runs the loop (uniform registers), one elected lane issues =================
        const bool leader = elect_one();
        const uint32_t tmem = __shfl_sync(0xffffffffu, tmem_slot, 0);       // (a shuffle from lane 0 is warp-uniform to the compiler)
        {
            // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (bit 4), A/B format at bits 7 / 10 (0 = f16,
            // 1 = bf16), both K-major, N>>3 at bit 17, M>>4 at bit 24
            const uint32_t f = p.fmt == 0 ? 1u : 0u;
            const uint32_t idesc = (1u << 4) | (f << 7) | (f << 10) | ((uint32_t)(p.N >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t acc_main = tmem + (p.nacc == 2 ? (uint32_t)p.N : 0u);
            const bool sw128 = p.kch == 64;
            const int k16 = p.kch >> 4;
            int ps = 0, ws = 0;
            uint32_t pph = 0, wph = 0;
            uint32_t started_cross = 0, started_main = 0;
            int pi = u0 % p.n_patches;
            const uint32_t row_bytes = (uint32_t)p.TW * (uint32_t)p.kch * 2u;
            long long waited = 0;
            for (int u = u0; u < u1; ++u) {
                const BfPatch pt = p.patch[pi];
                long long tw0 = prof ? clock64() : 0;
                mb_wait(&pfull[ps], pph);
                if (prof) { const long long tw1 = clock64(); waited += tw1 - tw0; if (u == u0 && leader) prof[2] = tw1; }
                const uint32_t pb = base + (uint32_t)ps * pslot;
                for (int t = pt.tap0; t < pt.tap0 + pt.ntaps; ++t) {
                    tw0 = prof ? clock64() : 0;
                    mb_wait(&wfull[ws], wph);
                    if (prof) waited += clock64() - tw0;
                    tc_fence_after();
                    const uint32_t boff = (uint32_t)p.tap[t].row_off * row_bytes;
                    const uint64_t xh = umma_desc_k(pb + boff, sw128), xl = umma_desc_k(pb + p.slot_bytes + boff, sw128);
                    const uint32_t wb = base + w_off + (uint32_t)ws * wslot;
                    const uint64_t wh = umma_desc_k(wb, sw128), wl = umma_desc_k(wb + p.wtile_bytes, sw128);
                    for (int j = 0; j < ((p.debug & 1) ? 0 : k16); ++j) {   // K = 16 elements = 32 bytes inside the swizzle row
                        const uint64_t o = (uint64_t)(j * 2);
                        if (p.nprod == 3) {
                            if (leader) {
                                tc_mma_f16(tmem, wl + o, xh + o, idesc, started_cross);
                                tc_mma_f16(tmem, wh + o, xl + o, idesc, 1u);
                            }
                            started_cross = 1u;
                            if (p.nacc == 1) started_main = 1u;
                        }
                        if (leader) tc_mma_f16(acc_main, wh + o, xh + o, idesc, started_main);
                        started_main = 1u;
                        if (p.nacc == 1) started_cross = 1u;
                    }
                    if (leader) tc_commit(&wempty[ws]);
                    if (++ws == p.NW) { ws = 0; wph ^= 1u; }
                }
                if (leader) tc_commit(&pempty[ps]);
                if (++ps == p.NP) { ps = 0; pph ^= 1u; }
                if (++pi == p.n_patches) pi = 0;
            }
            if (prof && leader) { prof[3] = clock64(); prof[7] = (unsigned long long)waited; }
            if (leader) tc_commit(&accum_bar);
            __syncwarp();
        }
    } else {
        // ================= epilogue (warps 2..9): thread <-> output channel, columns <-> pixels =================
        const int q = warp & 3;                         // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;               // which half of the pixel columns
        const int ch = blockIdx.y * 128 + q * 32 + lane;
        const bool chv = ch < p.cout;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const float bias = (chv && p.bias) ? __ldg(p.bias + ch) : 0.f;
        const int cbeg = half * (p.N >> 1), cend = cbeg + (p.N >> 1);
        const bool two = (p.nacc == 2) && (p.nprod == 3);
        const int tile_lin = blockIdx.x * gridDim.y + blockIdx.y;
        const float acc_scale = p.acc_scale, alpha = p.alpha;
        const bool has_res = p.res != nullptr, has_mask = p.mask != nullptr, has_acc = p.accumulate != 0, has_pl = p.ohi != nullptr;
        const int twm = p.TW - 1;
        const size_t img_pix = (size_t)img * p.Hout;
        unsigned short* const ohi = reinterpret_cast<unsigned short*>(p.ohi);
        unsigned short* const olo = reinterpret_cast<unsigned short*>(p.olo);

        // 16 consecutive columns = (TW == 8) two tile rows of 8 pixels, or (TW == 16) one row of 16: hoist the row part
        // scalar fallback (channel counts / strides that are not multiples of 4): thread <-> channel, one pixel at a time
        auto finish16_scalar = [&](int c0, const float (&v)[16]) {
            const int r0 = c0 >> p.tw_shift, px0 = c0 & twm;
#pragma unroll
            for (int hrow = 0; hrow < 2; ++hrow) {
                const int yy = y0 + r0 + (p.TW == 8 ? hrow : 0);
                const int jb = p.TW == 8 ? hrow * 8 : hrow * 8;
                if (yy >= p.H || !chv) continue;
                const size_t rowpix = (img_pix + (size_t)(yy * p.os + p.oy0)) * p.Wout + p.ox0;
                float* yrow = p.y + rowpix * p.ycs + ch;
                const float* rrow = has_res ? p.res + rowpix * p.res_cs + ch : nullptr;
                const float* mrow = has_mask ? p.mask + rowpix * p.mask_cs + ch : nullptr;
                unsigned short* hrow_p = has_pl ? ohi + rowpix * p.ocs + ch : nullptr;
                unsigned short* lrow_p = has_pl ? olo + rowpix * p.ocs + ch : nullptr;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int xx = x0 + (p.TW == 8 ? j : px0 + jb + j);
                    if (xx >= p.W) continue;
                    const int xo = xx * p.os;
                    float t = v[jb + j] * acc_scale + bias;
                    t = fmaxf(alpha * t, t);
                    if (has_res) t += rrow[(size_t)xo * p.res_cs];
                    if (has_acc) t += yrow[(size_t)xo * p.ycs];
                    if (has_mask) t *= (mrow[(size_t)xo * p.mask_cs] > 0.f) ? 1.f : p.mask_alpha;
                    if (p.debug & 8) continue;
                    yrow[(size_t)xo * p.ycs] = t;
                    if (has_pl) {
                        unsigned short h, l;
                        split16(t, p.ofmt, p.oscale, h, l);
                        hrow_p[(size_t)xo * p.ocs] = h;
                        lrow_p[(size_t)xo * p.ocs] = l;
                    }
                }
            }
        };


        // vector path: the warp's 16 px x 32 ch block is transposed through shared memory (the pipeline buffers are idle once
        // the accumulator barrier fired) so that a lane owns 4 consecutive channels of one pixel: 128-bit loads / stores for
        // y, residual, mask and accumulate, 64-bit stores for the two 16-bit planes, one address computation per 4 values.
        // (first version: thread <-> channel scalar stores, 67 warp instructions per pixel column -- the epilogue took 36.7 k
        // cycles per tile against 30 k for the whole main loop, MS_BF_PROF)
        const bool vec_ok = (p.cout & 3) == 0 && (p.ycs & 3) == 0 && (reinterpret_cast<uintptr_t>(p.y) & 15) == 0 &&
                            (!has_res || ((p.res_cs & 3) == 0 && (reinterpret_cast<uintptr_t>(p.res) & 15) == 0)) &&
                            (!has_mask || ((p.mask_cs & 3) == 0 && (reinterpret_cast<uintptr_t>(p.mask) & 15) == 0)) &&
                            (!has_pl || ((p.ocs & 3) == 0 && ((reinterpret_cast<uintptr_t>(p.ohi) | reinterpret_cast<uintptr_t>(p.olo)) & 7) == 0));
        float* const stage = reinterpret_cast<float*>(gbase) + (size_t)(warp - 2) * 512;      // 16 px x 32 ch per warp
        const int c4 = lane & 7, prow = lane >> 3;
        const int ch4 = blockIdx.y * 128 + q * 32 + c4 * 4;
        const bool ch4v = ch4 < p.cout;
        float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (vec_ok && ch4v && p.bias) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + ch4));
        const float mask_alpha = p.mask_alpha, oscale = p.oscale;
        const int ofmt = p.ofmt;
        auto finish16 = [&](int c0, const float (&v)[16]) {
            if (!vec_ok) { finish16_scalar(c0, v); return; }
            // pixel addresses of this lane's 4 pixels, and the operands that do not depend on the accumulator (residual,
            // previous value, mask) requested BEFORE the transpose so that their latency overlaps it
            size_t pix[4];
            bool ok[4];
            float4 rv[4], ov[4], mv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int col = c0 + i * 4 + prow;
                const int yy = y0 + (col >> p.tw_shift), xx = x0 + (col & twm);
                ok[i] = yy < p.H && xx < p.W && ch4v;
                pix[i] = (img_pix + (size_t)(yy * p.os + p.oy0)) * p.Wout + (size_t)(xx * p.os + p.ox0);
                if (ok[i]) {
                    if (has_res) rv[i] = *reinterpret_cast<const float4*>(p.res + pix[i] * p.res_cs + ch4);
                    if (has_acc) ov[i] = *reinterpret_cast<const float4*>(p.y + pix[i] * p.ycs + ch4);
                    if (has_mask) mv[i] = *reinterpret_cast<const float4*>(p.mask + pix[i] * p.mask_cs + ch4);
                }
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 16; ++j) stage[j * 32 + lane] = v[j];
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float4 t = *reinterpret_cast<const float4*>(stage + (i * 4 + prow) * 32 + c4 * 4);
                if (!ok[i]) continue;
                t.x = t.x * acc_scale + bias4.x; t.y = t.y * acc_scale + bias4.y; t.z = t.z * acc_scale + bias4.z; t.w = t.w * acc_scale + bias4.w;
                t.x = fmaxf(alpha * t.x, t.x); t.y = fmaxf(alpha * t.y, t.y); t.z = fmaxf(alpha * t.z, t.z); t.w = fmaxf(alpha * t.w, t.w);
                if (has_res) { t.x += rv[i].x; t.y += rv[i].y; t.z += rv[i].z; t.w += rv[i].w; }
                if (has_acc) { t.x += ov[i].x; t.y += ov[i].y; t.z += ov[i].z; t.w += ov[i].w; }
                if (has_mask) {
                    t.x *= mv[i].x > 0.f ? 1.f : mask_alpha; t.y *= mv[i].y > 0.f ? 1.f : mask_alpha;
                    t.z *= mv[i].z > 0.f ? 1.f : mask_alpha; t.w *= mv[i].w > 0.f ? 1.f : mask_alpha;
                }
                if (p.debug & 8) continue;
                *reinterpret_cast<float4*>(p.y + pix[i] * p.ycs + ch4) = t;
                if (has_pl) {
                    unsigned short h[4], l[4];
                    split16(t.x, ofmt, oscale, h[0], l[0]); split16(t.y, ofmt, oscale, h[1], l[1]);
                    split16(t.z, ofmt, oscale, h[2], l[2]); split16(t.w, ofmt, oscale, h[3], l[3]);
                    uint2 hv, lv;
                    hv.x = (uint32_t)h[0] | ((uint32_t)h[1] << 16); hv.y = (uint32_t)h[2] | ((uint32_t)h[3] << 16);
                    lv.x = (uint32_t)l[0] | ((uint32_t)l[1] << 16); lv.y = (uint32_t)l[2] | ((uint32_t)l[3] << 16);
                    *reinterpret_cast<uint2*>(ohi + pix[i] * p.ocs + ch4) = hv;
                    *reinterpret_cast<uint2*>(olo + pix[i] * p.ocs + ch4) = lv;
                }
            }
        };

        mb_wait(&accum_bar, 0);
        tc_fence_after();
        if (prof && threadIdx.x == 64) prof[4] = clock64();
        if (p.ksplit == 1) {
            for (int c0 = cbeg; c0 < cend; c0 += 16) {
                uint32_t r0[16], r1[16];
                float v[16];
                tc_ld16_nowait(tmem + lane_base + (uint32_t)c0, r0);
                if (two) tc_ld16_nowait(tmem + lane_base + (uint32_t)(p.N + c0), r1);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = two ? __uint_as_float(r0[j]) + __uint_as_float(r1[j]) : __uint_as_float(r0[j]);
                finish16(c0, v);
            }
        } else {
            // raw partial sums: part[(z * n_tiles + tile) * N + col][128 channels]
            const size_t n_tiles = (size_t)gridDim.x * gridDim.y;
            float* mine = p.part + (((size_t)blockIdx.z * n_tiles + tile_lin) * p.N) * 128 + q * 32 + lane;
            for (int c0 = cbeg; c0 < cend; c0 += 16) {
                uint32_t r0[16], r1[16];
                tc_ld16_nowait(tmem + lane_base + (uint32_t)c0, r0);
                if (two) tc_ld16_nowait(tmem + lane_base + (uint32_t)(p.N + c0), r1);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float t = __uint_as_float(r0[j]);
                    if (two) t += __uint_as_float(r1[j]);
                    mine[(size_t)(c0 + j) * 128] = t;
                }
            }
            __threadfence();
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (threadIdx.x == 64) {
                const unsigned int old = atomicAdd(p.tickets + tile_lin, 1u);
                const int last = (old == (unsigned int)(p.ksplit - 1)) ? 1 : 0;
                if (last) p.tickets[tile_lin] = 0u;        // self-resetting for the next launch
                last_flag = last;
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (last_flag) {
                __threadfence();
                const float* col0 = p.part + ((size_t)tile_lin * p.N) * 128 + q * 32 + lane;
                const size_t zstride = n_tiles * (size_t)p.N * 128;
                for (int c0 = cbeg; c0 < cend; c0 += 16) {
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = 0.f;
                    int z = 0;
                    for (; z + 2 <= p.ksplit; z += 2) {          // two partial sets in flight (32 independent loads per thread)
                        const float* s0 = col0 + (size_t)z * zstride + (size_t)c0 * 128;
                        const float* s1 = s0 + zstride;
                        float a[16], b[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) { a[j] = __ldcg(s0 + (size_t)j * 128); b[j] = __ldcg(s1 + (size_t)j * 128); }
#pragma unroll
                        for (int j = 0; j < 16; ++j) { v[j] += a[j]; v[j] += b[j]; }     // fixed order z, z+1: deterministic
                    }
                    for (; z < p.ksplit; ++z) {
                        const float* src = col0 + (size_t)z * zstride + (size_t)c0 * 128;
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] += __ldcg(src + (size_t)j * 128);
                    }
                    finish16(c0, v);
                }
            }
        }
    }
    if (prof && threadIdx.x == 64) prof[5] = clock64();
    tc_fence_before();
    __syncthreads();
    if (prof && threadIdx.x == 0) prof[6] = clock64();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

static unsigned long long* g_bf_prof = nullptr;
static int g_bf_prof_ctas = 0;
constexpr int BF_PROF_MAX = 8192;
// last profiled launch: per-CTA stamps (MS_BF_PROF=1); returns the number of CTAs copied
int conv_bf_read_prof(unsigned long long* out, int max_ctas) {
    if (!g_bf_prof || g_bf_prof_ctas <= 0) return 0;
    const int n = std::min(max_ctas, g_bf_prof_ctas);
    if (cudaMemcpy(out, g_bf_prof, (size_t)n * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return n;
}

// ------------------------------------------------------------------------------------------------
// 16-bit planes of an fp32 NHWC view (producers that are not conv_bf epilogues: correlation, resize, loss seeds ...)
// ------------------------------------------------------------------------------------------------
__global__ void split_planes_kernel(const float* __restrict__ x, int xcs, int C, size_t pixels,
                                    unsigned short* __restrict__ hi, unsigned short* __restrict__ lo, int pcs, int fmt, float scale) {
    pdl_prologue();
    const int cq = (C + 3) >> 2;
    const size_t total = pixels * cq;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t pix = i / cq;
        const int c = (int)(i - pix * cq) * 4;
        const float* src = x + pix * xcs + c;
        unsigned short h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float v = (c + j < C) ? src[j] : 0.f;
            split16(v, fmt, scale, h[j], l[j]);
        }
        unsigned short* dh = hi + pix * pcs + c;
        unsigned short* dl = lo + pix * pcs + c;
        if (c + 4 <= pcs) {
            *reinterpret_cast<uint2*>(dh) = *reinterpret_cast<const uint2*>(h);
            *reinterpret_cast<uint2*>(dl) = *reinterpret_cast<const uint2*>(l);
        } else {
            for (int j = 0; j < 4 && c + j < pcs; ++j) { dh[j] = h[j]; dl[j] = l[j]; }
        }
    }
}

int split_planes(const TView& x, const ActPlanes& pl, cudaStream_t st) {
    MS_REQUIRE(pl.hi && pl.lo && pl.cs >= x.c && (pl.cs & 7) == 0, "split_planes: bad plane buffers");
    const size_t total = x.pixels() * ((x.c + 3) / 4);
    const unsigned grid = (unsigned)std::min<size_t>(cdivz(total, 256), 148 * 16);
    launch_k(split_planes_kernel, dim3(grid), dim3(256), 0, st, x.p, x.cs, x.c, x.pixels(), reinterpret_cast<unsigned short*>(pl.hi),
                                              reinterpret_cast<unsigned short*>(pl.lo), pl.cs, pl.fmt, pl.fmt == 1 ? pl.scale : 1.f);
    return check_launch("split_planes");
}

// ------------------------------------------------------------------------------------------------
// weight preparation: the shared-memory image of every (M block, tap, K block) tile, hi tile | lo tile, swizzled,
// from canonical fp32 HWIO, batched over layers
//   transposed_src = 1 : src is [tap][K][M]  (forward conv: K = cin, M = cout)
//   transposed_src = 0 : src is [tap][M][K]  (dgrad: M = cin, K = cout)
// ------------------------------------------------------------------------------------------------
__global__ void bf_prep_weights_kernel(const BfPrepJob* __restrict__ jobs) {
    pdl_prologue();
    const BfPrepJob j = jobs[blockIdx.y];
    const int kch = j.Kpad > 32 ? 64 : 32;
    const int kblocks = j.Kpad / kch, mblocks = j.Mpad / 128;
    const size_t tile = (size_t)128 * kch;                         // elements per tile plane
    const size_t total = (size_t)mblocks * j.taps * kblocks * tile;
    unsigned short* dst = reinterpret_cast<unsigned short*>(j.tiles);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int kk = (int)(i % kch);
        size_t q = i / kch;
        const int r = (int)(q % 128); q /= 128;
        const int kb = (int)(q % kblocks); q /= kblocks;
        const int t = (int)(q % j.taps);
        const int mb = (int)(q / j.taps);
        const int m = mb * 128 + r, k = kb * kch + kk;
        float v = 0.f;
        if (m < j.M && k < j.K)
            v = j.transposed_src ? j.src[((size_t)t * j.K + k) * j.M + m] : j.src[((size_t)t * j.M + m) * j.K + k];
        unsigned short h, l;
        if (j.fmt == 0) {
            const __nv_bfloat16 hb = __float2bfloat16_rn(v);
            h = __bfloat16_as_ushort(hb); l = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(hb)));
        } else {                                                  // weights are not pre-scaled
            const __half hh = __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f));
            h = __half_as_ushort(hh); l = __half_as_ushort(__float2half_rn(v - __half2float(hh)));
        }
        // swizzled position inside the tile image (K-major rows of kch*2 bytes, 16-byte chunks XOR-ed with the row bits)
        const int chunk = kk >> 3, e = kk & 7;
        const int sw = kch == 64 ? (chunk ^ (r & 7)) : (chunk ^ ((r >> 1) & 3));
        const size_t off = (size_t)r * kch + (size_t)sw * 8 + e;
        const size_t tbase = ((((size_t)mb * j.taps + t) * kblocks + kb) * 2) * tile;
        dst[tbase + off] = h;
        dst[tbase + tile + off] = l;
    }
}

int bf_prep_weights(const BfPrepJob* jobs_dev, int njobs, size_t max_total, cudaStream_t st) {
    if (njobs <= 0) return 0;
    const unsigned gx = (unsigned)std::min<size_t>(cdivz(max_total / 2, 256), 512);
    launch_k(bf_prep_weights_kernel, dim3(dim3(gx, njobs)), dim3(256), 0, st, jobs_dev);
    return check_launch("bf_prep_weights");
}

void conv_bf_weight_dims(int M, int K, int& Mpad, int& Kpad) {
    Mpad = (M + 127) / 128 * 128;
    Kpad = K > 32 ? (K + 63) / 64 * 64 : 32;
}
size_t conv_bf_weight_halfs(int taps, int M, int K) {       // 16-bit elements of the tiled image, both planes
    int Mpad, Kpad; conv_bf_weight_dims(M, K, Mpad, Kpad);
    return (size_t)2 * taps * Mpad * Kpad;
}

// ------------------------------------------------------------------------------------------------
// tensor maps (16-bit elements, SWIZZLE_64B / 128B, zero OOB fill, optional element strides), cached
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn bf_get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* q = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(q);
    }
    return fn;
}
struct BfMapKey {
    uintptr_t addr; int rank; int swz; uint64_t d[4]; uint64_t s[3]; uint32_t b[4]; uint32_t es[4];
    bool operator<(const BfMapKey& o) const { return memcmp(this, &o, sizeof(BfMapKey)) < 0; }
};
// (BFLOAT16 as the element type for fp16 planes too: TMA moves 2-byte elements, the zero fill is format-agnostic)
int bf_get_map(const CUtensorMap** out, void* addr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, const cuuint32_t* estr, int swizzle_bytes) {
    static std::map<BfMapKey, CUtensorMap> cache;
    BfMapKey k;
    memset(&k, 0, sizeof k);
    k.addr = reinterpret_cast<uintptr_t>(addr); k.rank = rank; k.swz = swizzle_bytes;
    for (int i = 0; i < rank; ++i) { k.d[i] = dims[i]; k.b[i] = box[i]; k.es[i] = estr[i]; }
    for (int i = 0; i + 1 < rank; ++i) k.s[i] = strides_bytes[i];
    auto it = cache.find(k);
    if (it == cache.end()) {
        EncodeTiledFn enc = bf_get_encode();
        MS_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
        CUtensorMap m;
        CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, addr, dims, strides_bytes, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (16-bit planes) failed with code " + std::to_string((int)r)); return -1; }
        if (cache.size() >= 8192) {
            static thread_local CUtensorMap spill[16];
            static thread_local unsigned spill_i = 0;
            CUtensorMap* slot = &spill[spill_i++ & 15u];
            *slot = m;
            *out = slot;
            return 0;
        }
        it = cache.emplace(k, m).first;
    }
    *out = &it->second;
    return 0;
}

// ------------------------------------------------------------------------------------------------
bool conv_bf_supported(const ConvGemm& g) {
    if (g.div != 1 && !(g.div == 2 && g.mul == 1)) return false;       // forward (stride 1/2), dgrad / transposed (stride 1/2)
    if (g.mul != 1 && g.mul != 2) return false;
    if (g.mul == 2 && g.step != 1) return false;
    if (g.div == 2 && std::abs(g.step) != 1) return false;
    if (g.x.c < 3 || g.y.c < 8) return false;          // (3-channel images: the planes are padded to 8 channels, TMA zero-fills the K block)
    if (g.kh * g.kw > BF_MAX_TAPS) return false;
    if (g.y.h * g.y.w < 32) return false;
    return true;
}

int conv_bf_init() {
    static bool done = false;
    if (done) return 0;
    MS_CHECK_CUDA(cudaFuncSetAttribute(conv_bf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    done = true;
    return 0;
}

size_t conv_bf_part_floats() { return (size_t)8 << 20; }    // 32 MB of split-K partial sums
size_t conv_bf_ticket_words() { return 4096; }

struct BfTapSpec { int dy, dx, widx; };     // input pixel = out_lattice * sx + (dy, dx); weight tap index

// One launch: output lattice [Hj x Wj] (output pixel = j * os + o0), gather taps `taps`, input lattice stride sx.
static int conv_bf_launch(const ConvGemm& g, const ActPlanes& xp, const void* wtiles, const ActPlanes* yp,
                          float* part, unsigned int* tickets, int Hj, int Wj, int os, int oy0, int ox0, int sx,
                          const BfTapSpec* taps, int ntaps, int taps_total, cudaStream_t st) {
    const int K = g.x.c, M = g.y.c;
    int Mpad, Kpad; conv_bf_weight_dims(M, K, Mpad, Kpad);
    static ConvBfParams p;          // large (tables): filled in place, passed by value to the launch
    memset(&p, 0, sizeof p);
    p.H = Hj; p.W = Wj; p.NB = g.y.n; p.sx = sx;
    p.Hout = g.y.h; p.Wout = g.y.w; p.os = os; p.oy0 = oy0; p.ox0 = ox0;
    p.kch = Kpad > 32 ? 64 : 32;
    p.kblocks = Kpad / p.kch; p.cout = M; p.taps_total = taps_total;
    p.wtile_bytes = 128u * (uint32_t)p.kch * 2u;
    p.fmt = xp.fmt; p.acc_scale = xp.fmt == 1 ? 1.f / xp.scale : 1.f;
    MS_REQUIRE(xp.fmt == 0 || xp.scale > 0.f, "conv_bf: fp16 planes need a positive scale");
    const uint32_t row_unit = (uint32_t)p.kch * 2u;                 // bytes of one pixel of a patch plane
    // ---- patches: taps of one filter column (same dx; same row parity for an input lattice of stride 2) share a halo
    //      patch; a tap is a row offset into it
    auto posmod = [](int a, int m) { return ((a % m) + m) % m; };
    bool used[BF_MAX_TAPS] = {false};
    int np = 0, nt = 0, max_off = 0;
    for (int i = 0; i < ntaps; ++i) {
        if (used[i]) continue;
        int first_dy = taps[i].dy;
        for (int j = i; j < ntaps; ++j)
            if (!used[j] && taps[j].dx == taps[i].dx && posmod(taps[j].dy - taps[i].dy, sx) == 0) first_dy = std::min(first_dy, taps[j].dy);
        MS_REQUIRE(np < BF_MAX_PATCH, "conv_bf: too many patches");
        BfPatch& pt = p.patch[np];
        pt.dx = (short)taps[i].dx; pt.dy = (short)first_dy; pt.tap0 = (short)nt; pt.ntaps = 0;
        for (int j = i; j < ntaps; ++j) {
            if (used[j] || taps[j].dx != taps[i].dx || posmod(taps[j].dy - taps[i].dy, sx) != 0) continue;
            used[j] = true;
            const int off = (taps[j].dy - first_dy) / sx;
            p.tap[nt].row_off = (short)off; p.tap[nt].widx = (short)taps[j].widx;
            max_off = std::max(max_off, off);
            ++nt; ++pt.ntaps;
        }
        ++np;
    }
    // ---- pixel tile TW x TH (N = TW * TH MMA columns, a multiple of 32, 64 <= N <= 256).  One CTA per tile and no
    //      second wave to hide a ragged tail, so the tile shape decides how many of the 148 SMs work: a 96 x 320 map in
    //      8 x 32 tiles is 120 CTAs of 256 pixels (81 % of the SMs); in 16 x 14 tiles it is 140 CTAs of 224.
    //      cost = waves x (N + fixed overhead in pixel units); ties go to the taller tile (smaller halo).
    const int mblocks = Mpad / 128;
    static int force_n = -1, tile_search = -1;
    if (force_n < 0) { const char* e = getenv("MS_BF_N"); force_n = e ? atoi(e) : 0; }
    if (tile_search < 0) { const char* e = getenv("MS_BF_TILE_SEARCH"); tile_search = (e && e[0] == '0') ? 0 : 1; }
    int N = 64, TW = 8;
    if (force_n || !tile_search) {
        const int cand_n[3] = {256, 128, 64};
        for (int ci = 0; ci < 3; ++ci) {
            const int n = cand_n[ci];
            int tw = 8;
            if (n == 256 && (Hj % 32) != 0 && (Hj % 16) == 0) tw = 16;
            const int th = n / tw;
            const long tiles = (long)g.y.n * cdiv(Wj, tw) * cdiv(Hj, th) * mblocks;
            const bool take = force_n ? (n == force_n || ci == 2) : (tiles >= 100 || ci == 2);
            if (take) { N = n; TW = tw; break; }
        }
    } else {
        long best = -1; int best_th = 0;
        const int tws[3] = {8, 16, 32};
        for (int wi = 0; wi < 3; ++wi) {
            const int tw = tws[wi];
            if (tw * sx > 256) continue;
            for (int th = 1; th * tw <= 256; ++th) {
                const int n = th * tw;
                if (n < 64 || (n & 31)) continue;
                if ((th + max_off) * sx > 256) continue;
                const long tiles = (long)g.y.n * cdiv(Wj, tw) * cdiv(Hj, th) * mblocks;
                // (halo rows are loaded, not multiplied: a quarter weight keeps 32 x 2 tiles for the cases that save a wave)
                const long cost = cdiv((int)std::min<long>(tiles, 1 << 30), 148) * (long)(n + 32 + max_off * tw / 4);
                if (best < 0 || cost < best || (cost == best && th > best_th)) { best = cost; best_th = th; N = n; TW = tw; }
            }
        }
    }
    const int TH = N / TW;
    p.TW = TW; p.tw_shift = TW == 8 ? 3 : (TW == 16 ? 4 : 5); p.N = N;
    p.tiles_x = cdiv(Wj, TW); p.tiles_y = cdiv(Hj, TH);
    p.n_patches = np;
    int rows = TH + max_off;
    const size_t wslot = 2 * (size_t)p.wtile_bytes;
    // a tall halo (large dilation) costs more than one box per tap, or does not fit: one patch per tap instead
    if (max_off > 0 && ((size_t)rows * TW * row_unit * 2 * 2 + 2 * wslot > 220 * 1024 || rows * np >= TH * ntaps)) {
        MS_REQUIRE(ntaps <= BF_MAX_PATCH, "conv_bf: too many per-tap patches");
        for (int i = 0; i < ntaps; ++i) {
            BfPatch& pt = p.patch[i];
            pt.dx = (short)taps[i].dx; pt.dy = (short)taps[i].dy; pt.tap0 = (short)i; pt.ntaps = 1;
            p.tap[i].row_off = 0; p.tap[i].widx = (short)taps[i].widx;
        }
        p.n_patches = ntaps;
        rows = TH;
    }
    MS_REQUIRE(rows * sx <= 256 && TW * sx <= 256, "conv_bf: patch too large for one TMA box");
    p.slot_bytes = (uint32_t)rows * TW * row_unit;
    const size_t pslot = 2 * (size_t)p.slot_bytes;
    const size_t budget = 220 * 1024;
    MS_REQUIRE(2 * pslot + 2 * wslot <= budget, "conv_bf: patch does not fit shared memory");
    // MS_BF_SMEM_KB: cap on the two rings (default: all of the SM).  A CTA that leaves half of the shared memory free lets the
    // NEXT kernel's CTA become resident while this one drains (programmatic dependent launch: barrier set-up, TMEM
    // allocation and tensor-map fetch then overlap); deeper rings only help while loads are the bound.
    static long ring_cap = -1;
    if (ring_cap < 0) { const char* e = getenv("MS_BF_SMEM_KB"); ring_cap = e ? std::max(32L, atol(e)) * 1024 : (long)budget; }
    const size_t grow_budget = std::max<size_t>(std::min<size_t>(budget, (size_t)ring_cap), 2 * pslot + 2 * wslot);
    int NP = 2, NW = 2;
    for (;;) {                                       // grow the two rings alternately while they fit (weights first: smaller)
        bool grew = false;
        if (NW < 8 && (size_t)NP * pslot + (size_t)(NW + 1) * wslot <= grow_budget && NW <= 2 * NP) { ++NW; grew = true; }
        if (NP < 4 && (size_t)(NP + 1) * pslot + (size_t)NW * wslot <= grow_budget) { ++NP; grew = true; }
        if (!grew) break;
    }
    p.NP = NP; p.NW = NW;
    static int nacc_env = -1, nprod_env = -1;
    if (nacc_env < 0) { const char* e = getenv("MS_BF_NACC"); nacc_env = e ? atoi(e) : 2; }
    if (nprod_env < 0) { const char* e = getenv("MS_BF_NPROD"); nprod_env = e ? atoi(e) : 3; }
    p.nprod = nprod_env == 1 ? 1 : 3;
    p.nacc = (nacc_env == 1 || p.nprod == 1) ? 1 : 2;
    {
        const int need = p.nacc * N;
        p.tmem_cols = need <= 32 ? 32 : (need <= 64 ? 64 : (need <= 128 ? 128 : (need <= 256 ? 256 : 512)));
    }
    p.y = g.y.p; p.ycs = g.y.cs; p.bias = g.bias; p.alpha = g.alpha;
    p.res = g.res; p.res_cs = g.res_cs; p.mask = g.mask; p.mask_cs = g.mask_cs; p.mask_alpha = g.mask_alpha;
    p.accumulate = g.accumulate;
    if (yp && yp->hi) {
        MS_REQUIRE(yp->cs >= M && (yp->cs & 7) == 0, "conv_bf: bad output planes");
        p.ohi = yp->hi; p.olo = yp->lo; p.ocs = yp->cs; p.ofmt = yp->fmt; p.oscale = yp->fmt == 1 ? yp->scale : 1.f;
    }
    p.wtiles = static_cast<const unsigned char*>(wtiles);
    // ---- split K over (K block, patch) units when the map is too small to fill the GPU (at most 8 ways: the closing
    //      CTA reads every partial sum)
    const int grid_tiles = p.NB * p.tiles_x * p.tiles_y;
    const int units = p.kblocks * p.n_patches;
    int ksplit = 1;
    if (part && tickets && (long)grid_tiles * mblocks <= 74 && units > 1) {
        static int kmax = -1;
        if (kmax < 0) { const char* e = getenv("MS_BF_KSPLIT_MAX"); kmax = e ? std::max(1, atoi(e)) : 8; }
        ksplit = std::min(std::min(units, kmax), std::max(1, 148 / (grid_tiles * mblocks)));
        // MS_BF_SPLIT_CYCLES = c: split only while a CTA's share of the main loop stays above c MMA cycles (taps x k16 x
        // 3 products x N/2).  Measured (profiles/r2_split_heuristic.log): un-splitting the small maps (c = 8192) LOSES 5 % of
        // the step (521 vs 552 FPS) -- the serial K loop of a 3-30 CTA grid costs more than the partial-sum round trip --
        // so the default keeps every split (c = 1).
        static int min_cyc = -1;
        if (min_cyc < 0) { const char* e = getenv("MS_BF_SPLIT_CYCLES"); min_cyc = e ? atoi(e) : 1; }
        const long loop_cycles = (long)p.kblocks * nt * (p.kch / 16) * (p.nprod == 1 ? 1 : 3) * (N / 2);
        ksplit = (int)std::max<long>(1, std::min<long>(ksplit, loop_cycles / std::max(min_cyc, 1)));
        while (ksplit > 1 && (size_t)ksplit * grid_tiles * mblocks * N * 128 > conv_bf_part_floats()) --ksplit;
        if ((size_t)grid_tiles * mblocks > conv_bf_ticket_words()) ksplit = 1;
    }
    p.ksplit = ksplit; p.part = part; p.tickets = tickets;
    {
        static int prof_env = -1;
        if (prof_env < 0) { const char* e = getenv("MS_BF_PROF"); prof_env = e ? atoi(e) : 0; }
        p.prof = nullptr;
        if (prof_env) {
            if (!g_bf_prof) cudaMalloc(reinterpret_cast<void**>(&g_bf_prof), (size_t)BF_PROF_MAX * 8 * sizeof(unsigned long long));
            const int nctas = grid_tiles * mblocks * ksplit;
            if (g_bf_prof && nctas <= BF_PROF_MAX) { p.prof = g_bf_prof; g_bf_prof_ctas = nctas; }
        }
    }
    { static int dbg = -1; if (dbg < 0) { const char* e = getenv("MS_BF_DEBUG"); dbg = e ? atoi(e) : 0; } p.debug = dbg; }

    const CUtensorMap *mXh, *mXl;
    {
        cuuint64_t dims[4] = {(cuuint64_t)g.x.c, (cuuint64_t)g.x.w, (cuuint64_t)g.x.h, (cuuint64_t)g.x.n};
        cuuint64_t strides[3] = {(cuuint64_t)xp.cs * 2, (cuuint64_t)g.x.w * xp.cs * 2, (cuuint64_t)g.x.h * g.x.w * xp.cs * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.kch, (cuuint32_t)(TW * sx), (cuuint32_t)(rows * sx), 1};
        cuuint32_t es[4] = {1, (cuuint32_t)sx, (cuuint32_t)sx, 1};
        if (bf_get_map(&mXh, xp.hi, 4, dims, strides, box, es, p.kch == 64 ? 128 : 64)) return -1;
        if (bf_get_map(&mXl, xp.lo, 4, dims, strides, box, es, p.kch == 64 ? 128 : 64)) return -1;
    }
    const size_t smem = (size_t)NP * pslot + (size_t)NW * wslot + 1024;
    launch_k(conv_bf_kernel, dim3(grid_tiles, mblocks, ksplit), dim3(BF_THREADS), smem, st, *mXh, *mXl, p);
    return check_launch("conv_bf");
}

// xp: 16-bit planes of g.x;  wtiles: prepared weight tiles in the SAME format as xp;  yp: optional planes of g.y (written
// by the epilogue in yp->fmt)
int conv_bf(const ConvGemm& g, const ActPlanes& xp, const void* wtiles, const ActPlanes* yp,
            float* part, unsigned int* tickets, cudaStream_t st) {
    MS_REQUIRE(conv_bf_supported(g), "conv_bf: unsupported geometry");
    MS_REQUIRE(xp.hi && xp.lo && (xp.cs & 7) == 0 && xp.cs >= g.x.c, "conv_bf: input planes missing");
    if (conv_bf_init()) return -1;
    const int taps_total = g.kh * g.kw;
    BfTapSpec taps[BF_MAX_TAPS];
    if (g.div == 1) {
        // gathered input pixel = out * mul + off + tap * step
        int n = 0;
        for (int s = 0; s < g.kw; ++s)
            for (int r = 0; r < g.kh; ++r) taps[n++] = BfTapSpec{g.off_y + r * g.step, g.off_x + s * g.step, r * g.kw + s};
        return conv_bf_launch(g, xp, wtiles, yp, part, tickets, g.y.h, g.y.w, 1, 0, 0, g.mul, taps, n, taps_total, st);
    }
    // fractionally strided gather (stride-2 dgrad, conv_transpose): t = out + off + tap*step must be even, input = t / 2.
    // Output pixels of one parity class (py, px) see a fixed subset of the taps at unit input stride: four dense launches.
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
            const int Hj = (g.y.h - py + 1) / 2, Wj = (g.y.w - px + 1) / 2;
            if (Hj <= 0 || Wj <= 0) continue;
            int n = 0;
            for (int s = 0; s < g.kw; ++s) {
                const int tx = px + g.off_x + s * g.step;
                if (tx & 1) continue;
                for (int r = 0; r < g.kh; ++r) {
                    const int ty = py + g.off_y + r * g.step;
                    if (ty & 1) continue;
                    taps[n++] = BfTapSpec{ty / 2, tx / 2, r * g.kw + s};    // exact: ty, tx even (C++ division truncates toward 0)
                }
            }
            if (n == 0) { set_error("conv_bf: parity class without taps"); return -2; }
            if (conv_bf_launch(g, xp, wtiles, yp, part, tickets, Hj, Wj, 2, py, px, 1, taps, n, taps_total, st)) return -1;
        }
    return 0;
}

// one-shot convenience (operator-level C ABI / tests): splits the input, prepares the weights, runs the conv.
//   fmt: operand format (1 = fp16 forward planes, 0 = bf16 gradient planes)
//   scratch layout (bytes): [x hi | x lo | weight tiles | job | tickets | split-K partials]
size_t conv_bf_oneshot_scratch_bytes(const ConvGemm& g) {
    const size_t xe = g.x.pixels() * ((g.x.c + 7) / 8 * 8);
    const size_t we = conv_bf_weight_halfs(g.kh * g.kw, g.y.c, g.x.c);
    return 2 * (xe * 2 + 256) + (we * 2 + 256) + 1024 + conv_bf_ticket_words() * 4 + conv_bf_part_floats() * 4 + 4096;
}

int conv_bf_oneshot(const ConvGemm& g, int wmat_is_mk, int fmt, float act_scale, void* scratch, size_t scratch_bytes, cudaStream_t st) {
    MS_REQUIRE(conv_bf_supported(g), "conv_bf: unsupported geometry");
    MS_REQUIRE(scratch_bytes >= conv_bf_oneshot_scratch_bytes(g), "conv_bf: scratch too small");
    MS_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 255) == 0, "conv_bf: scratch must be 256B aligned");
    unsigned char* b = reinterpret_cast<unsigned char*>(scratch);
    auto take = [&](size_t bytes) { unsigned char* r = b; b += (bytes + 255) / 256 * 256; return r; };
    const int pcs = (g.x.c + 7) / 8 * 8;
    const size_t xe = g.x.pixels() * pcs;
    const size_t we = conv_bf_weight_halfs(g.kh * g.kw, g.y.c, g.x.c);
    ActPlanes xp; xp.hi = take(xe * 2); xp.lo = take(xe * 2); xp.cs = pcs; xp.fmt = fmt; xp.scale = fmt == 1 ? act_scale : 1.f;
    void* wt = take(we * 2);
    BfPrepJob* jd = reinterpret_cast<BfPrepJob*>(take(1024));
    unsigned int* tickets = reinterpret_cast<unsigned int*>(take(conv_bf_ticket_words() * 4));
    float* part = reinterpret_cast<float*>(take(conv_bf_part_floats() * 4));
    int Mpad, Kpad; conv_bf_weight_dims(g.y.c, g.x.c, Mpad, Kpad);
    BfPrepJob job{g.wmat, wt, g.kh * g.kw, g.y.c, g.x.c, Mpad, Kpad, wmat_is_mk ? 0 : 1, fmt};
    MS_CHECK_CUDA(cudaMemcpyAsync(jd, &job, sizeof job, cudaMemcpyHostToDevice, st));
    MS_CHECK_CUDA(cudaMemsetAsync(tickets, 0, conv_bf_ticket_words() * 4, st));
    if (bf_prep_weights(jd, 1, we, st)) return -1;
    if (split_planes(g.x, xp, st)) return -1;
    return conv_bf(g, xp, wt, nullptr, part, tickets, st);
}

}  // namespace ms
