// Direct fp32 kernels for the two full-resolution pyramid layers whose channel counts are too small for a GEMM tile:
// MADNet conv1 (3 -> 16, 3x3 stride 2) and conv2 (16 -> 16, 3x3), reference Nets/MadNet.py:173-190 built from
// sharedLayers.conv2d (Nets/sharedLayers.py:54-63), and the filter gradients tf.gradients derives for them in the
// module-2 train op (Stereo_Online_Adaptation.py:118).
//
// The launch list (profiles/r1_launches_final_summary.txt) had the gather GEMM at 105 us for conv1 forward (0.2 GFLOP,
// 27 MB: it should be a ~10 us HBM-bound kernel) and 319 + 271 us for the conv1 / conv2 weight gradients (432 / 2304
// outputs reduced over 245 760 pixels: a 16 x 16 output tile leaves the GEMM kernel with 9 CTAs per K split).
//   forward  : one thread computes two adjacent output pixels x all output channels; the weights sit in shared memory
//              and are read as broadcast float4.  105 -> 30 us for conv1.  (16 -> 16 | 32 instantiations exist but are
//              opt-in: without a staged input patch they are slower than the gather GEMM, see conv_small_fwd_supported.)
//   wgrad    : a thread owns one input channel ("role") and keeps all 9 taps x 16 output channels = 144 partial sums
//              in registers while it walks its share of the pixels (9 input loads + 16 dY loads per 144 FMAs, next
//              pixel prefetched); lanes of equal role are combined by shuffles, warps through shared memory, CTAs by
//              the fixed-order wgrad_reduce pass (deterministic).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace ms {

static __host__ __device__ bool al16s(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---------------------------------------------------------------------------------------------
// forward / stride-1 dgrad gather, 3x3, (cin, cout) in {(3,16), (16,16), (16,32)}
// ---------------------------------------------------------------------------------------------
constexpr int CS_NT = 128;

template <int CIN, int CO>
__global__ void __launch_bounds__(CS_NT) conv_small_fwd_kernel(ConvGemm p, int pairs_per_row, int total_pairs) {
    pdl_prologue();
    __shared__ __align__(16) float ws[9 * CIN * CO];                               // [tap][ci][co]
    __shared__ float bs[CO];
    for (int i = threadIdx.x; i < 9 * CIN * CO; i += CS_NT) ws[i] = p.wmat[i];
    for (int i = threadIdx.x; i < CO; i += CS_NT) bs[i] = p.bias ? p.bias[i] : 0.f;
    __syncthreads();
    const int e = blockIdx.x * CS_NT + threadIdx.x;
    if (e >= total_pairs) return;
    const int xp = e % pairs_per_row;
    const int q = e / pairs_per_row;
    const int oy = q % p.y.h, img = q / p.y.h;
    const int ox0 = xp * 2;
    float acc[2][CO];
#pragma unroll
    for (int j = 0; j < CO; ++j) { acc[0][j] = bs[j]; acc[1][j] = bs[j]; }
    const float* ximg = p.x.p + (size_t)img * p.x.h * p.x.w * p.x.cs;
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
        const int ty = tap / 3, tx = tap - ty * 3;
        const int iy = oy * p.mul + p.off_y + ty * p.step;
        const bool rok = iy >= 0 && iy < p.x.h;
        float xin[2][CIN];
#pragma unroll
        for (int pi = 0; pi < 2; ++pi) {
            const int ix = (ox0 + pi) * p.mul + p.off_x + tx * p.step;
            const bool ok = rok && ix >= 0 && ix < p.x.w;
            const float* s = ximg + ((size_t)(ok ? iy : 0) * p.x.w + (ok ? ix : 0)) * p.x.cs;
            if constexpr (CIN % 4 == 0) {
#pragma unroll
                for (int c4 = 0; c4 < CIN / 4; ++c4) {
                    const float4 v = ok ? __ldg(reinterpret_cast<const float4*>(s) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
                    xin[pi][4 * c4] = v.x; xin[pi][4 * c4 + 1] = v.y; xin[pi][4 * c4 + 2] = v.z; xin[pi][4 * c4 + 3] = v.w;
                }
            } else {
#pragma unroll
                for (int c = 0; c < CIN; ++c) xin[pi][c] = ok ? __ldg(s + c) : 0.f;
            }
        }
        const float4* wt = reinterpret_cast<const float4*>(ws + tap * CIN * CO);
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
            const float a0 = xin[0][c], a1 = xin[1][c];
#pragma unroll
            for (int j4 = 0; j4 < CO / 4; ++j4) {
                const float4 w = wt[c * (CO / 4) + j4];
                acc[0][4 * j4] = fmaf(a0, w.x, acc[0][4 * j4]); acc[0][4 * j4 + 1] = fmaf(a0, w.y, acc[0][4 * j4 + 1]);
                acc[0][4 * j4 + 2] = fmaf(a0, w.z, acc[0][4 * j4 + 2]); acc[0][4 * j4 + 3] = fmaf(a0, w.w, acc[0][4 * j4 + 3]);
                acc[1][4 * j4] = fmaf(a1, w.x, acc[1][4 * j4]); acc[1][4 * j4 + 1] = fmaf(a1, w.y, acc[1][4 * j4 + 1]);
                acc[1][4 * j4 + 2] = fmaf(a1, w.z, acc[1][4 * j4 + 2]); acc[1][4 * j4 + 3] = fmaf(a1, w.w, acc[1][4 * j4 + 3]);
            }
        }
    }
    const bool vec = (p.y.cs & 3) == 0 && al16s(p.y.p);
#pragma unroll
    for (int pi = 0; pi < 2; ++pi) {
        const int ox = ox0 + pi;
        if (ox >= p.y.w) break;
        const size_t pix = (size_t)(img * p.y.h + oy) * p.y.w + ox;
        float* yrow = p.y.p + pix * p.y.cs;
#pragma unroll
        for (int j = 0; j < CO; ++j) {                       // same epilogue order as conv_gemm_kernel
            float t = fmaxf(p.alpha * acc[pi][j], acc[pi][j]);
            if (p.res) t += p.res[pix * p.res_cs + j];
            if (p.accumulate) t += yrow[j];
            if (p.mask) t *= (p.mask[pix * p.mask_cs + j] > 0.f) ? 1.f : p.mask_alpha;
            acc[pi][j] = t;
        }
        if (vec) {
#pragma unroll
            for (int j = 0; j < CO; j += 4)
                *reinterpret_cast<float4*>(yrow + j) = make_float4(acc[pi][j], acc[pi][j + 1], acc[pi][j + 2], acc[pi][j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < CO; ++j) yrow[j] = acc[pi][j];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// 16 -> 16, 3x3, stride 1 (conv2 forward and its dgrad): shared-memory staged version.  A CTA owns an 8 x 32 output tile;
// the 10 x 34 input patch is loaded with coalesced 128-bit loads into shared memory with a 20-float pixel pitch (a
// quarter-warp's 128-bit reads at one-pixel lane stride then hit 32 distinct banks); a thread computes pixels (r, c) and
// (r, c + 16) so that lanes stay one pixel apart.  Default (MS_CONV_SMALL16=2; 0 = gather GEMM, 1 = untiled direct
// kernels): validated with the ops + MADNet GPU suites, conv_fwd 1.600 -> 1.575 ms per frame (profiles/r1_last_visit.log).
// ---------------------------------------------------------------------------------------------
constexpr int T16_TH = 8, T16_TW = 32, T16_PH = T16_TH + 2, T16_PW = T16_TW + 2, T16_PS = 20, T16_NT = 128;

__global__ void __launch_bounds__(T16_NT) conv_c16_tiled_kernel(ConvGemm p, int tiles_x, int tiles_y) {
    pdl_prologue();
    constexpr int CIN = 16, CO = 16;
    __shared__ __align__(16) float ws[9 * CIN * CO];
    __shared__ __align__(16) float patch[T16_PH * T16_PW * T16_PS];
    __shared__ float bs[CO];
    int bid = blockIdx.x;
    const int tx_ = bid % tiles_x; bid /= tiles_x;
    const int ty_ = bid % tiles_y;
    const int img = bid / tiles_y;
    const int y0 = ty_ * T16_TH, x0 = tx_ * T16_TW;
    const int miny = p.off_y + (p.step < 0 ? 2 * p.step : 0), minx = p.off_x + (p.step < 0 ? 2 * p.step : 0);
    for (int i = threadIdx.x; i < 9 * CIN * CO / 4; i += T16_NT)
        reinterpret_cast<float4*>(ws)[i] = __ldg(reinterpret_cast<const float4*>(p.wmat) + i);
    for (int i = threadIdx.x; i < CO; i += T16_NT) bs[i] = p.bias ? p.bias[i] : 0.f;
    const float* ximg = p.x.p + (size_t)img * p.x.h * p.x.w * p.x.cs;
    for (int e = threadIdx.x; e < T16_PH * T16_PW * 4; e += T16_NT) {
        const int pix = e >> 2, q = e & 3;
        const int py = pix / T16_PW, px = pix - py * T16_PW;
        const int iy = y0 + miny + py, ix = x0 + minx + px;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (iy >= 0 && iy < p.x.h && ix >= 0 && ix < p.x.w)
            v = __ldg(reinterpret_cast<const float4*>(ximg + ((size_t)iy * p.x.w + ix) * p.x.cs) + q);
        *reinterpret_cast<float4*>(patch + pix * T16_PS + q * 4) = v;
    }
    __syncthreads();
    const int r = threadIdx.x >> 4, c = threadIdx.x & 15;
    float acc[2][CO];
#pragma unroll
    for (int j = 0; j < CO; ++j) { acc[0][j] = bs[j]; acc[1][j] = bs[j]; }
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
        const int ty = tap / 3, tx = tap - ty * 3;
        const int pr = r + p.off_y + ty * p.step - miny, pc = c + p.off_x + tx * p.step - minx;
        const float* s0 = patch + (pr * T16_PW + pc) * T16_PS;
        float xin[2][CIN];
#pragma unroll
        for (int pi = 0; pi < 2; ++pi)
#pragma unroll
            for (int c4 = 0; c4 < CIN / 4; ++c4) {
                const float4 v = *reinterpret_cast<const float4*>(s0 + pi * 16 * T16_PS + c4 * 4);
                xin[pi][4 * c4] = v.x; xin[pi][4 * c4 + 1] = v.y; xin[pi][4 * c4 + 2] = v.z; xin[pi][4 * c4 + 3] = v.w;
            }
        const float4* wt = reinterpret_cast<const float4*>(ws + tap * CIN * CO);
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
            const float a0 = xin[0][ci], a1 = xin[1][ci];
#pragma unroll
            for (int j4 = 0; j4 < CO / 4; ++j4) {
                const float4 w = wt[ci * (CO / 4) + j4];
                acc[0][4 * j4] = fmaf(a0, w.x, acc[0][4 * j4]); acc[0][4 * j4 + 1] = fmaf(a0, w.y, acc[0][4 * j4 + 1]);
                acc[0][4 * j4 + 2] = fmaf(a0, w.z, acc[0][4 * j4 + 2]); acc[0][4 * j4 + 3] = fmaf(a0, w.w, acc[0][4 * j4 + 3]);
                acc[1][4 * j4] = fmaf(a1, w.x, acc[1][4 * j4]); acc[1][4 * j4 + 1] = fmaf(a1, w.y, acc[1][4 * j4 + 1]);
                acc[1][4 * j4 + 2] = fmaf(a1, w.z, acc[1][4 * j4 + 2]); acc[1][4 * j4 + 3] = fmaf(a1, w.w, acc[1][4 * j4 + 3]);
            }
        }
    }
    const bool vec = (p.y.cs & 3) == 0 && al16s(p.y.p);
    const int oy = y0 + r;
    if (oy >= p.y.h) return;
#pragma unroll
    for (int pi = 0; pi < 2; ++pi) {
        const int ox = x0 + c + pi * 16;
        if (ox >= p.y.w) continue;
        const size_t pix = (size_t)(img * p.y.h + oy) * p.y.w + ox;
        float* yrow = p.y.p + pix * p.y.cs;
#pragma unroll
        for (int j = 0; j < CO; ++j) {
            float t = fmaxf(p.alpha * acc[pi][j], acc[pi][j]);
            if (p.res) t += p.res[pix * p.res_cs + j];
            if (p.accumulate) t += yrow[j];
            if (p.mask) t *= (p.mask[pix * p.mask_cs + j] > 0.f) ? 1.f : p.mask_alpha;
            acc[pi][j] = t;
        }
        if (vec) {
#pragma unroll
            for (int j = 0; j < CO; j += 4)
                *reinterpret_cast<float4*>(yrow + j) = make_float4(acc[pi][j], acc[pi][j + 1], acc[pi][j + 2], acc[pi][j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < CO; ++j) yrow[j] = acc[pi][j];
        }
    }
}

static int small16_mode() {
    static int m = -1;
    if (m < 0) { const char* e = getenv("MS_CONV_SMALL16"); m = e ? atoi(e) : 2; }
    return m;
}

static bool conv_c16_tiled_supported(const ConvGemm& p) {
    return p.x.c == 16 && p.y.c == 16 && p.kh == 3 && p.kw == 3 && p.div == 1 && p.mul == 1 && (p.step == 1 || p.step == -1) &&
           p.x.h == p.y.h && p.x.w == p.y.w && p.x.n == p.y.n && (p.x.cs & 3) == 0 && al16s(p.x.p) && al16s(p.wmat) &&
           p.alpha <= 1.f && p.alpha >= 0.f;
}

bool conv_small_fwd_supported(const ConvGemm& p) {
    if (p.kh != 3 || p.kw != 3 || p.div != 1 || p.mul < 1 || p.x.n != p.y.n || p.alpha > 1.f || p.alpha < 0.f) return false;
    if (p.x.c == 3 && p.y.c == 16) return true;
    // The untiled 16-channel instantiations are opt-in (MS_CONV_SMALL16=1): measured 86 us (16->16) and 36 us (16->32
    // stride 2) against 71 / 32 us for the gather GEMM -- one thread reading its pixels' 64-byte channel rows straight
    // from global memory is LSU-bound (32 cache lines per load instruction).  The default (=2) is the shared-memory
    // tiled 16->16 stride-1 kernel above.
    if (small16_mode() == 2 && conv_c16_tiled_supported(p)) return true;
    if (small16_mode() == 1 && p.x.c == 16 && (p.y.c == 16 || p.y.c == 32)) return (p.x.cs & 3) == 0 && al16s(p.x.p);
    return false;
}

int conv_small_fwd(const ConvGemm& p, cudaStream_t st) {
    if (small16_mode() == 2 && conv_c16_tiled_supported(p)) {
        const int tiles_x = cdiv(p.y.w, T16_TW), tiles_y = cdiv(p.y.h, T16_TH);
        launch_k(conv_c16_tiled_kernel, dim3((unsigned)(tiles_x * tiles_y * p.y.n)), dim3(T16_NT), 0, st, p, tiles_x, tiles_y);
        return check_launch("conv_c16_tiled");
    }
    const int pairs_per_row = cdiv(p.y.w, 2);
    const size_t total = (size_t)p.y.n * p.y.h * pairs_per_row;
    MS_REQUIRE(total < (1u << 30), "conv_small_fwd: too many output pixels");
    const unsigned grid = (unsigned)cdivz(total, CS_NT);
    if (p.x.c == 3) launch_k(conv_small_fwd_kernel<3, 16>, dim3(grid), dim3(CS_NT), 0, st, p, pairs_per_row, (int)total);
    else if (p.y.c == 16) launch_k(conv_small_fwd_kernel<16, 16>, dim3(grid), dim3(CS_NT), 0, st, p, pairs_per_row, (int)total);
    else launch_k(conv_small_fwd_kernel<16, 32>, dim3(grid), dim3(CS_NT), 0, st, p, pairs_per_row, (int)total);
    return check_launch("conv_small_fwd");
}

// ---------------------------------------------------------------------------------------------
// weight gradient, 3x3, co = 16, ci <= 16
// ---------------------------------------------------------------------------------------------
constexpr int SW_NT = 256;
constexpr int SW_CO = 16;
constexpr int SW_TAPS = 9;
constexpr int SW_ACC = SW_TAPS * SW_CO;     // 144 partial sums per thread

struct SwOperands { float x[SW_TAPS]; float4 d[SW_CO / 4]; };

template <int RP>   // roles per pixel slot: ci padded to 4 / 8 / 16
__global__ void __launch_bounds__(SW_NT, 1) conv_small_wgrad_kernel(ConvWgrad p, int P, int chunk, float* __restrict__ partial) {
    pdl_prologue();
    extern __shared__ float sw_smem[];                       // [warps][RP][144]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int role = tid % RP, slot = tid / RP;
    constexpr int NSLOT = SW_NT / RP;
    const int ci = p.x.c;
    const bool live = role < ci;
    const int W = p.dy.w, H = p.dy.h;
    const bool dvec = (p.dy.cs & 3) == 0 && ((reinterpret_cast<uintptr_t>(p.dy.p) & 15) == 0);
    const int p_begin = blockIdx.x * chunk, p_end = min(P, p_begin + chunk);

    float acc[SW_TAPS][SW_CO];
#pragma unroll
    for (int t = 0; t < SW_TAPS; ++t)
#pragma unroll
        for (int j = 0; j < SW_CO; ++j) acc[t][j] = 0.f;

    int pp = p_begin + slot;
    int ox = 0, oy = 0, img = 0;
    if (pp < p_end) { ox = pp % W; const int q = pp / W; oy = q % H; img = q / H; }

    auto load = [&](int pix, int lx, int ly, int limg, SwOperands& o) {
        const bool ok = pix < p_end;
#pragma unroll
        for (int j4 = 0; j4 < SW_CO / 4; ++j4) o.d[j4] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) {
            const float* dsrc = p.dy.p + (size_t)pix * p.dy.cs;
            if (dvec) {
#pragma unroll
                for (int j4 = 0; j4 < SW_CO / 4; ++j4) o.d[j4] = __ldg(reinterpret_cast<const float4*>(dsrc) + j4);
            } else {
#pragma unroll
                for (int j4 = 0; j4 < SW_CO / 4; ++j4)
                    o.d[j4] = make_float4(__ldg(dsrc + 4 * j4), __ldg(dsrc + 4 * j4 + 1), __ldg(dsrc + 4 * j4 + 2), __ldg(dsrc + 4 * j4 + 3));
            }
        }
        const float* ximg = p.x.p + (size_t)limg * p.x.h * p.x.w * p.x.cs + role;
#pragma unroll
        for (int t = 0; t < SW_TAPS; ++t) {
            const int iy = ly * p.stride - p.pad_t + (t / 3) * p.dil;
            const int ix = lx * p.stride - p.pad_l + (t % 3) * p.dil;
            const bool in = ok && live && iy >= 0 && iy < p.x.h && ix >= 0 && ix < p.x.w;
            o.x[t] = in ? __ldg(ximg + ((size_t)iy * p.x.w + ix) * p.x.cs) : 0.f;
        }
    };
    auto advance = [&](int& lx, int& ly, int& limg) {
        lx += NSLOT;
        while (lx >= W) { lx -= W; if (++ly >= H) { ly = 0; ++limg; } }
    };

    SwOperands cur, nxt;
    load(pp, ox, oy, img, cur);
    while (pp < p_end) {
        const int pn = pp + NSLOT;
        advance(ox, oy, img);
        load(pn, ox, oy, img, nxt);
#pragma unroll
        for (int t = 0; t < SW_TAPS; ++t) {
            const float a = cur.x[t];
#pragma unroll
            for (int j4 = 0; j4 < SW_CO / 4; ++j4) {
                acc[t][4 * j4] = fmaf(a, cur.d[j4].x, acc[t][4 * j4]);
                acc[t][4 * j4 + 1] = fmaf(a, cur.d[j4].y, acc[t][4 * j4 + 1]);
                acc[t][4 * j4 + 2] = fmaf(a, cur.d[j4].z, acc[t][4 * j4 + 2]);
                acc[t][4 * j4 + 3] = fmaf(a, cur.d[j4].w, acc[t][4 * j4 + 3]);
            }
        }
        cur = nxt;
        pp = pn;
    }
    // lanes of equal role (lane % RP) -> lane < RP
#pragma unroll
    for (int t = 0; t < SW_TAPS; ++t)
#pragma unroll
        for (int j = 0; j < SW_CO; ++j) {
            float v = acc[t][j];
#pragma unroll
            for (int off = RP; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            acc[t][j] = v;
        }
    if (lane < RP) {
        float* dst = sw_smem + ((size_t)warp * RP + lane) * SW_ACC;
#pragma unroll
        for (int t = 0; t < SW_TAPS; ++t)
#pragma unroll
            for (int j = 0; j < SW_CO; ++j) dst[t * SW_CO + j] = acc[t][j];
    }
    __syncthreads();
    float* out = partial + (size_t)blockIdx.x * SW_TAPS * ci * SW_CO;        // [tap][ci][co]
    for (int e = tid; e < ci * SW_ACC; e += SW_NT) {
        const int r = e / SW_ACC, rem = e - r * SW_ACC;
        const int t = rem / SW_CO, j = rem - t * SW_CO;
        float s = 0.f;
#pragma unroll
        for (int wv = 0; wv < SW_NT / 32; ++wv) s += sw_smem[((size_t)wv * RP + r) * SW_ACC + rem];
        out[((size_t)t * ci + r) * SW_CO + j] = s;
    }
}

bool conv_small_wgrad_shape(int taps, int ci, int co) { return taps == 9 && co == SW_CO && ci >= 1 && ci <= 16; }

static int small_wgrad_split(size_t P) { return (int)std::min<size_t>(148, std::max<size_t>(1, P / 512)); }

size_t conv_small_wgrad_workspace_floats(int taps, int ci, int co, size_t P) {
    return (size_t)small_wgrad_split(P) * taps * ci * co;
}

bool conv_small_wgrad_supported(const ConvWgrad& p) {
    return p.kh == 3 && p.kw == 3 && conv_small_wgrad_shape(9, p.x.c, p.dy.c) && p.x.n == p.dy.n &&
           (size_t)p.dy.n * p.dy.h * p.dy.w >= 4096;
}

// partial sums -> p.workspace[0 .. split*taps*ci*co); returns the split through *split_out
int conv_small_wgrad(const ConvWgrad& p, int* split_out, cudaStream_t st) {
    const size_t Pz = (size_t)p.dy.n * p.dy.h * p.dy.w;
    MS_REQUIRE(Pz < (1u << 30), "conv_small_wgrad: too many pixels");
    const int P = (int)Pz, ci = p.x.c;
    const int split = small_wgrad_split(Pz);
    const int chunk = cdiv(P, split);
    MS_REQUIRE(p.workspace_floats >= (size_t)split * 9 * ci * SW_CO, "conv_small_wgrad: workspace too small");
    static bool attr = false;
    if (!attr) {
        MS_CHECK_CUDA(cudaFuncSetAttribute(conv_small_wgrad_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr = true;
    }
    const int rp = ci <= 4 ? 4 : (ci <= 8 ? 8 : 16);
    const size_t smem = (size_t)(SW_NT / 32) * rp * SW_ACC * sizeof(float);
    if (rp == 4) launch_k(conv_small_wgrad_kernel<4>, dim3(split), dim3(SW_NT), smem, st, p, P, chunk, p.workspace);
    else if (rp == 8) launch_k(conv_small_wgrad_kernel<8>, dim3(split), dim3(SW_NT), smem, st, p, P, chunk, p.workspace);
    else launch_k(conv_small_wgrad_kernel<16>, dim3(split), dim3(SW_NT), smem, st, p, P, chunk, p.workspace);
    *split_out = split;
    return check_launch("conv_small_wgrad");
}

}  // namespace ms
