// fp32 CUDA-core implicit-GEMM convolution family (sm_100a).
//
// Replaces, for the hot path, the cuDNN calls behind tf.nn.conv2d / atrous_conv2d / conv2d_transpose
// (reference Nets/sharedLayers.py:54-92) and the conv gradients tf.gradients derives for them.
// One "gather GEMM" kernel serves conv forward, conv dgrad and conv_transpose forward (see ConvGemm in
// common.cuh); a second kernel computes weight gradients as a split-K GEMM over pixels with a
// deterministic two-pass reduction.  This is the exact-fp32 path: the generic fallback for every layer shape the
// split-16-bit tensor-core path (conv_bf.cu, wgrad_bf.cu) does not take, and the op-level reference for it.
#include "common.cuh"
#include <algorithm>
#include <cstdlib>

namespace ms {

constexpr int BK = 16;
constexpr int NT = 256;

__device__ __forceinline__ float leaky_f(float v, float a) { return fmaxf(a * v, v); }

// ---------------------------------------------------------------------------------------------
// shared compute core: C[TM x TN per thread] += As[k][m] * Bs[k][n]
// ---------------------------------------------------------------------------------------------
template <int TM, int TN, int LDA, int LDB>
__device__ __forceinline__ void mma_tile(const float* __restrict__ As, const float* __restrict__ Bs,
                                         int tm, int tn, float (&acc)[TM][TN]) {
#pragma unroll
    for (int k = 0; k < BK; ++k) {
        float a[TM], b[TN];
        if constexpr (TM >= 4) {
#pragma unroll
            for (int i = 0; i < TM; i += 4) {
                float4 v = *reinterpret_cast<const float4*>(&As[k * LDA + tm * TM + i]);
                a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
            }
        } else if constexpr (TM == 2) {
            float2 v = *reinterpret_cast<const float2*>(&As[k * LDA + tm * TM]);
            a[0] = v.x; a[1] = v.y;
        } else {
            a[0] = As[k * LDA + tm];
        }
        if constexpr (TN == 8) {
            float4 v = *reinterpret_cast<const float4*>(&Bs[k * LDB + tn * 8]);
            float4 u = *reinterpret_cast<const float4*>(&Bs[k * LDB + tn * 8 + 4]);
            b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w; b[4] = u.x; b[5] = u.y; b[6] = u.z; b[7] = u.w;
        } else if constexpr (TN == 4) {
            float4 v = *reinterpret_cast<const float4*>(&Bs[k * LDB + tn * 4]);
            b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
        } else if constexpr (TN == 2) {
            float2 v = *reinterpret_cast<const float2*>(&Bs[k * LDB + tn * 2]);
            b[0] = v.x; b[1] = v.y;
        } else {
            b[0] = Bs[k * LDB + tn];
        }
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
}

// ---------------------------------------------------------------------------------------------
// gather GEMM: M = n*yh*yw output pixels, N = y.c, K = taps * x.c
// ---------------------------------------------------------------------------------------------
template <int TN, bool AVEC, bool BVEC>
__global__ void __launch_bounds__(NT) conv_gemm_kernel(ConvGemm p, int M) {
    constexpr int TM = 8, BM = 128, BN = 16 * TN, LDA = BM + 4, LDB = BN;
    constexpr int AR = AVEC ? 2 : 8;  // rows of A handled per thread
    __shared__ __align__(16) float As[2][BK * LDA];
    __shared__ __align__(16) float Bs[2][BK * LDB];

    const int t = threadIdx.x;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int xc = p.x.c, yc = p.y.c;
    const int kc_tiles = (xc + BK - 1) / BK;
    const int taps = p.kh * p.kw;
    const int total_all = taps * kc_tiles;
    const int it0 = (int)(((long)blockIdx.z * total_all) / p.ksplit), it1 = (int)(((long)(blockIdx.z + 1) * total_all) / p.ksplit);
    const int total = it1 - it0;

    // --- per-thread A row metadata
    int row_iy0[AR], row_ix0[AR], row_img[AR];
    const int a_k = AVEC ? (t & 3) * 4 : (t & 15);
#pragma unroll
    for (int j = 0; j < AR; ++j) {
        int r = AVEC ? ((t >> 2) + 64 * j) : ((t >> 4) + 16 * j);
        int m = m0 + r;
        if (m < M) {
            int ox = m % p.y.w;
            int q = m / p.y.w;
            int oy = q % p.y.h;
            row_img[j] = q / p.y.h;
            row_iy0[j] = oy * p.mul + p.off_y;
            row_ix0[j] = ox * p.mul + p.off_x;
        } else {
            row_img[j] = -1; row_iy0[j] = 0; row_ix0[j] = 0;
        }
    }

    float areg[8];
    float breg[4];

    auto load_tiles = [&](int tap, int c0) {
        const int r = tap / p.kw, s = tap - r * p.kw;
        // ---- A
#pragma unroll
        for (int j = 0; j < AR; ++j) {
            bool ok = row_img[j] >= 0;
            int ty = row_iy0[j] + r * p.step, tx = row_ix0[j] + s * p.step;
            if (p.div > 1) {
                ok = ok && ty >= 0 && tx >= 0 && (ty % p.div == 0) && (tx % p.div == 0);
                ty /= p.div; tx /= p.div;
            }
            ok = ok && ty >= 0 && ty < p.x.h && tx >= 0 && tx < p.x.w;
            const int c = c0 + a_k;
            if (AVEC) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok && c < xc) {
                    const float* src = p.x.p + ((size_t)(row_img[j] * p.x.h + ty) * p.x.w + tx) * p.x.cs + c;
                    v = *reinterpret_cast<const float4*>(src);
                    if (c + 1 >= xc) v.y = 0.f;
                    if (c + 2 >= xc) v.z = 0.f;
                    if (c + 3 >= xc) v.w = 0.f;
                }
                areg[4 * j] = v.x; areg[4 * j + 1] = v.y; areg[4 * j + 2] = v.z; areg[4 * j + 3] = v.w;
            } else {
                float v = 0.f;
                if (ok && c < xc)
                    v = p.x.p[((size_t)(row_img[j] * p.x.h + ty) * p.x.w + tx) * p.x.cs + c];
                areg[j] = v;
            }
        }
        // ---- B
        if (BVEC) {
            constexpr int F4 = BN / 4;  // float4 per k-row
            breg[0] = breg[1] = breg[2] = breg[3] = 0.f;
            if (t < BK * F4) {
                int k = t / F4, n = n0 + (t % F4) * 4;
                if (c0 + k < xc && n < yc) {
                    float4 v = *reinterpret_cast<const float4*>(p.wmat + ((size_t)tap * xc + c0 + k) * yc + n);
                    breg[0] = v.x; breg[1] = v.y; breg[2] = v.z; breg[3] = v.w;  // yc%4==0 in BVEC
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                int e = t + NT * j, k = e / BN, n = n0 + e % BN;
                float v = 0.f;
                if (c0 + k < xc && n < yc) v = p.wmat[((size_t)tap * xc + c0 + k) * yc + n];
                breg[j] = v;
            }
        }
    };

    auto store_tiles = [&](int buf) {
        float* as = As[buf];
        float* bs = Bs[buf];
        if (AVEC) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                int r = (t >> 2) + 64 * j;
#pragma unroll
                for (int q = 0; q < 4; ++q) as[(a_k + q) * LDA + r] = areg[4 * j + q];
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) as[a_k * LDA + (t >> 4) + 16 * j] = areg[j];
        }
        if (BVEC) {
            constexpr int F4 = BN / 4;
            if (t < BK * F4) {
                int k = t / F4, n = (t % F4) * 4;
                *reinterpret_cast<float4*>(&bs[k * LDB + n]) = make_float4(breg[0], breg[1], breg[2], breg[3]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                int e = t + NT * j;
                bs[(e / BN) * LDB + e % BN] = breg[j];
            }
        }
    };

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    const int tm = t >> 4, tn = t & 15;
    int tap = it0 / kc_tiles, kc = it0 - tap * kc_tiles;
    if (total > 0) {
    load_tiles(tap, kc * BK);
    store_tiles(0);
    }
    __syncthreads();
    for (int it = 0; it < total; ++it) {
        const int buf = it & 1;
        int ntap = tap, nkc = kc + 1;
        if (nkc == kc_tiles) { nkc = 0; ntap = tap + 1; }
        const bool more = (it + 1 < total);
        if (more) load_tiles(ntap, nkc * BK);
        mma_tile<TM, TN, LDA, LDB>(As[buf], Bs[buf], tm, tn, acc);
        if (more) store_tiles(buf ^ 1);
        __syncthreads();
        tap = ntap; kc = nkc;
    }

    // ---- epilogue
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int m = m0 + tm * TM + i;
        if (m >= M) continue;
        float* yrow = p.y.p + (size_t)m * p.y.cs;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int n = n0 + tn * TN + j;
            if (n >= yc) continue;
            float v = acc[i][j];
            if (p.ksplit > 1) { p.part[((size_t)blockIdx.z * M + m) * yc + n] = v; continue; }
            if (p.bias) v += p.bias[n];
            v = leaky_f(v, p.alpha);
            if (p.res) v += p.res[(size_t)m * p.res_cs + n];
            if (p.accumulate) v += yrow[n];
            if (p.mask) v *= (p.mask[(size_t)m * p.mask_cs + n] > 0.f) ? 1.f : p.mask_alpha;
            yrow[n] = v;
        }
    }
}

__global__ void gemm_splitk_reduce_kernel(ConvGemm p, int M) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int yc = p.y.c;
    if (i >= (size_t)M * yc) return;
    const size_t m = i / yc;
    const int n = (int)(i - m * yc);
    float v = 0.f;
    for (int z = 0; z < p.ksplit; ++z) v += p.part[((size_t)z * M + m) * yc + n];
    if (p.bias) v += p.bias[n];
    v = leaky_f(v, p.alpha);
    if (p.res) v += p.res[m * p.res_cs + n];
    float* yrow = p.y.p + m * p.y.cs;
    if (p.accumulate) v += yrow[n];
    if (p.mask) v *= (p.mask[m * p.mask_cs + n] > 0.f) ? 1.f : p.mask_alpha;
    yrow[n] = v;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

size_t conv_gemm_part_floats() { return (size_t)8 << 20; }      // 32 MB; conv_gemm splits K only as far as it fits

int conv_gemm(const ConvGemm& p_in, cudaStream_t st) {
    ConvGemm p = p_in;
    MS_REQUIRE(p.x.n == p.y.n, "conv_gemm: batch mismatch");
    {
        static int small_env = -1;
        if (small_env < 0) { const char* e = getenv("MS_CONV_SMALL"); small_env = (e && e[0] == '0') ? 0 : 1; }
        if (small_env && conv_small_fwd_supported(p)) return conv_small_fwd(p, st);     // cin = 3 (conv_small.cu)
    }
    const size_t Mz = (size_t)p.y.n * p.y.h * p.y.w;
    MS_REQUIRE(Mz < (1u << 30), "conv_gemm: too many output pixels");
    const int M = (int)Mz;
    const bool avec = (p.x.cs % 4 == 0) && aligned16(p.x.p) && p.x.c >= 4;
    const bool bvec = (p.y.c % 4 == 0) && aligned16(p.wmat);
    const int tn = p.y.c > 32 ? 4 : (p.y.c > 16 ? 2 : 1);
    dim3 grid(cdiv(M, 128), cdiv(p.y.c, 16 * tn));
    // few CTAs walking a long K loop (coarse pyramid levels, heads): split K across CTAs, reduce afterwards
    p.ksplit = 1;
    {
        const int ctas = grid.x * grid.y, total_k = p.kh * p.kw * cdiv(p.x.c, BK);
        if (p.part && ctas <= 74 && total_k >= 8) {
            int ks = std::min(total_k / 4, std::max(1, 296 / ctas));
            if (ks > 32) ks = 32;
            if (ks > 1 && (size_t)ks * M * p.y.c <= p.part_floats) { p.ksplit = ks; grid.z = ks; }
        }
    }
#define LAUNCH(TN_, AV_, BV_) conv_gemm_kernel<TN_, AV_, BV_><<<grid, NT, 0, st>>>(p, M)
#define DISPATCH_B(TN_, AV_) do { if (bvec) LAUNCH(TN_, AV_, true); else LAUNCH(TN_, AV_, false); } while (0)
#define DISPATCH_A(TN_) do { if (avec) DISPATCH_B(TN_, true); else DISPATCH_B(TN_, false); } while (0)
    if (tn == 4) DISPATCH_A(4); else if (tn == 2) DISPATCH_A(2); else DISPATCH_A(1);
#undef LAUNCH
#undef DISPATCH_A
#undef DISPATCH_B
    if (p.ksplit > 1) {
        gemm_splitk_reduce_kernel<<<(unsigned)cdivz((size_t)M * p.y.c, 256), 256, 0, st>>>(p, M);
        return check_launch("conv_gemm+reduce", 2);
    }
    return check_launch("conv_gemm");
}

// ---------------------------------------------------------------------------------------------
// weight gradient: per tap, dW[ci][co] = sum_pixels X[gather(p,tap)][ci] * dY[p][co]
// grid.x = taps * mtiles * ntiles, grid.y = split ; partials -> workspace, then wgrad_reduce.
// ---------------------------------------------------------------------------------------------
template <int TM, int TN, bool AVEC, bool BVEC>
__global__ void __launch_bounds__(NT) conv_wgrad_kernel(ConvWgrad p, int P, int chunk, int mtiles, int ntiles,
                                                        float* __restrict__ partial) {
    constexpr int BM = 16 * TM, BN = 16 * TN, LDA = BM, LDB = BN;
    __shared__ __align__(16) float As[2][BK * LDA];
    __shared__ __align__(16) float Bs[2][BK * LDB];
    const int t = threadIdx.x;
    int bx = blockIdx.x;
    const int nt_ = bx % ntiles; bx /= ntiles;
    const int mt_ = bx % mtiles;
    const int tap = bx / mtiles;
    const int r = tap / p.kw, s = tap - r * p.kw;
    const int m0 = mt_ * BM, n0 = nt_ * BN;
    const int ci = p.x.c, co = p.dy.c;
    const int p_begin = blockIdx.y * chunk;
    const int p_end = min(P, p_begin + chunk);
    const int iters = (p_end > p_begin) ? (p_end - p_begin + BK - 1) / BK : 0;

    constexpr int AF4 = (BK * BM / 4 + NT - 1) / NT;   // float4 loads per thread (vector path)
    constexpr int BF4 = (BK * BN / 4 + NT - 1) / NT;
    constexpr int ANV = AVEC ? AF4 : TM;   // loads per thread
    constexpr int BNV = BVEC ? BF4 : TN;
    float areg[AVEC ? 4 * AF4 : TM];
    float breg[BVEC ? 4 * BF4 : TN];

    auto load_tiles = [&](int pbase) {
        // ---- A: rows = pixels, cols = ci
#pragma unroll
        for (int j = 0; j < ANV; ++j) {
            int k, m;
            bool act;
            if (AVEC) { constexpr int F4 = BM / 4; int e = t + NT * j; act = e < BK * F4; k = e / F4; m = (e % F4) * 4; }
            else { int e = t + NT * j; act = true; k = e / BM; m = e % BM; }
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            int pp = pbase + k;
            if (act && pp < p_end && m0 + m < ci) {
                int ox = pp % p.dy.w;
                int q = pp / p.dy.w;
                int oy = q % p.dy.h;
                int img = q / p.dy.h;
                int iy = oy * p.stride - p.pad_t + r * p.dil;
                int ix = ox * p.stride - p.pad_l + s * p.dil;
                if (iy >= 0 && iy < p.x.h && ix >= 0 && ix < p.x.w) {
                    const float* src = p.x.p + ((size_t)(img * p.x.h + iy) * p.x.w + ix) * p.x.cs + m0 + m;
                    if (AVEC) {
                        v = *reinterpret_cast<const float4*>(src);
                        if (m0 + m + 1 >= ci) v.y = 0.f;
                        if (m0 + m + 2 >= ci) v.z = 0.f;
                        if (m0 + m + 3 >= ci) v.w = 0.f;
                    } else {
                        v.x = *src;
                    }
                }
            }
            if (AVEC) { areg[4 * j] = v.x; areg[4 * j + 1] = v.y; areg[4 * j + 2] = v.z; areg[4 * j + 3] = v.w; }
            else areg[j] = v.x;
        }
        // ---- B: rows = pixels, cols = co
#pragma unroll
        for (int j = 0; j < BNV; ++j) {
            int k, n;
            bool act;
            if (BVEC) { constexpr int F4 = BN / 4; int e = t + NT * j; act = e < BK * F4; k = e / F4; n = (e % F4) * 4; }
            else { int e = t + NT * j; act = true; k = e / BN; n = e % BN; }
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            int pp = pbase + k;
            if (act && pp < p_end && n0 + n < co) {
                const float* src = p.dy.p + (size_t)pp * p.dy.cs + n0 + n;
                if (BVEC) {
                    v = *reinterpret_cast<const float4*>(src);
                    if (n0 + n + 1 >= co) v.y = 0.f;
                    if (n0 + n + 2 >= co) v.z = 0.f;
                    if (n0 + n + 3 >= co) v.w = 0.f;
                } else {
                    v.x = *src;
                }
            }
            if (BVEC) { breg[4 * j] = v.x; breg[4 * j + 1] = v.y; breg[4 * j + 2] = v.z; breg[4 * j + 3] = v.w; }
            else breg[j] = v.x;
        }
    };
    auto store_tiles = [&](int buf) {
        float* as = As[buf];
        float* bs = Bs[buf];
        if (AVEC) {
            constexpr int F4 = BM / 4;
#pragma unroll
            for (int j = 0; j < AF4; ++j) {
                int e = t + NT * j;
                if (e < BK * F4)
                    *reinterpret_cast<float4*>(&as[(e / F4) * LDA + (e % F4) * 4]) =
                        make_float4(areg[4 * j], areg[4 * j + 1], areg[4 * j + 2], areg[4 * j + 3]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < TM; ++j) { int e = t + NT * j; as[(e / BM) * LDA + e % BM] = areg[j]; }
        }
        if (BVEC) {
            constexpr int F4 = BN / 4;
#pragma unroll
            for (int j = 0; j < BF4; ++j) {
                int e = t + NT * j;
                if (e < BK * F4)
                    *reinterpret_cast<float4*>(&bs[(e / F4) * LDB + (e % F4) * 4]) =
                        make_float4(breg[4 * j], breg[4 * j + 1], breg[4 * j + 2], breg[4 * j + 3]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < TN; ++j) { int e = t + NT * j; bs[(e / BN) * LDB + e % BN] = breg[j]; }
        }
    };

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    const int tm = t >> 4, tn = t & 15;

    if (iters > 0) {
        load_tiles(p_begin);
        store_tiles(0);
        __syncthreads();
        for (int it = 0; it < iters; ++it) {
            const int buf = it & 1;
            const bool more = it + 1 < iters;
            if (more) load_tiles(p_begin + (it + 1) * BK);
            mma_tile<TM, TN, LDA, LDB>(As[buf], Bs[buf], tm, tn, acc);
            if (more) store_tiles(buf ^ 1);
            __syncthreads();
        }
    }
    float* dst = partial + ((size_t)blockIdx.y * p.kh * p.kw + tap) * ci * co;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int m = m0 + tm * TM + i;
        if (m >= ci) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int n = n0 + tn * TN + j;
            if (n < co) dst[(size_t)m * co + n] = acc[i][j];
        }
    }
}

__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, size_t n,
                                    int split, int accumulate) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = accumulate ? dw[i] : 0.f;
    for (int k = 0; k < split; ++k) s += partial[(size_t)k * n + i];
    dw[i] = s;
}

// bias gradient partials: block (32 cols x 8 rows) over a pixel range
__global__ void bias_partial_kernel(const float* __restrict__ dy, int cs, int co, int P, int chunk,
                                    float* __restrict__ partial) {
    __shared__ float sm[8][33];
    const int cx = threadIdx.x, ry = threadIdx.y;
    const int n = blockIdx.x * 32 + cx;
    const int pb = blockIdx.y * chunk, pe = min(P, pb + chunk);
    float s = 0.f;
    if (n < co)
        for (int pp = pb + ry; pp < pe; pp += 8) s += dy[(size_t)pp * cs + n];
    sm[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && n < co) {
        float tot = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) tot += sm[k][cx];
        partial[(size_t)blockIdx.y * co + n] = tot;
    }
}

static int wgrad_split(int tiles, size_t P) {
    int split = cdiv(592, tiles);
    int maxs = (int)std::max<size_t>(1, P / 128);
    if (split > maxs) split = maxs;
    if (split > 96) split = 96;
    if (split < 1) split = 1;
    return split;
}
static void wgrad_tiles(int ci, int co, int& tm, int& tn) {
    // 8x8 thread tiles (128x128 CTA tiles) were measured slower than 4x4 here (fewer resident CTAs per SM)
    tm = ci > 32 ? 4 : (ci > 16 ? 2 : 1);
    tn = co > 32 ? 4 : (co > 16 ? 2 : 1);
}
static int bias_blocks(size_t P) { return (int)std::min<size_t>(128, std::max<size_t>(1, P / 256)); }

size_t conv_wgrad_workspace_floats(int taps, int ci, int co, size_t P) {
    int tm, tn; wgrad_tiles(ci, co, tm, tn);
    int tiles = taps * cdiv(ci, 16 * tm) * cdiv(co, 16 * tn);
    size_t main_part = (size_t)wgrad_split(tiles, P) * taps * ci * co;
    if (conv_small_wgrad_shape(taps, ci, co)) main_part = std::max(main_part, conv_small_wgrad_workspace_floats(taps, ci, co, P));
    if (co == 1) main_part = std::max(main_part, (size_t)2 * 148 * ((size_t)taps * ci + 1));      // conv_head_wgrad partials
    return main_part + (size_t)bias_blocks(P) * co + 64;
}

int conv_wgrad(const ConvWgrad& p, cudaStream_t st) {
    MS_REQUIRE(p.x.n == p.dy.n, "conv_wgrad: batch mismatch");
    const size_t Pz = (size_t)p.dy.n * p.dy.h * p.dy.w;
    MS_REQUIRE(Pz < (1u << 30), "conv_wgrad: too many pixels");
    const int P = (int)Pz;
    const int taps = p.kh * p.kw, ci = p.x.c, co = p.dy.c;
    {   // single output channel (disparity heads): dedicated reduction kernel, conv_head.cu
        static int heads = -1;
        if (heads < 0) { const char* e = getenv("MS_HEADS"); heads = (e && e[0] == '0') ? 0 : 1; }
        if (heads && conv_head_wgrad_supported(p) && p.workspace_floats >= conv_head_wgrad_workspace_floats(p)) return conv_head_wgrad(p, st);
    }
    int tm, tn; wgrad_tiles(ci, co, tm, tn);
    const int mtiles = cdiv(ci, 16 * tm), ntiles = cdiv(co, 16 * tn);
    const size_t wn = (size_t)taps * ci * co;
    const int nb = bias_blocks(Pz);
    static int small_env = -1;
    if (small_env < 0) { const char* e = getenv("MS_CONV_SMALL"); small_env = (e && e[0] == '0') ? 0 : 1; }
    const bool small = small_env && conv_small_wgrad_supported(p) &&
                       p.workspace_floats >= conv_small_wgrad_workspace_floats(taps, ci, co, Pz) + (size_t)nb * co;
    int split = wgrad_split(taps * mtiles * ntiles, Pz);
    int chunk = cdiv(P, split);
    chunk = cdiv(chunk, BK) * BK;
    if (small) {                                          // tiny channel counts: register-resident direct kernel (conv_small.cu)
        if (conv_small_wgrad(p, &split, st)) return -1;
    } else {
    MS_REQUIRE(p.workspace_floats >= (size_t)split * wn + (size_t)nb * co, "conv_wgrad: workspace too small");
    const bool avec = (p.x.cs % 4 == 0) && aligned16(p.x.p) && ci >= 4;
    const bool bvec = (p.dy.cs % 4 == 0) && aligned16(p.dy.p) && co >= 4;
    dim3 grid(taps * mtiles * ntiles, split);
#define L(TM_, TN_, AV_, BV_) conv_wgrad_kernel<TM_, TN_, AV_, BV_><<<grid, NT, 0, st>>>(p, P, chunk, mtiles, ntiles, p.workspace)
#define DB(TM_, TN_, AV_) do { if (bvec) L(TM_, TN_, AV_, true); else L(TM_, TN_, AV_, false); } while (0)
#define DA(TM_, TN_) do { if (avec) DB(TM_, TN_, true); else DB(TM_, TN_, false); } while (0)
#define DN(TM_) do { if (tn == 8) DA(TM_, 8); else if (tn == 4) DA(TM_, 4); else if (tn == 2) DA(TM_, 2); else DA(TM_, 1); } while (0)
    if (tm == 8) DN(8); else if (tm == 4) DN(4); else if (tm == 2) DN(2); else DN(1);
#undef L
#undef DB
#undef DA
#undef DN
    if (check_launch("conv_wgrad", 1)) return -1;
    }
    wgrad_reduce_kernel<<<(unsigned)cdivz(wn, 256), 256, 0, st>>>(p.workspace, p.dw, wn, split, p.accumulate);
    if (p.db) {
        float* bp = p.workspace + (size_t)split * wn;
        int bchunk = cdiv(P, nb);
        bias_partial_kernel<<<dim3(cdiv(co, 32), nb), dim3(32, 8), 0, st>>>(p.dy.p, p.dy.cs, co, P, bchunk, bp);
        wgrad_reduce_kernel<<<cdiv(co, 256), 256, 0, st>>>(bp, p.db, (size_t)co, nb, p.accumulate);
    }
    return check_launch("conv_wgrad_reduce", p.db ? 3 : 1);
}

int bias_grad(const TView& dy, float* db, float* workspace, size_t workspace_floats, cudaStream_t st) {
    const size_t Pz = dy.pixels();
    const int P = (int)Pz, co = dy.c, nb = bias_blocks(Pz);
    MS_REQUIRE(workspace_floats >= (size_t)nb * co, "bias_grad: workspace too small");
    bias_partial_kernel<<<dim3(cdiv(co, 32), nb), dim3(32, 8), 0, st>>>(dy.p, dy.cs, co, P, cdiv(P, nb), workspace);
    wgrad_reduce_kernel<<<cdiv(co, 256), 256, 0, st>>>(workspace, db, (size_t)co, nb, 0);
    return check_launch("bias_grad", 2);
}

// wt[tap][co][ci] = w[tap][ci][co]
__global__ void transpose_taps_kernel(const float* __restrict__ w, float* __restrict__ wt, int ci, int co) {
    __shared__ float tile[32][33];
    const int tap = blockIdx.z;
    const float* src = w + (size_t)tap * ci * co;
    float* dst = wt + (size_t)tap * ci * co;
    int c = blockIdx.x * 32 + threadIdx.x;   // co index
    for (int j = threadIdx.y; j < 32; j += 8) {
        int r = blockIdx.y * 32 + j;         // ci index
        tile[j][threadIdx.x] = (r < ci && c < co) ? src[(size_t)r * co + c] : 0.f;
    }
    __syncthreads();
    int r2 = blockIdx.y * 32 + threadIdx.x;  // ci index (fast)
    for (int j = threadIdx.y; j < 32; j += 8) {
        int c2 = blockIdx.x * 32 + j;        // co index
        if (r2 < ci && c2 < co) dst[(size_t)c2 * ci + r2] = tile[threadIdx.x][j];
    }
}

int transpose_taps(const float* w, float* wt, int taps, int ci, int co, cudaStream_t st) {
    transpose_taps_kernel<<<dim3(cdiv(co, 32), cdiv(ci, 32), taps), dim3(32, 8), 0, st>>>(w, wt, ci, co);
    return check_launch("transpose_taps");
}

}  // namespace ms
