// Horizontal correlation cost volume, fused with the MADNet linear warp and the cost-volume concat.
//
// Replaces sharedLayers.correlation / correlation_tf (reference Nets/sharedLayers.py:23-51), the native
// ShiftCorr op it can optionally call (Nets/Native/shift_corr.cu.cc:17-70,193-233 forward;
// :73-191,235-289 backward -- whose backward is defective, see DESIGN.md, so the *mathematical* gradient
// of correlation_tf is implemented), MadNet._linear_warping (Nets/MadNet.py:400-436) and
// MadNet._stereo_cost_volume_correlation's tf.concat (Nets/MadNet.py:370-375).
//
//   corr[b,y,x,i] = (1/C) * sum_c L[b,y,x,c] * RW[b,y,x+d_i,c],   d_i = -max_disp + i*stride, 0 outside
//   RW[x'] = wt0*R[x0s] + wt1*R[x1s]  with cx = x'+u[x'], x0=floor(cx), taps outside [0,w-1] weight 0
//
// One CTA owns one image row segment; the left/right feature rows are staged into shared memory with
// 1-D TMA bulk copies (cp.async.bulk + mbarrier); 8 lanes share a pixel (float4 channel chunks) and
// reduce the displacement sums with warp shuffles; results go out as 128-bit stores straight into the
// concat buffer the first estimator conv reads.  No tensor cores: it is a shifted inner product.
#include "common.cuh"
#include "corr_common.cuh"
#include <algorithm>
#include <cstdlib>

namespace ms {

// ---- PTX helpers (mbarrier + bulk async copy) ------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    const uint32_t a = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!ok);
}

// stage the contiguous feature row segment [wlo,whi) x C of one image row into smem
__device__ __forceinline__ void stage_row(float* dst, const float* src_row, int cs, int C, int wlo, int whi,
                                          bool use_tma, uint64_t* bar) {
    const int npx = whi - wlo;
    if (use_tma) {
        if (threadIdx.x == 0) {
            uint32_t bytes = (uint32_t)npx * C * 4u;
            uint32_t off = 0;
            while (off < bytes) {   // <=32 KB pieces keep each bulk request modest
                uint32_t n = min(bytes - off, 32768u);
                bulk_g2s(reinterpret_cast<char*>(dst) + off,
                         reinterpret_cast<const char*>(src_row + (size_t)wlo * cs) + off, n, bar);
                off += n;
            }
        }
    } else {
        const int nvec = C / 4;
        for (int e = threadIdx.x; e < npx * nvec; e += blockDim.x) {
            int px = e / nvec, q = e - px * nvec;
            reinterpret_cast<float4*>(dst)[e] =
                *reinterpret_cast<const float4*>(src_row + (size_t)(wlo + px) * cs + q * 4);
        }
    }
}

constexpr int CORR_NT = 256;
constexpr int LPP = 8;  // lanes per pixel

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CORR_NT) corr_fwd_kernel(CorrFwd p, int TW, int nd, int use_tma) {
    pdl_prologue();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    const int C = p.C, w = p.w, d = p.max_disp;
    const bool warped = p.u != nullptr;
    const int row = blockIdx.y;                 // b*h + y
    const int x0 = blockIdx.x * TW, x1 = min(w, x0 + TW);
    const int rlo = warped ? 0 : max(0, x0 - d), rhi = warped ? w : min(w, x1 + d);
    float* Ls = reinterpret_cast<float*>(smem_raw);                 // [TW][C]
    float* Rs = Ls + (size_t)TW * C;                                  // [rhi-rlo][C]
    float* Us = Rs + (size_t)(warped ? w : (TW + 2 * d)) * C;        // [w] (warped only)

    const float* lrow = p.left + (size_t)row * w * p.lcs;
    const float* rrow = p.right + (size_t)row * w * p.rcs;

    if (use_tma && threadIdx.x == 0) { mbar_init(&bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (use_tma && threadIdx.x == 0) mbar_expect_tx(&bar, (uint32_t)((x1 - x0) + (rhi - rlo)) * C * 4u);
    stage_row(Ls, lrow, p.lcs, C, x0, x1, use_tma, &bar);
    stage_row(Rs, rrow, p.rcs, C, rlo, rhi, use_tma, &bar);
    if (warped)
        for (int e = threadIdx.x; e < w; e += blockDim.x) Us[e] = p.u[((size_t)row * w + e) * p.ucs];
    __syncthreads();
    if (use_tma) mbar_wait(&bar, 0);

    const int lane = threadIdx.x & 31, sub = lane & (LPP - 1);
    const int grp = threadIdx.x / LPP, ngrp = CORR_NT / LPP;
    const int nchunk = C / 4;
    const float invC = 1.f / (float)C;
    float* orow = p.out + (size_t)row * w * p.ocs;
    float* o2row = p.out2 ? p.out2 + (size_t)row * w * p.o2cs : nullptr;
    const int coff = p.copy_left ? C : 0;
    const int tail0 = coff + nd + p.u_chan;            // first pad channel (the u channel is left untouched)

    for (int xb = x0; xb < x1; xb += ngrp) {   // uniform trip count: every lane reaches the shuffles
        const bool act = xb + grp < x1;
        const int x = act ? xb + grp : x0;       // x is uniform across the 8 lanes of a group
        const float4* L4 = reinterpret_cast<const float4*>(Ls + (size_t)(x - x0) * C);
        // copy of the left features into the concat buffer(s)
        if (p.copy_left && act) {
            for (int q = sub; q < nchunk; q += LPP) {
                float4 v = L4[q];
                *reinterpret_cast<float4*>(orow + (size_t)x * p.ocs + q * 4) = v;
                if (o2row) *reinterpret_cast<float4*>(o2row + (size_t)x * p.o2cs + q * 4) = v;
            }
        }
        for (int i = 0; i < nd; ++i) {
            const int xp = x + (-d + i * p.stride);
            float s = 0.f;
            if (act && xp >= 0 && xp < w) {
                WarpTap t = warp_tap(xp, warped ? Us[xp] : 0.f, w, warped);
                const float4* R0 = reinterpret_cast<const float4*>(Rs + (size_t)(t.i0 - rlo) * C);
                const float4* R1 = reinterpret_cast<const float4*>(Rs + (size_t)(t.i1 - rlo) * C);
                for (int q = sub; q < nchunk; q += LPP) {
                    float4 l = L4[q], a = R0[q];
                    if (warped) {
                        float4 b = R1[q];
                        a.x = t.w0 * a.x + t.w1 * b.x; a.y = t.w0 * a.y + t.w1 * b.y;
                        a.z = t.w0 * a.z + t.w1 * b.z; a.w = t.w0 * a.w + t.w1 * b.w;
                    }
                    s = fmaf(l.x, a.x, s); s = fmaf(l.y, a.y, s); s = fmaf(l.z, a.z, s); s = fmaf(l.w, a.w, s);
                }
            }
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            if (act && sub == (i & (LPP - 1))) orow[(size_t)x * p.ocs + coff + i] = s * invC;
        }
        if (act && sub == 0 && p.copy_left)
            for (int c = tail0; c < p.ocs; ++c) orow[(size_t)x * p.ocs + c] = 0.f;
    }
}

// ---------------------------------------------------------------------------------------------
// forward v2: small x-tiles (many CTAs per SM so loads / math / stores of different tiles overlap), warp taps
// computed once per column, the warped right row RW materialised once per tile in shared memory (each RW column feeds
// nd output columns), and a BOUNDED right-feature window staged by TMA: the window is sized from the actual taps of
// the tile; taps that fall outside the cap (pathological disparities) are read straight from global memory.
// ---------------------------------------------------------------------------------------------
template <int ND_CT>
__global__ void __launch_bounds__(CORR_NT) corr_fwd2_kernel(CorrFwd p, int TW, int RCAP, int nd_rt, int use_tma) {
    pdl_prologue();
    const int nd = ND_CT > 0 ? ND_CT : nd_rt;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ int s_lo, s_hi;
    const int C = p.C, w = p.w, d = p.max_disp;
    const bool warped = p.u != nullptr;
    const int row = blockIdx.y;
    const int x0 = blockIdx.x * TW, x1 = min(w, x0 + TW);
    const int wlo = max(0, x0 - d), whi = min(w, x1 + d);          // RW columns needed: [wlo, whi)
    const int NW = whi - wlo;
    float* Ls = reinterpret_cast<float*>(smem_raw);                  // [TW][C]
    float* RWs = Ls + (size_t)TW * C;                                 // [TW+2d][C]  warped right features
    float* Rs = RWs + (size_t)(TW + 2 * d) * C;                       // [RCAP][C]   raw right window (warped only)
    Tap* taps = reinterpret_cast<Tap*>(Rs + (size_t)(warped ? RCAP : 0) * C);   // [TW+2d]

    const float* lrow = p.left + (size_t)row * w * p.lcs;
    const float* rrow = p.right + (size_t)row * w * p.rcs;
    const float* urow = warped ? p.u + (size_t)row * w * p.ucs : nullptr;

    if (threadIdx.x == 0) { s_lo = w; s_hi = -1; if (use_tma) { mbar_init(&bar, 1); fence_mbar_init(); } }
    __syncthreads();
    // ---- phase 1: taps + the right-feature window they touch
    int rlo = wlo, rhi = whi;                                          // raw window [rlo, rhi)
    if (warped) {
        for (int t = threadIdx.x; t < NW; t += blockDim.x) {
            WarpTap wt = warp_tap(wlo + t, urow[(size_t)(wlo + t) * p.ucs], w, true);
            Tap tp; tp.i0 = wt.i0; tp.i1 = wt.i1; tp.w0 = wt.w0; tp.w1 = wt.w1;
            taps[t] = tp;
            if (wt.w0 != 0.f) { atomicMin(&s_lo, wt.i0); atomicMax(&s_hi, wt.i0); }
            if (wt.w1 != 0.f) { atomicMin(&s_lo, wt.i1); atomicMax(&s_hi, wt.i1); }
        }
        __syncthreads();
        rlo = s_lo; rhi = s_hi + 1;
        if (rhi <= rlo) { rlo = 0; rhi = 0; }
        if (rhi - rlo > RCAP) rhi = rlo + RCAP;                        // the rest goes through the global slow path
    }
    // ---- phase 2: stage L tile and the right window
    const uint32_t lbytes = (uint32_t)(x1 - x0) * C * 4u, rbytes = (uint32_t)(rhi - rlo) * C * 4u;
    float* rdst = warped ? Rs : RWs;
    if (use_tma && threadIdx.x == 0) mbar_expect_tx(&bar, lbytes + rbytes);
    stage_row(Ls, lrow, p.lcs, C, x0, x1, use_tma, &bar);
    if (rhi > rlo) stage_row(rdst, rrow, p.rcs, C, rlo, rhi, use_tma, &bar);
    __syncthreads();
    if (use_tma) mbar_wait(&bar, 0);

    const int lane = threadIdx.x & 31, sub = lane & (LPP - 1);
    const int grp = threadIdx.x / LPP, ngrp = CORR_NT / LPP;
    const int nchunk = C / 4;
    // ---- phase 3: RW[t] = w0*R[i0] + w1*R[i1]
    if (warped) {
        for (int t = grp; t < NW; t += ngrp) {
            const Tap tp = taps[t];
            const bool in0 = tp.i0 >= rlo && tp.i0 < rhi, in1 = tp.i1 >= rlo && tp.i1 < rhi;
            const float4* R0 = in0 ? reinterpret_cast<const float4*>(Rs + (size_t)(tp.i0 - rlo) * C)
                                   : reinterpret_cast<const float4*>(rrow + (size_t)tp.i0 * p.rcs);
            const float4* R1 = in1 ? reinterpret_cast<const float4*>(Rs + (size_t)(tp.i1 - rlo) * C)
                                   : reinterpret_cast<const float4*>(rrow + (size_t)tp.i1 * p.rcs);
            float4* dst = reinterpret_cast<float4*>(RWs + (size_t)t * C);
            for (int q = sub; q < nchunk; q += LPP) {
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (tp.w0 != 0.f) a = R0[q];
                if (tp.w1 != 0.f) b = R1[q];
                a.x = tp.w0 * a.x + tp.w1 * b.x; a.y = tp.w0 * a.y + tp.w1 * b.y;
                a.z = tp.w0 * a.z + tp.w1 * b.z; a.w = tp.w0 * a.w + tp.w1 * b.w;
                dst[q] = a;
            }
        }
        __syncthreads();
    }
    const int rwbase = warped ? wlo : rlo;                              // column held by RWs[0]
    const float invC = 1.f / (float)C;
    float* orow = p.out + (size_t)row * w * p.ocs;
    float* o2row = p.out2 ? p.out2 + (size_t)row * w * p.o2cs : nullptr;
    const int coff = p.copy_left ? C : 0;
    const int tail0 = coff + nd + p.u_chan;
    // ---- phase 5 (first, coalesced): left copy into the concat buffer(s)
    if (p.copy_left) {
        const int nvec = C / 4;
        for (int e = threadIdx.x; e < (x1 - x0) * nvec; e += blockDim.x) {
            const int px = e / nvec, q = e - px * nvec;
            const float4 v = reinterpret_cast<const float4*>(Ls)[e];
            *reinterpret_cast<float4*>(orow + (size_t)(x0 + px) * p.ocs + q * 4) = v;
            if (o2row) *reinterpret_cast<float4*>(o2row + (size_t)(x0 + px) * p.o2cs + q * 4) = v;
        }
    }
    // ---- phase 4: correlation
    const bool pack8 = p.copy_left && nd == 5 && (p.ocs & 3) == 0 && (coff & 3) == 0 && tail0 + (p.u_chan ? 0 : 0) <= coff + 8 &&
                       p.ocs >= coff + 8;
    for (int xb = x0; xb < x1; xb += ngrp) {
        const bool act = xb + grp < x1;
        const int x = act ? xb + grp : x0;
        const float4* L4 = reinterpret_cast<const float4*>(Ls + (size_t)(x - x0) * C);
        float keep0 = 0.f, keep1 = 0.f, keep2 = 0.f, keep3 = 0.f, keep4 = 0.f;
#pragma unroll
        for (int i = 0; i < nd; ++i) {
            const int xp = x + (-d + i * p.stride);
            float s = 0.f;
            if (act && xp >= 0 && xp < w) {
                const float4* R4 = reinterpret_cast<const float4*>(RWs + (size_t)(xp - rwbase) * C);
                for (int q = sub; q < nchunk; q += LPP) {
                    const float4 l = L4[q], a = R4[q];
                    s = fmaf(l.x, a.x, s); s = fmaf(l.y, a.y, s); s = fmaf(l.z, a.z, s); s = fmaf(l.w, a.w, s);
                }
            }
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s *= invC;
            if (pack8) {
                if (i == 0) keep0 = s; else if (i == 1) keep1 = s; else if (i == 2) keep2 = s; else if (i == 3) keep3 = s; else keep4 = s;
            } else if (act && sub == (i & (LPP - 1))) {
                orow[(size_t)x * p.ocs + coff + i] = s;
            }
        }
        if (act && pack8) {           // [c0 c1 c2 c3][c4 u 0 0] as two 128-bit stores
            float* o = orow + (size_t)x * p.ocs + coff;
            if (sub == 0) *reinterpret_cast<float4*>(o) = make_float4(keep0, keep1, keep2, keep3);
            if (sub == 1) {
                const float uu = p.u_chan ? o[5] : 0.f;                 // the u channel was written by the resize kernel
                *reinterpret_cast<float4*>(o + 4) = make_float4(keep4, uu, 0.f, 0.f);
            }
        } else if (act && sub == 0 && p.copy_left) {
            for (int c = tail0; c < p.ocs; ++c) orow[(size_t)x * p.ocs + c] = 0.f;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward v3: ncu on v2 (profiles/r1_ncu_corr_fwd2_L2_1920x1088_B8.txt) showed the kernel instruction-issue bound
// (155 M warp instructions for 1.04 M pixels, 66 % issue-active, DRAM 16 %): with 8 lanes per pixel every lane owns a
// single float4 chunk, so address arithmetic and the shuffle reductions dominate.  Here LP = 1..8 lanes share a pixel
// and each lane owns CPL >= 3 consecutive chunks; the left chunk is held in registers across the nd displacements;
// shared-memory tiles are stored with an XOR swizzle of the chunk index (low 3 bits ^ column&7) so that lane=column
// accesses are bank-conflict free.  Tiles are staged with coalesced 128-bit loads (the swizzle rules out the 1-D bulk
// copy used by v1/v2, which remain available: MS_CORR_V=1|2).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int swz_m(int q, int col, int m) { return (q & ~m) | ((q ^ col) & m); }

template <int ND_CT>
__global__ void __launch_bounds__(CORR_NT) corr_fwd3_kernel(CorrFwd p, int TW, int LP, int RCAP, int nd_rt, int smask) {
    pdl_prologue();
    auto swz = [smask](int q, int col) { return swz_m(q, col, smask); };
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_lo, s_hi;
    const int nd = ND_CT > 0 ? ND_CT : nd_rt;
    const int C = p.C, w = p.w, d = p.max_disp;
    const bool warped = p.u != nullptr;
    const int row = blockIdx.y;
    const int x0 = blockIdx.x * TW, x1 = min(w, x0 + TW);
    const int wlo = max(0, x0 - d), whi = min(w, x1 + d);
    const int NW = whi - wlo;
    const int nchunk = C / 4, CPL = nchunk / LP;
    float4* Ls = reinterpret_cast<float4*>(smem_raw);                        // [TW][nchunk]       swizzled by local column
    float4* RWs = Ls + (size_t)TW * nchunk;                                   // [TW+2d][nchunk]    swizzled by (column - wlo)
    float4* Rs = RWs + (size_t)(TW + 2 * d) * nchunk;                         // [RCAP][nchunk]     swizzled by (column - rlo)
    Tap* taps = reinterpret_cast<Tap*>(Rs + (size_t)(warped ? RCAP : 0) * nchunk);

    const float* lrow = p.left + (size_t)row * w * p.lcs;
    const float* rrow = p.right + (size_t)row * w * p.rcs;
    const float* urow = warped ? p.u + (size_t)row * w * p.ucs : nullptr;
    float* orow = p.out + (size_t)row * w * p.ocs;
    float* o2row = p.out2 ? p.out2 + (size_t)row * w * p.o2cs : nullptr;

    if (threadIdx.x == 0) { s_lo = w; s_hi = -1; }
    __syncthreads();
    int rlo = wlo, rhi = whi;
    if (warped) {
        for (int t = threadIdx.x; t < NW; t += blockDim.x) {
            WarpTap wt = warp_tap(wlo + t, urow[(size_t)(wlo + t) * p.ucs], w, true);
            Tap tp; tp.i0 = wt.i0; tp.i1 = wt.i1; tp.w0 = wt.w0; tp.w1 = wt.w1;
            taps[t] = tp;
            if (wt.w0 != 0.f) { atomicMin(&s_lo, wt.i0); atomicMax(&s_hi, wt.i0); }
            if (wt.w1 != 0.f) { atomicMin(&s_lo, wt.i1); atomicMax(&s_hi, wt.i1); }
        }
    }
    // ---- left tile: global -> (concat buffers) + swizzled smem
    for (int e = threadIdx.x; e < (x1 - x0) * nchunk; e += blockDim.x) {
        const int j = e / nchunk, q = e - j * nchunk;
        const float4 v = *reinterpret_cast<const float4*>(lrow + (size_t)(x0 + j) * p.lcs + q * 4);
        Ls[(size_t)j * nchunk + swz(q, j)] = v;
        if (p.copy_left) {
            *reinterpret_cast<float4*>(orow + (size_t)(x0 + j) * p.ocs + q * 4) = v;
            if (o2row) *reinterpret_cast<float4*>(o2row + (size_t)(x0 + j) * p.o2cs + q * 4) = v;
        }
    }
    __syncthreads();
    if (warped) {
        rlo = s_lo; rhi = s_hi + 1;
        if (rhi <= rlo) { rlo = 0; rhi = 0; }
        if (rhi - rlo > RCAP) rhi = rlo + RCAP;
    }
    // ---- right window: raw (warped) or final (unwarped) tile
    {
        float4* dst = warped ? Rs : RWs;
        for (int e = threadIdx.x; e < (rhi - rlo) * nchunk; e += blockDim.x) {
            const int j = e / nchunk, q = e - j * nchunk;
            dst[(size_t)j * nchunk + swz(q, j)] = *reinterpret_cast<const float4*>(rrow + (size_t)(rlo + j) * p.rcs + q * 4);
        }
    }
    __syncthreads();
    const int sub = threadIdx.x % LP, pl = threadIdx.x / LP, npl = CORR_NT / LP;   // lane-in-pixel, pixel slot
    if (warped) {
        for (int t = pl; t < NW; t += npl) {
            const Tap tp = taps[t];
            const int r0 = tp.i0 - rlo, r1 = tp.i1 - rlo;
            const bool in0 = r0 >= 0 && tp.i0 < rhi, in1 = r1 >= 0 && tp.i1 < rhi;
#pragma unroll 2
            for (int e = 0; e < CPL; ++e) {
                const int q = sub * CPL + e;
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (tp.w0 != 0.f) a = in0 ? Rs[(size_t)r0 * nchunk + swz(q, r0)] : *reinterpret_cast<const float4*>(rrow + (size_t)tp.i0 * p.rcs + q * 4);
                if (tp.w1 != 0.f) b = in1 ? Rs[(size_t)r1 * nchunk + swz(q, r1)] : *reinterpret_cast<const float4*>(rrow + (size_t)tp.i1 * p.rcs + q * 4);
                a.x = tp.w0 * a.x + tp.w1 * b.x; a.y = tp.w0 * a.y + tp.w1 * b.y;
                a.z = tp.w0 * a.z + tp.w1 * b.z; a.w = tp.w0 * a.w + tp.w1 * b.w;
                RWs[(size_t)t * nchunk + swz(q, t)] = a;
            }
        }
        __syncthreads();
    }
    const int rwbase = warped ? wlo : rlo;
    const float invC = 1.f / (float)C;
    const int coff = p.copy_left ? C : 0;
    const int tail0 = coff + nd + p.u_chan;
    const bool pack8 = p.copy_left && nd == 5 && (p.ocs & 3) == 0 && (coff & 3) == 0 && p.ocs >= coff + 8;
    constexpr int AB = ND_CT > 0 ? ND_CT : 8;                       // accumulators per pass
    for (int xb = x0; xb < x1; xb += npl) {                        // uniform trip count (shuffles below)
        const bool act = xb + pl < x1;
        const int x = act ? xb + pl : x0;
        const int j = x - x0;
        for (int i0 = 0; i0 < nd; i0 += AB) {
            float acc[AB];
#pragma unroll
            for (int k = 0; k < AB; ++k) acc[k] = 0.f;
            for (int e = 0; e < CPL; ++e) {
                const int q = sub * CPL + e;
                const float4 l = Ls[(size_t)j * nchunk + swz(q, j)];
#pragma unroll
                for (int k = 0; k < AB; ++k) {
                    const int i = i0 + k;
                    const int xp = x + (-d + i * p.stride);
                    if (i < nd && xp >= 0 && xp < w) {
                        const int t = xp - rwbase;
                        const float4 a = RWs[(size_t)t * nchunk + swz(q, t)];
                        acc[k] = fmaf(l.x, a.x, acc[k]); acc[k] = fmaf(l.y, a.y, acc[k]);
                        acc[k] = fmaf(l.z, a.z, acc[k]); acc[k] = fmaf(l.w, a.w, acc[k]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < AB; ++k) {
                for (int o = LP >> 1; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
                acc[k] *= invC;
            }
            if (act && sub == 0) {
                float* o = orow + (size_t)x * p.ocs + coff;
                if (ND_CT == 5 && pack8) {
                    const float uu = p.u_chan ? o[5] : 0.f;
                    *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                    *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4], uu, 0.f, 0.f);
                } else {
#pragma unroll
                    for (int k = 0; k < AB; ++k)
                        if (i0 + k < nd) o[i0 + k] = acc[k];
                }
            }
        }
        if (act && sub == 0 && p.copy_left && !(ND_CT == 5 && pack8))
            for (int c = tail0; c < p.ocs; ++c) orow[(size_t)x * p.ocs + c] = 0.f;
    }
}

static bool corr_use_tma() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MS_CORR_NO_TMA"); v = (e && e[0] == '1') ? 0 : 1; }
    return v == 1;
}
static bool a16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int pick_tw(int w, int C, int d, bool warped, size_t row_bufs_full, size_t budget, size_t extra) {
    // warped: windows are the full row regardless of TW
    const int cands[] = {w, 256, 128, 64, 32, 16, 8};
    for (int tw : cands) {
        if (tw > w) continue;
        size_t win = warped ? (size_t)w : (size_t)(tw + 2 * d);
        size_t bytes = (row_bufs_full * win + (size_t)tw) * C * 4 + extra;
        if (bytes <= budget) return tw;
        if (warped) break;
    }
    return -1;
}

int corr_fwd(const CorrFwd& p, cudaStream_t st) {
    MS_REQUIRE(p.C % 4 == 0 && p.lcs % 4 == 0 && p.rcs % 4 == 0, "corr_fwd: C and strides must be multiples of 4");
    MS_REQUIRE(a16(p.left) && a16(p.right) && a16(p.out), "corr_fwd: pointers must be 16B aligned");
    MS_REQUIRE(!p.copy_left || (p.ocs % 4 == 0), "corr_fwd: concat stride must be a multiple of 4");
    MS_REQUIRE(p.stride >= 1, "corr_fwd: stride");
    const bool warped = p.u != nullptr;
    const int nd = (2 * p.max_disp) / p.stride + 1;
    int tma = corr_use_tma() && p.lcs == p.C && p.rcs == p.C;
    if (corr_init()) return -1;
    static int ver = -1;
    if (ver < 0) { const char* e = getenv("MS_CORR_V"); ver = e ? atoi(e) : 4; }
    if (ver >= 4 && corr_mma_supported(p)) return corr_mma(p, st);      // DispNet: 81 displacements as a banded tensor-core product
    if (ver >= 4) {                                     // MADNet cost volume (d=2, C%32==0): tensor-map TMA kernel, corr_tma.cu
        const int r = corr_fwd4(p, st);
        if (r <= 0) return r;
    }
    if (ver >= 3) {
        const int nchunk = p.C / 4;
        const int LP = nchunk >= 24 ? 8 : (nchunk >= 16 ? 4 : (nchunk >= 8 ? 2 : 1));
        // measured (scripts/corr_bench.py): v3 wins for C<=32 (level 2, which moves most of the bytes), v2 for wider features / nd=81
        if (nchunk % LP == 0 && p.C <= 32 && nd <= 8) {
            const int TW = std::min(p.w, CORR_NT / LP);
            const int RCAP = warped ? TW + 2 * p.max_disp + 32 : 0;
            const size_t smem = ((size_t)TW + (size_t)(TW + 2 * p.max_disp) + (size_t)RCAP) * p.C * 4 +
                                (size_t)(TW + 2 * p.max_disp) * sizeof(Tap) + 64;
            if (smem <= 200 * 1024) {
                dim3 grid(cdiv(p.w, TW), p.B * p.h);
                const int smask = nchunk % 8 == 0 ? 7 : (nchunk % 4 == 0 ? 3 : (nchunk % 2 == 0 ? 1 : 0));
                if (nd == 5) launch_k(corr_fwd3_kernel<5>, dim3(grid), dim3(CORR_NT), smem, st, p, TW, LP, RCAP, nd, smask);
                else launch_k(corr_fwd3_kernel<0>, dim3(grid), dim3(CORR_NT), smem, st, p, TW, LP, RCAP, nd, smask);
                return check_launch("corr_fwd3");
            }
        }
    }
    if (ver >= 2) {
        // tile width: aim at >= 3 CTAs per SM
        static int tw_env = -1, slack_env = -1;
        if (tw_env < 0) { const char* e = getenv("MS_CORR_TW"); tw_env = e ? atoi(e) : 0; const char* f = getenv("MS_CORR_SLACK"); slack_env = f ? atoi(f) : 0; }
        int TW = std::min(p.w, tw_env > 0 ? tw_env : (p.C >= 128 ? 32 : 64));
        const int RCAP = warped ? TW + 2 * p.max_disp + (slack_env > 0 ? slack_env : 64) : 0;
        const size_t smem = ((size_t)TW + (size_t)(TW + 2 * p.max_disp) + (size_t)RCAP) * p.C * 4 +
                            (size_t)(TW + 2 * p.max_disp) * sizeof(Tap) + 64;
        if (smem <= 200 * 1024) {
            dim3 grid(cdiv(p.w, TW), p.B * p.h);
            if (nd == 5) launch_k(corr_fwd2_kernel<5>, dim3(grid), dim3(CORR_NT), smem, st, p, TW, RCAP, nd, tma);
            else launch_k(corr_fwd2_kernel<0>, dim3(grid), dim3(CORR_NT), smem, st, p, TW, RCAP, nd, tma);
            return check_launch("corr_fwd2");
        }
    }
    const size_t budget = 200 * 1024;
    int TW = pick_tw(p.w, p.C, p.max_disp, warped, 1, budget, (size_t)p.w * 4 + 64);
    MS_REQUIRE(TW > 0, "corr_fwd: row does not fit in shared memory");
    size_t smem = ((size_t)TW + (warped ? p.w : TW + 2 * p.max_disp)) * p.C * 4 + (warped ? (size_t)p.w * 4 : 0) + 64;
    dim3 grid(cdiv(p.w, TW), p.B * p.h);
    launch_k(corr_fwd_kernel, dim3(grid), dim3(CORR_NT), smem, st, p, TW, nd, tma);
    return check_launch("corr_fwd");
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CORR_NT) corr_bwd_kernel(CorrBwd p, int TW, int nd, int use_tma) {
    pdl_prologue();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    const int C = p.C, w = p.w, d = p.max_disp;
    const bool warped = p.u != nullptr;
    const int row = blockIdx.y;
    const int x0 = blockIdx.x * TW, x1 = min(w, x0 + TW);
    const int wlo = warped ? 0 : max(0, x0 - d), whi = warped ? w : min(w, x1 + d);
    const int WIN = warped ? w : (TW + 2 * d);
    float* Ls = reinterpret_cast<float*>(smem_raw);   // [WIN][C]   (later: scatter accumulator)
    float* Rs = Ls + (size_t)WIN * C;                   // [WIN][C]
    float* Ds = Rs + (size_t)WIN * C;                   // [TW][C]    d_rw (only when warped)
    float* Gs = Ds + (size_t)(warped ? TW : 0) * C;     // [WIN][nd]  corr grads
    float* Us = Gs + (size_t)WIN * nd;                  // [w]

    const float* lrow = p.left + (size_t)row * w * p.lcs;
    const float* rrow = p.right + (size_t)row * w * p.rcs;
    const float* grow = p.dcost + (size_t)row * w * p.dcs;
    const int gco = p.gcoff < 0 ? C : p.gcoff;

    if (use_tma && threadIdx.x == 0) { mbar_init(&bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (use_tma && threadIdx.x == 0) mbar_expect_tx(&bar, (uint32_t)(2 * (whi - wlo)) * C * 4u);
    stage_row(Ls, lrow, p.lcs, C, wlo, whi, use_tma, &bar);
    stage_row(Rs, rrow, p.rcs, C, wlo, whi, use_tma, &bar);
    for (int e = threadIdx.x; e < (whi - wlo) * nd; e += blockDim.x) {
        int px = e / nd, i = e - px * nd;
        Gs[e] = grow[(size_t)(wlo + px) * p.dcs + gco + i];
    }
    if (warped)
        for (int e = threadIdx.x; e < w; e += blockDim.x) Us[e] = p.u[((size_t)row * w + e) * p.ucs];
    __syncthreads();
    if (use_tma) mbar_wait(&bar, 0);

    const int lane = threadIdx.x & 31, sub = lane & (LPP - 1);
    const int grp = threadIdx.x / LPP, ngrp = CORR_NT / LPP;
    const int nchunk = C / 4;
    const float invC = 1.f / (float)C;
    float* dlrow = p.dleft + (size_t)row * w * p.dlcs;
    float* drrow = p.dright + (size_t)row * w * p.drcs;

    for (int xb = x0; xb < x1; xb += ngrp) {   // uniform trip count (shuffles below)
        const bool act = xb + grp < x1;
        const int x = act ? xb + grp : x0;
        // ---- dL[x,:] = slice + (1/C) sum_i g[x,i] * RW[x+d_i,:]
        for (int q = sub; q < nchunk && act; q += LPP) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < nd; ++i) {
                const int xp = x + (-d + i * p.stride);
                if (xp < 0 || xp >= w) continue;
                const float g = Gs[(size_t)(x - wlo) * nd + i];
                WarpTap t = warp_tap(xp, warped ? Us[xp] : 0.f, w, warped);
                float4 a = reinterpret_cast<const float4*>(Rs + (size_t)(t.i0 - wlo) * C)[q];
                if (warped) {
                    float4 b = reinterpret_cast<const float4*>(Rs + (size_t)(t.i1 - wlo) * C)[q];
                    a.x = t.w0 * a.x + t.w1 * b.x; a.y = t.w0 * a.y + t.w1 * b.y;
                    a.z = t.w0 * a.z + t.w1 * b.z; a.w = t.w0 * a.w + t.w1 * b.w;
                }
                acc.x = fmaf(g, a.x, acc.x); acc.y = fmaf(g, a.y, acc.y);
                acc.z = fmaf(g, a.z, acc.z); acc.w = fmaf(g, a.w, acc.w);
            }
            acc.x *= invC; acc.y *= invC; acc.z *= invC; acc.w *= invC;
            if (p.add_left_slice) {
                float4 sl = *reinterpret_cast<const float4*>(grow + (size_t)x * p.dcs + q * 4);
                acc.x += sl.x; acc.y += sl.y; acc.z += sl.z; acc.w += sl.w;
            }
            float4* dst = reinterpret_cast<float4*>(dlrow + (size_t)x * p.dlcs + q * 4);
            if (p.acc_left) { float4 o = *dst; acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w; }
            *dst = acc;
        }
        // ---- d_rw[x,:] = (1/C) sum_i g[x-d_i, i] * L[x-d_i,:]     (x plays the role of x')
        float du_part = 0.f;
        WarpTap tx_ = warp_tap(x, warped ? Us[x] : 0.f, w, warped);
        for (int q = sub; q < nchunk && act; q += LPP) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < nd; ++i) {
                const int xs = x - (-d + i * p.stride);
                if (xs < 0 || xs >= w) continue;
                const float g = Gs[(size_t)(xs - wlo) * nd + i];
                float4 l = reinterpret_cast<const float4*>(Ls + (size_t)(xs - wlo) * C)[q];
                acc.x = fmaf(g, l.x, acc.x); acc.y = fmaf(g, l.y, acc.y);
                acc.z = fmaf(g, l.z, acc.z); acc.w = fmaf(g, l.w, acc.w);
            }
            acc.x *= invC; acc.y *= invC; acc.z *= invC; acc.w *= invC;
            if (!warped) {
                float4* dst = reinterpret_cast<float4*>(drrow + (size_t)x * p.drcs + q * 4);
                if (p.acc_right) { float4 o = *dst; acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w; }
                *dst = acc;
            } else {
                reinterpret_cast<float4*>(Ds + (size_t)(x - x0) * C)[q] = acc;
                if (p.du) {
                    float4 a = reinterpret_cast<const float4*>(Rs + (size_t)(tx_.i0 - wlo) * C)[q];
                    float4 b = reinterpret_cast<const float4*>(Rs + (size_t)(tx_.i1 - wlo) * C)[q];
                    // d(wt0)/d(cx) = -mask0 ; d(wt1)/d(cx) = +mask1
                    float cx = (float)x + Us[x];
                    float f0 = floorf(cx);
                    float k0 = (f0 >= 0.f && f0 <= (float)(w - 1)) ? -1.f : 0.f;
                    float k1 = (f0 + 1.f >= 0.f && f0 + 1.f <= (float)(w - 1)) ? 1.f : 0.f;
                    du_part += acc.x * (k0 * a.x + k1 * b.x) + acc.y * (k0 * a.y + k1 * b.y) +
                               acc.z * (k0 * a.z + k1 * b.z) + acc.w * (k0 * a.w + k1 * b.w);
                }
            }
        }
        if (warped && p.du) {
            du_part += __shfl_xor_sync(0xffffffffu, du_part, 4);
            du_part += __shfl_xor_sync(0xffffffffu, du_part, 2);
            du_part += __shfl_xor_sync(0xffffffffu, du_part, 1);
            if (act && sub == 0) p.du[((size_t)row * w + x) * p.ducs] = du_part;
        }
    }
    if (!warped) return;

    // ---- deterministic scatter of d_rw through the warp taps: one thread per channel, x' in order
    __syncthreads();
    float* Acc = Ls;   // L no longer needed (warped => TW == w, single tile per row)
    for (int e = threadIdx.x; e < w * C; e += blockDim.x) Acc[e] = 0.f;
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        for (int xp = 0; xp < w; ++xp) {
            WarpTap t = warp_tap(xp, Us[xp], w, true);
            float v = Ds[(size_t)xp * C + c];
            Acc[(size_t)t.i0 * C + c] += t.w0 * v;
            Acc[(size_t)t.i1 * C + c] += t.w1 * v;
        }
    }
    __syncthreads();
    const int nvec = C / 4;
    for (int e = threadIdx.x; e < w * nvec; e += blockDim.x) {
        int px = e / nvec, q = e - px * nvec;
        float4 v = reinterpret_cast<const float4*>(Acc)[e];
        float4* dst = reinterpret_cast<float4*>(drrow + (size_t)px * p.drcs + q * 4);
        if (p.acc_right) { float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
        *dst = v;
    }
}

int corr_init() {
    static bool done = false;
    if (done) return 0;
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd2_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd3_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd3_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    MS_CHECK_CUDA(cudaFuncSetAttribute(corr_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    done = true;
    return 0;
}

int corr_bwd(const CorrBwd& p, cudaStream_t st) {
    MS_REQUIRE(p.C % 4 == 0 && p.lcs % 4 == 0 && p.rcs % 4 == 0 && p.dlcs % 4 == 0 && p.drcs % 4 == 0,
               "corr_bwd: C and strides must be multiples of 4");
    MS_REQUIRE(a16(p.left) && a16(p.right) && a16(p.dleft) && a16(p.dright), "corr_bwd: pointers must be 16B aligned");
    MS_REQUIRE(!p.add_left_slice || (p.dcs % 4 == 0 && a16(p.dcost)), "corr_bwd: dcost slice alignment");
    {
        static int ver = -1;
        if (ver < 0) { const char* e = getenv("MS_CORR_V"); ver = e ? atoi(e) : 4; }
        if (ver >= 4 && corr_mma_bwd_supported(p)) return corr_mma_bwd(p, st);     // DispNet: banded tensor-core products
    }
    const bool warped = p.u != nullptr;
    const int nd = (2 * p.max_disp) / p.stride + 1;
    const size_t budget = 220 * 1024;
    int TW;
    if (warped) {
        TW = p.w;
        size_t bytes = (size_t)3 * p.w * p.C * 4 + (size_t)p.w * nd * 4 + (size_t)p.w * 4 + 64;
        MS_REQUIRE(bytes <= budget, "corr_bwd: warped row does not fit in shared memory");
    } else {
        TW = -1;
        const int cands[] = {p.w, 128, 64, 32, 16, 8};
        for (int tw : cands) {
            if (tw > p.w) continue;
            size_t win = (size_t)tw + 2 * p.max_disp;
            size_t bytes = 2 * win * p.C * 4 + win * nd * 4 + 64;
            if (bytes <= (size_t)200 * 1024) { TW = tw; break; }
        }
        MS_REQUIRE(TW > 0, "corr_bwd: tile does not fit in shared memory");
    }
    const size_t WIN = warped ? p.w : TW + 2 * p.max_disp;
    size_t smem = 2 * WIN * p.C * 4 + (warped ? (size_t)TW * p.C * 4 : 0) + WIN * nd * 4 + (warped ? (size_t)p.w * 4 : 0) + 64;
    int tma = corr_use_tma() && p.lcs == p.C && p.rcs == p.C;
    if (corr_init()) return -1;
    dim3 grid(cdiv(p.w, TW), p.B * p.h);
    launch_k(corr_bwd_kernel, dim3(grid), dim3(CORR_NT), smem, st, p, TW, nd, tma);
    return check_launch("corr_bwd");
}

}  // namespace ms
