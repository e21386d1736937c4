// tcgen05 weight-gradient kernel for stride-1 convolutions (any dilation).
//
// Replaces the filter-gradient sub-graph tf.gradients derives for tf.nn.conv2d / atrous_conv2d
// (reference Nets/sharedLayers.py:58,72 inside the train ops of Stereo_Online_Adaptation.py:118,128).
//
//   dW[tap][ci][co] = sum over pixels p of  X[p + offset(tap)][ci] * dY[p][co]
//
// GEMM view per CTA (one tap, one 128-channel block of ci, one slice of the pixel range):
//   M = ci (128 TMEM lanes), N = co (<=192), K = pixels in chunks of 32 (a 1 x 32 row segment of one image; TMA pads
//   swizzled inner rows to the 128-byte swizzle span, so the inner box extent must be exactly 32 floats).
//   A (X^T)  : the tap-shifted X segment {128ch,32,1,1} arrives by TMA (zero fill outside the image = SAME padding);
//              each splitter thread owns one channel (= accumulator row), reads its 16 pixels from shared memory,
//              forms the tf32 hi/lo halves and writes them to TENSOR MEMORY (tcgen05.st) -> TS-mode MMAs.
//   B (dY^T) : dY is first transposed to NCHW (one small kernel) so that a TMA box {32,1,N,1} lands as the K-major
//              SWIZZLE_128B tile [N rows][32 pixels]; hi/lo split in shared memory.
//   3xTF32 with separated accumulators (cross terms | rotating hi*hi partial sums).
// Partial sums [split][tap][ci][co] go to the workspace; the existing fixed-order wgrad_reduce finishes (deterministic).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace ms {

struct WgradTCParams {
    int kh, kw, pad_y, pad_x, dil;
    int H, W, NB;                 // map size, batch
    int chunks_x, chunks_y;       // ceil(W/32), H
    int nchunks, chunk_per_split;
    int ci, co, BN, mblocks;
    int n_main, acc_stride, tmem_cols, nslots;
    int nop;                      // operand stages between splitter and MMA (64 TMEM columns + 2*BN*128 B each)
    float* part;                  // [split][tap][ci][co]
};

constexpr int WG_THREADS = 320;
constexpr int WG_SPLIT = 256;
constexpr int X_TILE_BYTES = 32 * 128 * 4;      // 32 pixels x 128 channels

__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapD, const WgradTCParams p) {
    extern __shared__ unsigned char smem_dyn[];
    __shared__ __align__(8) uint64_t full_bar[6], empty_bar[6], ready_bar[4], free_bar[4], accum_bar;
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t base = (s_addr(smem_dyn) + 1023u) & ~1023u;
    unsigned char* gbase = smem_dyn + (base - s_addr(smem_dyn));
    const uint32_t b_bytes = (uint32_t)p.BN * 128u;
    const uint32_t op_bytes = 2u * b_bytes;                         // B_hi, B_lo
    const int NOP = p.nop;
    const uint32_t ring_off = (uint32_t)NOP * op_bytes;
    const uint32_t slot_bytes = (uint32_t)X_TILE_BYTES + b_bytes;   // X tile | raw dY^T tile
    const int NS = p.nslots;
    const uint32_t a_col0 = (uint32_t)((p.n_main + 1) * p.acc_stride);

    const int tap = blockIdx.x / p.mblocks, mb = blockIdx.x - tap * p.mblocks;
    const int tr = tap / p.kw, ts = tap - tr * p.kw;
    const int offy = tr * p.dil - p.pad_y, offx = ts * p.dil - p.pad_x;
    const int c_begin = blockIdx.y * p.chunk_per_split;
    const int c_end = min(p.nchunks, c_begin + p.chunk_per_split);
    const int total = max(0, c_end - c_begin);

    if (threadIdx.x == 0) {
        for (int i = 0; i < NS; ++i) { mb_init(&full_bar[i], 1); mb_init(&empty_bar[i], WG_SPLIT / 32); }
        for (int i = 0; i < NOP; ++i) { mb_init(&ready_bar[i], WG_SPLIT / 32); mb_init(&free_bar[i], 1); }
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

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int slot = 0;
            uint32_t ph = 0;
            for (int it = 0; it < total; ++it) {
                int c = c_begin + it;
                const int cx = c % p.chunks_x; c /= p.chunks_x;
                const int cy = c % p.chunks_y;
                const int img = c / p.chunks_y;
                const int x0 = cx * 32, y0 = cy;
                mb_wait(&empty_bar[slot], ph ^ 1u);
                unsigned char* sl = gbase + ring_off + (size_t)slot * slot_bytes;
                mb_expect_tx(&full_bar[slot], slot_bytes);
                tma_load_4d(sl, &mapX, &full_bar[slot], mb * 128, x0 + offx, y0 + offy, img);
                tma_load_4d(sl + X_TILE_BYTES, &mapD, &full_bar[slot], x0, y0, 0, img);
                if (++slot == NS) { slot = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (TS mode: A from tensor memory) =================
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.BN >> 3) << 17) | ((128u >> 4) << 24);
            int s = 0, rot = 0, gcount = 0;
            uint32_t oph = 0;
            for (int it = 0; it < total; ++it) {
                mb_wait(&ready_bar[s], oph);
                tc_fence_after();
                const uint32_t sb = base + (uint32_t)s * op_bytes;
                const uint64_t b_hi = umma_desc_sw128(sb), b_lo = umma_desc_sw128(sb + b_bytes);
                const uint32_t a_hi = tmem + a_col0 + (uint32_t)s * 64u, a_lo = a_hi + 32u;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint64_t o = (uint64_t)(j * 2);
                    const uint32_t ao = (uint32_t)(j * 8);
                    tc_mma_tf32_ts(tmem, a_lo + ao, b_hi + o, idesc, gcount > 0 ? 1u : 0u);
                    tc_mma_tf32_ts(tmem, a_hi + ao, b_lo + o, idesc, 1u);
                    const uint32_t dmain = tmem + (uint32_t)((1 + rot) * p.acc_stride);
                    tc_mma_tf32_ts(dmain, a_hi + ao, b_hi + o, idesc, gcount >= p.n_main ? 1u : 0u);
                    ++gcount;
                    if (++rot == p.n_main) rot = 0;
                }
                tc_commit(&free_bar[s]);
                if (++s == NOP) { s = 0; oph ^= 1u; }
            }
            tc_commit(&accum_bar);
        }
    } else {
        // ================= splitter (warps 2..9): thread <-> input channel (accumulator row) =================
        const int st_tid = threadIdx.x - 64;
        const int b_f4 = p.BN * 8;
        const int q = warp & 3;
        const int hsel = (warp - 2) >> 2;              // which 16 of the 32 pixels of the chunk
        const int m = q * 32 + lane;                   // channel inside the 128-block
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        {
            int slot = 0, s = 0;
            uint32_t ph = 0, oph = 0;
            for (int it = 0; it < total; ++it) {
                mb_wait(&free_bar[s], oph ^ 1u);
                mb_wait(&full_bar[slot], ph);
                const unsigned char* sl = gbase + ring_off + (size_t)slot * slot_bytes;
                // ---- A: X^T. pixel k of the chunk sits at k*512 bytes, channel m at +4m  (conflict-free across lanes)
                const float* xs = reinterpret_cast<const float*>(sl) + m;
                float hi[16], lo[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float v = xs[(hsel * 16 + e) * 128];
                    hi[e] = tf32_hi(v);
                    lo[e] = v - hi[e];
                }
                const uint32_t acol = tmem + lane_base + a_col0 + (uint32_t)s * 64u + (uint32_t)hsel * 16u;
                tc_st16(acol, hi);
                tc_st16(acol + 32u, lo);
                // ---- B: dY^T tile (already K-major swizzled by TMA): elementwise hi/lo split
                unsigned char* stg = gbase + (size_t)s * op_bytes;
                float4* __restrict__ bhi = reinterpret_cast<float4*>(stg);
                float4* __restrict__ blo = reinterpret_cast<float4*>(stg + b_bytes);
                const float4* __restrict__ braw = reinterpret_cast<const float4*>(sl + X_TILE_BYTES);
                for (int i0 = st_tid; i0 < b_f4; i0 += 2 * WG_SPLIT) {
                    const int i1 = i0 + WG_SPLIT;
                    const bool two = i1 < b_f4;
                    float4 w0 = braw[i0], w1 = two ? braw[i1] : make_float4(0.f, 0.f, 0.f, 0.f);
                    float4 h, l;
                    h.x = tf32_hi(w0.x); h.y = tf32_hi(w0.y); h.z = tf32_hi(w0.z); h.w = tf32_hi(w0.w);
                    l.x = w0.x - h.x; l.y = w0.y - h.y; l.z = w0.z - h.z; l.w = w0.w - h.w;
                    bhi[i0] = h; blo[i0] = l;
                    if (two) {
                        h.x = tf32_hi(w1.x); h.y = tf32_hi(w1.y); h.z = tf32_hi(w1.z); h.w = tf32_hi(w1.w);
                        l.x = w1.x - h.x; l.y = w1.y - h.y; l.z = w1.z - h.z; l.w = w1.w - h.w;
                        bhi[i1] = h; blo[i1] = l;
                    }
                }
                tc_wait_st();
                fence_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { mb_arrive(&ready_bar[s]); mb_arrive(&empty_bar[slot]); }
                if (++slot == NS) { slot = 0; ph ^= 1u; }
                if (++s == NOP) { s = 0; oph ^= 1u; }
            }
        }
        // ================= epilogue: raw partial sums [ci][co] =================
        if (total > 0) {
            mb_wait(&accum_bar, 0);
            tc_fence_after();
        }
        const int ci_g = mb * 128 + m;
        const bool valid = ci_g < p.ci;
        float* prow = p.part + (((size_t)blockIdx.y * p.kh * p.kw + tap) * p.ci + ci_g) * p.co;
        const bool vec = (p.co & 3) == 0;
        const int chunks = p.BN / 16, half = (chunks + 1) / 2;
        const int cbeg = (warp < 6 ? 0 : half) * 16, cend = (warp < 6 ? half : chunks) * 16;
        for (int c0 = cbeg; c0 < cend; c0 += 16) {
            float v[16];
            if (total > 0) {
                uint32_t r0[16], r1[16], r2[16], r3[16];
                tc_ld16_nowait(tmem + lane_base + (uint32_t)c0, r0);
                tc_ld16_nowait(tmem + lane_base + (uint32_t)(p.acc_stride + c0), r1);
                if (p.n_main > 1) tc_ld16_nowait(tmem + lane_base + (uint32_t)(2 * p.acc_stride + c0), r2);
                if (p.n_main > 2) tc_ld16_nowait(tmem + lane_base + (uint32_t)(3 * p.acc_stride + c0), r3);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float t = __uint_as_float(r0[j]) + __uint_as_float(r1[j]);
                    if (p.n_main > 1) t += __uint_as_float(r2[j]);
                    if (p.n_main > 2) t += __uint_as_float(r3[j]);
                    v[j] = t;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = 0.f;
            }
            if (!valid) continue;
            if (vec && c0 + 16 <= p.co) {
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4*>(prow + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (c0 + j < p.co) prow[c0 + j] = v[j];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// dY [img][pixels][co] (channel stride cs) -> dYT [img][co][pixels]
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ src, int cs, int co, int P, float* __restrict__ dst) {
    __shared__ float tile[32][33];
    const int img = blockIdx.z;
    const float* s = src + (size_t)img * P * cs;
    float* d = dst + (size_t)img * co * P;
    const int c = blockIdx.x * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int px = blockIdx.y * 32 + j;
        tile[j][threadIdx.x] = (px < P && c < co) ? s[(size_t)px * cs + c] : 0.f;
    }
    __syncthreads();
    const int px2 = blockIdx.y * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c2 = blockIdx.x * 32 + j;
        if (px2 < P && c2 < co) d[(size_t)c2 * P + px2] = tile[threadIdx.x][j];
    }
}

__global__ void wgrad_tc_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, size_t n, int split) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
    for (int k = 0; k < split; ++k) s += partial[(size_t)k * n + i];
    dw[i] = s;
}

static int wg_splits(int ctas_per_split, int nchunks) {
    int s = std::max(1, 296 / std::max(1, ctas_per_split));
    s = std::min(s, std::max(1, nchunks / 4));
    return std::min(s, 64);
}

bool wgrad_tc_supported(const ConvWgrad& q) {
    if (q.stride != 1) return false;
    if (q.x.h != q.dy.h || q.x.w != q.dy.w) return false;
    const int ci = q.x.c, co = q.dy.c;
    if (ci < 16 || co < 16 || co > 192 || (co & 3)) return false;
    if ((long)ci * co < 2048) return false;
    if ((q.x.cs & 3) || (reinterpret_cast<uintptr_t>(q.x.p) & 15)) return false;
    if ((q.dy.w & 3) || q.dy.h * q.dy.w < 256) return false;
    return true;
}

// floats needed in q.workspace: NCHW copy of dy + split partials (+ bias partials, handled by bias_grad afterwards)
size_t wgrad_tc_workspace_floats(int taps, int ci, int co, int n, int h, int w) {
    const int nchunks = n * h * cdiv(w, 32);
    const int split = wg_splits(taps * cdiv(ci, 128), nchunks);
    return (size_t)n * co * h * w + 64 + (size_t)split * taps * ci * co + 128 * (size_t)co + 4096;
}

int wgrad_tc_init() {
    static bool done = false;
    if (done) return 0;
    MS_CHECK_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    done = true;
    return 0;
}

int wgrad_tc(const ConvWgrad& q, cudaStream_t st) {
    MS_REQUIRE(wgrad_tc_supported(q), "wgrad_tc: unsupported geometry");
    if (wgrad_tc_init()) return -1;
    const int taps = q.kh * q.kw, ci = q.x.c, co = q.dy.c;
    const int n = q.dy.n, h = q.dy.h, w = q.dy.w, P = h * w;
    WgradTCParams p{};
    p.kh = q.kh; p.kw = q.kw; p.pad_y = q.pad_t; p.pad_x = q.pad_l; p.dil = q.dil;
    p.H = h; p.W = w; p.NB = n;
    p.chunks_x = cdiv(w, 32); p.chunks_y = h;
    p.nchunks = n * p.chunks_x * p.chunks_y;
    p.ci = ci; p.co = co; p.BN = (co + 15) / 16 * 16; p.mblocks = cdiv(ci, 128);
    p.acc_stride = (p.BN + 31) / 32 * 32;
    static int nop_env = -1;
    if (nop_env < 0) { const char* e = getenv("MS_WG_NS"); nop_env = e ? atoi(e) : 2; }     // measured: 3 stages gain nothing and cost an accumulator
    int nop = std::max(2, std::min(4, nop_env));
    while (nop > 2 && 2 * p.acc_stride + nop * 64 > 512) --nop;
    p.nop = nop;
    p.n_main = std::max(1, std::min(3, (512 - nop * 64) / p.acc_stride - 1));
    const int need = (p.n_main + 1) * p.acc_stride + nop * 64;
    MS_REQUIRE(need <= 512, "wgrad_tc: accumulators do not fit tensor memory");
    p.tmem_cols = need <= 256 ? 256 : 512;
    const int split = wg_splits(taps * p.mblocks, p.nchunks);
    p.chunk_per_split = cdiv(p.nchunks, split);
    const size_t dyt_floats = ((size_t)n * co * P + 63) / 64 * 64;
    const size_t wn = (size_t)taps * ci * co;
    MS_REQUIRE(q.workspace_floats >= dyt_floats + (size_t)split * wn, "wgrad_tc: workspace too small");
    float* dyt = q.workspace;
    p.part = q.workspace + dyt_floats;
    const size_t b_bytes = (size_t)p.BN * 128, op_bytes = 2 * b_bytes, slot_bytes = X_TILE_BYTES + b_bytes;
    const size_t fixed = (size_t)p.nop * op_bytes + 1024;
    int ns = (int)std::min<size_t>(6, (224 * 1024 - fixed) / slot_bytes);
    MS_REQUIRE(ns >= 2, "wgrad_tc: tiles do not fit shared memory");
    p.nslots = ns;

    nhwc_to_nchw_kernel<<<dim3(cdiv(co, 32), cdiv(P, 32), n), dim3(32, 8), 0, st>>>(q.dy.p, q.dy.cs, co, P, dyt);
    const CUtensorMap *mapX, *mapD;
    {
        cuuint64_t dims[4] = {(cuuint64_t)ci, (cuuint64_t)q.x.w, (cuuint64_t)q.x.h, (cuuint64_t)q.x.n};
        cuuint64_t strides[3] = {(cuuint64_t)q.x.cs * 4, (cuuint64_t)q.x.w * q.x.cs * 4, (cuuint64_t)q.x.h * q.x.w * q.x.cs * 4};
        cuuint32_t box[4] = {128, 32, 1, 1};
        if (tc_get_map(&mapX, q.x.p, 4, dims, strides, box, false)) return -1;
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)co, (cuuint64_t)n};
        cuuint64_t strides[3] = {(cuuint64_t)w * 4, (cuuint64_t)P * 4, (cuuint64_t)co * P * 4};
        cuuint32_t box[4] = {32, 1, (cuuint32_t)p.BN, 1};
        if (tc_get_map(&mapD, dyt, 4, dims, strides, box, true)) return -1;
    }
    const size_t smem = fixed + (size_t)ns * slot_bytes;
    wgrad_tc_kernel<<<dim3(taps * p.mblocks, split), WG_THREADS, smem, st>>>(*mapX, *mapD, p);
    wgrad_tc_reduce_kernel<<<(unsigned)cdivz(wn, 256), 256, 0, st>>>(p.part, q.dw, wn, split);
    if (check_launch("wgrad_tc", 3)) return -1;
    if (q.db) {
        float* bws = p.part + (size_t)split * wn;
        const size_t left = q.workspace_floats - dyt_floats - (size_t)split * wn;
        return bias_grad(q.dy, q.db, bws, left, st);
    }
    return 0;
}

}  // namespace ms
