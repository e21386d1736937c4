// Correlation forward v4: tensor-map TMA staging, one (or two) threads per pixel.
//
// Same operator as corr.cu (reference Nets/sharedLayers.py:23-51 correlation, Nets/MadNet.py:370-375 concat,
// Nets/MadNet.py:400-436 linear warp; native launcher Nets/Native/shift_corr.cu.cc:193-233), specialised for the MADNet
// cost volume: max_disp = 2, stride 1 (5 displacements), C a multiple of 32.
//
// ncu on v3 (profiles/r1_ncu_corr_fwd3_L2_1920x1088_B8.txt) showed ~3000 thread instructions per pixel: staging loops
// (index division, swizzle, 64-bit address math), bounds predicates in the inner loop and shuffle reductions, i.e. the
// kernel was instruction-issue bound at 28 % of HBM.  Here
//   * the left tile, the right window and the left half of the concat buffer move by TMA tensor copies
//     (cp.async.bulk.tensor, SWIZZLE_128B: a pixel's 32-channel block is one 128-byte row, its 16-byte chunks XOR-ed
//     with row&7), so staging and the concat copy cost no thread instructions and reads are bank-conflict free with
//     lane == pixel;
//   * out-of-image columns are zero rows (TMA zero fill for the un-warped window, zero taps for the warped one), so the
//     displacement loop has no bounds predicates;
//   * the warped right row RW is materialised once per tile in shared memory, every RW column feeds 5 outputs;
//   * each pixel is owned by LP (1 or 2) lanes that keep the 5 running sums in registers; results leave as two 128-bit
//     stores per pixel into the concat buffer ([c0 c1 c2 c3][c4 u 0 0]).
// The right window of a warped tile is data dependent: taps are computed first, the window [min tap, max tap] is then
// fetched by one TMA copy per 32-channel block (bounded by RB rows; taps outside read global memory directly).
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <map>

#include "common.cuh"
#include "corr_common.cuh"
#include "tc_ptx.cuh"

namespace ms {

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
                 "r"(s_addr(src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// shared-memory byte address of row r of a swizzled tile, pre-XORed so that chunk q sits at rowkey(..) ^ (q << 4):
// the row base is 128-byte aligned and the swizzled chunk offset is < 128, so OR == ADD and the XOR distributes.
__device__ __forceinline__ uint32_t rowkey(uint32_t tile_s, int r) { return (tile_s + (uint32_t)r * 128u) | (((uint32_t)r & 7u) << 4); }

struct Corr4Params {
    CorrFwd p;
    int TW, WB, RB, ncb;     // tile width, RW rows (>= TW+4), raw right window rows, 32-channel blocks
    int store_o, store_o2;   // left -> concat copy by TMA store
    float invC;
};

// float4 index of chunk q of row r in 32-channel block cb of a [ncb][rows][8] swizzled tile
__device__ __forceinline__ int t4(int cb, int rows, int r, int q) { return ((cb * rows + r) << 3) + (q ^ (r & 7)); }

template <int LP, int NCB_CT>     // NCB_CT > 0: number of 32-channel blocks known at compile time (loops unroll)
__global__ void __launch_bounds__(256) corr_fwd4_kernel(const __grid_constant__ CUtensorMap mapL,
                                                        const __grid_constant__ CUtensorMap mapR,
                                                        const __grid_constant__ CUtensorMap mapO,
                                                        const __grid_constant__ CUtensorMap mapO2, const Corr4Params k) {
    pdl_prologue();
    constexpr int ND = 5, D = 2, QPL = 8 / LP;
    const CorrFwd& p = k.p;
    extern __shared__ unsigned char smem_dyn[];
    __shared__ __align__(8) uint64_t barL, barR;
    __shared__ int s_lo, s_hi;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
    const int TW = k.TW, WB = k.WB, RB = k.RB, ncb = NCB_CT > 0 ? NCB_CT : k.ncb;
    const int w = p.w;
    const bool warped = p.u != nullptr;
    const int row = blockIdx.y, x0 = blockIdx.x * TW;
    const int NW = TW + 2 * D;                                        // RW column t <-> image column x0 - D + t
    const uint32_t base = (s_addr(smem_dyn) + 1023u) & ~1023u;
    unsigned char* g = smem_dyn + (base - s_addr(smem_dyn));
    float4* Ls = reinterpret_cast<float4*>(g);                        // [ncb][TW][8]
    float4* RWs = Ls + (size_t)ncb * TW * 8;                           // [ncb][WB][8]
    float4* Rs = RWs + (size_t)ncb * WB * 8;                           // [ncb][RB][8]   (warped only)
    Tap* taps = reinterpret_cast<Tap*>(Rs + (warped ? (size_t)ncb * RB * 8 : 0));   // [WB]
    const uint32_t Ls_s = base, RWs_s = Ls_s + (uint32_t)(ncb * TW) * 128u, Rs_s = RWs_s + (uint32_t)(ncb * WB) * 128u;

    const float* rrow = p.right + (size_t)row * w * p.rcs;
    float* orow = p.out + (size_t)row * w * p.ocs;

    if (tid == 0) {
        mb_init(&barL, 1); mb_init(&barR, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_lo = INT_MAX; s_hi = -1;
    }
    __syncthreads();
    if (tid == 0) {
        mb_expect_tx(&barL, (uint32_t)(ncb * TW) * 128u);
        for (int cb = 0; cb < ncb; ++cb) tma_load_3d(Ls + (size_t)cb * TW * 8, &mapL, &barL, cb * 32, x0, row);
        if (!warped) {
            mb_expect_tx(&barR, (uint32_t)(ncb * WB) * 128u);
            for (int cb = 0; cb < ncb; ++cb) tma_load_3d(RWs + (size_t)cb * WB * 8, &mapR, &barR, cb * 32, x0 - D, row);
        }
    }
    int rlo = 0, rhi = 0;
    if (warped) {
        const float* urow = p.u + (size_t)row * w * p.ucs;
        int lo = INT_MAX, hi = -1;
        for (int t = tid; t < NW; t += nthr) {
            const int xc = x0 - D + t;
            Tap tp; tp.i0 = 0; tp.i1 = 0; tp.w0 = 0.f; tp.w1 = 0.f;       // columns outside the image: RW = 0
            if (xc >= 0 && xc < w) {
                const WarpTap wt = warp_tap(xc, urow[(size_t)xc * p.ucs], w, true);
                tp.i0 = wt.i0; tp.i1 = wt.i1; tp.w0 = wt.w0; tp.w1 = wt.w1;
                if (wt.w0 != 0.f) { lo = min(lo, wt.i0); hi = max(hi, wt.i0); }
                if (wt.w1 != 0.f) { lo = min(lo, wt.i1); hi = max(hi, wt.i1); }
            }
            taps[t] = tp;
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (lane == 0 && hi >= 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
        __syncthreads();
        rlo = s_lo; rhi = s_hi + 1;
        if (rhi <= rlo) { rlo = 0; rhi = 0; }
        if (rhi - rlo > RB) rhi = rlo + RB;                              // further taps take the global path
        if (tid == 0 && rhi > rlo) {
            mb_expect_tx(&barR, (uint32_t)(ncb * RB) * 128u);
            for (int cb = 0; cb < ncb; ++cb) tma_load_3d(Rs + (size_t)cb * RB * 8, &mapR, &barR, cb * 32, rlo, row);
        }
    }
    // ---- left tile -> concat buffer(s)
    const bool any_store = p.copy_left && (k.store_o || (p.out2 && k.store_o2));
    if (tid == 0 && any_store) {
        mb_wait(&barL, 0);
        for (int cb = 0; cb < ncb; ++cb) {
            if (k.store_o) tma_store_3d(&mapO, Ls + (size_t)cb * TW * 8, cb * 32, x0, row);
            if (p.out2 && k.store_o2) tma_store_3d(&mapO2, Ls + (size_t)cb * TW * 8, cb * 32, x0, row);
        }
        bulk_commit();
    }
    mb_wait(&barL, 0);
    if (p.copy_left && (!k.store_o || (p.out2 && !k.store_o2))) {
        float* o2row = p.out2 ? p.out2 + (size_t)row * w * p.o2cs : nullptr;
        const int per = ncb * 8;
        for (int e = tid; e < TW * per; e += nthr) {
            const int j = e / per, r = e - j * per, cb = r >> 3, q = r & 7;
            if (x0 + j >= w) continue;
            const float4 v = Ls[t4(cb, TW, j, q)];
            if (!k.store_o) *reinterpret_cast<float4*>(orow + (size_t)(x0 + j) * p.ocs + cb * 32 + q * 4) = v;
            if (o2row && !k.store_o2) *reinterpret_cast<float4*>(o2row + (size_t)(x0 + j) * p.o2cs + cb * 32 + q * 4) = v;
        }
    }
    const int sub = tid % LP, pl = tid / LP, npl = nthr / LP;          // lane within pixel, pixel slot
    const int q0 = sub * QPL;
    // ---- RW[t] = w0 * R[i0] + w1 * R[i1]
    if (warped) {
        if (rhi > rlo) mb_wait(&barR, 0);
        const uint32_t subk = (uint32_t)q0 << 4;
        for (int t = pl; t < NW; t += npl) {
            const Tap tp = taps[t];
            const int r0 = tp.i0 - rlo, r1 = tp.i1 - rlo;
            const bool in0 = r0 >= 0 && tp.i0 < rhi, in1 = r1 >= 0 && tp.i1 < rhi;
            const bool z0 = tp.w0 == 0.f, z1 = tp.w1 == 0.f;
            uint32_t dk = rowkey(RWs_s, t) ^ subk;
            if (!z0 && !z1 && in0 && in1) {                  // common case: both taps staged
                uint32_t ak = rowkey(Rs_s, r0) ^ subk, bk = rowkey(Rs_s, r1) ^ subk;
#pragma unroll
                for (int cb = 0; cb < ncb; ++cb) {
#pragma unroll
                    for (int qq = 0; qq < QPL; ++qq) {
                        float4 a = lds128(ak ^ (uint32_t)(qq << 4));
                        const float4 b = lds128(bk ^ (uint32_t)(qq << 4));
                        a.x = tp.w0 * a.x + tp.w1 * b.x; a.y = tp.w0 * a.y + tp.w1 * b.y;
                        a.z = tp.w0 * a.z + tp.w1 * b.z; a.w = tp.w0 * a.w + tp.w1 * b.w;
                        sts128(dk ^ (uint32_t)(qq << 4), a);
                    }
                    ak += (uint32_t)RB * 128u; bk += (uint32_t)RB * 128u; dk += (uint32_t)WB * 128u;
                }
            } else {                                         // border columns (zero weights) / taps outside the staged window
                for (int cb = 0; cb < ncb; ++cb) {
#pragma unroll
                    for (int qq = 0; qq < QPL; ++qq) {
                        const int q = q0 + qq;
                        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                        if (!z0) a = in0 ? Rs[t4(cb, RB, r0, q)] : *reinterpret_cast<const float4*>(rrow + (size_t)tp.i0 * p.rcs + cb * 32 + q * 4);
                        if (!z1) b = in1 ? Rs[t4(cb, RB, r1, q)] : *reinterpret_cast<const float4*>(rrow + (size_t)tp.i1 * p.rcs + cb * 32 + q * 4);
                        a.x = tp.w0 * a.x + tp.w1 * b.x; a.y = tp.w0 * a.y + tp.w1 * b.y;
                        a.z = tp.w0 * a.z + tp.w1 * b.z; a.w = tp.w0 * a.w + tp.w1 * b.w;
                        RWs[t4(cb, WB, t, q)] = a;
                    }
                }
            }
        }
        __syncthreads();
    } else {
        mb_wait(&barR, 0);
    }
    // ---- correlation: thread (pl, sub) owns pixel x0+pl, chunks [q0, q0+QPL) of every channel block
    {
        const bool act = pl < TW && x0 + pl < w;
        const int j = pl < TW ? pl : TW - 1;
        float acc[ND];
#pragma unroll
        for (int i = 0; i < ND; ++i) acc[i] = 0.f;
        {
            const uint32_t subk = (uint32_t)q0 << 4;
            uint32_t lk = rowkey(Ls_s, j) ^ subk;
            uint32_t rk[ND];
#pragma unroll
            for (int i = 0; i < ND; ++i) rk[i] = rowkey(RWs_s, j + i) ^ subk;
#pragma unroll
            for (int cb = 0; cb < ncb; ++cb) {
#pragma unroll
                for (int qq = 0; qq < QPL; ++qq) {
                    const float4 l = lds128(lk ^ (uint32_t)(qq << 4));
#pragma unroll
                    for (int i = 0; i < ND; ++i) {
                        const float4 a = lds128(rk[i] ^ (uint32_t)(qq << 4));
                        acc[i] = fmaf(l.x, a.x, acc[i]); acc[i] = fmaf(l.y, a.y, acc[i]);
                        acc[i] = fmaf(l.z, a.z, acc[i]); acc[i] = fmaf(l.w, a.w, acc[i]);
                    }
                }
                lk += (uint32_t)TW * 128u;
#pragma unroll
                for (int i = 0; i < ND; ++i) rk[i] += (uint32_t)WB * 128u;
            }
        }
        const float invC = k.invC;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            if (LP == 2) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 1);
            acc[i] *= invC;
        }
        if (act && sub == 0) {
            const int x = x0 + pl;
            const int coff = p.copy_left ? p.C : 0;
            float* o = orow + (size_t)x * p.ocs + coff;
            const bool pack8 = p.copy_left && (p.ocs & 3) == 0 && p.ocs >= coff + 8;
            if (pack8) {
                const float uu = p.u_chan ? o[5] : 0.f;            // the u channel was written by the resize kernel
                *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4], uu, 0.f, 0.f);
                for (int c = coff + 8; c < p.ocs; ++c) orow[(size_t)x * p.ocs + c] = 0.f;
            } else {
#pragma unroll
                for (int i = 0; i < ND; ++i) o[i] = acc[i];
                if (p.copy_left)
                    for (int c = coff + ND + p.u_chan; c < p.ocs; ++c) orow[(size_t)x * p.ocs + c] = 0.f;
            }
        }
    }
    if (tid == 0 && any_store) bulk_wait_read0();       // the TMA stores read Ls: keep the CTA's smem alive until done
}

static int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

struct MapKey {
    uintptr_t addr; int rank; int swz; uint64_t d[4]; uint64_t s[3]; uint32_t b[4];
    bool operator<(const MapKey& o) const { return memcmp(this, &o, sizeof(MapKey)) < 0; }
};

// fp32 tensor maps for the TMA copies here and in wgrad_tc.cu (declared in tc_ptx.cuh)
int tc_get_map(const CUtensorMap** out, void* addr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, bool swizzle128) {
    static std::map<MapKey, CUtensorMap> cache;
    MapKey k;
    memset(&k, 0, sizeof k);
    k.addr = reinterpret_cast<uintptr_t>(addr); k.rank = rank; k.swz = swizzle128 ? 1 : 0;
    for (int i = 0; i < rank; ++i) { k.d[i] = dims[i]; k.b[i] = box[i]; }
    for (int i = 0; i + 1 < rank; ++i) k.s[i] = strides_bytes[i];
    auto it = cache.find(k);
    if (it == cache.end()) {
        EncodeTiledFn enc = get_encode();
        MS_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
        cuuint32_t es[5] = {1, 1, 1, 1, 1};
        CUtensorMap m;
        CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, addr, dims, strides_bytes, box, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r)); return -1; }
        if (cache.size() >= 4096) {
            // cache full (callers that keep passing fresh pointers): do not evict -- pointers handed out earlier in the same
            // launch sequence must stay valid -- but serve this descriptor from a small ring of uncached slots
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

// 3-D view {channels, w, B*h} of an NHWC tensor with channel stride cs; box {32, rows, 1}
static int feat_map(CUtensorMap* out, const float* ptr, int chans, int cs, int w, int rows_total, int box_rows) {
    const cuuint64_t dims[3] = {(cuuint64_t)chans, (cuuint64_t)w, (cuuint64_t)rows_total};
    const cuuint64_t strides[2] = {(cuuint64_t)cs * 4, (cuuint64_t)w * cs * 4};
    const cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
    const CUtensorMap* m = nullptr;
    if (tc_get_map(&m, const_cast<float*>(ptr), 3, dims, strides, box, true)) return -1;
    *out = *m;                                            // by value: the cache may be recycled by a later lookup
    return 0;
}

// returns 0 = launched, 1 = shape not handled by this kernel (caller uses v1..v3), -1 = error
int corr_fwd4(const CorrFwd& p, cudaStream_t st) {
    const bool warped = p.u != nullptr;
    if (p.stride != 1 || p.max_disp != 2 || p.C % 32 != 0 || p.C > 256 || p.w < 8) return 1;
    if ((p.lcs & 3) || (p.rcs & 3) || !al16(p.left) || !al16(p.right) || !al16(p.out)) return 1;
    if (p.copy_left && (p.ocs & 3)) return 1;
    static int tw_env = -2, lp_env, st_env, slack_env;
    if (tw_env == -2) {
        lp_env = env_int("MS_CORR4_LP", 2); st_env = env_int("MS_CORR4_ST", 1); slack_env = env_int("MS_CORR4_SLACK", 16);
        tw_env = env_int("MS_CORR4_TW", 0);
    }
    const int LP = lp_env == 1 ? 1 : 2;
    const int ncb = p.C / 32;
    // measured (profiles/r1_corr_v4_ab.log): 64-pixel tiles (7 CTAs per SM at C=32) beat 128; slack 16 beats 32
    int TW = tw_env > 0 ? tw_env : std::max(32, std::min(64, (128 / ncb + 7) / 8 * 8));
    TW = std::min(TW, 256 / LP);
    TW = std::min(TW, (p.w + 7) / 8 * 8);
    TW = std::max(8, TW / 8 * 8);
    const int WB = (TW + 4 + 7) / 8 * 8;
    const int RB = warped ? std::min(256, (TW + 4 + std::max(8, slack_env) + 7) / 8 * 8) : 0;
    const size_t smem = (size_t)ncb * (TW + WB + RB) * 128 + (size_t)WB * sizeof(Tap) + 1024 + 64;
    if (smem > 200 * 1024) return 1;

    Corr4Params k;
    k.invC = 1.f / (float)p.C;
    k.p = p; k.TW = TW; k.WB = WB; k.RB = RB; k.ncb = ncb;
    k.store_o = (p.copy_left && st_env) ? 1 : 0;
    k.store_o2 = (p.copy_left && p.out2 && st_env && (p.o2cs & 3) == 0 && al16(p.out2)) ? 1 : 0;
    const int rows = p.B * p.h;
    CUtensorMap mL, mR, mO, mO2;
    if (feat_map(&mL, p.left, p.C, p.lcs, p.w, rows, TW)) return -1;
    if (feat_map(&mR, p.right, p.C, p.rcs, p.w, rows, warped ? RB : WB)) return -1;
    mO = mL; mO2 = mL;
    if (k.store_o && feat_map(&mO, p.out, p.C, p.ocs, p.w, rows, TW)) return -1;
    if (k.store_o2 && feat_map(&mO2, p.out2, p.C, p.o2cs, p.w, rows, TW)) return -1;

    static bool attr = false;
    if (!attr) {
        MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd4_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
        MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd4_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
        MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd4_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
        MS_CHECK_CUDA(cudaFuncSetAttribute(corr_fwd4_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
        attr = true;
    }
    const dim3 grid(cdiv(p.w, TW), rows);
    const int threads = (TW * LP + 31) / 32 * 32;
    if (LP == 1) launch_k(corr_fwd4_kernel<1, 0>, dim3(grid), dim3(threads), smem, st, mL, mR, mO, mO2, k);
    else if (ncb == 1) launch_k(corr_fwd4_kernel<2, 1>, dim3(grid), dim3(threads), smem, st, mL, mR, mO, mO2, k);
    else if (ncb == 2) launch_k(corr_fwd4_kernel<2, 2>, dim3(grid), dim3(threads), smem, st, mL, mR, mO, mO2, k);
    else launch_k(corr_fwd4_kernel<2, 0>, dim3(grid), dim3(threads), smem, st, mL, mR, mO, mO2, k);
    return check_launch("corr_fwd4");
}

}  // namespace ms
