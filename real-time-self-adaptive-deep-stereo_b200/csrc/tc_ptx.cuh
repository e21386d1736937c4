// tcgen05 / TMA / mbarrier PTX wrappers shared by the tensor-core kernels (conv_bf.cu, wgrad_bf.cu, wgrad_tc.cu) and the
// TMA-staged correlation (corr_tma.cu).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace ms {

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mb_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_addr(bar)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t a = s_addr(bar);
    uint32_t ok = 0;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(s_addr(dst)), "l"(map), "r"(s_addr(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(s_addr(dst)), "l"(map), "r"(s_addr(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// One lane of a converged warp (cute::elect_one_sync).  The tcgen05 / TMA instructions take their descriptors from UNIFORM
// registers: issued from a loop that only lane 0 runs (`if (lane == 0)`), the descriptors are computed in vector registers and
// every operand crosses over with an ELECT + R2UR.BROADCAST pair in front of each instruction -- wgrad_bf spent 200 cycles
// per MMA with its loads switched off (profiles/r2_wgrad_bf_killswitch.log) where the instruction itself costs
// max(N / 2, 50) cycles (scripts/mma_probe.py, profiles/r2_mma_probe.log).  Run the loop on the whole warp with warp-uniform
// control flow (warp index through a shuffle) and predicate only the instruction itself: the descriptor arithmetic then
// runs on the uniform datapath (UIADD3 / UMOV) and nothing crosses over.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_addr(bar)) : "memory");
}

__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
          "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
          "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
          "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
          "r"(__float_as_uint(v[15]))
        : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO=1 | SBO=1024B |
// version=1 (sm100) | layout_type=2 (SWIZZLE_128B).  Tile base must be 1024-byte aligned.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_byte_addr) {
    return (uint64_t)((smem_byte_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// tf32 "hi" half by truncation: the top 19 bits of x (exactly representable in tf32 whatever rounding the tensor core
// applies to its inputs); lo = x - hi is then exact in fp32 with |lo| < 2^-10 |x|.  One LOP3 instead of the 4-5
// instruction sequence cvt.rna.tf32.f32 expands to -- ncu showed the splitter loop to be instruction-latency bound
// (349 instructions per warp per K step, 128 of them from the 32 cvt.rna).
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }


// cached cuTensorMapEncodeTiled (fp32, zero OOB fill); swizzle128=false => SWIZZLE_NONE.  (corr_tma.cu)
int tc_get_map(const CUtensorMap** out, void* addr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, bool swizzle128);

// cached cuTensorMapEncodeTiled for bf16 planes (zero OOB fill, element strides); swizzle_bytes 64 or 128.  (conv_bf.cu)
int bf_get_map(const CUtensorMap** out, void* addr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, const cuuint32_t* estr, int swizzle_bytes = 64);

}  // namespace ms
