// avd_umma.cuh -- thin PTX wrappers for the Blackwell (sm_100a) tensor-core path:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05.{alloc,mma,commit,ld,fence}, shared-memory matrix descriptors.
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor" tables.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace avd {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cnt(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes (or the hint expires) instead
// of returning after a short system-dependent interval.  A waiting warp then costs no issue slots -- without the hint the
// consumer warps' polling loops (SYNCS / BRA / YIELD, ~30 % of all executed instructions) competed with the single MMA-issuing
// warp for its scheduler, and that warp's serial instruction stream is the critical path of every persistent kernel here.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMA -----------------------------------------------------------------------------------------
// Host: 3-D bf16 tensor map {inner, rows, batch} with a {box_inner, box_rows, 1} box and 128-byte swizzle; pitch and batch_stride
// in elements (a single batch may pass batch_stride = 0).  Returns AVD_OK, or AVD_ERR_CUDA with the error text set (avd_lib.cu).
int make_tensor_map(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t pitch, uint64_t batch_stride,
                    uint32_t box_inner, uint32_t box_rows);

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// shared -> global tile store (bulk async-group completion); the source tile must stay intact until bulk_wait_read0()
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---- tcgen05 -------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp; writes the TMEM base address (lane 0, column c) to *dst_smem
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives when all previously issued MMAs of this thread have completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane (warp w may only touch lanes 32*(w%4) .. +31)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 64 consecutive fp32 columns: both 32-column loads are in flight before the single wait
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float* v) {
    uint32_t r[64];
#pragma unroll
    for (int h = 0; h < 2; ++h)
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[32 * h + 0]), "=r"(r[32 * h + 1]), "=r"(r[32 * h + 2]), "=r"(r[32 * h + 3]), "=r"(r[32 * h + 4]), "=r"(r[32 * h + 5]),
              "=r"(r[32 * h + 6]), "=r"(r[32 * h + 7]), "=r"(r[32 * h + 8]), "=r"(r[32 * h + 9]), "=r"(r[32 * h + 10]), "=r"(r[32 * h + 11]),
              "=r"(r[32 * h + 12]), "=r"(r[32 * h + 13]), "=r"(r[32 * h + 14]), "=r"(r[32 * h + 15]), "=r"(r[32 * h + 16]), "=r"(r[32 * h + 17]),
              "=r"(r[32 * h + 18]), "=r"(r[32 * h + 19]), "=r"(r[32 * h + 20]), "=r"(r[32 * h + 21]), "=r"(r[32 * h + 22]), "=r"(r[32 * h + 23]),
              "=r"(r[32 * h + 24]), "=r"(r[32 * h + 25]), "=r"(r[32 * h + 26]), "=r"(r[32 * h + 27]), "=r"(r[32 * h + 28]), "=r"(r[32 * h + 29]),
              "=r"(r[32 * h + 30]), "=r"(r[32 * h + 31])
            : "r"(taddr + 32u * h));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}

// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// relu + round-to-nearest bf16 + pack in ONE instruction (F2FP.RELU): the max() never touches the half-rate ALU pipe
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// fp16 variant for precision = 2 (11-bit significand instead of 8): relu + round + SATURATE to the largest finite half
// (F2FP.SATFINITE.RELU.F16), so an activation beyond 65504 clamps instead of turning the whole row into inf / NaN
__device__ __forceinline__ uint32_t pack_relu_f16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.satfinite.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
template <bool F16>
__device__ __forceinline__ uint32_t pack_relu_x2(float lo, float hi) {
    return F16 ? pack_relu_f16x2(lo, hi) : pack_relu_bf16x2(lo, hi);
}
// round + pack without the relu: bf16, or fp16 saturating to the largest finite half
template <bool F16>
__device__ __forceinline__ uint32_t pack_x2(float lo, float hi) {
    uint32_t d;
    if (F16) asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// ---- coalesced store of a 32 x 32 fp32 block held one-row-per-lane -----------------------------------
// After tcgen05.ld.32x32b every lane owns 32 consecutive columns of ITS row, so a direct store makes each
// instruction touch 32 different 128-byte lines (32 L1 wavefronts).  Staging the block through a padded
// per-warp shared-memory scratch ([32][33] floats) and reading it back with lane = column-quad turns every
// store instruction into four fully used 128-byte lines.  `row_ptr0` points at (row 0 of the block, column 0
// of the block); rows are `ld` floats apart; rows >= nrows and columns >= ncols are masked.
__device__ __forceinline__ void store_block_32x32(float* scratch, const float* v, float* row_ptr0, int64_t ld, int nrows, int ncols, int lane) {
#pragma unroll
    for (int j = 0; j < 32; ++j) scratch[lane * 33 + j] = v[j];
    __syncwarp();
    const int cq = (lane & 7) * 4;       // first of my four columns
    const int rsub = lane >> 3;          // 0..3
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(row_ptr0) & 15) == 0) && ((ld & 3) == 0) && (ncols == 32);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int r = i * 4 + rsub;
        const float a = scratch[r * 33 + cq], b = scratch[r * 33 + cq + 1], c = scratch[r * 33 + cq + 2], d = scratch[r * 33 + cq + 3];
        if (r < nrows) {
            float* dst = row_ptr0 + (int64_t)r * ld + cq;
            if (vec_ok) {
                *reinterpret_cast<float4*>(dst) = make_float4(a, b, c, d);
            } else {
                if (cq < ncols) dst[0] = a;
                if (cq + 1 < ncols) dst[1] = b;
                if (cq + 2 < ncols) dst[2] = c;
                if (cq + 3 < ncols) dst[3] = d;
            }
        }
    }
    __syncwarp();
}

// ---- descriptors ---------------------------------------------------------------------------------
// shared-memory matrix descriptor, SWIZZLE_128B, version 1 (Blackwell):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4 | [46,48) = 1 | [61,64) = 2
// K-major tile  (rows x 64 bf16, 128 B per row, 8-row swizzle groups of 1024 B): LBO unused (1), SBO = 1024
// MN-major tile (64 contiguous MN elements x K rows of 128 B): LBO = stride between 64-element MN chunks,
//                                                              SBO = 1024 (stride between 8-row K groups)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
}

// instruction descriptor for kind::f16 with bf16 A/B and fp32 D:
//   [4,6) D fmt = 1 (f32) | [7,10) A fmt = 1 (bf16) | [10,13) B fmt = 1 | [15] A MN-major | [16] B MN-major | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// kind::f16 operand formats (0 = fp16, 1 = bf16).  The descriptor has one field per operand, but B200 executes only EQUAL
// formats: fp16 x bf16 traps with "illegal instruction" (tests/test_gpu_umma.py::test_mixed_operand_formats pins this), so
// precision = 2 switches whole products to fp16 (11-bit significand) and scales the operands whose range needs it.
constexpr uint32_t FMT_F16 = 0u, FMT_BF16 = 1u;
__host__ __device__ constexpr uint32_t make_idesc_f16kind(int M, int N, bool a_mn, bool b_mn, uint32_t a_fmt, uint32_t b_fmt) {
    return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// ---- single-issuer helpers -----------------------------------------------------------------------
// The issuing warp keeps WARP-UNIFORM control flow (all 32 lanes run the loops and the barrier waits) and predicates the
// one-thread instructions on an elected lane inside the asm block.  With divergent `if (lane == 0)` code the compiler has to
// wrap every uniform-datapath instruction (UTCHMMA, UTCBAR, UTMALDG) in a waterfall loop (ELECT / R2UR / BRA.U.ANY, ~17 SASS
// instructions per MMA), and the serial latency of that single thread becomes the critical path of the whole CTA.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void mma_bf16_p(uint32_t leader, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void mma_commit_p(uint32_t leader, uint64_t* bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %1, 0;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(leader)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_p(uint32_t leader, uint64_t* bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %1, 0;\n"
        "@q mbarrier.arrive.shared::cta.b64 _, [%0];\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(leader)
        : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_p(uint32_t leader, uint64_t* bar, uint32_t bytes) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %2, 0;\n"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(bytes), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d_p(uint32_t leader, void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %6, 0;\n"
        "@q cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n"
        "}\n" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_store_3d_p(uint32_t leader, const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];\n"
        "}\n" ::"l"(reinterpret_cast<uint64_t>(map)),
        "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(leader)
        : "memory");
}
// L2 prefetch of a tile (no shared-memory destination): issued a few tiles ahead, it turns the HBM latency of the later
// cp.async.bulk.tensor load into an L2 hit when shared memory is too small for a deeper ring
__device__ __forceinline__ void tma_prefetch_3d_p(uint32_t leader, const CUtensorMap* map, int c0, int c1, int c2) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.b32 q, %4, 0;\n"
        "@q cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];\n"
        "}\n" ::"l"(reinterpret_cast<uint64_t>(map)),
        "r"(c0), "r"(c1), "r"(c2), "r"(leader)
        : "memory");
}
// SWIZZLE_128B descriptor with the 16-byte-unit address added to a precomputed base (address field: bits [0,14))
__device__ __forceinline__ uint64_t desc_add(uint64_t base_desc, uint32_t byte_offset) { return base_desc + (uint64_t)(byte_offset >> 4); }

}  // namespace umma
}  // namespace avd
