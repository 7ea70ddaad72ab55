// wb_tc.cuh -- tcgen05 / TMEM / mbarrier / bulk-copy primitives for the tensor-core decoder kernels (sm_100a).
//
// Operand layouts (no swizzle, "interleaved" canonical form of the UMMA shared-memory descriptor):
//   core matrix = 8 rows x 16 bytes (8 fp16), stored contiguously (128 B).
//   SAMPLE TILE  [128 samples x C features], C multiple of 8, "slab" layout:
//        element (s, f) at byte (f/8)*2048 + s*16 + (f%8)*2            (one slab = 8 features of all 128 samples)
//     as K-major  A (M = sample,  K = feature): LBO = 2048 (next 8 features), SBO = 128  (next 8 samples)
//     as MN-major A/B (MN = feature, K = sample): SBO = 2048 (next 8 features), LBO = 128 (next 8 samples)
//   WEIGHT PACK  W[N x K] (nn.Linear weight, N = out, K = in), N multiple of 8, K multiple of 8:
//        element (n, k) at byte (k/8)*(N*16) + n*16 + (k%8)*2
//     as K-major  B (N = out, K = in):  LBO = N*16, SBO = 128
//     as MN-major B (N' = in, K' = out) for data-grad:  SBO = N*16, LBO = 128
// Accumulators: D[128 x N] fp32 in TMEM, row r <-> TMEM lane r, column n <-> TMEM column (base + n).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout) --------------------------------
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);            // start address  [0,14)
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;       // leading byte offset [16,30)
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;       // stride byte offset  [32,46)
    d |= (uint64_t)1 << 46;                                  // descriptor version 1 (Blackwell) [46,48)
    return d;                                                // base_offset 0, lbo_mode 0, layout SWIZZLE_NONE
}
// ---- instruction descriptor for kind::f16, fp16 x fp16 -> fp32 (cute::UMMA::InstrDescriptor) -----------------
__host__ __device__ __forceinline__ uint32_t tc_idesc(int M, int N, int a_mn_major, int b_mn_major)
{
    return (1u << 4)                       // c_format = F32
         | (0u << 7) | (0u << 10)          // a_format = b_format = F16
         | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16)
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// advance a descriptor's start address by `bytes` (multiple of 16; the 14-bit address field must not wrap: smem < 256 KB)
__device__ __forceinline__ uint64_t tc_desc_adv(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }
// one lane of a converged warp (warp-uniform context: lets ptxas keep descriptors in uniform registers)
__device__ __forceinline__ uint32_t tc_elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(pred));
    return pred;
}
// A operand read from TENSOR MEMORY (dense fp16: lane = row, two halfs per 32-bit column, K-major only), B from shared memory.
// Used by the TMEM-A forward kernel (F == 2 'cat' hash grids; see wb_shade_tc.cu): activations never touch shared memory.
__device__ __forceinline__ void tc_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// make all previously issued MMAs of this thread arrive on an mbarrier when they complete
__device__ __forceinline__ void tc_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tensor core operand fetch)
__device__ __forceinline__ void tc_fence_smem_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM allocation (one warp, power-of-two columns >= 32) --------------------------------------------------
__device__ __forceinline__ void tc_tmem_alloc(uint32_t* dst_smem, uint32_t ncols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(tc_smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_tmem_dealloc(uint32_t taddr, uint32_t ncols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane (warp w of a warpgroup reads lanes 32*(w%4) .. +31)
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float v[16])
{
    uint32_t r[16];
    __syncwarp();                                   // warp-collective (.sync.aligned): reconverge after predicated epilogue code
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 consecutive fp32 columns in one instruction
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float v[32])
{
    uint32_t r[32];
    __syncwarp();
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// named barrier over `nthreads` threads (sub-tile groups of a CTA synchronise independently of each other)
__device__ __forceinline__ void tc_group_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}
// 64 consecutive fp32 columns in one instruction (one wait instead of four round trips)
__device__ __forceinline__ void tc_ld64(uint32_t taddr, float v[64])
{
    uint32_t r[64];
    __syncwarp();
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}
// zero 16 consecutive fp32 columns of this thread's TMEM lane (warp-collective)
__device__ __forceinline__ void tc_st16_zero(uint32_t taddr)
{
    const uint32_t z = 0;
    __syncwarp();
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};\n"
                 :: "r"(taddr), "r"(z) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// store 4 / 16 consecutive 32-bit columns of this thread's TMEM lane (warp-collective); tc_st_wait() before the hand-over
__device__ __forceinline__ void tc_st4(uint32_t taddr, uint4 v)
{
    __syncwarp();
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};\n" :: "r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t r[16])
{
    __syncwarp();
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
                 :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                    "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tc_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- mbarrier ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(tc_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(tc_smem_u32(bar)), "r"(parity) : "memory");
    }
}
// TMA bulk copy global -> shared (bytes multiple of 16, both addresses 16-byte aligned); SASS: UBLKCP
__device__ __forceinline__ void tc_bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(tc_smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(tc_smem_u32(bar)) : "memory");
}

// ---- fp16 packing ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tc_pack2(float a, float b)
{
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// {relu(lo), relu(hi)} -> packed fp16x2 in ONE instruction (F2FP.RELU): the whole hidden-layer activation
__device__ __forceinline__ uint32_t tc_pack2_relu(float lo, float hi)
{
    uint32_t d;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// byte offset of (sample s, feature f) in a slab tile
__device__ __forceinline__ uint32_t tc_slab_off(int s, int f) { return (uint32_t)((f >> 3) * 2048 + s * 16 + (f & 7) * 2); }
