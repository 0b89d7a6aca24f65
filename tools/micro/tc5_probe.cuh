// tcgen05 primitives only the probes in this directory use: kind::tf32 MMAs on the 4-byte panel layout (one panel per
// 4-column chunk, R rows of 16 bytes) and the wider TMEM accesses.  The kernels of the package use the bf16x3 toolkit
// (motionmixerconv_b200/csrc/mmx_tc5.cuh) instead.
#pragma once
#include "../../motionmixerconv_b200/csrc/mmx_tc5.cuh"

namespace mmx {
namespace tc5 {

// 4-byte panel operand, rows = M/N index, cols = K index; k0 = first column of this K=8 step (multiple of 8)
MMX_D uint64_t desc_kmajor(uint32_t base, uint32_t panel_bytes, int k0) {
    return smem_desc(base + (uint32_t)(k0 >> 2) * panel_bytes, panel_bytes, 128u);
}
// 4-byte panel operand, rows = K index, cols = M/N index; r0 = first row of this K=8 step (multiple of 8), c0 = first M/N column
MMX_D uint64_t desc_mnmajor(uint32_t base, uint32_t panel_bytes, int r0, int c0) {
    return smem_desc(base + (uint32_t)(c0 >> 2) * panel_bytes + (uint32_t)r0 * 16u, 128u, panel_bytes);
}
// instruction descriptor: kind::tf32, fp32 accumulate, dense
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem], kind::tf32 (ONE thread)
MMX_D void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]   (A: one row per lane, one K element per 32-bit column; K-major only)
MMX_D void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

MMX_D void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
MMX_D void tmem_st4(uint32_t taddr, float a, float b, float c, float d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(__float_as_uint(a)),
                 "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d))
                 : "memory");
}

}  // namespace tc5
}  // namespace mmx
