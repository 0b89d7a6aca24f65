// The bf16x3 toolkit of the tcgen05 kernels (sm_100a): tensor memory (TMEM) allocation and access, tcgen05.mma on
// shared-memory operands, mbarriers, the bulk-copy engine (cp.async.bulk) and the proxy fences between them, plus what every
// kernel of the family builds on top: the split operand format, the three-MMA product, tile staging, the dropout hash and
// the CTA set-up / teardown.  Device-only; everything is inline PTX (no CUTLASS).
//
// Contractions: tcgen05.mma kind::f16 on bf16 operands with fp32 accumulation in TMEM.  Every fp32 operand x is split as
// x = hi + lo (+ <= 2^-18 |x|), hi = bf16(x), lo = bf16(x - hi), and a product is issued as three MMAs hi*hi + lo*hi + hi*lo
// ("bf16x3"): measured 5e-6 .. 2e-5 on predictions / gradients of the whole model against the fp64 oracle.
// Operands live in shared memory in the 16-bit PANEL layout
//     element (row r, col c)  ->  plane + (c / 8) * (R * 16) + r * 16 + (c % 8) * 2        (hi plane, lo plane)
// which the tensor core reads in both orientations (SWIZZLE_NONE canonical layouts, checked by tools/micro/umma_layout_probe_bf16):
//   K-major  (rows = M/N index, cols = K): SBO = 128, LBO = R*16     -> forward GEMMs   D = A W^T
//   MN-major (rows = K index, cols = M/N): SBO = R*16, LBO = 128     -> weight gradients dW = dY^T A  (K = the tile's rows)
//                                                                       and data gradients dA = dY W with the UNtransposed weight
// so one copy of each activation / weight serves the forward, the data-gradient and the weight-gradient product.
#pragma once
#include "mmx_common.cuh"

namespace mmx {
namespace tc5 {

// CTA shape: four warps per TMEM lane quarter; they split a row's 8-column chunks between them
constexpr int kHalves = 4;
constexpr int kCtaThreads = 128 * kHalves;

MMX_D uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------ mbarrier
MMX_D void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make mbarrier.init visible to the async proxy (TMA / tcgen05.commit arrive on it)
MMX_D void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
MMX_D void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
MMX_D void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
MMX_D bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a mis-programmed pipeline must end the kernel (and fail the test) instead of hanging the GPU.  `*abort_flag`
// (shared) is set on timeout; callers check it after the kernel's join points.
MMX_D bool mbar_wait(uint64_t* bar, uint32_t parity, volatile int* abort_flag) {
    for (uint32_t it = 0; it < (1u << 22); ++it) {
        if (mbar_try_wait(bar, parity)) return true;
        if (it > 64 && *abort_flag) return false;
    }
    *abort_flag = 1;
    return false;
}

// ------------------------------------------------------------------------------------------ proxy / tcgen05 fences
// generic-proxy writes to shared memory (st.shared) -> visible to the async proxy (tcgen05.mma operand reads, bulk stores)
MMX_D void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
MMX_D void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
MMX_D void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
MMX_D void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
MMX_D void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------ TMEM allocation (one full warp)
template <int COLS>
MMX_D void tmem_alloc(uint32_t* slot_in_smem) {
    static_assert(COLS == 32 || COLS == 64 || COLS == 128 || COLS == 256 || COLS == 512, "TMEM columns: power of two >= 32");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
MMX_D void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

// ------------------------------------------------------------------------------------------ descriptors and MMA issue
// shared-memory matrix descriptor, SWIZZLE_NONE, Blackwell version field = 1
MMX_D uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}
// instruction descriptor: kind::f16, bf16 x bf16 -> fp32
MMX_HD uint32_t idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem], issued by ONE thread
MMX_D void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all MMAs issued so far by this thread arrive on `bar` when they have completed (implies fence::before_thread_sync)
MMX_D void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------ TMEM <-> registers (whole warp)
// Lane l of warp w (w % 4 = lane quarter) touches TMEM lane 32*(w%4) + l, columns [col, col + N).
MMX_D uint32_t tmem_addr(uint32_t base, int lane_quarter, int col) { return base + ((uint32_t)(lane_quarter * 32) << 16) + (uint32_t)col; }

MMX_D void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
                 : "r"(taddr));
    v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
    v[4] = __uint_as_float(r4); v[5] = __uint_as_float(r5); v[6] = __uint_as_float(r6); v[7] = __uint_as_float(r7);
}
MMX_D void tmem_st8(uint32_t taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}

// ------------------------------------------------------------------------------------------ bulk copies (TMA engine, 1-D)
// global -> shared, completes `bytes` on the mbarrier; addresses and size multiples of 16
MMX_D void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global (bulk async-group)
MMX_D void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
MMX_D void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the source shared memory of all committed bulk stores has been read (buffer reusable)
MMX_D void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
MMX_D void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------------------------------ CTA set-up and teardown
// start of a tcgen05 CTA: nbars mbarriers (arrival count 1), the abort flag cleared, TM_COLS TMEM columns allocated by warp 0
template <int TM_COLS>
MMX_D void cta_begin(uint64_t* bars, int nbars, volatile int* abortf, uint32_t* tslot, int tid) {
    if (tid == 0) {
        for (int i = 0; i < nbars; ++i) mbar_init(&bars[i], 1);
        *abortf = 0;
        fence_mbar_init();
    }
    if ((tid >> 5) == 0) tmem_alloc<TM_COLS>(tslot);
}
// end of a tcgen05 CTA: bulk stores complete, a timed-out wait counted in *abort_count, TMEM freed.  Contains a CTA barrier.
template <int TM_COLS>
MMX_D void cta_end(volatile int* abortf, int* abort_count, uint32_t tmem, int tid) {
    if ((tid >> 5) == 0) bulk_wait_all0();
    if (tid == 0 && *abortf) atomicAdd(abort_count, 1);
    tc_fence_before();
    __syncthreads();
    if ((tid >> 5) == 0) tmem_dealloc<TM_COLS>(tmem);
}

// ------------------------------------------------------------------------------------------ programmatic dependent launch
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start while its predecessor in the stream is
// still running: everything before pdl_wait() (barrier / TMEM set-up, staging of the weights -- nothing the predecessor
// writes) overlaps the predecessor's tail; pdl_wait() returns once the predecessor has completed and its writes are visible.
// pdl_launch_dependents() lets the NEXT kernel's CTAs be scheduled as soon as this kernel's CTAs have all started.
MMX_D void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
MMX_D void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------ dropout masks of the tcgen05 family
// A dropout site is a [rows][W] tensor; chunk c8 of row `row` covers its columns [8*c8, 8*c8+8).  Four counter-based 32-bit
// hashes (lowbias32 finaliser over counter ^ key) give 16 random bits per element; an element is kept iff its field >=
// thresh16.  The key mixes (seed, site, step).  tests/masks_np.py is the numpy twin (bit-exact; pinned by a GPU test), which
// lets the parity tests hand the very same masks to the oracle.
MMX_HD uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
    return x;
}
MMX_HD uint32_t drop_key(uint32_t seed_lo, uint32_t seed_hi, uint32_t site, uint32_t step) {
    return mix32(seed_lo ^ mix32(seed_hi ^ mix32(site * 0x9E3779B1u + step)));
}
// bit j of the result = keep element 8*c8 + j
MMX_HD uint32_t keep8(uint32_t key, uint32_t thresh16, uint32_t row, uint32_t W8, uint32_t c8) {
    const uint32_t base = (row * W8 + c8) * 4u;
    uint32_t bits = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t i = 0; i < 4; ++i) {
        const uint32_t r = mix32((base + i) ^ key);
        bits |= ((r & 0xffffu) >= thresh16 ? 1u : 0u) << (2 * i);
        bits |= ((r >> 16) >= thresh16 ? 1u : 0u) << (2 * i + 1);
    }
    return bits;
}

// ------------------------------------------------------------------------------------------ split operands, panel layout
// Geometry of the operands at padded width KP: activation tiles of 128 rows and KP x KP weights, hi plane then lo plane.
template <int KP>
struct Panels {
    static constexpr uint32_t PS = 128 * 16;                 // activation panel: 128 rows x 16 B
    static constexpr uint32_t PLANE = (KP / 8) * PS;
    static constexpr uint32_t BUF = 2 * PLANE;               // hi plane + lo plane
    static constexpr uint32_t WPS = KP * 16;                 // weight panel: KP rows x 16 B
    static constexpr uint32_t WPLANE = (KP / 8) * WPS;
    static constexpr uint32_t WBUF = 2 * WPLANE;
};
MMX_HD uint32_t up128(uint32_t v) { return (v + 127u) / 128u * 128u; }
MMX_HD uint32_t umax(uint32_t a, uint32_t b) { return a > b ? a : b; }
// byte offset of element (row, col) in one plane whose panels are panel_bytes long
MMX_HD uint32_t panel_off(int row, int col, uint32_t panel_bytes) {
    return (uint32_t)(col >> 3) * panel_bytes + (uint32_t)row * 16u + (uint32_t)(col & 7) * 2u;
}

MMX_D uint32_t pack_bf16x2(float lo_elem, float hi_elem) {   // lo_elem -> bits [0,16) (lower address)
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
    return r;
}
struct Split { uint32_t hi, lo; };
// two fp32 values -> bf16x2 hi and lo words (a in the lower half)
MMX_D Split split2(float a, float b) {
    const uint32_t h = pack_bf16x2(a, b);
    return {h, pack_bf16x2(a - __uint_as_float(h << 16), b - __uint_as_float(h & 0xffff0000u))};
}
// one fp32 value -> bf16 hi and lo in bits [0,16)
MMX_D Split split1(float v) {
    const uint32_t h = pack_bf16x2(v, 0.0f) & 0xffffu;
    return {h, pack_bf16x2(v - __uint_as_float(h << 16), 0.0f) & 0xffffu};
}
// 8 fp32 values -> 8 bf16 "hi" (16 bytes) + 8 bf16 "lo" (16 bytes)
MMX_D void split8(const float (&v)[8], uint4& hi, uint4& lo) {
    Split s[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) s[i] = split2(v[2 * i], v[2 * i + 1]);
    hi = make_uint4(s[0].hi, s[1].hi, s[2].hi, s[3].hi);
    lo = make_uint4(s[0].lo, s[1].lo, s[2].lo, s[3].lo);
}

// 16-bit panel operand, rows = M/N index, cols = K index; k0 = first column of this K=16 step
MMX_D uint64_t dk(uint32_t plane, uint32_t panel_bytes, int k0) { return smem_desc(plane + (uint32_t)(k0 >> 3) * panel_bytes, panel_bytes, 128u); }
// 16-bit panel operand, rows = K index, cols = M/N index; r0 = first row of this K=16 step
MMX_D uint64_t dmn(uint32_t plane, uint32_t panel_bytes, int r0) { return smem_desc(plane + (uint32_t)r0 * 16u, 128u, panel_bytes); }

// D (+)= A B^T with split operands: hi*hi + lo*hi + hi*lo.  A: buffer (planes a_hi, a_lo, panel bytes a_ps), B likewise.
// A_MN / B_MN: orientation of each operand; ksteps K=16 steps.  Issued by ONE thread.
template <int A_MN, int B_MN>
MMX_D void gemm3(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t a_ps, uint32_t b_hi, uint32_t b_lo, uint32_t b_ps, int N,
                 int ksteps, bool accumulate_first) {
    const uint32_t id = idesc_bf16(128, N, A_MN, B_MN);
#pragma unroll 1
    for (int s = 0; s < ksteps; ++s) {
        const int k0 = 16 * s;
        const uint64_t ah = A_MN ? dmn(a_hi, a_ps, k0) : dk(a_hi, a_ps, k0);
        const uint64_t al = A_MN ? dmn(a_lo, a_ps, k0) : dk(a_lo, a_ps, k0);
        const uint64_t bh = B_MN ? dmn(b_hi, b_ps, k0) : dk(b_hi, b_ps, k0);
        const uint64_t bl = B_MN ? dmn(b_lo, b_ps, k0) : dk(b_lo, b_ps, k0);
        mma_f16(d_tmem, ah, bh, id, (s > 0 || accumulate_first) ? 1u : 0u);
        mma_f16(d_tmem, al, bh, id, 1u);
        mma_f16(d_tmem, ah, bl, id, 1u);
    }
}

// ------------------------------------------------------------------------------------------ staging
// bulk copy of a tile of activation rows global -> shared (issued by warp 0), completion on `bar`
template <int VEC>
MMX_D void stage_in(float* S, const float* g, size_t row0, int nrows, int H, int pitch, uint64_t* bar, int lane) {
    if (lane == 0) mbar_expect_tx(bar, (uint32_t)nrows * H * 4u);
    __syncwarp();
    if (VEC == 2) {
        if (lane == 0) bulk_g2s(S, g + row0 * H, (uint32_t)nrows * H * 4u, bar);
    } else {
        for (int r = lane; r < nrows; r += 32) bulk_g2s(S + (size_t)r * pitch, g + (row0 + r) * H, (uint32_t)H * 4u, bar);
    }
}
template <int VEC>
MMX_D void stage_out(float* g, const float* S, size_t row0, int nrows, int H, int pitch, int lane) {
    if (VEC == 2) {
        if (lane == 0) bulk_s2g(g + row0 * H, S, (uint32_t)nrows * H * 4u);
    } else {
        for (int r = lane; r < nrows; r += 32) bulk_s2g(g + (row0 + r) * H, S + (size_t)r * pitch, (uint32_t)H * 4u);
    }
    bulk_commit();
}

// 8 consecutive columns [k0, k0+8) of a staged row; columns >= H read as zero (H % VEC == 0)
template <int VEC>
MMX_D void ld8(const float* srow, int k0, int H, float (&v)[8]) {
#pragma unroll
    for (int j = 0; j < 8; j += VEC) {
        if (k0 + j < H) {
            if (VEC == 4) { const float4 t = *reinterpret_cast<const float4*>(srow + k0 + j); v[j] = t.x; v[j + 1] = t.y; v[j + 2] = t.z; v[j + 3] = t.w; }
            else { const float2 t = *reinterpret_cast<const float2*>(srow + k0 + j); v[j] = t.x; v[j + 1] = t.y; }
        } else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) v[j + i] = 0.0f;
        }
    }
}
template <int VEC>
MMX_D void st8(float* srow, int k0, int H, const float (&v)[8]) {
#pragma unroll
    for (int j = 0; j < 8; j += VEC) {
        if (k0 + j < H) {
            if (VEC == 4) *reinterpret_cast<float4*>(srow + k0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            else *reinterpret_cast<float2*>(srow + k0 + j) = make_float2(v[j], v[j + 1]);
        }
    }
}
MMX_D void ld8s(const float* p, float (&v)[8]) {   // 8 floats from a 16-byte aligned shared array
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

MMX_D void put_chunk(uint8_t* buf, uint32_t plane_bytes, uint32_t ps, int row, int c8, const float (&t)[8]) {
    uint4 hi, lo;
    split8(t, hi, lo);
    *reinterpret_cast<uint4*>(buf + c8 * ps + row * 16) = hi;
    *reinterpret_cast<uint4*>(buf + plane_bytes + c8 * ps + row * 16) = lo;
}

// stage one weight matrix W[rows][cols] (row-major, optional per-column scale) into a weight buffer (panel layout, KP x KP,
// zero padded; the buffer must have been zeroed)
template <int KP>
MMX_D void stage_weight(uint8_t* wbuf, const float* W, int rows, int cols, const float* colscale, int tid) {
    using P = Panels<KP>;
    if ((cols & 1) == 0) {
        const int n2 = rows * cols / 2;
        for (int i = tid; i < n2; i += kCtaThreads) {
            const int e = 2 * i, r = e / cols, c = e - r * cols;
            float2 v = *reinterpret_cast<const float2*>(W + e);
            if (colscale) { v.x *= colscale[c]; v.y *= colscale[c + 1]; }
            const Split s = split2(v.x, v.y);
            const uint32_t off = panel_off(r, c, P::WPS);
            *reinterpret_cast<uint32_t*>(wbuf + off) = s.hi;
            *reinterpret_cast<uint32_t*>(wbuf + P::WPLANE + off) = s.lo;
        }
    } else {
        for (int i = tid; i < rows * cols; i += kCtaThreads) {
            const int r = i / cols, c = i - r * cols;
            float v = W[i];
            if (colscale) v *= colscale[c];
            const Split s = split1(v);
            const uint32_t off = panel_off(r, c, P::WPS);
            *reinterpret_cast<uint16_t*>(wbuf + off) = (uint16_t)s.hi;
            *reinterpret_cast<uint16_t*>(wbuf + P::WPLANE + off) = (uint16_t)s.lo;
        }
    }
}

// sum the halves' partial sums of a row (every half gets the totals).  Contains a CTA barrier.
MMX_D void row_exchange(float* ex, int half, int prow, float& a, float& b) {
    ex[(0 * kHalves + half) * 128 + prow] = a;
    ex[(1 * kHalves + half) * 128 + prow] = b;
    __syncthreads();
    a = 0.0f; b = 0.0f;
#pragma unroll
    for (int i = 0; i < kHalves; ++i) { a += ex[(0 * kHalves + i) * 128 + prow]; b += ex[(1 * kHalves + i) * 128 + prow]; }
}

}  // namespace tc5
}  // namespace mmx
