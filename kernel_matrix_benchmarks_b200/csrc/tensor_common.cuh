// Shared pieces of the tensor-core kernels (kprod_tensor.cu, kprod_tensor_pv.cu, kprod_tensor_pv16.cu): tcgen05 / TMA
// PTX wrappers, UMMA descriptors, kernel functions on (2u.v, |u|^2, |v|^2), the prepass, the wave schedule.
#pragma once
#include <cuda.h>

#include "kmb_common.cuh"

namespace kmb {
namespace tc {

constexpr int TM = 128;            // target rows per tile  (UMMA M, one TMEM lane per row)
constexpr int TK = 32;             // floats per K block = one 128-byte swizzle atom
constexpr int UMMA_K = 8;          // TF32: 32 bytes per instruction
constexpr int ELT_TF32 = 0;        // operand element: TF32 hi / lo planes (fp32 storage)
constexpr int ELT_F16 = 1;         // FP16 hi / lo planes of power-of-two scaled data (see tensor_prepass_f16)
constexpr int ELT_F16X1 = 2;       // the hi planes of ELT_F16 alone, one hi.hi MMA term (KMB_PATH_TENSOR_1XF16)

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// One lane of a converged warp.  The MMA-issuing warp walks its loop with all 32 lanes (uniform control
// flow, so ptxas keeps descriptors and TMEM addresses in uniform registers) and issues tcgen05.mma /
// tcgen05.commit under this predicate.  Wrapping the whole loop in `if (lane == 0)` instead makes every
// UTCHMMA a waterfall loop (ELECT + 4 R2UR + BRA.U.ANY): ~125 cycles per MMA, measured.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.b32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with the A operand read from tensor memory
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// tcgen05.wait::ld that the 16 destination registers of a preceding tcgen05.ld depend on.  A bare wait is only
// ordered against other volatile asm: ptxas / nvcc may (and did, in kprod_tensor_pv16) schedule arithmetic that
// consumes the loaded registers ABOVE it.  Passing the registers through the wait as "+r" operands pins every
// consumer below it.
#define KMB_DEP16(u)                                                                                                      \
    "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]), "+r"(u[8]), "+r"(u[9]), \
        "+r"(u[10]), "+r"(u[11]), "+r"(u[12]), "+r"(u[13]), "+r"(u[14]), "+r"(u[15])
__device__ __forceinline__ void tmem_ld_wait16(float* r) {
    uint32_t* u = reinterpret_cast<uint32_t*>(r);
    asm volatile("tcgen05.wait::ld.sync.aligned;" : KMB_DEP16(u)::"memory");
}
__device__ __forceinline__ void tmem_ld_dep16(float* r) {   // after tmem_ld_wait16: the same pin for 16 more registers
    uint32_t* u = reinterpret_cast<uint32_t*>(r);
    asm volatile("" : KMB_DEP16(u)::"memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const float* r) {
    const uint32_t* u = reinterpret_cast<const uint32_t*>(r);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
        "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
        : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = lane = row)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&r)[32]) {
    uint32_t* u = reinterpret_cast<uint32_t*>(r);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
          "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
          "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
        : "r"(taddr)
        : "memory");
    tmem_ld_wait16(r);
    tmem_ld_dep16(r + 16);
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 version 1): rows are 128 bytes,
// 8-row atoms are 1024 bytes apart; the tile base is 1024-byte aligned.
__device__ __forceinline__ uint64_t umma_desc_sw128(const void* smem_tile, int byte_offset) {
    const uint32_t addr = smem_u32(smem_tile) + byte_offset;
    return static_cast<uint64_t>((addr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t idesc_tf32(int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(TM >> 4) << 24);
}
// D = F32, A = B = F16, both K-major; m = 256 for the MMAs of a CTA pair (two CTAs x 128 rows)
__host__ __device__ constexpr uint32_t idesc_f16(int n, int m = TM) {
    return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// same MMA with the A operand read from tensor memory (lane = row, one 32-bit column per K element)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// registers -> 32 lanes x 32 consecutive columns of tensor memory
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const float (&r)[32]) {
    const uint32_t* u = reinterpret_cast<const uint32_t*>(r);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
        "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]), "r"(u[16]), "r"(u[17]), "r"(u[18]),
        "r"(u[19]), "r"(u[20]), "r"(u[21]), "r"(u[22]), "r"(u[23]), "r"(u[24]), "r"(u[25]), "r"(u[26]), "r"(u[27]),
        "r"(u[28]), "r"(u[29]), "r"(u[30]), "r"(u[31])
        : "memory");
}
// 16-column variants (column-split epilogues: each warp group owns a slice of the tile's columns)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, float* r) {
    uint32_t* u = reinterpret_cast<uint32_t*>(r);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// CPT (16 or 32) consecutive columns of this warp's 32 lanes <-> registers
template <int CPT>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&r)[CPT]) {
    static_assert(CPT % 16 == 0, "16-column chunks");
#pragma unroll
    for (int c = 0; c < CPT; c += 16) tmem_ld_32x16(taddr + c, r + c);
    tmem_ld_wait16(r);
#pragma unroll
    for (int c = 16; c < CPT; c += 16) tmem_ld_dep16(r + c);
}
template <int CPT>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const float (&r)[CPT]) {
#pragma unroll
    for (int c = 0; c < CPT; c += 16) tmem_st_32x16(taddr + c, r + c);
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster drive one tcgen05.mma of M = 256 ---------------------------
namespace pair {
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared-memory object of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
    uint32_t a;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
    return a;
}
// Arrive on a barrier of another CTA of the cluster.  Default semantics (.release.cta), as CUTLASS's ClusterBarrier
// does: what the waiter must see was published by tcgen05.wait::st + tcgen05.fence::before_thread_sync or is TMA
// traffic; an explicit .release.cluster here cost ~1300 cycles per arrival in kprod_tensor_pv16 (measured).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion bytes are counted on the LEADER CTA's barrier at the same offset as `bar`
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once the MMAs issued so far are done
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void umma2_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
}  // namespace pair

template <int KID>
__device__ __forceinline__ float kernel_from_parts(float s, float un, float vn) {
    // s = 2 u.v (log2-scaled data), so -(|u|^2 + |v|^2 - s) is the log2 of the Gaussian
    if constexpr (KID == KMB_KERNEL_GAUSSIAN) return ex2_approx((s - vn) - un);
    else {
        const float d2 = fmaxf((un + vn) - s, 0.f);  // bruteforce.py:21 / :10: maximum(sqdists, 0)
        if constexpr (KID == KMB_KERNEL_ABSOLUTE_EXPONENTIAL) return ex2_approx(-sqrt_approx(d2));
        else return rsqrt_approx(d2);
    }
}
template <int KID>
__device__ __forceinline__ float log2_kernel_from_parts(float s, float un, float vn) {
    if constexpr (KID == KMB_KERNEL_GAUSSIAN) return (s - vn) - un;
    else return -sqrt_approx(fmaxf((un + vn) - s, 0.f));
}

// The instantiation a kernel's tensor-path product launches.  The dot-exponential kernel has none of its own: its prepass
// (no centre, multiplier 1 on both planes, |u|^2 = |v|^2 = 0) makes S = log2(e) <x, y>, so the Gaussian epilogues'
// log2 k = S - |u|^2 - |v|^2 is log2 exp(<x, y>) exactly (DESIGN.md, "The dot-exponential kernel").
__host__ __device__ constexpr int epilogue_kid(int kid) { return kid == KMB_KERNEL_DOT_EXPONENTIAL ? KMB_KERNEL_GAUSSIAN : kid; }

// ---- host helpers shared by the tensor kernels (defined in kprod_tensor.cu) ----------------------
// (rows, cols) row-major plane of `elt` elements (ELT_TF32: fp32, otherwise FP16); box = one 128-byte swizzle atom of
// columns (32 floats / 64 halves) x box_rows rows, 128-byte swizzle, out-of-bounds reads as zero
int make_tensor_map(CUtensorMap* map, int elt, const void* base, long long rows, int cols, int box_rows);
// centre (column means of y), TF32 hi/lo split of A = 2 s (x - c) and B = s (y - c), squared norms
int tensor_prepass(const float* x, const float* y, int64_t N, int64_t M, int D, int Dp, int kid, float* center,
                   float* cpart, float* uh, float* ul, float* vh, float* vl, float* un, float* vn, cudaStream_t stream);
constexpr int CENTER_BLOCKS = 128;

// FP16 operands: centre (column means of y); p = power of two that brings max |s (point - c)| over x and y into [2^13, 2^14);
// FP16 hi / lo split of A = 2 s 2^p (x - c) and B = s 2^p (y - c) (Dp16 = D rounded up to 16 columns, zero
// padded), squared norms of s (point - c) in FP32; sscale[0] = 2^p, sscale[1] = 2^-2p (device).
// stats: 6 * CENTER_BLOCKS * D floats of scratch.
int tensor_prepass_f16(const float* x, const float* y, int64_t N, int64_t M, int D, int Dp16, int kid, float* center,
                       float* stats, float* sscale, void* uh, void* ul, void* vh, void* vl, float* un, float* vn,
                       cudaStream_t stream);

// L2-aware wave schedule shared by the tensor kernels (see kprod_tensor.cu): full waves of R row tiles x C CTAs,
// a last wave of R_last x C_last.
struct WavePlan { int R, C, W, R_last, C_last, slots_per_wave; long long partial_slots; };
void plan_waves(long long n_tiles, long long nsb, int grid, size_t row_tile_bytes, WavePlan* wp);

// Work of `unit` in wave w: row tile, source-block range [sb_lo, sb_hi), range index c of Cw.  The unit is a CTA, or the
// cluster of a CTA pair, whose wave plan counts pairs of row tiles (`tile` is then the pair's index).
//
// CAUSAL (KMB_FLAG_CAUSAL, row i sees sources j <= row_offset + i): the Cw ranges split only the nb_t source blocks of
// BLOCK sources that the unit's last row can see, nb_t = min(nsb, (row_offset + last row) / BLOCK + 1), so nothing above
// the diagonal is scheduled; a range is empty when nb_t < Cw.  The tiles of odd waves are taken in reverse order
// (serpentine): tile work grows with the tile index, and unit u then gets a light tile in one wave and a heavy one in the
// next.  Host and device: kmb_debug_causal_work checks the plan without a GPU.
struct WaveWork { int tile, sb_lo, sb_hi, c, Cw, tile_in_wave; };
template <bool CAUSAL = false, int BLOCK = 1, bool PAIR = false, class Params>
__host__ __device__ __forceinline__ bool wave_work(const Params& P, int w, int unit, WaveWork& ww) {
    const bool last = (w == P.W - 1);
    const int Rw = last ? P.R_last : P.R, Cw = last ? P.C_last : P.C;
    if (unit >= Rw * Cw) return false;
    ww.Cw = Cw;
    ww.tile_in_wave = unit / Cw;
    ww.c = unit - ww.tile_in_wave * Cw;
    if constexpr (CAUSAL) {
        if (w & 1) ww.tile_in_wave = Rw - 1 - ww.tile_in_wave;
        ww.tile = w * P.R + ww.tile_in_wave;
        const long long rows_end = static_cast<long long>(ww.tile + 1) * TM * (PAIR ? 2 : 1);
        const long long last_row = (rows_end < P.N ? rows_end : P.N) - 1;
        const long long nb_t = (P.row_offset + last_row) / BLOCK + 1;
        const long long nb = nb_t < P.nsb ? nb_t : P.nsb;
        ww.sb_lo = static_cast<int>(nb * ww.c / Cw);
        ww.sb_hi = static_cast<int>(nb * (ww.c + 1) / Cw);
    } else {
        ww.tile = w * P.R + ww.tile_in_wave;
        ww.sb_lo = static_cast<int>(static_cast<long long>(P.nsb) * ww.c / Cw);
        ww.sb_hi = static_cast<int>(static_cast<long long>(P.nsb) * (ww.c + 1) / Cw);
    }
    return true;
}

}  // namespace tc

// CTA pairs (cta_group::2) for an FP16-plane problem of n_tiles row tiles on `sms` SMs: at least two row tiles, unless
// KMB_TENSOR_PAIR=0 (read once per process).  Host logic only (kprod_tensor.cu; kprod_tensor and kprod_tensor_pv16).
bool tensor_use_pair(long long n_tiles, int sms);

// What a P.B kernel launches (kmb_debug_pv_plan, include/kmb_b200.h): the fields of its `out`, in this order.
enum {
    PVQ_FAMILY, PVQ_PAIR, PVQ_GRID, PVQ_STAGES, PVQ_KBLOCKS, PVQ_KSTEPS_LAST, PVQ_PASSES, PVQ_EB_FIRST, PVQ_EBP_FIRST,
    PVQ_EB_LAST, PVQ_EBP_LAST, PVQ_ROW_TILES, PVQ_SOURCE_BLOCKS, PVQ_R, PVQ_C, PVQ_W, PVQ_R_LAST, PVQ_C_LAST,
    PVQ_FLUSH_BLOCKS, PVQ_FIELDS
};
// the fields both P.B kernels derive alike: signal passes of max_eb columns (each padded to 32), tiling, wave plan
inline void pv_plan_fill(int E, int max_eb, long long n_tiles, long long nsb, const tc::WavePlan& w, long long* out) {
    const int passes = (E + max_eb - 1) / max_eb;
    const int eb_first = E < max_eb ? E : max_eb, eb_last = E - (passes - 1) * max_eb;
    out[PVQ_PASSES] = passes;
    out[PVQ_EB_FIRST] = eb_first;
    out[PVQ_EBP_FIRST] = (eb_first + 31) / 32 * 32;
    out[PVQ_EB_LAST] = eb_last;
    out[PVQ_EBP_LAST] = (eb_last + 31) / 32 * 32;
    out[PVQ_ROW_TILES] = n_tiles;
    out[PVQ_SOURCE_BLOCKS] = nsb;
    out[PVQ_R] = w.R;
    out[PVQ_C] = w.C;
    out[PVQ_W] = w.W;
    out[PVQ_R_LAST] = w.R_last;
    out[PVQ_C_LAST] = w.C_last;
}

// What a causal tensor kernel schedules (kmb_debug_causal_work, include/kmb_b200.h): the fields of its `out`, in this order.
enum { CWQ_FAMILY, CWQ_WAVES, CWQ_UNITS, CWQ_BLOCK, CWQ_TILE, CWQ_SB_LO, CWQ_SB_HI, CWQ_C, CWQ_CW, CWQ_FIELDS };
inline void causal_work_fill(int family, int waves, int units, int block, const tc::WaveWork* ww, long long* out) {
    out[CWQ_FAMILY] = family;
    out[CWQ_WAVES] = waves;
    out[CWQ_UNITS] = units;
    out[CWQ_BLOCK] = block;
    if (!ww) return;   // the unit has no row tile in this wave
    out[CWQ_TILE] = ww->tile;
    out[CWQ_SB_LO] = ww->sb_lo;
    out[CWQ_SB_HI] = ww->sb_hi;
    out[CWQ_C] = ww->c;
    out[CWQ_CW] = ww->Cw;
}
// as tensor_causal_work_debug (kprod_tensor.cuh), for kprod_tensor_pv16 (kprod_tensor_pv16.cu)
int tensor_pv16_causal_work_debug(int64_t N, int64_t M, int D, int E, int64_t row_offset, int sms, int smem_optin, int wave, int unit,
                                  long long out[CWQ_FIELDS]);

// E > 4 with D <= 128: second GEMM on the tensor cores (kprod_tensor_pv.cu)
bool tensor_pv_applicable(int D, int E);
// The plan of kprod_tensor_pv on a device of `sms` SMs with `smem_optin` bytes of opt-in shared memory per block (host
// logic only, the launcher's own): fills every PVQ_* field but PVQ_FAMILY.  Errors as the launcher's plan.
int tensor_pv_plan_debug(int64_t N, int64_t M, int D, int E, int sms, int smem_optin, long long out[PVQ_FIELDS]);
int tensor_pv_signal_block();     // signal columns per pass of kprod_tensor_pv
int tensor_pv16_signal_block();   // ... of kprod_tensor_pv16
int tensor_pv_workspace_bytes(int64_t N, int64_t M, int D, int E, size_t* bytes);
int tensor_pv_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E,
                      int kid, int flags, int64_t row_offset, void* workspace, size_t workspace_bytes,
                      cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1);


// the same with FP16 hi/lo operand planes (kprod_tensor_pv16.cu): Gaussian and exponential kernels
bool tensor_pv16_applicable(int D, int E, int kid);
// source blocks the P.B accumulators collect between two flushes: KMB_PV16_FLUSH_BLOCKS (read once per process), else 128
int tensor_pv16_flush_blocks();
// as tensor_pv_plan_debug, for kprod_tensor_pv16 (PVQ_PAIR: the CTA-pair kernel)
int tensor_pv16_plan_debug(int64_t N, int64_t M, int D, int E, int sms, int smem_optin, long long out[PVQ_FIELDS]);
int tensor_pv16_workspace_bytes(int64_t N, int64_t M, int D, int E, size_t* bytes);
// elt: tc::ELT_F16 (three-term S and P.B) or tc::ELT_F16X1 (hi.hi only; the lo planes are neither loaded nor written)
int tensor_pv16_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E, int kid,
                        int flags, int elt, int64_t row_offset, void* workspace, size_t workspace_bytes, cudaStream_t stream, cudaEvent_t ev0,
                        cudaEvent_t ev1, bool prepared);

// Head of the workspace of both FP16-plane kernels: everything the prepass writes from the points alone.  The layout
// depends on (N, M, D) only, so that it survives from fit() to query() whatever the signal width turns out to be.
struct F16PointsLayout {
    int Dp;          // D rounded up to 16
    long long Mv;    // entries of |v|^2: M rounded up to 256, the tail filled with 3.4e38 (padded sources weigh nothing)
    size_t off_center, off_stats, off_sscale, off_uh, off_ul, off_vh, off_vl, off_un, off_vn, end;
};
void f16_points_layout(int64_t N, int64_t M, int D, F16PointsLayout* L);
int f16_points_prepass(const float* x, const float* y, int64_t N, int64_t M, int D, int kid, const F16PointsLayout& L,
                       char* ws, cudaStream_t stream);

}  // namespace kmb
