// kprod_tensor_pv16: a_i = sum_j k(x_i, y_j) b_j for 16 < D <= 128 and E > 4, Gaussian and exponential kernels --
// both contractions on the tensor cores with FP16 hi / lo operand planes (config C4: exponential-kernel
// attention, N = M = 262144, D = E = 64).  Same algorithm as kprod_tensor_pv.cu (TF32 planes), re-shaped after
// tools/ubench_umma.cu: a 128 x 64 x 8 SS MMA takes 60 cycles for 32 cycles of math, a 128 x 128 x 16 one 75 for
// 64, and kind::f16 does twice the work of kind::tf32 per instruction.
//
//   S = 2 u.v^T   (exponential kernel: 2 u.v - |u|^2 - |v|^2, the squared norms as one more BF16 K step -- extra_k)
//                 128 rows x 128 sources per block; tcgen05.mma kind::f16, three-term split
//                 (lo.hi + hi.lo + hi.hi), A = u tile (hi, lo) resident in shared memory for the whole row
//                 tile, B = v blocks streamed by TMA, FP32 accumulator in TMEM (SST = 3 stages)
//   P = k(S)      8 epilogue warps = NG = 2 column groups x 4 TMEM lane quarters.  Group g owns columns [64g, 64g+64)
//                 of every S block and runs its OWN online-softmax stream over those sources: tcgen05.ld S, log2
//                 of the kernel, a running reference exponent per (row, group) (lazy rescale of the group's O
//                 when the maximum outgrows it by 2^8, so P <= 2^8 fits FP16 and rows whose kernel values all
//                 underflow FP32 still normalise), P = 2^(log2 k - ref) split into FP16 hi + lo, packed two per
//                 32-bit column and stored IN PLACE over the thread's own S columns (tcgen05.st).  No
//                 block-level synchronisation between epilogue warps inside a row tile.  Gaussian kernel: one fused
//                 pass per block with the reference the row already has (kFused); the two phases only when it moves.
//   O_g += P_g.B  tcgen05.mma with A = P from TMEM (hi, lo), B = transposed signal block (FP16 hi, lo, scaled per
//                 signal column by a power of two) from shared memory; one accumulator O_g (128 x E) per column
//                 group, kept in TMEM for the whole row tile; the NG of them are merged (weights 2^(ref_g - ref)) when
//                 the row tile ends -- every thread can read all four because TMEM lanes are rows.
//
// TMEM columns: S/P stages at 128 a, a < SST | O_g at 128 SST + 64 g  (3 x 128 + 2 x 64 = 512).
// S(n + SST) overwrites stage n % SST after PV(n) has been issued (tensor-pipe order): the issue order is
// S(0) .. S(SST-1), PV(0), S(SST), PV(1), ..., so the tensor side runs SST - 1 blocks ahead of the epilogue.
// Work split: the wave schedule of kprod_tensor.cu -- every CTA of a wave walks the SAME source blocks at the same
// time (all of them when there are at least as many row tiles as CTAs), so v and b blocks come from L2.
// TERMS = 1 (KMB_PATH_TENSOR_1XF16): S = hi.hi and O_g += P_hi.B_hi, one MMA per K step each.  The lo planes of u, v and
// the signal are neither loaded nor counted on the barriers, the epilogue writes P hi only and sums the weights as the
// MMA sees them (P rounded to FP16); the extra K step, the online maximum and the flushes are those of TERMS = 3.
#include <algorithm>
#include <cstdlib>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "tensor_common.cuh"

namespace kmb {
namespace pv16 {

using namespace tc;

constexpr int TNS = 128;               // sources per S block
constexpr int SLOT_BYTES = 32768;      // ring slot: v block of one K block (hi 16 KB | lo 16 KB) or one signal block
                                       // (CTA pairs: each CTA holds half of either, 16 KB slots)
constexpr int A_TILE_BYTES = TM * 128; // 16 KB: 128 rows of one 128-byte K block
constexpr int PANEL_BYTES = 64 * 128;  // signal: 64 signal columns x 64 sources (one swizzle atom wide)
// Shape of the epilogue (build-time; rounds 1 and 2 began with NG = 4, SST = 2, two phases per block):
//   NG  column groups = online-softmax streams (4 warps each, one per TMEM lane quarter), own accumulator O_g each
//   SST S / P stages in tensor memory
// 512 TMEM columns = SST * 128 (S / P) + NG * 64 (O_g).  With two stages the epilogue of block n + 2 cannot start before
// P(n) of the SLOWEST group + P.B(n) + S(n + 2); with three the tensor side is always a block ahead.  What was measured on
// the way (16 warps in pairs sharing a group, the groups skewed or staggered by a barrier, parts of the kernel removed,
// SM clock inside the kernel): tools/experiments/README.md, profiles/r2_pv16_*.
#ifndef KMB_PV16_NG
#define KMB_PV16_NG 2
#endif
#ifndef KMB_PV16_SST
#define KMB_PV16_SST 3
#endif
#ifndef KMB_PV16_FUSED
#define KMB_PV16_FUSED 2
#endif
#ifndef KMB_PV16_FHSPLIT
#define KMB_PV16_FHSPLIT 1
#endif
#ifndef KMB_PV16_EXTRAK
#define KMB_PV16_EXTRAK 1
#endif
constexpr int NG = KMB_PV16_NG;        // epilogue column groups (4 warps each)
constexpr int SST = KMB_PV16_SST;      // S / P stages
constexpr int kFused = KMB_PV16_FUSED;   // one pass per block with the row's current reference: 0 never, 1 Gaussian, 2 both kernels
// |u|^2 + |v|^2 through the tensor cores: one more K step (BF16: FP32's exponent range) whose operands are three BF16 pieces of
// -2^2p |u_i|^2 against ones and ones against three pieces of -2^2p |v_j|^2, so that the accumulator holds (2 u.v - |u|^2 - |v|^2) / sscale
// = -d2 / sscale and the epilogue needs neither the shared-memory line of |v|^2 nor a packed add per pair.  0 never, 1 exponential
// kernel, 2 both kernels.
// hi / lo split of a weight: 1 = hi by one F2FP (round to nearest), -lo = hi - w by the mixed-precision FHADD of sm_100a (f16 + f32),
// the lo plane stored negated and the P_lo.B_hi MMA negating its A operand (instruction descriptor bit 13): 4 instructions per two
// weights; 0 = mask + packed subtract + two F2FP: 5.
constexpr bool kFhSplit = KMB_PV16_FHSPLIT != 0;
constexpr int kExtraK = KMB_PV16_EXTRAK;
template <int KID>
__host__ __device__ constexpr bool extra_k() { return kExtraK == 2 || (kExtraK == 1 && KID == KMB_KERNEL_ABSOLUTE_EXPONENTIAL); }
constexpr int CPT = TNS / NG;          // S columns per epilogue thread
constexpr int EPI_WARPS = 4 * NG;
constexpr int EPI_THREADS = 32 * EPI_WARPS;
constexpr int THREADS = 64 + EPI_THREADS;
constexpr int TMEM_COLS = 512;
constexpr int MAX_EB = 64;             // signal columns per pass
constexpr int COL_S = 0, COL_O = SST * TNS;
static_assert(COL_O + NG * MAX_EB <= TMEM_COLS, "S / P stages and the O_g must fit 512 tensor-memory columns");
static_assert(CPT % 32 == 0 && SST >= 2 && SST <= 4, "epilogue shape");
constexpr float kLazyRescale = 8.f;    // rescale O only when the row maximum outgrew the reference by 2^8
constexpr int PS = MAX_EB + 2;         // partial record: O row, sum of weights, reference exponent
// The tensor cores add into the FP32 accumulator with truncation, not round-to-nearest: every accumulating MMA shrinks
// O_g by ~2^-25 of its magnitude, and a row tile at M = 262144 makes 12288 of them per group -- measured 2.4e-4 relative
// (every row alike, the sum of weights on the CUDA cores does not shrink with it) against the 1e-4 the path is held to.
// So O_g only collects kFlushBlocks source blocks; then the epilogue adds it (round-to-nearest, L2 reductions the thread
// does not wait for) to a per-(CTA, group) FP32 accumulator in global memory and the next P.B starts from zero.
// Measured at C4 (M = 262144): flush every 2048 blocks (= never) 2.4e-4, every 32 blocks 3.6e-6 at +6 % time (the L2
// reductions of 148 CTAs arrive together).  With NG = 2 a group makes 12 accumulating MMAs per block: every 128 blocks
// (1536 MMAs) 3.0e-5, every 64 blocks 1.4e-5 at +0.3 % (exponential) / +1.5 % (Gaussian) -- profiles/r2_pv16_variants_ab.jsonl.
constexpr int kFlushBlocks = 128;        // default of Params::flush_blocks

struct Params {
    const float* un;
    const float* vn;
    const float* sscale;       // [1] = 2^-2p: S = sscale[1] * accumulator
    const float* binv;         // (Ep) 2^-q_e: undoes the per-column scale of the signal planes
    float* out;
    float* partial;
    float* olong;              // grid x NG x MAX_EB x TM: long accumulators of the O_g, [column][row] (see kFlushBlocks)
    int* tile_counter;
    long long N, M;
    int E, e0, eb, ebp;        // this pass covers signal columns e0 .. e0+eb-1; ebp = eb rounded up to 32
    int n_tiles, nsb, kblocks, ksteps_last, stages, ep_rows, flush_blocks;
    int R, C, W, R_last, C_last, slots_per_wave;
};

// `unit`: the CTA (single-CTA kernel) or the cluster (CTA pairs: the wave plan then counts pairs of row tiles)
struct WaveWork { int tile, sb_lo, sb_hi, c, Cw, tile_in_wave; };
__device__ __forceinline__ bool wave_work(const Params& P, int w, int cta, WaveWork& ww) {
    const bool last = (w == P.W - 1);
    const int Rw = last ? P.R_last : P.R, Cw = last ? P.C_last : P.C;
    if (cta >= Rw * Cw) return false;
    ww.Cw = Cw;
    ww.tile_in_wave = cta / Cw;
    ww.c = cta - ww.tile_in_wave * Cw;
    ww.tile = w * P.R + ww.tile_in_wave;
    ww.sb_lo = static_cast<int>(static_cast<long long>(P.nsb) * ww.c / Cw);
    ww.sb_hi = static_cast<int>(static_cast<long long>(P.nsb) * (ww.c + 1) / Cw);
    return true;
}

__device__ __forceinline__ void umma_f16_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d),
                 "l"(a), "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
__device__ __forceinline__ void umma_f16_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n" ::"r"(d),
                 "r"(a), "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
__host__ __device__ constexpr uint32_t idesc_f16(int n) {   // D = F32, A = B = F16, K-major
    return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(TM >> 4) << 24);
}
// two floats -> one 32-bit word of two halves: `even` in bits [0,16), `odd` in bits [16,32)
__device__ __forceinline__ uint32_t pack_half2(float even, float odd) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(odd), "f"(even));
    return r;
}

// T = -log2 k / t_scale<KID> for two sources at once (packed FP32: FFMA2 / FADD2), from the raw accumulators:
// s_raw sscale = 2 u.v on log2-scaled data, w = |u|^2 + |v|^2
template <int KID>
__device__ __forceinline__ constexpr float t_scale() { return KID == KMB_KERNEL_GAUSSIAN ? 1.f : 0.70710678118654752f; }
__device__ __forceinline__ float sqrt_mufu(float x) {   // one MUFU.SQRT (x >= 0)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// shared-memory accesses in the shared state space (a pointer derived from the aligned dynamic base is generic to nvcc)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
template <int KID>
__device__ __forceinline__ float2 neg_log2_kernel2(float2 s_raw, float2 nsscale, float2 w) {
    const float2 d2 = fma2(s_raw, nsscale, w);          // log2(e) |x - y|^2 (Gaussian) or (log2(e) |x - y|)^2
    if constexpr (KID == KMB_KERNEL_GAUSSIAN) return d2;
    else {
        // bruteforce.py:21: sqrt(maximum(sqdists, 0)).  d2 + |d2| = 2 max(d2, 0) is ONE packed instruction (FADD2 takes
        // |.| on a packed operand; there is no packed max), the factor sqrt(2) leaves with t_scale in the FFMA2 that
        // forms the exponent; sqrt.approx.ftz is a single MUFU.SQRT on sm_100a (sqrt(0) = 0: no clamp away from zero).
        // Padded sources (|v|^2 = 3.39e38): 2 d2 = +inf, sqrt = +inf, exponent -inf, weight 0 -- no NaN on the way.
        const float2 r = add2(d2, make_float2(fabsf(d2.x), fabsf(d2.y)));
        return make_float2(sqrt_mufu(r.x), sqrt_mufu(r.y));
    }
}

// PAIR: two CTAs of a cluster (cta_group::2) work on two adjacent row tiles and the same source blocks: every MMA is
// 256 rows tall (half as many instructions per row tile -- the issuing warp is what bounds the single-CTA kernel),
// each CTA streams half of every v block (64 sources) and half of every signal block (32 signal columns), the leader
// CTA issues, tcgen05.commit multicasts to both CTAs' barriers and the peer's epilogue warps arrive on the leader's.
template <int KID, bool NORM, bool PAIR, int TERMS>
__device__ __forceinline__ void pv16_body(const CUtensorMap& map_ah, const CUtensorMap& map_al, const CUtensorMap& map_bh,
                                          const CUtensorMap& map_bl, const CUtensorMap& map_sh, const CUtensorMap& map_sl,
                                          const CUtensorMap& map_ue, const CUtensorMap& map_ve, const Params& P) {
    constexpr bool XK = extra_k<KID>();                            // the squared norms come out of the tensor cores
    constexpr int SLOT = PAIR ? SLOT_BYTES / 2 : SLOT_BYTES;       // V: hi | lo halves of the slot
    constexpr int PANEL = PAIR ? PANEL_BYTES / 2 : PANEL_BYTES;    // signal: 4 panels (hi 0, hi 1, lo 0, lo 1)
    constexpr bool LO = TERMS == 3;                                // the lo planes take part
    static_assert(TERMS == 3 || TERMS == 1, "three-term or one-term split");
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
    unsigned char* u_region = smem;                                   // kblocks x [A hi 16 KB | A lo 16 KB] (+ the norm tile)
    unsigned char* u_extra = u_region + P.kblocks * 2 * A_TILE_BYTES; // XK: 128 rows x [3 pieces of -2^2p |u|^2, 1, 1, 1, 0 ..] (BF16)
    unsigned char* ring = u_extra + (XK ? A_TILE_BYTES : 0);          // stages x 32 KB
    float* vline = reinterpret_cast<float*>(ring + P.stages * SLOT);    // EPI_WARPS x 2 x CPT: per-warp |v|^2 lines
    float* refbuf = vline + EPI_WARPS * 2 * CPT;                               // NG x TM: per-group reference exponents
    float* ksbuf = refbuf + NG * TM;                                           // NG x TM: per-group sums of weights
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ksbuf + NG * TM);
    uint64_t* empty_bar = full_bar + P.stages;
    uint64_t* acc_full = empty_bar + P.stages;     // [SST] S(n) complete in stage n % SST
    uint64_t* p_ready = acc_full + SST;            // [SST] P(n) stored in stage n % SST
    uint64_t* pv_done = p_ready + SST;             // [SST] PV(n) complete
    uint64_t* u_full = pv_done + SST;
    uint64_t* u_free = u_full + 1;
    uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(u_free + 1);
    int* s_flag = reinterpret_cast<int*>(tmem_base_smem + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = PAIR ? pair::cluster_ctarank() : 0;   // 0 = leader (issues the MMAs)
    const int cta = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);   // unit of the wave plan
    const int ST = P.stages;
    constexpr int NCTA = PAIR ? 2 : 1;

    if (tid == 0) {
        for (int s = 0; s < ST; ++s) { mbar_init(&full_bar[s], NCTA); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < SST; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&p_ready[a], NCTA * EPI_WARPS); mbar_init(&pv_done[a], 1); }
        mbar_init(u_full, NCTA);
        mbar_init(u_free, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        if constexpr (PAIR) pair::tmem_alloc2(tmem_base_smem, TMEM_COLS);
        else tmem_alloc(tmem_base_smem, TMEM_COLS);
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) pair::cluster_sync_all();   // the peer's barriers exist before anything arrives on them
    tc_fence_after();
    // barrier-side helpers: where TMA bytes are counted / how the producers arm a full barrier
    auto arm_full = [&](uint64_t* bar, uint32_t bytes_per_cta) {   // elected lane only
        if constexpr (PAIR) {
            if (rank == 0) mbar_arrive_expect_tx(bar, 2 * bytes_per_cta);
            else pair::mbar_arrive_cluster(pair::map_to_cta(bar, 0));
        } else {
            mbar_arrive_expect_tx(bar, bytes_per_cta);
        }
    };
    auto load2d = [&](void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
        if constexpr (PAIR) pair::tma_load_2d_pair(dst, map, c0, c1, pair::map_to_cta(bar, 0));
        else tma_load_2d(dst, map, c0, c1, bar);
    };
    auto commit = [&](uint64_t* bar) {
        if constexpr (PAIR) pair::umma2_commit_both(bar);
        else umma_commit(bar);
    };
    const uint32_t tmem_base = *tmem_base_smem;

    if (warp == 0) {
        // ------------------------------------ TMA producer ------------------------------------
        // all 32 lanes walk the loop (uniform control flow); one elected lane issues (see elect_one)
        // ring position as (slot, phase) counters: `it % stages` with a run-time divisor is ~30 instructions and a MUFU.RCP
        // that queues behind the epilogue's exponentials
        uint32_t seg = 0;
        int slot = 0;
        uint32_t ring_phase = 0;
        auto ring_next = [&]() { if (++slot == ST) { slot = 0; ring_phase ^= 1u; } };
        auto emit_signal = [&](int sb) {   // one slot: hi panels 0, 1 | lo panels 0, 1
            // slab sb, signal column e0 (CTA pairs: this CTA's half of the pass's signal columns)
            const int row0 = sb * P.ep_rows + P.e0 + (PAIR ? static_cast<int>(rank) * (P.ebp / 2) : 0);
            mbar_wait(&empty_bar[slot], ring_phase ^ 1u);
            unsigned char* dst = ring + slot * SLOT;
            if (elect_one()) {
                constexpr uint32_t panels = LO ? 4u : 2u;
                arm_full(&full_bar[slot], PAIR ? panels * (P.ebp / 2) * 128u : panels * PANEL_BYTES);
                load2d(dst + 0 * PANEL, &map_sh, 0, row0, &full_bar[slot]);
                load2d(dst + 1 * PANEL, &map_sh, 64, row0, &full_bar[slot]);
                if constexpr (LO) {
                    load2d(dst + 2 * PANEL, &map_sl, 0, row0, &full_bar[slot]);
                    load2d(dst + 3 * PANEL, &map_sl, 64, row0, &full_bar[slot]);
                }
            }
            __syncwarp();
            ring_next();
        };
        // the signal block of P.B(n - (SST - 1)) is consumed after the v block of S(n): a queue of SST - 1 source blocks
        int pend[SST - 1];
#pragma unroll
        for (int q = 0; q < SST - 1; ++q) pend[q] = -1;
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!wave_work(P, w, cta, ww)) continue;
            // new row tile: (re)load the resident u tile once the last S of the previous tile has read it
            mbar_wait(u_free, (seg & 1) ^ 1);
            const int my_row0 = (PAIR ? ww.tile * 2 + static_cast<int>(rank) : ww.tile) * TM;
            if (elect_one()) {
                arm_full(u_full, (P.kblocks * (LO ? 2 : 1) + (XK ? 1 : 0)) * A_TILE_BYTES);
                for (int kb = 0; kb < P.kblocks; ++kb) {
                    load2d(u_region + (kb * 2 + 0) * A_TILE_BYTES, &map_ah, kb * 64, my_row0, u_full);
                    if constexpr (LO) load2d(u_region + (kb * 2 + 1) * A_TILE_BYTES, &map_al, kb * 64, my_row0, u_full);
                }
                if constexpr (XK) load2d(u_extra, &map_ue, 0, my_row0, u_full);
            }
            __syncwarp();
            ++seg;
            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb) {
                for (int kb = 0; kb < P.kblocks; ++kb) {
                    mbar_wait(&empty_bar[slot], ring_phase ^ 1u);
                    unsigned char* dst = ring + slot * SLOT;
                    const int src0 = sb * TNS + (PAIR ? static_cast<int>(rank) * (TNS / 2) : 0);   // pairs: this CTA's 64 sources
                    if (elect_one()) {
                        arm_full(&full_bar[slot], LO ? SLOT : SLOT / 2);
                        load2d(dst, &map_bh, kb * 64, src0, &full_bar[slot]);
                        if constexpr (LO) load2d(dst + SLOT / 2, &map_bl, kb * 64, src0, &full_bar[slot]);
                    }
                    __syncwarp();
                    ring_next();
                }
                if constexpr (XK) {   // the block's norm tile: its own ring slot (half of it used)
                    mbar_wait(&empty_bar[slot], ring_phase ^ 1u);
                    const int src0 = sb * TNS + (PAIR ? static_cast<int>(rank) * (TNS / 2) : 0);
                    if (elect_one()) {
                        arm_full(&full_bar[slot], SLOT / 2);
                        load2d(ring + slot * SLOT, &map_ve, 0, src0, &full_bar[slot]);
                    }
                    __syncwarp();
                    ring_next();
                }
                if (pend[0] >= 0) emit_signal(pend[0]);   // consumed by PV(n - (SST - 1)), issued after S(n)
#pragma unroll
                for (int q = 0; q + 1 < SST - 1; ++q) pend[q] = pend[q + 1];
                pend[SST - 2] = sb;
            }
        }
#pragma unroll
        for (int q = 0; q < SST - 1; ++q)
            if (pend[q] >= 0) emit_signal(pend[q]);
    } else if (warp == 1 && rank == 0) {
        // ------------------------------------- MMA issuer (pairs: the leader CTA's) -------------------------------------
        // All 32 lanes walk the loop and wait on the barriers; one elected lane issues (see elect_one).
        // Order: S(0), .., S(SST - 1), PV(0), S(SST), PV(1), ...
        uint32_t n = 0, seg = 0;
        int slot = 0;                 // ring position as counters (see the producer)
        uint32_t ring_phase = 0;
        auto ring_next = [&]() { if (++slot == ST) { slot = 0; ring_phase ^= 1u; } };
        const uint32_t d_o = tmem_base + COL_O;
        constexpr uint32_t m_bits = PAIR ? (static_cast<uint32_t>(256 >> 4) << 24) : (static_cast<uint32_t>(TM >> 4) << 24);
        const uint32_t idesc_s = (1u << 4) | (static_cast<uint32_t>(TNS >> 3) << 17) | m_bits;
        const uint32_t idesc_o = (1u << 4) | (static_cast<uint32_t>(P.ebp >> 3) << 17) | m_bits;
        auto mma_ss = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
            if constexpr (PAIR) pair::umma2_f16(d, a, b, idesc, acc);
            else umma_f16_ss(d, a, b, idesc, acc);
        };
        auto mma_ts = [&](uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
            if constexpr (PAIR) pair::umma2_f16_ts(d, a, b, idesc, acc);
            else umma_f16_ts(d, a, b, idesc, acc);
        };
#ifdef KMB_PV16_TIMING
        long long macc[6] = {0, 0, 0, 0, 0, 0}, mprev = clock64();
#define KMB_M(i) do { const long long t_ = clock64(); macc[i] += t_ - mprev; mprev = t_; } while (0)
#else
#define KMB_M(i) do { } while (0)
#endif
        auto issue_pv = [&](uint32_t m, bool from_zero) {   // from_zero: the O_g were flushed (or the tile starts)
            const int a = m % SST;
            KMB_M(0);
            mbar_wait(&p_ready[a], (m / SST) & 1);
            KMB_M(1);
            mbar_wait(&full_bar[slot], ring_phase);
            tc_fence_after();
            KMB_M(2);
            const unsigned char* sg = ring + slot * SLOT;
            const uint32_t p_base = tmem_base + COL_S + a * TNS;
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < TNS / 16; ++k) {   // 16 sources per instruction; column group g = k / (CPT / 16)
                    constexpr int KPG = CPT / 16;      // instructions (of each of the three terms) per group
                    const int g = k / KPG, kk = k % KPG, panel = k >> 2, koff = (k & 3) * 32;
                    const uint64_t bh = umma_desc_sw128(sg + panel * PANEL, koff);
                    const uint64_t bl = umma_desc_sw128(sg + (2 + panel) * PANEL, koff);
                    const uint32_t a_hi = p_base + g * CPT + kk * 8, a_lo = a_hi + CPT / 2;
                    const uint32_t d_g = d_o + g * MAX_EB;
                    if constexpr (LO) {
                        mma_ts(d_g, a_lo, bh, idesc_o | (kFhSplit ? (1u << 13) : 0u), !(from_zero && kk == 0));   // (-) P_lo . B_hi
                        mma_ts(d_g, a_hi, bl, idesc_o, 1);
                        mma_ts(d_g, a_hi, bh, idesc_o, 1);
                    } else {
                        mma_ts(d_g, a_hi, bh, idesc_o, !(from_zero && kk == 0));
                    }
                }
                commit(&empty_bar[slot]);
                commit(&pv_done[a]);
            }
            __syncwarp();
            ring_next();
        };
        uint32_t first_bits = 0;   // bit q: block n - q starts its O_g from zero
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!wave_work(P, w, cta, ww)) continue;
            mbar_wait(u_full, seg & 1);
            ++seg;
            int until_flush = 0;   // blocks until the epilogue flushes the O_g again (a countdown: no division in the loop)
            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++n) {
                const bool first = (until_flush == 0);
                until_flush = first ? P.flush_blocks - 1 : until_flush - 1;
                first_bits = (first_bits << 1) | (first ? 1u : 0u);
                const int a = n % SST;   // stage a held P(n - SST): PV(n - SST) was issued in the previous iteration
                const uint32_t d_s = tmem_base + COL_S + a * TNS;
                for (int kb = 0; kb < P.kblocks; ++kb) {
                    KMB_M(3);
                    mbar_wait(&full_bar[slot], ring_phase);
                    tc_fence_after();
                    KMB_M(4);
                    const unsigned char* bt = ring + slot * SLOT;
                    const unsigned char* at = u_region + kb * 2 * A_TILE_BYTES;
                    const int ksteps = (kb == P.kblocks - 1) ? P.ksteps_last : 4;
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (k < ksteps) {
                                const uint64_t ah = umma_desc_sw128(at, k * 32);
                                const uint64_t al = umma_desc_sw128(at + A_TILE_BYTES, k * 32);
                                const uint64_t bh = umma_desc_sw128(bt, k * 32);
                                const uint64_t bl = umma_desc_sw128(bt + SLOT / 2, k * 32);
                                if constexpr (LO) {
                                    mma_ss(d_s, al, bh, idesc_s, (kb | k) != 0);
                                    mma_ss(d_s, ah, bl, idesc_s, 1);
                                    mma_ss(d_s, ah, bh, idesc_s, 1);
                                } else {
                                    mma_ss(d_s, ah, bh, idesc_s, (kb | k) != 0);
                                }
                            }
                        }
                        commit(&empty_bar[slot]);
                    }
                    __syncwarp();
                    ring_next();
                }
                if constexpr (XK) {   // S -= (|u|^2 + |v|^2) / sscale: one BF16 MMA, K = 16
                    mbar_wait(&full_bar[slot], ring_phase);
                    tc_fence_after();
                    if (elect_one()) {
                        constexpr uint32_t bf16_ab = (1u << 7) | (1u << 10);   // A and B formats: BF16
                        mma_ss(d_s, umma_desc_sw128(u_extra, 0), umma_desc_sw128(ring + slot * SLOT, 0), idesc_s | bf16_ab, 1);
                        commit(&empty_bar[slot]);
                    }
                    __syncwarp();
                    ring_next();
                }
                const bool last_of_tile = (sb + 1 == ww.sb_hi);
                if (elect_one()) {
                    commit(&acc_full[a]);
                    if (last_of_tile) commit(u_free);   // last S of this row tile
                }
                __syncwarp();
                if (n >= static_cast<uint32_t>(SST - 1)) issue_pv(n - (SST - 1), ((first_bits >> (SST - 1)) & 1u) != 0);
            }
        }
        // drain: the last SST - 1 blocks (n = number of blocks issued)
#pragma unroll
        for (int q = SST - 1; q >= 1; --q)
            if (n >= static_cast<uint32_t>(q)) issue_pv(n - q, ((first_bits >> (q - 1)) & 1u) != 0);
#ifdef KMB_PV16_TIMING
        if (blockIdx.x == 0 && lane == 0) {
            for (int i = 0; i < 5; ++i) P.out[8 + i] = static_cast<float>(macc[i]) / n;
        }
#endif
    } else if (warp >= 2) {
        // -------------------------------------- epilogue --------------------------------------
        const int et = tid - 64;
        const int lane_group = warp & 3;             // TMEM lane quarter this warp may touch
        const int cg = (warp - 2) >> 2;              // column group = online-softmax stream (own reference, sum, O_g)
        const int col0 = cg * CPT;                   // first S column of this thread
        const int row_in_tile = lane_group * 32 + lane;
        const uint32_t lane_addr = static_cast<uint32_t>(lane_group * 32) << 16;
        const uint32_t o_mine = tmem_base + COL_O + cg * MAX_EB + lane_addr;   // this group's accumulator
        const float sscale = __ldg(P.sscale + 1);
        uint32_t n = 0;   // blocks this CTA has processed (all waves)
#ifdef KMB_PV16_TIMING
        long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = clock64();
        const long long t_start = tprev;
        unsigned long long ns_start;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_start));
#define KMB_T(i) do { const long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } while (0)
#else
#define KMB_T(i) do { } while (0)
#endif
        auto wait_pv = [&](uint32_t m) {   // PV(m) has read P(m) and finished accumulating into the O_g
            mbar_wait(&pv_done[m % SST], (m / SST) & 1);
            tc_fence_after();
        };

        // |v|^2 of this group's CPT sources: lane l fetches sources l, l + 32, .. of the NEXT block (coalesced loads, a
        // block ahead of their use), parks them in the warp's shared-memory line and every lane reads the line back as float4s
        constexpr int VQ = CPT / 32;
        const uint32_t my_line_addr = smem_u32(vline + (warp - 2) * 2 * CPT);
        float vn_next[VQ];
#pragma unroll
        for (int q = 0; q < VQ; ++q) vn_next[q] = 0.f;
        auto fetch_vn = [&](int sb) {   // padded to whole blocks with 3.4e38
#pragma unroll
            for (int q = 0; q < VQ; ++q) vn_next[q] = __ldg(P.vn + static_cast<long long>(sb) * TNS + col0 + q * 32 + lane);
        };
        bool primed = false;
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!wave_work(P, w, cta, ww)) continue;
            const int tile = PAIR ? ww.tile * 2 + static_cast<int>(rank) : ww.tile;
            const long long row = static_cast<long long>(tile) * TM + row_in_tile;
            const bool row_ok = row < P.N;
            const float un = row_ok ? __ldg(P.un + row) : 0.f;
            float ksum = 0.f, ref = -INFINITY;   // this group's stream
            // long accumulator of this thread's O_g row: zero, then only ever touched by this thread until the merge
            float* olong = P.olong + (static_cast<size_t>(blockIdx.x) * NG + cg) * (MAX_EB * TM) + row_in_tile;
            for (int c = 0; c < P.ebp; ++c) __stcg(olong + c * TM, 0.f);
            auto flush_o = [&]() {   // olong += O_g (after the last P.B into it has completed)
                for (int c0 = 0; c0 < P.ebp; c0 += 16) {
                    float o[16];
                    tmem_ld_cols<16>(o_mine + c0, o);
#pragma unroll
                    for (int c = 0; c < 16; ++c) atomicAdd(olong + (c0 + c) * TM, o[c]);   // RED: nothing to wait for
                }
            };
            if (!XK && !primed) {
                fetch_vn(ww.sb_lo);
                primed = true;
            }
            // first block of the next wave this CTA works in (for the prefetch across the tile boundary)
            int sb_next_tile = -1;
            {
                WaveWork wn;
                for (int w2 = w + 1; w2 < P.W && sb_next_tile < 0; ++w2)
                    if (wave_work(P, w2, cta, wn)) sb_next_tile = wn.sb_lo;
            }

            int until_flush = P.flush_blocks;   // blocks until this thread moves its O_g row to the long accumulator
            bool flushed = false;               // ... which has happened at least once in this tile
            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++n) {
                const int a = n % SST;
                const uint32_t st_addr = tmem_base + COL_S + a * TNS + col0 + lane_addr;
                const uint32_t line = my_line_addr + (n & 1) * (CPT * 4);
                if constexpr (!XK) {
#pragma unroll
                    for (int q = 0; q < VQ; ++q) sts32(line + (q * 32 + lane) * 4, vn_next[q]);
                    const int sbn = (sb + 1 < ww.sb_hi) ? sb + 1 : sb_next_tile;
                    if (sbn >= 0) fetch_vn(sbn);
                    __syncwarp();
                }
                KMB_T(0);
                mbar_wait(&acc_full[a], (n / SST) & 1);
                tc_fence_after();
                KMB_T(1);
                float2 t2[CPT / 2];   // S as pairs of sources, then T = -log2 k / t_scale
                tmem_ld_cols<CPT>(st_addr, reinterpret_cast<float(&)[CPT]>(t2));
                KMB_T(2);

                // Padded sources need no branch: their |v|^2 is 3.39e38, so their exponent is -3.39e38 or -inf and their
                // weight an exact zero whatever the reference is.
                constexpr bool kRowTermOut = (KID == KMB_KERNEL_GAUSSIAN) && !XK;   // the Gaussian t leaves the row's |u|^2 out
                const float2 nss2 = make_float2(-sscale, -sscale), un2 = make_float2(un, un);
                // XK: the accumulator is -d2 / sscale.  Gaussian: t = -sscale S.  Exponential: |S| - S = 2 max(d2, 0) / sscale in one
                // packed add, T = its MUFU.SQRT, t = sqrt(sscale / 2) T -- the factor leaves with the FFMA2 that forms the exponent.
                const float xk_tscale = (KID == KMB_KERNEL_GAUSSIAN) ? 1.f : sqrtf(0.5f * sscale);
                auto xk_t = [&](float2 sv) -> float2 {
                    if constexpr (KID == KMB_KERNEL_GAUSSIAN) return mul2(sv, nss2);
                    else {
                        const float2 r = add2(make_float2(fabsf(sv.x), fabsf(sv.y)), make_float2(-sv.x, -sv.y));
                        return make_float2(sqrt_mufu(r.x), sqrt_mufu(r.y));
                    }
                };
                uint32_t ph[CPT / 2], pl[CPT / 2];       // P = 2^(log2 k - ref): FP16 hi / lo, two sources per TMEM column
                float2 kacc = make_float2(0.f, 0.f);     // two-level sum of the weights (see kprod_direct.cuh)
                auto weight = [&](int c, float2 e) {     // exponent -> weight -> planes (2 MUFU.EX2 + 7 instructions)
                    const float2 pw = make_float2(ex2_approx(e.x), ex2_approx(e.y));
                    if constexpr (!LO) {
                        // one plane: the row's sum takes the weights the MMA multiplies, P rounded to FP16
                        ph[c] = pack_half2(pw.x, pw.y);
                        if constexpr (NORM) kacc = add2(kacc, __half22float2(*reinterpret_cast<const __half2*>(&ph[c])));
                        return;
                    }
                    if constexpr (NORM) kacc = add2(kacc, pw);   // the plain product never divides by the sum of the weights
                    if constexpr (kFhSplit) {
                        const uint32_t hi2 = pack_half2(pw.x, pw.y);
                        float nlx, nly;   // hi - w: exact in FP32 (hi is within 2^-11 of w)
                        asm("{\n.reg .b16 l, h;\nmov.b32 {l, h}, %2;\nsub.rn.f32.f16 %0, l, %3;\nsub.rn.f32.f16 %1, h, %4;\n}"
                            : "=f"(nlx), "=f"(nly)
                            : "r"(hi2), "f"(pw.x), "f"(pw.y));
                        ph[c] = hi2;
                        pl[c] = pack_half2(nlx, nly);   // -lo
                    } else {
                        // 11 significant bits: exact in FP16
                        const float2 h = make_float2(__uint_as_float(__float_as_uint(pw.x) & 0xffffe000u),
                                                     __uint_as_float(__float_as_uint(pw.y) & 0xffffe000u));
                        const float2 l = sub2(pw, h);
                        ph[c] = pack_half2(h.x, h.y);
                        pl[c] = pack_half2(l.x, l.y);
                    }
                };
                bool done = false;
                if constexpr (kFused == 2 || (kFused == 1 && KID == KMB_KERNEL_GAUSSIAN)) {
                    // One pass with the reference the row already has: S -> exponent -> weight, the largest exponent on the
                    // side.  The lazy reference moves in a handful of blocks per row tile; only then (or while a row has
                    // no reference yet) is the block redone in two phases below, from S, which is still in tensor memory.
                    // Gaussian kernel: the two phases leave the MUFU pipe idle through the whole log2 k phase (C4 shape:
                    // 45.1 -> 42.7 ms).  Exponential kernel: sqrt -> exponent -> ex2 in one chain was slower than the two
                    // MUFU-bound phases while the chain began with the |v|^2 line (52.3 against 51.4 ms); with the norms out of
                    // the tensor cores (extra_k) it is level to slightly ahead (49.8 against 50.2 ms) and used for both
                    // (profiles/r2_pv16_fused_ab.jsonl, r2_pv16_extra_k_ab.jsonl).
                    if (__all_sync(0xffffffffu, ref != -INFINITY)) {
                        const float nref = kRowTermOut ? -ref - un : -ref;
                        const float2 nref2 = make_float2(nref, nref), ss2 = make_float2(sscale, sscale);
                        const float2 nts2 = XK ? make_float2(-xk_tscale, -xk_tscale) : make_float2(-t_scale<KID>(), -t_scale<KID>());
                        float emax = -INFINITY, emax_b = -INFINITY;   // two chains
#pragma unroll
                        for (int c = 0; c < CPT / 4; ++c) {
                            float4 vq = make_float4(0.f, 0.f, 0.f, 0.f);
                            if constexpr (!XK) vq = lds128(line + c * 16);   // broadcast read of the warp's line
                            const float2 wa = make_float2(vq.x, vq.y), wb = make_float2(vq.z, vq.w);
                            float2 ea, eb;
                            if constexpr (XK) {
                                if constexpr (KID == KMB_KERNEL_GAUSSIAN) {
                                    ea = fma2(t2[2 * c], ss2, nref2);
                                    eb = fma2(t2[2 * c + 1], ss2, nref2);
                                } else {
                                    ea = fma2(xk_t(t2[2 * c]), nts2, nref2);
                                    eb = fma2(xk_t(t2[2 * c + 1]), nts2, nref2);
                                }
                            } else if constexpr (KID == KMB_KERNEL_GAUSSIAN) {
                                ea = fma2(t2[2 * c], ss2, sub2(nref2, wa));
                                eb = fma2(t2[2 * c + 1], ss2, sub2(nref2, wb));
                            } else {
                                ea = fma2(neg_log2_kernel2<KID>(t2[2 * c], nss2, add2(wa, un2)), nts2, nref2);
                                eb = fma2(neg_log2_kernel2<KID>(t2[2 * c + 1], nss2, add2(wb, un2)), nts2, nref2);
                            }
                            emax = fmaxf(fmaxf(emax, ea.x), ea.y);
                            emax_b = fmaxf(fmaxf(emax_b, eb.x), eb.y);
                            weight(2 * c, ea);
                            weight(2 * c + 1, eb);
                        }
                        const bool need = fmaxf(emax, emax_b) > kLazyRescale;
                        done = !__any_sync(0xffffffffu, need);
                        if (!done) {
                            tmem_ld_cols<CPT>(st_addr, reinterpret_cast<float(&)[CPT]>(t2));
                            kacc = make_float2(0.f, 0.f);
                        }
                    }
                }
                KMB_T(3);
                if (!done) {
                    // t = -log2 of the kernel values (packed pairs) and their minimum over this thread's columns
                    float tmin = INFINITY, tmin_b = INFINITY;   // two chains
#pragma unroll
                    for (int c = 0; c < CPT / 4; ++c) {
                        float2 ta, tb;
                        if constexpr (XK) {
                            ta = xk_t(t2[2 * c]);
                            tb = xk_t(t2[2 * c + 1]);
                        } else {
                            const float4 vq = lds128(line + c * 16);   // broadcast read of the warp's line
                            // Gaussian: |u|^2 is the same for the whole row, so it is left out of t here and added to the
                            // block minimum / subtracted with the reference exponent below (one FADD2 per four values less)
                            const float2 wa = make_float2(vq.x, vq.y), wb = make_float2(vq.z, vq.w);
                            ta = neg_log2_kernel2<KID>(t2[2 * c], nss2, KID == KMB_KERNEL_GAUSSIAN ? wa : add2(wa, un2));
                            tb = neg_log2_kernel2<KID>(t2[2 * c + 1], nss2, KID == KMB_KERNEL_GAUSSIAN ? wb : add2(wb, un2));
                        }
                        t2[2 * c] = ta;
                        t2[2 * c + 1] = tb;
                        tmin = fminf(fminf(tmin, ta.x), ta.y);
                        tmin_b = fminf(fminf(tmin_b, tb.x), tb.y);
                    }
                    tmin = fminf(tmin, tmin_b);
                    const float tsc = XK ? xk_tscale : t_scale<KID>();                 // t = tsc T
                    const float cm = kRowTermOut ? -(tmin + un) : -tmin * tsc;         // largest log2 k of the block
                    // lazy rescale: keep the reference exponent unless the maximum outgrew it by 2^8
                    bool need = false;
                    if (ref == -INFINITY) ref = cm;   // nothing but zero weights so far
                    else need = cm > ref + kLazyRescale;
                    if (__any_sync(0xffffffffu, need)) {
                        const float sc = need ? ex2_approx(ref - cm) : 1.f;
                        if (sb > ww.sb_lo) {   // O_g holds this tile's sums
                            wait_pv(n - 1);
                            for (int c0 = 0; c0 < P.ebp; c0 += 16) {
                                float o[16];
                                tmem_ld_cols<16>(o_mine + c0, o);
#pragma unroll
                                for (int c = 0; c < 16; ++c) o[c] *= sc;
                                tmem_st_cols<16>(o_mine + c0, o);
                            }
                            tmem_st_wait();
                            if (flushed && sc != 1.f)   // something was flushed already
                                for (int c = 0; c < P.ebp; ++c) __stcg(olong + c * TM, sc * __ldcg(olong + c * TM));
                        }
                        ksum *= sc;
                        if (need) ref = cm;
                    }
                    // all -inf so far: every weight is 2^-inf = 0
                    const float nref = (ref == -INFINITY) ? 0.f : (kRowTermOut ? -ref - un : -ref);
                    const float2 nref2 = make_float2(nref, nref);
#pragma unroll
                    for (int c = 0; c < CPT / 2; ++c)
                        weight(c, (KID == KMB_KERNEL_GAUSSIAN) ? sub2(nref2, t2[c]) : fma2(t2[c], make_float2(-tsc, -tsc), nref2));
                }
                KMB_T(4);
                {
                    // the group's P over the thread's own S columns: hi planes in the first half, lo planes in the second
                    const uint32_t p_addr = tmem_base + COL_S + a * TNS + col0 + lane_addr;
                    tmem_st_cols<CPT / 2>(p_addr, reinterpret_cast<const float(&)[CPT / 2]>(ph));
                    if constexpr (LO) tmem_st_cols<CPT / 2>(p_addr + CPT / 2, reinterpret_cast<const float(&)[CPT / 2]>(pl));
                    ksum += kacc.x + kacc.y;
                }
                KMB_T(5);
                tmem_st_wait();
                if (until_flush == 0) {   // P.B(n) starts the O_g from zero
                    wait_pv(n - 1);
                    flush_o();
                    until_flush = P.flush_blocks;
                    flushed = true;
                }
                --until_flush;
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (PAIR && rank != 0) pair::mbar_arrive_cluster(pair::map_to_cta(&p_ready[a], 0));
                    else mbar_arrive(&p_ready[a]);
                }
                KMB_T(6);
            }
#ifdef KMB_PV16_TIMING
            if (blockIdx.x == 0 && et == 0) {
                for (int i = 0; i < 7; ++i) P.out[i] = static_cast<float>(tacc[i]) / n;
                P.out[7] = static_cast<float>(n);
                unsigned long long ns_now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_now));
                P.out[13] = static_cast<float>(clock64() - t_start) / n;                         // cycles per block, all in
                P.out[14] = static_cast<float>(clock64() - t_start) / static_cast<float>(ns_now - ns_start) * 1e3f;   // MHz
            }
#endif


            // ------------------------------ row tile done: merge the streams of the column groups ------------------------------
            refbuf[cg * TM + row_in_tile] = ref;
            ksbuf[cg * TM + row_in_tile] = ksum;
            wait_pv(n - 1);   // the tile's last PV
            flush_o();        // the long accumulators now hold the whole tile
            __threadfence();
            named_bar_sync(2, EPI_THREADS);
            float rmax = -INFINITY, wg[NG], ktot = 0.f;
#pragma unroll
            for (int g = 0; g < NG; ++g) rmax = fmaxf(rmax, refbuf[g * TM + row_in_tile]);
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                const float rg = refbuf[g * TM + row_in_tile];
                wg[g] = (rg == -INFINITY) ? 0.f : ex2_approx(rg - rmax);
                ktot = fmaf(wg[g], ksbuf[g * TM + row_in_tile], ktot);   // fixed order
            }
            const bool complete = (ww.Cw == 1);
            const bool ghost = tile >= P.n_tiles;   // pairs: an odd number of row tiles leaves the last peer without one
            // partial records of one wave: [row tile or pair in wave][range c]([rank])
            const size_t slot0 = static_cast<size_t>(w) * P.slots_per_wave + static_cast<size_t>(ww.tile_in_wave) * ww.Cw * NCTA + rank;
            float* mine = P.partial + (slot0 + static_cast<size_t>(ww.c) * NCTA) * (TM * PS);
            // plain product: undo the reference exponent (2^ref may underflow exactly where FP32 K b would)
            const float row_scale = NORM ? 1.f / ktot : ((rmax == -INFINITY) ? 0.f : ex2_approx(rmax));
            for (int c0 = cg * 16; c0 < P.ebp; c0 += NG * 16) {   // this thread merges 16-column chunks c0 of all O_g
                float o[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) o[c] = 0.f;
#pragma unroll
                for (int g = 0; g < NG; ++g) {
                    const float* og = P.olong + (static_cast<size_t>(blockIdx.x) * NG + g) * (MAX_EB * TM) + row_in_tile;
#pragma unroll
                    for (int c = 0; c < 16; ++c) o[c] = fmaf(wg[g], __ldcg(og + (c0 + c) * TM), o[c]);
                }
                if (ghost) continue;
                if (complete) {
                    if (row_ok) {
#pragma unroll
                        for (int c = 0; c < 16; ++c)
                            if (c0 + c < P.eb) P.out[row * P.E + P.e0 + c0 + c] = o[c] * __ldg(P.binv + P.e0 + c0 + c) * row_scale;
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < 16; ++c) mine[(c0 + c) * TM + row_in_tile] = o[c];
                }
            }
            tc_fence_before();
            if (!complete && !ghost) {
                if (cg == 0) {
                    mine[MAX_EB * TM + row_in_tile] = ktot;
                    mine[(MAX_EB + 1) * TM + row_in_tile] = rmax;
                }
                __threadfence();
                named_bar_sync(2, EPI_THREADS);
                if (et == 0) {
                    const int old = atomicAdd(&P.tile_counter[tile], 1);
                    const int last = (old == ww.Cw - 1);
                    if (last) P.tile_counter[tile] = 0;
                    *s_flag = last;
                }
                named_bar_sync(2, EPI_THREADS);
                const bool is_last = *s_flag != 0;
                named_bar_sync(2, EPI_THREADS);
                if (is_last && row_ok) {
                    __threadfence();
                    float mx = -INFINITY;
                    for (int c = 0; c < ww.Cw; ++c)
                        mx = fmaxf(mx, __ldcg(P.partial + (slot0 + static_cast<size_t>(c) * NCTA) * (TM * PS) + (MAX_EB + 1) * TM + row_in_tile));
                    for (int e = cg; e < P.eb; e += NG) {   // the groups share the signal columns of the row
                        float sum = 0.f, l = 0.f;
                        for (int c = 0; c < ww.Cw; ++c) {
                            const float* ps = P.partial + (slot0 + static_cast<size_t>(c) * NCTA) * (TM * PS);
                            const float m = __ldcg(ps + (MAX_EB + 1) * TM + row_in_tile);
                            const float wgt = (m == -INFINITY) ? 0.f : ex2_approx(m - mx);
                            sum = fmaf(wgt, __ldcg(ps + e * TM + row_in_tile), sum);
                            l = fmaf(wgt, __ldcg(ps + MAX_EB * TM + row_in_tile), l);
                        }
                        const float rs = NORM ? 1.f / l : ((mx == -INFINITY) ? 0.f : ex2_approx(mx));
                        P.out[row * P.E + P.e0 + e] = sum * __ldg(P.binv + P.e0 + e) * rs;
                    }
                }
            } else {
                named_bar_sync(2, EPI_THREADS);   // refbuf / ksbuf are rewritten at the end of the next tile
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) pair::cluster_sync_all();   // neither CTA frees tensor memory (or exits) while the other may signal it
    if (warp == 1) {
        if constexpr (PAIR) pair::tmem_dealloc2(tmem_base, TMEM_COLS);
        else tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int KID, bool NORM, int TERMS>
__global__ void __launch_bounds__(THREADS, 1)
kprod_tensor_pv16_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                         const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                         const __grid_constant__ CUtensorMap map_sh, const __grid_constant__ CUtensorMap map_sl,
                         const __grid_constant__ CUtensorMap map_ue, const __grid_constant__ CUtensorMap map_ve, const Params P) {
    pv16_body<KID, NORM, false, TERMS>(map_ah, map_al, map_bh, map_bl, map_sh, map_sl, map_ue, map_ve, P);
}
template <int KID, bool NORM, int TERMS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
kprod_tensor_pv16_pair_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                              const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                              const __grid_constant__ CUtensorMap map_sh, const __grid_constant__ CUtensorMap map_sl,
                              const __grid_constant__ CUtensorMap map_ue, const __grid_constant__ CUtensorMap map_ve, const Params P) {
    pv16_body<KID, NORM, true, TERMS>(map_ah, map_al, map_bh, map_bl, map_sh, map_sl, map_ue, map_ve, P);
}

// ---- signal planes -----------------------------------------------------------------------------------
// per block: column maxima of |b|
static __global__ void __launch_bounds__(256) signal_absmax_kernel(const float* __restrict__ b, long long M, int E,
                                                                   float* __restrict__ pmax) {
    __shared__ float sm[8][32];
    const int col = blockIdx.y * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;
    float hi = 0.f;
    if (col < E)
        for (long long r = blockIdx.x * 8 + rl; r < M; r += static_cast<long long>(gridDim.x) * 8) hi = fmaxf(hi, fabsf(b[r * E + col]));
    sm[rl][threadIdx.x & 31] = hi;
    __syncthreads();
    if (rl == 0 && col < E) {
        float h = 0.f;
        for (int i = 0; i < 8; ++i) h = fmaxf(h, sm[i][threadIdx.x]);
        pmax[static_cast<size_t>(blockIdx.x) * E + col] = h;
    }
}
// bscale[e] = 2^q with 2^q max_j |b[j][e]| in [2^13, 2^14); binv[e] = 2^-q.  q is clamped to [-114, 126], the range in
// which both 2^q and 2^-q are finite FP32 normals: every column whose largest |b| is an FP32 normal number then lands in
// [2^13, 2^14) (max |b| >= 2^-113) or in [1, 2^14) (the smallest normals), never above FP16's 65504 and never where the
// lo plane would lose bits to FP16 subnormals (tests/test_split_accuracy_cpu.py)
static __global__ void signal_scale_kernel(const float* __restrict__ pmax, int blocks, int E, int Ep, float* __restrict__ bscale,
                                           float* __restrict__ binv) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= Ep) return;
    float m = 0.f;
    if (e < E)
        for (int b = 0; b < blocks; ++b) m = fmaxf(m, pmax[static_cast<size_t>(b) * E + e]);
    int q = 0;
    if (m > 0.f && m < INFINITY) q = 13 - ilogbf(m);
    q = max(-114, min(126, q));
    bscale[e] = exp2f(static_cast<float>(q));
    binv[e] = exp2f(static_cast<float>(-q));
}
// hi/lo[sb][e][jj] = FP16 hi/lo of 2^q_e b[128 sb + jj][e]: the K-major signal of the P.B contraction, one contiguous
// (Ep x 128) slab per source block (a TMA box then reads 64 rows of 128 bytes 256 bytes apart, not 64 rows that are
// 2 Mp bytes apart), zero padded.  TERMS = 1 writes the hi plane only.
template <int TERMS>
static __global__ void transpose_split_signal_f16_kernel(const float* __restrict__ b, long long M, long long Mp, int E, int Ep,
                                                         const float* __restrict__ bscale, __half* __restrict__ hi,
                                                         __half* __restrict__ lo) {
    const long long j = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const int e = blockIdx.y;
    if (j >= Mp) return;
    const float v = (j < M && e < E) ? b[j * E + e] * bscale[e] : 0.f;
    const __half h = __float2half_rn(v);
    const long long at = ((j / TNS) * Ep + e) * TNS + (j % TNS);
    hi[at] = h;
    if constexpr (TERMS == 3) lo[at] = __float2half_rn(v - __half2float(h));
}

// Norm tiles of the extra K step (extra_k): rows of 64 BF16 (one 128-byte swizzle atom wide, 16 columns used).
//   ue[i] = [a0 a1 a2 1 1 1 0 ..]   a0 + a1 + a2 = -|u_i|^2 / sscale  (three BF16 pieces: 24 significant bits)
//   ve[j] = [1 1 1 b0 b1 b2 0 ..]   b0 + b1 + b2 = -|v_j|^2 / sscale;  padded sources (j >= M): b0 = -3e38, so that their
//                                   accumulator is -3e38 and their weight an exact zero (their v rows are zero-filled by TMA)
static __global__ void __launch_bounds__(256) norm_tiles_kernel(const float* __restrict__ un, const float* __restrict__ vn,
                                                                const float* __restrict__ sscale, long long N, long long M, long long Mp,
                                                                __nv_bfloat16* __restrict__ ue, __nv_bfloat16* __restrict__ ve) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= N + Mp) return;
    const bool is_u = i < N;
    const long long j = is_u ? i : i - N;
    const float inv = 1.f / __ldg(sscale + 1);   // 2^2p: exact
    float val = is_u ? -un[j] * inv : (j < M ? -vn[j] * inv : -3.0e38f);
    __nv_bfloat16 pc[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        pc[k] = __float2bfloat16_rn(val);
        val -= __bfloat162float(pc[k]);
    }
    // one 16-byte store of the six live columns (+ two zeros), seven of zeros: rows are 128 bytes
    const unsigned short one = 0x3f80;   // BF16 1.0
    unsigned short h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        h[k] = is_u ? __bfloat16_as_ushort(pc[k]) : one;
        h[3 + k] = is_u ? one : __bfloat16_as_ushort(pc[k]);
    }
    uint4* row = reinterpret_cast<uint4*>((is_u ? ue : ve) + j * 64);
    row[0] = make_uint4(h[0] | (static_cast<unsigned>(h[1]) << 16), h[2] | (static_cast<unsigned>(h[3]) << 16),
                        h[4] | (static_cast<unsigned>(h[5]) << 16), 0u);
#pragma unroll
    for (int c = 1; c < 8; ++c) row[c] = make_uint4(0u, 0u, 0u, 0u);
}

}  // namespace pv16

namespace {

size_t align_up_pv16(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Pv16Plan {
    bool pair;   // CTA pairs (cta_group::2): at least two row tiles
    int Dp, Ep, kblocks, ksteps_last, stages, grid, smem;
    long long n_tiles, nsb, Mp;
    tc::WavePlan waves;
    size_t off_center, off_stats, off_sscale, off_uh, off_ul, off_vh, off_vl, off_un, off_vn, off_sh, off_sl, off_bmax, off_bscale,
        off_binv, off_partial, off_olong, off_counter, off_ue, off_ve, total;
};

// host arithmetic only, for a device of `sms` SMs and `smem_max` bytes of opt-in shared memory per block: the launcher
// (plan_pv16) and the plan query (tensor_pv16_plan_debug) share it
int plan_pv16_host(int64_t N, int64_t M, int D, int E, int sms, int smem_max, Pv16Plan* pl) {
    pl->Dp = (D + 15) / 16 * 16;
    pl->kblocks = (pl->Dp + 63) / 64;
    pl->ksteps_last = (pl->Dp - (pl->kblocks - 1) * 64) / 16;
    pl->Ep = (E + pv16::MAX_EB - 1) / pv16::MAX_EB * pv16::MAX_EB;
    pl->Mp = (M + pv16::TNS - 1) / pv16::TNS * pv16::TNS;
    pl->n_tiles = (N + tc::TM - 1) / tc::TM;
    pl->nsb = (M + pv16::TNS - 1) / pv16::TNS;
    pl->pair = tensor_use_pair(pl->n_tiles, sms);
    pl->grid = pl->pair ? sms / 2 * 2 : sms;
    const int slot = pl->pair ? pv16::SLOT_BYTES / 2 : pv16::SLOT_BYTES;
    const int fixed = 1024 + (pl->kblocks * 2 + (pv16::kExtraK ? 1 : 0)) * pv16::A_TILE_BYTES + pv16::EPI_WARPS * 2 * pv16::CPT * 4 + 2 * pv16::NG * tc::TM * 4 + 512;
    pl->stages = std::min(pl->pair ? 10 : 6, (smem_max - fixed) / slot);
    if (pl->stages < 3) return set_error(KMB_ERR_UNSUPPORTED, "not enough shared memory for D=%d", D);
    pl->smem = fixed + pl->stages * slot;
    if (pl->pair) {   // the wave plan counts pairs of row tiles and clusters
        tc::plan_waves((pl->n_tiles + 1) / 2, pl->nsb, pl->grid / 2, static_cast<size_t>(tc::TM) * pl->Dp * 8, &pl->waves);
        pl->waves.slots_per_wave *= 2;
        pl->waves.partial_slots *= 2;
    } else {
        tc::plan_waves(pl->n_tiles, pl->nsb, pl->grid, static_cast<size_t>(tc::TM) * pl->Dp * 4, &pl->waves);
    }
    F16PointsLayout L;   // the points-only head shared with kprod_tensor (kmb_product_prepare_f32)
    f16_points_layout(N, M, D, &L);
    pl->off_center = L.off_center; pl->off_stats = L.off_stats; pl->off_sscale = L.off_sscale;
    pl->off_uh = L.off_uh; pl->off_ul = L.off_ul; pl->off_vh = L.off_vh; pl->off_vl = L.off_vl;
    pl->off_un = L.off_un; pl->off_vn = L.off_vn;
    size_t o = L.end;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up_pv16(bytes, 256); return at; };
    pl->off_sh = take(2 * static_cast<size_t>(pl->Ep) * pl->Mp);
    pl->off_sl = take(2 * static_cast<size_t>(pl->Ep) * pl->Mp);
    pl->off_bmax = take(sizeof(float) * tc::CENTER_BLOCKS * E);
    pl->off_bscale = take(sizeof(float) * pl->Ep);
    pl->off_binv = take(sizeof(float) * pl->Ep);
    pl->off_partial = take(sizeof(float) * pl->waves.partial_slots * tc::TM * pv16::PS);
    pl->off_olong = take(sizeof(float) * pl->grid * pv16::NG * pv16::MAX_EB * tc::TM);
    pl->off_counter = take(sizeof(int) * pl->n_tiles);
    pl->off_ue = take(pv16::kExtraK ? static_cast<size_t>(N) * 128 : 0);     // norm tiles of the extra K step: 64 BF16 per row
    pl->off_ve = take(pv16::kExtraK ? static_cast<size_t>(pl->Mp) * 128 : 0);
    pl->total = o;
    return KMB_OK;
}

int plan_pv16(int64_t N, int64_t M, int D, int E, Pv16Plan* pl) {
    int dev = 0, sms = 0, smem_max = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    return plan_pv16_host(N, M, D, E, sms, smem_max, pl);
}

template <int KID, bool NORM, int TERMS>
int launch_pv16(const CUtensorMap* m, const pv16::Params& P, int grid, int smem, bool pair, cudaStream_t stream) {
    if (pair) {
        auto fn = pv16::kprod_tensor_pv16_pair_kernel<KID, NORM, TERMS>;
        if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), smem)) return rc;
        fn<<<grid, pv16::THREADS, smem, stream>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], P);
    } else {
        auto fn = pv16::kprod_tensor_pv16_kernel<KID, NORM, TERMS>;
        if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), smem)) return rc;
        fn<<<grid, pv16::THREADS, smem, stream>>>(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], P);
    }
    KMB_CUDA_CHECK(cudaGetLastError());
    return KMB_OK;
}

}  // namespace

bool tensor_pv16_applicable(int D, int E, int kid) {
    return E > 4 && D <= 128 && (kid == KMB_KERNEL_GAUSSIAN || kid == KMB_KERNEL_ABSOLUTE_EXPONENTIAL || kid == KMB_KERNEL_DOT_EXPONENTIAL);
}
int tensor_pv16_signal_block() { return pv16::MAX_EB; }

int tensor_pv16_flush_blocks() {
    static const int flush_blocks = [] {   // tuning knob
        const char* e = getenv("KMB_PV16_FLUSH_BLOCKS");
        const int v = e ? atoi(e) : pv16::kFlushBlocks;
        return v < 1 ? 1 : v;
    }();
    return flush_blocks;
}

int tensor_pv16_plan_debug(int64_t N, int64_t M, int D, int E, int sms, int smem_optin, long long out[PVQ_FIELDS]) {
    Pv16Plan pl{};
    if (int rc = plan_pv16_host(N, M, D, E, sms, smem_optin, &pl)) return rc;
    pv_plan_fill(E, pv16::MAX_EB, pl.n_tiles, pl.nsb, pl.waves, out);   // pairs: R, C, R_last count pairs of row tiles
    out[PVQ_PAIR] = pl.pair ? 1 : 0;
    out[PVQ_GRID] = pl.grid;
    out[PVQ_STAGES] = pl.stages;
    out[PVQ_KBLOCKS] = pl.kblocks;
    out[PVQ_KSTEPS_LAST] = pl.ksteps_last;
    out[PVQ_FLUSH_BLOCKS] = tensor_pv16_flush_blocks();
    return KMB_OK;
}

int tensor_pv16_workspace_bytes(int64_t N, int64_t M, int D, int E, size_t* bytes) {
    Pv16Plan pl{};
    if (int rc = plan_pv16(N, M, D, E, &pl)) return rc;
    *bytes = pl.total;
    return KMB_OK;
}

int tensor_pv16_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E, int kid,
                        int flags, int elt, void* workspace, size_t workspace_bytes, cudaStream_t stream, cudaEvent_t ev0,
                        cudaEvent_t ev1, bool prepared) {
    Pv16Plan pl{};
    if (int rc = plan_pv16(N, M, D, E, &pl)) return rc;
    if (!workspace || workspace_bytes < pl.total)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.total, workspace_bytes);
    if (N >= (1ll << 31) - tc::TM || M >= (1ll << 31) - pv16::TNS)
        return set_error(KMB_ERR_UNSUPPORTED, "tensor path indexes rows with 32-bit TMA coordinates");
    if (!b) return set_error(KMB_ERR_INVALID, "signal is NULL");
    char* ws = static_cast<char*>(workspace);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
    void *uh = ws + pl.off_uh, *ul = ws + pl.off_ul, *vh = ws + pl.off_vh, *vl = ws + pl.off_vl, *sh = ws + pl.off_sh, *sl = ws + pl.off_sl;
    int* counters = reinterpret_cast<int*>(ws + pl.off_counter);
    const bool norm = flags & KMB_FLAG_NORMALIZE_ROWS;
    const bool x1 = elt == tc::ELT_F16X1;   // one term: the lo planes are not read, their maps repeat the hi ones

    KMB_CUDA_CHECK(cudaMemsetAsync(counters, 0, sizeof(int) * pl.n_tiles, stream));
    if (!prepared) {
        F16PointsLayout L;
        f16_points_layout(N, M, D, &L);
        if (int rc = f16_points_prepass(x, y, N, M, D, kid, L, ws, stream)) return rc;
    }
    {
        const int blocks = static_cast<int>(std::min<long long>(tc::CENTER_BLOCKS, (M + 7) / 8));
        pv16::signal_absmax_kernel<<<dim3(blocks, (E + 31) / 32), 256, 0, stream>>>(b, M, E, F(pl.off_bmax));
        KMB_CUDA_CHECK(cudaGetLastError());
        pv16::signal_scale_kernel<<<(pl.Ep + 127) / 128, 128, 0, stream>>>(F(pl.off_bmax), blocks, E, pl.Ep, F(pl.off_bscale), F(pl.off_binv));
        KMB_CUDA_CHECK(cudaGetLastError());
        dim3 g(static_cast<unsigned>((pl.Mp + 255) / 256), pl.Ep);
        if (x1)
            pv16::transpose_split_signal_f16_kernel<1><<<g, 256, 0, stream>>>(b, M, pl.Mp, E, pl.Ep, F(pl.off_bscale),
                                                                               static_cast<__half*>(sh), static_cast<__half*>(sl));
        else
            pv16::transpose_split_signal_f16_kernel<3><<<g, 256, 0, stream>>>(b, M, pl.Mp, E, pl.Ep, F(pl.off_bscale),
                                                                               static_cast<__half*>(sh), static_cast<__half*>(sl));
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch(3);
    }
    CUtensorMap maps[8];
    if (int rc = tc::make_tensor_map_f16(&maps[0], uh, N, pl.Dp, tc::TM)) return rc;
    if (int rc = tc::make_tensor_map_f16(&maps[1], x1 ? uh : ul, N, pl.Dp, tc::TM)) return rc;
    // CTA pairs: each CTA loads 64 of a block's 128 sources and half of the pass's signal columns
    if (int rc = tc::make_tensor_map_f16(&maps[2], vh, M, pl.Dp, pl.pair ? pv16::TNS / 2 : pv16::TNS)) return rc;
    if (int rc = tc::make_tensor_map_f16(&maps[3], x1 ? vh : vl, M, pl.Dp, pl.pair ? pv16::TNS / 2 : pv16::TNS)) return rc;
    const int ekid = tc::epilogue_kid(kid);   // dot-exponential: the Gaussian instantiations
    const bool xk = (ekid == KMB_KERNEL_GAUSSIAN) ? pv16::extra_k<KMB_KERNEL_GAUSSIAN>() : pv16::extra_k<KMB_KERNEL_ABSOLUTE_EXPONENTIAL>();
    if (xk) {   // |u|^2, |v|^2 as operands of one more K step (16-bit elements: the FP16 map serves BF16 rows as well)
        const long long rows = N + pl.Mp;
        pv16::norm_tiles_kernel<<<static_cast<unsigned>((rows + 255) / 256), 256, 0, stream>>>(
            F(pl.off_un), F(pl.off_vn), F(pl.off_sscale), N, M, pl.Mp, reinterpret_cast<__nv_bfloat16*>(ws + pl.off_ue),
            reinterpret_cast<__nv_bfloat16*>(ws + pl.off_ve));
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
        if (int rc = tc::make_tensor_map_f16(&maps[6], ws + pl.off_ue, N, 64, tc::TM)) return rc;
        if (int rc = tc::make_tensor_map_f16(&maps[7], ws + pl.off_ve, pl.Mp, 64, pl.pair ? pv16::TNS / 2 : pv16::TNS)) return rc;
    } else {
        maps[6] = maps[0];
        maps[7] = maps[2];
    }

    const int n_passes = pl.Ep / pv16::MAX_EB;
    for (int pass = 0; pass < n_passes; ++pass) {
        pv16::Params P;
        P.un = F(pl.off_un);
        P.vn = F(pl.off_vn);
        P.sscale = F(pl.off_sscale);
        P.binv = F(pl.off_binv);
        P.out = out;
        P.partial = F(pl.off_partial);
        P.olong = F(pl.off_olong);
        P.tile_counter = counters;
        P.N = N;
        P.M = M;
        P.E = E;
        P.e0 = pass * pv16::MAX_EB;
        P.eb = std::min(pv16::MAX_EB, E - P.e0);
        P.ebp = (P.eb + 31) / 32 * 32;
        {
            const int box_rows = pl.pair ? P.ebp / 2 : pv16::MAX_EB;
            if (int rc = tc::make_tensor_map_f16(&maps[4], sh, pl.nsb * pl.Ep, pv16::TNS, box_rows)) return rc;
            if (int rc = tc::make_tensor_map_f16(&maps[5], x1 ? sh : sl, pl.nsb * pl.Ep, pv16::TNS, box_rows)) return rc;
        }
        P.n_tiles = static_cast<int>(pl.n_tiles);
        P.nsb = static_cast<int>(pl.nsb);
        P.kblocks = pl.kblocks;
        P.ksteps_last = pl.ksteps_last;
        P.stages = pl.stages;
        P.ep_rows = pl.Ep;
        P.flush_blocks = tensor_pv16_flush_blocks();
        P.R = pl.waves.R;
        P.C = pl.waves.C;
        P.W = pl.waves.W;
        P.R_last = pl.waves.R_last;
        P.C_last = pl.waves.C_last;
        P.slots_per_wave = pl.waves.slots_per_wave;
        if (ev0 && pass == n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev0, stream));
        int rc;
        switch (ekid * 4 + (norm ? 2 : 0) + (x1 ? 1 : 0)) {
            case 0: rc = launch_pv16<KMB_KERNEL_GAUSSIAN, false, 3>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 1: rc = launch_pv16<KMB_KERNEL_GAUSSIAN, false, 1>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 2: rc = launch_pv16<KMB_KERNEL_GAUSSIAN, true, 3>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 3: rc = launch_pv16<KMB_KERNEL_GAUSSIAN, true, 1>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 4: rc = launch_pv16<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, false, 3>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 5: rc = launch_pv16<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, false, 1>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            case 6: rc = launch_pv16<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, true, 3>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
            default: rc = launch_pv16<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, true, 1>(maps, P, pl.grid, pl.smem, pl.pair, stream); break;
        }
        if (rc) return rc;
        if (ev1 && pass == n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev1, stream));
        count_launch();
    }
    return KMB_OK;
}

}  // namespace kmb
