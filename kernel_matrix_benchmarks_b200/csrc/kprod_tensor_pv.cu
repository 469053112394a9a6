// kprod_tensor_pv: a_i = sum_j k(x_i, y_j) b_j for 16 < D <= 128 and E > 4 -- both contractions on the
// tensor cores, flash-attention style (config C4: exponential-kernel attention, D = 64, E = 64).
//
//   S = 2 u.v^T   tcgen05.mma kind::tf32 (3xTF32), A = u tile resident in shared memory for a whole row
//                 tile, B = v tiles streamed by TMA, accumulator in TMEM (two stages)
//   P = k(S)      epilogue warps: tcgen05.ld S, kernel function (MUFU), lazy online max-rescale for the
//                 row-normalised variant, TF32 hi/lo split of P written back to TMEM (tcgen05.st)
//   O += P.B      tcgen05.mma with A = P from TMEM (hi, lo), B = transposed signal tile (hi, lo) from
//                 shared memory, accumulator O (128 x E) in TMEM; read once per row tile
//
// The epilogue is the critical resource (MUFU + the hi/lo split, ~12 instructions per kernel value against
// 48 MMAs of 32 cycles per 128 x 64 tile), so it is spread over NG groups of four warps: group g owns
// columns [g TN/NG, (g+1) TN/NG) of every S tile (all 128 rows: TMEM lane quarter = warp % 4), the groups
// agree on the row maximum through shared memory, and each one rescales / stores its own share of O.
//
// TMEM columns: S stage 0 [0,64) | S stage 1 [64,128) | P hi [128,192) | P lo [192,256) | O [256,256+E).
// Warp roles and the wave schedule (every CTA of a wave walks the same source blocks at the same time) are those of
// kprod_tensor.cu.  This is the first version of the E > 4 kernel; FP16 planes take kprod_tensor_pv16.cu.
#include <algorithm>

#include "tensor_common.cuh"

namespace kmb {
namespace pv {

using namespace tc;

constexpr int TN = 64;                 // sources per S tile
constexpr int SLOT_BYTES = 16384;      // ring slot: v tile hi+lo of one K block, or one half (hi / lo) of a signal tile
constexpr int HALF_SLOT = SLOT_BYTES / 2;
constexpr int A_TILE_BYTES = TM * TK * 4;   // 16 KB
constexpr int NG = 4;                  // epilogue column groups (4 warps each)
constexpr int CPT = TN / NG;           // S columns per epilogue thread
constexpr int EPI_WARPS = 4 * NG;
constexpr int EPI_THREADS = 32 * EPI_WARPS;
constexpr int THREADS = 64 + EPI_THREADS;
static_assert(CPT % 16 == 0, "tcgen05.ld/st in 16-column chunks");
constexpr int TMEM_COLS = 512;
constexpr int COL_S = 0, COL_PH = 128, COL_PL = 192, COL_O = 256;
constexpr int MAX_EB = 64;             // signal columns per pass
constexpr float kLazyRescale = 64.f;   // rescale O only when the row maximum grows by more than 2^64
// The tensor cores add into the FP32 accumulator with truncation (see kprod_tensor_pv16.cu: 2.4e-4 relative after 12288
// accumulating MMAs); this kernel makes 24 per 64-source block.  O therefore only collects kFlushBlocks blocks; then each
// epilogue thread adds its chunks of O (round-to-nearest, L2 reductions it does not wait for) to a per-CTA FP32
// accumulator in global memory and the next P.B starts from zero.
constexpr int kFlushBlocks = 64;

struct Params {
    const float* un;
    const float* vn;
    float* out;
    float* partial;
    float* olong;              // grid x MAX_EB x TM: long accumulator of O, [column][row] (see kFlushBlocks)
    int* tile_counter;
    long long N, M, row_offset;
    int E, e0, eb;             // this pass covers signal columns e0 .. e0+eb-1; ebp = eb rounded up to 32
    int ebp;
    int n_tiles, nsb, kblocks, stages;
    int R, C, W, R_last, C_last, slots_per_wave;   // wave schedule (tc::plan_waves, see kprod_tensor.cu)
};

// unit range [u0, u1) (units = row tile * nsb + source block) of CTA `cta` in wave w: one row tile, a contiguous range
// of its source blocks; every CTA of a wave with the same range index walks the same source blocks at the same time
struct WaveRange { long long u0, u1; int c, Cw, tile_in_wave; };
__device__ __forceinline__ bool wave_range(const Params& P, int w, int cta, WaveRange& wr) {
    const bool last = (w == P.W - 1);
    const int Rw = last ? P.R_last : P.R, Cw = last ? P.C_last : P.C;
    if (cta >= Rw * Cw) return false;
    wr.Cw = Cw;
    wr.tile_in_wave = cta / Cw;
    wr.c = cta - wr.tile_in_wave * Cw;
    const long long tile = static_cast<long long>(w) * P.R + wr.tile_in_wave;
    wr.u0 = tile * P.nsb + static_cast<long long>(P.nsb) * wr.c / Cw;
    wr.u1 = tile * P.nsb + static_cast<long long>(P.nsb) * (wr.c + 1) / Cw;
    return true;
}

template <int KID, bool NORM>
struct Cfg {
    static constexpr bool ONLINE_MAX = NORM && KID != KMB_KERNEL_INVERSE_DISTANCE;
    static constexpr int PS = MAX_EB + 2;   // O row, sum of weights, reference exponent
};

template <int KID, bool NORM>
__global__ void __launch_bounds__(THREADS, 1)
kprod_tensor_pv_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                       const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                       const __grid_constant__ CUtensorMap map_sh, const __grid_constant__ CUtensorMap map_sl,
                       const Params P) {
    using C = Cfg<KID, NORM>;
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
    unsigned char* u_region = smem;                                   // kblocks x [A hi 16 KB | A lo 16 KB]
    unsigned char* ring = u_region + P.kblocks * 2 * A_TILE_BYTES;    // stages x 16 KB
    float* aux = reinterpret_cast<float*>(ring + P.stages * SLOT_BYTES);   // 2 x TN floats (|v|^2)
    float* cmbuf = aux + 2 * TN;                                            // 2 x NG x TM: per-group row maxima of a tile
    float* ksbuf = cmbuf + 2 * NG * TM;                                     // NG x TM: per-group sums of weights
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ksbuf + NG * TM);
    uint64_t* empty_bar = full_bar + P.stages;
    uint64_t* acc_full = empty_bar + P.stages;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* u_full = acc_empty + 2;
    uint64_t* u_free = u_full + 1;
    uint64_t* p_ready = u_free + 1;
    uint64_t* p_free = p_ready + 1;
    uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(p_free + 1);
    int* s_flag = reinterpret_cast<int*>(tmem_base_smem + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int G = gridDim.x;
    const long long nsb = P.nsb;
    const int cta = blockIdx.x;
    (void)G;
    const int ST = P.stages;

    if (tid == 0) {
        for (int s = 0; s < ST; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], EPI_WARPS); }
        mbar_init(u_full, 1);
        mbar_init(u_free, 1);
        mbar_init(p_ready, EPI_WARPS);
        mbar_init(p_free, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(tmem_base_smem, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_smem;
    const uint32_t idesc_s = idesc_tf32(TN), idesc_o = idesc_tf32(P.ebp);

    if (warp == 0) {
        // ------------------------------------ TMA producer ------------------------------------
        // all 32 lanes walk the loop (uniform control flow); one elected lane issues (see elect_one)
        {
            uint32_t it = 0, seg = 0;
            auto emit_signal = [&](long long u) {
                const int src0 = static_cast<int>(u % nsb) * TN;
                for (int h = 0; h < 2; ++h, ++it) {
                    const int slot = it % ST;
                    mbar_wait(&empty_bar[slot], ((it / ST) & 1) ^ 1);
                    unsigned char* dst = ring + slot * SLOT_BYTES;
                    const CUtensorMap* m = h == 0 ? &map_sh : &map_sl;
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&full_bar[slot], SLOT_BYTES);
                        tma_load_2d(dst, m, src0, P.e0, &full_bar[slot]);                  // K columns src0 .. +31
                        tma_load_2d(dst + HALF_SLOT, m, src0 + TK, P.e0, &full_bar[slot]); // K columns src0+32 .. +63
                    }
                    __syncwarp();
                }
            };
            long long prev = -1;
            WaveRange wr;
            for (int w = 0; w < P.W; ++w) {
            if (!wave_range(P, w, cta, wr)) continue;
            const long long u0 = wr.u0, u1 = wr.u1;
            for (long long u = u0; u < u1; ++u) {
                const int tile = static_cast<int>(u / nsb);
                if (u == u0 || u % nsb == 0) {   // new row tile: (re)load the resident u tile
                    mbar_wait(u_free, (seg & 1) ^ 1);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(u_full, P.kblocks * 2 * A_TILE_BYTES);
                        for (int kb = 0; kb < P.kblocks; ++kb) {
                            tma_load_2d(u_region + (kb * 2 + 0) * A_TILE_BYTES, &map_ah, kb * TK, tile * TM, u_full);
                            tma_load_2d(u_region + (kb * 2 + 1) * A_TILE_BYTES, &map_al, kb * TK, tile * TM, u_full);
                        }
                    }
                    __syncwarp();
                    ++seg;
                }
                const int src0 = static_cast<int>(u % nsb) * TN;
                for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                    const int slot = it % ST;
                    mbar_wait(&empty_bar[slot], ((it / ST) & 1) ^ 1);
                    unsigned char* dst = ring + slot * SLOT_BYTES;
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&full_bar[slot], SLOT_BYTES);
                        tma_load_2d(dst, &map_bh, kb * TK, src0, &full_bar[slot]);
                        tma_load_2d(dst + HALF_SLOT, &map_bl, kb * TK, src0, &full_bar[slot]);
                    }
                    __syncwarp();
                }
                if (prev >= 0) emit_signal(prev);   // consumed by PV(n-1), issued after S(n)
                prev = u;
            }
            }
            if (prev >= 0) emit_signal(prev);
        }
    } else if (warp == 1) {
        // ------------------------------------- MMA issuer -------------------------------------
        // All 32 lanes walk the loop and wait on the barriers; one elected lane issues (see elect_one).
        // Order: S(0), S(1), PV(0), S(2), PV(1), ...
        {
            uint32_t it = 0, n = 0, seg = 0;
            const uint32_t d_o = tmem_base + COL_O;
            auto issue_pv = [&](uint32_t m, bool from_zero) {   // from_zero: O was flushed (or the segment starts)
                mbar_wait(p_ready, m & 1);
                const int slot_h = it % ST;
                mbar_wait(&full_bar[slot_h], (it / ST) & 1);
                ++it;
                const int slot_l = it % ST;
                mbar_wait(&full_bar[slot_l], (it / ST) & 1);
                ++it;
                tc_fence_after();
                const unsigned char* sh = ring + slot_h * SLOT_BYTES;
                const unsigned char* sl = ring + slot_l * SLOT_BYTES;
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < TN / UMMA_K; ++k) {
                        const int panel = k >> 2, koff = (k & 3) * UMMA_K * 4;
                        const uint64_t bh = umma_desc_sw128(sh + panel * HALF_SLOT, koff);
                        const uint64_t bl = umma_desc_sw128(sl + panel * HALF_SLOT, koff);
                        const uint32_t a_hi = tmem_base + COL_PH + k * UMMA_K, a_lo = tmem_base + COL_PL + k * UMMA_K;
                        umma_tf32_ts(d_o, a_lo, bh, idesc_o, !(from_zero && k == 0));
                        umma_tf32_ts(d_o, a_hi, bl, idesc_o, 1);
                        umma_tf32_ts(d_o, a_hi, bh, idesc_o, 1);
                    }
                    umma_commit(&empty_bar[slot_h]);
                    umma_commit(&empty_bar[slot_l]);
                    umma_commit(p_free);
                }
                __syncwarp();
            };
            bool prev_first = false, pv_pending = false;
            WaveRange wr;
            for (int w = 0; w < P.W; ++w) {
            if (!wave_range(P, w, cta, wr)) continue;
            const long long u0 = wr.u0, u1 = wr.u1;
            long long seg_u0 = u0;
            for (long long u = u0; u < u1; ++u, ++n) {
                bool first = (u == u0) || (u % nsb == 0);
                if (first) {
                    mbar_wait(u_full, seg & 1);
                    ++seg;
                    seg_u0 = u;
                }
                first = ((u - seg_u0) % kFlushBlocks == 0);   // O restarts from zero at every flush
                const int a = n & 1;
                mbar_wait(&acc_empty[a], ((n >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_s = tmem_base + COL_S + a * TN;
                for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                    const int slot = it % ST;
                    mbar_wait(&full_bar[slot], (it / ST) & 1);
                    tc_fence_after();
                    const unsigned char* bt = ring + slot * SLOT_BYTES;
                    const unsigned char* at = u_region + kb * 2 * A_TILE_BYTES;
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < TK / UMMA_K; ++k) {
                            const uint64_t ah = umma_desc_sw128(at, k * UMMA_K * 4);
                            const uint64_t al = umma_desc_sw128(at + A_TILE_BYTES, k * UMMA_K * 4);
                            const uint64_t bh = umma_desc_sw128(bt, k * UMMA_K * 4);
                            const uint64_t bl = umma_desc_sw128(bt + HALF_SLOT, k * UMMA_K * 4);
                            umma_tf32(d_s, al, bh, idesc_s, (kb | k) != 0);
                            umma_tf32(d_s, ah, bl, idesc_s, 1);
                            umma_tf32(d_s, ah, bh, idesc_s, 1);
                        }
                        umma_commit(&empty_bar[slot]);
                    }
                    __syncwarp();
                }
                const bool last_of_tile = (u + 1 == u1 || (u + 1) % nsb == 0);
                if (elect_one()) {
                    umma_commit(&acc_full[a]);
                    if (last_of_tile) umma_commit(u_free);   // last S of this row tile
                }
                __syncwarp();
                if (pv_pending) issue_pv(n - 1, prev_first);
                pv_pending = true;
                prev_first = first;
            }
            }
            if (pv_pending) issue_pv(n - 1, prev_first);
        }
    } else {
        // -------------------------------------- epilogue --------------------------------------
        const int et = tid - 64;
        const int lane_group = warp & 3;             // TMEM lane quarter this warp may touch
        const int cg = (warp - 2) >> 2;              // column group
        const int col0 = cg * CPT;                   // first S / P column of this thread
        const int row_in_tile = lane_group * 32 + lane;
        const uint32_t lane_addr = static_cast<uint32_t>(lane_group * 32) << 16;
        uint32_t n = 0, pv_seen = 0;
#ifdef KMB_PV_TIMING
        long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = clock64();
#define KMB_T(i) do { const long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } while (0)
#else
#define KMB_T(i) do { } while (0)
#endif
        auto ensure_pv_done = [&](uint32_t count) {   // PV(0 .. count-1) have completed
            while (pv_seen < count) {
                mbar_wait(p_free, pv_seen & 1);
                ++pv_seen;
            }
            tc_fence_after();
        };
        WaveRange wr;
        for (int w = 0; w < P.W; ++w) {
        if (!wave_range(P, w, cta, wr)) continue;
        const long long u0 = wr.u0, u1 = wr.u1;
        long long u = u0;
        float vn_next = 1.0e30f;   // |v|^2 of source (next block) + et, for the threads that stage it
        if (et < TN && u0 < u1) {
            const long long j = (u0 % nsb) * TN + et;
            if (j < P.M) vn_next = __ldg(P.vn + j);
        }
        while (u < u1) {
            const int tile = static_cast<int>(u / nsb);
            const long long sb0 = u - tile * nsb;
            const int cnt = static_cast<int>(min(nsb - sb0, u1 - u));
            const long long row = static_cast<long long>(tile) * TM + row_in_tile;
            const bool row_ok = row < P.N;
            const float un = row_ok ? __ldg(P.un + row) : 0.f;
            [[maybe_unused]] const long long jz = (P.row_offset + row) % (P.M + 1);
            float ksum = 0.f, ref = -INFINITY;   // ksum: this group's columns only
            // long accumulator of this thread's 16-column chunks of O: zero, then only ever touched by this thread
            float* olong = P.olong + static_cast<size_t>(blockIdx.x) * (MAX_EB * TM) + row_in_tile;
            for (int c0 = cg * 16; c0 < P.ebp; c0 += NG * 16)
#pragma unroll
                for (int c = 0; c < 16; ++c) __stcg(olong + (c0 + c) * TM, 0.f);

            for (int k = 0; k < cnt; ++k, ++n) {
                const long long j0 = (sb0 + k) * TN;
                float* ax = aux + (n & 1) * TN;
                if (et < TN) {
                    ax[et] = vn_next;   // loaded one tile ago: the global-load latency stays off the critical path
                    const long long un1 = u + k + 1;
                    const long long j = (un1 % nsb) * TN + et;
                    vn_next = (un1 < u1 && j < P.M) ? __ldg(P.vn + j) : 1.0e30f;
                }
                KMB_T(0);
                named_bar_sync(1, EPI_THREADS);
                KMB_T(1);
                const int a = n & 1;
                mbar_wait(&acc_full[a], (n >> 1) & 1);
                tc_fence_after();
                KMB_T(2);
                float s[CPT];
                tmem_ld_cols<CPT>(tmem_base + COL_S + a * TN + col0 + lane_addr, s);
                KMB_T(3);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[a]);   // S is in registers: the MMA warp may refill this stage

                // kernel values (or their log2 under the online max)
                float cm = -INFINITY;
#pragma unroll
                for (int c = 0; c < CPT; ++c) {
                    if constexpr (C::ONLINE_MAX) {
                        s[c] = log2_kernel_from_parts<KID>(s[c], un, ax[col0 + c]);
                        cm = fmaxf(cm, s[c]);
                    } else {
                        s[c] = kernel_from_parts<KID>(s[c], un, ax[col0 + c]);
                        if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE) {
                            if (j0 + col0 + c == jz || j0 + col0 + c >= P.M) s[c] = 0.f;
                        }
                    }
                }
                if constexpr (C::ONLINE_MAX) {
                    // the groups agree on the row maximum of the tile (so that they take the same decisions)
                    float* cmb = cmbuf + (n & 1) * (NG * TM);
                    cmb[cg * TM + row_in_tile] = cm;
                    named_bar_sync(3, EPI_THREADS);
#pragma unroll
                    for (int g = 0; g < NG; ++g) cm = fmaxf(cm, cmb[g * TM + row_in_tile]);
                }
                KMB_T(4);
                ensure_pv_done(n);   // PV(n-1) has read P and finished accumulating into O
                if (k > 0 && k % kFlushBlocks == 0) {   // PV(n) starts O from zero: move what it holds to the long accumulator
                    for (int c0 = cg * 16; c0 < P.ebp; c0 += NG * 16) {
                        float o[16];
                        tmem_ld_cols<16>(tmem_base + COL_O + c0 + lane_addr, o);
#pragma unroll
                        for (int c = 0; c < 16; ++c) atomicAdd(olong + (c0 + c) * TM, o[c]);   // RED: nothing to wait for
                    }
                }
                KMB_T(5);
                if constexpr (C::ONLINE_MAX) {
                    // lazy rescale: keep the reference exponent unless the row maximum outgrew it by 2^64
                    bool need = false;
                    if (ref == -INFINITY) ref = cm;   // first tile of the row (O is overwritten by its PV)
                    else need = cm > ref + kLazyRescale;
                    if (__any_sync(0xffffffffu, need)) {   // same lanes, same data in every group: same branch
                        const float sc = need ? ex2_approx(ref - cm) : 1.f;
                        for (int c0 = cg * 16; c0 < P.ebp; c0 += NG * 16) {   // this group's 16-column chunks of O
                            float o[16];
                            tmem_ld_cols<16>(tmem_base + COL_O + c0 + lane_addr, o);
#pragma unroll
                            for (int c = 0; c < 16; ++c) o[c] *= sc;
                            tmem_st_cols<16>(tmem_base + COL_O + c0 + lane_addr, o);
                            if (k >= kFlushBlocks && sc != 1.f)   // something was flushed already
#pragma unroll
                                for (int c = 0; c < 16; ++c) __stcg(olong + (c0 + c) * TM, sc * __ldcg(olong + (c0 + c) * TM));
                        }
                        tmem_st_wait();
                        ksum *= sc;
                        if (need) ref = cm;
                    }
#pragma unroll
                    for (int c = 0; c < CPT; ++c) s[c] = ex2_approx(s[c] - ref);
                }
                // TF32 hi / lo split of P -> TMEM; the weights summed for the normaliser are the split ones
                {
                    float lo[CPT], kacc = 0.f;   // two-level sum of the weights (see kprod_direct.cuh)
#pragma unroll
                    for (int c = 0; c < CPT; ++c) {
                        const float hi = to_tf32(s[c]);
                        lo[c] = to_tf32(s[c] - hi);
                        s[c] = hi;
                        kacc += hi + lo[c];
                    }
                    tmem_st_cols<CPT>(tmem_base + COL_PH + col0 + lane_addr, s);
                    tmem_st_cols<CPT>(tmem_base + COL_PL + col0 + lane_addr, lo);
                    ksum += kacc;
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(p_ready);
                KMB_T(6);
            }
#ifdef KMB_PV_TIMING
            if (blockIdx.x == 0 && et == 0 && u + cnt >= u1) {
                for (int i = 0; i < 7; ++i) P.out[i] = static_cast<float>(tacc[i]) / n;
                P.out[7] = static_cast<float>(n);
            }
#endif

            // ------------------------------ row tile (segment) done ------------------------------
            ensure_pv_done(n);
            // the row's sum of weights over all column groups, in a fixed order
            ksbuf[cg * TM + row_in_tile] = ksum;
            named_bar_sync(2, EPI_THREADS);
            float ktot = 0.f;
#pragma unroll
            for (int g = 0; g < NG; ++g) ktot += ksbuf[g * TM + row_in_tile];
            const bool complete = (wr.Cw == 1);
            // one partial record per (wave, CTA); the last CTA of the row tile to arrive adds them in range order
            const size_t slot0 = static_cast<size_t>(w) * P.slots_per_wave + static_cast<size_t>(wr.tile_in_wave) * wr.Cw;
            float* mine = P.partial + (slot0 + wr.c) * (TM * C::PS);
            for (int c0 = cg * 16; c0 < P.ebp; c0 += NG * 16) {   // this group's 16-column chunks of O
                float o[16];
                tmem_ld_cols<16>(tmem_base + COL_O + c0 + lane_addr, o);
#pragma unroll
                for (int c = 0; c < 16; ++c) o[c] += __ldcg(olong + (c0 + c) * TM);   // what earlier flushes moved out of O
                if (complete) {
                    if (row_ok) {
#pragma unroll
                        for (int c = 0; c < 16; ++c)
                            if (c0 + c < P.eb) P.out[row * P.E + P.e0 + c0 + c] = NORM ? o[c] / ktot : o[c];
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < 16; ++c) mine[(c0 + c) * TM + row_in_tile] = o[c];
                }
            }
            tc_fence_before();
            if (!complete) {
                if (cg == 0) {
                    mine[MAX_EB * TM + row_in_tile] = ktot;
                    mine[(MAX_EB + 1) * TM + row_in_tile] = ref;
                }
                __threadfence();
                named_bar_sync(2, EPI_THREADS);
                const int c_first = 0, c_last = wr.Cw - 1;
                if (et == 0) {
                    const int old = atomicAdd(&P.tile_counter[tile], 1);
                    const int last = (old == c_last - c_first);
                    if (last) P.tile_counter[tile] = 0;
                    *s_flag = last;
                }
                named_bar_sync(2, EPI_THREADS);
                const bool is_last = *s_flag != 0;
                named_bar_sync(2, EPI_THREADS);
                if (is_last && row_ok) {
                    __threadfence();
                    float mx = -INFINITY, l = 0.f;
                    if constexpr (C::ONLINE_MAX) {
                        for (int c = c_first; c <= c_last; ++c) {
                            const float* ps = P.partial + (slot0 + c) * (TM * C::PS);
                            mx = fmaxf(mx, __ldcg(ps + (MAX_EB + 1) * TM + row_in_tile));
                        }
                    }
                    for (int e = cg; e < P.eb; e += NG) {   // the groups share the signal columns of the row
                        float sum = 0.f;
                        l = 0.f;
                        for (int c = c_first; c <= c_last; ++c) {
                            const float* ps = P.partial + (slot0 + c) * (TM * C::PS);
                            float w = 1.f;
                            if constexpr (C::ONLINE_MAX) {
                                const float m = __ldcg(ps + (MAX_EB + 1) * TM + row_in_tile);
                                w = (m == -INFINITY) ? 0.f : ex2_approx(m - mx);
                            }
                            sum = fmaf(w, __ldcg(ps + e * TM + row_in_tile), sum);
                            l = fmaf(w, __ldcg(ps + MAX_EB * TM + row_in_tile), l);
                        }
                        P.out[row * P.E + P.e0 + e] = NORM ? sum / l : sum;
                    }
                }
            } else {
                named_bar_sync(2, EPI_THREADS);   // ksbuf is rewritten at the end of the next segment
            }
            u += cnt;
        }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// bt_hi/bt_lo[e][j] = TF32 hi/lo of b[j][e]  (K-major signal for the P.B contraction), zero padded
static __global__ void transpose_split_signal_kernel(const float* __restrict__ b, long long M, long long Mp, int E, int Ep,
                                                     float* __restrict__ hi, float* __restrict__ lo) {
    const long long j = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const int e = blockIdx.y;
    if (j >= Mp) return;
    const float v = (j < M && e < E) ? b[j * E + e] : 0.f;
    const float h = to_tf32(v);
    hi[e * Mp + j] = h;
    lo[e * Mp + j] = to_tf32(v - h);
    (void)Ep;
}

}  // namespace pv

namespace {

size_t align_up_pv(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct PvPlan {
    int Dp, Ep, kblocks, stages, grid_max, smem;
    long long n_tiles, nsb, Mp;
    tc::WavePlan waves;
    size_t off_center, off_cpart, off_uh, off_ul, off_vh, off_vl, off_un, off_vn, off_sh, off_sl, off_partial, off_olong, off_counter, total;
};

// host arithmetic only, for a device of `sms` SMs and `smem_max` bytes of opt-in shared memory per block: the launcher
// (plan_pv) and the plan query (tensor_pv_plan_debug) share it
int plan_pv_host(int64_t N, int64_t M, int D, int E, int sms, int smem_max, PvPlan* pl) {
    pl->Dp = (D + tc::TK - 1) / tc::TK * tc::TK;
    pl->kblocks = pl->Dp / tc::TK;
    pl->Ep = (E + pv::MAX_EB - 1) / pv::MAX_EB * pv::MAX_EB;
    pl->Mp = (M + pv::TN - 1) / pv::TN * pv::TN;
    pl->n_tiles = (N + tc::TM - 1) / tc::TM;
    pl->nsb = (M + pv::TN - 1) / pv::TN;
    pl->grid_max = sms;
    const int fixed = 1024 + pl->kblocks * 2 * pv::A_TILE_BYTES + 2 * pv::TN * 4 + 3 * pv::NG * tc::TM * 4 + 512;
    pl->stages = std::min(12, (smem_max - fixed) / pv::SLOT_BYTES);
    if (pl->stages < 4) return set_error(KMB_ERR_UNSUPPORTED, "not enough shared memory for D=%d", D);
    pl->smem = fixed + pl->stages * pv::SLOT_BYTES;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up_pv(bytes, 256); return at; };
    pl->off_center = take(sizeof(float) * pl->Dp);
    pl->off_cpart = take(sizeof(float) * tc::CENTER_BLOCKS * D);
    pl->off_uh = take(sizeof(float) * N * pl->Dp);
    pl->off_ul = take(sizeof(float) * N * pl->Dp);
    pl->off_vh = take(sizeof(float) * M * pl->Dp);
    pl->off_vl = take(sizeof(float) * M * pl->Dp);
    pl->off_un = take(sizeof(float) * N);
    pl->off_vn = take(sizeof(float) * M);
    pl->off_sh = take(sizeof(float) * pl->Ep * pl->Mp);
    pl->off_sl = take(sizeof(float) * pl->Ep * pl->Mp);
    tc::plan_waves(pl->n_tiles, pl->nsb, pl->grid_max, static_cast<size_t>(tc::TM) * pl->Dp * 8, &pl->waves);
    pl->off_partial = take(sizeof(float) * pl->waves.partial_slots * tc::TM * (pv::MAX_EB + 2));
    pl->off_olong = take(sizeof(float) * pl->grid_max * pv::MAX_EB * tc::TM);
    pl->off_counter = take(sizeof(int) * pl->n_tiles);
    pl->total = o;
    return KMB_OK;
}

int plan_pv(int64_t N, int64_t M, int D, int E, PvPlan* pl) {
    int dev = 0, sms = 0, smem_max = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    return plan_pv_host(N, M, D, E, sms, smem_max, pl);
}

template <int KID, bool NORM>
int launch_pv(const CUtensorMap* m, const pv::Params& P, int grid, int smem, cudaStream_t stream) {
    auto fn = pv::kprod_tensor_pv_kernel<KID, NORM>;
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), smem)) return rc;
    fn<<<grid, pv::THREADS, smem, stream>>>(m[0], m[1], m[2], m[3], m[4], m[5], P);
    KMB_CUDA_CHECK(cudaGetLastError());
    return KMB_OK;
}

}  // namespace

bool tensor_pv_applicable(int D, int E) { return E > 4 && D <= 128; }
int tensor_pv_signal_block() { return pv::MAX_EB; }

int tensor_pv_plan_debug(int64_t N, int64_t M, int D, int E, int sms, int smem_optin, long long out[PVQ_FIELDS]) {
    PvPlan pl{};
    if (int rc = plan_pv_host(N, M, D, E, sms, smem_optin, &pl)) return rc;
    pv_plan_fill(E, pv::MAX_EB, pl.n_tiles, pl.nsb, pl.waves, out);
    out[PVQ_PAIR] = 0;
    out[PVQ_GRID] = pl.grid_max;
    out[PVQ_STAGES] = pl.stages;
    out[PVQ_KBLOCKS] = pl.kblocks;
    out[PVQ_KSTEPS_LAST] = tc::TK / tc::UMMA_K;   // D is zero-padded to whole K blocks
    out[PVQ_FLUSH_BLOCKS] = pv::kFlushBlocks;
    return KMB_OK;
}

int tensor_pv_workspace_bytes(int64_t N, int64_t M, int D, int E, size_t* bytes) {
    PvPlan pl{};
    if (int rc = plan_pv(N, M, D, E, &pl)) return rc;
    *bytes = pl.total;
    return KMB_OK;
}

int tensor_pv_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E,
                      int kid, int flags, int64_t row_offset, void* workspace, size_t workspace_bytes, cudaStream_t stream,
                      cudaEvent_t ev0, cudaEvent_t ev1) {
    PvPlan pl{};
    if (int rc = plan_pv(N, M, D, E, &pl)) return rc;
    if (!workspace || workspace_bytes < pl.total)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.total, workspace_bytes);
    if (N >= (1ll << 31) - tc::TM || M >= (1ll << 31) - pv::TN)
        return set_error(KMB_ERR_UNSUPPORTED, "tensor path indexes rows with 32-bit TMA coordinates");
    if (!b) return set_error(KMB_ERR_INVALID, "signal is NULL");
    char* ws = static_cast<char*>(workspace);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
    float *uh = F(pl.off_uh), *ul = F(pl.off_ul), *vh = F(pl.off_vh), *vl = F(pl.off_vl), *sh = F(pl.off_sh), *sl = F(pl.off_sl);
    int* counters = reinterpret_cast<int*>(ws + pl.off_counter);
    const bool norm = flags & KMB_FLAG_NORMALIZE_ROWS;

    KMB_CUDA_CHECK(cudaMemsetAsync(counters, 0, sizeof(int) * pl.n_tiles, stream));
    if (int rc = tc::tensor_prepass(x, y, N, M, D, pl.Dp, kid, F(pl.off_center), F(pl.off_cpart), uh, ul, vh, vl, F(pl.off_un),
                                    F(pl.off_vn), stream))
        return rc;
    {
        dim3 g(static_cast<unsigned>((pl.Mp + 255) / 256), pl.Ep);
        pv::transpose_split_signal_kernel<<<g, 256, 0, stream>>>(b, M, pl.Mp, E, pl.Ep, sh, sl);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
    }
    CUtensorMap maps[6];
    if (int rc = tc::make_tensor_map(&maps[0], uh, N, pl.Dp, tc::TM)) return rc;
    if (int rc = tc::make_tensor_map(&maps[1], ul, N, pl.Dp, tc::TM)) return rc;
    if (int rc = tc::make_tensor_map(&maps[2], vh, M, pl.Dp, pv::TN)) return rc;
    if (int rc = tc::make_tensor_map(&maps[3], vl, M, pl.Dp, pv::TN)) return rc;
    if (int rc = tc::make_tensor_map(&maps[4], sh, pl.Ep, static_cast<int>(pl.Mp), pv::MAX_EB)) return rc;
    if (int rc = tc::make_tensor_map(&maps[5], sl, pl.Ep, static_cast<int>(pl.Mp), pv::MAX_EB)) return rc;

    const int grid = pl.grid_max;
    const int n_passes = pl.Ep / pv::MAX_EB;
    for (int pass = 0; pass < n_passes; ++pass) {
        pv::Params P;
        P.un = F(pl.off_un);
        P.vn = F(pl.off_vn);
        P.out = out;
        P.partial = F(pl.off_partial);
        P.olong = F(pl.off_olong);
        P.tile_counter = counters;
        P.N = N;
        P.M = M;
        P.row_offset = row_offset;
        P.E = E;
        P.e0 = pass * pv::MAX_EB;
        P.eb = std::min(pv::MAX_EB, E - P.e0);
        P.ebp = (P.eb + 31) / 32 * 32;
        P.n_tiles = static_cast<int>(pl.n_tiles);
        P.nsb = static_cast<int>(pl.nsb);
        P.kblocks = pl.kblocks;
        P.stages = pl.stages;
        P.R = pl.waves.R;
        P.C = pl.waves.C;
        P.W = pl.waves.W;
        P.R_last = pl.waves.R_last;
        P.C_last = pl.waves.C_last;
        P.slots_per_wave = pl.waves.slots_per_wave;
        if (ev0 && pass == n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev0, stream));
        int rc;
        switch (tc::epilogue_kid(kid) * 2 + (norm ? 1 : 0)) {   // dot-exponential: the Gaussian instantiations
            case 0: rc = launch_pv<KMB_KERNEL_GAUSSIAN, false>(maps, P, grid, pl.smem, stream); break;
            case 1: rc = launch_pv<KMB_KERNEL_GAUSSIAN, true>(maps, P, grid, pl.smem, stream); break;
            case 2: rc = launch_pv<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, false>(maps, P, grid, pl.smem, stream); break;
            case 3: rc = launch_pv<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, true>(maps, P, grid, pl.smem, stream); break;
            case 4: rc = launch_pv<KMB_KERNEL_INVERSE_DISTANCE, false>(maps, P, grid, pl.smem, stream); break;
            default: rc = launch_pv<KMB_KERNEL_INVERSE_DISTANCE, true>(maps, P, grid, pl.smem, stream); break;
        }
        if (rc) return rc;
        if (ev1 && pass == n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev1, stream));
        count_launch();
    }
    return KMB_OK;
}

}  // namespace kmb
