// kprod_tensor: a_i = sum_j k(x_i, y_j) b_j for D > 16 on the 5th-generation tensor cores.
//
//   prepass   u = s (x - c), v = s (y - c)  (c = column means of y, s folds log2 e into the data),
//             split into TF32 hi / lo parts (3xTF32: hi.hi + hi.lo + lo.hi), squared norms in FP32.
//   main      persistent CTAs, warp-specialised:
//               warp 0      TMA producer: 128 x 32-float tiles of A = 2u (hi, lo), 256 x 32 of B = v (hi, lo),
//                           SWIZZLE_128B, 2-stage mbarrier ring of 96 KB stages
//               warp 1      MMA issuer: tcgen05.mma kind::tf32, M = 128, N = 256, K = 8 per instruction,
//                           S = 2 u.v accumulated in TMEM (two accumulator stages)
//               warps 2-5   epilogue: tcgen05.ld the S tile (one target row per thread), d2 = |u|^2 + |v|^2 - S,
//                           kernel function (MUFU), reduce against b in registers; online max-rescale for
//                           the row-normalised variant
//   work      waves of R row tiles x C CTAs per tile (R C <= grid): the CTAs of one row tile split its source
//             blocks into C contiguous ranges, and all R CTAs with the same range index walk the SAME
//             source blocks at the same time, so a v block is fetched from HBM once per wave and served to the
//             other R - 1 CTAs by L2 (with equal contiguous unit ranges per CTA, the first version, every CTA
//             sat at a different source block: 46.7 GB of DRAM reads per C3 product, 86 % of HBM peak).
//             Row tiles split over C > 1 CTAs are combined in range order by the last CTA to arrive.
//   operands  ELT_TF32: 3xTF32 (hi.hi + hi.lo + lo.hi), 32 floats per 128-byte K block.
//             ELT_F16:  the same three-term split with FP16 hi / lo parts of the data scaled by a power of
//             two (max |operand| in [2^13, 2^15)): 22 significand bits as 3xTF32, kind::f16 runs at twice
//             the TF32 rate and moves half the bytes; 64 halves per K block; S is rescaled in the epilogue.
//             ELT_F16X1: the hi planes of ELT_F16 alone (KMB_PATH_TENSOR_1XF16): one hi.hi MMA per K step, the lo
//             planes neither loaded nor counted on the barrier: 11 significand bits per operand, float16-class S.
#include <algorithm>
#include <cstdlib>

#include <cuda_fp16.h>

#include "kprod_tensor.cuh"
#include "tensor_common.cuh"

namespace kmb {

namespace tc {

#ifndef KMB_TC_TN
#define KMB_TC_TN 256
#endif
constexpr int TN = KMB_TC_TN;      // sources per tile      (UMMA N, one TMEM column per source): 128 or 256
static_assert(TN == 128 || TN == 256, "TN");
constexpr int STAGES = TN == 256 ? 2 : 3;
constexpr int TILE_BYTES = TM * 128;           // 16 KB: one 128-row A tile of 128-byte K blocks
constexpr int B_TILE_BYTES = TN * 128;         // one TN-row B tile
constexpr int STAGE_BYTES = 2 * TILE_BYTES + 2 * B_TILE_BYTES;    // A hi, A lo, B hi, B lo
constexpr int ACC_STAGES = 2;
constexpr int TMEM_COLS = ACC_STAGES * TN;     // 256 columns of 32-bit
constexpr int EPI_THREADS = 128;
constexpr int THREADS = 64 + EPI_THREADS;      // producer warp, MMA warp, 4 epilogue warps
constexpr int MAX_EP = 4;

struct Params {
    const float* un;     // (N) |u_i|^2
    const float* vn;     // (M) |v_j|^2
    const float* b;      // (M, E) signal or nullptr (density)
    float* out;          // (N, E)
    float* partial;
    int* tile_counter;
    const float* sscale; // FP16 planes: S = sscale[1] * accumulator (2^-2p); unused for TF32
    long long N, M, row_offset;
    int E, e0;
    int n_tiles, nsb, kblocks, ksteps_last;
    int R, C, W, R_last, C_last, slots_per_wave;   // wave schedule (plan_waves)
};

// work of CTA `cta` in wave w: row tile, source-block range [sb_lo, sb_hi), range index c of Cw
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
// instruction descriptor: D = F32, A = B = F16, both K-major
__host__ __device__ constexpr uint32_t idesc_f16(int n) {
    return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(TM >> 4) << 24);
}

template <int EP, int KID, bool NORM>
struct Cfg {
    static constexpr bool ONLINE_MAX = NORM && KID != KMB_KERNEL_INVERSE_DISTANCE;
    static constexpr int PS = EP + (NORM ? 1 : 0) + (ONLINE_MAX ? 1 : 0);
    static constexpr int AUX_FLOATS = TN * (1 + EP);   // |v|^2 and the signal chunk of one source block
    static constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGES * STAGE_BYTES + 2 * AUX_FLOATS * 4 +
                                      (2 * STAGES + 2 * ACC_STAGES) * 8 + 16;
};

template <int EP, int KID, bool NORM, int ELT>
__global__ void __launch_bounds__(THREADS, 1)
kprod_tensor_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                    const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                    const Params P) {
    using C = Cfg<EP, KID, NORM>;
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
    unsigned char* stages = smem;
    float* aux = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux + 2 * C::AUX_FLOATS);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* acc_full = empty_bar + STAGES;
    uint64_t* acc_empty = acc_full + ACC_STAGES;
    uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(acc_empty + ACC_STAGES);
    int* s_flag = reinterpret_cast<int*>(tmem_base_smem + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int cta = blockIdx.x;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], EPI_THREADS / 32); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc(tmem_base_smem, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_smem;

    if (warp == 0) {
        // ------------------------------------ TMA producer ------------------------------------
        // all 32 lanes walk the loop (uniform control flow); one elected lane issues (see elect_one)
        {
            constexpr int TKE = ELT == ELT_TF32 ? 32 : 64;   // elements per 128-byte K block
            constexpr bool LO = ELT != ELT_F16X1;             // the lo planes take part
            constexpr uint32_t TX_BYTES = LO ? STAGE_BYTES : TILE_BYTES + B_TILE_BYTES;
            uint32_t it = 0;
            WaveWork ww;
            for (int w = 0; w < P.W; ++w) {
                if (!wave_work(P, w, cta, ww)) continue;
                const int row0 = ww.tile * TM;
                for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb) {
                    const int src0 = sb * TN;
                    for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                        const int stage = it % STAGES;
                        mbar_wait(&empty_bar[stage], ((it / STAGES) & 1) ^ 1);
                        unsigned char* st = stages + stage * STAGE_BYTES;
                        if (elect_one()) {
                            mbar_arrive_expect_tx(&full_bar[stage], TX_BYTES);
                            tma_load_2d(st + 0 * TILE_BYTES, &map_ah, kb * TKE, row0, &full_bar[stage]);
                            if constexpr (LO) tma_load_2d(st + 1 * TILE_BYTES, &map_al, kb * TKE, row0, &full_bar[stage]);
                            tma_load_2d(st + 2 * TILE_BYTES, &map_bh, kb * TKE, src0, &full_bar[stage]);
                            if constexpr (LO) tma_load_2d(st + 2 * TILE_BYTES + B_TILE_BYTES, &map_bl, kb * TKE, src0, &full_bar[stage]);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------- MMA issuer -------------------------------------
        // all 32 lanes walk the loop and wait on the barriers; one elected lane issues (see elect_one)
        {
            uint32_t it = 0, unit = 0;
            WaveWork ww;
            for (int w = 0; w < P.W; ++w) {
                if (!wave_work(P, w, cta, ww)) continue;
                for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++unit) {
                    const int a = unit % ACC_STAGES;
                    mbar_wait(&acc_empty[a], ((unit / ACC_STAGES) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + a * TN;
                    for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                        const int stage = it % STAGES;
                        mbar_wait(&full_bar[stage], (it / STAGES) & 1);
                        tc_fence_after();
                        const unsigned char* st = stages + stage * STAGE_BYTES;
                        const int ksteps = (kb == P.kblocks - 1) ? P.ksteps_last : 4;
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) {   // 32 bytes of K per instruction
                                if (k < ksteps) {
                                    const uint64_t ah = umma_desc_sw128(st + 0 * TILE_BYTES, k * 32);
                                    const uint64_t al = umma_desc_sw128(st + 1 * TILE_BYTES, k * 32);
                                    const uint64_t bh = umma_desc_sw128(st + 2 * TILE_BYTES, k * 32);
                                    const uint64_t bl = umma_desc_sw128(st + 2 * TILE_BYTES + B_TILE_BYTES, k * 32);
                                    // three-term split: the two small cross terms first, then hi.hi
                                    if constexpr (ELT == ELT_F16X1) {
                                        umma_f16(d_tmem, ah, bh, idesc_f16(TN), (kb | k) != 0);
                                    } else if constexpr (ELT == ELT_F16) {
                                        umma_f16(d_tmem, al, bh, idesc_f16(TN), (kb | k) != 0);
                                        umma_f16(d_tmem, ah, bl, idesc_f16(TN), 1);
                                        umma_f16(d_tmem, ah, bh, idesc_f16(TN), 1);
                                    } else {
                                        umma_tf32(d_tmem, al, bh, idesc_tf32(TN), (kb | k) != 0);
                                        umma_tf32(d_tmem, ah, bl, idesc_tf32(TN), 1);
                                        umma_tf32(d_tmem, ah, bh, idesc_tf32(TN), 1);
                                    }
                                }
                            }
                            umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs have read it
                        }
                        __syncwarp();
                    }
                    if (elect_one()) umma_commit(&acc_full[a]);   // accumulator complete
                    __syncwarp();
                }
            }
        }
    } else {
        // -------------------------------------- epilogue --------------------------------------
        const int et = tid - 64;                       // 0..127
        const int lane_group = warp & 3;               // TMEM lanes this warp may access
        const int row_in_tile = lane_group * 32 + lane;
        [[maybe_unused]] float sscale = 1.f;
        if constexpr (ELT != ELT_TF32) sscale = __ldg(P.sscale + 1);
        uint32_t unit = 0;
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!wave_work(P, w, cta, ww)) continue;
            const int tile = ww.tile;
            const long long row = static_cast<long long>(tile) * TM + row_in_tile;
            const bool row_ok = row < P.N;
            const float un = row_ok ? __ldg(P.un + row) : 0.f;
            [[maybe_unused]] const long long jz = (P.row_offset + row) % (P.M + 1);

            float tot[EP], ktot = 0.f, kmax = -INFINITY;
#pragma unroll
            for (int e = 0; e < EP; ++e) tot[e] = 0.f;

            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++unit) {
                const long long j0 = static_cast<long long>(sb) * TN;
                // stage |v|^2 and the signal of this source block in shared memory (double buffered)
                float* ax = aux + (unit & 1) * C::AUX_FLOATS;
#pragma unroll
                for (int jt = et; jt < TN; jt += EPI_THREADS) {
                    const long long j = j0 + jt;
                    const bool live = j < P.M;
                    ax[jt] = live ? __ldg(P.vn + j) : 1.0e30f;   // padded sources: k underflows to 0
#pragma unroll
                    for (int e = 0; e < EP; ++e) {
                        float v = 0.f;
                        if (live && P.e0 + e < P.E) v = P.b ? __ldg(P.b + j * P.E + P.e0 + e) : 1.f;
                        ax[TN + jt * EP + e] = v;
                    }
                }
                named_bar_sync(1, EPI_THREADS);
                const int a = unit % ACC_STAGES;
                mbar_wait(&acc_full[a], (unit / ACC_STAGES) & 1);
                tc_fence_after();
                const uint32_t t_addr = tmem_base + a * TN + (static_cast<uint32_t>(lane_group * 32) << 16);

                float acc[EP], ksum = 0.f;
#pragma unroll
                for (int e = 0; e < EP; ++e) acc[e] = 0.f;
#pragma unroll 1
                for (int ch = 0; ch < TN / 32; ++ch) {
                    float s[32];
                    tmem_ld_32x32(t_addr + ch * 32, s);
                    if constexpr (ELT != ELT_TF32) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) s[c] *= sscale;   // exact: a power of two
                    }
                    if constexpr (!C::ONLINE_MAX) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            const int jj = ch * 32 + c;
                            float kv = kernel_from_parts<KID>(s[c], un, ax[jj]);
                            if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE)
                                if (j0 + jj == jz || j0 + jj >= P.M) kv = 0.f;  // zeroing rule; padding adds exactly 0
#pragma unroll
                            for (int e = 0; e < EP; ++e) acc[e] = fmaf(kv, ax[TN + jj * EP + e], acc[e]);
                            if constexpr (NORM) ksum += kv;
                        }
                    } else {
                        float cm = -INFINITY;
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            s[c] = log2_kernel_from_parts<KID>(s[c], un, ax[ch * 32 + c]);
                            cm = fmaxf(cm, s[c]);
                        }
                        const float mnew = fmaxf(kmax, cm);
                        const float sc = (mnew == -INFINITY) ? 1.f : ex2_approx(kmax - mnew);
                        const float moff = (mnew == -INFINITY) ? 0.f : mnew;
                        kmax = mnew;
                        // rescale everything accumulated so far (this unit and the tile totals)
                        ksum *= sc;
                        ktot *= sc;
#pragma unroll
                        for (int e = 0; e < EP; ++e) { acc[e] *= sc; tot[e] *= sc; }
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            const int jj = ch * 32 + c;
                            const float kv = ex2_approx(s[c] - moff);
#pragma unroll
                            for (int e = 0; e < EP; ++e) acc[e] = fmaf(kv, ax[TN + jj * EP + e], acc[e]);
                            ksum += kv;
                        }
                    }
                }
                // accumulator drained: hand the TMEM stage back to the MMA warp
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[a]);
                // two-level summation (see kprod_direct.cuh)
#pragma unroll
                for (int e = 0; e < EP; ++e) tot[e] += acc[e];
                ktot += ksum;
            }

            // ------------------------------ write this row tile ------------------------------
            if (ww.Cw == 1) {
                if (row_ok) {
#pragma unroll
                    for (int e = 0; e < EP; ++e)
                        if (P.e0 + e < P.E) P.out[row * P.E + P.e0 + e] = NORM ? tot[e] / ktot : tot[e];
                }
            } else {
                // one partial per (wave, CTA); the last CTA of the row tile to arrive adds them in range order
                const size_t slot0 = static_cast<size_t>(w) * P.slots_per_wave + static_cast<size_t>(ww.tile_in_wave) * ww.Cw;
                float* mine = P.partial + (slot0 + ww.c) * (TM * C::PS);
#pragma unroll
                for (int e = 0; e < EP; ++e) mine[e * TM + row_in_tile] = tot[e];
                if constexpr (NORM) mine[EP * TM + row_in_tile] = ktot;
                if constexpr (C::ONLINE_MAX) mine[(EP + 1) * TM + row_in_tile] = kmax;
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
                    float sum[EP], l = 0.f, mx = -INFINITY;
#pragma unroll
                    for (int e = 0; e < EP; ++e) sum[e] = 0.f;
                    if constexpr (C::ONLINE_MAX) {
                        for (int c = 0; c < ww.Cw; ++c)
                            mx = fmaxf(mx, __ldcg(P.partial + (slot0 + c) * (TM * C::PS) + (EP + 1) * TM + row_in_tile));
                    }
                    for (int c = 0; c < ww.Cw; ++c) {
                        const float* ps = P.partial + (slot0 + c) * (TM * C::PS);
                        float wgt = 1.f;
                        if constexpr (C::ONLINE_MAX) {
                            const float m = __ldcg(ps + (EP + 1) * TM + row_in_tile);
                            wgt = (m == -INFINITY) ? 0.f : ex2_approx(m - mx);
                        }
#pragma unroll
                        for (int e = 0; e < EP; ++e) sum[e] = fmaf(wgt, __ldcg(ps + e * TM + row_in_tile), sum[e]);
                        if constexpr (NORM) l = fmaf(wgt, __ldcg(ps + EP * TM + row_in_tile), l);
                    }
#pragma unroll
                    for (int e = 0; e < EP; ++e)
                        if (P.e0 + e < P.E) P.out[row * P.E + P.e0 + e] = NORM ? sum[e] / l : sum[e];
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ---- CTA pairs (cta_group::2), FP16 planes -----------------------------------------------------------------
// The single-CTA kernel above fetches 48 KB of operands from L2 per 6 MMAs and runs into the L2 -> SM bandwidth
// (ncu: 11.6 TB/s, tensor pipe 72 %).  Here two CTAs on neighbouring SMs work on two adjacent 128-row tiles and the
// same 256 sources: each loads its own A tile and HALF of the B block, and one tcgen05.mma.cta_group::2 of shape
// 256 x 256 x 16 (issued by the leader CTA) reads A from both CTAs' shared memory and the two B halves, leaving each
// CTA its own 128 x 256 accumulator in its own TMEM.  Operand bytes per CTA and K block: 32 KB of A + 32 KB of B
// (was 32 + 64), and a stage of 64 KB lets three stages fit.
//   full_bar   leader's; both producers' TMA bytes land on it (cp.async.bulk.tensor ... cta_group::2), the leader's
//              producer arms it with the bytes of both CTAs, the peer's producer arrives remotely
//   empty_bar  one per CTA; the leader's tcgen05.commit multicasts to both
//   acc_full   one per CTA (multicast commit); acc_empty: leader's, 8 arrivals (4 epilogue warps of each CTA)
// TERMS = 3: lo.hi + hi.lo + hi.hi (KMB_PATH_TENSOR_3XF16); TERMS = 1: hi.hi only, the lo planes are not loaded
// (KMB_PATH_TENSOR_1XF16).
namespace pair {

constexpr int STAGES2 = 3;
constexpr int BH_BYTES = 128 * 128;                      // this CTA's half of a B tile: 128 sources x 128 bytes
constexpr int STAGE2_BYTES = 2 * TILE_BYTES + 2 * BH_BYTES;   // A hi, A lo, B-half hi, B-half lo = 64 KB

// D = F32, A = B = F16, K-major, M = 256 (two CTAs x 128 rows), N = 256
__host__ __device__ constexpr uint32_t idesc2_f16() {
    return (1u << 4) | (static_cast<uint32_t>(TN >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);
}

template <int EP, int KID, bool NORM>
struct Cfg2 {
    static constexpr int SMEM_BYTES = 1024 + STAGES2 * STAGE2_BYTES + 2 * Cfg<EP, KID, NORM>::AUX_FLOATS * 4 +
                                      (2 * STAGES2 + 2 * ACC_STAGES) * 8 + 16;
};

// work of cluster `cid` in wave w (the wave plan counts pairs of row tiles and clusters)
__device__ __forceinline__ bool pair_wave_work(const Params& P, int w, int cid, WaveWork& ww) {
    const bool last = (w == P.W - 1);
    const int Rw = last ? P.R_last : P.R, Cw = last ? P.C_last : P.C;
    if (cid >= Rw * Cw) return false;
    ww.Cw = Cw;
    ww.tile_in_wave = cid / Cw;              // pair of row tiles within the wave
    ww.c = cid - ww.tile_in_wave * Cw;
    ww.tile = w * P.R + ww.tile_in_wave;     // pair index
    ww.sb_lo = static_cast<int>(static_cast<long long>(P.nsb) * ww.c / Cw);
    ww.sb_hi = static_cast<int>(static_cast<long long>(P.nsb) * (ww.c + 1) / Cw);
    return true;
}

template <int EP, int KID, bool NORM, int TERMS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
kprod_tensor_pair_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                         const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                         const Params P) {
    using C = Cfg<EP, KID, NORM>;
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
    unsigned char* stages = smem;
    float* aux = reinterpret_cast<float*>(smem + STAGES2 * STAGE2_BYTES);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux + 2 * C::AUX_FLOATS);
    uint64_t* empty_bar = full_bar + STAGES2;
    uint64_t* acc_full = empty_bar + STAGES2;
    uint64_t* acc_empty = acc_full + ACC_STAGES;
    uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(acc_empty + ACC_STAGES);
    int* s_flag = reinterpret_cast<int*>(tmem_base_smem + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();          // 0 = leader (issues the MMAs), 1 = peer
    const int cid = blockIdx.x >> 1;

    if (tid == 0) {
        for (int s = 0; s < STAGES2; ++s) { mbar_init(&full_bar[s], 2); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 2 * (EPI_THREADS / 32)); }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc2(tmem_base_smem, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // the peer's barriers are initialised before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_smem;

    if (warp == 0) {
        // ------------------------------------ TMA producer (both CTAs) ------------------------------------
        uint32_t it = 0;
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!pair_wave_work(P, w, cid, ww)) continue;
            const int row0 = (ww.tile * 2 + static_cast<int>(rank)) * TM;
            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb) {
                const int src0 = sb * TN + static_cast<int>(rank) * 128;   // this CTA's half of the source block
                for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                    const int stage = it % STAGES2;
                    mbar_wait(&empty_bar[stage], ((it / STAGES2) & 1) ^ 1);
                    unsigned char* st = stages + stage * STAGE2_BYTES;
                    const uint32_t leader_full = map_to_cta(&full_bar[stage], 0);
                    if (elect_one()) {
                        constexpr uint32_t tx = TERMS == 3 ? STAGE2_BYTES : TILE_BYTES + BH_BYTES;
                        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * tx);   // both CTAs' bytes
                        else mbar_arrive_cluster(leader_full);
                        tma_load_2d_pair(st + 0 * TILE_BYTES, &map_ah, kb * 64, row0, leader_full);
                        if constexpr (TERMS == 3) tma_load_2d_pair(st + 1 * TILE_BYTES, &map_al, kb * 64, row0, leader_full);
                        tma_load_2d_pair(st + 2 * TILE_BYTES, &map_bh, kb * 64, src0, leader_full);
                        if constexpr (TERMS == 3) tma_load_2d_pair(st + 2 * TILE_BYTES + BH_BYTES, &map_bl, kb * 64, src0, leader_full);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------- MMA issuer (leader CTA only) -------------------------------------
        if (rank == 0) {
            uint32_t it = 0, unit = 0;
            WaveWork ww;
            for (int w = 0; w < P.W; ++w) {
                if (!pair_wave_work(P, w, cid, ww)) continue;
                for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++unit) {
                    const int a = unit % ACC_STAGES;
                    mbar_wait(&acc_empty[a], ((unit / ACC_STAGES) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + a * TN;
                    for (int kb = 0; kb < P.kblocks; ++kb, ++it) {
                        const int stage = it % STAGES2;
                        mbar_wait(&full_bar[stage], (it / STAGES2) & 1);
                        tc_fence_after();
                        const unsigned char* st = stages + stage * STAGE2_BYTES;
                        const int ksteps = (kb == P.kblocks - 1) ? P.ksteps_last : 4;
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (k < ksteps) {
                                    const uint64_t ah = umma_desc_sw128(st + 0 * TILE_BYTES, k * 32);
                                    const uint64_t al = umma_desc_sw128(st + 1 * TILE_BYTES, k * 32);
                                    const uint64_t bh = umma_desc_sw128(st + 2 * TILE_BYTES, k * 32);
                                    const uint64_t bl = umma_desc_sw128(st + 2 * TILE_BYTES + BH_BYTES, k * 32);
                                    if constexpr (TERMS == 3) {
                                        umma2_f16(d_tmem, al, bh, idesc2_f16(), (kb | k) != 0);
                                        umma2_f16(d_tmem, ah, bl, idesc2_f16(), 1);
                                        umma2_f16(d_tmem, ah, bh, idesc2_f16(), 1);
                                    } else {
                                        umma2_f16(d_tmem, ah, bh, idesc2_f16(), (kb | k) != 0);
                                    }
                                }
                            }
                            umma2_commit_both(&empty_bar[stage]);   // both CTAs' slots are reusable
                        }
                        __syncwarp();
                    }
                    if (elect_one()) umma2_commit_both(&acc_full[a]);   // both CTAs' accumulators are complete
                    __syncwarp();
                }
            }
        }
    } else {
        // -------------------------------------- epilogue (both CTAs) --------------------------------------
        const int et = tid - 64;
        const int lane_group = warp & 3;
        const int row_in_tile = lane_group * 32 + lane;
        const float sscale = __ldg(P.sscale + 1);
        uint32_t unit = 0;
        WaveWork ww;
        for (int w = 0; w < P.W; ++w) {
            if (!pair_wave_work(P, w, cid, ww)) continue;
            const int tile = ww.tile * 2 + static_cast<int>(rank);
            const long long row = static_cast<long long>(tile) * TM + row_in_tile;
            const bool row_ok = row < P.N;
            const float un = row_ok ? __ldg(P.un + row) : 0.f;
            [[maybe_unused]] const long long jz = (P.row_offset + row) % (P.M + 1);

            float tot[EP], ktot = 0.f, kmax = -INFINITY;
#pragma unroll
            for (int e = 0; e < EP; ++e) tot[e] = 0.f;

            for (int sb = ww.sb_lo; sb < ww.sb_hi; ++sb, ++unit) {
                const long long j0 = static_cast<long long>(sb) * TN;
                float* ax = aux + (unit & 1) * C::AUX_FLOATS;
#pragma unroll
                for (int jt = et; jt < TN; jt += EPI_THREADS) {
                    const long long j = j0 + jt;
                    const bool live = j < P.M;
                    ax[jt] = live ? __ldg(P.vn + j) : 1.0e30f;
#pragma unroll
                    for (int e = 0; e < EP; ++e) {
                        float v = 0.f;
                        if (live && P.e0 + e < P.E) v = P.b ? __ldg(P.b + j * P.E + P.e0 + e) : 1.f;
                        ax[TN + jt * EP + e] = v;
                    }
                }
                named_bar_sync(1, EPI_THREADS);
                const int a = unit % ACC_STAGES;
                mbar_wait(&acc_full[a], (unit / ACC_STAGES) & 1);
                tc_fence_after();
                const uint32_t t_addr = tmem_base + a * TN + (static_cast<uint32_t>(lane_group * 32) << 16);

                float acc[EP], ksum = 0.f;
#pragma unroll
                for (int e = 0; e < EP; ++e) acc[e] = 0.f;
#pragma unroll 1
                for (int ch = 0; ch < TN / 32; ++ch) {
                    float s[32];
                    tmem_ld_32x32(t_addr + ch * 32, s);
#pragma unroll
                    for (int c = 0; c < 32; ++c) s[c] *= sscale;
                    if constexpr (!C::ONLINE_MAX) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            const int jj = ch * 32 + c;
                            float kv = kernel_from_parts<KID>(s[c], un, ax[jj]);
                            if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE)
                                if (j0 + jj == jz || j0 + jj >= P.M) kv = 0.f;
#pragma unroll
                            for (int e = 0; e < EP; ++e) acc[e] = fmaf(kv, ax[TN + jj * EP + e], acc[e]);
                            if constexpr (NORM) ksum += kv;
                        }
                    } else {
                        float cm = -INFINITY;
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            s[c] = log2_kernel_from_parts<KID>(s[c], un, ax[ch * 32 + c]);
                            cm = fmaxf(cm, s[c]);
                        }
                        const float mnew = fmaxf(kmax, cm);
                        const float sc = (mnew == -INFINITY) ? 1.f : ex2_approx(kmax - mnew);
                        const float moff = (mnew == -INFINITY) ? 0.f : mnew;
                        kmax = mnew;
                        ksum *= sc;
                        ktot *= sc;
#pragma unroll
                        for (int e = 0; e < EP; ++e) { acc[e] *= sc; tot[e] *= sc; }
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            const int jj = ch * 32 + c;
                            const float kv = ex2_approx(s[c] - moff);
#pragma unroll
                            for (int e = 0; e < EP; ++e) acc[e] = fmaf(kv, ax[TN + jj * EP + e], acc[e]);
                            ksum += kv;
                        }
                    }
                }
                // accumulator drained: tell the leader's MMA warp (remote arrive from the peer)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (rank != 0) mbar_arrive_cluster(map_to_cta(&acc_empty[a], 0));
                    else mbar_arrive(&acc_empty[a]);
                }
#pragma unroll
                for (int e = 0; e < EP; ++e) tot[e] += acc[e];
                ktot += ksum;
            }

            // ------------------------------ write this row tile ------------------------------
            if (tile < P.n_tiles) {   // the last pair may hold a ghost tile (odd number of row tiles)
                if (ww.Cw == 1) {
                    if (row_ok) {
#pragma unroll
                        for (int e = 0; e < EP; ++e)
                            if (P.e0 + e < P.E) P.out[row * P.E + P.e0 + e] = NORM ? tot[e] / ktot : tot[e];
                    }
                } else {
                    // partial records of one wave: [pair in wave][range c][rank]
                    const size_t slot0 = static_cast<size_t>(w) * P.slots_per_wave + static_cast<size_t>(ww.tile_in_wave) * ww.Cw * 2 + rank;
                    float* mine = P.partial + (slot0 + ww.c * 2) * (TM * C::PS);
#pragma unroll
                    for (int e = 0; e < EP; ++e) mine[e * TM + row_in_tile] = tot[e];
                    if constexpr (NORM) mine[EP * TM + row_in_tile] = ktot;
                    if constexpr (C::ONLINE_MAX) mine[(EP + 1) * TM + row_in_tile] = kmax;
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
                        float sum[EP], l = 0.f, mx = -INFINITY;
#pragma unroll
                        for (int e = 0; e < EP; ++e) sum[e] = 0.f;
                        if constexpr (C::ONLINE_MAX) {
                            for (int c = 0; c < ww.Cw; ++c)
                                mx = fmaxf(mx, __ldcg(P.partial + (slot0 + c * 2) * (TM * C::PS) + (EP + 1) * TM + row_in_tile));
                        }
                        for (int c = 0; c < ww.Cw; ++c) {
                            const float* ps = P.partial + (slot0 + c * 2) * (TM * C::PS);
                            float wgt = 1.f;
                            if constexpr (C::ONLINE_MAX) {
                                const float m = __ldcg(ps + (EP + 1) * TM + row_in_tile);
                                wgt = (m == -INFINITY) ? 0.f : ex2_approx(m - mx);
                            }
#pragma unroll
                            for (int e = 0; e < EP; ++e) sum[e] = fmaf(wgt, __ldcg(ps + e * TM + row_in_tile), sum[e]);
                            if constexpr (NORM) l = fmaf(wgt, __ldcg(ps + EP * TM + row_in_tile), l);
                        }
#pragma unroll
                        for (int e = 0; e < EP; ++e)
                            if (P.e0 + e < P.E) P.out[row * P.E + P.e0 + e] = NORM ? sum[e] / l : sum[e];
                    }
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // neither CTA frees tensor memory (or exits) while the other may still signal it
    if (warp == 1) tmem_dealloc2(tmem_base, TMEM_COLS);
}

}  // namespace pair

// ---- prepass ---------------------------------------------------------------------------------------

// partial[blk][col] = sum over this block's rows of y[row][col]
static __global__ void __launch_bounds__(256) column_sum_kernel(const float* __restrict__ y, long long M, int D,
                                                                float* __restrict__ partial) {
    __shared__ float sm[8][32];
    const int col = blockIdx.y * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;
    float acc = 0.f;
    if (col < D)
        for (long long r = blockIdx.x * 8 + rl; r < M; r += static_cast<long long>(gridDim.x) * 8) acc += y[r * D + col];
    sm[rl][threadIdx.x & 31] = acc;
    __syncthreads();
    if (rl == 0 && col < D) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += sm[i][threadIdx.x];
        partial[static_cast<size_t>(blockIdx.x) * D + col] = t;
    }
}
static __global__ void column_mean_kernel(const float* __restrict__ partial, int blocks, long long M, int D, int Dp,
                                          float* __restrict__ center) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= Dp) return;
    float t = 0.f;
    if (col < D)
        for (int b = 0; b < blocks; ++b) t += partial[static_cast<size_t>(b) * D + col];
    center[col] = col < D ? t / static_cast<float>(M) : 0.f;
}

// One warp per point: w = mult * s * (p - c); hi = tf32(w), lo = tf32(w - hi); norm2 = |s (p - c)|^2.
static __global__ void __launch_bounds__(256) split_points_kernel(const float* __restrict__ pts, long long n, int D, int Dp,
                                                                  const float* __restrict__ center, float scale, float mult,
                                                                  float* __restrict__ hi, float* __restrict__ lo,
                                                                  float* __restrict__ norm2) {
    const long long row = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    float acc = 0.f;
    for (int d = lane; d < Dp; d += 32) {
        float w = 0.f;
        if (d < D) w = scale * (pts[row * D + d] - center[d]);
        acc = fmaf(w, w, acc);
        w *= mult;
        const float h = to_tf32(w);
        hi[row * Dp + d] = h;
        lo[row * Dp + d] = to_tf32(w - h);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) norm2[row] = acc;
}

// One warp per point of the dot-exponential kernel: operand = s p (TF32) or s 2^p p (FP16; 2^p = sscale[0]), uncentred and
// with multiplier 1 on both planes, split into hi + lo; norm2 = 0.  S = s^2 <x, y> = log2(e) <x, y> is then what the
// Gaussian epilogue's S - |u|^2 - |v|^2 evaluates: the log2 of exp(<x, y>).
constexpr float kDotScale = 1.2011224087864498f;   // sqrt(log2 e)
template <int ELT>
static __global__ void __launch_bounds__(256) split_points_dot_kernel(const float* __restrict__ pts, long long n, int D, int Dp,
                                                                      float scale, const float* __restrict__ sscale, void* hi,
                                                                      void* lo, float* __restrict__ norm2) {
    const long long row = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const float m = ELT == ELT_F16 ? scale * __ldg(sscale) : scale;
    for (int d = lane; d < Dp; d += 32) {
        const float w = d < D ? m * pts[row * D + d] : 0.f;
        if constexpr (ELT == ELT_F16) {
            const __half h = __float2half_rn(w);
            static_cast<__half*>(hi)[row * Dp + d] = h;
            static_cast<__half*>(lo)[row * Dp + d] = __float2half_rn(w - __half2float(h));
        } else {
            const float h = to_tf32(w);
            static_cast<float*>(hi)[row * Dp + d] = h;
            static_cast<float*>(lo)[row * Dp + d] = to_tf32(w - h);
        }
    }
    if (lane == 0) norm2[row] = 0.f;
}

// (rows, cols) fp32 row-major; box = 32 floats x box_rows rows, 128-byte swizzle, out-of-bounds reads as zero
int make_tensor_map(CUtensorMap* map, const float* base, long long rows, int cols, int box_rows) {
    using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn enc = nullptr;
    if (!enc) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        KMB_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess) return set_error(KMB_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        enc = reinterpret_cast<EncodeFn>(p);
    }
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 4};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(TK), static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(KMB_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", static_cast<int>(r));
    return KMB_OK;
}

int tensor_prepass(const float* x, const float* y, int64_t N, int64_t M, int D, int Dp, int kid, float* center, float* cpart,
                   float* uh, float* ul, float* vh, float* vl, float* un, float* vn, cudaStream_t stream) {
    if (kid == KMB_KERNEL_DOT_EXPONENTIAL) {   // no centre, no squared norms
        split_points_dot_kernel<ELT_TF32><<<static_cast<unsigned>((N * 32 + 255) / 256), 256, 0, stream>>>(x, N, D, Dp, kDotScale, nullptr, uh, ul, un);
        KMB_CUDA_CHECK(cudaGetLastError());
        split_points_dot_kernel<ELT_TF32><<<static_cast<unsigned>((M * 32 + 255) / 256), 256, 0, stream>>>(y, M, D, Dp, kDotScale, nullptr, vh, vl, vn);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch(2);
        return KMB_OK;
    }
    // scale folds log2(e) into the data as in the direct path; the A operand carries the factor 2 of 2 u.v
    const float scale = kid == KMB_KERNEL_GAUSSIAN ? 1.2011224087864498f : kid == KMB_KERNEL_ABSOLUTE_EXPONENTIAL ? 1.4426950408889634f : 1.f;
    const int cblocks = static_cast<int>(std::min<long long>(CENTER_BLOCKS, (M + 7) / 8));
    dim3 g(cblocks, (D + 31) / 32);
    column_sum_kernel<<<g, 256, 0, stream>>>(y, M, D, cpart);
    KMB_CUDA_CHECK(cudaGetLastError());
    column_mean_kernel<<<(Dp + 127) / 128, 128, 0, stream>>>(cpart, cblocks, M, D, Dp, center);
    KMB_CUDA_CHECK(cudaGetLastError());
    split_points_kernel<<<static_cast<unsigned>((N * 32 + 255) / 256), 256, 0, stream>>>(x, N, D, Dp, center, scale, 2.f, uh, ul, un);
    KMB_CUDA_CHECK(cudaGetLastError());
    split_points_kernel<<<static_cast<unsigned>((M * 32 + 255) / 256), 256, 0, stream>>>(y, M, D, Dp, center, scale, 1.f, vh, vl, vn);
    KMB_CUDA_CHECK(cudaGetLastError());
    count_launch(4);
    return KMB_OK;
}


// ---- FP16 operands ---------------------------------------------------------------------------------

// per block: column sums, minima and maxima of its rows
static __global__ void __launch_bounds__(256) column_stats_kernel(const float* __restrict__ pts, long long n, int D,
                                                                  float* __restrict__ psum, float* __restrict__ pmin,
                                                                  float* __restrict__ pmax) {
    __shared__ float sm[3][8][32];
    const int col = blockIdx.y * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;
    float acc = 0.f, lo = INFINITY, hi = -INFINITY;
    if (col < D)
        for (long long r = blockIdx.x * 8 + rl; r < n; r += static_cast<long long>(gridDim.x) * 8) {
            const float v = pts[r * D + col];
            acc += v;
            lo = fminf(lo, v);
            hi = fmaxf(hi, v);
        }
    sm[0][rl][threadIdx.x & 31] = acc;
    sm[1][rl][threadIdx.x & 31] = lo;
    sm[2][rl][threadIdx.x & 31] = hi;
    __syncthreads();
    if (rl == 0 && col < D) {
        float t = 0.f, l = INFINITY, h = -INFINITY;
        for (int i = 0; i < 8; ++i) {
            t += sm[0][i][threadIdx.x];
            l = fminf(l, sm[1][i][threadIdx.x]);
            h = fmaxf(h, sm[2][i][threadIdx.x]);
        }
        psum[static_cast<size_t>(blockIdx.x) * D + col] = t;
        pmin[static_cast<size_t>(blockIdx.x) * D + col] = l;
        pmax[static_cast<size_t>(blockIdx.x) * D + col] = h;
    }
}
// red[0 .. 255] = per-thread largest |coordinate| (before the scale s): max-reduce, then sscale[0] = 2^p with
// 2^p s max in [2^13, 2^14), sscale[1] = 2^-2p
__device__ __forceinline__ void operand_scale(float* red, float scale, float* __restrict__ sscale) {
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float mw = scale * red[0];
        int p = 0;
        if (mw > 0.f && mw < INFINITY) p = 13 - ilogbf(mw);   // 2^p mw in [2^13, 2^14)
        p = max(-60, min(60, p));
        sscale[0] = exp2f(static_cast<float>(p));
        sscale[1] = exp2f(static_cast<float>(-2 * p));
    }
}
// one block: centre = column means of y; the largest |point - centre| follows from the column extrema
static __global__ void __launch_bounds__(256) center_scale_kernel(const float* __restrict__ ystats, int yblocks,
                                                                  const float* __restrict__ xstats, int xblocks, long long M,
                                                                  int D, int Dp, float scale, float* __restrict__ center,
                                                                  float* __restrict__ sscale) {
    __shared__ float red[256];
    const size_t plane_y = static_cast<size_t>(CENTER_BLOCKS) * D;
    float dev = 0.f;
    for (int col = threadIdx.x; col < Dp; col += 256) {
        float c = 0.f;
        if (col < D) {
            float t = 0.f, lo = INFINITY, hi = -INFINITY;
            for (int b = 0; b < yblocks; ++b) {
                t += ystats[static_cast<size_t>(b) * D + col];
                lo = fminf(lo, ystats[plane_y + static_cast<size_t>(b) * D + col]);
                hi = fmaxf(hi, ystats[2 * plane_y + static_cast<size_t>(b) * D + col]);
            }
            for (int b = 0; b < xblocks; ++b) {
                lo = fminf(lo, xstats[plane_y + static_cast<size_t>(b) * D + col]);
                hi = fmaxf(hi, xstats[2 * plane_y + static_cast<size_t>(b) * D + col]);
            }
            c = t / static_cast<float>(M);
            dev = fmaxf(dev, fmaxf(hi - c, c - lo));
        }
        center[col] = c;
    }
    red[threadIdx.x] = dev;
    operand_scale(red, scale, sscale);
}
// one block: the dot-exponential kernel's operands are not centred, so p follows from the largest |coordinate| of x and y
static __global__ void __launch_bounds__(256) dot_scale_kernel(const float* __restrict__ ystats, int yblocks,
                                                               const float* __restrict__ xstats, int xblocks, int D, float scale,
                                                               float* __restrict__ sscale) {
    __shared__ float red[256];
    const size_t plane = static_cast<size_t>(CENTER_BLOCKS) * D;
    float mag = 0.f;
    for (int col = threadIdx.x; col < D; col += 256) {
        for (int b = 0; b < yblocks; ++b)
            mag = fmaxf(mag, fmaxf(-ystats[plane + static_cast<size_t>(b) * D + col], ystats[2 * plane + static_cast<size_t>(b) * D + col]));
        for (int b = 0; b < xblocks; ++b)
            mag = fmaxf(mag, fmaxf(-xstats[plane + static_cast<size_t>(b) * D + col], xstats[2 * plane + static_cast<size_t>(b) * D + col]));
    }
    red[threadIdx.x] = mag;
    operand_scale(red, scale, sscale);
}
// One warp per point: w = s (p - c); operand = mult 2^p w split into FP16 hi + lo; norm2 = |w|^2.
static __global__ void __launch_bounds__(256) split_points_f16_kernel(const float* __restrict__ pts, long long n, int D, int Dp,
                                                                      const float* __restrict__ center, float scale, float mult,
                                                                      const float* __restrict__ sscale, __half* __restrict__ hi,
                                                                      __half* __restrict__ lo, float* __restrict__ norm2) {
    const long long row = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const float m2 = mult * __ldg(sscale);
    float acc = 0.f;
    for (int d = lane; d < Dp; d += 32) {
        float w = 0.f;
        if (d < D) w = scale * (pts[row * D + d] - center[d]);
        acc = fmaf(w, w, acc);
        w *= m2;
        const __half h = __float2half_rn(w);
        hi[row * Dp + d] = h;
        lo[row * Dp + d] = __float2half_rn(w - __half2float(h));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) norm2[row] = acc;
}

int make_tensor_map_f16(CUtensorMap* map, const void* base, long long rows, int cols, int box_rows) {
    using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn enc = nullptr;
    if (!enc) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        KMB_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess) return set_error(KMB_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        enc = reinterpret_cast<EncodeFn>(p);
    }
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
    const cuuint32_t box[2] = {64u, static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(KMB_ERR_CUDA, "cuTensorMapEncodeTiled (f16) failed with %d", static_cast<int>(r));
    return KMB_OK;
}

int tensor_prepass_f16(const float* x, const float* y, int64_t N, int64_t M, int D, int Dp16, int kid, float* center,
                       float* stats, float* sscale, void* uh, void* ul, void* vh, void* vl, float* un, float* vn,
                       cudaStream_t stream) {
    const float scale = kid == KMB_KERNEL_GAUSSIAN ? 1.2011224087864498f : kid == KMB_KERNEL_ABSOLUTE_EXPONENTIAL ? 1.4426950408889634f : 1.f;
    const size_t plane = static_cast<size_t>(CENTER_BLOCKS) * D;
    float* ys = stats;
    float* xs = stats + 3 * plane;
    const int yblocks = static_cast<int>(std::min<long long>(CENTER_BLOCKS, (M + 7) / 8));
    const int xblocks = static_cast<int>(std::min<long long>(CENTER_BLOCKS, (N + 7) / 8));
    column_stats_kernel<<<dim3(yblocks, (D + 31) / 32), 256, 0, stream>>>(y, M, D, ys, ys + plane, ys + 2 * plane);
    KMB_CUDA_CHECK(cudaGetLastError());
    column_stats_kernel<<<dim3(xblocks, (D + 31) / 32), 256, 0, stream>>>(x, N, D, xs, xs + plane, xs + 2 * plane);
    KMB_CUDA_CHECK(cudaGetLastError());
    if (kid == KMB_KERNEL_DOT_EXPONENTIAL) {   // no centre, no squared norms (|v|^2 of padded sources: f16_points_prepass)
        dot_scale_kernel<<<1, 256, 0, stream>>>(ys, yblocks, xs, xblocks, D, kDotScale, sscale);
        KMB_CUDA_CHECK(cudaGetLastError());
        split_points_dot_kernel<ELT_F16><<<static_cast<unsigned>((N * 32 + 255) / 256), 256, 0, stream>>>(x, N, D, Dp16, kDotScale, sscale, uh, ul, un);
        KMB_CUDA_CHECK(cudaGetLastError());
        split_points_dot_kernel<ELT_F16><<<static_cast<unsigned>((M * 32 + 255) / 256), 256, 0, stream>>>(y, M, D, Dp16, kDotScale, sscale, vh, vl, vn);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch(5);
        return KMB_OK;
    }
    center_scale_kernel<<<1, 256, 0, stream>>>(ys, yblocks, xs, xblocks, M, D, Dp16, scale, center, sscale);
    KMB_CUDA_CHECK(cudaGetLastError());
    split_points_f16_kernel<<<static_cast<unsigned>((N * 32 + 255) / 256), 256, 0, stream>>>(
        x, N, D, Dp16, center, scale, 2.f, sscale, static_cast<__half*>(uh), static_cast<__half*>(ul), un);
    KMB_CUDA_CHECK(cudaGetLastError());
    split_points_f16_kernel<<<static_cast<unsigned>((M * 32 + 255) / 256), 256, 0, stream>>>(
        y, M, D, Dp16, center, scale, 1.f, sscale, static_cast<__half*>(vh), static_cast<__half*>(vl), vn);
    KMB_CUDA_CHECK(cudaGetLastError());
    count_launch(5);
    return KMB_OK;
}

// Choose R (row tiles per wave) to minimise the number of source-block steps a CTA walks; ties go to the
// larger R (each v block is read from HBM once per wave).  R row tiles of u must stay L2-resident.
void plan_waves(long long n_tiles, long long nsb, int grid, size_t row_tile_bytes, WavePlan* wp) {
    const size_t l2_budget = 48u << 20;
    long long rmax = static_cast<long long>(l2_budget / std::max<size_t>(row_tile_bytes, 1));
    rmax = std::max<long long>(rmax, (grid + nsb - 1) / nsb);   // few source blocks: enough row tiles to keep every CTA busy
    rmax = std::max<long long>(1, std::min<long long>({rmax, static_cast<long long>(grid), n_tiles}));
    long long best_steps = -1;
    for (long long R = 1; R <= rmax; ++R) {
        const long long C = std::max<long long>(1, std::min<long long>(grid / R, nsb));
        const long long W = (n_tiles + R - 1) / R;
        const long long Rl = n_tiles - (W - 1) * R;
        const long long Cl = std::max<long long>(1, std::min<long long>(grid / Rl, nsb));
        const long long steps = (W - 1) * ((nsb + C - 1) / C) + (nsb + Cl - 1) / Cl;
        if (best_steps < 0 || steps <= best_steps) {
            best_steps = steps;
            wp->R = static_cast<int>(R);
            wp->C = static_cast<int>(C);
            wp->W = static_cast<int>(W);
            wp->R_last = static_cast<int>(Rl);
            wp->C_last = static_cast<int>(Cl);
        }
    }
    // partial results: one slot per (wave, CTA) when the full waves split row tiles, else only the last wave does
    const bool all = wp->C > 1 && wp->W > 1;
    const bool any = all || wp->C_last > 1;
    wp->slots_per_wave = all ? grid : 0;
    wp->partial_slots = all ? static_cast<long long>(wp->W) * grid : (any ? grid : 1);
}

}  // namespace tc

// ---- host side ---------------------------------------------------------------------------------------
void f16_points_layout(int64_t N, int64_t M, int D, F16PointsLayout* L) {
    auto up = [](size_t v, size_t a) { return (v + a - 1) / a * a; };
    L->Dp = (D + 15) / 16 * 16;
    L->Mv = (M + 255) / 256 * 256;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += up(bytes, 256); return at; };
    L->off_center = take(sizeof(float) * L->Dp);
    L->off_stats = take(sizeof(float) * tc::CENTER_BLOCKS * D * 6);
    L->off_sscale = take(sizeof(float) * 2);
    L->off_uh = take(2 * static_cast<size_t>(N) * L->Dp);
    L->off_ul = take(2 * static_cast<size_t>(N) * L->Dp);
    L->off_vh = take(2 * static_cast<size_t>(M) * L->Dp);
    L->off_vl = take(2 * static_cast<size_t>(M) * L->Dp);
    L->off_un = take(sizeof(float) * N);
    L->off_vn = take(sizeof(float) * L->Mv);
    L->end = o;
}

int f16_points_prepass(const float* x, const float* y, int64_t N, int64_t M, int D, int kid, const F16PointsLayout& L, char* ws,
                       cudaStream_t stream) {
    auto F = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
    if (L.Mv > M)   // |v|^2 of padded sources: 0x7f7f7f7f = 3.4e38, their weights underflow to zero
        KMB_CUDA_CHECK(cudaMemsetAsync(F(L.off_vn) + M, 0x7f, sizeof(float) * (L.Mv - M), stream));
    return tc::tensor_prepass_f16(x, y, N, M, D, L.Dp, kid, F(L.off_center), F(L.off_stats), F(L.off_sscale), ws + L.off_uh,
                                  ws + L.off_ul, ws + L.off_vh, ws + L.off_vl, F(L.off_un), F(L.off_vn), stream);
}

bool tensor_use_pair(long long n_tiles, int sms) {
    static const bool pair_enabled = [] {   // tuning knob: KMB_TENSOR_PAIR=0 keeps the single-CTA kernels
        const char* e = getenv("KMB_TENSOR_PAIR");
        return !(e && e[0] == '0');
    }();
    return pair_enabled && n_tiles >= 2 && sms >= 2;
}

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// signal columns per pass of kprod_tensor (E = 3 runs on the EP = 4 instantiation, see launch_ep)
int tensor_e_chunk(int E) { return E >= 4 ? 4 : E; }

// which kernel family tensor_product hands the product to (KIND_NONE: the one-term path has no TF32 P.B kernel)
enum { KIND_TENSOR, KIND_PV, KIND_PV16, KIND_NONE };
int tensor_kind(int D, int E, int kid, int elt) {
    if (elt != tc::ELT_TF32 && tensor_pv16_applicable(D, E, kid)) return KIND_PV16;
    if (tensor_pv_applicable(D, E)) return elt == tc::ELT_F16X1 ? KIND_NONE : KIND_PV;
    return KIND_TENSOR;
}
int kind_unsupported(int D, int E) {
    return set_error(KMB_ERR_UNSUPPORTED, "the one-term FP16 path has no kernel for this shape (D=%d, E=%d: the TF32 P.B family)", D, E);
}

struct TensorPlan {
    bool pair;   // CTA-pair kernel (cta_group::2): FP16 planes, at least two row tiles
    int Dp, e_chunk, n_passes, grid, kblocks, ksteps_last;
    long long n_tiles, nsb;
    tc::WavePlan waves;
    size_t esz;   // bytes per stored operand element
    size_t off_center, off_cpart, off_sscale, off_uh, off_ul, off_vh, off_vl, off_un, off_vn, off_partial, off_counter, total;
};

int plan_tensor(int64_t N, int64_t M, int D, int E, int elt, TensorPlan* pl) {
    const bool f16 = elt != tc::ELT_TF32;
    pl->Dp = f16 ? (D + 15) / 16 * 16 : (D + tc::TK - 1) / tc::TK * tc::TK;
    const int tke = f16 ? 64 : 32;
    pl->kblocks = (pl->Dp + tke - 1) / tke;
    pl->ksteps_last = (pl->Dp - (pl->kblocks - 1) * tke) / (f16 ? 16 : 8);
    pl->esz = f16 ? 2 : 4;
    pl->e_chunk = tensor_e_chunk(E);
    pl->n_passes = (E + pl->e_chunk - 1) / pl->e_chunk;
    pl->n_tiles = (N + tc::TM - 1) / tc::TM;
    pl->nsb = (M + tc::TN - 1) / tc::TN;
    int dev = 0, sms = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    pl->grid = sms;
    pl->pair = f16 && tensor_use_pair(pl->n_tiles, sms);
    if (pl->pair) {
        // the wave plan counts pairs of row tiles and clusters of two CTAs
        pl->grid = sms / 2 * 2;
        tc::plan_waves((pl->n_tiles + 1) / 2, pl->nsb, pl->grid / 2, static_cast<size_t>(tc::TM) * pl->Dp * pl->esz * 4, &pl->waves);
        pl->waves.slots_per_wave *= 2;
        pl->waves.partial_slots *= 2;
    } else {
        tc::plan_waves(pl->n_tiles, pl->nsb, pl->grid, static_cast<size_t>(tc::TM) * pl->Dp * pl->esz * 2, &pl->waves);
    }
    const int PS = tc::MAX_EP + 2;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    if (f16) {   // the points-only head shared with kprod_tensor_pv16 (kmb_product_prepare_f32)
        F16PointsLayout L;
        f16_points_layout(N, M, D, &L);
        pl->off_center = L.off_center; pl->off_cpart = L.off_stats; pl->off_sscale = L.off_sscale;
        pl->off_uh = L.off_uh; pl->off_ul = L.off_ul; pl->off_vh = L.off_vh; pl->off_vl = L.off_vl;
        pl->off_un = L.off_un; pl->off_vn = L.off_vn;
        o = L.end;
    } else {
        pl->off_center = take(sizeof(float) * pl->Dp);
        pl->off_cpart = take(sizeof(float) * tc::CENTER_BLOCKS * D);
        pl->off_sscale = take(sizeof(float) * 2);
        pl->off_uh = take(pl->esz * N * pl->Dp);
        pl->off_ul = take(pl->esz * N * pl->Dp);
        pl->off_vh = take(pl->esz * M * pl->Dp);
        pl->off_vl = take(pl->esz * M * pl->Dp);
        pl->off_un = take(sizeof(float) * N);
        pl->off_vn = take(sizeof(float) * M);
    }
    pl->off_partial = take(sizeof(float) * pl->waves.partial_slots * tc::TM * PS);
    pl->off_counter = take(sizeof(int) * pl->n_tiles);
    pl->total = o;
    return KMB_OK;
}

using KernelFn = void (*)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const tc::Params);

template <int EP, int KID, bool NORM, int ELT>
int launch_one(const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    using C = tc::Cfg<EP, KID, NORM>;
    auto fn = tc::kprod_tensor_kernel<EP, KID, NORM, ELT>;
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), C::SMEM_BYTES)) return rc;
    fn<<<grid, tc::THREADS, C::SMEM_BYTES, stream>>>(maps[0], maps[1], maps[2], maps[3], P);
    KMB_CUDA_CHECK(cudaGetLastError());
    return KMB_OK;
}

template <int EP, int KID, bool NORM, int TERMS>
int launch_pair_one(const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    using C = tc::pair::Cfg2<EP, KID, NORM>;
    auto fn = tc::pair::kprod_tensor_pair_kernel<EP, KID, NORM, TERMS>;
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), C::SMEM_BYTES)) return rc;
    fn<<<grid, tc::THREADS, C::SMEM_BYTES, stream>>>(maps[0], maps[1], maps[2], maps[3], P);
    KMB_CUDA_CHECK(cudaGetLastError());
    return KMB_OK;
}

template <int KID, bool NORM, int TERMS>
int launch_pair_ep(int ep, const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    if (ep == 1) return launch_pair_one<1, KID, NORM, TERMS>(maps, P, grid, stream);
    if (ep == 2) return launch_pair_one<2, KID, NORM, TERMS>(maps, P, grid, stream);
    return launch_pair_one<4, KID, NORM, TERMS>(maps, P, grid, stream);
}

// TERMS = 1 (one-term path): Gaussian and exponential epilogues only (the inverse distance is rejected by the C ABI)
template <int TERMS>
int launch_pair_any(int kid, bool norm, int ep, const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    switch (kid * 2 + (norm ? 1 : 0)) {
        case 0: return launch_pair_ep<KMB_KERNEL_GAUSSIAN, false, TERMS>(ep, maps, P, grid, stream);
        case 1: return launch_pair_ep<KMB_KERNEL_GAUSSIAN, true, TERMS>(ep, maps, P, grid, stream);
        case 2: return launch_pair_ep<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, false, TERMS>(ep, maps, P, grid, stream);
        case 3: return launch_pair_ep<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, true, TERMS>(ep, maps, P, grid, stream);
    }
    if constexpr (TERMS == 1) return set_error(KMB_ERR_UNSUPPORTED, "no one-term kernel for kernel id %d", kid);
    else if (norm) return launch_pair_ep<KMB_KERNEL_INVERSE_DISTANCE, true, TERMS>(ep, maps, P, grid, stream);
    else return launch_pair_ep<KMB_KERNEL_INVERSE_DISTANCE, false, TERMS>(ep, maps, P, grid, stream);
}

template <int KID, bool NORM, int ELT>
int launch_ep(int ep, const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    if (ep == 1) return launch_one<1, KID, NORM, ELT>(maps, P, grid, stream);
    if (ep == 2) return launch_one<2, KID, NORM, ELT>(maps, P, grid, stream);
    return launch_one<4, KID, NORM, ELT>(maps, P, grid, stream);
}

template <int ELT>
int launch_any(int kid, bool norm, int ep, const CUtensorMap* maps, const tc::Params& P, int grid, cudaStream_t stream) {
    switch (kid * 2 + (norm ? 1 : 0)) {
        case 0: return launch_ep<KMB_KERNEL_GAUSSIAN, false, ELT>(ep, maps, P, grid, stream);
        case 1: return launch_ep<KMB_KERNEL_GAUSSIAN, true, ELT>(ep, maps, P, grid, stream);
        case 2: return launch_ep<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, false, ELT>(ep, maps, P, grid, stream);
        case 3: return launch_ep<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, true, ELT>(ep, maps, P, grid, stream);
    }
    if constexpr (ELT == tc::ELT_F16X1) return set_error(KMB_ERR_UNSUPPORTED, "no one-term kernel for kernel id %d", kid);
    else if (norm) return launch_ep<KMB_KERNEL_INVERSE_DISTANCE, true, ELT>(ep, maps, P, grid, stream);
    else return launch_ep<KMB_KERNEL_INVERSE_DISTANCE, false, ELT>(ep, maps, P, grid, stream);
}

}  // namespace

void tensor_plan_waves_debug(long long n_tiles, long long nsb, int grid, size_t row_tile_bytes, long long out[7]) {
    tc::WavePlan wp{};
    tc::plan_waves(n_tiles, nsb, grid, row_tile_bytes, &wp);
    out[0] = wp.R; out[1] = wp.C; out[2] = wp.W; out[3] = wp.R_last; out[4] = wp.C_last; out[5] = wp.slots_per_wave;
    out[6] = wp.partial_slots;
}

void tensor_plan_debug(int64_t N, int D, int E, int kid, int elt, int sms, long long out[4]) {
    const long long n_tiles = (N + tc::TM - 1) / tc::TM;
    const int kind = tensor_kind(D, E, kid, elt);
    int chunk;
    if (kind == KIND_NONE) {
        out[0] = KMB_FAMILY_UNSUPPORTED;
        out[1] = out[2] = -1;
        out[3] = n_tiles;
        return;
    }
    if (kind == KIND_TENSOR) {
        out[0] = (elt != tc::ELT_TF32 && tensor_use_pair(n_tiles, sms)) ? KMB_FAMILY_TENSOR_PAIR : KMB_FAMILY_TENSOR;
        chunk = tensor_e_chunk(E);
    } else if (kind == KIND_PV) {
        out[0] = KMB_FAMILY_PV;
        chunk = tensor_pv_signal_block();
    } else {
        out[0] = tensor_use_pair(n_tiles, sms) ? KMB_FAMILY_PV16_PAIR : KMB_FAMILY_PV16;
        chunk = tensor_pv16_signal_block();
    }
    out[1] = chunk;
    out[2] = (E + chunk - 1) / chunk;
    out[3] = n_tiles;
}

int tensor_pv_plan_query(int64_t N, int64_t M, int D, int E, int kid, int elt, int sms, int smem_optin, long long* out) {
    static_assert(PVQ_FIELDS == KMB_PV_PLAN_FIELDS, "kmb_debug_pv_plan fields");
    for (int i = 0; i < PVQ_FIELDS; ++i) out[i] = -1;
    long long t[4];
    tensor_plan_debug(N, D, E, kid, elt, sms, t);
    out[PVQ_FAMILY] = t[0];
    const int kind = tensor_kind(D, E, kid, elt);
    if (kind == KIND_PV16) return tensor_pv16_plan_debug(N, M, D, E, sms, smem_optin, out);
    if (kind == KIND_PV) return tensor_pv_plan_debug(N, M, D, E, sms, smem_optin, out);
    return KMB_OK;   // an E <= 4 kernel: only the family
}

int tensor_workspace_bytes(int64_t N, int64_t M, int D, int E, int kid, int flags, int elt, size_t* bytes) {
    (void)flags;
    const int kind = tensor_kind(D, E, kid, elt);
    if (kind == KIND_NONE) return kind_unsupported(D, E);
    if (kind == KIND_PV16) return tensor_pv16_workspace_bytes(N, M, D, E, bytes);
    if (kind == KIND_PV) return tensor_pv_workspace_bytes(N, M, D, E, bytes);
    TensorPlan pl{};
    if (int rc = plan_tensor(N, M, D, E, elt, &pl)) return rc;
    *bytes = pl.total;
    return KMB_OK;
}

int tensor_prepare(const float* x, const float* y, int64_t N, int64_t M, int D, int kid, int elt, void* workspace,
                   size_t workspace_bytes, cudaStream_t stream) {
    if (elt == tc::ELT_TF32) return KMB_OK;
    F16PointsLayout L;
    f16_points_layout(N, M, D, &L);
    if (!workspace || workspace_bytes < L.end)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", L.end, workspace_bytes);
    return f16_points_prepass(x, y, N, M, D, kid, L, static_cast<char*>(workspace), stream);
}

int tensor_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E,
                   int kid, int flags, int elt, int64_t row_offset, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1, bool prepared) {
    const int kind = tensor_kind(D, E, kid, elt);
    if (kind == KIND_NONE) return kind_unsupported(D, E);
    if (kind == KIND_PV16)
        return tensor_pv16_product(x, y, b, out, N, M, D, E, kid, flags, elt, workspace, workspace_bytes, stream, ev0, ev1, prepared);
    if (kind == KIND_PV)
        return tensor_pv_product(x, y, b, out, N, M, D, E, kid, flags, row_offset, workspace, workspace_bytes, stream, ev0, ev1);
    TensorPlan pl{};
    if (int rc = plan_tensor(N, M, D, E, elt, &pl)) return rc;
    if (!workspace || workspace_bytes < pl.total)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.total, workspace_bytes);
    if (N >= (1ll << 31) - tc::TM || M >= (1ll << 31) - tc::TN)
        return set_error(KMB_ERR_UNSUPPORTED, "tensor path indexes rows with 32-bit TMA coordinates");
    const bool f16 = elt != tc::ELT_TF32;
    const bool x1 = elt == tc::ELT_F16X1;   // the lo planes are not read: their maps repeat the hi ones
    char* ws = static_cast<char*>(workspace);
    float* center = reinterpret_cast<float*>(ws + pl.off_center);
    float* cpart = reinterpret_cast<float*>(ws + pl.off_cpart);
    float* sscale = reinterpret_cast<float*>(ws + pl.off_sscale);
    void* uh = ws + pl.off_uh;
    void* ul = ws + pl.off_ul;
    void* vh = ws + pl.off_vh;
    void* vl = ws + pl.off_vl;
    float* un = reinterpret_cast<float*>(ws + pl.off_un);
    float* vn = reinterpret_cast<float*>(ws + pl.off_vn);
    float* partial = reinterpret_cast<float*>(ws + pl.off_partial);
    int* counters = reinterpret_cast<int*>(ws + pl.off_counter);
    const bool norm = flags & KMB_FLAG_NORMALIZE_ROWS;
    const bool density = flags & KMB_FLAG_DENSITY;

    KMB_CUDA_CHECK(cudaMemsetAsync(counters, 0, sizeof(int) * pl.n_tiles, stream));
    CUtensorMap maps[4];
    if (f16) {
        if (!prepared) {
            F16PointsLayout L;
            f16_points_layout(N, M, D, &L);
            if (int rc = f16_points_prepass(x, y, N, M, D, kid, L, ws, stream)) return rc;
        }
        if (int rc = tc::make_tensor_map_f16(&maps[0], uh, N, pl.Dp, tc::TM)) return rc;
        if (int rc = tc::make_tensor_map_f16(&maps[1], x1 ? uh : ul, N, pl.Dp, tc::TM)) return rc;
        // the pair kernel's CTAs each load half a source block (128 rows)
        if (int rc = tc::make_tensor_map_f16(&maps[2], vh, M, pl.Dp, pl.pair ? 128 : tc::TN)) return rc;
        if (int rc = tc::make_tensor_map_f16(&maps[3], x1 ? vh : vl, M, pl.Dp, pl.pair ? 128 : tc::TN)) return rc;
    } else {
        if (int rc = tc::tensor_prepass(x, y, N, M, D, pl.Dp, kid, center, cpart, static_cast<float*>(uh), static_cast<float*>(ul),
                                        static_cast<float*>(vh), static_cast<float*>(vl), un, vn, stream))
            return rc;
        if (int rc = tc::make_tensor_map(&maps[0], static_cast<float*>(uh), N, pl.Dp, tc::TM)) return rc;
        if (int rc = tc::make_tensor_map(&maps[1], static_cast<float*>(ul), N, pl.Dp, tc::TM)) return rc;
        if (int rc = tc::make_tensor_map(&maps[2], static_cast<float*>(vh), M, pl.Dp, tc::TN)) return rc;
        if (int rc = tc::make_tensor_map(&maps[3], static_cast<float*>(vl), M, pl.Dp, tc::TN)) return rc;
    }

    const int grid = pl.grid;
    for (int pass = 0; pass < pl.n_passes; ++pass) {
        tc::Params P;
        P.un = un;
        P.vn = vn;
        P.b = density ? nullptr : b;
        P.out = out;
        P.partial = partial;
        P.tile_counter = counters;
        P.sscale = sscale;
        P.N = N;
        P.M = M;
        P.row_offset = row_offset;
        P.E = E;
        P.e0 = pass * pl.e_chunk;
        P.n_tiles = static_cast<int>(pl.n_tiles);
        P.nsb = static_cast<int>(pl.nsb);
        P.kblocks = pl.kblocks;
        P.ksteps_last = pl.ksteps_last;
        P.R = pl.waves.R;
        P.C = pl.waves.C;
        P.W = pl.waves.W;
        P.R_last = pl.waves.R_last;
        P.C_last = pl.waves.C_last;
        P.slots_per_wave = pl.waves.slots_per_wave;
        if (ev0 && pass == pl.n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev0, stream));
        const int ekid = tc::epilogue_kid(kid);
        int rc;
        if (pl.pair) rc = x1 ? launch_pair_any<1>(ekid, norm, pl.e_chunk, maps, P, grid, stream)
                             : launch_pair_any<3>(ekid, norm, pl.e_chunk, maps, P, grid, stream);
        else if (x1) rc = launch_any<tc::ELT_F16X1>(ekid, norm, pl.e_chunk, maps, P, grid, stream);
        else if (f16) rc = launch_any<tc::ELT_F16>(ekid, norm, pl.e_chunk, maps, P, grid, stream);
        else rc = launch_any<tc::ELT_TF32>(ekid, norm, pl.e_chunk, maps, P, grid, stream);
        if (rc) return rc;
        if (ev1 && pass == pl.n_passes - 1) KMB_CUDA_CHECK(cudaEventRecord(ev1, stream));
        count_launch();
    }
    return KMB_OK;
}

}  // namespace kmb
