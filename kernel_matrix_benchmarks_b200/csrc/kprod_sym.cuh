// kprod_sym: a_i = sum_j k(y_i, y_j) b_j when targets and sources are the same points (the reference's
// `same_points` flag, base.py:56-79; always the case in the kernel solve, bruteforce.py:193-199).
// Every kernel of bruteforce.py:18-22 is a function of |x - y|, so K is symmetric and each kernel value is
// evaluated ONCE and used twice:
//     a_i += k_ij b_j   (row sum, as in kprod_direct)      a_j += k_ij b_i   (column sum)
// which halves the MUFU work -- the binding pipe of kprod_direct at D = 3 (SURVEY.md section 8d).
//
// Shape of the computation
//   * FORM 1 (Gaussian, data small enough -- DirectStats::use_product): product form of kprod_direct.cuh,
//     k_ij = 2^(-|u_i|^2) e_ij 2^(-|u_j|^2), e_ij = 2^(2 u_i.u_j), with w_j = b_j 2^(-|u_j|^2) riding in the
//     packed records.  Row sums R_i = sum_j e_ij w_j and column sums C_j = sum_i e_ij w_i share e_ij;
//     out_i = 2^(-|u_i|^2) (R_i + C_i).
//     FORM 0 (any kernel): difference form, k_ij = f(|v_i - v_j|^2), w_j = b_j, out_i = R_i + C_i.
//   * The N x N pair matrix is cut into units of (TILE_ROWS target rows) x (SB sources).  Only units on or above
//     the block diagonal are evaluated: the TB = TILE_ROWS / SB units that intersect a tile's own rows
//     ("diagonal" units) are evaluated in full with row sums only, the units to their right feed both the row
//     sums of the tile and the column sums of the block.
//   * Unit order: the source blocks are cut into STRIPS of Wb blocks; the list runs strip by strip, inside a
//     strip tile by tile, inside a (strip, tile) SEGMENT block by block.  The list is cut stream-K style into
//     equal contiguous ranges -- first across `n_parts` GPUs, then across the resident CTAs.  With
//     Wb ~ nsb / sqrt(2 G) a CTA's range is a roughly square patch of the pair matrix (Wb blocks wide, a few
//     tiles tall), which minimises what it has to hand over: one row-sum vector per segment and ONE column-sum
//     slab per (CTA, strip), Wb * SB floats.  The slab lives in global memory but is private to the CTA:
//     zero-filled when the CTA enters the strip, then read-modify-written once per unit by the same thread
//     (plain program order, no atomics), so it stays in L2.  Workspace is O(N sqrt(G)) floats (77 MB at
//     N = 10^6, 0.3 GB at 4 10^6) instead of one column vector per tile (O(N^2 / TILE_ROWS): 0.98 GB / 15.6 GB).
//   * Column sums of a unit: each thread reduces its R rows, each warp reduces its 32 lanes with a transposing
//     shuffle butterfly (16 SHFL per 16 sources instead of 80), the 16 warps meet in shared memory.
//   * sym_combine_kernel adds, in a fixed order, the row pieces of a row's tile (one per strip, plus the pieces of
//     segments cut by a CTA boundary) and the column pieces of its strip (one per CTA that worked in the strip):
//     bitwise deterministic; with n_parts > 1 the caller sums the parts' outputs (one all-reduce of N floats).
#pragma once
#include "kprod_direct.cuh"

namespace kmb {

constexpr int SYM_MAX_STRIPS = 96;

// Geometry of the strip-ordered unit list; built on the host (sym_build_geom), passed by value.
struct SymGeom {
    long long nsb;                                 // source blocks
    int n_tiles, Wb, Wt, n_strips;                 // strip width in blocks / in tiles (Wb = TB * Wt)
    long long strip_prefix[SYM_MAX_STRIPS + 1];    // units before strip s
    int seg_prefix[SYM_MAX_STRIPS + 1];            // (strip, tile) segments before strip s
};

struct SymSeg {     // one (strip, tile) segment: units [begin, begin + len), source blocks jb0 .. jb0 + len - 1
    int strip, tile, len;
    long long begin, jb0;
};

struct SymParams {
    const DirectStats* stats;
    const float4* rec;     // packed records (pack_sources_kernel), nsb * SB of them: sources AND targets
    float* rowseg;         // row sums of the segments finished by one CTA, slot = seg_prefix[strip] + tile - seg_base
    float* rowpart;        // grid * 2 * TILE_ROWS: row sums of each CTA's first / last (cut) segment
    float* colpart;        // (grid + strips of this part) slabs of piece_floats: column sums per (CTA, strip)
    float* out;            // N
    long long N, M;
    long long unit_begin, unit_end;   // this launch's share of the unit list
    long long piece_floats;           // Wb * SB
    int grid, seg_base, strip_base;   // first segment slot / first strip of this part
    SymGeom g;
};

template <int TB>
__host__ __device__ __forceinline__ long long sym_tri(long long k, long long w) {   // units of the first k diagonal tiles of a strip
    return k * w - (TB * k * (k - 1)) / 2;
}
__host__ __device__ __forceinline__ long long sym_strip_width(const SymGeom& g, int s) {
    const long long e = static_cast<long long>(s + 1) * g.Wb;
    return (e < g.nsb ? e : g.nsb) - static_cast<long long>(s) * g.Wb;
}
// the segment of tile `tile` in strip s (tile < tiles of the strip)
template <int TB>
__host__ __device__ __forceinline__ SymSeg sym_seg(const SymGeom& g, int s, int tile) {
    const long long w = sym_strip_width(g, s), F = static_cast<long long>(s) * g.Wt;
    SymSeg r;
    r.strip = s;
    r.tile = tile;
    if (tile < F) {
        r.begin = g.strip_prefix[s] + tile * w;
        r.len = static_cast<int>(w);
        r.jb0 = static_cast<long long>(s) * g.Wb;
    } else {
        const long long k = tile - F;
        r.begin = g.strip_prefix[s] + F * w + sym_tri<TB>(k, w);
        r.len = static_cast<int>(w - TB * k);
        r.jb0 = static_cast<long long>(TB) * tile;
    }
    return r;
}
// the segment that holds unit u
template <int TB>
__host__ __device__ __forceinline__ SymSeg sym_seg_of(const SymGeom& g, long long u) {
    int lo = 0, hi = g.n_strips - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (g.strip_prefix[mid] <= u) lo = mid; else hi = mid - 1;
    }
    const int s = lo;
    const long long w = sym_strip_width(g, s), F = static_cast<long long>(s) * g.Wt;
    long long v = u - g.strip_prefix[s];
    if (v < F * w) return sym_seg<TB>(g, s, static_cast<int>(v / w));
    v -= F * w;
    const long long kt = (w + TB - 1) / TB;
    const double h = static_cast<double>(w) + 0.5 * TB;
    double disc = h * h - 2.0 * TB * static_cast<double>(v);
    if (disc < 0.0) disc = 0.0;
    long long k = static_cast<long long>((h - sqrt(disc)) / TB);
    if (k < 0) k = 0;
    if (k > kt - 1) k = kt - 1;
    while (k + 1 < kt && sym_tri<TB>(k + 1, w) <= v) ++k;
    while (k > 0 && sym_tri<TB>(k, w) > v) --k;
    return sym_seg<TB>(g, s, static_cast<int>(F + k));
}

// Host: strip width in tiles that `total_ctas` CTAs over all parts ask for (Wb ~ nsb / sqrt(2 G)), before the
// strip-count cap.
template <int TB>
inline long long sym_cta_strip_tiles(long long nsb, long long total_ctas) {
    double ideal = static_cast<double>(nsb) / sqrt(2.0 * static_cast<double>(total_ctas < 1 ? 1 : total_ctas));
    long long Wt = static_cast<long long>(ceil(ideal / TB));
    return Wt < 1 ? 1 : Wt;
}

// Host: strip width for `total_ctas` CTAs over all parts, prefix tables.
template <int TB>
inline void sym_build_geom(long long n_tiles, long long nsb, long long total_ctas, SymGeom* g) {
    long long Wt = sym_cta_strip_tiles<TB>(nsb, total_ctas);
    const long long min_wt = (n_tiles + SYM_MAX_STRIPS - 1) / SYM_MAX_STRIPS;
    if (Wt < min_wt) Wt = min_wt;
    g->nsb = nsb;
    g->n_tiles = static_cast<int>(n_tiles);
    g->Wt = static_cast<int>(Wt);
    g->Wb = static_cast<int>(Wt * TB);
    g->n_strips = static_cast<int>((nsb + g->Wb - 1) / g->Wb);
    g->strip_prefix[0] = 0;
    g->seg_prefix[0] = 0;
    for (int s = 0; s < g->n_strips; ++s) {
        const long long w = sym_strip_width(*g, s), F = static_cast<long long>(s) * Wt, kt = (w + TB - 1) / TB;
        g->strip_prefix[s + 1] = g->strip_prefix[s] + F * w + sym_tri<TB>(kt, w);
        g->seg_prefix[s + 1] = g->seg_prefix[s] + static_cast<int>(F + kt);
    }
    for (int s = g->n_strips + 1; s <= SYM_MAX_STRIPS; ++s) {
        g->strip_prefix[s] = g->strip_prefix[g->n_strips];
        g->seg_prefix[s] = g->seg_prefix[g->n_strips];
    }
}

// KID_/FORM_: kernel and evaluation form (FORM_ 1 = Gaussian product form); POLY_: every POLY_-th exponential of the
// product form on the FMA pipe (see DirectCfg); CH_: sources per shuffle butterfly
template <int DP_, int KID_ = KMB_KERNEL_GAUSSIAN, int FORM_ = 1, int POLY_ = 0, int MINB_ = 1, int CH_ = 16, int CONSUMERS_ = 512,
          int R_ = 8, int STAGES_ = 4>
struct SymCfg {
    static constexpr int DP = DP_, KID = KID_, FORM = FORM_, POLY = POLY_, MINB = MINB_, CH = CH_;
    static_assert(FORM == 0 || KID == KMB_KERNEL_GAUSSIAN, "product form is Gaussian-only");
    static_assert(POLY == 0 || FORM == 1, "the polynomial exp2 needs the bounded exponents of the product form");
    static constexpr int R = R_, RP = R_ / 2, CONSUMERS = CONSUMERS_, THREADS = CONSUMERS + 32, WARPS = CONSUMERS / 32;
    static_assert(R % 2 == 0 && (CH == 8 || CH == 16), "rows are processed as packed pairs; butterflies of 8 or 16 sources");
    static constexpr int TILE_ROWS = CONSUMERS * R;
    static constexpr int STAGES = STAGES_;
    static constexpr int PAIRS = DP + 1, RECV = (PAIRS + 1) / 2;
    static_assert(RECV == 2, "32-byte records (D <= 3, E = 1)");
    static constexpr int SB = 512;
    static_assert(SB % CONSUMERS == 0 && TILE_ROWS % SB == 0, "whole sources per thread when the warps' column sums are combined");
    static constexpr int TB = TILE_ROWS / SB;
    static constexpr int STAGE_BYTES = SB * RECV * 16;
    static constexpr int COLBUF_BYTES = WARPS * SB * 4;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + COLBUF_BYTES + 2 * STAGES * 8 + 16;
};

// first coordinate of a padding target row (difference form): far from the data AND from the padding records
// (+1e18 in pack_sources_kernel), so its kernel values are exactly zero (exponentials) or finite (inverse
// distance, where they meet a zero signal entry)
constexpr float kSymPadCoord = -1.0e18f;

template <class C>
__global__ void __launch_bounds__(C::THREADS, C::MINB)
kprod_sym_kernel(const SymParams P) {
    constexpr int DP = C::DP, RP = C::RP, R = C::R, SB = C::SB, STAGES = C::STAGES, RECV = C::RECV, TB = C::TB, CH = C::CH;
    constexpr int KID = C::KID, FORM = C::FORM;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4* stage_base = reinterpret_cast<float4*>(smem_raw);
    float* colbuf = reinterpret_cast<float*>(smem_raw + STAGES * C::STAGE_BYTES);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + STAGES * C::STAGE_BYTES + C::COLBUF_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;

    // both forms of a Gaussian product are enqueued; the data decide (on the device) which one runs
    if ((P.stats->use_product != 0) != (FORM == 1)) return;

    const int tid = threadIdx.x;
    const int G = gridDim.x;
    const long long Ur = P.unit_end - P.unit_begin;
    const long long u0 = P.unit_begin + Ur * blockIdx.x / G;
    const long long u1 = P.unit_begin + Ur * (blockIdx.x + 1) / G;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], C::WARPS);
        }
        fence_mbar_init();
    }
    __syncthreads();

    if (tid >= C::CONSUMERS) {
        // ------------------------------ producer warp ------------------------------
        if (tid == C::CONSUMERS) {
            uint32_t it = 0;
            long long u = u0;
            while (u < u1) {
                const SymSeg sg = sym_seg_of<TB>(P.g, u);
                long long jb = sg.jb0 + (u - sg.begin);
                const long long end = min(sg.begin + sg.len, u1);
                for (; u < end; ++u, ++jb, ++it) {
                    const int stage = it % STAGES;
                    mbar_wait_backoff(&empty_bar[stage], ((it / STAGES) & 1) ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], C::STAGE_BYTES);
                    tma_bulk_g2s(stage_base + stage * (SB * RECV), P.rec + jb * (SB * RECV), C::STAGE_BYTES, &full_bar[stage]);
                }
            }
        }
        return;
    }

    // -------------------------------- consumers --------------------------------
    const int lane = tid & 31, warp = tid >> 5;
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4, h2 = lane & 2;
    // the source of a chunk this lane ends up holding, and whether it is the lane that stores it
    const int jl = CH == 16 ? (h16 ? 8 : 0) + (h8 ? 4 : 0) + (h4 ? 2 : 0) + (h2 ? 1 : 0) : (h16 ? 4 : 0) + (h8 ? 2 : 0) + (h4 ? 1 : 0);
    float* my_col = colbuf + warp * SB + jl;
    const bool col_writer = CH == 16 ? (lane & 1) == 0 : (lane & 3) == 0;

    uint32_t it = 0;
    long long u = u0;
    int cur_strip = -1;
    float* piece = nullptr;   // this CTA's column-sum slab of the strip it is in
    long long strip_jb0 = 0;
    while (u < u1) {
        const SymSeg sg = sym_seg_of<TB>(P.g, u);
        const int tile = sg.tile;
        const long long jb0 = sg.jb0 + (u - sg.begin);
        const int cnt = static_cast<int>(min(sg.begin + sg.len, u1) - u);
        const long long row_base = static_cast<long long>(tile) * C::TILE_ROWS + tid;

        if (sg.strip != cur_strip) {
            // entering a strip: zero this CTA's slab.  Thread t owns column t of every block (zero-fill and every
            // later read-modify-write of an address come from the same thread: program order is all that is needed)
            cur_strip = sg.strip;
            strip_jb0 = static_cast<long long>(cur_strip) * P.g.Wb;
            piece = P.colpart + static_cast<size_t>(blockIdx.x + cur_strip - P.strip_base) * P.piece_floats;
            const int w = static_cast<int>(sym_strip_width(P.g, cur_strip));
            for (int k = 0; k < w; ++k)
#pragma unroll
                for (int sidx = tid; sidx < SB; sidx += C::CONSUMERS) __stcg(piece + static_cast<size_t>(k) * SB + sidx, 0.f);
        }

        // this thread's rows, straight from the packed records: the row operand of the exponent (2u, product form) or of
        // the difference (-v), and w = what the row contributes to the column sums (its signal entry)
        float2 xr[DP][RP], w[RP];
        [[maybe_unused]] long long grow[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const long long row = row_base + static_cast<long long>(r) * C::CONSUMERS;
            grow[r] = row;
            float4 q0 = make_float4(FORM == 1 ? 0.f : kSymPadCoord, 0.f, 0.f, 0.f), q1 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < P.N) {
                q0 = __ldg(P.rec + row * RECV);
                q1 = __ldg(P.rec + row * RECV + 1);
            }
            const float c[4] = {q0.x, q0.z, q1.x, q1.z};   // pairs are duplicated: [v0 v0 v1 v1 | v2 v2 w w]
#pragma unroll
            for (int d = 0; d < DP; ++d) {
                const float v = FORM == 1 ? 2.f * c[d] : -c[d];
                if (r & 1) xr[d][r >> 1].y = v; else xr[d][r >> 1].x = v;
            }
            if (r & 1) w[r >> 1].y = c[DP]; else w[r >> 1].x = c[DP];
        }
        float2 acc[RP], tot[RP];
#pragma unroll
        for (int p = 0; p < RP; ++p) acc[p] = tot[p] = make_float2(0.f, 0.f);

        // kernel values of one source record for the thread's row pair p
        auto eval = [&](const float2* pr, int p, bool poly) -> float2 {
            float2 s;
            if constexpr (FORM == 1) {
#pragma unroll
                for (int d = 0; d < DP; ++d) s = (d == 0) ? mul2(xr[d][p], pr[d]) : fma2(xr[d][p], pr[d], s);
                return poly ? ex2_poly2(s) : make_float2(ex2_approx(s.x), ex2_approx(s.y));
            } else {
#pragma unroll
                for (int d = 0; d < DP; ++d) {
                    const float2 diff = add2(xr[d][p], pr[d]);
                    s = (d == 0) ? mul2(diff, diff) : fma2(diff, diff, s);
                }
                return make_float2(kernel_value<KID>(s.x), kernel_value<KID>(s.y));
            }
        };

        for (int k = 0; k < cnt; ++k, ++it) {
            const int stage = it % STAGES;
            mbar_wait(&full_bar[stage], (it / STAGES) & 1);
            const float4* rec = stage_base + stage * (SB * RECV);
            const long long jb = jb0 + k;
            const bool off_diagonal = jb >= static_cast<long long>(TB) * (tile + 1);

            if (!off_diagonal) {
                // sources are this tile's own rows: every (i, j) of the block is evaluated, row sums only
                [[maybe_unused]] const long long j_base = jb * SB;
#pragma unroll(CH)
                for (int j = 0; j < SB; ++j) {
                    const float4 v0 = rec[j * RECV], v1 = rec[j * RECV + 1];
                    const float2 pr[4] = {make_float2(v0.x, v0.y), make_float2(v0.z, v0.w), make_float2(v1.x, v1.y), make_float2(v1.z, v1.w)};
#pragma unroll
                    for (int p = 0; p < RP; ++p) {
                        const bool poly = C::POLY > 0 && (RP * CH) % C::POLY == 0 && ((j % CH) * RP + p) % C::POLY == C::POLY - 1;
                        float2 kv = eval(pr, p, poly);
                        if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE) {
                            // the reference's zeroing rule (bruteforce.py:12-14) with N == M: the diagonal; padding
                            // sources carry b == 0 and a finite kernel value
                            if (j_base + j == grow[2 * p]) kv.x = 0.f;
                            if (j_base + j == grow[2 * p + 1]) kv.y = 0.f;
                        }
                        acc[p] = fma2(kv, pr[DP], acc[p]);
                    }
                }
            } else {
#pragma unroll 1
                for (int j = 0; j < SB; j += CH) {
                    float t[CH];
#pragma unroll
                    for (int c = 0; c < CH; ++c) {
                        const float4 v0 = rec[(j + c) * RECV], v1 = rec[(j + c) * RECV + 1];
                        const float2 pr[4] = {make_float2(v0.x, v0.y), make_float2(v0.z, v0.w), make_float2(v1.x, v1.y), make_float2(v1.z, v1.w)};
                        float2 kv[RP];
#pragma unroll
                        for (int p = 0; p < RP; ++p) {
                            const bool poly = C::POLY > 0 && (RP * CH) % C::POLY == 0 && (c * RP + p) % C::POLY == C::POLY - 1;
                            kv[p] = eval(pr, p, poly);
                            acc[p] = fma2(kv[p], pr[DP], acc[p]);
                        }
                        // what this thread's R rows add to column j + c
                        float2 tt = mul2(kv[0], w[0]);
#pragma unroll
                        for (int p = 1; p < RP; ++p) tt = fma2(kv[p], w[p], tt);
                        t[c] = tt.x + tt.y;
                    }
                    // transposing butterfly: each xor step halves the columns a lane carries, until one is left
                    float cs;
                    if constexpr (CH == 16) {
                        float s8[8], s4[4], s2[2];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float send = h16 ? t[q] : t[q + 8], keep = h16 ? t[q + 8] : t[q];
                            s8[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float send = h8 ? s8[q] : s8[q + 4], keep = h8 ? s8[q + 4] : s8[q];
                            s4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                        }
#pragma unroll
                        for (int q = 0; q < 2; ++q) {
                            const float send = h4 ? s4[q] : s4[q + 2], keep = h4 ? s4[q + 2] : s4[q];
                            s2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                        }
                        const float send = h2 ? s2[0] : s2[1], keep = h2 ? s2[1] : s2[0];
                        cs = keep + __shfl_xor_sync(0xffffffffu, send, 2);
                        cs += __shfl_xor_sync(0xffffffffu, cs, 1);
                    } else {
                        float s4[4], s2[2];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float send = h16 ? t[q] : t[q + 4], keep = h16 ? t[q + 4] : t[q];
                            s4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                        }
#pragma unroll
                        for (int q = 0; q < 2; ++q) {
                            const float send = h8 ? s4[q] : s4[q + 2], keep = h8 ? s4[q + 2] : s4[q];
                            s2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                        }
                        const float send = h4 ? s2[0] : s2[1], keep = h4 ? s2[1] : s2[0];
                        cs = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                        cs += __shfl_xor_sync(0xffffffffu, cs, 2);
                        cs += __shfl_xor_sync(0xffffffffu, cs, 1);
                    }
                    if (col_writer) my_col[j] = cs;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[stage]);
            // two-level summation of the row sums (see kprod_direct.cuh)
#pragma unroll
            for (int p = 0; p < RP; ++p) {
                tot[p] = add2(tot[p], acc[p]);
                acc[p] = make_float2(0.f, 0.f);
            }
            if (off_diagonal) {
                // the 16 warps' column sums of this unit -> one value per source, added to the CTA's slab (L2)
                float* dst = piece + static_cast<size_t>(jb - strip_jb0) * SB;
                float old[SB / C::CONSUMERS];
#pragma unroll
                for (int q = 0; q < SB / C::CONSUMERS; ++q) old[q] = __ldcg(dst + tid + q * C::CONSUMERS);
                named_bar_sync(1, C::CONSUMERS);
#pragma unroll
                for (int q = 0; q < SB / C::CONSUMERS; ++q) {
                    const int sidx = tid + q * C::CONSUMERS;
                    float cs = 0.f;
#pragma unroll
                    for (int wv = 0; wv < C::WARPS; ++wv) cs += colbuf[wv * SB + sidx];
                    __stcg(dst + sidx, old[q] + cs);
                }
                named_bar_sync(1, C::CONSUMERS);
            }
        }

        // ---------------------------- row sums of this segment ----------------------------
        const bool complete = (u == sg.begin) && (cnt == sg.len);
        float* dst = complete ? P.rowseg + static_cast<size_t>(P.g.seg_prefix[sg.strip] + tile - P.seg_base) * C::TILE_ROWS
                              : P.rowpart + (static_cast<size_t>(blockIdx.x) * 2 + (u == u0 ? 0 : 1)) * C::TILE_ROWS;
        // (streaming / evict-first stores here did not lower the DRAM traffic: 229 MB per launch against 220 MB, measured)
#pragma unroll
        for (int r = 0; r < R; ++r) dst[tid + r * C::CONSUMERS] = (r & 1) ? tot[r >> 1].y : tot[r >> 1].x;
        u += cnt;
    }
}

// out_i = scale_i * (row pieces + column pieces of this part), fixed summation order.
template <class C>
__global__ void __launch_bounds__(256)
sym_combine_kernel(const SymParams P) {
    constexpr int TB = C::TB, SB = C::SB, RECV = C::RECV, DP = C::DP;
    if ((P.stats->use_product != 0) != (C::FORM == 1)) return;
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= P.N) return;
    const int G = P.grid;
    const long long ub = P.unit_begin, ue = P.unit_end, Ur = ue - ub;
    const int tile = static_cast<int>(i / C::TILE_ROWS);
    const int lr = static_cast<int>(i - static_cast<long long>(tile) * C::TILE_ROWS);

    // row pieces: the segments (s, tile) of every strip at or right of the tile's diagonal
    float rs = 0.f;
    for (int s = (TB * tile) / P.g.Wb; s < P.g.n_strips && Ur > 0; ++s) {
        const SymSeg sg = sym_seg<TB>(P.g, s, tile);
        const long long t_begin = sg.begin, t_end = sg.begin + sg.len;
        const long long a = max(t_begin, ub), b = min(t_end, ue);
        if (a >= b) continue;
        const int c_first = static_cast<int>(((a - ub + 1) * G - 1) / Ur);
        const int c_last = static_cast<int>(((b - ub) * G - 1) / Ur);
        for (int c = c_first; c <= c_last; ++c) {
            const long long c0 = ub + Ur * c / G, c1 = ub + Ur * (c + 1) / G;
            const long long s0 = max(c0, t_begin), s1 = min(c1, t_end);
            if (s0 >= s1) continue;
            if (s0 == t_begin && s1 == t_end) rs += __ldcg(P.rowseg + static_cast<size_t>(P.g.seg_prefix[s] + tile - P.seg_base) * C::TILE_ROWS + lr);
            else rs += __ldcg(P.rowpart + (static_cast<size_t>(c) * 2 + (s0 == c0 ? 0 : 1)) * C::TILE_ROWS + lr);
        }
    }
    // column pieces: one slab per CTA whose range meets the strip of source i
    float cs = 0.f;
    {
        const long long jb = i / SB;
        const int s = static_cast<int>(jb / P.g.Wb);
        const long long a = max(P.g.strip_prefix[s], ub), b = min(P.g.strip_prefix[s + 1], ue);
        if (a < b) {
            const int c_first = static_cast<int>(((a - ub + 1) * G - 1) / Ur);
            const int c_last = static_cast<int>(((b - ub) * G - 1) / Ur);
            const size_t off = static_cast<size_t>(jb - static_cast<long long>(s) * P.g.Wb) * SB + static_cast<size_t>(i % SB);
            for (int c = c_first; c <= c_last; ++c) {
                const long long c0 = ub + Ur * c / G, c1 = ub + Ur * (c + 1) / G;
                if (max(c0, a) >= min(c1, b)) continue;
                cs += __ldcg(P.colpart + static_cast<size_t>(c + s - P.strip_base) * P.piece_floats + off);
            }
        }
    }
    float scale = 1.f;
    if constexpr (C::FORM == 1) {
        const float4 q0 = __ldg(P.rec + i * RECV), q1 = __ldg(P.rec + i * RECV + 1);
        const float c[4] = {q0.x, q0.z, q1.x, q1.z};
        float n2 = 0.f;
#pragma unroll
        for (int d = 0; d < DP; ++d) n2 = fmaf(c[d], c[d], n2);
        scale = exp2f(-n2);
    }
    P.out[i] = scale * (rs + cs);
}

}  // namespace kmb
