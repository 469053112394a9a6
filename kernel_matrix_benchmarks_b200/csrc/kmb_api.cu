// C ABI of libkmb_b200.so (see include/kmb_b200.h): argument checking, path selection,
// workspace carving and kernel launches.  No allocation, no synchronisation.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <mutex>
#include <vector>

#include "kprod_direct.cuh"
#include "kprod_sym.cuh"
#include "kprod_tensor.cuh"

namespace kmb {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;
// optional CUDA-event bracket around the dominant (main) kernel of the last product call
static thread_local bool g_profile = false;
static thread_local cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
static thread_local bool g_ev_valid = false;

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
void count_launch(int n) { g_launches += n; }
int launch_count() { return g_launches; }
void set_launch_count(int n) { g_launches = n; }

#define KMB_DECLARE_TABLE(NAME)      \
    extern const DirectEntry NAME[]; \
    extern const int NAME##_count;
KMB_DECLARE_TABLE(kDirect_gauss_n0)
KMB_DECLARE_TABLE(kDirect_gauss_n1)
KMB_DECLARE_TABLE(kDirect_absexp_n0)
KMB_DECLARE_TABLE(kDirect_absexp_n1)
KMB_DECLARE_TABLE(kDirect_invdist_n0)
KMB_DECLARE_TABLE(kDirect_invdist_n1)
KMB_DECLARE_TABLE(kDirect_gaussprod_n0)
KMB_DECLARE_TABLE(kDirect_gaussprod_n1)

// kprod_f64.cu
int product_f64(const double* x, const double* y, const double* b, double* out, int64_t N, int64_t M, int D, int E,
                int kernel_id, int flags, int64_t row_offset, cudaStream_t stream);
int kernel_block_f64(const double* x, const double* y, double* out, int64_t n, int64_t m, int D, int kernel_id, cudaStream_t stream);
// kprod_sym.cu
bool sym_supported(int D);
int sym_tile_rows();
int sym_block_sources();
int sym_grid(int sms, int* grid);
void sym_geometry(long long n_tiles, long long nsb, long long total_ctas, SymGeom* g);
long long sym_cta_strip_width(long long nsb, long long total_ctas);
SymSeg sym_segment_of(const SymGeom& g, long long u);
int sym_launch(int D, int kernel_id, int form, const SymParams& P, cudaStream_t stream);

// the direct tables in the order above (kmb_debug_direct_entry numbers them so)
struct DirectTable { const DirectEntry* tab; const int* count; };
static const DirectTable kDirectTables[8] = {
    {kDirect_gauss_n0, &kDirect_gauss_n0_count},       {kDirect_gauss_n1, &kDirect_gauss_n1_count},
    {kDirect_absexp_n0, &kDirect_absexp_n0_count},     {kDirect_absexp_n1, &kDirect_absexp_n1_count},
    {kDirect_invdist_n0, &kDirect_invdist_n0_count},   {kDirect_invdist_n1, &kDirect_invdist_n1_count},
    {kDirect_gaussprod_n0, &kDirect_gaussprod_n0_count}, {kDirect_gaussprod_n1, &kDirect_gaussprod_n1_count}};

static const DirectEntry* find_direct(int D, int e_chunk, int kid, bool norm, int form) {
    if (form == 1 && kid != KMB_KERNEL_GAUSSIAN) return nullptr;
    const DirectTable& t = kDirectTables[form == 1 ? 6 + norm : kid * 2 + norm];
    const DirectEntry* best = nullptr;
    for (int i = 0; i < *t.count; ++i) {
        const DirectEntry& e = t.tab[i];
        if (e.DP < D || e.EP < e_chunk) continue;
        if (!best || e.DP < best->DP || (e.DP == best->DP && e.EP < best->EP)) best = &e;
    }
    return best;
}

// The direct kernels of a product: signal columns per pass and the entry of each evaluation form (D <= 16).
struct DirectChoice {
    const DirectEntry* ent[2];   // [0] difference form (nullptr: no kernel), [1] Gaussian product form (optional)
    int e_chunk, n_passes;
};
static void choose_direct(int D, int E, int kid, bool norm, int path, DirectChoice* c) {
    // signal columns per pass: every pass re-evaluates the kernel (~8 FMA-pipe slots' worth per pair, MUFU included) and
    // adds one FMA per column; pick the width that minimises passes x (8 + width)
    static const int max_chunk = [] {   // tuning knob: KMB_DIRECT_MAX_EP=4 restores one pass per 4 columns
        const char* e = getenv("KMB_DIRECT_MAX_EP");
        const int v = e ? atoi(e) : 16;
        return v < 1 ? 1 : v > 16 ? 16 : v;
    }();
    c->e_chunk = 1;
    for (int w = 1, best = 0; w <= max_chunk; w *= 2) {
        const int cost = ((E + w - 1) / w) * (8 + w);
        if (best == 0 || cost < best) { best = cost; c->e_chunk = w; }
    }
    c->n_passes = (E + c->e_chunk - 1) / c->e_chunk;
    c->ent[0] = find_direct(D, c->e_chunk, kid, norm, 0);
    c->ent[1] = (kid == KMB_KERNEL_GAUSSIAN && path != KMB_PATH_DIRECT_DIFF) ? find_direct(D, c->e_chunk, kid, norm, 1) : nullptr;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct FormPlan {   // one evaluation form's kernel and geometry
    const DirectEntry* ent = nullptr;
    long long n_tiles = 0, nsb = 0, M_pad = 0;
};
struct DirectPlan {
    FormPlan form[2];   // [0] difference form (always), [1] Gaussian product form (optional)
    int e_chunk, n_passes;
    int grid_max;
    size_t stats_bytes, rec_bytes, partial_bytes, counter_bytes, total_bytes;
};

// ---- per-(function, device) launch state (declared in kmb_common.cuh) ---------------------------
namespace {
struct FuncState { const void* fn; int dev, smem, threads, per_sm; };
std::mutex g_func_mutex;
std::vector<FuncState> g_func_state;
int g_sm_count[64];   // 0 = not asked yet

FuncState* func_state(const void* fn, int dev) {   // g_func_mutex held
    for (FuncState& f : g_func_state)
        if (f.fn == fn && f.dev == dev) return &f;
    g_func_state.push_back(FuncState{fn, dev, 0, 0, 0});
    return &g_func_state.back();
}
}  // namespace

int ensure_dyn_smem(const void* fn, int smem_bytes) {
    int dev = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_func_mutex);
    FuncState* f = func_state(fn, dev);
    if (f->smem < smem_bytes) {
        KMB_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        f->smem = smem_bytes;
        f->per_sm = 0;
    }
    return KMB_OK;
}

int resident_ctas(const void* fn, int threads, int smem_bytes, int* per_sm) {
    if (int rc = ensure_dyn_smem(fn, smem_bytes)) return rc;
    int dev = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_func_mutex);
    FuncState* f = func_state(fn, dev);
    if (f->per_sm == 0 || f->threads != threads) {
        int n = 0;
        KMB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fn, threads, smem_bytes));
        if (n < 1) return set_error(KMB_ERR_CUDA, "kernel does not fit on an SM (%d threads, smem %d B)", threads, smem_bytes);
        f->threads = threads;
        f->per_sm = n;
    }
    *per_sm = f->per_sm;
    return KMB_OK;
}

int device_sm_count(int* sms) {
    int dev = 0;
    KMB_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_func_mutex);
    if (dev < 0 || dev >= 64 || g_sm_count[dev] == 0) {
        int n = 0;
        KMB_CUDA_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        if (dev < 0 || dev >= 64) { *sms = n; return KMB_OK; }
        g_sm_count[dev] = n;
    }
    *sms = g_sm_count[dev];
    return KMB_OK;
}

static int plan_direct(int64_t N, int64_t M, int D, int E, int kid, int flags, int path, DirectPlan* pl) {
    const bool norm = flags & KMB_FLAG_NORMALIZE_ROWS;
    if (D > 16) return set_error(KMB_ERR_UNSUPPORTED, "direct FP32 path supports D <= 16 (got D=%d)", D);
    DirectChoice ch;
    choose_direct(D, E, kid, norm, path, &ch);
    pl->e_chunk = ch.e_chunk;
    pl->n_passes = ch.n_passes;
    pl->form[0].ent = ch.ent[0];
    if (!pl->form[0].ent) return set_error(KMB_ERR_UNSUPPORTED, "no direct kernel for D=%d E=%d kernel=%d", D, E, kid);
    pl->form[1].ent = ch.ent[1];
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    pl->grid_max = sms * 2;
    pl->stats_bytes = align_up(sizeof(DirectStats), 256) + align_up(sizeof(float) * STATS_MAX_BLOCKS * 2 * 16, 256);
    pl->rec_bytes = pl->partial_bytes = pl->counter_bytes = 0;
    for (FormPlan& f : pl->form) {
        if (!f.ent) continue;
        const DirectEntry& e = *f.ent;
        f.n_tiles = (N + e.TILE_ROWS - 1) / e.TILE_ROWS;
        f.nsb = (M + e.SB - 1) / e.SB;
        f.M_pad = f.nsb * e.SB;
        pl->rec_bytes = std::max(pl->rec_bytes, align_up(static_cast<size_t>(f.M_pad) * e.RECV * 16, 256));
        pl->partial_bytes = std::max(pl->partial_bytes, align_up(static_cast<size_t>(pl->grid_max) * 2 * e.TILE_ROWS * e.PS * 4, 256));
        pl->counter_bytes = std::max(pl->counter_bytes, align_up(static_cast<size_t>(f.n_tiles) * 4, 256));
    }
    pl->total_bytes = pl->stats_bytes + pl->rec_bytes + pl->partial_bytes + pl->counter_bytes;
    return KMB_OK;
}

// Symmetric (same_points) product: the record / statistics buffers of the direct pipeline (the symmetric kernels read
// the same packed records) + the strip geometry and the hand-over buffers of kprod_sym.
struct SymPlan {
    DirectPlan direct;          // record layout of both evaluation forms (32-byte records, 512-record blocks)
    SymGeom geom;
    long long unit_begin, unit_end;   // this part's share of the unit list
    int grid, seg_base, strip_base;
    int n_segs, n_strips_part;        // (strip, tile) segments and strips this part's units meet (0 for an empty part)
    size_t rowseg_bytes, rowpart_bytes, colpart_bytes, total_bytes;
};

// Arguments of a symmetric product and the direct kernels whose record layout it reads (host logic only).
static int sym_check(int D, int kernel_id, int part, int n_parts, DirectChoice* ch) {
    if (!sym_supported(D)) return set_error(KMB_ERR_UNSUPPORTED, "symmetric path supports D <= 3 (got D=%d)", D);
    if (n_parts < 1 || part < 0 || part >= n_parts) return set_error(KMB_ERR_INVALID, "bad part %d of %d", part, n_parts);
    if (kernel_id < KMB_KERNEL_GAUSSIAN || kernel_id > KMB_KERNEL_INVERSE_DISTANCE) return set_error(KMB_ERR_UNSUPPORTED, "unknown kernel id %d", kernel_id);
    choose_direct(D, 1, kernel_id, false, KMB_PATH_DIRECT_F32, ch);
    if (!ch->ent[0]) return set_error(KMB_ERR_UNSUPPORTED, "no direct kernel for D=%d E=1 kernel=%d", D, kernel_id);
    for (const DirectEntry* e : ch->ent)
        if (e && (e->SB != sym_block_sources() || e->RECV != 2))
            return set_error(KMB_ERR_UNSUPPORTED, "no 32-byte record layout for D=%d", D);
    return KMB_OK;
}

// Host: the strip geometry for sp->grid CTAs per part, this part's share of the unit list and the hand-over buffers.
static void sym_partition(int64_t n, int part, int n_parts, SymPlan* sp) {
    const long long nsb = (n + sym_block_sources() - 1) / sym_block_sources();
    const long long n_tiles = (n + sym_tile_rows() - 1) / sym_tile_rows();
    sym_geometry(n_tiles, nsb, static_cast<long long>(sp->grid) * n_parts, &sp->geom);
    const long long units = sp->geom.strip_prefix[sp->geom.n_strips];
    sp->unit_begin = units * part / n_parts;
    sp->unit_end = units * (part + 1) / n_parts;
    sp->n_segs = sp->n_strips_part = 0;
    sp->seg_base = sp->strip_base = 0;
    if (sp->unit_end > sp->unit_begin) {
        const SymSeg first = sym_segment_of(sp->geom, sp->unit_begin), last = sym_segment_of(sp->geom, sp->unit_end - 1);
        sp->seg_base = sp->geom.seg_prefix[first.strip] + first.tile;
        sp->strip_base = first.strip;
        sp->n_segs = sp->geom.seg_prefix[last.strip] + last.tile - sp->seg_base + 1;
        sp->n_strips_part = last.strip - first.strip + 1;
    }
    const size_t piece_bytes = static_cast<size_t>(sp->geom.Wb) * sym_block_sources() * 4;
    sp->rowseg_bytes = align_up(static_cast<size_t>(std::max(sp->n_segs, 1)) * sym_tile_rows() * 4, 256);
    sp->rowpart_bytes = align_up(static_cast<size_t>(sp->grid) * 2 * sym_tile_rows() * 4, 256);
    sp->colpart_bytes = align_up(static_cast<size_t>(sp->grid + std::max(sp->n_strips_part, 1)) * piece_bytes, 256);
}

static int plan_sym(int64_t n, int D, int kernel_id, int part, int n_parts, SymPlan* sp) {
    DirectChoice ch;
    if (int rc = sym_check(D, kernel_id, part, n_parts, &ch)) return rc;
    if (int rc = plan_direct(n, n, D, 1, kernel_id, 0, KMB_PATH_DIRECT_F32, &sp->direct)) return rc;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    if (int rc = sym_grid(sms, &sp->grid)) return rc;
    sym_partition(n, part, n_parts, sp);
    sp->total_bytes = sp->direct.total_bytes + sp->rowseg_bytes + sp->rowpart_bytes + sp->colpart_bytes;
    return KMB_OK;
}

__global__ void fill_kernel(float* out, long long n, float v) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < n) out[i] = v;
}

static int check_product_args(int64_t N, int64_t M, int D, int E, int kid, int flags, int path) {
    if (N < 0 || M < 1 || D < 1 || E < 1) return set_error(KMB_ERR_INVALID, "bad sizes N=%lld M=%lld D=%d E=%d", (long long)N, (long long)M, D, E);
    if (kid < 0 || kid > KMB_KERNEL_DOT_EXPONENTIAL) return set_error(KMB_ERR_UNSUPPORTED, "unknown kernel id %d", kid);
    if (kid == KMB_KERNEL_DOT_EXPONENTIAL && (path == KMB_PATH_DIRECT_F32 || path == KMB_PATH_DIRECT_DIFF || path == KMB_PATH_DIRECT_SYM))
        return set_error(KMB_ERR_UNSUPPORTED, "the dot-exponential kernel runs on the tensor paths only (path %d)", path);
    if (kid == KMB_KERNEL_INVERSE_DISTANCE && path == KMB_PATH_TENSOR_1XF16)
        return set_error(KMB_ERR_UNSUPPORTED, "the one-term FP16 path does not support the inverse-distance kernel (1/|x-y| amplifies "
                                              "the error of a one-term S near coincident points)");
    if (flags & ~(KMB_FLAG_NORMALIZE_ROWS | KMB_FLAG_DENSITY | KMB_FLAG_PREPARED | KMB_FLAG_CAUSAL))
        return set_error(KMB_ERR_INVALID, "unknown flags 0x%x", flags);
    if ((flags & KMB_FLAG_DENSITY) && E != 1) return set_error(KMB_ERR_INVALID, "density estimation implies E == 1 (got %d)", E);
    if (path < KMB_PATH_AUTO || path > KMB_PATH_TENSOR_1XF16) return set_error(KMB_ERR_INVALID, "unknown path %d", path);
    if (path == KMB_PATH_DIRECT_SYM) {
        if (N != M) return set_error(KMB_ERR_INVALID, "the symmetric path needs targets == sources (N=%lld, M=%lld)", (long long)N, (long long)M);
        if ((flags & KMB_FLAG_NORMALIZE_ROWS) || E != 1 || !sym_supported(D))
            return set_error(KMB_ERR_UNSUPPORTED, "the symmetric path covers the plain product / density with D <= 3, E = 1");
    }
    return KMB_OK;
}

// KMB_PATH_AUTO.  D > 16: tensor path.  D <= 16: the direct FP32 kernel -- unless the signal is wide (E >= 32) and the
// kernel is one the FP16-plane P.B kernel covers: then K b is a dense contraction and belongs on the tensor cores too
// (D = 3, E = 64: 1531 against 231 Gpairs/s, 1.4e-5 against 7e-7 relative -- the tensor path's tolerance is 1e-4).
// The dot-exponential kernel has no direct kernel: the FP16-plane tensor path at every D (the planes pad D to 16).
constexpr int kWideSignal = 32;
// the operand planes of a tensor path (kprod_tensor.cuh: elt), -1 for the other paths
static int tensor_elt(int path) {
    return path == KMB_PATH_TENSOR_3XTF32 ? 0 : path == KMB_PATH_TENSOR_3XF16 ? 1 : path == KMB_PATH_TENSOR_1XF16 ? 2 : -1;
}
// KMB_FLAG_CAUSAL: the causal kernels are the three-term FP16 ones, so the tensor path at every D as well.
bool tensor_pv16_applicable(int D, int E, int kid);   // kprod_tensor_pv16.cu
bool tensor_pv_applicable(int D, int E);              // kprod_tensor_pv.cu
static int resolve_path(int D, int E, int kid, int flags, int path) {
    if (path != KMB_PATH_AUTO) return path;
    if (D > 16 || kid == KMB_KERNEL_DOT_EXPONENTIAL || (flags & KMB_FLAG_CAUSAL)) return KMB_PATH_TENSOR_3XF16;
    return (E >= kWideSignal && tensor_pv16_applicable(D, E, kid)) ? KMB_PATH_TENSOR_3XF16 : KMB_PATH_DIRECT_F32;
}

// KMB_FLAG_CAUSAL runs on the three-term FP16 kernels (kprod_tensor, _pair, pv16, pv16_pair) only: the other paths, and
// the one shape the FP16 path hands to the TF32 P.B kernel (inverse distance, E > 4, D <= 128), have no causal kernel.
static int check_causal(int D, int E, int kid, int flags, int path) {
    if (!(flags & KMB_FLAG_CAUSAL)) return KMB_OK;
    if (resolve_path(D, E, kid, flags, path) != KMB_PATH_TENSOR_3XF16)
        return set_error(KMB_ERR_UNSUPPORTED, "causal products run on the three-term FP16 tensor path only (path %d)", path);
    if (!((flags & KMB_FLAG_NORMALIZE_ROWS) && (flags & KMB_FLAG_DENSITY)) && tensor_pv_applicable(D, E) &&
        !tensor_pv16_applicable(D, E, kid))
        return set_error(KMB_ERR_UNSUPPORTED, "no causal kernel for the TF32 P.B family (inverse distance, E > 4, D <= 128)");
    return KMB_OK;
}

// Enqueue the direct pipeline on `stream`: bounding-box statistics -> source packing -> main kernels.
//   sym == nullptr  out (N x E) = product of the N targets x with all M sources.
//   sym != nullptr  targets == sources == y (x is y, N == M, E == 1).  The symmetric kernel (Gaussian: product form
//                   and difference form both enqueued, the data decide) runs over this part's share of the unit
//                   list and writes this part's contribution to all N rows of out: the parts' outputs add up to
//                   the product.
static int run_direct(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E,
                      int kernel_id, int flags, int64_t row_offset, const DirectPlan& pl, const SymPlan* sym, char* ws,
                      cudaStream_t stream) {
    const bool density = b == nullptr;
    (void)flags;
    DirectStats* stats = reinterpret_cast<DirectStats*>(ws);
    float* block_box = reinterpret_cast<float*>(ws + align_up(sizeof(DirectStats), 256));
    float2* rec = reinterpret_cast<float2*>(ws + pl.stats_bytes);
    float* partial = reinterpret_cast<float*>(ws + pl.stats_bytes + pl.rec_bytes);
    int* counters = reinterpret_cast<int*>(ws + pl.stats_bytes + pl.rec_bytes + pl.partial_bytes);
    KMB_CUDA_CHECK(cudaMemsetAsync(stats, 0, sizeof(DirectStats), stream));
    KMB_CUDA_CHECK(cudaMemsetAsync(counters, 0, pl.counter_bytes, stream));

    // bounding box -> centre, radius, evaluation form (stays on the device)
    {
        const long long pts = M + ((x == y && N == M) ? 0 : N);
        long long blocks = (pts + STATS_THREADS * 8 - 1) / (STATS_THREADS * 8);
        blocks = std::max(1LL, std::min<long long>(blocks, STATS_MAX_BLOCKS));
        direct_stats_kernel<<<static_cast<unsigned>(blocks), STATS_THREADS, 0, stream>>>(x, N, y, M, D, block_box, stats,
                                                                                         pl.form[1].ent ? 1 : 0);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
    }

    // resident CTAs per SM of each instantiation (cached per kernel function and device)
    auto resident = [&](const DirectEntry& ent, int* per_sm) -> int {
        if (int rc = resident_ctas(ent.func, ent.THREADS, ent.SMEM, per_sm)) return rc;
        if (*per_sm > 2) *per_sm = 2;
        return KMB_OK;
    };

    const float scale = coord_scale(kernel_id);
    const DirectEntry& e0ent = *pl.form[0].ent;
    PackLayout lay[2];
    for (int f = 0; f < 2; ++f) {
        const DirectEntry* e = pl.form[f].ent ? pl.form[f].ent : pl.form[0].ent;
        const FormPlan& fp = pl.form[f].ent ? pl.form[f] : pl.form[0];
        lay[f].M_pad = fp.M_pad;
        lay[f].wcol = e->WCOL;
        lay[f].pairs_per_rec = e->RECV * 2;
    }
    const long long pack_rows = std::max(lay[0].M_pad, lay[1].M_pad);
    for (int pass = 0; pass < pl.n_passes; ++pass) {
        const int e0 = pass * pl.e_chunk;
        pack_sources_kernel<<<static_cast<unsigned>((pack_rows + 255) / 256), 256, 0, stream>>>(
            y, density ? nullptr : b, rec, stats, M, D, E, e0ent.DP, e0ent.EP, lay[0], lay[1], e0, scale);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
        if (g_profile) {
            if (!g_ev0) {
                KMB_CUDA_CHECK(cudaEventCreate(&g_ev0));
                KMB_CUDA_CHECK(cudaEventCreate(&g_ev1));
            }
            KMB_CUDA_CHECK(cudaEventRecord(g_ev0, stream));
        }
        if (sym) {
            // this part's share of the strip-ordered unit list -> kprod_sym + combine, once per evaluation form
            char* sb = ws + pl.total_bytes;
            SymParams S;
            S.stats = stats;
            S.rec = reinterpret_cast<const float4*>(rec);
            S.rowseg = reinterpret_cast<float*>(sb);
            S.rowpart = reinterpret_cast<float*>(sb + sym->rowseg_bytes);
            S.colpart = reinterpret_cast<float*>(sb + sym->rowseg_bytes + sym->rowpart_bytes);
            S.out = out;
            S.N = N;
            S.M = M;
            S.unit_begin = sym->unit_begin;
            S.unit_end = sym->unit_end;
            S.piece_floats = static_cast<long long>(sym->geom.Wb) * sym_block_sources();
            S.grid = sym->grid;
            S.seg_base = sym->seg_base;
            S.strip_base = sym->strip_base;
            S.g = sym->geom;
            for (int f = 1; f >= 0; --f) {
                if (!pl.form[f].ent) continue;
                if (int rc = sym_launch(D, kernel_id, f, S, stream)) return rc;
            }
        }
        // both forms are enqueued; the one the data did not select returns at once
        for (int f = 1; f >= 0 && !sym; --f) {
            if (!pl.form[f].ent) continue;
            const DirectEntry& ent = *pl.form[f].ent;
            int per_sm = 0;
            if (int rc = resident(ent, &per_sm)) return rc;
            const long long units = pl.form[f].n_tiles * pl.form[f].nsb;
            long long grid = static_cast<long long>(pl.grid_max / 2) * per_sm;
            if (grid > units) grid = units;
            DirectParams P;
            P.x = x;
            P.stats = stats;
            P.rec = reinterpret_cast<const float4*>(rec);
            P.out = out;
            P.partial = partial;
            P.tile_counter = counters;
            P.N = N;
            P.M = M;
            P.row_offset = row_offset;
            P.D = D;
            P.E = E;
            P.e0 = e0;
            P.n_tiles = static_cast<int>(pl.form[f].n_tiles);
            P.n_src_blocks = static_cast<int>(pl.form[f].nsb);
            P.xscale = scale;
            KMB_CUDA_CHECK(ent.launch(P, static_cast<int>(grid), stream));
            count_launch();
        }
        if (g_profile) {
            KMB_CUDA_CHECK(cudaEventRecord(g_ev1, stream));
            g_ev_valid = true;
        }
    }
    return KMB_OK;
}

}  // namespace kmb

using namespace kmb;

extern "C" {

int kmb_abi_version(void) { return KMB_ABI_VERSION; }
const char* kmb_last_error(void) { return g_err; }
int kmb_last_launch_count(void) { return g_launches; }

int kmb_set_profiling(int enabled) {
    g_profile = enabled != 0;
    g_ev_valid = false;
    return KMB_OK;
}
int kmb_last_main_kernel_ms(float* ms) {
    if (!ms) return set_error(KMB_ERR_INVALID, "ms is NULL");
    if (!g_ev_valid) return set_error(KMB_ERR_INVALID, "no profiled product call on this thread");
    KMB_CUDA_CHECK(cudaEventSynchronize(g_ev1));
    KMB_CUDA_CHECK(cudaEventElapsedTime(ms, g_ev0, g_ev1));
    return KMB_OK;
}

int kmb_get_device_info(int device, kmb_device_info* info) {
    if (!info) return set_error(KMB_ERR_INVALID, "info is NULL");
    cudaDeviceProp p;
    KMB_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    info->sm_count = p.multiProcessorCount;
    info->cc_major = p.major;
    info->cc_minor = p.minor;
    KMB_CUDA_CHECK(cudaDeviceGetAttribute(&info->clock_khz, cudaDevAttrClockRate, device));
    info->l2_bytes = p.l2CacheSize;
    info->smem_per_block_optin = static_cast<int>(p.sharedMemPerBlockOptin);
    info->total_mem = p.totalGlobalMem;
    return KMB_OK;
}

int kmb_product_workspace_bytes(int64_t N, int64_t M, int D, int E, int kernel_id, int flags, int path,
                                size_t* bytes) {
    if (!bytes) return set_error(KMB_ERR_INVALID, "bytes is NULL");
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, path)) return rc;
    if (int rc = check_causal(D, E, kernel_id, flags, path)) return rc;
    *bytes = 256;
    if ((flags & KMB_FLAG_NORMALIZE_ROWS) && (flags & KMB_FLAG_DENSITY)) return KMB_OK;
    const int p = resolve_path(D, E, kernel_id, flags, path);
    if (p == KMB_PATH_DIRECT_SYM) return kmb_product_sym_workspace_bytes(N, D, 0, 1, bytes);
    if (p == KMB_PATH_DIRECT_F32 || p == KMB_PATH_DIRECT_DIFF) {
        DirectPlan pl;
        if (int rc = plan_direct(N, M, D, E, kernel_id, flags, p, &pl)) return rc;
        *bytes = pl.total_bytes;
        return KMB_OK;
    }
    return tensor_workspace_bytes(N, M, D, E, kernel_id, flags, tensor_elt(p), bytes);
}

int kmb_product_f32(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D,
                    int E, int kernel_id, int flags, int path, int64_t row_offset, void* workspace,
                    size_t workspace_bytes, void* stream_) {
    g_launches = 0;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, path)) return rc;
    if (int rc = check_causal(D, E, kernel_id, flags, path)) return rc;
    if (N == 0) return KMB_OK;   // an empty row shard (x and out may then be NULL: empty tensors have no storage)
    if (!x || !y || !out) return set_error(KMB_ERR_INVALID, "x, y and out must not be NULL");
    const bool density = flags & KMB_FLAG_DENSITY;
    if (!density && !b) return set_error(KMB_ERR_INVALID, "b is NULL without KMB_FLAG_DENSITY");

    if ((flags & KMB_FLAG_NORMALIZE_ROWS) && density) {  // bruteforce.py:134-138
        fill_kernel<<<static_cast<unsigned>((N + 255) / 256), 256, 0, stream>>>(out, N, 1.0f);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
        return KMB_OK;
    }
    const int p = resolve_path(D, E, kernel_id, flags, path);
    if (reinterpret_cast<uintptr_t>(workspace) % 256)
        return set_error(KMB_ERR_INVALID, "workspace must be 256-byte aligned");
    if (tensor_elt(p) >= 0) {
        if (g_profile && !g_ev0) {
            KMB_CUDA_CHECK(cudaEventCreate(&g_ev0));
            KMB_CUDA_CHECK(cudaEventCreate(&g_ev1));
        }
        const int rc = tensor_product(x, y, density ? nullptr : b, out, N, M, D, E, kernel_id, flags, tensor_elt(p), row_offset, workspace,
                                      workspace_bytes, stream, g_profile ? g_ev0 : nullptr, g_profile ? g_ev1 : nullptr,
                                      (flags & KMB_FLAG_PREPARED) != 0);
        if (rc == KMB_OK && g_profile) g_ev_valid = true;
        return rc;
    }

    if (p == KMB_PATH_DIRECT_SYM) {
        if (x != y) return set_error(KMB_ERR_INVALID, "the symmetric path needs x == y (same_points)");
        return kmb_product_sym_f32(y, density ? nullptr : b, out, N, D, kernel_id, 0, 1, workspace, workspace_bytes, stream_);
    }
    DirectPlan pl;
    if (int rc = plan_direct(N, M, D, E, kernel_id, flags, p, &pl)) return rc;
    if (!workspace || workspace_bytes < pl.total_bytes)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", pl.total_bytes, workspace_bytes);
    return run_direct(x, y, density ? nullptr : b, out, N, M, D, E, kernel_id, flags, row_offset, pl, nullptr,
                      static_cast<char*>(workspace), stream);
}

int kmb_product_prepare_f32(const float* x, const float* y, int64_t N, int64_t M, int D, int kernel_id, int flags, int path,
                            void* workspace, size_t workspace_bytes, void* stream_) {
    g_launches = 0;
    if (int rc = check_product_args(N, M, D, 1, kernel_id, flags & ~KMB_FLAG_DENSITY, path)) return rc;
    if (int rc = check_causal(D, 1, kernel_id, flags & ~KMB_FLAG_DENSITY, path)) return rc;
    if (!x || !y) return set_error(KMB_ERR_INVALID, "x and y must not be NULL");
    if (N == 0) return KMB_OK;
    const int p = resolve_path(D, 1, kernel_id, flags, path);   // (D <= 16 under KMB_PATH_AUTO: the signal width decides at query time)
    if (p != KMB_PATH_TENSOR_3XF16 && p != KMB_PATH_TENSOR_1XF16) return KMB_OK;   // nothing worth keeping on the other paths
    if (reinterpret_cast<uintptr_t>(workspace) % 256) return set_error(KMB_ERR_INVALID, "workspace must be 256-byte aligned");
    return tensor_prepare(x, y, N, M, D, kernel_id, tensor_elt(p), workspace, workspace_bytes, static_cast<cudaStream_t>(stream_));
}

int kmb_product_f64(const double* x, const double* y, const double* b, double* out, int64_t N, int64_t M, int D, int E,
                    int kernel_id, int flags, int64_t row_offset, void* stream_) {
    g_launches = 0;
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, KMB_PATH_AUTO)) return rc;
    if (N == 0) return KMB_OK;
    if (!x || !y || !out) return set_error(KMB_ERR_INVALID, "x, y and out must not be NULL");
    if (!(flags & KMB_FLAG_DENSITY) && !b) return set_error(KMB_ERR_INVALID, "b is NULL without KMB_FLAG_DENSITY");
    return product_f64(x, y, b, out, N, M, D, E, kernel_id, flags, row_offset, static_cast<cudaStream_t>(stream_));
}

int kmb_debug_plan_waves(int64_t n_tiles, int64_t n_source_blocks, int grid, size_t row_tile_bytes, int64_t* out7) {
    if (!out7 || n_tiles < 1 || n_source_blocks < 1 || grid < 1) return set_error(KMB_ERR_INVALID, "bad arguments");
    long long o[7];
    tensor_plan_waves_debug(n_tiles, n_source_blocks, grid, row_tile_bytes, o);
    for (int i = 0; i < 7; ++i) out7[i] = o[i];
    return KMB_OK;
}

int kmb_resolved_path(int D, int E, int kernel_id, int path) {
    if (D < 1 || E < 1 || kernel_id < KMB_KERNEL_GAUSSIAN || kernel_id > KMB_KERNEL_DOT_EXPONENTIAL || path < KMB_PATH_AUTO ||
        path > KMB_PATH_TENSOR_1XF16)
        return -1;
    return resolve_path(D, E, kernel_id, 0, path);
}

int kmb_debug_direct_entry(int table, int index, int32_t* out11) {
    if (!out11 || table < 0 || table >= 8) return set_error(KMB_ERR_INVALID, "bad arguments");
    const DirectTable& t = kDirectTables[table];
    out11[0] = *t.count;
    for (int i = 1; i < 11; ++i) out11[i] = -1;
    if (index < 0 || index >= *t.count) return KMB_OK;
    const DirectEntry& e = t.tab[index];
    const int32_t v[10] = {e.KID, e.NORM, e.FORM, e.DP, e.EP, e.R, e.TILE_ROWS, e.SB, e.RECV, e.PS};
    for (int i = 0; i < 10; ++i) out11[1 + i] = v[i];
    return KMB_OK;
}

int kmb_debug_product_plan(int64_t N, int64_t M, int D, int E, int kernel_id, int flags, int path, int sms, int64_t* out10) {
    if (!out10 || sms < 1) return set_error(KMB_ERR_INVALID, "bad arguments");
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, path)) return rc;
    if (int rc = check_causal(D, E, kernel_id, flags, path)) return rc;
    for (int i = 0; i < 10; ++i) out10[i] = -1;
    const int p = resolve_path(D, E, kernel_id, flags, path);
    out10[0] = p;
    if ((flags & KMB_FLAG_NORMALIZE_ROWS) && (flags & KMB_FLAG_DENSITY)) {
        out10[1] = KMB_FAMILY_FILL;
        return KMB_OK;
    }
    if (p == KMB_PATH_DIRECT_SYM) {
        out10[1] = KMB_FAMILY_SYM;
        return KMB_OK;
    }
    if (tensor_elt(p) >= 0) {
        long long t[4];
        tensor_plan_debug(N, D, E, kernel_id, tensor_elt(p), sms, t);
        out10[1] = t[0];
        out10[6] = t[1];
        out10[7] = t[2];
        out10[8] = t[3];
        return KMB_OK;
    }
    DirectChoice ch;
    if (D <= 16) choose_direct(D, E, kernel_id, flags & KMB_FLAG_NORMALIZE_ROWS, p, &ch);
    if (D > 16 || !ch.ent[0]) {
        out10[1] = KMB_FAMILY_UNSUPPORTED;
        return KMB_OK;
    }
    out10[1] = KMB_FAMILY_DIRECT;
    for (int f = 0; f < 2; ++f) {
        if (!ch.ent[f]) continue;
        for (int t = 0; t < 8; ++t) {
            const DirectTable& tab = kDirectTables[t];
            if (ch.ent[f] >= tab.tab && ch.ent[f] < tab.tab + *tab.count) {
                out10[2 + 2 * f] = t;
                out10[3 + 2 * f] = ch.ent[f] - tab.tab;
            }
        }
    }
    out10[6] = ch.e_chunk;
    out10[7] = ch.n_passes;
    out10[8] = (N + ch.ent[0]->TILE_ROWS - 1) / ch.ent[0]->TILE_ROWS;
    out10[9] = (M + ch.ent[0]->SB - 1) / ch.ent[0]->SB;
    return KMB_OK;
}

int kmb_debug_pv_plan(int64_t N, int64_t M, int D, int E, int kernel_id, int flags, int path, int sms, int smem_optin,
                      int64_t* out19) {
    if (!out19 || sms < 1 || smem_optin < 1) return set_error(KMB_ERR_INVALID, "bad arguments");
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, path)) return rc;
    int64_t plan[10];
    if (int rc = kmb_debug_product_plan(N, M, D, E, kernel_id, flags, path, sms, plan)) return rc;
    long long o[KMB_PV_PLAN_FIELDS];
    for (int i = 0; i < KMB_PV_PLAN_FIELDS; ++i) o[i] = -1;
    o[0] = plan[1];
    if (plan[1] == KMB_FAMILY_PV || plan[1] == KMB_FAMILY_PV16 || plan[1] == KMB_FAMILY_PV16_PAIR)
        if (int rc = tensor_pv_plan_query(N, M, D, E, kernel_id, tensor_elt(static_cast<int>(plan[0])), sms, smem_optin, o))
            return rc;
    for (int i = 0; i < KMB_PV_PLAN_FIELDS; ++i) out19[i] = o[i];
    return KMB_OK;
}

int kmb_debug_causal_work(int64_t N, int64_t M, int D, int E, int kernel_id, int flags, int path, int64_t row_offset, int sms,
                          int smem_optin, int wave, int unit, int64_t* out9) {
    if (!out9 || N < 1 || sms < 1 || smem_optin < 1 || row_offset < 0) return set_error(KMB_ERR_INVALID, "bad arguments");
    if (!(flags & KMB_FLAG_CAUSAL)) return set_error(KMB_ERR_INVALID, "kmb_debug_causal_work needs KMB_FLAG_CAUSAL");
    if ((flags & KMB_FLAG_NORMALIZE_ROWS) && (flags & KMB_FLAG_DENSITY)) return set_error(KMB_ERR_INVALID, "a filled result has no plan");
    if (int rc = check_product_args(N, M, D, E, kernel_id, flags, path)) return rc;
    if (int rc = check_causal(D, E, kernel_id, flags, path)) return rc;
    long long o[KMB_CAUSAL_WORK_FIELDS];
    if (int rc = tensor_causal_work_debug(N, M, D, E, kernel_id, row_offset, sms, smem_optin, wave, unit, o)) return rc;
    for (int i = 0; i < KMB_CAUSAL_WORK_FIELDS; ++i) out9[i] = o[i];
    return KMB_OK;
}

int kmb_debug_sym_unit(int64_t n, int64_t total_ctas, int64_t u, int64_t* out8) {
    if (!out8 || n < 1 || total_ctas < 1) return set_error(KMB_ERR_INVALID, "bad arguments");
    SymGeom g;
    sym_geometry((n + sym_tile_rows() - 1) / sym_tile_rows(), (n + sym_block_sources() - 1) / sym_block_sources(), total_ctas, &g);
    out8[0] = g.strip_prefix[g.n_strips];
    out8[1] = g.n_strips;
    out8[2] = g.Wb;
    for (int i = 3; i < 8; ++i) out8[i] = -1;
    if (u < 0 || u >= out8[0]) return KMB_OK;
    const SymSeg sg = sym_segment_of(g, u);
    out8[3] = sg.strip;
    out8[4] = sg.tile;
    out8[5] = sg.jb0 + (u - sg.begin);
    out8[6] = sg.begin;
    out8[7] = sg.len;
    return KMB_OK;
}

int kmb_debug_sym_plan(int64_t n, int D, int kernel_id, int part, int n_parts, int sms, int64_t* out) {
    if (!out || n < 1 || sms < 1) return set_error(KMB_ERR_INVALID, "bad arguments");
    DirectChoice ch;
    if (int rc = sym_check(D, kernel_id, part, n_parts, &ch)) return rc;
    SymPlan sp;
    sp.grid = sms;   // sym_grid: one CTA per SM
    sym_partition(n, part, n_parts, &sp);
    const SymGeom& g = sp.geom;
    // the strip-count cap binds when it makes the strips wider than the CTA count alone would
    const bool capped = g.Wb > sym_cta_strip_width(g.nsb, static_cast<long long>(sms) * n_parts);
    const long long v[KMB_SYM_PLAN_FIELDS] = {sym_tile_rows(), sym_block_sources(), sym_tile_rows() / sym_block_sources(),
                                              g.strip_prefix[g.n_strips], sp.unit_begin, sp.unit_end,
                                              std::min<long long>(sms, sp.unit_end - sp.unit_begin), g.n_strips, g.Wb,
                                              sp.seg_base, sp.strip_base, sp.n_segs, sp.n_strips_part,
                                              (ch.ent[0] ? 1 : 0) | (ch.ent[1] ? 2 : 0), capped ? 1 : 0};
    for (int i = 0; i < KMB_SYM_PLAN_FIELDS; ++i) out[i] = v[i];
    return KMB_OK;
}

int kmb_kernel_block_f64(const double* x, const double* y, double* out, int64_t n, int64_t m, int D, int kernel_id, void* stream_) {
    g_launches = 0;
    if (n < 0 || m < 1 || D < 1) return set_error(KMB_ERR_INVALID, "bad sizes n=%lld m=%lld D=%d", (long long)n, (long long)m, D);
    if (kernel_id < KMB_KERNEL_GAUSSIAN || kernel_id > KMB_KERNEL_DOT_EXPONENTIAL) return set_error(KMB_ERR_UNSUPPORTED, "unknown kernel %d", kernel_id);
    if (!x || !y || !out) return set_error(KMB_ERR_INVALID, "x, y and out must not be NULL");
    if (n == 0) return KMB_OK;
    return kernel_block_f64(x, y, out, n, m, D, kernel_id, static_cast<cudaStream_t>(stream_));
}

int kmb_product_sym_workspace_bytes(int64_t n, int D, int part, int n_parts, size_t* bytes) {
    if (!bytes) return set_error(KMB_ERR_INVALID, "bytes is NULL");
    if (n < 1) return set_error(KMB_ERR_INVALID, "bad size n=%lld", (long long)n);
    SymPlan sp;
    if (int rc = plan_sym(n, D, KMB_KERNEL_GAUSSIAN, part, n_parts, &sp)) return rc;   // the Gaussian plan (two forms) is the largest
    *bytes = sp.total_bytes;
    return KMB_OK;
}

int kmb_product_sym_f32(const float* y, const float* b, float* out, int64_t n, int D, int kernel_id, int part, int n_parts,
                        void* workspace, size_t workspace_bytes, void* stream_) {
    g_launches = 0;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n < 1 || D < 1) return set_error(KMB_ERR_INVALID, "bad sizes n=%lld D=%d", (long long)n, D);
    if (!y || !out) return set_error(KMB_ERR_INVALID, "y and out must not be NULL");   // b == NULL: density (b == 1)
    SymPlan sp;
    if (int rc = plan_sym(n, D, kernel_id, part, n_parts, &sp)) return rc;
    if (!workspace || workspace_bytes < sp.total_bytes)
        return set_error(KMB_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", sp.total_bytes, workspace_bytes);
    if (reinterpret_cast<uintptr_t>(workspace) % 256)
        return set_error(KMB_ERR_INVALID, "workspace must be 256-byte aligned");
    return run_direct(y, y, b, out, n, n, D, 1, kernel_id, 0, 0, sp.direct, &sp, static_cast<char*>(workspace), stream);
}

}  // extern "C"
