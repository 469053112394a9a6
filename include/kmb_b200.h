/* kmb_b200.h -- C ABI of libkmb_b200.so: the B200 (sm_100a) kernel-matrix hot path.
 *
 * The reference (kernel-matrix-benchmarks) is pure Python: its hot path is
 * kernel_matrix_benchmarks/algorithms/bruteforce.py, called through the plugin
 * interface of algorithms/base.py.  It has no FFI of its own, so this header
 * declares what a ctypes binding for that path binds (INTEGRATION.md shows the
 * stub); each entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a KMB_ERR_* code otherwise; the
 *     message for the calling thread is kmb_last_error().  No exceptions, no
 *     torch types, no hidden allocation: all device buffers (inputs, outputs,
 *     workspace) belong to the caller.
 *   - "device pointer" arguments are fp32, row-major, contiguous, 16-byte
 *     aligned, resident on the current CUDA device; `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).  Calls are asynchronous
 *     on `stream` unless stated otherwise.
 *   - sizes are int64_t; D (point dimension) and E (signal dimension) are int.
 *   - not thread-safe per stream/workspace (the reference's caller,
 *     runner.py:70-176, is single-threaded).
 */
#ifndef KMB_B200_H
#define KMB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMB_ABI_VERSION 1

/* error codes */
enum {
    KMB_OK = 0,
    KMB_ERR_INVALID = 1,     /* bad argument (NULL pointer, negative size, ...) */
    KMB_ERR_UNSUPPORTED = 2, /* kernel / path / shape not implemented -> NotImplementedError in Python,
                                as bruteforce.py:82-85 does for unknown kernels */
    KMB_ERR_WORKSPACE = 3,   /* workspace too small */
    KMB_ERR_CUDA = 4         /* a CUDA runtime call failed; message carries cudaGetErrorString */
};

/* kernel functions: bruteforce.py:18-22 */
enum {
    KMB_KERNEL_GAUSSIAN = 0,             /* exp(-|x-y|^2)              :20 */
    KMB_KERNEL_ABSOLUTE_EXPONENTIAL = 1, /* exp(-|x-y|)                :21 */
    KMB_KERNEL_INVERSE_DISTANCE = 2,     /* 1/|x-y|, flat indices k(M+1) zeroed  :8-15 */
    KMB_KERNEL_DOT_EXPONENTIAL = 3       /* exp(<x, y>): NOT in bruteforce.py (an extension; with KMB_FLAG_NORMALIZE_ROWS
                                            this is softmax attention softmax(x y^T) b).  Tensor paths only
                                            (KMB_PATH_AUTO resolves to KMB_PATH_TENSOR_3XF16 at every D); the direct and
                                            symmetric paths return KMB_ERR_UNSUPPORTED.  The plain product is FP32 and
                                            overflows to inf where exp(<x, y>) does (<x, y> > ~88); row normalisation
                                            runs under an online maximum and stays finite beyond that. */
};

/* query modes: BruteForceProductBLAS.query, bruteforce.py:130-153 */
enum {
    KMB_FLAG_NORMALIZE_ROWS = 1, /* attention: (K @ [b,1])[:, :-1] / [:, -1:]     :139-145 */
    KMB_FLAG_DENSITY = 2,        /* b == 1, E == 1: K.sum(-1)                      :150    */
    KMB_FLAG_PREPARED = 4        /* the points-only work was done by kmb_product_prepare_f32 on this workspace (below) */
};

/* evaluation paths */
enum {
    KMB_PATH_AUTO = 0,
    KMB_PATH_DIRECT_F32 = 1,   /* FP32 FMA + MUFU path, D <= 16.  Squared distances as a sum of squared
                                  differences (bruteforce.py:53-54); for the Gaussian kernel on data whose
                                  centred bounding box is small (log2(e) * half-diagonal^2 <= 6, decided on
                                  the device) the algebraically equal product form
                                  2^(-|u|^2) 2^(2u.v) 2^(-|v|^2) is used instead (4 FMA slots per pair, not 7) */
    KMB_PATH_TENSOR_3XTF32 = 2, /* |x|^2+|y|^2-2x.y (bruteforce.py:36-49) on tcgen05, 3xTF32 split, D >= 32 */
    KMB_PATH_DIRECT_DIFF = 3,  /* KMB_PATH_DIRECT_F32 restricted to the difference form */
    KMB_PATH_TENSOR_3XF16 = 5, /* the same tensor path with FP16 hi/lo operand planes instead of TF32 ones: the data are
                                  centred and scaled by a power of two (chosen on the device from the column extrema)
                                  so that the largest operand lies in [2^13, 2^15); hi + lo carry 22 significand
                                  bits as the TF32 split does, kind::f16 MMAs run at twice the TF32 rate and the
                                  operand planes are half as large.  What KMB_PATH_AUTO picks for D > 16. */
    KMB_PATH_TENSOR_1XF16 = 6, /* KMB_PATH_TENSOR_3XF16 with only the hi.hi term: the same prepass and hi planes (11 significand
                                  bits per operand), but the lo planes of the points and of the signal are neither loaded
                                  nor multiplied, S = u.v and (E > 4) P.B are one kind::f16 MMA per K step where the
                                  three-term path issues three, and P is written to tensor memory as one FP16 plane (the
                                  row sums use the same rounded weights).  Float16-class results: about 1e-5 relative for
                                  E <= 4 (S alone), about 3e-4 to 1e-3 for E > 4 (dominated by rounding P and b to FP16),
                                  still well inside what a float16 evaluation of the reference gives.  Gaussian,
                                  exponential and dot-exponential kernels; the inverse distance (1/|x - y| amplifies the
                                  cancellation error of S near coincident points) and shapes whose three-term product
                                  would take the TF32 P.B kernel return KMB_ERR_UNSUPPORTED.  Never chosen by
                                  KMB_PATH_AUTO.  A workspace prepared for one path belongs to that path. */
    KMB_PATH_DIRECT_SYM = 4    /* targets == sources (the reference's same_points, base.py:56-79): x must be the
                                  same pointer as y.  Plain product or density of any kernel, D <= 3, E == 1: every kernel
                                  value is evaluated once and feeds a_i += k b_j and a_j += k b_i (K is
                                  symmetric), see kmb_product_sym_f32.  Never chosen by KMB_PATH_AUTO (the
                                  library cannot see aliasing in kmb_product_workspace_bytes) */
};

typedef struct {
    int sm_count;
    int cc_major, cc_minor;
    int clock_khz;           /* cudaDevAttrClockRate */
    int l2_bytes;
    int smem_per_block_optin;
    size_t total_mem;
} kmb_device_info;

int kmb_abi_version(void);
const char* kmb_last_error(void);
int kmb_get_device_info(int device, kmb_device_info* info);

/* Workspace (bytes) kmb_product_f32 needs for this shape; *bytes is a multiple of 256. */
int kmb_product_workspace_bytes(int64_t n_targets, int64_t n_sources, int D, int E, int kernel_id,
                                int flags, int path, size_t* bytes);

/* out[i, :] = sum_j k(x_i, y_j) b[j, :]   (K is never materialised)
 *
 * Replaces kernel_matrix(...) + the matrix product of
 * BruteForceProductBLAS.fit/query (bruteforce.py:25-58, 113-120, 130-153).
 *
 *   x   (n_targets, D)  target points  (device)   -- may alias y (same_points)
 *   y   (n_sources, D)  source points  (device)
 *   b   (n_sources, E)  source signal  (device); NULL with KMB_FLAG_DENSITY (then E must be 1)
 *   out (n_targets, E)  result         (device)
 *   row_offset: global index of x's first row in the full target set.  Only
 *     the inverse-distance kernel looks at it (its zeroing rule depends on the
 *     global flat index, bruteforce.py:12-14); pass 0 unless rows are sharded.
 *   KMB_FLAG_NORMALIZE_ROWS | KMB_FLAG_DENSITY fills out with ones (bruteforce.py:134-138).
 */
int kmb_product_f32(const float* x, const float* y, const float* b, float* out, int64_t n_targets,
                    int64_t n_sources, int D, int E, int kernel_id, int flags, int path,
                    int64_t row_offset, void* workspace, size_t workspace_bytes, void* stream);

/* The points-only part of a product: what the reference does in fit() (bruteforce.py:113-120 builds the kernel matrix
 * from the points; query() only multiplies, :130-153).  For the FP16 tensor paths (KMB_PATH_TENSOR_3XF16 / KMB_PATH_AUTO
 * with D > 16, KMB_PATH_TENSOR_1XF16 at every D) this is the prepass -- column statistics, centre, power-of-two scale, FP16 hi/lo operand planes, squared
 * norms -- written to the head of `workspace`, whose layout does not depend on E.  A later kmb_product_f32 with the same
 * x, y, sizes, kernel and path on the SAME workspace memory may then pass KMB_FLAG_PREPARED and skips it; the caller
 * must prepare again if the workspace was reallocated (e.g. grown for a wider signal) or the points changed.  Other
 * paths have nothing worth keeping: the call is a no-op and KMB_FLAG_PREPARED is ignored.  `flags` as for the product
 * (KMB_FLAG_PREPARED itself is ignored here); workspace_bytes >= kmb_product_workspace_bytes(..., E = 1, ...). */
int kmb_product_prepare_f32(const float* x, const float* y, int64_t n_targets, int64_t n_sources, int D, int kernel_id,
                            int flags, int path, void* workspace, size_t workspace_bytes, void* stream);

/* Symmetric product for targets == sources (same_points):
 *     out[i] = this part's share of  sum_j k(y_i, y_j) b[j]        (E == 1, D <= 3, any kernel_id)
 *
 * Same arithmetic as kmb_product_f32(y, y, b, ...) -- kernel_matrix + K @ b of bruteforce.py:25-58,
 * 153 with target_points = None (:27-28, :113-120) -- but K's symmetry is used (every kernel of
 * bruteforce.py:18-22 is a function of |x - y|; the inverse-distance zeroing rule :12-14 zeroes the
 * diagonal when N == M): the n x n pair matrix is cut into (4096 rows x 512 sources) units, only units
 * on or above the block diagonal are evaluated, and each kernel value is added to both its row's and
 * its column's sum.  The unit list (ordered in strips of source blocks so that a CTA works on a
 * compact patch of the matrix, csrc/kprod_sym.cuh) is split into `n_parts` equal contiguous ranges;
 * this call evaluates range `part` and writes the sums it produced to ALL n entries of out (zero where
 * it contributed nothing).  With n_parts > 1 (one part per GPU) the caller adds the parts' outputs --
 * one all-reduce of n floats; with n_parts == 1 out is the product.  Deterministic for a given
 * (n, n_parts, device).  The Gaussian kernel uses the product form when the data allow it and the
 * difference form otherwise (see KMB_PATH_DIRECT_F32; decided on the device), symmetric either way.
 * b == NULL means b == 1 (density estimation, bruteforce.py:150).
 * Workspace: O(n sqrt(CTAs)) floats (77 MB at n = 10^6 on one GPU), the same for every kernel_id.
 * KMB_KERNEL_DOT_EXPONENTIAL is not symmetric in this sense (not a function of |x - y|): KMB_ERR_UNSUPPORTED.
 */
int kmb_product_sym_workspace_bytes(int64_t n, int D, int part, int n_parts, size_t* bytes);
int kmb_product_sym_f32(const float* y, const float* b, float* out, int64_t n, int D, int kernel_id,
                        int part, int n_parts, void* workspace, size_t workspace_bytes, void* stream);

/* ---- several GPUs driven by one host thread --------------------------------------------------------
 * The reference's caller is ONE Python process that calls query() and waits (runner.py:118-148,
 * main.py:299-308), so a plugin that uses G GPUs has to drive them from that one thread.  The calls below
 * take one kmb_device_shard per GPU, launch every shard's product on its own device and stream, and
 * fork/join on shard 0's stream: all work starts after what shard 0's stream held at the call and
 * shard 0's stream continues after every shard is done -- for the caller it is as if the product had
 * run on shard 0's stream (synchronise that one).  No host synchronisation, no NCCL: partial results
 * cross GPUs through NVLink peer memory (kmb_enable_peer_access first).  Pointers in a shard are
 * resident on shard.device unless stated otherwise; b and out MAY point into a peer GPU's memory.
 */
typedef struct {
    int device;             /* CUDA device ordinal of this shard */
    int flags;              /* extra per-shard flags (KMB_FLAG_PREPARED: this shard's workspace holds its prepass) */
    const float* x;         /* rows mode: this shard's block of target rows (n_targets, D), on shard.device */
    const float* y;         /* all source points (n_sources, D), replicated on shard.device */
    const float* b;         /* source signal (n_sources, E); may live on shard 0's device (read once per pass by the packing /
                               transposing kernel, over NVLink); NULL with KMB_FLAG_DENSITY */
    float* out;             /* rows mode: where this shard's rows go -- typically a peer pointer into the gathered
                               (N, E) result on shard 0's device (plain stores over NVLink: the gather costs nothing);
                               symmetric mode: this shard's partial N-vector, on shard.device */
    int64_t n_targets;      /* rows mode: rows in this shard (0 allowed) */
    int64_t row_offset;     /* rows mode: global index of the shard's first row */
    void* workspace;        /* on shard.device, 256-byte aligned */
    size_t workspace_bytes;
    void* stream;           /* a stream of shard.device */
} kmb_device_shard;

/* Peer access in both directions between all listed devices (idempotent).  KMB_ERR_UNSUPPORTED if a pair has no peer path. */
int kmb_enable_peer_access(const int* devices, int n_devices);

/* Rows mode (any kernel / path / query mode of kmb_product_f32): shard s computes its n_targets rows against all sources
 * and stores them at shard.out.  No collective at all. */
int kmb_product_rows_multi_f32(const kmb_device_shard* shards, int n_shards, int64_t n_sources, int D, int E, int kernel_id,
                               int flags, int path);

/* Symmetric mode (kmb_product_sym_f32 with n_parts = n_shards): shard s evaluates range s of the triangular unit list
 * into its own partial vector shard.out (n floats on shard.device; workspace_bytes >= kmb_product_sym_workspace_bytes(n, D,
 * s, n_shards)), then shard 0's device adds the parts in shard order (deterministic) into `out` (n floats on shard 0's
 * device), reading the other parts through peer memory: the path's one exchange step, N floats per GPU over NVLink.
 * With n_shards == 1 the product is written to `out` directly. */
int kmb_product_sym_multi_f32(const kmb_device_shard* shards, int n_shards, float* out, int64_t n, int D, int kernel_id);

/* out[i] = parts[0][i] + ... + parts[n_parts-1][i], fixed order; parts[k] may be peer-device pointers (16-byte aligned,
 * n_parts <= 16).  Runs on the current device / `stream`. */
int kmb_reduce_parts_f32(float* out, const float* const* parts, int n_parts, int64_t n, void* stream);

/* out[i, :] = sum_j k(x_i, y_j) b[j, :] in double precision: the `precision=float64` variant of the
 * reference's plugin (bruteforce.py:64-87, 100-106; algos.yaml:156-162), same arithmetic as its float64
 * difference-form path (bruteforce.py:53-54).  All pointers are float64 device arrays; any D (one row per thread for
 * D <= 16, a tiled kernel above: what the D = 784 / D = 64 ground truth is written with); flags and
 * row_offset as kmb_product_f32.  No workspace.  Row normalisation divides by the plain row sum as the
 * reference does (a row whose kernels all underflow is 0/0 = NaN there and here).  KMB_KERNEL_DOT_EXPONENTIAL:
 * exp(sum_d x_d y_d) in double, the same way (as in kmb_kernel_block_f64).
 */
int kmb_product_f64(const double* x, const double* y, const double* b, double* out, int64_t n_targets,
                    int64_t n_sources, int D, int E, int kernel_id, int flags, int64_t row_offset,
                    void* stream);

/* out[i, j] = k(x_i, y_j) in double precision: an explicit (n, m) block of the kernel matrix -- kernel_matrix(...)
 * of bruteforce.py:25-58 (difference form, :53-54) restricted to m source points.  Used for the m landmark columns of
 * the Nystrom preconditioner of the CG solve (m ~ 10^3; the full matrix is never formed).  x (n, D), y (m, D),
 * out (n, m): float64 device arrays, row-major.  The inverse-distance kernel returns +inf on coincident points (the
 * reference zeroes those by flat index, bruteforce.py:12-14; not applied here). */
int kmb_kernel_block_f64(const double* x, const double* y, double* out, int64_t n, int64_t m, int D, int kernel_id,
                         void* stream);

/* Diagnostics (host logic only, no GPU needed): the wave schedule the tensor-path kernels would use for n_tiles row
 * tiles x n_source_blocks source blocks on `grid` CTAs (CTA pairs: pairs of row tiles on grid / 2 clusters).
 * out7 = {R, C, W, R_last, C_last, slots_per_wave, partial_slots}: W - 1 waves of R row tiles x C CTAs per tile and a
 * last wave of R_last x C_last; CTA b of a wave works on row tile b / C and on source blocks
 * [n_source_blocks (b % C) / C, n_source_blocks (b % C + 1) / C). */
int kmb_debug_plan_waves(int64_t n_tiles, int64_t n_source_blocks, int grid, size_t row_tile_bytes, int64_t* out7);

/* The path KMB_PATH_AUTO stands for with this D, E and kernel (any other `path`, KMB_PATH_TENSOR_1XF16 included, is returned
 * unchanged; -1 on bad arguments):
 * D > 16 -> KMB_PATH_TENSOR_3XF16; D <= 16 -> KMB_PATH_DIRECT_F32, except wide signals (E >= 32) of the Gaussian /
 * exponential kernels, whose K b is a dense contraction and runs on the tensor cores as well.  The dot-exponential
 * kernel resolves to KMB_PATH_TENSOR_3XF16 at every D.  Host logic only. */
int kmb_resolved_path(int D, int E, int kernel_id, int path);

/* Diagnostics (host logic only, no GPU needed): what kmb_product_f32 would launch for this problem on a device with
 * `sms` SMs.  out10 = {resolved path, family (KMB_FAMILY_*), difference-form table, index, product-form table, index,
 * signal columns per pass, passes, row tiles, source blocks}; -1 where a field does not apply.
 *   direct:  (table, index) name kmb_debug_direct_entry entries (the product form only for the Gaussian kernel off
 *            KMB_PATH_DIRECT_DIFF; the data pick one of the two forms on the device); row tiles and source blocks
 *            are those of the difference form.
 *   tensor families: signal columns per pass is min(E, 4) for kprod_tensor (E = 3 runs on its EP = 4
 *            instantiation) and the signal block of the P.B kernels.
 * The CTA-pair decision honours the KMB_TENSOR_PAIR this process has read.  Errors as kmb_product_workspace_bytes. */
enum {
    KMB_FAMILY_DIRECT = 0,       /* kprod_direct (FP32, D <= 16) */
    KMB_FAMILY_SYM = 1,          /* kprod_sym (KMB_PATH_DIRECT_SYM) */
    KMB_FAMILY_TENSOR = 2,       /* kprod_tensor, one CTA per row tile (TF32 or FP16 planes), E <= 4 per pass */
    KMB_FAMILY_TENSOR_PAIR = 3,  /* kprod_tensor_pair: CTA pairs, FP16 planes */
    KMB_FAMILY_PV = 4,           /* kprod_tensor_pv: P.B on the tensor cores, TF32 planes (E > 4, D <= 128) */
    KMB_FAMILY_PV16 = 5,         /* kprod_tensor_pv16, one CTA per row tile (FP16 planes, Gaussian / exponential) */
    KMB_FAMILY_PV16_PAIR = 6,    /* kprod_tensor_pv16_pair */
    KMB_FAMILY_FILL = 7,         /* normalised density: out = 1 */
    KMB_FAMILY_UNSUPPORTED = 8   /* kmb_product_f32 would return KMB_ERR_UNSUPPORTED */
};
int kmb_debug_product_plan(int64_t n_targets, int64_t n_sources, int D, int E, int kernel_id, int flags, int path, int sms,
                           int64_t* out10);

/* Diagnostics (host logic only, no GPU needed): how the P.B kernel (KMB_FAMILY_PV, _PV16, _PV16_PAIR) would run this
 * problem on a device with `sms` SMs and `smem_optin` bytes of opt-in shared memory per block -- the launchers' own
 * plan.  out19 = {family, CTA pairs (0 / 1), grid (CTAs), ring stages, K blocks, K steps of the last K block, signal
 * passes, columns of the first pass, the same padded to 32, columns of the last pass, the same padded to 32, row tiles,
 * source blocks, R, C, W, R_last, C_last (the wave plan, see kmb_debug_plan_waves; with CTA pairs R and R_last count
 * pairs of row tiles), source blocks the P.B accumulators collect between two flushes}.  Another family only fills
 * out19[0] (the others are -1).  The CTA-pair decision and the flush interval honour the KMB_TENSOR_PAIR and
 * KMB_PV16_FLUSH_BLOCKS this process has read.  Errors as kmb_product_workspace_bytes; KMB_ERR_UNSUPPORTED when the
 * kernel's ring does not fit `smem_optin`. */
#define KMB_PV_PLAN_FIELDS 19
int kmb_debug_pv_plan(int64_t n_targets, int64_t n_sources, int D, int E, int kernel_id, int flags, int path, int sms,
                      int smem_optin, int64_t* out19);

/* Diagnostics (host logic only): entry `index` of direct-kernel table `table` (0..7: Gaussian difference form n0, n1,
 * exponential n0, n1, inverse distance n0, n1, Gaussian product form n0, n1; nK = row normalisation off / on).
 * out11 = {entries in the table, KID, NORM, FORM, DP, EP, R (rows per thread), TILE_ROWS, SB (sources per block),
 * RECV (float4 per source record), PS (partial floats per row)}; an index outside the table only fills the first. */
int kmb_debug_direct_entry(int table, int index, int32_t* out11);

/* Diagnostics (host logic only, no GPU needed): where unit `u` of the strip-ordered unit list of the symmetric path
 * sits when n points are worked on by `total_ctas` CTAs over all parts (kprod_sym.cuh).
 * out8 = {total units, strips, strip width in source blocks, strip, row tile, source block, first unit of the
 * (strip, row tile) segment, units in the segment}; u outside [0, total units) only fills the first three. */
int kmb_debug_sym_unit(int64_t n, int64_t total_ctas, int64_t u, int64_t* out8);

/* Diagnostics (host logic only, no GPU needed): how kmb_product_sym_f32 would run part `part` of `n_parts` on a device
 * with `sms` SMs -- the launcher's own geometry and partition (one CTA per SM and part).  out = {row tile rows, sources
 * per block, TB (source blocks per row tile), units in total, this part's first unit, its end (exclusive), CTAs the part
 * launches (min(sms, its units); 0 launches no main kernel), strips, strip width in source blocks, first (strip, tile)
 * segment of the part, its first strip, segments and strips the part meets (0 for an empty part), evaluation forms
 * enqueued (bit 0: difference form, bit 1: Gaussian product form), 1 if the strip-count cap widened the strips beyond
 * what the CTA count asks for}.  Errors as kmb_product_sym_workspace_bytes; KMB_ERR_INVALID for sms < 1. */
#define KMB_SYM_PLAN_FIELDS 15
int kmb_debug_sym_plan(int64_t n, int D, int kernel_id, int part, int n_parts, int sms, int64_t* out);

/* Number of this library's kernels the last kmb_product_f32 / kmb_cg_* call on this
 * thread launched (bench.py's gpu_launches). */
int kmb_last_launch_count(void);

/* Measurement hooks (bench.py's roofline leg).  With profiling enabled on this thread,
 * kmb_product_f32 records a CUDA event on `stream` immediately before and after its dominant
 * kernel (the last pass's main kernel, not the source packing); kmb_last_main_kernel_ms waits
 * for the second event and returns the elapsed device time. */
int kmb_set_profiling(int enabled);
int kmb_last_main_kernel_ms(float* ms);

/* ---- conjugate gradients on (K + lambda I) b = a: fused vector steps -------------------
 * The reference solves K b = a densely (BruteForceSolverLAPACK.query, bruteforce.py:205-207);
 * at N = 10^6 the build iterates with the product above as its matvec.  All vectors are
 * (n_local, E) row shards; scalars live on the device as E floats per quantity so the
 * loop needs no host synchronisation.  *_local outputs are this shard's partial sums: the
 * caller all-reduces them across ranks when rows are sharded.  Reductions are deterministic
 * (fixed block order).  `scratch`: kmb_cg_scratch_bytes() bytes, zeroed once by the caller,
 * 256-byte aligned, reusable across calls on one stream.  E <= 16 per call.
 */
size_t kmb_cg_scratch_bytes(void);

/* x = 0, r = a, p_shard = a, rs_local[e] = sum_i r[i,e]^2 */
int kmb_cg_init_f32(const float* a, float* x, float* r, float* p_shard, float* rs_local,
                    int64_t n_local, int E, void* scratch, void* stream);
/* Ap += lambda * p ; pAp_local[e] = sum_i p[i,e] * Ap[i,e] */
int kmb_cg_shift_dot_f32(float* Ap, const float* p_shard, float lambda, float* pAp_local,
                         int64_t n_local, int E, void* scratch, void* stream);
/* alpha = rs/pAp ; x += alpha p ; r -= alpha Ap ; rs_new_local[e] = sum_i r[i,e]^2 */
int kmb_cg_update_f32(float* x, float* r, const float* p_shard, const float* Ap, const float* rs,
                      const float* pAp, float* rs_new_local, int64_t n_local, int E, void* scratch,
                      void* stream);
/* beta = rs_new/rs ; p = r + beta p */
int kmb_cg_direction_f32(float* p_shard, const float* r, const float* rs_new, const float* rs,
                         int64_t n_local, int E, void* stream);

/* The same four steps in double precision: the `precision: float64` variant of the solver (the reference's
 * algos.yaml:164-181 sweeps float16 / float32 / float64 for BruteForceSolverLAPACK); the matvec is kmb_product_f64. */
int kmb_cg_init_f64(const double* a, double* x, double* r, double* p_shard, double* rs_local,
                    int64_t n_local, int E, void* scratch, void* stream);
int kmb_cg_shift_dot_f64(double* Ap, const double* p_shard, double lambda, double* pAp_local,
                         int64_t n_local, int E, void* scratch, void* stream);
int kmb_cg_update_f64(double* x, double* r, const double* p_shard, const double* Ap, const double* rs,
                      const double* pAp, double* rs_new_local, int64_t n_local, int E, void* scratch,
                      void* stream);
int kmb_cg_direction_f64(double* p_shard, const double* r, const double* rs_new, const double* rs,
                         int64_t n_local, int E, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KMB_B200_H */
