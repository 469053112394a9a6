// kprod_f64: a_i = sum_j k(x_i, y_j) b_j in double precision -- the `precision=float64` variant of the
// reference (/root/reference/kernel_matrix_benchmarks/algorithms/bruteforce.py:64-87, 100-106; algos.yaml:156-162
// sweeps float16 / float32 / float64).  Same arithmetic as the reference's float64 slow path
// (bruteforce.py:53-54: sum of squared differences; :18-22 kernel functions; :130-153 query modes), K never
// materialised.  This is the accuracy end of the Pareto front, not the headline path: one target row per
// thread, sources staged through shared memory, FP64 pipe (64 DFMA/clk/SM) + libdevice exp.
//
// Row normalisation divides by the plain row sum like the reference does (no running maximum): a row
// whose kernels all underflow in float64 is 0/0 = NaN there and here.
//
// The dot-exponential kernel exp(<x, y>) (not in bruteforce.py) runs through the same kernels: its pair term is the
// product x_d y_d where the others have (x_d - y_d)^2.
#include "kmb_common.cuh"

namespace kmb {

namespace {

constexpr int F64_THREADS = 128;
constexpr int F64_SB = 256;        // sources per shared-memory stage
constexpr int F64_MAX_D = 16, F64_MAX_E = 8;

// what one coordinate adds to the kernel's argument: (a - b)^2 (squared distance, bruteforce.py:53-54) or a b (<x, y>)
template <int KID>
__device__ __forceinline__ double pair_term(double a, double b, double acc) {
    if constexpr (KID == KMB_KERNEL_DOT_EXPONENTIAL) return fma(a, b, acc);
    else {
        const double diff = a - b;
        return fma(diff, diff, acc);
    }
}
template <int KID>
__device__ __forceinline__ double kernel_value_f64(double d2) {   // d2: the sum of pair_term
    if constexpr (KID == KMB_KERNEL_GAUSSIAN) return exp(-d2);
    else if constexpr (KID == KMB_KERNEL_DOT_EXPONENTIAL) return exp(d2);
    else if constexpr (KID == KMB_KERNEL_ABSOLUTE_EXPONENTIAL) return exp(-sqrt(fmax(d2, 0.0)));   // bruteforce.py:21
    else return 1.0 / sqrt(fmax(d2, 0.0));                                                          // bruteforce.py:10-11
}

// E columns e0 .. e0+EC-1 of the signal per launch (EC <= F64_MAX_E).  CAUSAL (KMB_FLAG_CAUSAL): row i sums the sources
// j <= row_offset + i only, and the CTA stops at the last source its last row sees.
template <int KID, int EC, bool CAUSAL>
__device__ __forceinline__ void f64_rows_body(const uint32_t tid, const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                                              double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                                              long long row_offset) {
    extern __shared__ double sm[];
    double* sy = sm;                        // F64_SB x D
    double* sb = sm + F64_SB * D;           // F64_SB x EC
    const long long row = blockIdx.x * static_cast<long long>(F64_THREADS) + tid;
    const bool ok = row < N;
    double xr[F64_MAX_D];
#pragma unroll
    for (int d = 0; d < F64_MAX_D; ++d) xr[d] = (ok && d < D) ? x[row * D + d] : 0.0;
    double acc[EC], ksum = 0.0;
#pragma unroll
    for (int e = 0; e < EC; ++e) acc[e] = 0.0;
    [[maybe_unused]] const long long jz = (row_offset + row) % (M + 1);   // inverse-distance zeroing (bruteforce.py:12-14)
    long long m_end = M;
    if constexpr (CAUSAL) m_end = min(M, row_offset + min(N, (blockIdx.x + 1ll) * F64_THREADS));

    for (long long j0 = 0; j0 < m_end; j0 += F64_SB) {
        const int cnt = static_cast<int>(min(static_cast<long long>(F64_SB), m_end - j0));
        __syncthreads();
        for (int i = tid; i < cnt * D; i += F64_THREADS) sy[i] = y[j0 * D + i];
        for (int i = tid; i < cnt * EC; i += F64_THREADS) {
            const int j = i / EC, e = i % EC;
            sb[i] = (e0 + e < E) ? (b ? b[(j0 + j) * E + e0 + e] : 1.0) : 0.0;
        }
        __syncthreads();
        if (ok) {
            for (int j = 0; j < cnt; ++j) {
                double d2 = 0.0;
#pragma unroll
                for (int d = 0; d < F64_MAX_D; ++d) {
                    if (d < D) d2 = pair_term<KID>(xr[d], sy[j * D + d], d2);
                }
                double k = kernel_value_f64<KID>(d2);
                if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE) {
                    if (j0 + j == jz) k = 0.0;
                }
                if constexpr (CAUSAL) {
                    if (j0 + j > row_offset + row) k = 0.0;
                }
                ksum += k;
#pragma unroll
                for (int e = 0; e < EC; ++e) acc[e] = fma(k, sb[j * EC + e], acc[e]);
            }
        }
    }
    if (ok) {
#pragma unroll
        for (int e = 0; e < EC; ++e)
            if (e0 + e < E) out[row * E + e0 + e] = normalize ? acc[e] / ksum : acc[e];
    }
}
template <int KID, int EC>
__global__ void __launch_bounds__(F64_THREADS)
kprod_f64_kernel(const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                 double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                 long long row_offset) {
    f64_rows_body<KID, EC, false>(threadIdx.x, x, y, b, out, N, M, D, E, e0, normalize, row_offset);
}
template <int KID, int EC>
__global__ void __launch_bounds__(F64_THREADS)
kprod_f64_causal_kernel(const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                        double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                        long long row_offset) {
    f64_rows_body<KID, EC, true>(threadIdx.x, x, y, b, out, N, M, D, E, e0, normalize, row_offset);
}

// ---- any D (D > 16): tiled version --------------------------------------------------------------------
// The reference's ground truth for every dataset is its float64 brute force (datasets.py:180-195), also for the
// D = 784 and D = 64 configs whose (N, M, D) temporaries it cannot hold; this kernel is the float64 path for those
// (precision="float64" with D > 16, and the chunked truth writer of harness/datasets_ext.py).
// One CTA = 64 target rows x 64 sources per step.  Phase 1: squared distances as sums of squared differences
// (bruteforce.py:53-54), D staged through shared memory in chunks of 16, a 4 x 4 micro-tile per thread, then the kernel
// function -> k tile in shared memory.  Phase 2: out[64 x EC] += k[64 x 64] b[64 x EC] (EC <= 64 signal columns per
// pass), 16 accumulators per thread in registers across all source tiles; row sums of k ride along for normalize_rows.
constexpr int W_T = 64, W_DC = 16, W_EC = 64, W_THREADS = 256;

template <int KID, bool CAUSAL>
__device__ __forceinline__ void f64_wide_body(const uint32_t tid_, const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                                              double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                                              long long row_offset) {
    extern __shared__ double wide_smem[];
    double (*xs)[W_DC + 1] = reinterpret_cast<double (*)[W_DC + 1]>(wide_smem);
    double (*ys)[W_DC + 1] = xs + W_T;
    double (*ks)[W_T + 1] = reinterpret_cast<double (*)[W_T + 1]>(wide_smem + 2 * W_T * (W_DC + 1));
    double (*bs)[W_EC] = reinterpret_cast<double (*)[W_EC]>(wide_smem + 2 * W_T * (W_DC + 1) + W_T * (W_T + 1));
    const int tid = tid_, tx = tid & 15, ty = tid >> 4;
    const long long row0 = blockIdx.x * static_cast<long long>(W_T);
    const int ec = min(W_EC, E - e0);
    const int pr = tid >> 2, pc = tid & 3;   // phase 2: row pr, signal columns pc, pc + 4, ...
    double acc[W_EC / 4], ksum = 0.0;
#pragma unroll
    for (int q = 0; q < W_EC / 4; ++q) acc[q] = 0.0;

    long long m_end = M;
    if constexpr (CAUSAL) m_end = min(M, row_offset + min(N, row0 + W_T));
    for (long long j0 = 0; j0 < m_end; j0 += W_T) {
        double d2[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) d2[i][j] = 0.0;
        for (int dc = 0; dc < D; dc += W_DC) {
            __syncthreads();
            for (int i = tid; i < W_T * W_DC; i += W_THREADS) {
                const int r = i / W_DC, d = i % W_DC;
                xs[r][d] = (row0 + r < N && dc + d < D) ? x[(row0 + r) * D + dc + d] : 0.0;
                ys[r][d] = (j0 + r < M && dc + d < D) ? y[(j0 + r) * D + dc + d] : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int d = 0; d < W_DC; ++d) {
                double xv[4], yv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) xv[i] = xs[ty + 16 * i][d];
#pragma unroll
                for (int j = 0; j < 4; ++j) yv[j] = ys[tx + 16 * j][d];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) d2[i][j] = pair_term<KID>(xv[i], yv[j], d2[i][j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const long long src = j0 + tx + 16 * j, row = row0 + ty + 16 * i;
                double k = (src < M && row < N) ? kernel_value_f64<KID>(d2[i][j]) : 0.0;
                if constexpr (KID == KMB_KERNEL_INVERSE_DISTANCE) {
                    if (src == (row_offset + row) % (M + 1)) k = 0.0;   // bruteforce.py:12-14
                }
                if constexpr (CAUSAL) {
                    if (src > row_offset + row) k = 0.0;
                }
                ks[ty + 16 * i][tx + 16 * j] = k;
            }
        for (int i = tid; i < W_T * W_EC; i += W_THREADS) {
            const int j = i / W_EC, e = i % W_EC;
            bs[j][e] = (j0 + j < M && e < ec) ? (b ? b[(j0 + j) * E + e0 + e] : 1.0) : 0.0;
        }
        __syncthreads();
        for (int j = 0; j < W_T; ++j) {
            const double k = ks[pr][j];
            if (pc == 0) ksum += k;
#pragma unroll
            for (int q = 0; q < W_EC / 4; ++q) acc[q] = fma(k, bs[j][pc + 4 * q], acc[q]);
        }
    }
    const double total = __shfl_sync(0xffffffffu, ksum, (tid & 31) & ~3);   // the row's sum lives in its pc == 0 lane
    if (row0 + pr < N) {
#pragma unroll
        for (int q = 0; q < W_EC / 4; ++q) {
            const int e = pc + 4 * q;
            if (e < ec) out[(row0 + pr) * E + e0 + e] = normalize ? acc[q] / total : acc[q];
        }
    }
}
template <int KID>
__global__ void __launch_bounds__(W_THREADS)
kprod_f64_wide_kernel(const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                      double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                      long long row_offset) {
    f64_wide_body<KID, false>(threadIdx.x, x, y, b, out, N, M, D, E, e0, normalize, row_offset);
}
template <int KID>
__global__ void __launch_bounds__(W_THREADS)
kprod_f64_wide_causal_kernel(const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ b,
                             double* __restrict__ out, long long N, long long M, int D, int E, int e0, int normalize,
                             long long row_offset) {
    f64_wide_body<KID, true>(threadIdx.x, x, y, b, out, N, M, D, E, e0, normalize, row_offset);
}

template <int KID>
int launch_f64_wide(const double* x, const double* y, const double* b, double* out, int64_t N, int64_t M, int D, int E, int flags,
                    int64_t row_offset, cudaStream_t stream) {
    const int normalize = (flags & KMB_FLAG_NORMALIZE_ROWS) ? 1 : 0;
    const unsigned grid = static_cast<unsigned>((N + W_T - 1) / W_T);
    constexpr int smem = sizeof(double) * (2 * W_T * (W_DC + 1) + W_T * (W_T + 1) + W_T * W_EC);
    auto fn = (flags & KMB_FLAG_CAUSAL) ? &kprod_f64_wide_causal_kernel<KID> : &kprod_f64_wide_kernel<KID>;
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(fn), smem)) return rc;
    for (int e0 = 0; e0 < E; e0 += W_EC) {
        fn<<<grid, W_THREADS, smem, stream>>>(x, y, b, out, N, M, D, E, e0, normalize, row_offset);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
    }
    return KMB_OK;
}

__global__ void fill_f64_kernel(double* out, long long n, double v) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < n) out[i] = v;
}

template <int KID>
int launch_f64(const double* x, const double* y, const double* b, double* out, int64_t N, int64_t M, int D, int E, int flags,
               int64_t row_offset, cudaStream_t stream) {
    const int normalize = (flags & KMB_FLAG_NORMALIZE_ROWS) ? 1 : 0;
    const unsigned grid = static_cast<unsigned>((N + F64_THREADS - 1) / F64_THREADS);
    for (int e0 = 0; e0 < E; e0 += F64_MAX_E) {
        const int ec = std::min(F64_MAX_E, E - e0);
        const size_t smem = sizeof(double) * F64_SB * (D + (ec <= 1 ? 1 : ec <= 2 ? 2 : ec <= 4 ? 4 : 8));
        const bool causal = flags & KMB_FLAG_CAUSAL;
        auto fn = ec <= 1 ? (causal ? &kprod_f64_causal_kernel<KID, 1> : &kprod_f64_kernel<KID, 1>)
                : ec <= 2 ? (causal ? &kprod_f64_causal_kernel<KID, 2> : &kprod_f64_kernel<KID, 2>)
                : ec <= 4 ? (causal ? &kprod_f64_causal_kernel<KID, 4> : &kprod_f64_kernel<KID, 4>)
                          : (causal ? &kprod_f64_causal_kernel<KID, 8> : &kprod_f64_kernel<KID, 8>);
        fn<<<grid, F64_THREADS, smem, stream>>>(x, y, b, out, N, M, D, E, e0, normalize, row_offset);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
    }
    return KMB_OK;
}

// out[i][j] = k(x_i, y_j): an explicit (n x m) block of the kernel matrix, m small (the landmark columns of the
// Nystrom preconditioner, solver.py).  kernel_matrix(...) of bruteforce.py:25-58 restricted to m source points.
template <int KID>
__global__ void __launch_bounds__(256) kernel_block_f64_kernel(const double* __restrict__ x, const double* __restrict__ y,
                                                                double* __restrict__ out, long long n, long long m, int D) {
    const long long j = blockIdx.y * 32ll + threadIdx.x;
    const long long i = blockIdx.x * 8ll + threadIdx.y;
    if (i >= n || j >= m) return;
    double d2 = 0.0;
    for (int d = 0; d < D; ++d) d2 = pair_term<KID>(x[i * D + d], y[j * D + d], d2);
    out[i * m + j] = kernel_value_f64<KID>(d2);
}

}  // namespace

int kernel_block_f64(const double* x, const double* y, double* out, int64_t n, int64_t m, int D, int kernel_id, cudaStream_t stream) {
    if ((m + 31) / 32 > 65535 || (n + 7) / 8 > 2147483647ll) return set_error(KMB_ERR_UNSUPPORTED, "block too large (n=%lld, m=%lld)", (long long)n, (long long)m);
    const dim3 block(32, 8), grid(static_cast<unsigned>((n + 7) / 8), static_cast<unsigned>((m + 31) / 32));
    switch (kernel_id) {
        case KMB_KERNEL_GAUSSIAN: kernel_block_f64_kernel<KMB_KERNEL_GAUSSIAN><<<grid, block, 0, stream>>>(x, y, out, n, m, D); break;
        case KMB_KERNEL_ABSOLUTE_EXPONENTIAL: kernel_block_f64_kernel<KMB_KERNEL_ABSOLUTE_EXPONENTIAL><<<grid, block, 0, stream>>>(x, y, out, n, m, D); break;
        case KMB_KERNEL_DOT_EXPONENTIAL: kernel_block_f64_kernel<KMB_KERNEL_DOT_EXPONENTIAL><<<grid, block, 0, stream>>>(x, y, out, n, m, D); break;
        default: kernel_block_f64_kernel<KMB_KERNEL_INVERSE_DISTANCE><<<grid, block, 0, stream>>>(x, y, out, n, m, D); break;
    }
    KMB_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return KMB_OK;
}

int product_f64(const double* x, const double* y, const double* b, double* out, int64_t N, int64_t M, int D, int E,
                int kernel_id, int flags, int64_t row_offset, cudaStream_t stream) {
    if ((flags & KMB_FLAG_NORMALIZE_ROWS) && (flags & KMB_FLAG_DENSITY)) {   // bruteforce.py:134-138
        fill_f64_kernel<<<static_cast<unsigned>((N + 255) / 256), 256, 0, stream>>>(out, N, 1.0);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
        return KMB_OK;
    }
    const double* sig = (flags & KMB_FLAG_DENSITY) ? nullptr : b;
    if (D > F64_MAX_D) {
        switch (kernel_id) {
            case KMB_KERNEL_GAUSSIAN: return launch_f64_wide<KMB_KERNEL_GAUSSIAN>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
            case KMB_KERNEL_ABSOLUTE_EXPONENTIAL: return launch_f64_wide<KMB_KERNEL_ABSOLUTE_EXPONENTIAL>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
            case KMB_KERNEL_DOT_EXPONENTIAL: return launch_f64_wide<KMB_KERNEL_DOT_EXPONENTIAL>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
            default: return launch_f64_wide<KMB_KERNEL_INVERSE_DISTANCE>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
        }
    }
    switch (kernel_id) {
        case KMB_KERNEL_GAUSSIAN: return launch_f64<KMB_KERNEL_GAUSSIAN>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
        case KMB_KERNEL_ABSOLUTE_EXPONENTIAL: return launch_f64<KMB_KERNEL_ABSOLUTE_EXPONENTIAL>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
        case KMB_KERNEL_DOT_EXPONENTIAL: return launch_f64<KMB_KERNEL_DOT_EXPONENTIAL>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
        default: return launch_f64<KMB_KERNEL_INVERSE_DISTANCE>(x, y, sig, out, N, M, D, E, flags, row_offset, stream);
    }
}

}  // namespace kmb
