// tcgen05.mma pacing micro-benchmark: cycles per MMA instruction for the shapes the tensor kernels use.
// One CTA per SM issues a long chain of M = 128 MMAs into one TMEM accumulator (kind::tf32 or kind::f16,
// A from shared memory (SS) or from tensor memory (TS), N = 64 / 128 / 256, SWIZZLE_128B K-major operands
// walked in four 32-byte K steps per 128-byte atom exactly as the kernels walk them) and times the chain with
// clock64.  The math floor is 128 N / 256 cycles per instruction (B300_MICROARCH.md, "tcgen05 floor"); what
// is measured above it is the operand fetch.  Prints one JSON object per configuration.
//   pattern 0: (A0, B0) repeated          pattern 1: the 3-term split order (A1,B0), (A0,B1), (A0,B0)
#include <cstdio>
#include <cstdlib>

#include "../kernel_matrix_benchmarks_b200/csrc/tensor_common.cuh"

using namespace kmb;
using namespace kmb::tc;

#define CHECK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

constexpr int A_BYTES = 128 * 128;    // 128 rows x one 128-byte swizzle atom
constexpr int B_BYTES = 256 * 128;
constexpr int SMEM = 1024 + 2 * A_BYTES + 2 * B_BYTES + 64;

// traffic: 0 = none; 1 = 4 warps stream tcgen05.ld (x32) from TMEM while the chain runs; 2 = tcgen05.ld + tcgen05.st;
// 3 = 16 warps of tcgen05.ld + tcgen05.st (the epilogue of kprod_tensor_pv16)
template <int KIND, bool TS>
__global__ void __launch_bounds__(544, 1) umma_bench(int N, int reps, int pattern, int traffic, int n_acc, long long* cycles) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
    unsigned char* a0 = smem;
    unsigned char* a1 = a0 + A_BYTES;
    unsigned char* b0 = a1 + A_BYTES;
    unsigned char* b1 = b0 + B_BYTES;
    uint64_t* bar = reinterpret_cast<uint64_t*>(b1 + B_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
    volatile int* stop = reinterpret_cast<volatile int*>(tmem_slot + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) *stop = 0;
    // operand bits: finite values of the kind's element type
    for (int i = tid; i < (2 * A_BYTES + 2 * B_BYTES) / 4; i += blockDim.x) {
        const uint32_t h = (i * 2654435761u) >> 9;
        reinterpret_cast<uint32_t*>(smem)[i] = KIND == 0 ? (0x3f000000u | (h & 0x7fe000u)) : (0x38003800u | (h & 0x03ff03ffu));
    }
    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t idesc = (1u << 4) | (KIND == 0 ? ((2u << 7) | (2u << 10)) : 0u) | (static_cast<uint32_t>(N >> 3) << 17) | (8u << 24);
    if (warp == 0) {
        const long long t0 = clock64();
        for (int r = 0; r < reps; ++r) {
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // n_acc < 0: descriptors rebuilt from a run-time slot offset every iteration, as a kernel with a
                    // shared-memory ring does (the offset is zero, but ptxas cannot know)
                    const int so = n_acc < 0 ? (r % 5) * (n_acc + 1) : 0;
                    const uint64_t da0 = umma_desc_sw128(a0 + so, k * 32), da1 = umma_desc_sw128(a1 + so, k * 32);
                    const uint64_t db0 = umma_desc_sw128(b0 + so, k * 32), db1 = umma_desc_sw128(b1 + so, k * 32);
                    const uint32_t ta0 = tmem + 256 + k * 8, ta1 = tmem + 320 + k * 8;
                    const uint32_t dd = tmem + (n_acc > 1 ? ((r + k) & (n_acc - 1)) * 64 : 0);   // n_acc accumulators in turn
                    auto mma = [&](uint64_t da, uint32_t ta, uint64_t db, uint32_t acc) {
                        if constexpr (KIND == 0) { if constexpr (TS) umma_tf32_ts(dd, ta, db, idesc, acc); else umma_tf32(dd, da, db, idesc, acc); }
                        else { if constexpr (TS) umma_f16_ts(dd, ta, db, idesc, acc); else umma_f16(dd, da, db, idesc, acc); }
                    };
                    if (pattern == 0) {
                        mma(da0, ta0, db0, (r | k) != 0);
                    } else {
                        mma(da1, ta1, db0, (r | k) != 0);
                        mma(da0, ta0, db1, 1);
                        mma(da0, ta0, db0, 1);
                    }
                }
            }
            __syncwarp();
        }
        if (elect_one()) umma_commit(bar);
        __syncwarp();
        mbar_wait(bar, 0);
        const long long t1 = clock64();
        if (tid == 0) cycles[blockIdx.x] = t1 - t0;
        *stop = 1;
    } else if (traffic == 4) {
        // 16 warps of arithmetic (FFMA2 + MUFU, no TMEM access): do they starve the issuing warp of issue slots?
        float2 acc = make_float2(threadIdx.x * 1e-3f, 1.f);
        float m = 0.5f;
        while (!*stop) {
#pragma unroll
            for (int i = 0; i < 64; ++i) {
                acc = __ffma2_rn(acc, make_float2(0.999f, 1.001f), make_float2(m, m));
                if ((i & 3) == 0) m = ex2_approx(m - 1.f);
            }
        }
        if (acc.x == 123.f) cycles[0] = 0;
    } else if (traffic > 0 && (warp <= 4 || traffic == 3)) {
        // TMEM traffic beside the MMA chain: columns [384, 416) + 32 (warp / 4) of this warp's lane quarter
        const uint32_t addr = tmem + 384 + 32 * ((warp - 1) >> 2) + (static_cast<uint32_t>((warp & 3) * 32) << 16);
        float v[32];
        while (!*stop) {
            tmem_ld_32x32(addr, v);
            if (traffic >= 2) {
                tmem_st_32x32(addr, v);
                tmem_st_wait();
            }
        }
        if (v[0] == 123.f) cycles[0] = 0;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int KIND, bool TS>
int run(int N, int pattern, long long* d_cycles, int sms, int traffic = 0, int n_acc = 1) {
    auto fn = umma_bench<KIND, TS>;
    CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    const int reps = 1024;
    const int per_rep = 4 * (pattern == 0 ? 1 : 3);
    fn<<<sms, 544, SMEM>>>(N, 64, pattern, traffic, n_acc, d_cycles);   // warm-up
    fn<<<sms, 544, SMEM>>>(N, reps, pattern, traffic, n_acc, d_cycles);
    CHECK(cudaDeviceSynchronize());
    long long* h = static_cast<long long*>(malloc(sizeof(long long) * sms));
    CHECK(cudaMemcpy(h, d_cycles, sizeof(long long) * sms, cudaMemcpyDeviceToHost));
    long long mx = 0, mn = 1ll << 62;
    for (int i = 0; i < sms; ++i) { mx = h[i] > mx ? h[i] : mx; mn = h[i] < mn ? h[i] : mn; }
    free(h);
    const double n_mma = static_cast<double>(reps) * per_rep;
    const int a_bytes = TS ? 0 : 128 * 32, b_bytes = N * 32;
    printf("{\"kind\": \"%s\", \"a\": \"%s\", \"M\": 128, \"N\": %d, \"pattern\": %d, \"tmem_traffic\": %d, \"accumulators\": %d, \"cycles_per_mma_min\": %.1f, \"cycles_per_mma_max\": %.1f, "
           "\"math_floor\": %d, \"smem_operand_bytes\": %d}\n",
           KIND == 0 ? "tf32" : "f16", TS ? "tmem" : "smem", N, pattern, traffic, n_acc, mn / n_mma, mx / n_mma, N / 2, a_bytes + b_bytes);
    return 0;
}

int main() {
    int sms = 0;
    CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    long long* d_cycles;
    CHECK(cudaMalloc(&d_cycles, sizeof(long long) * sms));
    const int ns[3] = {64, 128, 256};
    for (int pattern = 0; pattern < 2; ++pattern)
        for (int n : ns) {
            if (run<0, false>(n, pattern, d_cycles, sms)) return 1;
            if (run<0, true>(n, pattern, d_cycles, sms)) return 1;
            if (run<1, false>(n, pattern, d_cycles, sms)) return 1;
            if (run<1, true>(n, pattern, d_cycles, sms)) return 1;
        }
    // the shapes of kprod_tensor_pv16 beside TMEM traffic from other warps, and with 4 accumulators in turn
    for (int traffic = 0; traffic <= 4; ++traffic) {
        if (run<1, true>(64, 1, d_cycles, sms, traffic, 1)) return 1;
        if (run<1, true>(64, 1, d_cycles, sms, traffic, 4)) return 1;
        if (run<1, true>(64, 1, d_cycles, sms, traffic, -1)) return 1;
        if (run<1, false>(128, 1, d_cycles, sms, traffic, 1)) return 1;
        if (run<1, false>(128, 1, d_cycles, sms, traffic, -1)) return 1;
    }
    return 0;
}
