// Tensor-core path (D > 16): squared distances through |x|^2 + |y|^2 - 2 x.y with the dot products on tcgen05
// (FP32 accumulators in TMEM) and a three-term hi/lo split of the operands for FP32-class accuracy: FP16 planes of
// power-of-two scaled data (KMB_PATH_TENSOR_3XF16, the default) or TF32 planes (KMB_PATH_TENSOR_3XTF32).
// Replaces kernel_matrix(..., fast_sqdists=True) + K @ b of the reference
// (/root/reference/kernel_matrix_benchmarks/algorithms/bruteforce.py:36-49, 18-22, 130-153).
#pragma once
#include "kmb_common.cuh"

namespace kmb {

// elt: 0 = TF32 hi/lo operands (KMB_PATH_TENSOR_3XTF32), 1 = FP16 hi/lo operands (KMB_PATH_TENSOR_3XF16),
//      2 = the FP16 hi operands alone, one MMA term (KMB_PATH_TENSOR_1XF16)
int tensor_workspace_bytes(int64_t N, int64_t M, int D, int E, int kid, int flags, int elt, size_t* bytes);

// Enqueue the whole tensor-path product on `stream` (prepass + main kernel per signal chunk).
// ev0/ev1: optional events recorded around the last main kernel.
int tensor_product(const float* x, const float* y, const float* b, float* out, int64_t N, int64_t M, int D, int E,
                   int kid, int flags, int elt, int64_t row_offset, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1, bool prepared = false);

// Points-only prepass of the FP16-plane kernels into the head of the workspace (E-independent layout; see
// kmb_product_prepare_f32).  tensor_product skips it when `prepared` is set.  No-op for TF32 planes.
int tensor_prepare(const float* x, const float* y, int64_t N, int64_t M, int D, int kid, int elt, void* workspace,
                   size_t workspace_bytes, cudaStream_t stream);

// The wave schedule of the tensor kernels for a (row tiles x source blocks) problem on `grid` CTAs (or clusters):
// out = {R, C, W, R_last, C_last, slots_per_wave, partial_slots}.  Host logic only (tests/test_abi_cpu.py).
void tensor_plan_waves_debug(long long n_tiles, long long nsb, int grid, size_t row_tile_bytes, long long out[7]);

// What tensor_product launches for this shape on `sms` SMs: out = {KMB_FAMILY_*, signal columns per pass, passes, row
// tiles}.  Host logic only, the same decisions as tensor_product (kmb_debug_product_plan).
void tensor_plan_debug(int64_t N, int D, int E, int kid, int elt, int sms, long long out[4]);

// What the P.B kernel (kprod_tensor_pv / kprod_tensor_pv16) launches for this shape on a device of `sms` SMs with
// `smem_optin` bytes of opt-in shared memory per block: out = the KMB_PV_PLAN_FIELDS of kmb_debug_pv_plan.  Host logic
// only, the launchers' own plan functions; for an E <= 4 kernel only the family is filled.
int tensor_pv_plan_query(int64_t N, int64_t M, int D, int E, int kid, int elt, int sms, int smem_optin, long long* out);

}  // namespace kmb
