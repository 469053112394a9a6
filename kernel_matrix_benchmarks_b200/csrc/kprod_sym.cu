// Instantiations and launchers of the symmetric (same_points) product, D <= 3, E = 1: the Gaussian product
// form plus the difference form of every kernel of bruteforce.py:18-22.
#include "kprod_sym.cuh"

namespace kmb {

namespace {

// Production shape (tools/tune_sym.cu on B200, profiles/r1_tune_sym.log): 512 consumer threads x 8 rows,
// one CTA per SM, butterflies of 16 sources, every exponential on the MUFU pipe -- 13.1 kernel
// evaluations/clk/SM = 26 pairs/clk/SM at N = 10^6 (4 rows x 2 CTAs/SM: 12.5; with 1/16 of the
// exponentials on the FMA pipe: 12.0 -- here the FMA pipe and the issue slots are the scarce resource).
template <int DP, int KID, int FORM>
using Sym = SymCfg<DP, KID, FORM, 0, 1, 16, 512, 8, 4>;
using SymRef = Sym<3, KMB_KERNEL_GAUSSIAN, 1>;   // geometry (tile rows, block sources) is the same for all

template <class C>
int sym_launch_of(SymParams P, cudaStream_t stream) {
    static_assert(C::TILE_ROWS == SymRef::TILE_ROWS && C::SB == SymRef::SB, "one geometry for every instantiation");
    const long long units = P.unit_end - P.unit_begin;
    if (units > 0) {
        const int grid = static_cast<int>(std::min<long long>(P.grid, units));
        P.grid = grid;
        if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(&kprod_sym_kernel<C>), C::SMEM_BYTES)) return rc;
        kprod_sym_kernel<C><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(P);
        KMB_CUDA_CHECK(cudaGetLastError());
        count_launch();
    }
    sym_combine_kernel<C><<<static_cast<unsigned>((P.N + 255) / 256), 256, 0, stream>>>(P);
    KMB_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return KMB_OK;
}

template <int KID, int FORM>
int sym_launch_dp(int D, const SymParams& P, cudaStream_t stream) {
    return D <= 2 ? sym_launch_of<Sym<2, KID, FORM>>(P, stream) : sym_launch_of<Sym<3, KID, FORM>>(P, stream);
}

}  // namespace

bool sym_supported(int D) { return D >= 1 && D <= 3; }
int sym_tile_rows() { return SymRef::TILE_ROWS; }
int sym_block_sources() { return SymRef::SB; }

// one persistent CTA per SM (544 threads, ~110 registers)
int sym_grid(int sms, int* grid) {
    int per_sm = 0;
    if (int rc = resident_ctas(reinterpret_cast<const void*>(&kprod_sym_kernel<SymRef>), SymRef::THREADS, SymRef::SMEM_BYTES, &per_sm)) return rc;
    *grid = sms;
    return KMB_OK;
}

void sym_geometry(long long n_tiles, long long nsb, long long total_ctas, SymGeom* g) { sym_build_geom<SymRef::TB>(n_tiles, nsb, total_ctas, g); }
long long sym_cta_strip_width(long long nsb, long long total_ctas) { return sym_cta_strip_tiles<SymRef::TB>(nsb, total_ctas) * SymRef::TB; }
SymSeg sym_segment_of(const SymGeom& g, long long u) { return sym_seg_of<SymRef::TB>(g, u); }

// the main kernel over P.unit_begin .. P.unit_end on P.grid CTAs, then the combine kernel.
// form 1: Gaussian product form; form 0: difference form of `kernel_id`.  Each returns at once on the device
// when DirectStats::use_product selects the other form.
int sym_launch(int D, int kernel_id, int form, const SymParams& P, cudaStream_t stream) {
    if (form == 1) return sym_launch_dp<KMB_KERNEL_GAUSSIAN, 1>(D, P, stream);
    switch (kernel_id) {
        case KMB_KERNEL_GAUSSIAN: return sym_launch_dp<KMB_KERNEL_GAUSSIAN, 0>(D, P, stream);
        case KMB_KERNEL_ABSOLUTE_EXPONENTIAL: return sym_launch_dp<KMB_KERNEL_ABSOLUTE_EXPONENTIAL, 0>(D, P, stream);
        case KMB_KERNEL_INVERSE_DISTANCE: return sym_launch_dp<KMB_KERNEL_INVERSE_DISTANCE, 0>(D, P, stream);
    }
    return set_error(KMB_ERR_UNSUPPORTED, "unknown kernel id %d", kernel_id);
}

}  // namespace kmb
