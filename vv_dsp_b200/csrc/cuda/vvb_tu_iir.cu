/* vvb_tu_iir.cu -- the IIR second-order-section kernels (vvb_iir_kernels.cuh): iir_tile_kernel for the segment end states
 * (launch A, STATES) and the filtered output (launch C), iir_chain_kernel for the chain of segment states (launch B). */
#include "vvb_rt.cuh"
#include "vvb_iir_kernels.cuh"

namespace vvb {

template <int L, bool STATES> static int launch_iir_tile(const IirArgs& a, int sms, void* stream)
{
    static OccCache occ;
    auto kern = iir_tile_kernel<L, STATES>;
    const size_t smem = iir_smem_bytes<L>(a.sections);
    const int per_sm = occ.get(kern, IIR_THREADS, smem);
    if (per_sm == 0) return rt_fail(4, "iir_tile_kernel", "does not fit on this device");
    /* named in full so that VVB_ROUTE_DEBUG prints the kernel as well as its configuration */
    VVB_LAUNCH((iir_tile_kernel<L, STATES>), persistent_grid(a.count, per_sm, sms), IIR_THREADS, smem, stream, a);
    return 0;
}

template <int THREADS> static int launch_iir_chain(const IirArgs& a, int sms, void* stream)
{
    static OccCache occ;
    auto kern = iir_chain_kernel<THREADS>;
    const size_t smem = sizeof(float) * THREADS;
    const int per_sm = occ.get(kern, THREADS, smem);
    if (per_sm == 0) return rt_fail(4, "iir_chain_kernel", "does not fit on this device");
    VVB_LAUNCH((iir_chain_kernel<THREADS>), persistent_grid(a.count, per_sm, sms), THREADS, smem, stream, a);
    return 0;
}

int tu_iir(char pass, const IirArgs& a, int sms, void* stream)
{
    if (pass == 'A') return launch_iir_tile<VVB_IIR_RUN, true>(a, sms, stream);
    if (pass == 'B') return launch_iir_chain<IIR_CHAIN_THREADS>(a, sms, stream);
    return launch_iir_tile<VVB_IIR_RUN, false>(a, sms, stream);
}

}  // namespace vvb
