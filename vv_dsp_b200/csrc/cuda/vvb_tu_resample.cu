/* vvb_tu_resample.cu -- resample_poly_kernel instantiations (polyphase FIR resampling, vvb_resample_kernels.cuh): runs of
 * RS_RUN outputs, the input span of a tile staged in shared memory or read through L1. */
#include "vvb_rt.cuh"
#include "vvb_resample_kernels.cuh"

namespace vvb {

template <int R, bool SMEM> static int launch_resample(const ResampleArgs& a, int sms, void* stream)
{
    static OccCache occ;
    auto kern = resample_poly_kernel<R, SMEM>;
    const size_t smem = SMEM ? resample_smem_bytes(a.span) : 0;
    const int per_sm = occ.get(kern, RS_THREADS, smem);
    if (per_sm == 0) return rt_fail(4, "resample_poly_kernel", "does not fit on this device");
    /* named in full so that VVB_ROUTE_DEBUG prints the kernel as well as its configuration */
    VVB_LAUNCH((resample_poly_kernel<R, SMEM>), persistent_grid(a.count, per_sm, sms), RS_THREADS, smem, stream, a);
    return 0;
}

int tu_resample(const ResampleArgs& a, int sms, void* stream)
{
    return a.span > 0 ? launch_resample<RS_RUN, true>(a, sms, stream) : launch_resample<RS_RUN, false>(a, sms, stream);
}

}  // namespace vvb
