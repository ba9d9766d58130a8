/* vvb_tu_fir.cu -- fir_ols_kernel instantiations (overlap-save FIR on the M-point register FFT, M = 128 ... 8192) and the
 * partition padding kernel of the filter spectra. */
#include "vvb_rt.cuh"
#include "vvb_fir_kernels.cuh"

namespace vvb {

__global__ void fir_pad_kernel(const FirPadArgs a)
{
    const float inv_m = 1.0f / (float)a.m;          /* a power of two: the scaling is exact */
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < a.total; idx += (long long)gridDim.x * blockDim.x) {
        const long long row = idx / a.m;
        const int i = (int)(idx - row * a.m);
        const long long f = row / a.parts;
        const long long j = (row - f * a.parts) * a.lp + i;
        float v = 0.0f;
        if (i < a.lp && j < a.taps) v = __ldg(a.h + f * a.h_pitch + j) * inv_m;
        a.out[idx] = make_float2(v, 0.0f);
    }
}

template <class C, bool ACCUM> static int launch_fir(const FirArgs& a, int sms, void* stream)
{
    constexpr int G = Teams<C>::G;
    static OccCache occ;
    auto kern = fir_ols_kernel<C, G, ACCUM>;
    const size_t smem = smem_c2c<C>();
    const int per_sm = occ.get(kern, C::T * G, smem);
    if (per_sm == 0) return rt_fail(4, "fir_ols_kernel", "does not fit on this device");
    /* named in full so that VVB_ROUTE_DEBUG prints the kernel as well as its configuration */
    VVB_LAUNCH((fir_ols_kernel<C, G, ACCUM>), persistent_grid((a.count + G - 1) / G, per_sm, sms), C::T * G, smem, stream, a);
    return 0;
}
template <class C> static int launch_fir_pass(const FirArgs& a, bool accum, int sms, void* stream)
{
    return accum ? launch_fir<C, true>(a, sms, stream) : launch_fir<C, false>(a, sms, stream);
}

int tu_fir(int m, const FirArgs& a, bool accum, int sms, void* stream)
{
    switch (m) {
    case 128: return launch_fir_pass<Cfg128>(a, accum, sms, stream);
    case 256: return launch_fir_pass<Cfg256>(a, accum, sms, stream);
    case 512: return launch_fir_pass<Cfg512>(a, accum, sms, stream);
    case 1024: return launch_fir_pass<Cfg1024>(a, accum, sms, stream);
    case 2048: return launch_fir_pass<Cfg2048>(a, accum, sms, stream);
    case 4096: return launch_fir_pass<Cfg4096>(a, accum, sms, stream);
    case 8192: return launch_fir_pass<Cfg8192>(a, accum, sms, stream);
    default: return rt_fail(6, "fir_ols_kernel", "no Stockham kernel for this size");
    }
}

int tu_fir_pad(const FirPadArgs& a, int sms, void* stream)
{
    VVB_LAUNCH(fir_pad_kernel, persistent_grid((a.total + 255) / 256, 8, sms), 256, 0, stream, a);
    return 0;
}

}  // namespace vvb
