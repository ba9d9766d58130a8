/* vvb_tu_inv_generic.cu -- stft_inverse_kernel instantiations: slot overlap-add for hops without a marching / pair
 * kernel, and windowed frames without overlap-add (vv_dsp_stft_reconstruct, C2R plans). */
#include "vvb_rt.cuh"

namespace vvb {

template <class C, bool OLA> static int launch_inverse_t(InvArgs a, long long batch, int sms, void* stream)
{
    constexpr int G = Teams<C>::G;
    static OccCache occ;
    auto kern = stft_inverse_kernel<C, G, OLA>;
    const size_t smem = smem_inv<C>(a.hop, OLA);
    const int per_sm = occ.get(kern, C::T * G, smem);
    if (per_sm == 0) return rt_fail(4, "stft_inverse_kernel", "does not fit on this device");
    long long items;
    if (OLA) {
        /* split every signal into chunks of frames so the persistent grid has >= ~4 items per CTA;
         * each chunk re-synthesises up to K-1 halo frames, so chunks are kept long (>= 16 rounds) */
        const long long cap = (long long)per_sm * sms;
        long long want = (4 * cap + batch - 1) / batch;                 /* chunks per signal wanted */
        long long max_chunks = a.frames / (16 * G);
        if (max_chunks < 1) max_chunks = 1;
        if (want > max_chunks) want = max_chunks;
        if (want < 1) want = 1;
        long long cf = (a.frames + want - 1) / want;
        cf = (cf + G - 1) / G * G;                                      /* whole rounds */
        a.chunk_frames = (int)cf;
        a.chunks_per_signal = (int)((a.frames + cf - 1) / cf);
        items = batch * a.chunks_per_signal;
        if (getenv("VVB_ROUTE_DEBUG"))
            fprintf(stderr, "vvb: stft_inverse_kernel overlap-add: chunks_per_signal %d, chunk_frames %d\n", a.chunks_per_signal, a.chunk_frames);
    } else {
        items = (a.frames + G - 1) / G;
    }
    if (items > 0x7fffffffLL) return rt_fail(2, "vvb_stft_inverse", "too many work items");
    a.num_items = (int)items;
    if (items == 0) return 0;
    VVB_LAUNCH(kern, persistent_grid(items, per_sm, sms), C::T * G, smem, stream, a);
    return 0;
}

template <bool OLA> static int dispatch_inverse(int m, const InvArgs& a, long long batch, int sms, void* stream)
{
    switch (m) {
    case 128: return launch_inverse_t<Cfg128, OLA>(a, batch, sms, stream);
    case 160: return launch_inverse_t<Cfg160, OLA>(a, batch, sms, stream);
    case 200: return launch_inverse_t<Cfg200, OLA>(a, batch, sms, stream);
    case 240: return launch_inverse_t<Cfg240, OLA>(a, batch, sms, stream);
    case 320: return launch_inverse_t<Cfg320, OLA>(a, batch, sms, stream);
    case 256: return launch_inverse_t<Cfg256, OLA>(a, batch, sms, stream);
    case 512: return launch_inverse_t<Cfg512, OLA>(a, batch, sms, stream);
    case 1024: return launch_inverse_t<Cfg1024, OLA>(a, batch, sms, stream);
    case 2048: return launch_inverse_t<Cfg2048, OLA>(a, batch, sms, stream);
    case 4096: return launch_inverse_t<Cfg4096, OLA>(a, batch, sms, stream);
    default: return rt_fail(6, "vvb_stft_inverse", "no Stockham kernel for this size");
    }
}

int tu_inv_generic(int m, bool ola, const InvArgs& a, long long batch, int sms, void* stream)
{
    return ola ? dispatch_inverse<true>(m, a, batch, sms, stream) : dispatch_inverse<false>(m, a, batch, sms, stream);
}

}  // namespace vvb
