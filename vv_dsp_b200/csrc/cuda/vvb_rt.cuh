/*
 * vvb_rt.cuh -- what the CUDA translation units of the library share: error plumbing, the launch
 * macro, per-device occupancy caching, the kernel configurations and the per-family launch entry
 * points.  One family of kernel instantiations per translation unit (vvb_tu_*.cu) so that they
 * compile in parallel and every hot kernel is code-generated in isolation; vvb_cuda.cu holds the
 * C-ABI of include/vvb200_cuda.h and dispatches to the families.
 */
#pragma once
#include "vvb_chirp_kernels.cuh"
#include "../../../include/vvb200_cuda.h"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace vvb {

/* ------------------------------------------------------------------ error plumbing (vvb_cuda.cu) */
int rt_fail(int code, const char* what, const char* detail);     /* records the text for vvb_last_error() */
extern std::atomic<unsigned long long> g_launches;
int rt_num_sms();                                                 /* SMs of the current device */

enum { VVB_MAX_DEVICES = 32 };

/* VVB_ROUTE_DEBUG=1: one stderr line per launch naming the kernel and the function that launches it.  Inside the
 * per-family launchers (vvb_tu_*.cu, vvb_launch_march.cuh) the function's signature carries the kernel family and its
 * compile-time configuration, so a test can tell which kernel a (fft_size, hop) reached. */
inline void rt_route_debug(const char* kern, const char* where)
{
    if (getenv("VVB_ROUTE_DEBUG")) fprintf(stderr, "vvb: launch %s in %s\n", kern, where);
}

#ifdef VVB_EMU
#define CK(expr) do { if ((expr) != 0) return ::vvb::rt_fail(4, #expr, "emu"); } while (0)
#define VVB_LAUNCH(kern, grid, block, smem, stream, ...) \
    do { ::vvb::g_launches++; ::vvb::rt_route_debug(#kern, __PRETTY_FUNCTION__); \
         vvb_emu::launch(dim3(grid), dim3(block), smem, [&] { kern(__VA_ARGS__); }); } while (0)
inline int rt_device() { return 0; }
template <class K> static int rt_blocks_per_sm(K, int, size_t) { return 1; }
#else
#define CK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return ::vvb::rt_fail(4, #expr, cudaGetErrorString(e_)); } while (0)
#define VVB_LAUNCH(kern, grid, block, smem, stream, ...) \
    do { ::vvb::g_launches++; ::vvb::rt_route_debug(#kern, __PRETTY_FUNCTION__); \
         kern<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__); CK(cudaGetLastError()); } while (0)
inline int rt_device() { int d = 0; return cudaGetDevice(&d) == cudaSuccess ? d : 0; }
/* opt in to the dynamic shared memory the kernel needs (a per-device attribute) and ask how many CTAs fit per SM */
template <class K> static int rt_blocks_per_sm(K kern, int threads, size_t smem)
{
    cudaError_t e1 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int nb = 0;
    cudaError_t e2 = (e1 == cudaSuccess) ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, smem) : e1;
    if (e2 != cudaSuccess || nb == 0) {
        cudaFuncAttributes fa;
        memset(&fa, 0, sizeof(fa));
        cudaFuncGetAttributes(&fa, kern);
        fprintf(stderr, "vvb: kernel does not fit: %s (threads %d, dyn smem %zu, regs %d, static smem %zu, maxThreadsPerBlock %d)\n",
                cudaGetErrorString(e2), threads, smem, fa.numRegs, fa.sharedSizeBytes, fa.maxThreadsPerBlock);
        cudaGetLastError();
        return 0;
    }
    return nb;
}
#endif

/* CTAs per SM of one kernel instantiation, remembered PER DEVICE (the shared-memory opt-in is a per-device
 * function attribute) and per dynamic shared-memory size; safe to call from several host threads. */
struct OccCache {
    std::mutex mu;
    int per_sm[VVB_MAX_DEVICES];
    size_t smem[VVB_MAX_DEVICES];
    OccCache() { for (int i = 0; i < VVB_MAX_DEVICES; ++i) { per_sm[i] = -1; smem[i] = 0; } }
    template <class K> int get(K kern, int threads, size_t bytes)
    {
        const int dev = rt_device() % VVB_MAX_DEVICES;
        std::lock_guard<std::mutex> lock(mu);
        if (per_sm[dev] < 0 || smem[dev] != bytes) { per_sm[dev] = rt_blocks_per_sm(kern, threads, bytes); smem[dev] = bytes; }
        return per_sm[dev];
    }
};

inline int persistent_grid(long long work, int per_sm, int sms)
{
    long long cap = (long long)(per_sm > 0 ? per_sm : 1) * (sms > 0 ? sms : 1);
    long long g = work < cap ? work : cap;
    return (int)(g < 1 ? 1 : g);
}

/* ------------------------------------------------------------------ kernel configurations */
/* M complex points = fft_size/2 for the real transforms */
using Cfg128 = Cfg<128, 16, 16, 8>;
using Cfg256 = Cfg<256, 16, 16, 16>;
using Cfg256m = Cfg<256, 8, 8, 8, 4>;       /* T = 32: whole-warp team for the marching ISTFT (own table blob) */
using Cfg512 = Cfg<512, 32, 32, 16>;
using Cfg512m = Cfg<512, 16, 16, 16, 2>;    /* T = 32 */
using Cfg1024 = Cfg<1024, 32, 32, 32>;
using Cfg2048 = Cfg<2048, 32, 32, 8, 8>;      /* T = 64 (two warps per frame), E = 32 */
using Cfg4096 = Cfg<4096, 32, 32, 16, 8>;     /* T = 128, E = 32 */
using Cfg8192 = Cfg<8192, 32, 32, 16, 16>;    /* T = 256, E = 32: plan-API C2C only */
/* mixed radix (a 5-point leaf under the radix-2 tree): the speech framings fft_size 400 (25 ms at 16 kHz) and 320 (20 ms) */
using Cfg200 = Cfg<200, 50, 10, 10, 2>;       /* T = 4 */
using Cfg160 = Cfg<160, 20, 10, 4, 4>;        /* T = 8 */
/* ... and with a 3-point leaf as well: fft_size 480 (30 ms at 16 kHz) and 640 (40 ms).  (960 = 2 x 12.20.2 with 60 points
 * per thread spills ~200 bytes in every kernel: it stays on the chirp-z path.) */
using Cfg240 = Cfg<240, 60, 12, 20>;          /* T = 4 */
using Cfg320 = Cfg<320, 20, 20, 4, 4>;        /* T = 16 */
template <class C> struct Teams { static constexpr int G = (C::T >= 256) ? 1 : 256 / C::T; };   /* 256 threads per CTA */

template <class C> constexpr size_t smem_fwd() { return sizeof(float) * (2 * C::M + 2 * (C::TW2 + C::TW3 + C::POST + 1) + 2 * Teams<C>::G * C::XBUF); }
template <class C> inline size_t smem_inv(int hop, bool ola) { return smem_fwd<C>() + (ola ? sizeof(float) * 2 * (2 * C::M - hop) : 0); }
template <class C> constexpr size_t smem_c2c() { return sizeof(float) * (2 * (C::TW2 + C::TW3) + 2 * Teams<C>::G * C::XBUF); }

/* team-marching kernels (whole-warp teams: fft_size 2048 / 4096 / 8192, hop = 2*T*S dividing fft_size).
 * G teams per CTA and CTAs per SM chosen per configuration: registers are partitioned per SM sub-partition
 * (16 K each), so 8 warps per SM may use 255 registers per thread but 9..12 warps cap at 168. */
template <class C> struct March;
template <> struct March<Cfg256m> { static constexpr int G = 8, MINB = 3; };    /* 256 thr, <= 80 regs */
template <> struct March<Cfg512m> { static constexpr int G = 8, MINB = 2; };    /* 256 thr, <= 128 regs */
template <> struct March<Cfg1024> { static constexpr int G = 8, MINB = 1; };   /* 256 thr, 232 regs, 1 CTA/SM */
template <> struct March<Cfg2048> { static constexpr int G = 4, MINB = 1; };   /* 256 thr, 1 CTA/SM, up to 255 regs */
template <> struct March<Cfg4096> { static constexpr int G = 2, MINB = 1; };   /* 256 thr, 1 CTA/SM, up to 255 regs */

/* ------------------------------------------------------------------ family entry points (vvb_tu_*.cu) */
/* m = fft_size / 2 of a size with a Stockham kernel; `batch` of a forward launch travels in FwdArgs::num_groups.
 * The marching / pair entries return -1 when (fft_size, hop) has no such kernel. */
int tu_fwd_generic(int m, const FwdArgs& a, int kind, int sms, void* stream);
int tu_fwd_logmel(int m, const FwdArgs& a, int sms, void* stream, bool probe);      /* generic kernel + mel_phase per warp; 6: no such kernel / schedule too long */
int tu_fwd_march_2048(size_t hop, const FwdArgs& a, int kind, int sms, void* stream);
int tu_fwd_march_4096(size_t hop, const FwdArgs& a, int kind, int sms, void* stream);
int tu_fwd_march_8192(size_t hop, const FwdArgs& a, int kind, int sms, void* stream);
int tu_inv_generic(int m, bool ola, const InvArgs& a, long long batch, int sms, void* stream);
int tu_inv_march_small(int nfft, size_t hop, const InvArgs& a, long long batch, int sms, void* stream);   /* 512 / 1024 */
int tu_inv_march_2048(size_t hop, const InvArgs& a, long long batch, int sms, void* stream);
int tu_inv_ws_2048(size_t hop, const InvArgs& a, long long batch, int sms, void* stream);      /* warp-specialised (vvb_istft_ws.cuh) */
int tu_inv_march_4096(size_t hop, const InvArgs& a, long long batch, int sms, void* stream);
int tu_inv_march_8192(size_t hop, const InvArgs& a, long long batch, int sms, void* stream);
/* two frames per complex transform (fft_size 256 / 512 / 1024): tables_p = twiddles of the N-point complex plan,
 * tables_real = Tables blob of the real plan (windows, steady-state norm) */
int tu_inv_pair(int nfft, size_t hop, const InvArgs& a, long long batch, int sms, const float* tables_p, const float* tables_real, void* stream);
int tu_c2c(int n, const C2CArgs& a, int sms, void* stream);
int tu_chirp_fused(size_t M, const ChirpFusedArgs& a, int sms, void* stream);
struct FirArgs;
struct FirPadArgs;
int tu_fir(int m, const FirArgs& a, bool accum, int sms, void* stream);    /* one overlap-save pass (vvb_fir_kernels.cuh) */
int tu_fir_pad(const FirPadArgs& a, int sms, void* stream);
struct ResampleArgs;
int tu_resample(const ResampleArgs& a, int sms, void* stream);   /* polyphase resampling (vvb_resample_kernels.cuh) */
struct IirArgs;
int tu_iir(char pass, const IirArgs& a, int sms, void* stream);   /* IIR launch 'A', 'B' or 'C' (vvb_iir_kernels.cuh) */

}  // namespace vvb
