/*
 * vvb_cuda.cu -- implementation of the thin C-ABI in include/vvb200_cuda.h: device
 * plans (tables resident in HBM), kernel dispatch, memory / stream plumbing.
 *
 * Built by nvcc for sm_100a only (vv_dsp_b200/build.py).  There is no CPU code path:
 * without a usable CUDA device every entry returns 6 (VV_DSP_ERROR_UNSUPPORTED) or
 * 4 (VV_DSP_ERROR_INTERNAL) and the host library fails loudly.
 * (-DVVB_EMU is the test-only emulator build under tests/emu/, see cuda_emu.h.)
 */
#include "vvb_rt.cuh"
#include "vvb_direct_kernels.cuh"
#include "vvb_fir_kernels.cuh"
#include "vvb_resample_kernels.cuh"
#include "vvb_iir_kernels.cuh"

#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

using namespace vvb;

/* ------------------------------------------------------------------ error plumbing */
static thread_local char g_err[512] = "";
std::atomic<unsigned long long> vvb::g_launches{0};

extern "C" const char* vvb_last_error(void) { return g_err; }
extern "C" unsigned long long vvb_kernel_launches(void) { return g_launches.load(); }

int vvb::rt_fail(int code, const char* what, const char* detail)
{
    snprintf(g_err, sizeof(g_err), "%s: %s", what, detail ? detail : "");
    return code;
}
static int fail(int code, const char* what, const char* detail) { return rt_fail(code, what, detail); }

#ifdef VVB_EMU
/* ---- emulator runtime: host memory stands in for HBM, streams are no-ops */
namespace vvb_emu {
Cta* g_cta = nullptr;
uint3_emu g_threadIdx, g_blockIdx;
dim3 g_blockDim, g_gridDim;
char* g_dyn_smem = nullptr;
}
int vvb::rt_num_sms() { return 3; }
extern "C" int vvb_device_ready(void) { return 0; }
extern "C" int vvb_malloc(void** p, size_t bytes) { *p = malloc(bytes ? bytes : 1); return *p ? 0 : fail(4, "malloc", "oom"); }
extern "C" int vvb_free(void* p) { free(p); return 0; }
extern "C" int vvb_host_alloc(void** p, size_t bytes) { return vvb_malloc(p, bytes); }
extern "C" int vvb_host_memory_is_device_visible(void) { return 0; }
extern "C" int vvb_host_free(void* p) { free(p); return 0; }
extern "C" int vvb_memcpy_h2d(void* d, const void* s, size_t n, void*) { memcpy(d, s, n); return 0; }
extern "C" int vvb_memcpy_d2h(void* d, const void* s, size_t n, void*) { memcpy(d, s, n); return 0; }
static int emu_copy2d(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h)
{
    for (size_t r = 0; r < h; ++r) memcpy((char*)d + r * dp, (const char*)s + r * sp, w);
    return 0;
}
extern "C" int vvb_memcpy2d_h2d(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void*) { return emu_copy2d(d, dp, s, sp, w, h); }
extern "C" int vvb_memcpy2d_d2h(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void*) { return emu_copy2d(d, dp, s, sp, w, h); }
extern "C" int vvb_memcpy2d_d2d(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void*) { return emu_copy2d(d, dp, s, sp, w, h); }
extern "C" int vvb_memset(void* d, int v, size_t n, void*) { memset(d, v, n); return 0; }
extern "C" int vvb_stream_create(void** s) { *s = malloc(1); return 0; }
extern "C" int vvb_stream_destroy(void* s) { free(s); return 0; }
extern "C" int vvb_stream_sync(void*) { return 0; }
extern "C" int vvb_event_create(void** e) { *e = malloc(1); return 0; }
extern "C" int vvb_event_destroy(void* e) { free(e); return 0; }
extern "C" int vvb_event_record(void*, void*) { return 0; }
extern "C" int vvb_event_sync(void*) { return 0; }
extern "C" int vvb_device_count(int* n) { *n = 1; return 0; }
extern "C" int vvb_get_device(int* d) { *d = 0; return 0; }
extern "C" int vvb_set_device(int) { return 0; }
extern "C" int vvb_enable_peer_access(int, int) { return 0; }
extern "C" int vvb_event_create_timing(void** e) { *e = malloc(1); return 0; }
extern "C" int vvb_event_elapsed_ms(void*, void*, float* ms) { *ms = 0.f; return 0; }
extern "C" int vvb_graph_capture_begin(void*) { return 6; }
extern "C" int vvb_graph_capture_end(void*, void**) { return 6; }
extern "C" int vvb_graph_launch(void*, void*) { return 6; }
extern "C" int vvb_graph_destroy(void*) { return 0; }
extern "C" int vvb_stream_wait_event(void*, void*) { return 0; }
#else
/* ---- CUDA runtime */
int vvb::rt_num_sms()
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}
extern "C" int vvb_device_ready(void)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return fail(6, "no CUDA device", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    int dev = 0, major = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) return fail(6, "device is not sm_100-class", "this library ships sm_100a code only");
    return 0;
}
extern "C" int vvb_malloc(void** p, size_t bytes) { CK(cudaMalloc(p, bytes ? bytes : 1)); return 0; }
extern "C" int vvb_free(void* p) { if (p) CK(cudaFree(p)); return 0; }
extern "C" int vvb_host_alloc(void** p, size_t bytes) { CK(cudaMallocHost(p, bytes ? bytes : 1)); return 0; }
extern "C" int vvb_host_memory_is_device_visible(void)
{
    int dev = 0, uva = 0, native = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (cudaDeviceGetAttribute(&uva, cudaDevAttrUnifiedAddressing, dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (cudaDeviceGetAttribute(&native, cudaDevAttrCanUseHostPointerForRegisteredMem, dev) != cudaSuccess) { cudaGetLastError(); native = 0; }
    return uva && native;
}
extern "C" int vvb_host_free(void* p) { if (p) CK(cudaFreeHost(p)); return 0; }
extern "C" int vvb_memcpy_h2d(void* d, const void* s, size_t n, void* st) { CK(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, (cudaStream_t)st)); return 0; }
extern "C" int vvb_memcpy_d2h(void* d, const void* s, size_t n, void* st) { CK(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, (cudaStream_t)st)); return 0; }
extern "C" int vvb_memcpy2d_h2d(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void* st)
{
    CK(cudaMemcpy2DAsync(d, dp, s, sp, w, h, cudaMemcpyHostToDevice, (cudaStream_t)st)); return 0;
}
extern "C" int vvb_memcpy2d_d2h(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void* st)
{
    CK(cudaMemcpy2DAsync(d, dp, s, sp, w, h, cudaMemcpyDeviceToHost, (cudaStream_t)st)); return 0;
}
extern "C" int vvb_memcpy2d_d2d(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, void* st)
{
    CK(cudaMemcpy2DAsync(d, dp, s, sp, w, h, cudaMemcpyDeviceToDevice, (cudaStream_t)st)); return 0;
}
extern "C" int vvb_memset(void* d, int v, size_t n, void* st) { CK(cudaMemsetAsync(d, v, n, (cudaStream_t)st)); return 0; }
extern "C" int vvb_stream_create(void** s) { cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); *s = st; return 0; }
extern "C" int vvb_stream_destroy(void* s) { if (s) CK(cudaStreamDestroy((cudaStream_t)s)); return 0; }
extern "C" int vvb_stream_sync(void* s) { CK(cudaStreamSynchronize((cudaStream_t)s)); return 0; }
extern "C" int vvb_event_create(void** e) { cudaEvent_t ev; CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)); *e = ev; return 0; }
extern "C" int vvb_event_destroy(void* e) { if (e) CK(cudaEventDestroy((cudaEvent_t)e)); return 0; }
extern "C" int vvb_event_record(void* e, void* s) { CK(cudaEventRecord((cudaEvent_t)e, (cudaStream_t)s)); return 0; }
extern "C" int vvb_event_sync(void* e) { CK(cudaEventSynchronize((cudaEvent_t)e)); return 0; }
extern "C" int vvb_device_count(int* n) { CK(cudaGetDeviceCount(n)); return 0; }
extern "C" int vvb_get_device(int* d) { CK(cudaGetDevice(d)); return 0; }
extern "C" int vvb_set_device(int d) { CK(cudaSetDevice(d)); return 0; }
extern "C" int vvb_enable_peer_access(int device, int peer)
{
    if (device == peer) return 0;
    int can = 0, cur = 0;
    CK(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) return fail(6, "vvb_enable_peer_access", "devices are not peers");
    CK(cudaGetDevice(&cur));
    CK(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
    cudaSetDevice(cur);
    CK(e);
    return 0;
}
extern "C" int vvb_event_create_timing(void** e) { cudaEvent_t ev; CK(cudaEventCreate(&ev)); *e = ev; return 0; }
extern "C" int vvb_event_elapsed_ms(void* e0, void* e1, float* ms) { CK(cudaEventElapsedTime(ms, (cudaEvent_t)e0, (cudaEvent_t)e1)); return 0; }
extern "C" int vvb_graph_capture_begin(void* st) { CK(cudaStreamBeginCapture((cudaStream_t)st, cudaStreamCaptureModeThreadLocal)); return 0; }
extern "C" int vvb_graph_capture_end(void* st, void** exec)
{
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    *exec = nullptr;
    CK(cudaStreamEndCapture((cudaStream_t)st, &g));
    cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    CK(e);
    *exec = ge;
    return 0;
}
extern "C" int vvb_graph_launch(void* exec, void* st) { CK(cudaGraphLaunch((cudaGraphExec_t)exec, (cudaStream_t)st)); return 0; }
extern "C" int vvb_graph_destroy(void* exec) { if (exec) CK(cudaGraphExecDestroy((cudaGraphExec_t)exec)); return 0; }
extern "C" int vvb_stream_wait_event(void* s, void* e) { CK(cudaStreamWaitEvent((cudaStream_t)s, (cudaEvent_t)e, 0)); return 0; }
#endif

/* -------------------------------------------------------------------- plan tables */
/* Everything trigonometric is computed in double on the host and rounded once. */
template <class C> static void build_tables(std::vector<float>& blob, const float* window, size_t hop = 0)
{
    using TB = Tables<C>;
    constexpr int M = C::M, N = 2 * M;
    blob.assign(TB::TOTAL, 0.f);
    for (int i = 0; i < N; ++i) {
        const float w = window ? window[i] : 1.0f;
        blob[TB::WIN + i] = w;
        /* 1/M folded into the synthesis window: exact for the power-of-two sizes, one rounding otherwise */
        blob[TB::WSYN + i] = ((M & (M - 1)) == 0) ? w * (1.0f / (float)M) : (float)((double)w / (double)M);
    }
    auto fill = [&](int off, int R, int NS) {
        for (int r = 1; r < R; ++r)
            for (int jm = 0; jm < NS; ++jm) {
                const double ang = -2.0 * M_PI * (double)r * (double)jm / ((double)NS * R);
                blob[off + 2 * ((r - 1) * NS + jm)] = (float)cos(ang);
                blob[off + 2 * ((r - 1) * NS + jm) + 1] = (float)sin(ang);
            }
    };
    fill(TB::TW2, C::R2, C::R1);
    if (C::NP == 3) fill(TB::TW3, C::R3, C::R1 * C::R2);
    for (int k = 0; k <= M / 2; ++k) {
        const double ang = 2.0 * M_PI * (double)k / (double)N;
        blob[TB::POST + 2 * k] = (float)(0.5 * cos(ang));
        blob[TB::POST + 2 * k + 1] = (float)(0.5 * sin(ang));
    }
    /* steady-state window-sum sum_w2[c] = sum of w[c + i*hop]^2 over the frames covering a position,
     * accumulated in ASCENDING frame order (descending i) in float32 like the reference's norm_add
     * (src/spectral/stft.c:107), and the synthesis window with 1/sum_w2 folded in (guard 1e-12 as in
     * tools/dump_stft_roundtrip.c:50-52) */
    if (hop > 0 && hop <= (size_t)N) {
        for (size_t c = 0; c < hop; ++c) {
            float acc = 0.0f;
            for (long long i = ((long long)N - 1 - (long long)c) / (long long)hop; i >= 0; --i) {
                const float w = blob[TB::WIN + c + (size_t)i * hop];
                acc += w * w;
            }
            blob[TB::MIDNORM + c] = acc;
        }
        for (int p = 0; p < N; ++p) {
            const float nrm = blob[TB::MIDNORM + (size_t)p % hop];
            blob[TB::WSYN_NORM + p] = nrm > 1e-12f ? blob[TB::WSYN + p] * (1.0f / nrm) : 0.0f;
        }
    }
}

static bool fast_size(size_t m) { return m == 128 || m == 256 || m == 512 || m == 1024 || m == 2048 || m == 4096; }
/* real transforms of fft_size 2 m: the powers of two plus the mixed-radix speech / audio framings 320, 400, 480, 640;
 * VVB_NO_MIXED_RADIX=1 sends those through the chirp-z path like any other non-power-of-two size (read at creation) */
static bool fast_real_size(size_t m)
{
    return fast_size(m) || ((m == 160 || m == 200 || m == 240 || m == 320) && getenv("VVB_NO_MIXED_RADIX") == nullptr);
}
/* plan-API C2C (and the chirp-z transform built on it) also has a 256-thread, three-pass 8192-point kernel */
static bool fast_c2c_size(size_t n) { return fast_size(n) || n == 8192; }
static void build_c2c_tables(size_t n, std::vector<float>& blob);

/* twiddle tables of the n-point complex plan (no window) */
static void build_c2c_tables(size_t n, std::vector<float>& blob)
{
    switch (n) {
    case 128: build_tables<Cfg128>(blob, nullptr); break;
    case 256: build_tables<Cfg256>(blob, nullptr); break;
    case 512: build_tables<Cfg512>(blob, nullptr); break;
    case 1024: build_tables<Cfg1024>(blob, nullptr); break;
    case 2048: build_tables<Cfg2048>(blob, nullptr); break;
    case 4096: build_tables<Cfg4096>(blob, nullptr); break;
    default: build_tables<Cfg8192>(blob, nullptr); break;
    }
}

/* Bluestein plan for a size without a Stockham kernel (see vvb_direct_kernels.cuh): chirp table, spectrum of the
 * wrapped conjugate chirp, two power-of-two C2C engines and a work buffer grown on demand. */
struct Chirp {
    size_t n = 0, M = 0;
    float2* d_chirp = nullptr;       /* exp(-j pi i^2 / n), i < n */
    float2* d_bspec = nullptr;       /* FFT_M of the wrapped conjugate chirp */
    float2* d_bspec_m = nullptr;     /* the same divided by M (fused kernel: inverse scale folded in) */
    float* d_tables = nullptr;       /* Tables<C> blob of the M-point plan (fused kernel) */
    bool fused = true;
    vvb_fft_engine* fwd = nullptr;   /* C2C size M forward */
    vvb_fft_engine* bwd = nullptr;   /* C2C size M backward (scaled 1/M) */
    float2* d_work = nullptr;
    size_t work_elems = 0;
};
/* M = pow2 >= 2n-1: one fused kernel up to M = 8192 (n <= 4096), the multi-kernel pipeline on four-step plans up to M = 2^23 */
static bool chirp_size(size_t n) { return n >= 32 && n <= ((size_t)1 << 22) && getenv("VVB_NO_BLUESTEIN") == nullptr; }
static void chirp_destroy(Chirp* c);
static int chirp_create(size_t n, Chirp** out);
static int chirp_reserve(Chirp* c, size_t transforms, size_t* chunk);
static int chirp_convolve(Chirp* c, size_t count, void* stream);
static int chirp_fused(Chirp* c, ChirpFusedArgs a, int sms, void* stream);

struct vvb_engine {
    Chirp* chirp = nullptr;          /* sizes served by the Bluestein path */
    size_t nfft = 0, hop = 0;
    bool fast = false;
    int sms = 0;
    float* d_tables = nullptr;       /* fast: Tables<C> blob */
    float* d_tables_m = nullptr;     /* fft_size 512 / 1024: blob of the whole-warp config used by the marching ISTFT */
    float* d_tables_p = nullptr;     /* fft_size 256 / 512 / 1024: twiddles of the N-point complex plan of istft_pair_kernel */
    float* d_win = nullptr;          /* direct: window */
    float2* d_wtab = nullptr;        /* direct: (cos,-sin)(2 pi j/n) */
    float* d_scratch = nullptr;      /* direct: synthesis frames */
    size_t scratch_bytes = 0;
};

static void make_wtab(std::vector<float>& t, size_t n)
{
    t.resize(2 * n);
    for (size_t j = 0; j < n; ++j) {
        const double ang = 2.0 * M_PI * (double)j / (double)n;
        t[2 * j] = (float)cos(ang);
        t[2 * j + 1] = (float)-sin(ang);
    }
}

static int upload(float** d, const std::vector<float>& h)
{
    int st = vvb_malloc((void**)d, h.size() * sizeof(float));
    if (st) return st;
    st = vvb_memcpy_h2d(*d, h.data(), h.size() * sizeof(float), nullptr);
    if (st) return st;
    return vvb_stream_sync(nullptr);
}

extern "C" int vvb_engine_create(size_t nfft, size_t hop, const float* window, vvb_engine** out)
{
    if (!out || !window) return fail(1, "vvb_engine_create", "null");
    *out = nullptr;
    if (nfft == 0 || hop == 0 || hop > nfft) return fail(2, "vvb_engine_create", "size");
#ifndef VVB_EMU
    if (int st = vvb_device_ready()) return st;
#endif
    vvb_engine* e = new (std::nothrow) vvb_engine();
    if (!e) return fail(4, "vvb_engine_create", "oom");
    e->nfft = nfft; e->hop = hop; e->sms = rt_num_sms();
    e->fast = (nfft % 2 == 0) && fast_real_size(nfft / 2);
    int st = 0;
    std::vector<float> blob;
    if (e->fast) {
        switch (nfft / 2) {
        case 128: build_tables<Cfg128>(blob, window, hop); break;
        case 160: build_tables<Cfg160>(blob, window, hop); break;
        case 200: build_tables<Cfg200>(blob, window, hop); break;
        case 240: build_tables<Cfg240>(blob, window, hop); break;
        case 320: build_tables<Cfg320>(blob, window, hop); break;
        case 256: build_tables<Cfg256>(blob, window, hop); break;
        case 512: build_tables<Cfg512>(blob, window, hop); break;
        case 1024: build_tables<Cfg1024>(blob, window, hop); break;
        case 2048: build_tables<Cfg2048>(blob, window, hop); break;
        default: build_tables<Cfg4096>(blob, window, hop); break;
        }
        st = upload(&e->d_tables, blob);
        if (!st && (nfft == 512 || nfft == 1024)) {
            if (nfft == 512) build_tables<Cfg256m>(blob, window, hop); else build_tables<Cfg512m>(blob, window, hop);
            st = upload(&e->d_tables_m, blob);
        }
        if (!st && (nfft == 256 || nfft == 512 || nfft == 1024)) {
            if (nfft == 256) build_tables<Cfg256m>(blob, nullptr);
            else if (nfft == 512) build_tables<Cfg512m>(blob, nullptr);
            else build_tables<Cfg1024>(blob, nullptr);
            st = upload(&e->d_tables_p, blob);
        }
    } else {
        std::vector<float> w(window, window + nfft), t;
        make_wtab(t, nfft);
        st = upload(&e->d_win, w);
        if (!st) st = upload((float**)&e->d_wtab, t);
        if (!st && chirp_size(nfft)) st = chirp_create(nfft, &e->chirp);
    }
    if (st) { vvb_engine_destroy(e); return st; }
    *out = e;
    return 0;
}

extern "C" void vvb_engine_destroy(vvb_engine* e)
{
    if (!e) return;
    vvb_free(e->d_tables); vvb_free(e->d_tables_m); vvb_free(e->d_tables_p); vvb_free(e->d_win); vvb_free(e->d_wtab); vvb_free(e->d_scratch);
    chirp_destroy(e->chirp);
    delete e;
}

extern "C" int vvb_engine_is_fast(const vvb_engine* e) { return e && e->fast; }

extern "C" int vvb_stft_forward(vvb_engine* e, const float* d_x, size_t batch, size_t n, size_t x_pitch, size_t frames,
                                int pad_mode, int out_kind, void* d_out, size_t out_pitch, void* stream)
{
    if (!e || !d_x || !d_out) return fail(1, "vvb_stft_forward", "null");
    if (batch == 0 || frames == 0) return 0;
    if (frames > 0x7fffffffu || batch > 0x7fffffffu) return fail(2, "vvb_stft_forward", "too many frames");
    if (out_pitch < e->nfft / 2 + 1) return fail(2, "vvb_stft_forward", "out_pitch < bins");
    if (e->fast) {
        FwdArgs a;
        a.x = d_x; a.x_pitch = (long long)x_pitch; a.n = (long long)n;
        a.frames = (int)frames; a.hop = (int)e->hop; a.pad_mode = pad_mode;
        a.out = d_out; a.out_pitch = (long long)out_pitch; a.tables = e->d_tables;
        a.num_groups = (int)batch; a.groups_per_signal = 0;
        a.mel_w = nullptr; a.mel_seg = nullptr; a.mel_S = 0; a.mel_prow = 0; a.n_mels = 0; a.mel_eps = 0.f; a.mel_pair = 0; a.mel_unit = 0;
        if (!getenv("VVB_NO_MARCH")) {           /* zero padding and centred reflect padding both */
            int r = -1;
            /* (at fft_size 512 / 1024 the 2-pass generic forward kernel is faster than a 3-pass marching one) */
            /* (a producer / consumer split of the forward kernel like istft_ws_kernel was measured slower: the window then
             * lives in shared memory and the kernel becomes wavefront-bound, profiles/r02_ncu_full_forward_ws_experiment.csv) */
            if (e->nfft == 2048) r = tu_fwd_march_2048(e->hop, a, out_kind, e->sms, stream);
            else if (e->nfft == 4096) r = tu_fwd_march_4096(e->hop, a, out_kind, e->sms, stream);
            else if (e->nfft == 8192) r = tu_fwd_march_8192(e->hop, a, out_kind, e->sms, stream);
            if (r >= 0) return r;
        }
        return tu_fwd_generic((int)(e->nfft / 2), a, out_kind, e->sms, stream);
    }
    if (e->chirp && e->chirp->fused) {
        ChirpFusedArgs a;
        memset(&a, 0, sizeof(a));
        a.count = (long long)(batch * frames); a.mode = CHIRP_STFT_FWD; a.win = e->d_win;
        a.x = d_x; a.x_pitch = (long long)x_pitch; a.n_sig = (long long)n; a.frames = (int)frames; a.hop = (int)e->hop;
        a.pad_mode = pad_mode; a.out_kind = out_kind; a.out = d_out; a.out_pitch = (long long)out_pitch;
        return chirp_fused(e->chirp, a, e->sms, stream);
    }
    if (e->chirp) {
        Chirp* c = e->chirp;
        const size_t count = batch * frames;
        size_t chunk = 0;
        if (int st = chirp_reserve(c, count, &chunk)) return st;
        for (size_t g0 = 0; g0 < count; g0 += chunk) {
            ChirpFwdArgs a;
            a.x = d_x; a.x_pitch = (long long)x_pitch; a.n_sig = (long long)n;
            a.frames = (int)frames; a.hop = (int)e->hop; a.nfft = (int)e->nfft; a.pad_mode = pad_mode; a.M = (int)c->M;
            a.g0 = (long long)g0; a.count = (long long)std::min(chunk, count - g0);
            a.win = e->d_win; a.chirp = c->d_chirp; a.work = c->d_work;
            a.out_kind = out_kind; a.out = d_out; a.out_pitch = (long long)out_pitch;
            VVB_LAUNCH(chirp_pre_stft_kernel, persistent_grid((a.count * a.M + 255) / 256, 8, e->sms), 256, 0, stream, a);
            if (int st = chirp_convolve(c, (size_t)a.count, stream)) return st;
            VVB_LAUNCH(chirp_post_stft_kernel, persistent_grid((a.count * (a.nfft / 2 + 1) + 255) / 256, 8, e->sms), 256, 0, stream, a);
        }
        return 0;
    }
    DirFwdArgs a;
    a.x = d_x; a.x_pitch = (long long)x_pitch; a.n = (long long)n;
    a.batch = (int)batch; a.frames = (int)frames; a.hop = (int)e->hop; a.nfft = (int)e->nfft;
    a.pad_mode = pad_mode; a.out_kind = out_kind; a.out = d_out; a.out_pitch = (long long)out_pitch;
    a.win = e->d_win; a.wtab = e->d_wtab;
    const long long total = (long long)batch * frames * (e->nfft / 2 + 1);
    VVB_LAUNCH(stft_forward_direct_kernel, persistent_grid((total + 127) / 128, 16, e->sms), 128, 0, stream, a);
    return 0;
}

/* STFT -> power -> log-mel in ONE kernel (stft_march_kernel<..., OUT_LOGMEL>, see mel_phase): no power spectrogram in HBM.
 * Returns 6 when this plan / schedule has no fused kernel (the caller then chains the power and log-mel kernels). */
static FwdArgs logmel_probe_args(size_t mel_segments, size_t mel_prow, size_t mel_unit, size_t n_mels)
{
    FwdArgs a;
    memset(&a, 0, sizeof(a));
    a.mel_S = (int)mel_segments; a.mel_prow = (int)mel_prow; a.mel_unit = (int)mel_unit; a.n_mels = (int)n_mels;
    return a;
}
/* does this plan / schedule have a fused STFT -> log-mel kernel?  (same conditions as the launch below, nothing is enqueued) */
extern "C" int vvb_stft_forward_logmel_ok(const vvb_engine* e, size_t mel_segments, size_t mel_prow, size_t mel_unit, size_t n_mels)
{
    using C = Cfg1024;
    if (!e || !e->fast || getenv("VVB_MEL_UNFUSED")) return 0;
    if (e->nfft <= 1024) {        /* generic forward kernel, sub-warp teams: any hop; 3 = the band sums run per warp on pairs of its frames */
        if (mel_segments == 0 || mel_segments > 64 || n_mels == 0 || n_mels > 1024 || (mel_prow & 3) || mel_prow < e->nfft / 2 + 1) return 0;
        if (mel_unit != 2 && mel_unit != 4) return 0;
        if (getenv("VVB_MEL_NO_GENERIC")) return 0;
        return tu_fwd_logmel((int)(e->nfft / 2), logmel_probe_args(mel_segments, mel_prow, mel_unit, n_mels), e->sms, nullptr, true) == 0 ? 3 : 0;
    }
    if (e->nfft != 2048 || mel_unit != MEL_U || getenv("VVB_NO_MARCH")) return 0;
    if (e->hop != 256 && e->hop != 512 && e->hop != 1024) return 0;
    if (mel_segments == 0 || mel_segments > 64 || n_mels == 0 || n_mels > 1024 || (mel_prow & 3)) return 0;
    /* the power row sits in the lower half of the exchange buffer; its tail past the last bin is re-zeroed by one store per lane */
    if (mel_prow < C::M + 1 || mel_prow > C::M + 1 + 32 || mel_prow > 2 * (size_t)(C::M / 2 + C::M / 2 / C::R1)) return 0;
    constexpr size_t G = March<C>::G;
    const size_t slots = e->hop / (2 * C::T);                  /* S of the kernel: register slots per hop */
    const size_t base = sizeof(float) * 2 * (C::TW2 + C::TW3 + C::POST + 1 + G * C::XBUF + G * (C::E / slots + 1) * C::T * slots) + 8 * G;
    /* 2: two frames per band-sum phase (a second row buffer per warp); 1: one frame, where shared memory is short (hop 1024) */
    if (!getenv("VVB_MEL_SINGLE") && base + mel_smem_bytes((int)G, (int)mel_segments, (int)n_mels, (int)mel_prow, 1) <= 227 * 1024) return 2;
    return base + mel_smem_bytes((int)G, (int)mel_segments, (int)n_mels, (int)mel_prow, 0) <= 227 * 1024 ? 1 : 0;
}

extern "C" int vvb_stft_forward_logmel(vvb_engine* e, const float* d_x, size_t batch, size_t n, size_t x_pitch, size_t frames, int pad_mode,
                                       const float* d_mel_w, const int* d_mel_seg, size_t mel_segments, size_t mel_prow, size_t mel_unit,
                                       size_t n_mels, float eps, float* d_out, void* stream)
{
    if (!e || !d_x || !d_out || !d_mel_w || !d_mel_seg) return fail(1, "vvb_stft_forward_logmel", "null");
    if (batch == 0 || frames == 0) return 0;
    if (frames > 0x7fffffffu || batch > 0x7fffffffu) return fail(2, "vvb_stft_forward_logmel", "too many frames");
    const int mode = vvb_stft_forward_logmel_ok(e, mel_segments, mel_prow, mel_unit, n_mels);
    if (!mode) return 6;
    FwdArgs a;
    a.x = d_x; a.x_pitch = (long long)x_pitch; a.n = (long long)n;
    a.frames = (int)frames; a.hop = (int)e->hop; a.pad_mode = pad_mode;
    a.out = d_out; a.out_pitch = (long long)n_mels; a.tables = e->d_tables;
    a.num_groups = (int)batch; a.groups_per_signal = 0;
    a.mel_w = reinterpret_cast<const float4*>(d_mel_w); a.mel_seg = reinterpret_cast<const int2*>(d_mel_seg);
    a.mel_S = (int)mel_segments; a.mel_prow = (int)mel_prow; a.mel_unit = (int)mel_unit; a.n_mels = (int)n_mels; a.mel_eps = eps; a.mel_pair = mode == 2;
    if (mode == 3) return tu_fwd_logmel((int)(e->nfft / 2), a, e->sms, stream, false);
    const int r = tu_fwd_march_2048(e->hop, a, OUT_LOGMEL, e->sms, stream);
    return r < 0 ? 6 : r;
}

/* ------------------------------------------------------------------ inverse launch */
static int ensure_scratch(vvb_engine* e, size_t bytes)
{
    if (e->scratch_bytes >= bytes) return 0;
    vvb_free(e->d_scratch); e->d_scratch = nullptr; e->scratch_bytes = 0;
    int st = vvb_malloc((void**)&e->d_scratch, bytes);
    if (!st) e->scratch_bytes = bytes;
    return st;
}

/* Bluestein synthesis of `count` frames: Hermitian half spectra -> real frames times `win` (nullptr: none) */
static int chirp_inverse_frames(vvb_engine* e, const float2* d_spec, size_t count, size_t spec_pitch, float* d_frames,
                                const float* win, void* stream)
{
    Chirp* c = e->chirp;
    if (c->fused) {
        ChirpFusedArgs a;
        memset(&a, 0, sizeof(a));
        a.count = (long long)count; a.mode = CHIRP_STFT_INV; a.win = win;
        a.spec = d_spec; a.spec_pitch = (long long)spec_pitch; a.frames_out = d_frames;
        return chirp_fused(c, a, e->sms, stream);
    }
    size_t chunk = 0;
    if (int st = chirp_reserve(c, count, &chunk)) return st;
    for (size_t g0 = 0; g0 < count; g0 += chunk) {
        ChirpInvArgs a;
        a.spec = d_spec; a.spec_pitch = (long long)spec_pitch; a.g0 = (long long)g0; a.count = (long long)std::min(chunk, count - g0);
        a.nfft = (int)e->nfft; a.M = (int)c->M; a.win = win; a.chirp = c->d_chirp; a.work = c->d_work; a.frames_out = d_frames;
        VVB_LAUNCH(chirp_pre_spec_kernel, persistent_grid((a.count * a.M + 255) / 256, 8, e->sms), 256, 0, stream, a);
        if (int st = chirp_convolve(c, (size_t)a.count, stream)) return st;
        VVB_LAUNCH(chirp_post_frames_kernel, persistent_grid((a.count * a.nfft + 255) / 256, 8, e->sms), 256, 0, stream, a);
    }
    return 0;
}

extern "C" int vvb_stft_inverse_frames(vvb_engine* e, const vvb_cpx* d_spec, size_t count, size_t spec_pitch,
                                       float* d_frames, void* stream)
{
    if (!e || !d_spec || !d_frames) return fail(1, "vvb_stft_inverse_frames", "null");
    if (count == 0) return 0;
    if (count > 0x7fffffffu) return fail(2, "vvb_stft_inverse_frames", "too many frames");
    if (e->fast) {
        InvArgs a;
        memset(&a, 0, sizeof(a));
        a.spec = reinterpret_cast<const float2*>(d_spec); a.spec_pitch = (long long)spec_pitch;
        a.frames = (int)count; a.hop = (int)e->hop; a.y = d_frames; a.tables = e->d_tables;
        return tu_inv_generic((int)(e->nfft / 2), false, a, 1, e->sms, stream);
    }
    if (e->chirp) return chirp_inverse_frames(e, reinterpret_cast<const float2*>(d_spec), count, spec_pitch, d_frames, e->d_win, stream);
    DirInvArgs a;
    a.spec = reinterpret_cast<const float2*>(d_spec); a.spec_pitch = (long long)spec_pitch;
    a.count = (long long)count; a.nfft = (int)e->nfft; a.frames_out = d_frames; a.win = e->d_win; a.wtab = e->d_wtab;
    const long long total = (long long)count * e->nfft;
    VVB_LAUNCH(stft_inverse_direct_kernel, persistent_grid((total + 127) / 128, 16, e->sms), 128, 0, stream, a);
    return 0;
}

/* marching / warp-specialised launch for one (fft_size, hop); -1 when there is none */
static int launch_inverse_marching(vvb_engine* e, const InvArgs& a, long long batch, void* stream)
{
    int r = -1;
    InvArgs am = a;
    am.tables = e->d_tables_m;
    if (e->nfft == 512 || e->nfft == 1024) r = tu_inv_march_small((int)e->nfft, e->hop, am, batch, e->sms, stream);
    else if (e->nfft == 2048) {
        if (!getenv("VVB_NO_WS")) r = tu_inv_ws_2048(e->hop, a, batch, e->sms, stream);
        if (r < 0) r = tu_inv_march_2048(e->hop, a, batch, e->sms, stream);
    }
    /* (a producer / consumer split between two-warp teams was built for fft_size 4096 and measured slower: the consumer team
     * holds two of the three passes and loses the half exchange, profiles/r02_ncu_full_istft_ws3_experiment.csv) */
    else if (e->nfft == 4096) r = tu_inv_march_4096(e->hop, a, batch, e->sms, stream);
    else if (e->nfft == 8192) r = tu_inv_march_8192(e->hop, a, batch, e->sms, stream);
    return r;
}

/* One frame-range shard of a longer stream (see InvArgs::halo_frames): d_spec holds halo_frames + own frames. */
extern "C" int vvb_stft_inverse_shard(vvb_engine* e, const vvb_cpx* d_spec, size_t frames, size_t halo_frames, int head_edge,
                                      int tail_edge, size_t spec_pitch, float* d_y, size_t n_out, const float* d_inv_norm, void* stream)
{
    if (!e || !d_y || !d_spec) return fail(1, "vvb_stft_inverse_shard", "null");
    if (frames == 0 || frames > 0x7fffffffu || halo_frames >= frames || n_out == 0) return fail(2, "vvb_stft_inverse_shard", "size");
    if (halo_frames && head_edge) return fail(2, "vvb_stft_inverse_shard", "the first shard has no halo");
    if (!e->fast) return fail(6, "vvb_stft_inverse_shard", "needs a marching kernel (fft_size 512 ... 8192)");
    InvArgs a;
    memset(&a, 0, sizeof(a));
    a.spec = reinterpret_cast<const float2*>(d_spec); a.spec_pitch = (long long)spec_pitch;
    a.frames = (int)frames; a.hop = (int)e->hop;
    a.y = d_y; a.y_pitch = (long long)((n_out + 1) & ~(size_t)1); a.n_out = (long long)n_out;
    a.inv_norm = d_inv_norm; a.tables = e->d_tables;
    a.halo_frames = (int)halo_frames; a.head_edge = head_edge ? 1 : 0; a.tail_edge = tail_edge ? 1 : 0;
    const int r = launch_inverse_marching(e, a, 1, stream);
    return r >= 0 ? r : fail(6, "vvb_stft_inverse_shard", "no marching kernel for this (fft_size, hop)");
}

extern "C" int vvb_stft_inverse(vvb_engine* e, const vvb_cpx* d_spec, size_t batch, size_t frames, size_t spec_pitch,
                                float* d_y, size_t n_out, size_t y_pitch, const float* d_inv_norm, void* stream)
{
    if (!e || !d_y || (!d_spec && frames)) return fail(1, "vvb_stft_inverse", "null");
    if (batch == 0 || n_out == 0) return 0;
    if (frames > 0x7fffffffu) return fail(2, "vvb_stft_inverse", "too many frames");
    if (frames == 0) {
        for (size_t b = 0; b < batch; ++b)
            if (int st = vvb_memset(d_y + b * y_pitch, 0, n_out * sizeof(float), stream)) return st;
        return 0;
    }
    if (e->fast) {
        InvArgs a;
        memset(&a, 0, sizeof(a));
        a.spec = reinterpret_cast<const float2*>(d_spec); a.spec_pitch = (long long)spec_pitch;
        a.frames = (int)frames; a.hop = (int)e->hop;
        a.y = d_y; a.y_pitch = (long long)y_pitch; a.n_out = (long long)n_out;
        a.inv_norm = d_inv_norm; a.tables = e->d_tables;
        a.halo_frames = 0; a.head_edge = 1; a.tail_edge = 1;          /* whole signals */
        if (e->d_tables_p && !getenv("VVB_NO_PAIR") && !getenv("VVB_NO_MARCH")) {
            const int r = tu_inv_pair((int)e->nfft, e->hop, a, (long long)batch, e->sms, e->d_tables_p, e->d_tables, stream);
            if (r >= 0) return r;
        }
        if (!getenv("VVB_NO_MARCH")) {          /* (rows that are not 8-byte aligned are stored with 32-bit stores) */
            const int r = launch_inverse_marching(e, a, (long long)batch, stream);
            if (r >= 0) return r;
        }
        return tu_inv_generic((int)(e->nfft / 2), true, a, (long long)batch, e->sms, stream);
    }
    /* direct path: synthesis frames to HBM scratch, then the stand-alone overlap-add kernel */
    const size_t count = batch * frames;
    if (int st = ensure_scratch(e, count * e->nfft * sizeof(float))) return st;
    if (e->chirp) {
        if (int st = chirp_inverse_frames(e, reinterpret_cast<const float2*>(d_spec), count, spec_pitch, e->d_scratch, e->d_win, stream)) return st;
    } else {
        DirInvArgs d;
        d.spec = reinterpret_cast<const float2*>(d_spec); d.spec_pitch = (long long)spec_pitch;
        d.count = (long long)count; d.nfft = (int)e->nfft; d.frames_out = e->d_scratch; d.win = e->d_win; d.wtab = e->d_wtab;
        const long long total = (long long)count * e->nfft;
        VVB_LAUNCH(stft_inverse_direct_kernel, persistent_grid((total + 127) / 128, 16, e->sms), 128, 0, stream, d);
    }
    OlaArgs o;
    o.frames_in = e->d_scratch; o.batch = (int)batch; o.frames = (int)frames; o.hop = (int)e->hop; o.nfft = (int)e->nfft;
    o.y = d_y; o.y_pitch = (long long)y_pitch; o.n_out = (long long)n_out; o.inv_norm = d_inv_norm;
    const long long tot2 = (long long)batch * n_out;
    VVB_LAUNCH(overlap_add_kernel, persistent_grid((tot2 + 255) / 256, 8, e->sms), 256, 0, stream, o);
    return 0;
}

/* ---------------------------------------------------------------------- FFT engine */
struct vvb_fft_engine {
    size_t n = 0;
    int type = 0, dir = 0, sms = 0;
    bool fast_c2c = false;
    float* d_tables = nullptr;       /* C2C fast: Tables<C> blob with M = n */
    float2* d_wtab = nullptr;        /* direct C2C */
    vvb_engine* real = nullptr;      /* R2C / C2R: STFT engine with a boxcar window, hop = n */
    Chirp* chirp = nullptr;          /* C2C sizes served by the Bluestein path */
    /* four-step (n = n1 n2, powers of two above 8192): two batched Stockham plans + transposes through work buffers */
    size_t n1 = 0, n2 = 0;
    vvb_fft_engine* sub1 = nullptr;  /* C2C size n1, same direction */
    vvb_fft_engine* sub2 = nullptr;  /* C2C size n2 */
    vvb_fft_engine* c2c = nullptr;   /* R2C / C2R of a four-step size: the complex plan underneath */
    float2* d_work[2] = {nullptr, nullptr};
    size_t work_elems = 0;
};

/* powers of two in (8192, 2^26]: n1 = 2^ceil(log2(n)/2) <= 8192, n2 = n / n1 >= 128 */
static bool four_step_size(size_t n) { return n > 8192 && n <= ((size_t)1 << 26) && (n & (n - 1)) == 0; }

extern "C" int vvb_fft_engine_create(size_t n, int type, int dir, vvb_fft_engine** out)
{
    if (!out) return fail(1, "vvb_fft_engine_create", "null");
    *out = nullptr;
    if (n == 0) return fail(2, "vvb_fft_engine_create", "n == 0");
    if (type < 0 || type > 2 || (dir != 1 && dir != -1)) return fail(3, "vvb_fft_engine_create", "enum");
#ifndef VVB_EMU
    if (int st = vvb_device_ready()) return st;
#endif
    vvb_fft_engine* e = new (std::nothrow) vvb_fft_engine();
    if (!e) return fail(4, "vvb_fft_engine_create", "oom");
    e->n = n; e->type = type; e->dir = dir; e->sms = rt_num_sms();
    int st = 0;
    if (type == 0) {
        e->fast_c2c = fast_c2c_size(n);
        std::vector<float> blob;
        if (e->fast_c2c) {
            build_c2c_tables(n, blob);
            st = upload(&e->d_tables, blob);
        } else if (four_step_size(n)) {
            int lg = 0;
            while (((size_t)1 << lg) < n) ++lg;
            e->n1 = (size_t)1 << ((lg + 1) / 2); e->n2 = n / e->n1;
            st = vvb_fft_engine_create(e->n1, 0, dir, &e->sub1);
            if (!st) st = vvb_fft_engine_create(e->n2, 0, dir, &e->sub2);
        } else {
            make_wtab(blob, n);
            st = upload((float**)&e->d_wtab, blob);
            if (!st && chirp_size(n)) st = chirp_create(n, &e->chirp);
        }
    } else if (four_step_size(n)) {
        st = vvb_fft_engine_create(n, 0, dir, &e->c2c);       /* R2C = C2C of (x, 0), half kept; C2R = C2C of the Hermitian extension */
    } else {
        std::vector<float> ones(n, 1.0f);
        st = vvb_engine_create(n, n, ones.data(), &e->real);
    }
    if (st) { vvb_fft_engine_destroy(e); return st; }
    *out = e;
    return 0;
}

/* 1 when one transform is ONE kernel that reads its input once (Stockham, fused chirp-z): such a plan may run straight on
 * mapped host memory; the multi-kernel pipelines and the O(n^2) kernels may not */
extern "C" int vvb_fft_engine_is_single_kernel(const vvb_fft_engine* e)
{
    if (!e) return 0;
    if (e->type == 0) return e->fast_c2c || (e->chirp && e->chirp->fused);
    return e->real && (e->real->fast || (e->real->chirp && e->real->chirp->fused));
}

extern "C" void vvb_fft_engine_destroy(vvb_fft_engine* e)
{
    if (!e) return;
    vvb_free(e->d_tables); vvb_free(e->d_wtab); vvb_engine_destroy(e->real);
    chirp_destroy(e->chirp);
    vvb_fft_engine_destroy(e->sub1); vvb_fft_engine_destroy(e->sub2); vvb_fft_engine_destroy(e->c2c);
    vvb_free(e->d_work[0]); vvb_free(e->d_work[1]);
    delete e;
}

/* work buffers for `want` transforms of n points, bounded at 256 MB each: *chunk = transforms per pass */
static int four_step_reserve(vvb_fft_engine* e, size_t want, size_t* chunk)
{
    const size_t cap = std::max<size_t>(((size_t)256 << 20) / (e->n * sizeof(float2)), 1);
    want = std::min(want, cap);
    if (e->work_elems < want * e->n) {
        for (int i = 0; i < 2; ++i) { vvb_free(e->d_work[i]); e->d_work[i] = nullptr; }
        e->work_elems = 0;
        for (int i = 0; i < 2; ++i)
            if (int st = vvb_malloc((void**)&e->d_work[i], want * e->n * sizeof(float2))) return st;
        e->work_elems = want * e->n;
    }
    *chunk = e->work_elems / e->n;
    return 0;
}

static int four_step_transpose(const float2* in, float2* out, size_t rows, size_t cols, size_t batch, size_t twiddle_n, int inverse, int sms,
                               void* stream)
{
    FourStepArgs a;
    a.in = in; a.out = out; a.rows = (int)rows; a.cols = (int)cols; a.batch = (long long)batch; a.twiddle_n = (long long)twiddle_n; a.inverse = inverse;
    const long long tiles = (long long)((rows + 31) / 32) * ((cols + 31) / 32) * (long long)batch;
    VVB_LAUNCH(fourstep_transpose_kernel, persistent_grid(tiles, 8, sms), 256, 0, stream, a);
    return 0;
}

/* X[k1 + n1 k2] = sum_j2 W_n2^(j2 k2) [ W_n^(j2 k1) sum_j1 x[j1 n2 + j2] W_n1^(j1 k1) ]: transpose, n2 transforms of n1 points,
 * twiddle + transpose, n1 transforms of n2 points, transpose.  in == out is fine (everything goes through the work buffers). */
static int four_step_exec(vvb_fft_engine* e, const float2* d_in, float2* d_out, size_t batch, void* stream)
{
    const int inv = e->dir < 0;
    size_t chunk = 0;
    if (int st = four_step_reserve(e, batch, &chunk)) return st;
    for (size_t b0 = 0; b0 < batch; b0 += chunk) {
        const size_t nb = std::min(chunk, batch - b0);
        const float2* x = d_in + b0 * e->n;
        float2* y = d_out + b0 * e->n;
        if (int st = four_step_transpose(x, e->d_work[0], e->n1, e->n2, nb, 0, inv, e->sms, stream)) return st;
        if (int st = vvb_fft_exec(e->sub1, e->d_work[0], e->d_work[0], nb * e->n2, stream)) return st;
        if (int st = four_step_transpose(e->d_work[0], e->d_work[1], e->n2, e->n1, nb, e->n, inv, e->sms, stream)) return st;
        if (int st = vvb_fft_exec(e->sub2, e->d_work[1], e->d_work[1], nb * e->n1, stream)) return st;
        if (int st = four_step_transpose(e->d_work[1], y, e->n1, e->n2, nb, 0, inv, e->sms, stream)) return st;
    }
    return 0;
}

static int four_step_real_exec(vvb_fft_engine* e, const void* d_in, void* d_out, size_t batch, void* stream)
{
    vvb_fft_engine* c = e->c2c;
    size_t chunk = 0;
    if (int st = four_step_reserve(e, batch, &chunk)) return st;        /* e->d_work[0]: the complex signal / spectrum */
    const size_t bins = e->n / 2 + 1;
    for (size_t b0 = 0; b0 < batch; b0 += chunk) {
        const size_t nb = std::min(chunk, batch - b0);
        const long long total = (long long)(nb * e->n);
        const int grid = persistent_grid((total + 255) / 256, 8, e->sms);
        if (e->type == 1) {
            VVB_LAUNCH(real_to_cpx_kernel, grid, 256, 0, stream, (const float*)d_in + b0 * e->n, e->d_work[0], total);
            if (int st = vvb_fft_exec(c, e->d_work[0], e->d_work[0], nb, stream)) return st;
            VVB_LAUNCH(cpx_keep_half_kernel, grid, 256, 0, stream, (const float2*)e->d_work[0], (float2*)d_out + b0 * bins, (long long)nb, (int)e->n);
        } else {
            VVB_LAUNCH(hermitian_extend_kernel, grid, 256, 0, stream, (const float2*)d_in + b0 * bins, e->d_work[0], (long long)nb, (int)e->n);
            if (int st = vvb_fft_exec(c, e->d_work[0], e->d_work[0], nb, stream)) return st;
            VVB_LAUNCH(cpx_real_part_kernel, grid, 256, 0, stream, (const float2*)e->d_work[0], (float*)d_out + b0 * e->n, total);
        }
    }
    return 0;
}

extern "C" int vvb_fft_exec(vvb_fft_engine* e, const void* d_in, void* d_out, size_t batch, void* stream)
{
    if (!e || !d_in || !d_out) return fail(1, "vvb_fft_exec", "null");
    if (batch == 0) return 0;
    if (batch > 0x7fffffffu) return fail(2, "vvb_fft_exec", "batch");
    if (e->type == 0 && e->sub1) return four_step_exec(e, (const float2*)d_in, (float2*)d_out, batch, stream);
    if (e->type != 0 && e->c2c) return four_step_real_exec(e, d_in, d_out, batch, stream);
    if (e->type == 0) {
        if (e->fast_c2c) {
            C2CArgs a;
            a.in = (const float2*)d_in; a.out = (float2*)d_out; a.batch = (int)batch; a.inverse = e->dir < 0; a.tables = e->d_tables;
            return tu_c2c((int)e->n, a, e->sms, stream);
        }
        if (e->chirp && e->chirp->fused) {      /* in place is fine: a team reads its whole transform before it writes */
            ChirpFusedArgs a;
            memset(&a, 0, sizeof(a));
            a.count = (long long)batch; a.mode = CHIRP_C2C; a.cin = (const float2*)d_in; a.cout = (float2*)d_out; a.inverse = e->dir < 0;
            return chirp_fused(e->chirp, a, e->sms, stream);
        }
        if (e->chirp) {
            Chirp* c = e->chirp;
            size_t chunk = 0;
            if (int st = chirp_reserve(c, batch, &chunk)) return st;
            for (size_t g0 = 0; g0 < batch; g0 += chunk) {
                ChirpC2CArgs a;
                a.in = (const float2*)d_in + g0 * e->n; a.out = (float2*)d_out + g0 * e->n;
                a.count = (long long)std::min(chunk, batch - g0); a.n = (int)e->n; a.M = (int)c->M; a.inverse = e->dir < 0;
                a.chirp = c->d_chirp; a.work = c->d_work;
                VVB_LAUNCH(chirp_pre_c2c_kernel, persistent_grid((a.count * a.M + 255) / 256, 8, e->sms), 256, 0, stream, a);
                if (int st = chirp_convolve(c, (size_t)a.count, stream)) return st;
                VVB_LAUNCH(chirp_post_c2c_kernel, persistent_grid((a.count * a.n + 255) / 256, 8, e->sms), 256, 0, stream, a);
            }
            return 0;
        }
        /* the direct kernel reads every input of a transform for every output: out must not alias in */
        DirC2CArgs a;
        a.in = (const float2*)d_in; a.out = (float2*)d_out; a.batch = (long long)batch; a.n = (int)e->n;
        a.inverse = e->dir < 0; a.wtab = e->d_wtab;
        if (d_in == d_out) return fail(3, "vvb_fft_exec", "direct C2C cannot run in place (host stages a copy)");
        const long long total = (long long)batch * e->n;
        VVB_LAUNCH(fft_c2c_direct_kernel, persistent_grid((total + 127) / 128, 16, e->sms), 128, 0, stream, a);
        return 0;
    }
    const size_t bins = e->n / 2 + 1;
    if (e->type == 1)   /* R2C: one frame per transform, boxcar window, complex half spectrum */
        return vvb_stft_forward(e->real, (const float*)d_in, batch, e->n, e->n, 1, PAD_ZERO, OUT_COMPLEX, d_out, bins, stream);
    return vvb_stft_inverse_frames(e->real, (const vvb_cpx*)d_in, batch, bins, (float*)d_out, stream);   /* C2R */
}

/* ------------------------------------------------------------------ FIR by overlap-save */
/* the forward C2C plan of the transform size: its tables feed fir_ols_kernel, its kernel makes the filter spectra */
struct vvb_fir_engine {
    vvb_fft_engine* fwd = nullptr;
};

extern "C" int vvb_fir_engine_create(size_t m, vvb_fir_engine** out)
{
    if (!out) return fail(1, "vvb_fir_engine_create", "null");
    *out = nullptr;
    if (m < 128 || m > 8192 || (m & (m - 1)) != 0) return fail(6, "vvb_fir_engine_create", "no Stockham kernel for this size");
    vvb_fir_engine* e = new (std::nothrow) vvb_fir_engine();
    if (!e) return fail(4, "vvb_fir_engine_create", "oom");
    if (int st = vvb_fft_engine_create(m, 0, 1, &e->fwd)) { delete e; return st; }
    *out = e;
    return 0;
}

extern "C" void vvb_fir_engine_destroy(vvb_fir_engine* e)
{
    if (!e) return;
    vvb_fft_engine_destroy(e->fwd);
    delete e;
}

extern "C" int vvb_fir_spectra(vvb_fir_engine* e, const float* d_h, size_t filters, size_t h_pitch, size_t num_taps, size_t lp,
                               size_t parts, vvb_cpx* d_spec, void* stream)
{
    if (!e || !d_h || !d_spec) return fail(1, "vvb_fir_spectra", "null");
    if (filters == 0) return 0;
    const size_t m = e->fwd->n;
    if (lp == 0 || lp > m || parts == 0) return fail(2, "vvb_fir_spectra", "partition");
    FirPadArgs a;
    a.h = d_h; a.h_pitch = (long long)h_pitch; a.taps = (long long)num_taps; a.out = (float2*)d_spec;
    a.total = (long long)(filters * parts * m); a.m = (int)m; a.lp = (int)lp; a.parts = (int)parts;
    if (int st = tu_fir_pad(a, e->fwd->sms, stream)) return st;
    return vvb_fft_exec(e->fwd, d_spec, d_spec, filters * parts, stream);      /* in place: each team reads before it writes */
}

extern "C" int vvb_fir_filter(vvb_fir_engine* e, const vvb_cpx* d_spec, size_t spec_stride, size_t num_taps, size_t lp, size_t parts,
                              const float* d_x, size_t batch, size_t n, size_t x_pitch, float* d_y, size_t n_out, size_t y_pitch,
                              void* stream)
{
    if (!e || !d_spec || !d_x || !d_y) return fail(1, "vvb_fir_filter", "null");
    if (batch == 0 || n_out == 0) return 0;
    const size_t m = e->fwd->n;
    if (lp == 0 || lp > m || parts == 0 || (parts - 1) * lp >= num_taps) return fail(2, "vvb_fir_filter", "partition");
    FirArgs a;
    a.x = d_x; a.x_pitch = (long long)x_pitch; a.n = (long long)n;
    a.y = d_y; a.y_pitch = (long long)y_pitch; a.n_out = (long long)n_out; a.n_full = (long long)(n + num_taps - 1);
    a.h_stride = (long long)spec_stride;
    a.lp = (int)lp; a.L = (int)(m - lp + 1);
    a.blocks = ((long long)n_out + a.L - 1) / a.L;
    a.pairs = (a.blocks + 1) / 2;
    a.count = (long long)batch * a.pairs;
    a.tables = e->fwd->d_tables;
    for (size_t p = 0; p < parts; ++p) {          /* ascending partitions: every output sample sums its passes in one order */
        a.H = (const float2*)d_spec + p * m;
        a.delay = (long long)(p * lp);
        if (int st = tu_fir((int)m, a, p > 0, e->fwd->sms, stream)) return st;
    }
    return 0;
}

/* ------------------------------------------------------------------ polyphase resampling */
/* the largest shared-memory input span a launch stages; beyond it the kernel reads its inputs through L1 */
#define VVB_RESAMPLE_SMEM_MAX ((size_t)200 << 10)

extern "C" int vvb_resample_poly(const float* d_bank, size_t up, size_t down, size_t taps_per_phase, size_t half,
                                 const float* d_x, size_t batch, size_t n, size_t x_pitch, float* d_y, size_t n_out,
                                 size_t y_pitch, void* stream)
{
    if (!d_bank || !d_x || !d_y) return fail(1, "vvb_resample_poly", "null");
    if (up == 0 || down == 0 || taps_per_phase == 0) return fail(2, "vvb_resample_poly", "ratio");
    if (batch == 0 || n_out == 0) return 0;
    ResampleArgs a;
    a.x = d_x; a.x_pitch = (long long)x_pitch; a.n = (long long)n;
    a.y = d_y; a.y_pitch = (long long)y_pitch; a.n_out = (long long)n_out;
    a.bank = d_bank;
    a.up = (long long)up; a.down = (long long)down; a.half = (long long)half;
    a.half_mod = (long long)(half % up);
    a.taps = (int)taps_per_phase;
    {   /* down^-1 mod up by the extended Euclidean algorithm (gcd(up, down) == 1) */
        long long r0 = a.up, r1 = a.down % a.up, t0 = 0, t1 = 1;
        while (r1) { const long long qq = r0 / r1, r2 = r0 - qq * r1, t2 = t0 - qq * t1; r0 = r1; r1 = r2; t0 = t1; t1 = t2; }
        if (r0 != 1 && up != 1) return fail(2, "vvb_resample_poly", "up and down are not coprime");
        a.dinv = up == 1 ? 0 : ((t0 % a.up) + a.up) % a.up;
    }
    const long long band = (long long)RS_RUN * a.up;
    const long long bands = (a.n_out + band - 1) / band;
    a.tiles = (bands * a.up + RS_THREADS - 1) / RS_THREADS;
    a.count = (long long)batch * a.tiles;
    /* a tile's runs lie in at most (RS_THREADS - 1) / up + 2 bands, which read at most that times R down inputs plus T */
    const double span = ((double)((RS_THREADS - 1) / a.up) + 2.0) * RS_RUN * (double)down + (double)taps_per_phase + 1.0;
    a.span = span < 1e8 && resample_smem_bytes((long long)span) <= VVB_RESAMPLE_SMEM_MAX ? (int)span : 0;
    return tu_resample(a, rt_num_sms(), stream);
}

/* ------------------------------------------------------------------ IIR second-order sections */
extern "C" int vvb_iir_sos(const vvb_iir_call* c, void* stream)
{
    if (!c || !c->d_table || !c->x || !c->y) return fail(1, "vvb_iir_sos", "null");
    if (c->sections == 0 || 2 * c->sections > (size_t)IIR_CHAIN_THREADS || c->segment == 0 ||
        c->segment % ((size_t)IIR_THREADS * VVB_IIR_RUN) != 0)
        return fail(2, "vvb_iir_sos", "sections / segment");
    if (c->batch == 0 || c->nv == 0) return 0;
    IirArgs a;
    a.x = c->x; a.x_pitch = (long long)c->x_pitch; a.n = (long long)c->n;
    a.in_mode = c->in_mode; a.padtype = c->padtype; a.pad = (long long)c->pad; a.nv = (long long)c->nv;
    a.y = c->y; a.y_pitch = (long long)c->y_pitch; a.out_mode = c->out_mode;
    a.table = c->d_table; a.sections = (int)c->sections; a.phi = c->d_phi;
    a.zi = c->zi; a.zi_sstride = (long long)c->zi_sstride; a.zi_rstride = (long long)c->zi_rstride;
    a.zi_scale_first = c->zi_scale_first;
    a.zf = c->zf; a.zf_sstride = (long long)c->zf_sstride;
    a.seg = c->d_seg;
    a.segment = (long long)c->segment;
    a.segs = (a.nv + a.segment - 1) / a.segment;
    const long long batch = (long long)c->batch;
    const int sms = rt_num_sms();
    if (a.segs > 1) {
        if (!c->d_seg || !c->d_phi) return fail(1, "vvb_iir_sos", "segment scratch");
        a.count = batch * (a.segs - 1);               /* A: end states of every segment but the last, from zero */
        if (int st = tu_iir('A', a, sms, stream)) return st;
        a.count = batch;                              /* B: the true entering state of every segment */
        if (int st = tu_iir('B', a, sms, stream)) return st;
    }
    a.count = batch * a.segs;                         /* C: every segment from its entering state */
    return tu_iir('C', a, sms, stream);
}

/* ---------------------------------------------------------------------- Bluestein plumbing */
static void chirp_destroy(Chirp* c)
{
    if (!c) return;
    vvb_free(c->d_chirp); vvb_free(c->d_bspec); vvb_free(c->d_bspec_m); vvb_free(c->d_tables); vvb_free(c->d_work);
    vvb_fft_engine_destroy(c->fwd); vvb_fft_engine_destroy(c->bwd);
    delete c;
}

static int chirp_create(size_t n, Chirp** out)
{
    *out = nullptr;
    Chirp* c = new (std::nothrow) Chirp();
    if (!c) return fail(4, "chirp_create", "oom");
    c->n = n;
    c->M = 128;
    while (c->M < 2 * n - 1) c->M *= 2;
    const size_t M = c->M;
    /* chirp in double with the exponent reduced mod 2n; spectrum of the wrapped conjugate chirp by a direct
     * double-precision DFT (M * (2n-1) terms, once per plan) */
    std::vector<double> cr(n), ci(n), twr(M), twi(M);
    std::vector<float> chirp(2 * n), bspec(2 * M);
    for (size_t i = 0; i < n; ++i) {
        const double ang = M_PI * (double)((i * i) % (2 * n)) / (double)n;
        cr[i] = cos(ang); ci[i] = -sin(ang);
        chirp[2 * i] = (float)cr[i]; chirp[2 * i + 1] = (float)ci[i];
    }
    for (size_t j = 0; j < M; ++j) { const double ang = 2.0 * M_PI * (double)j / (double)M; twr[j] = cos(ang); twi[j] = -sin(ang); }
    if (M <= 8192) {
        for (size_t k = 0; k < M; ++k) {
            double sr = cr[0], si = -ci[0];                      /* b[0] = conj(c[0]) = 1 */
            for (size_t i = 1; i < n; ++i) {
                /* b[i] = b[M-i] = conj(c[i]):  b[i] (W^{ki} + W^{-ki}) = 2 b[i] cos(2 pi k i / M) */
                const double w = 2.0 * twr[(k * i) % M];
                sr += cr[i] * w; si += -ci[i] * w;
            }
            bspec[2 * k] = (float)sr; bspec[2 * k + 1] = (float)si;
        }
    } else {
        /* large sizes: the same spectrum by a double-precision radix-2 FFT on the host (M log M instead of M n terms) */
        std::vector<double> br(M, 0.0), bi(M, 0.0);
        br[0] = cr[0]; bi[0] = -ci[0];
        for (size_t i = 1; i < n; ++i) { br[i] = br[M - i] = cr[i]; bi[i] = bi[M - i] = -ci[i]; }
        for (size_t i = 1, j = 0; i < M; ++i) {                  /* bit reversal */
            size_t bit = M >> 1;
            for (; j & bit; bit >>= 1) j ^= bit;
            j ^= bit;
            if (i < j) { std::swap(br[i], br[j]); std::swap(bi[i], bi[j]); }
        }
        for (size_t len = 2; len <= M; len <<= 1) {
            const size_t half = len >> 1, step = M / len;
            for (size_t base = 0; base < M; base += len)
                for (size_t q = 0; q < half; ++q) {
                    const double wr = twr[q * step], wi = twi[q * step];
                    const size_t u = base + q, v = u + half;
                    const double xr = br[v] * wr - bi[v] * wi, xi = br[v] * wi + bi[v] * wr;
                    br[v] = br[u] - xr; bi[v] = bi[u] - xi;
                    br[u] += xr; bi[u] += xi;
                }
        }
        for (size_t k = 0; k < M; ++k) { bspec[2 * k] = (float)br[k]; bspec[2 * k + 1] = (float)bi[k]; }
    }
    int st = upload((float**)&c->d_chirp, chirp);
    if (!st) st = upload((float**)&c->d_bspec, bspec);
    c->fused = M <= 8192 && getenv("VVB_BLUESTEIN_UNFUSED") == nullptr;     /* beyond 8192 the M-point transforms are four-step plans */
    if (!st && c->fused) {
        std::vector<float> bm(bspec), blob;
        for (auto& v : bm) v = (float)((double)v / (double)M);
        st = upload((float**)&c->d_bspec_m, bm);
        build_c2c_tables(M, blob);
        if (!st) st = upload(&c->d_tables, blob);
    }
    if (!st) st = vvb_fft_engine_create(M, 0, +1, &c->fwd);
    if (!st) st = vvb_fft_engine_create(M, 0, -1, &c->bwd);
    if (st) { chirp_destroy(c); return st; }
    *out = c;
    return 0;
}

/* work buffer for up to `transforms` transforms, bounded at 256 MB: *chunk = transforms per pass */
static int chirp_reserve(Chirp* c, size_t transforms, size_t* chunk)
{
    const size_t cap = ((size_t)256 << 20) / (c->M * sizeof(float2));
    size_t want = std::min(transforms, std::max<size_t>(cap, 1));
    if (want == 0) want = 1;
    if (c->work_elems < want * c->M) {
        vvb_free(c->d_work); c->d_work = nullptr; c->work_elems = 0;
        if (int st = vvb_malloc((void**)&c->d_work, want * c->M * sizeof(float2))) return st;
        c->work_elems = want * c->M;
    }
    *chunk = c->work_elems / c->M;
    return 0;
}

/* work <- IFFT_M(FFT_M(work) * bspec), in place, `count` transforms */
static int chirp_convolve(Chirp* c, size_t count, void* stream)
{
    if (int st = vvb_fft_exec(c->fwd, c->d_work, c->d_work, count, stream)) return st;
    VVB_LAUNCH(chirp_mul_kernel, persistent_grid(((long long)count * (long long)c->M + 255) / 256, 8, rt_num_sms()), 256, 0, stream,
               c->d_work, c->d_bspec, (long long)count, (int)c->M);
    return vvb_fft_exec(c->bwd, c->d_work, c->d_work, count, stream);
}

static int chirp_fused(Chirp* c, ChirpFusedArgs a, int sms, void* stream)
{
    a.n = (int)c->n; a.chirp = c->d_chirp; a.bspec_over_m = c->d_bspec_m; a.tables = c->d_tables;
    return tu_chirp_fused(c->M, a, sms, stream);
}

/* ---------------------------------------------------------------------- log-mel */
#ifndef VVB_MEL_FPT
#define VVB_MEL_FPT 1                 /* frames per thread of logmel_tma_kernel: 1 = 16 warps per CTA (measured 9 % faster), 2 = 8 warps */
#endif
template <int R> static int launch_logmel_tma(const MelArgs& a, int grid, size_t smem, int stages, int stage_floats, int n_groups, void* stream)
{
    static OccCache occ;                                   /* per device and dynamic shared-memory size */
    if (occ.get(logmel_tma_kernel<R, VVB_MEL_FPT>, 256 * (2 / VVB_MEL_FPT), smem) == 0) return fail(4, "logmel_tma_kernel", "does not fit on this device");
    VVB_LAUNCH((logmel_tma_kernel<R, VVB_MEL_FPT>), grid, 256 * (2 / VVB_MEL_FPT), smem, stream, a, stages, stage_floats, n_groups);
    return 0;
}

extern "C" int vvb_logmel(const float* d_power, size_t frames, size_t bins, size_t power_pitch, const int* d_meta, const float* d_w,
                          size_t n_mels, size_t n_groups, float eps, float* d_out, void* stream)
{
    if (!d_power || !d_meta || !d_w || !d_out) return fail(1, "vvb_logmel", "null");
    if (frames == 0 || n_mels == 0) return 0;
    if (bins > 0x7fffffffu || n_mels > 0x7fffffffu) return fail(2, "vvb_logmel", "size");
#ifndef VVB_EMU
    if (int st = vvb_device_ready()) return st;
#endif
    MelArgs a;
    a.power = d_power; a.pitch = (long long)power_pitch; a.frames = (long long)frames; a.bins = (int)bins; a.n_mels = (int)n_mels;
    a.meta = d_meta; a.w = d_w; a.eps = eps; a.out = d_out;
    /* densely packed, aligned rows: the TMA-fed kernel, with the largest frame tile that still leaves a
     * three-deep ring (then two, then one) inside 220 KB of shared memory */
    if (power_pitch == bins && ((uintptr_t)d_power & 15u) == 0 && n_mels <= MEL_TMA_MAX_MELS && n_groups > 0 &&
        n_groups <= 3072 && getenv("VVB_MEL_NO_TMA") == nullptr) {
        const size_t budget = 226 * 1024;
        for (int want = 3; want >= 1; --want) {
            for (int R = 32; R >= 4; R >>= 1) {
                const size_t stage_bytes = (size_t)R * bins * 4, fixed = MEL_HDR + n_groups * 32 + (size_t)R * (n_mels | 1) * 4 + 16;
                if (fixed + want * stage_bytes > budget) continue;
                int stages = (int)((budget - fixed) / stage_bytes);
                if (stages > 4) stages = 4;
                const size_t smem = fixed + (size_t)stages * stage_bytes;
                const long long tiles = (long long)((frames + R - 1) / R);
                const int grid = (int)std::min<long long>(tiles, rt_num_sms());
                const int sf = (int)(stage_bytes / 4);
                switch (R) {
                    case 32: return launch_logmel_tma<32>(a, grid, smem, stages, sf, (int)n_groups, stream);
                    case 16: return launch_logmel_tma<16>(a, grid, smem, stages, sf, (int)n_groups, stream);
                    case 8:  return launch_logmel_tma<8>(a, grid, smem, stages, sf, (int)n_groups, stream);
                    default: return launch_logmel_tma<4>(a, grid, smem, stages, sf, (int)n_groups, stream);
                }
            }
        }
    }
    static OccCache occ;
    const size_t smem = sizeof(float) * MEL_KC * 33;
    const int per_sm = occ.get(logmel_kernel, 256, smem);
    if (per_sm == 0) return fail(4, "logmel_kernel", "does not fit on this device");
    VVB_LAUNCH(logmel_kernel, persistent_grid((long long)((frames + 31) / 32), per_sm, rt_num_sms()), 256, smem, stream, a);
    return 0;
}

extern "C" int vvb_mfcc(const float* d_logmel, size_t frames, size_t n_mels, size_t n_coeffs, const float* d_table,
                        const float* d_lifter, float* d_out, void* stream)
{
    if (!d_logmel || !d_table || !d_lifter || !d_out) return fail(1, "vvb_mfcc", "null");
    if (frames == 0 || n_coeffs == 0) return 0;
    const size_t smem = sizeof(float) * (32 * (n_mels | 1) + n_coeffs * n_mels + 32 * (n_coeffs | 1));
    if (n_mels > 0x7fffffffu || smem > 200 * 1024) return fail(2, "vvb_mfcc", "n_mels x n_coeffs table does not fit in shared memory");
#ifndef VVB_EMU
    if (int st = vvb_device_ready()) return st;
#endif
    MfccArgs a;
    a.logmel = d_logmel; a.frames = (long long)frames; a.n_mels = (int)n_mels; a.n_coeffs = (int)n_coeffs;
    a.table = d_table; a.lifter = d_lifter; a.out = d_out;
    static OccCache occ;
    const int per_sm = occ.get(mfcc_kernel, 256, smem);
    if (per_sm == 0) return fail(4, "mfcc_kernel", "does not fit on this device");
    VVB_LAUNCH(mfcc_kernel, persistent_grid((long long)((frames + 31) / 32), per_sm, rt_num_sms()), 256, smem, stream, a);
    return 0;
}

extern "C" int vvb_pcm_to_planar(const void* d_interleaved, int format, size_t num_samples, size_t channels, float* d_planar,
                                 size_t pitch, void* stream)
{
    if (!d_interleaved || !d_planar) return fail(1, "vvb_pcm_to_planar", "null");
    if (num_samples == 0 || channels == 0) return 0;
    if (channels > 0x7fffffffu) return fail(2, "vvb_pcm_to_planar", "size");
#ifndef VVB_EMU
    if (int st = vvb_device_ready()) return st;
#endif
    PcmArgs a;
    a.in = (const unsigned char*)d_interleaved; a.format = format; a.num_samples = (long long)num_samples; a.channels = (int)channels;
    a.out = d_planar; a.pitch = (long long)pitch;
    const long long total = (long long)(num_samples * channels);
    const int grid = (int)std::min<long long>((total + 255) / 256, (long long)rt_num_sms() * 16);
    VVB_LAUNCH(pcm_to_planar_kernel, grid, 256, 0, stream, a);
    return 0;
}

/* ---------------------------------------------------------------- FP32 peak probe */
/* Measures the FP32 FMA throughput the roofline is quoted against: 16 independent dependent-FMA
 * chains per thread, scalar FFMA or packed FFMA2.  Diagnostics only (bench.py's roofline_fp32). */
template <bool PACKED> __global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters)
{
    float2 a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = make_float2(threadIdx.x * 1e-3f + i, 1.0f - i * 1e-2f);
    const float2 m = make_float2(0.999f, 1.001f), c = make_float2(1e-3f, -1e-3f);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if constexpr (PACKED) a[i] = __ffma2_rn(a[i], m, c);
                else { a[i].x = fmaf(a[i].x, m.x, c.x); a[i].y = fmaf(a[i].y, m.y, c.y); }
            }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += a[i].x + a[i].y;
    if (s == 123.456f) out[0] = s;
}

extern "C" int vvb_fp32_peak(int packed, double* tflops)
{
    if (!tflops) return fail(1, "vvb_fp32_peak", "null");
#ifdef VVB_EMU
    (void)packed; *tflops = 0.0; return 0;
#else
    if (int st = vvb_device_ready()) return st;
    float* d = nullptr;
    CK(cudaMalloc(&d, 4));
    const int iters = 4096, grid = rt_num_sms() * 8;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(e0));
        if (packed) fp32_peak_kernel<true><<<grid, 256>>>(d, iters); else fp32_peak_kernel<false><<<grid, 256>>>(d, iters);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = (double)grid * 256 * iters * 4 * 8 * 2 * 2;   /* 64 FMA lanes-ops per iteration, 2 flop each */
        if (rep > 0 && flops / (ms * 1e-3) / 1e12 > best) best = flops / (ms * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops = best;
    return 0;
#endif
}

/* ---------------------------------------------------------------- halo gather (one stream over several GPUs) */
/* The two sample halos of a frame-range shard, fetched by the shard's OWN device with plain loads from its neighbours'
 * memory (peer access over NVLink; the same pointers work when both shards live on one device).  A kernel, not a
 * copy-engine transfer: 12 KB per halo is latency-, not bandwidth-bound, and a kernel node replays inside the step's
 * CUDA graph. */
__global__ void __launch_bounds__(256) halo_gather_kernel(float* dst_left, const float* src_left, float* dst_right, const float* src_right,
                                                        long long count)
{
    const float* src = blockIdx.y ? src_right : src_left;
    float* dst = blockIdx.y ? dst_right : dst_left;
    if (!src || !dst) return;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) dst[i] = src[i];
}

extern "C" int vvb_halo_gather(float* dst_left, const float* src_left, float* dst_right, const float* src_right, size_t count, void* stream)
{
    if (count == 0 || (!dst_left && !dst_right)) return 0;
    const int blocks = (int)std::min<size_t>((count + 255) / 256, 16);
    VVB_LAUNCH(halo_gather_kernel, dim3(blocks, 2), 256, 0, stream, dst_left, src_left, dst_right, src_right, (long long)count);
    return 0;
}

/* ---------------------------------------------------------------- SM clock probe */
/* One warp spins for ~50 us and reports SM cycles per nanosecond of the global timer: the SM clock the GPU is
 * ACTUALLY running at that moment (nvidia-smi samples every 100 ms and misses short excursions).  Diagnostics
 * for bench.py / benchmarks: lets a measurement say which clock it was taken at. */
__global__ void sm_clock_probe_kernel(double* out, long long spin_cycles)
{
#ifndef VVB_EMU
    unsigned long long g0, g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
    const long long c0 = clock64();
    long long c1 = c0;
    while (c1 - c0 < spin_cycles) c1 = clock64();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    if (threadIdx.x == 0) out[0] = (g1 > g0) ? (double)(c1 - c0) / (double)(g1 - g0) * 1000.0 : 0.0;
#else
    (void)spin_cycles; out[0] = 0.0;
#endif
}

extern "C" int vvb_sm_clock_mhz(void* stream, double* mhz)
{
    if (!mhz) return fail(1, "vvb_sm_clock_mhz", "null");
#ifdef VVB_EMU
    (void)stream; *mhz = 0.0; return 0;
#else
    if (int st = vvb_device_ready()) return st;
    static thread_local double* d_out = nullptr;
    static thread_local double* h_out = nullptr;
    if (!d_out) { CK(cudaMalloc(&d_out, sizeof(double))); CK(cudaMallocHost(&h_out, sizeof(double))); }
    sm_clock_probe_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_out, 100000);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h_out, d_out, sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    *mhz = *h_out;
    return 0;
#endif
}
