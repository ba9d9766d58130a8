/*
 * sos.c -- batched IIR filtering by second-order sections on the device: vv_dsp_sos_* of include/vv_dsp/b200.h (host,
 * C99).  This file validates the cascade, builds its tables in double once per handle (the scan matrices of every
 * section, the cascade's transition over one segment, sosfilt_zi), and stages HOST buffers in chunks of rows; the
 * arithmetic is iir_tile_kernel / iir_chain_kernel (csrc/cuda/vvb_iir_kernels.cuh).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

typedef char sos_tile_is_the_kernels[(VV_DSP_SOS_TILE == VVB_IIR_THREADS * VVB_IIR_RUN) ? 1 : -1];
typedef char sos_chain_fits[(2 * VV_DSP_SOS_MAX_SECTIONS <= 128) ? 1 : -1];

struct vv_dsp_sos {
    size_t sections, segment;
    size_t default_padlen;            /* scipy's 3 (2S + 1 - min(#{b2 == 0}, #{a2 == 0})) */
    handle_core core;
    double* d_table;                  /* [S][VVB_IIR_TABLE] */
    float* d_phi;                     /* [2S][2S] */
    float* d_zi_unit;                 /* [S][2]: sosfilt_zi(sos) */
    float* d_x;     size_t x_bytes;   /* signals staged from HOST */
    float* d_y;     size_t y_bytes;   /* output staged for HOST */
    float* d_fwd;   size_t fwd_bytes; /* filtfilt: the forward pass over the padded rows */
    float* d_seg;   size_t seg_bytes; /* segment states of long rows */
    float* d_zi;    size_t zi_bytes;  /* zi staged from HOST */
    float* d_zf;    size_t zf_bytes;  /* zf staged for HOST */
};

/* c = a b, n x n row-major; c may not alias a or b */
static void matmul(const double* a, const double* b, double* c, size_t n)
{
    size_t i, j, k;
    for (i = 0; i < n; ++i) {
        for (j = 0; j < n; ++j) c[i * n + j] = 0.0;
        for (k = 0; k < n; ++k) {
            const double aik = a[i * n + k];
            if (aik != 0.0) for (j = 0; j < n; ++j) c[i * n + j] += aik * b[k * n + j];
        }
    }
}

/* m = a^e by binary exponentiation, n x n; returns 0, or 4 when out of memory */
static int matpow(const double* a, size_t e, double* m, size_t n)
{
    double* base = (double*)malloc(n * n * sizeof(double));
    double* tmp = (double*)malloc(n * n * sizeof(double));
    size_t i;
    if (!base || !tmp) { free(base); free(tmp); return 4; }
    memcpy(base, a, n * n * sizeof(double));
    for (i = 0; i < n * n; ++i) m[i] = (i % (n + 1)) == 0 ? 1.0 : 0.0;
    while (e) {
        if (e & 1) { matmul(m, base, tmp, n); memcpy(m, tmp, n * n * sizeof(double)); }
        e >>= 1;
        if (e) { matmul(base, base, tmp, n); memcpy(base, tmp, n * n * sizeof(double)); }
    }
    free(base); free(tmp);
    return 0;
}

/* the tables of one handle, in double from the float32 coefficients: the scan matrices stay double (the scan runs in
 * float64), Phi and sosfilt_zi are rounded to float32 once */
static int build_tables(const float* sos, size_t S, size_t segment, double* table, float* phi, float* zi_unit)
{
    const size_t n2 = 2 * S;
    double* step = (double*)calloc(n2 * n2, sizeof(double));
    double* big = (double*)malloc(n2 * n2 * sizeof(double));
    double scale = 1.0;
    size_t s, k, d;
    int st = 0;
    if (!step || !big) st = 4;
    for (s = 0; s < S && !st; ++s) {
        const double b0 = sos[6 * s], b1 = sos[6 * s + 1], b2 = sos[6 * s + 2], a1 = sos[6 * s + 4], a2 = sos[6 * s + 5];
        const double A[4] = { -a1, 1.0, -a2, 0.0 };
        double m[4], t[4];
        double* row = table + s * VVB_IIR_TABLE;
        row[0] = b0; row[1] = b1; row[2] = b2; row[3] = a1; row[4] = a2;
        row[5] = row[6] = row[7] = 0.0;
        matpow(A, VVB_IIR_RUN, m, 2);                 /* A^L, then squared once per level: A^(L 2^d) */
        for (d = 0; d < VVB_IIR_LEVELS; ++d) {
            for (k = 0; k < 4; ++k) row[8 + 4 * d + k] = m[k];
            matmul(m, m, t, 2);
            memcpy(m, t, sizeof(m));
        }
        {   /* sosfilt_zi: lfilter_zi of the section, (I - A) zi = (b1 - a1 b0, b2 - a2 b0), times the DC gain before it */
            const double B0 = b1 - a1 * b0, B1 = b2 - a2 * b0, det = 1.0 + a1 + a2;
            zi_unit[2 * s] = (float)(scale * (B0 + B1) / det);
            zi_unit[2 * s + 1] = (float)(scale * ((1.0 + a1) * B1 - a2 * B0) / det);
            scale *= (b0 + b1 + b2) / det;
        }
    }
    /* one step of the whole cascade with zero input: column k is the response to the unit state e_k */
    for (k = 0; k < n2 && !st; ++k) {
        double u = 0.0;
        for (s = 0; s < S; ++s) {
            const double b0 = sos[6 * s], b1 = sos[6 * s + 1], b2 = sos[6 * s + 2], a1 = sos[6 * s + 4], a2 = sos[6 * s + 5];
            const double z0 = (k == 2 * s) ? 1.0 : 0.0, z1 = (k == 2 * s + 1) ? 1.0 : 0.0;
            const double y = b0 * u + z0;
            step[(2 * s) * n2 + k] = b1 * u - a1 * y + z1;
            step[(2 * s + 1) * n2 + k] = b2 * u - a2 * y;
            u = y;
        }
    }
    if (!st) st = matpow(step, segment, big, n2);
    if (!st) for (k = 0; k < n2 * n2; ++k) phi[k] = (float)big[k];
    free(step); free(big);
    return st;
}

static void sos_free(vv_dsp_sos* h)
{
    if (!h) return;
    vvb_free(h->d_table); vvb_free(h->d_phi); vvb_free(h->d_zi_unit);
    vvb_free(h->d_x); vvb_free(h->d_y); vvb_free(h->d_fwd); vvb_free(h->d_seg); vvb_free(h->d_zi); vvb_free(h->d_zf);
    vvdsp_internal_core_free(&h->core);
    free(h);
}

vv_dsp_status vv_dsp_sos_create(const vv_dsp_real* sos, size_t n_sections, vv_dsp_sos** out)
{
    vv_dsp_sos* h;
    size_t s, zb2 = 0, za2 = 0;
    int st;
    if (!out) return VV_DSP_ERROR_NULL_POINTER;
    *out = NULL;
    if (!sos) return VV_DSP_ERROR_NULL_POINTER;
    if (n_sections < 1 || n_sections > VV_DSP_SOS_MAX_SECTIONS) return VV_DSP_ERROR_INVALID_SIZE;
    for (s = 0; s < 6 * n_sections; ++s)
        if (!isfinite(sos[s])) return VV_DSP_ERROR_NAN_INF;
    for (s = 0; s < n_sections; ++s) {
        const double a1 = sos[6 * s + 4], a2 = sos[6 * s + 5];
        if (sos[6 * s + 3] != 1.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
        /* both roots of z^2 + a1 z + a2 strictly inside the unit circle (the stability triangle) */
        if (!(fabs(a2) < 1.0 && fabs(a1) < 1.0 + a2)) return VV_DSP_ERROR_OUT_OF_RANGE;
        zb2 += sos[6 * s + 2] == 0.0f;
        za2 += a2 == 0.0;
    }
    h = (vv_dsp_sos*)calloc(1, sizeof(*h));
    if (!h) return VV_DSP_ERROR_INTERNAL;
    h->sections = n_sections;
    h->default_padlen = 3 * (2 * n_sections + 1 - (zb2 < za2 ? zb2 : za2));
    h->segment = VV_DSP_SOS_SEGMENT;
    {   /* a short segment lets a small row span several (tests); rounded up to a whole number of tiles */
        const char* env = getenv("VVB_IIR_SEGMENT");
        if (env && atol(env) > 0) h->segment = ((size_t)atol(env) + VV_DSP_SOS_TILE - 1) / VV_DSP_SOS_TILE * VV_DSP_SOS_TILE;
    }
    st = vvdsp_internal_core_init(&h->core);
    if (!st) {
        const size_t S = n_sections, nt = S * VVB_IIR_TABLE, np = 4 * S * S;
        double* table = (double*)malloc(nt * sizeof(double));
        float* phi = (float*)malloc(np * sizeof(float));
        float* zi = (float*)malloc(2 * S * sizeof(float));
        st = (!table || !phi || !zi) ? 4 : build_tables(sos, S, h->segment, table, phi, zi);
        if (!st) st = vvb_malloc((void**)&h->d_table, nt * sizeof(double));
        if (!st) st = vvb_malloc((void**)&h->d_phi, np * sizeof(float));
        if (!st) st = vvb_malloc((void**)&h->d_zi_unit, 2 * S * sizeof(float));
        if (!st) st = vvb_memcpy_h2d(h->d_table, table, nt * sizeof(double), h->core.stream);
        if (!st) st = vvb_memcpy_h2d(h->d_phi, phi, np * sizeof(float), h->core.stream);
        if (!st) st = vvb_memcpy_h2d(h->d_zi_unit, zi, 2 * S * sizeof(float), h->core.stream);
        if (!st) st = vvb_stream_sync(h->core.stream);
        free(table); free(phi); free(zi);
    }
    if (st) { sos_free(h); return st == 6 ? VV_DSP_ERROR_UNSUPPORTED : VV_DSP_ERROR_INTERNAL; }
    *out = h;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_sos_destroy(vv_dsp_sos* h)
{
    int prev;
    if (!h) return VV_DSP_ERROR_NULL_POINTER;
    prev = vvdsp_internal_enter(&h->core);
    sos_free(h);
    vvdsp_internal_leave(prev);
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_sos_set_stream(vv_dsp_sos* h, void* cuda_stream)
{
    return vvdsp_internal_set_stream(h ? &h->core : NULL, cuda_stream);
}

vv_dsp_status vv_dsp_sos_synchronize(vv_dsp_sos* h)
{
    return vvdsp_internal_synchronize(h ? &h->core : NULL);
}

vv_dsp_status vv_dsp_sos_get_config(const vv_dsp_sos* h, size_t* n_sections, size_t* segment_length)
{
    if (!h || !n_sections || !segment_length) return VV_DSP_ERROR_NULL_POINTER;
    *n_sections = h->sections;
    *segment_length = h->segment;
    return VV_DSP_OK;
}

/* the segment-state scratch of nb rows of nv samples (none when a row fits one segment) */
static int reserve_segments(vv_dsp_sos* h, size_t nb, size_t nv)
{
    const size_t segs = (nv + h->segment - 1) / h->segment;
    if (segs < 2) return 0;
    return vvdsp_internal_reserve(&h->core, (void**)&h->d_seg, &h->seg_bytes, nb * segs * 2 * h->sections * sizeof(float));
}

static void call_init(const vv_dsp_sos* h, vvb_iir_call* c)
{
    memset(c, 0, sizeof(*c));
    c->d_table = h->d_table; c->d_phi = h->d_phi; c->sections = h->sections; c->segment = h->segment;
    c->d_seg = h->d_seg;
}

static int bad_space(vv_dsp_mem_space s) { return (unsigned)s > 1u; }

/* zf = zi, or zeros, for every row: the filter of an empty signal */
static int pass_state(vv_dsp_sos* h, const vv_dsp_real* zi, vv_dsp_mem_space zi_space, vv_dsp_real* zf,
                      vv_dsp_mem_space zf_space, size_t batch)
{
    const size_t bytes = 2 * h->sections * batch * sizeof(float);
    int st = 0;
    if (!zf || (const void*)zf == (const void*)zi) return 0;
    if (!zi) st = zf_space == VV_DSP_MEM_HOST ? (memset(zf, 0, bytes), 0) : vvb_memset(zf, 0, bytes, h->core.stream);
    else if (zi_space == VV_DSP_MEM_HOST && zf_space == VV_DSP_MEM_HOST) memcpy(zf, zi, bytes);
    else if (zi_space == VV_DSP_MEM_HOST) st = vvb_memcpy_h2d(zf, zi, bytes, h->core.stream);
    else if (zf_space == VV_DSP_MEM_HOST) st = vvb_memcpy_d2h(zf, zi, bytes, h->core.stream);
    else st = vvb_memcpy2d_d2d(zf, bytes, zi, bytes, bytes, 1, h->core.stream);
    if (!st && (zi_space == VV_DSP_MEM_HOST || zf_space == VV_DSP_MEM_HOST)) st = vvb_stream_sync(h->core.stream);
    return st;
}

static int filter_impl(vv_dsp_sos* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n,
                       size_t signal_pitch, const vv_dsp_real* zi, vv_dsp_mem_space zi_space, vv_dsp_real* zf,
                       vv_dsp_mem_space zf_space, vv_dsp_real* out, vv_dsp_mem_space out_space, size_t out_pitch)
{
    const size_t S = h->sections, row_bytes = n * sizeof(float), state_row = 2 * S * sizeof(float);
    const size_t x_per = signals_space == VV_DSP_MEM_HOST ? row_bytes : 0;
    const size_t y_per = out_space == VV_DSP_MEM_HOST ? row_bytes : 0;
    const int zi_host = zi && zi_space == VV_DSP_MEM_HOST, zf_host = zf && zf_space == VV_DSP_MEM_HOST;
    const int any_host = x_per || y_per || zi_host || zf_host;
    const size_t cs = vvdsp_internal_chunk_rows(&h->core, batch, x_per > y_per ? x_per : y_per);
    size_t done;
    int st = 0;
    if (x_per) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_x, &h->x_bytes, cs * x_per);
    if (!st && y_per) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_y, &h->y_bytes, cs * y_per);
    if (!st && zi_host) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_zi, &h->zi_bytes, cs * state_row);
    if (!st && zf_host) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_zf, &h->zf_bytes, cs * state_row);
    if (!st) st = reserve_segments(h, cs, n);
    /* every chunk runs on the handle's stream, so stream order keeps the scratch buffers of consecutive chunks apart */
    for (done = 0; done < batch && !st; done += cs) {
        const size_t nb = batch - done < cs ? batch - done : cs;
        vvb_iir_call c;
        call_init(h, &c);
        c.x = signals + done * signal_pitch; c.x_pitch = signal_pitch; c.n = n; c.nv = n; c.in_mode = VVB_IIR_IN_PLAIN;
        c.y = out + done * out_pitch; c.y_pitch = out_pitch; c.out_mode = VVB_IIR_OUT_DIRECT;
        c.batch = nb;
        if (x_per) {
            st = vvb_memcpy2d_h2d(h->d_x, row_bytes, c.x, signal_pitch * sizeof(float), row_bytes, nb, h->core.stream);
            c.x = h->d_x; c.x_pitch = n;
        }
        if (y_per) { c.y = h->d_y; c.y_pitch = n; }
        if (zi) {                                     /* [S][batch][2]: the chunk's rows of every section */
            c.zi = zi + 2 * done; c.zi_sstride = 2 * batch; c.zi_rstride = 2;
            if (zi_host && !st) {
                st = vvb_memcpy2d_h2d(h->d_zi, 2 * nb * sizeof(float), c.zi, 2 * batch * sizeof(float), 2 * nb * sizeof(float),
                                      S, h->core.stream);
                c.zi = h->d_zi; c.zi_sstride = 2 * nb;
            }
        }
        if (zf) {
            c.zf = zf_host ? h->d_zf : zf + 2 * done;
            c.zf_sstride = zf_host ? 2 * nb : 2 * batch;
        }
        if (!st) st = vvb_iir_sos(&c, h->core.stream);
        if (!st && y_per)
            st = vvb_memcpy2d_d2h(out + done * out_pitch, out_pitch * sizeof(float), h->d_y, row_bytes, row_bytes, nb,
                                  h->core.stream);
        if (!st && zf_host)
            st = vvb_memcpy2d_d2h(zf + 2 * done, 2 * batch * sizeof(float), h->d_zf, 2 * nb * sizeof(float),
                                  2 * nb * sizeof(float), S, h->core.stream);
    }
    return vvdsp_internal_finish(&h->core, st, any_host);
}

vv_dsp_status vv_dsp_sos_filter_batch(vv_dsp_sos* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch,
                                      size_t n, size_t signal_pitch, const vv_dsp_real* zi, vv_dsp_mem_space zi_space,
                                      vv_dsp_real* zf, vv_dsp_mem_space zf_space, vv_dsp_real* out,
                                      vv_dsp_mem_space out_space, size_t out_pitch)
{
    int prev, st;
    if (!h || !signals || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (bad_space(signals_space) || bad_space(out_space) || (zi && bad_space(zi_space)) || (zf && bad_space(zf_space)))
        return VV_DSP_ERROR_OUT_OF_RANGE;
    if (signal_pitch == 0) signal_pitch = n;
    if (out_pitch == 0) out_pitch = n;
    if (signal_pitch < n || out_pitch < n) return VV_DSP_ERROR_INVALID_SIZE;
    if ((const void*)out == (const void*)signals) return VV_DSP_ERROR_UNSUPPORTED;      /* no in-place filtering */
    if (batch == 0) return VV_DSP_OK;
    prev = vvdsp_internal_enter(&h->core);
    st = n == 0 ? pass_state(h, zi, zi_space, zf, zf_space, batch)
                : filter_impl(h, signals, signals_space, batch, n, signal_pitch, zi, zi_space, zf, zf_space, out, out_space,
                              out_pitch);
    vvdsp_internal_leave(prev);
    return vvdsp_internal_status(st);
}

static int filtfilt_impl(vv_dsp_sos* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n,
                         size_t signal_pitch, int padtype, size_t pad, vv_dsp_real* out, vv_dsp_mem_space out_space,
                         size_t out_pitch)
{
    const size_t nv = n + 2 * pad, row_bytes = n * sizeof(float);
    const size_t x_per = signals_space == VV_DSP_MEM_HOST ? row_bytes : 0;
    const size_t y_per = out_space == VV_DSP_MEM_HOST ? row_bytes : 0;
    const size_t cs = vvdsp_internal_chunk_rows(&h->core, batch, x_per > y_per ? x_per : y_per);
    size_t done;
    int st = 0;
    if (x_per) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_x, &h->x_bytes, cs * x_per);
    if (!st && y_per) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_y, &h->y_bytes, cs * y_per);
    if (!st) st = vvdsp_internal_reserve(&h->core, (void**)&h->d_fwd, &h->fwd_bytes, cs * nv * sizeof(float));
    if (!st) st = reserve_segments(h, cs, nv);
    for (done = 0; done < batch && !st; done += cs) {
        const size_t nb = batch - done < cs ? batch - done : cs;
        vvb_iir_call c;
        const float* x = signals + done * signal_pitch;
        size_t xp = signal_pitch;
        if (x_per) {
            st = vvb_memcpy2d_h2d(h->d_x, row_bytes, x, signal_pitch * sizeof(float), row_bytes, nb, h->core.stream);
            x = h->d_x; xp = n;
        }
        /* forward over the padded rows, from sosfilt_zi x_ext[0], into the scratch */
        call_init(h, &c);
        c.x = x; c.x_pitch = xp; c.n = n; c.in_mode = VVB_IIR_IN_EXT; c.padtype = padtype; c.pad = pad; c.nv = nv;
        c.y = h->d_fwd; c.y_pitch = nv; c.out_mode = VVB_IIR_OUT_DIRECT;
        c.zi = h->d_zi_unit; c.zi_sstride = 2; c.zi_rstride = 0; c.zi_scale_first = 1;
        c.batch = nb;
        if (!st) st = vvb_iir_sos(&c, h->core.stream);
        /* backward over the reversed scratch, from sosfilt_zi y_fwd[last], reversed again and trimmed into out */
        c.x = h->d_fwd; c.x_pitch = nv; c.in_mode = VVB_IIR_IN_REV;
        c.y = y_per ? h->d_y : out + done * out_pitch; c.y_pitch = y_per ? n : out_pitch; c.out_mode = VVB_IIR_OUT_REVTRIM;
        if (!st) st = vvb_iir_sos(&c, h->core.stream);
        if (!st && y_per)
            st = vvb_memcpy2d_d2h(out + done * out_pitch, out_pitch * sizeof(float), h->d_y, row_bytes, row_bytes, nb,
                                  h->core.stream);
    }
    return vvdsp_internal_finish(&h->core, st, x_per || y_per);
}

vv_dsp_status vv_dsp_sos_filtfilt_batch(vv_dsp_sos* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space,
                                        size_t batch, size_t n, size_t signal_pitch, int padtype, size_t padlen,
                                        vv_dsp_real* out, vv_dsp_mem_space out_space, size_t out_pitch)
{
    int prev, st;
    size_t pad;
    if (!h || !signals || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (bad_space(signals_space) || bad_space(out_space) || padtype < VV_DSP_PAD_NONE || padtype > VV_DSP_PAD_CONSTANT)
        return VV_DSP_ERROR_OUT_OF_RANGE;
    if (signal_pitch == 0) signal_pitch = n;
    if (out_pitch == 0) out_pitch = n;
    if (signal_pitch < n || out_pitch < n) return VV_DSP_ERROR_INVALID_SIZE;
    /* scipy's _validate_pad: no padding for padtype None, and the signal must be longer than the padding */
    pad = padtype == VV_DSP_PAD_NONE ? 0 : padlen == (size_t)-1 ? h->default_padlen : padlen;
    if (n > 0 && n <= pad) return VV_DSP_ERROR_INVALID_SIZE;
    if ((const void*)out == (const void*)signals) return VV_DSP_ERROR_UNSUPPORTED;
    if (batch == 0 || n == 0) return VV_DSP_OK;
    prev = vvdsp_internal_enter(&h->core);
    st = filtfilt_impl(h, signals, signals_space, batch, n, signal_pitch, padtype, pad, out, out_space, out_pitch);
    vvdsp_internal_leave(prev);
    return vvdsp_internal_status(st);
}
