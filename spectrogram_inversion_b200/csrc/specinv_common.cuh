// Shared device/host helpers for the specinv_b200 kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/specinv_b200.h"

namespace specinv {

template <typename T> struct cx_of;
template <> struct cx_of<float> { using type = float2; };
template <> struct cx_of<double> { using type = double2; };
template <typename T> using cx_t = typename cx_of<T>::type;

template <typename T> __host__ __device__ __forceinline__ cx_t<T> mk(T re, T im) {
    cx_t<T> r; r.x = re; r.y = im; return r;
}
template <typename C> __device__ __forceinline__ C cadd(C a, C b) { a.x += b.x; a.y += b.y; return a; }
template <typename C> __device__ __forceinline__ C csub(C a, C b) { a.x -= b.x; a.y -= b.y; return a; }
template <typename C> __device__ __forceinline__ C cmul(C a, C b) {
    C r; r.x = a.x * b.x - a.y * b.y; r.y = a.x * b.y + a.y * b.x; return r;
}
// a * conj(b)
template <typename C> __device__ __forceinline__ C cmulc(C a, C b) {
    C r; r.x = a.x * b.x + a.y * b.y; r.y = a.y * b.x - a.x * b.y; return r;
}
// a * (-i)
template <typename C> __device__ __forceinline__ C mul_mi(C a) { C r; r.x = a.y; r.y = -a.x; return r; }
// a * (+i)
template <typename C> __device__ __forceinline__ C mul_pi(C a) { C r; r.x = -a.y; r.y = a.x; return r; }

__device__ __forceinline__ float fast_sqrt(float v) { return sqrtf(v); }
__device__ __forceinline__ double fast_sqrt(double v) { return sqrt(v); }

// Projection onto the magnitude constraint, methods.py:246-247: q * mag / (|q| + 1e-16).
// |q| == 0 gives 0 (not NaN) exactly like the reference.
template <typename T> __device__ __forceinline__ cx_t<T> project(cx_t<T> q, T mag) {
    T r = fast_sqrt(q.x * q.x + q.y * q.y);
    T s = mag / (r + T(1e-16));
    return mk<T>(q.x * s, q.y * s);
}
// fp32: q * mag * rsqrt(|q|^2 + 1e-32), the form the specialised kernels use (one MUFU op instead of an IEEE square root
// and an IEEE division: ~15 instructions less per bin in the instruction-bound generic kernels).  Identical up to
// rounding (2 ulp) unless |q| ~ 1e-16; |q| == 0 still gives 0.
template <> __device__ __forceinline__ float2 project<float>(float2 q, float mag) {
    const float s = mag * rsqrtf(fmaf(q.x, q.x, fmaf(q.y, q.y, 1e-32f)));
    return mk<float>(q.x * s, q.y * s);
}

// Dimensions derived from a specinv_desc (host side and kernels share it).
struct Dims {
    int N;        // n_fft
    int M;        // N/2 (floor): size of the complex FFT used for the real transform; top bin of the half spectrum
    int logM;
    int pow2;     // n_fft is a power of two (FFT kernels); otherwise the direct-DFT tile kernel of specinv_generic.cu
    int hop;
    int T;        // frames
    int B;        // batch
    int P;        // one-sided centre padding (N/2 or 0)
    int K;        // halo frames = ceil(N/hop) - 1 = (N-1)/hop
    int pad_mode;
    int onesided;
    int row;      // main row length (M onesided, N two-sided)
    long long L;  // output samples per signal
    long long Lp; // padded length = (T-1)*hop + N
};

// Offsets (bytes) of the tables inside a plan buffer.
struct PlanLayout {
    size_t tw;       // M complex:  exp(-2 pi i j / M)
    size_t twr;      // M/2+1 complex: exp(-2 pi i k / N)
    size_t wa;       // N real: analysis window * forward scale
    size_t ws;       // N real: synthesis window * inverse scale
    size_t env;      // L real
    size_t inv_env;  // L real
    size_t total;
};

// Where one RTISI-LA launch reads its magnitudes and writes its samples (include/specinv_b200.h:
// specinv_rtisi_la_stream).  A whole-signal run is frame0 = 0, n_rows = T, x0 = 0, x_len = L, final = 1.
struct RtisiWindow {
    int frame0, n_rows;       // magnitude row r of a signal is spectrogram frame frame0 + r
    long long x0, x_len;      // x_out column c of a signal is output sample x0 + c; x_len is also the row stride
    const void* inv_env;      // 1/envelope of samples [x0, x0 + x_len), shared by the batch
    int final;                // n_frames is the total: zero magnitudes past it, the last frame flushes the carry
};

inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

inline int make_dims(const specinv_desc* d, Dims* o) {
    if (!d) return SPECINV_ERR_INVALID;
    const int N = d->n_fft;
    if (N < 16 || N > 32768) return SPECINV_ERR_INVALID;
    if ((N & 1) && d->onesided) return SPECINV_ERR_INVALID;   // an odd n_fft only exists two-sided (bin count = n_fft): direct DFT
    if (d->hop < 1 || d->hop > N) return SPECINV_ERR_INVALID;
    if (d->n_frames < 1 || d->batch < 1) return SPECINV_ERR_INVALID;
    if (d->dtype != SPECINV_F32 && d->dtype != SPECINV_F64) return SPECINV_ERR_INVALID;
    if (d->pad_mode < 0 || d->pad_mode > 3) return SPECINV_ERR_INVALID;
    o->N = N; o->M = N / 2; o->logM = ilog2(N / 2); o->hop = d->hop; o->T = d->n_frames; o->B = d->batch;
    o->pow2 = (N & (N - 1)) == 0;
    o->P = d->center ? N / 2 : 0;
    o->K = (N - 1) / d->hop;
    o->pad_mode = d->pad_mode;
    o->onesided = d->onesided ? 1 : 0;
    o->row = d->onesided ? N / 2 : N;
    o->Lp = (long long)(d->n_frames - 1) * d->hop + N;
    o->L = o->Lp - 2LL * o->P;
    if (o->L < 1) return SPECINV_ERR_INVALID;
    // reflect / circular padding need pad < L (torch.stft raises otherwise)
    if (d->center && (d->pad_mode == SPECINV_PAD_REFLECT || d->pad_mode == SPECINV_PAD_CIRCULAR) && o->P >= o->L)
        return SPECINV_ERR_INVALID;
    return SPECINV_OK;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Programmatic-dependent-launch guard (defined in specinv_api.cu).  The fused iteration kernels read the plan's
// window / twiddle tables in their prologue, BEFORE griddepcontrol.wait, i.e. possibly while the previous kernel of
// the stream is still running.  That is only safe when that previous kernel does not write those tables:
// `note_tables_launch(st)` records that the tables kernel was the library's latest launch on stream `st`,
// `note_other_launch(st)` that some other library kernel followed it, and `pdl_prologue_safe(st)` -- called by the
// iteration launchers -- returns false (launch fully serialised) in the first case and clears the mark.
void note_tables_launch(cudaStream_t st);
void note_other_launch(cudaStream_t st);
bool pdl_prologue_safe(cudaStream_t st);

inline PlanLayout plan_layout(const Dims& dm, int dtype) {
    const size_t es = dtype == SPECINV_F64 ? 8 : 4;
    PlanLayout p; size_t off = 0;
    // power of two: W_M^j, j < M (the M-point complex FFT); otherwise W_N^j, j < N (direct DFT)
    p.tw = off;      off = align_up(off + (size_t)(dm.pow2 ? dm.M : dm.N) * 2 * es, 256);
    p.twr = off;     off = align_up(off + (size_t)(dm.M / 2 + 1) * 2 * es, 256);
    p.wa = off;      off = align_up(off + (size_t)dm.N * es, 256);
    p.ws = off;      off = align_up(off + (size_t)dm.N * es, 256);
    p.env = off;     off = align_up(off + (size_t)dm.L * es, 256);
    p.inv_env = off; off = align_up(off + (size_t)dm.L * es, 256);
    p.total = off;
    return p;
}

// Map a position in the (centre-)padded signal to an index into x, or -1 for a zero sample.
// torch.stft pads n_fft//2 on both sides with pad_mode (torch/functional.py:676-679).
__device__ __forceinline__ long long pad_index(long long pp, int P, long long L, int pad_mode) {
    long long m = pp - P;
    if (m >= 0 && m < L) return m;
    switch (pad_mode) {
        case SPECINV_PAD_REFLECT:   return m < 0 ? -m : 2 * (L - 1) - m;
        case SPECINV_PAD_REPLICATE: return m < 0 ? 0 : L - 1;
        case SPECINV_PAD_CIRCULAR:  return m < 0 ? m + L : m - L;
        default:                    return -1;
    }
}

}  // namespace specinv
