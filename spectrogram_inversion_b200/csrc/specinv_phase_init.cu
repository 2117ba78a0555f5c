// One-shot kernels that run before the iteration loop, on the split frame-major layout:
//   * phase_init : the reference's simplified single-pass spectrogram inversion start
//                  (torch_specinv/methods.py:572-615), fused into ONE pass over the magnitude:
//                  strict spectral peaks along frequency (:597-598), parabolic interpolation (:604),
//                  instantaneous frequency (:605) assigned to the peak bin and its two neighbours with
//                  the reference's write order (:607-609: a peak at k-1 wins over a peak at k+1),
//                  running sum over time (:611) and C = mag * exp(i*phi) (:612-614).
//                  The reference does this with ~15 full-tensor PyTorch ops.
//   * spec_abs   : |C| for a complex initial estimate (methods.py:110).
#include "specinv_common.cuh"

namespace specinv {

template <typename T> __device__ __forceinline__ void sincos_t(T x, T* s, T* c);
// The running phase reaches 1e5..1e6 rad (omega = pi/2 * k per frame at hop = n_fft/4), ~5e8 rad after one hour at
// n_fft = 4096: far into the slow (Payne-Hanek) range of sincosf.  The float phase is exactly representable in double, so reduce it modulo 2 pi
// there (two-term 2 pi, error < 1e-10 rad) and take the fast path on the remainder.
template <> __device__ __forceinline__ void sincos_t<float>(float x, float* s, float* c) {
    const double xd = (double)x;
    const double n = rint(xd * 0.15915494309189533576888);
    double r = fma(-n, 6.283185307179586231996, xd);
    r = fma(-n, 2.449293598294706353906e-16, r);
    sincosf((float)r, s, c);
}
template <> __device__ __forceinline__ void sincos_t<double>(double x, double* s, double* c) { sincos(x, s, c); }

// magnitude of bin k (0..F-1) of frame row `fr`; out-of-range bins are never peaks
template <typename T>
__device__ __forceinline__ T mag_at(const T* __restrict__ main, const T* __restrict__ nyq, const Dims& dm, long long fr,
                                    int k) {
    if (dm.onesided && k == dm.M) return __ldg(nyq + fr);
    return __ldg(main + fr * dm.row + k);
}

// One thread per (signal, bin); it walks over time carrying the running phase.  A warp covers 30 consecutive
// bins plus one halo bin on each side: every lane tests ITS bin for a peak and interpolates its frequency once
// (one IEEE division), the two neighbours' results arrive by warp shuffle.  Consecutive lanes handle consecutive
// bins, so the loads / stores of a time step are coalesced in the frame-major layout.  (signal, 30-bin segment)
// pairs are numbered linearly over the warps so that the batched shapes fit one wave of resident blocks.
//
// Small batches do not have enough (signal, segment) pairs to fill the machine, so time is split into `chunks`
// ranges that run in parallel (MODE 1 / 2; MODE 0 is the single pass):
//   MODE 1: every (signal, segment, chunk) warp sums its chunk's phase advances (no output yet) and leaves the
//           double in the 8 / 16 output bytes of (first frame of the chunk, bin);
//   scan  : an exclusive scan over the chunks of every (signal, bin), in place;
//   MODE 2: the warp reads ITS start phase from that slot and then writes C for its frames (the slot is overwritten
//           by the first of them).
// The double accumulation is then associated per chunk instead of strictly left to right.  For float32 magnitudes
// that changes nothing: the omegas of one bin come from peaks at k-1 .. k+1 and lie within a factor 7 of each other,
// so every partial sum is a multiple of the smallest float ulp u among them and below 7 * 2^24 * T * u: exact in
// double for T < 2^26, and the chunked phase is bit-identical to the left-to-right sum.  In float64 the sums re-associate
// (<= T * 2^-53 * |phi|).
constexpr int PI_SEG = 30;

template <typename T>
__device__ __forceinline__ double* chunk_slot(const Dims& dm, cx_t<T>* c_main, cx_t<T>* c_nyq, long long fr, int k) {
    return reinterpret_cast<double*>((dm.onesided && k == dm.M) ? c_nyq + fr : c_main + fr * dm.row + k);
}

// POW2: n_fft is a power of two, where x * (1 / n_fft) IS the IEEE quotient x / n_fft (1 / n_fft is exact); the
// division costs 6 % of the kernel's time at cfg2 (1.73 vs 1.63 ms on a B200 at 1000 W), so it is only paid where
// it changes the result.
template <typename T, int MODE, bool POW2>
__global__ void __launch_bounds__(128) phase_init_kernel(Dims dm, int F, int segs, int chunks, int chunk_len, T hop,
                                                         T n_fft, const T* __restrict__ mag_main,
                                                         const T* __restrict__ mag_nyq, cx_t<T>* __restrict__ c_main,
                                                         cx_t<T>* __restrict__ c_nyq, const double* __restrict__ phase_in,
                                                         double* __restrict__ phase_out) {
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // global warp
    const int lane = threadIdx.x & 31;
    if (w >= (long long)dm.B * segs * chunks) return;                                  // whole warp
    const int chunk = (int)(w % chunks);
    const long long ws = w / chunks;
    const int b = (int)(ws / segs);
    const int k = (int)(ws - (long long)b * segs) * PI_SEG - 1 + lane;                 // lanes 0 and 31: halo bins
    const int ta = chunk * chunk_len, tb = min(dm.T, ta + chunk_len);                  // this warp's frames
    const bool in_spec = k >= 0 && k < F;
    const bool owner = in_spec && lane >= 1 && lane <= PI_SEG;
    const bool can_peak = k >= 1 && k <= F - 2;       // strict local maxima exist for 1 <= k <= F-2 only (:597-598)
    const T pi2 = (T)6.283185307179586476925286766559;
    const T inv_n_fft = T(1) / n_fft;                  // exact when POW2
    // torch's CPU cumsum accumulates float32 in float64 and rounds each output; phase_in (frame-range
    // sharding) is the phase accumulated by the frames before this range
    double phase = 0.0;
    if (MODE == 0) phase = (owner && phase_in) ? phase_in[(long long)b * F + k] : 0.0;
    if (MODE == 2 && owner) phase = *chunk_slot<T>(dm, c_main, c_nyq, (long long)b * dm.T + ta, k);
    // The running phase is the only loop-carried value: the loads of U consecutive frames are issued together.
    constexpr int U = 4;
    for (int t0 = ta; t0 < tb; t0 += U) {
        T m[U][3];                      // mag[k-1 .. k+1] of frames t0 .. t0+U-1
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long fr = (long long)b * dm.T + min(t0 + u, tb - 1);
            m[u][1] = in_spec ? mag_at(mag_main, mag_nyq, dm, fr, k) : T(0);
            m[u][0] = can_peak ? mag_at(mag_main, mag_nyq, dm, fr, k - 1) : T(0);
            m[u][2] = can_peak ? mag_at(mag_main, mag_nyq, dm, fr, k + 1) : T(0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (t0 + u < tb) {          // warp-uniform
                const long long fr = (long long)b * dm.T + t0 + u;
                const T lo = m[u][0], mid = m[u][1], hi = m[u][2];
                // own peak: interpolated angular frequency * hop (:604-605), or -1 (omega is never negative).
                // The operations and their order are the reference's: 2 pi * (k + p), an IEEE division by n_fft
                // (a multiplication by 1 / n_fft differs in the last bit when n_fft is not a power of two), * hop.
                T own = T(-1);
                if (can_peak && mid > hi && mid > lo) {
                    const T p = T(0.5) * (lo - hi) / (lo - T(2) * mid + hi);
                    own = POW2 ? pi2 * ((T)k + p) * inv_n_fft * hop : pi2 * ((T)k + p) / n_fft * hop;
                }
                const T up = __shfl_down_sync(0xffffffffu, own, 1);      // bin k + 1
                const T dn = __shfl_up_sync(0xffffffffu, own, 1);        // bin k - 1
                // reference write order: own peak, then peak at k+1 (writes k), then peak at k-1 (writes k): last wins
                T omega = T(0);
                if (own >= T(0)) omega = own;
                if (up >= T(0)) omega = up;
                if (dn >= T(0)) omega = dn;
                if (owner) {
                    phase += (double)omega;
                    if (MODE != 1) {
                        const T ph = (T)phase;
                        T sn, cs;
                        sincos_t<T>(ph, &sn, &cs);
                        const cx_t<T> v = mk<T>(mid * cs, mid * sn);
                        if (dm.onesided && k == dm.M) c_nyq[fr] = v;
                        else c_main[fr * dm.row + k] = v;
                    }
                }
            }
        }
    }
    if (MODE == 1) { if (owner) *chunk_slot<T>(dm, c_main, c_nyq, (long long)b * dm.T + ta, k) = phase; }
    else if (owner && phase_out && tb == dm.T) phase_out[(long long)b * F + k] = phase;
}

// exclusive scan of the chunk sums of every (signal, bin), in place, starting from phase_in
template <typename T>
__global__ void phase_scan_kernel(Dims dm, int F, int chunks, int chunk_len, cx_t<T>* c_main, cx_t<T>* c_nyq,
                                  const double* __restrict__ phase_in) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)dm.B * F) return;
    const int b = (int)(i / F), k = (int)(i - (long long)b * F);
    double run = phase_in ? phase_in[i] : 0.0;
    for (int c = 0; c < chunks; ++c) {
        double* slot = chunk_slot<T>(dm, c_main, c_nyq, (long long)b * dm.T + (long long)c * chunk_len, k);
        const double v = *slot;
        *slot = run;
        run += v;
    }
}

template <typename T>
__global__ void spec_abs_kernel(const cx_t<T>* __restrict__ c, T* __restrict__ m, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const cx_t<T> v = c[i];
        m[i] = hypot(v.x, v.y);      // torch's complex abs is hypot
    }
}

template <typename T, bool POW2>
static void phase_init_launch(const Dims& dm, int F, int segs, long long chunks, int chunk_len, long long blocks,
                              const T* mm, const T* mn, cx_t<T>* cm, cx_t<T>* cn, const double* phase_in,
                              double* phase_out, cudaStream_t st) {
    const T hop = (T)dm.hop, n_fft = (T)dm.N;
    if (chunks == 1) {
        phase_init_kernel<T, 0, POW2><<<(unsigned)blocks, 128, 0, st>>>(dm, F, segs, 1, dm.T, hop, n_fft, mm, mn, cm, cn,
                                                                        phase_in, phase_out);
    } else {
        phase_init_kernel<T, 1, POW2><<<(unsigned)blocks, 128, 0, st>>>(dm, F, segs, (int)chunks, chunk_len, hop, n_fft, mm,
                                                                        mn, cm, cn, nullptr, nullptr);
        const long long nbf = (long long)dm.B * F;
        phase_scan_kernel<T><<<(unsigned)((nbf + 127) / 128), 128, 0, st>>>(dm, F, (int)chunks, chunk_len, cm, cn, phase_in);
        phase_init_kernel<T, 2, POW2><<<(unsigned)blocks, 128, 0, st>>>(dm, F, segs, (int)chunks, chunk_len, hop, n_fft, mm,
                                                                        mn, cm, cn, nullptr, phase_out);
    }
}

template <typename T>
static int phase_init_t(const Dims& dm, const void* mag_main, const void* mag_nyq, void* c_main, void* c_nyq,
                        const double* phase_in, double* phase_out, cudaStream_t st) {
    const int F = dm.onesided ? dm.M + 1 : dm.N;
    const int segs = (F + PI_SEG - 1) / PI_SEG;
    // split time only when the (signal, segment) pairs leave more than half of the 148 x 64 warp slots idle (the
    // split costs a second pass over the magnitudes); chunks of at least 32 frames
    const long long pairs = (long long)dm.B * segs;
    long long chunks = (148LL * 64) / pairs;
    if (chunks > dm.T / 32) chunks = dm.T / 32;
    if (chunks < 1) chunks = 1;
    const int chunk_len = (int)((dm.T + chunks - 1) / chunks);
    chunks = (dm.T + chunk_len - 1) / chunk_len;
    const long long blocks = (pairs * chunks + 3) / 4;                  // 4 warps per block
    if (blocks > 0x7fffffffLL) return SPECINV_ERR_UNSUPPORTED;
    const T* mm = (const T*)mag_main; const T* mn = (const T*)mag_nyq;
    cx_t<T>* cm = (cx_t<T>*)c_main; cx_t<T>* cn = (cx_t<T>*)c_nyq;
    if ((dm.N & (dm.N - 1)) == 0)
        phase_init_launch<T, true>(dm, F, segs, chunks, chunk_len, blocks, mm, mn, cm, cn, phase_in, phase_out, st);
    else
        phase_init_launch<T, false>(dm, F, segs, chunks, chunk_len, blocks, mm, mn, cm, cn, phase_in, phase_out, st);
    return (int)cudaGetLastError();
}

template <typename T>
static int spec_abs_t(const Dims& dm, const void* c_main, const void* c_nyq, void* m_main, void* m_nyq, cudaStream_t st) {
    const long long n = (long long)dm.B * dm.T * dm.row;
    long long blocks = (n + 1023) / 1024;
    if (blocks > 148 * 16) blocks = 148 * 16;
    spec_abs_kernel<T><<<(unsigned)blocks, 256, 0, st>>>((const cx_t<T>*)c_main, (T*)m_main, n);
    if (dm.onesided) {
        const long long nn = (long long)dm.B * dm.T;
        spec_abs_kernel<T><<<(unsigned)((nn + 255) / 256 > 1184 ? 1184 : (nn + 255) / 256), 256, 0, st>>>(
            (const cx_t<T>*)c_nyq, (T*)m_nyq, nn);
    }
    return (int)cudaGetLastError();
}

}  // namespace specinv

using namespace specinv;

extern "C" {

int specinv_phase_init_ex(const specinv_desc* d, const void* mag_main, const void* mag_nyq, void* c_main, void* c_nyq,
                          const double* phase_in, double* phase_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!mag_main || !c_main || (dm.onesided && (!mag_nyq || !c_nyq))) return SPECINV_ERR_INVALID;
    return d->dtype == SPECINV_F64
               ? phase_init_t<double>(dm, mag_main, mag_nyq, c_main, c_nyq, phase_in, phase_out, (cudaStream_t)stream)
               : phase_init_t<float>(dm, mag_main, mag_nyq, c_main, c_nyq, phase_in, phase_out, (cudaStream_t)stream);
}

int specinv_phase_init(const specinv_desc* d, const void* mag_main, const void* mag_nyq, void* c_main, void* c_nyq,
                       void* stream) {
    return specinv_phase_init_ex(d, mag_main, mag_nyq, c_main, c_nyq, nullptr, nullptr, stream);
}

int specinv_spec_abs(const specinv_desc* d, const void* c_main, const void* c_nyq, void* mag_main, void* mag_nyq,
                     void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!mag_main || !c_main || (dm.onesided && (!mag_nyq || !c_nyq))) return SPECINV_ERR_INVALID;
    return d->dtype == SPECINV_F64 ? spec_abs_t<double>(dm, c_main, c_nyq, mag_main, mag_nyq, (cudaStream_t)stream)
                                   : spec_abs_t<float>(dm, c_main, c_nyq, mag_main, mag_nyq, (cudaStream_t)stream);
}

}  // extern "C"
