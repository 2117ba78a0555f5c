// RTISI-LA (real-time iterative spectrogram inversion with look-ahead), torch_specinv/methods.py:273-412,
// as ONE persistent kernel: a CTA owns one signal and keeps the whole sliding state on chip for all
// (T + LA) * max_iter inner iterations -- K kept frames, LA+1 active frames (which double as the FFT
// work space), the LA+1 momentum spectra, the partial overlap-add and the output carry.  HBM traffic is
// one read of the magnitudes per outer step and one write of the output signal; the reference issues
// ~20 PyTorch ops per inner iteration instead (dispatch bound, SURVEY.md section 3.5).
//
// Per inner iteration (methods.py:365-398):
//   y      = sum_f frame_f * (w * c) overlap-added at hop spacing, first K*hop samples dropped   (:365-370)
//   S[a]   = rfft(y[a*hop : a*hop+N] * w)   (last frame: asym_window1/2 when asymmetric)          (:371-385)
//   S     -= lr * pre   (j > 0);   S[a] -= lr * pre[a+1] for a < LA  (j == 0, i > 0)              (:387-392)
//   S      = S * mag[i+a] / (|S| + 1e-16);  active frames = irfft(S)                               (:394-398)
// After max_iter iterations the oldest active frame is committed (:401-404): it joins the kept ring and
// is overlap-added (window w, 1/envelope, centre trimming) into the output (:406-408, fused here).
// Frame / spectrum slots rotate by index ((a + i) mod (LA+1)), so "pre[a] <- pre[a+1]" and the slide of
// the active frames cost nothing.
#include <cstdlib>

#include "specinv_common.cuh"
#include "generic_fft.cuh"
#include "mixed_radix.cuh"

namespace specinv {

// implemented in specinv_rtisi_fast.cu; returns SPECINV_ERR_UNSUPPORTED when the shape is not its own
int rtisi_fast(const specinv_desc* d, const Dims& dm, const void* plan, const void* mag_main, const void* mag_nyq,
               void* x_out, const RtisiWindow& win, const void* asym1, const void* asym2, int look_ahead, int asymmetric,
               int max_iter, double alpha, double synth_coeff, int step_begin, int step_end, void* state, cudaStream_t st);

// Elements (of the real type) of the sliding state of ONE signal between two outer steps, the layout both kernels
// save / restore (include/specinv_b200.h: specinv_rtisi_la_steps): active frames [NA][N] (logical order, oldest
// first; the kernels' unscaled inverse-FFT samples), momentum spectra [NA][F] complex, kept frames [K][N] already
// multiplied by window * synth_coeff, output overlap-add carry [N].
size_t rtisi_state_elems(const Dims& dm, int LA) {
    const size_t NA = LA + 1, F = dm.onesided ? dm.M + 1 : dm.N;
    return NA * dm.N + 2 * NA * F + (size_t)dm.K * dm.N + dm.N;
}

struct RtisiArgs {
    const void* mag_main; const void* mag_nyq;
    void* x_out;
    const void* tw; const void* twr; const void* wa; const void* ws;
    RtisiWindow win;                          // magnitude / output / 1/envelope windows
    const void* asym1; const void* asym2;     // analysis windows of the newest frame (already * forward scale)
    double synth_coeff;                       // c = hop / (w . w)
    double lr;                                // alpha / (1 + alpha)
    Dims dm;
    int LA, max_iter, asymmetric, Mp;
    int step_begin, step_end;                 // outer steps [step_begin, step_end) of the T + LA steps of a run
    void* state;                              // per-signal sliding state in / out (rtisi_state_elems), or nullptr
    size_t state_elems;
    int use_mr;                               // mixed-radix passes (any n_fft whose half factors into 2 .. 13)
    mr::Plan mp;
};

template <typename T>
__global__ void __launch_bounds__(256) rtisi_kernel(const RtisiArgs a) {
    using C = cx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Dims& dm = a.dm;
    const int N = dm.N, M = dm.M, hop = dm.hop, K = dm.K, LA = a.LA, NA = a.LA + 1, Mp = a.Mp;
    const int F = dm.onesided ? M + 1 : N;
    const int ylen = LA * hop + N;

    C* work = reinterpret_cast<C*>(smem_raw);                 // [NA][Mp] active frames / FFT work space
    C* pre = work + (size_t)NA * Mp;                          // [NA][F] momentum spectra
    T* kept = reinterpret_cast<T*>(pre + (size_t)NA * F);     // [K][N] committed frames (unscaled samples)
    T* y = kept + (size_t)K * N;                              // [ylen] overlap-add of the current buffer
    T* ykept = y + ylen;                                      // [ylen] part of y that comes from kept frames
    T* carry = ykept + ylen;                                  // [N] output overlap-add carry
    unsigned short* perm = reinterpret_cast<unsigned short*>(carry + N);   // [M] padded position of bin k after the forward passes

    const int tid = threadIdx.x, NT = blockDim.x;
    const int b = blockIdx.x;
    const C* tw = (const C*)a.tw;
    const C* twr = (const C*)a.twr;
    const T* wa = (const T*)a.wa;
    const T* ws = (const T*)a.ws;
    const T* asym1 = (const T*)a.asym1;
    const T* asym2 = (const T*)a.asym2;
    const T* mag_main = (const T*)a.mag_main;
    const T* mag_nyq = (const T*)a.mag_nyq;
    const T* ienv = (const T*)a.win.inv_env;
    const long long x0 = a.win.x0, x1 = a.win.x0 + a.win.x_len;
    T* xo = (T*)a.x_out + (long long)b * a.win.x_len;
    const T coef = (T)a.synth_coeff, lr = (T)a.lr;
    T* workf = reinterpret_cast<T*>(work);
    for (int k = tid; k < M; k += NT)
        perm[k] = (unsigned short)padidx(a.use_mr ? mr::mr_position(a.mp, k) : (int)(__brev((unsigned)k) >> (32 - dm.logM)));
    // the transforms of `nf` frames at v: mixed-radix passes (mixed_radix.cuh) or the radix-2^2 passes (generic_fft.cuh);
    // both end with __syncthreads()
    auto forward = [&](C* v, int nf) {
        if (a.use_mr) {
            for (int s = 0; s < a.mp.nst; ++s) { mr::pass<T, false>(v, nf, Mp, a.mp, s, tw, tid, NT); __syncthreads(); }
        } else {
            fft_forward_inplace<T>(v, nf, M, Mp, tw);
        }
    };
    auto inverse = [&](C* v, int nf) {
        if (a.use_mr) {
            for (int s = a.mp.nst - 1; s >= 0; --s) { mr::pass<T, true>(v, nf, Mp, a.mp, s, tw, tid, NT); __syncthreads(); }
        } else {
            fft_inverse_inplace<T>(v, nf, M, dm.logM, Mp, tw);
        }
    };

    // magnitude of bin kk of spectrogram frame t (zero outside [0, T): the reference pads with zeros, :339)
    auto mag_of = [&](int t, int kk) -> T {
        if (t < 0 || t >= dm.T) return T(0);
        const long long fr = (long long)b * a.win.n_rows + (t - a.win.frame0);
        if (dm.onesided && kk == M) return mag_nyq[fr];
        return mag_main[fr * dm.row + kk];
    };
    // sample n of the frame stored in work slot s
    auto wsample = [&](int s, int n) -> T { return workf[2 * ((size_t)s * Mp + padidx(n >> 1)) + (n & 1)]; };

    // ---- init (methods.py:353-358): everything zero, newest active frame = irfft(first magnitude frame)
    for (int i = tid; i < NA * Mp; i += NT) work[i] = mk<T>(T(0), T(0));
    for (int i = tid; i < NA * F; i += NT) pre[i] = mk<T>(T(0), T(0));
    for (int i = tid; i < K * N; i += NT) kept[i] = T(0);
    for (int i = tid; i < N; i += NT) carry[i] = T(0);
    __syncthreads();
    T* st_frames = a.state ? (T*)a.state + (size_t)b * a.state_elems : nullptr;
    T* st_pre = st_frames + (size_t)NA * N;
    T* st_kept = st_pre + 2 * (size_t)NA * F;
    T* st_carry = st_kept + (size_t)K * N;
    if (a.step_begin > 0) {
        // ---- resume: the state another launch saved before outer step step_begin
        for (int idx = tid; idx < NA * N; idx += NT) {
            const int aa = idx / N, n = idx - aa * N;
            workf[2 * ((size_t)((aa + a.step_begin) % NA) * Mp + padidx(n >> 1)) + (n & 1)] = st_frames[idx];
        }
        for (int idx = tid; idx < NA * F; idx += NT) {
            const int aa = idx / F, k = idx - aa * F;
            pre[(size_t)((aa + a.step_begin) % NA) * F + k] = mk<T>(st_pre[2 * idx], st_pre[2 * idx + 1]);
        }
        for (int i = tid; i < K * N; i += NT) kept[i] = st_kept[i];
        for (int i = tid; i < N; i += NT) carry[i] = st_carry[i];
        __syncthreads();
    } else {
        // logical frame LA at step 0 lives in slot (LA + 0) % NA = LA
        C* v = work + (size_t)LA * Mp;
        for (int k = tid; k <= M / 2; k += NT) {
            const int kA = k, kB = M - k;
            const int pA = perm[kA], pB = perm[kB == M ? 0 : kB];
            C hA = mk<T>(mag_of(0, kA), T(0)), hB = mk<T>(mag_of(0, kB), T(0));
            if (!dm.onesided) {   // Hermitian part of a real two-sided spectrum: (m[k] + m[N-k]) / 2
                if (kA != 0) hA.x = T(0.5) * (hA.x + mag_of(0, N - kA));
                if (kB != M) hB.x = T(0.5) * (hB.x + mag_of(0, N - kB));
            }
            C zA, zB;
            irfft_pre_pair<T>(hA, hB, twr[k], zA, zB);
            v[pA] = zA;
            if (kB != kA && k != 0) v[pB] = zB;
        }
        __syncthreads();
        inverse(v, 1);
    }

    int kslot = 0;   // kept ring: logical kept frame f (0 = oldest) lives in slot (kslot + f) % K
    for (int i = a.step_begin; i < a.step_end; ++i) {
        // part of y contributed by the kept frames: constant over the inner iterations
        for (int p = tid; p < ylen; p += NT) {
            T acc = T(0);
            for (int f = 0; f < K; ++f) {
                const int idx = p + (K - f) * hop;          // index inside kept frame f
                if (idx < N) acc += kept[(size_t)((kslot + f) % K) * N + idx];   // stored as frame * (ws * coef)
            }
            ykept[p] = acc;
        }
        __syncthreads();

        for (int j = 0; j < a.max_iter; ++j) {
            // ---- overlap-add of the active frames on top of the kept part (:365-370)
            for (int p = tid; p < ylen; p += NT) {
                T acc = ykept[p];
                const int alo = p >= N ? (p - N) / hop + 1 : 0;
                const int ahi = min(LA, p / hop);
                for (int aa = alo; aa <= ahi; ++aa) {
                    const int idx = p - aa * hop;
                    acc += wsample((aa + i) % NA, idx) * (ws[idx] * coef);
                }
                y[p] = acc;
            }
            __syncthreads();
            // ---- frame + analysis window (:371-385)
            for (int idx = tid; idx < NA * M; idx += NT) {
                const int aa = idx / M, n = idx - aa * M;
                const T* win = (a.asymmetric && aa == LA) ? (j ? asym2 : asym1) : wa;
                work[(size_t)((aa + i) % NA) * Mp + padidx(n)] =
                    mk<T>(y[aa * hop + 2 * n] * win[2 * n], y[aa * hop + 2 * n + 1] * win[2 * n + 1]);
            }
            __syncthreads();
            forward(work, NA);
            // ---- momentum, projection (:387-396), real-FFT post / pre-processing
            const int npair = M / 2 + 1;
            for (int idx = tid; idx < NA * npair; idx += NT) {
                const int aa = idx / npair, k = idx - aa * npair;
                const int slot = (aa + i) % NA;
                C* v = work + (size_t)slot * Mp;
                C* pr = pre + (size_t)slot * F;
                const int t = i + aa - LA;                  // spectrogram frame of this active frame
                const bool mom = j > 0 || (i > 0 && aa < LA);
                const int kA = k, kB = M - k;
                const int pA = perm[kA], pB = perm[kB == M ? 0 : kB];
                const C w = twr[k];
                C sA, sB;
                rfft_post_pair<T>(v[pA], v[pB], w, sA, sB);
                auto upd = [&](int kk, C s) -> C {
                    if (mom) { const C p0 = pr[kk]; s = mk<T>(s.x - lr * p0.x, s.y - lr * p0.y); }
                    pr[kk] = s;
                    return project<T>(s, mag_of(t, kk));
                };
                C hA, hB;
                if (dm.onesided) {
                    hA = upd(kA, sA);
                    hB = (kB != kA) ? upd(kB, sB) : hA;
                } else {
                    hA = upd(kA, sA);
                    if (kA != 0) {
                        const C m = upd(N - kA, mk<T>(sA.x, -sA.y));
                        hA = mk<T>(T(0.5) * (hA.x + m.x), T(0.5) * (hA.y - m.y));
                    }
                    if (kB != kA) {
                        hB = upd(kB, sB);
                        if (kB != M) {
                            const C m = upd(N - kB, mk<T>(sB.x, -sB.y));
                            hB = mk<T>(T(0.5) * (hB.x + m.x), T(0.5) * (hB.y - m.y));
                        }
                    } else {
                        hB = hA;
                    }
                }
                if (k == 0) { hA.y = T(0); hB.y = T(0); }
                C zA, zB;
                irfft_pre_pair<T>(hA, hB, w, zA, zB);
                v[pA] = zA;
                if (kB != kA && k != 0) v[pB] = zB;
            }
            __syncthreads();
            inverse(work, NA);                                       // ends with __syncthreads()
        }

        // ---- commit the oldest active frame (:401-404) and fuse the final overlap-add (:406-408)
        const int s0 = i % NA;                                  // slot of logical frame 0
        if (i >= LA) {
            const int t = i - LA;                               // index of the committed frame in the output OLA
            for (int n = tid; n < N; n += NT) carry[n] += wsample(s0, n) * ws[n];
            __syncthreads();
            const bool last = a.win.final && t == dm.T - 1;
            const int nout = last ? N : hop;                    // the last frame flushes the whole carry
            for (int n = tid; n < nout; n += NT) {
                const long long m = (long long)t * hop + n - dm.P;
                if (m >= x0 && m < x1) xo[m - x0] = carry[n] * ienv[m - x0];
            }
            __syncthreads();
            if (!last) {
                // shift the carry by one hop (two passes through registers to avoid the overlap hazard)
                for (int base = 0; base < N; base += NT) {
                    const int n = base + tid;
                    const T v = (n < N && n + hop < N) ? carry[n + hop] : T(0);
                    __syncthreads();
                    if (n < N) carry[n] = v;
                    __syncthreads();
                }
            }
        }
        if (K > 0) {
            // the committed frame replaces the oldest kept frame
            T* dst = kept + (size_t)kslot * N;
            for (int n = tid; n < N; n += NT) dst[n] = wsample(s0, n) * (ws[n] * coef);
            kslot = (kslot + 1) % K;
        }
        __syncthreads();
        // slot s0 becomes the newest (all-zero) active frame of the next step
        for (int n = tid; n < Mp; n += NT) work[(size_t)s0 * Mp + n] = mk<T>(T(0), T(0));
        __syncthreads();
    }
    if (a.step_begin == a.step_end) {
        // a final launch with no step left (look_ahead = 0, frame T-1 committed by an earlier launch): release the
        // carry that commit shifted by one hop -- the values its flush would have written
        for (int n = tid; n < N - hop; n += NT) {
            const long long m = (long long)dm.T * hop + n - dm.P;
            if (m >= x0 && m < x1) xo[m - x0] = carry[n] * ienv[m - x0];
        }
    }
    if (a.state && !(a.win.final && a.step_end == dm.T + LA)) {
        // ---- save the state before outer step step_end (logical order; the newest frame's momentum is not used)
        for (int idx = tid; idx < NA * N; idx += NT) {
            const int aa = idx / N, n = idx - aa * N;
            st_frames[idx] = wsample((aa + a.step_end) % NA, n);
        }
        for (int idx = tid; idx < NA * F; idx += NT) {
            const int aa = idx / F, k = idx - aa * F;
            const C v = aa == LA ? mk<T>(T(0), T(0)) : pre[(size_t)((aa + a.step_end) % NA) * F + k];
            st_pre[2 * idx] = v.x; st_pre[2 * idx + 1] = v.y;
        }
        for (int idx = tid; idx < K * N; idx += NT) {
            const int f = idx / N, n = idx - f * N;
            st_kept[idx] = kept[(size_t)((kslot + f) % K) * N + n];
        }
        for (int i = tid; i < N; i += NT) st_carry[i] = carry[i];
    }
}

// asym_window1 / asym_window2 of methods.py:326-336 (times the forward scale of the analysis side)
template <typename T>
__global__ void rtisi_windows_kernel(int N, int hop, int K, const T* __restrict__ w, double coef, double fscale,
                                     T* asym1, T* asym2) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= N) return;
    T a1 = T(0), a2 = T(0);
    for (int i = 0; i <= K; ++i) {
        const int s = i * hop;
        if (m >= s) {
            const T v = w[N - 1 - (m - s)];           // window.flip(0)[m - s]
            a2 += v;
            if (i >= 1) a1 += v;
        }
    }
    asym1[m] = (T)((double)(a1 * (T)coef) * fscale);
    asym2[m] = (T)((double)(a2 * (T)coef) * fscale);
}

template <typename T>
static int rtisi_t(const specinv_desc* d, const Dims& dm, const void* plan, const void* window, const void* mag_main,
                   const void* mag_nyq, void* x_out, const RtisiWindow& win, void* scratch, int look_ahead, int asymmetric,
                   int max_iter, double alpha, double synth_coeff, int step_begin, int step_end, void* state,
                   cudaStream_t st) {
    RtisiArgs a{};
    const PlanLayout pl = plan_layout(dm, d->dtype);
    const char* p = (const char*)plan;
    a.tw = p + pl.tw; a.twr = p + pl.twr; a.wa = p + pl.wa; a.ws = p + pl.ws; a.win = win;
    a.dm = dm;
    a.LA = look_ahead < 0 ? dm.K : look_ahead;
    a.max_iter = max_iter; a.asymmetric = asymmetric;
    a.synth_coeff = synth_coeff; a.lr = alpha / (1.0 + alpha);
    a.mag_main = mag_main; a.mag_nyq = mag_nyq; a.x_out = x_out;
    a.Mp = mr::padded_len(dm.M);
    {
        // mixed-radix passes whenever the half size factors into 2 .. 13 (the only path for a non-power-of-two n_fft,
        // whose root table is W_N); SPECINV_GENERIC_MR=0 keeps the radix-2^2 passes for the powers of two
        const char* e = getenv("SPECINV_GENERIC_MR");
        const bool want = !(e && e[0] == '0') || !dm.pow2;
        a.use_mr = want && dm.M <= 4096 && !(dm.N & 1) && mr::make_plan(dm.M, dm.pow2 ? dm.M : dm.N, &a.mp, sizeof(T) == 4) ? 1 : 0;
        if (!a.use_mr && !dm.pow2) return SPECINV_ERR_UNSUPPORTED;    // a prime factor > 13: no RTISI-LA kernel
    }
    a.step_begin = step_begin; a.step_end = step_end; a.state = state; a.state_elems = rtisi_state_elems(dm, a.LA);
    T* asym = (T*)scratch;
    a.asym1 = asym; a.asym2 = asym + dm.N;
    const double fscale = d->normalized ? 1.0 / sqrt((double)dm.N) : 1.0;
    rtisi_windows_kernel<T><<<(dm.N + 255) / 256, 256, 0, st>>>(dm.N, dm.hop, dm.K, (const T*)window, synth_coeff, fscale,
                                                                asym, asym + dm.N);
    if (sizeof(T) == 4) {
        // the register-FFT kernel of specinv_rtisi_fast.cu covers n_fft = 1024 / hop = 256 / look_ahead <= 3
        const char* fg = getenv("SPECINV_FORCE_GENERIC");
        if (!(fg && fg[0] == '1')) {
            const int rf = rtisi_fast(d, dm, plan, mag_main, mag_nyq, x_out, win, asym, asym + dm.N, look_ahead,
                                      asymmetric, max_iter, alpha, synth_coeff, step_begin, step_end, state, st);
            if (rf != SPECINV_ERR_UNSUPPORTED) return rf;
        }
    }
    const int NA = a.LA + 1, F = dm.onesided ? dm.M + 1 : dm.N, ylen = a.LA * dm.hop + dm.N;
    const size_t smem = ((size_t)NA * a.Mp + (size_t)NA * F) * 2 * sizeof(T) +
                        ((size_t)dm.K * dm.N + 2 * (size_t)ylen + dm.N) * sizeof(T) + (size_t)dm.M * 2;
    int dev = 0, optin = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if ((long long)smem > (long long)optin) return SPECINV_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(rtisi_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    rtisi_kernel<T><<<dm.B, 256, smem, st>>>(a);
    return (int)cudaGetLastError();
}

}  // namespace specinv

using namespace specinv;

extern "C" {

int specinv_rtisi_state_bytes(const specinv_desc* d, int look_ahead, size_t* bytes) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!bytes) return SPECINV_ERR_INVALID;
    const int LA = look_ahead < 0 ? dm.K : look_ahead;
    *bytes = (size_t)dm.B * rtisi_state_elems(dm, LA) * (d->dtype == SPECINV_F64 ? 8 : 4);
    return SPECINV_OK;
}

int specinv_rtisi_la_steps(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                           const void* mag_nyq, void* x_out, void* scratch, int look_ahead, int asymmetric_window,
                           int max_iter, double alpha, double synth_coeff, int step_begin, int step_end, void* state,
                           void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !window || !mag_main || !x_out || !scratch || (dm.onesided && !mag_nyq)) return SPECINV_ERR_INVALID;
    if (max_iter < 1 || alpha < 0) return SPECINV_ERR_INVALID;
    const int steps = dm.T + (look_ahead < 0 ? dm.K : look_ahead);
    if (step_begin < 0 || step_end > steps || step_begin >= step_end) return SPECINV_ERR_INVALID;
    if ((step_begin > 0 || step_end < steps) && !state) return SPECINV_ERR_INVALID;
    // the whole signal is the window: every launch addresses all T frames and all L samples
    const RtisiWindow win{0, dm.T, 0, dm.L, (const char*)plan + plan_layout(dm, d->dtype).inv_env, 1};
    return d->dtype == SPECINV_F64
               ? rtisi_t<double>(d, dm, plan, window, mag_main, mag_nyq, x_out, win, scratch, look_ahead,
                                 asymmetric_window, max_iter, alpha, synth_coeff, step_begin, step_end, state,
                                 (cudaStream_t)stream)
               : rtisi_t<float>(d, dm, plan, window, mag_main, mag_nyq, x_out, win, scratch, look_ahead,
                                asymmetric_window, max_iter, alpha, synth_coeff, step_begin, step_end, state,
                                (cudaStream_t)stream);
}

int specinv_rtisi_la_stream(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                            const void* mag_nyq, int frame0, int n_rows, void* x_out, const void* inv_env, int64_t x0,
                            int64_t x_len, void* scratch, int look_ahead, int asymmetric_window, int max_iter,
                            double alpha, double synth_coeff, int step_begin, int step_end, int final, void* state,
                            void* stream) {
    if (!d || d->n_frames < 1) return SPECINV_ERR_INVALID;
    // RTISI-LA never pads, and one centred frame has no output sample yet (L = 0), which make_dims refuses for a
    // whole signal: derive the dimensions as for two frames, then put the real frame count back
    specinv_desc dd = *d;
    dd.pad_mode = SPECINV_PAD_CONSTANT;
    if (dd.n_frames < 2) dd.n_frames = 2;
    Dims dm; int rc = make_dims(&dd, &dm); if (rc) return rc;
    dm.T = d->n_frames;
    dm.Lp = (long long)(dm.T - 1) * dm.hop + dm.N;
    dm.L = dm.Lp - 2LL * dm.P;
    if (!plan || !window || !scratch || !state) return SPECINV_ERR_INVALID;
    if (n_rows > 0 && (!mag_main || (dm.onesided && !mag_nyq))) return SPECINV_ERR_INVALID;
    if (x_len > 0 && (!x_out || !inv_env)) return SPECINV_ERR_INVALID;
    if (max_iter < 1 || alpha < 0 || (final != 0 && final != 1)) return SPECINV_ERR_INVALID;
    const int LA = look_ahead < 0 ? dm.K : look_ahead;
    // steps: step i reads frame i, so a launch that is not final stops at the frames pushed so far
    if (step_begin < 0 || step_end > dm.T + (final ? LA : 0)) return SPECINV_ERR_INVALID;
    // an empty range only as the final launch that releases the carry left by an earlier commit of frame T-1
    if (step_begin > step_end || (step_begin == step_end && !(final && step_end == dm.T + LA))) return SPECINV_ERR_INVALID;
    // magnitude rows: from the oldest frame a resume re-reads up to the newest one a step reads
    const int need0 = step_begin - LA > 0 ? step_begin - LA : 0;
    const int need1 = step_end < dm.T ? step_end : dm.T;
    if (frame0 < 0 || n_rows < 0 || frame0 > need0 || (long long)frame0 + n_rows > dm.T || frame0 + n_rows < need1)
        return SPECINV_ERR_INVALID;
    // samples: exactly those these steps finish (the commit of step i finishes [(i-LA)*hop - P, (i-LA+1)*hop - P);
    // the final launch also finishes everything up to L)
    auto block_end = [&](long long i) { const long long e = (i - LA) * dm.hop - dm.P; return e > 0 ? e : 0LL; };
    long long lo = block_end(step_begin), hi = block_end(step_end);
    if (final) {
        const long long L = dm.L > 0 ? dm.L : 0;
        lo = lo < L ? lo : L;
        hi = step_end == dm.T + LA || hi > L ? L : hi;
    }
    if (x0 != lo || x_len != hi - lo) return SPECINV_ERR_INVALID;
    const RtisiWindow win{frame0, n_rows, x0, x_len, inv_env, final};
    return d->dtype == SPECINV_F64
               ? rtisi_t<double>(d, dm, plan, window, mag_main, mag_nyq, x_out, win, scratch, look_ahead,
                                 asymmetric_window, max_iter, alpha, synth_coeff, step_begin, step_end, state,
                                 (cudaStream_t)stream)
               : rtisi_t<float>(d, dm, plan, window, mag_main, mag_nyq, x_out, win, scratch, look_ahead,
                                asymmetric_window, max_iter, alpha, synth_coeff, step_begin, step_end, state,
                                (cudaStream_t)stream);
}

int specinv_rtisi_la(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                     const void* mag_nyq, void* x_out, void* scratch, int look_ahead, int asymmetric_window,
                     int max_iter, double alpha, double synth_coeff, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    return specinv_rtisi_la_steps(d, plan, window, mag_main, mag_nyq, x_out, scratch, look_ahead, asymmetric_window,
                                  max_iter, alpha, synth_coeff, 0, dm.T + (look_ahead < 0 ? dm.K : look_ahead), nullptr,
                                  stream);
}

}  // extern "C"
