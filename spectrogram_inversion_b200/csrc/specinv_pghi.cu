// PGHI: phase-gradient heap integration (Průša, Balazs and Søndergaard, IEEE/ACM TASLP 25(5), 2017), in the
// frame-causal form of Průša and Holighaus (EUSIPCO 2017).  The definition is pghi_heap of tests/golden/pghi_ref.py;
// this file computes its scan formulation, pghi_ref.pghi (DESIGN.md section 3.7):
//   * which neighbour reaches a bin of frame n (time, left, right) depends on the magnitudes of frames n-1 and n only:
//     a widest-path problem inside every run of significant bins, solved by (min, max) clamp scans over the bins;
//   * the phase of bin m in frame n is phi[g[m], n-1] + c[m] (g: the root of m's run, c: the root's time step plus
//     the bin steps along the run, a segmented prefix sum in each direction); these maps compose over frames, so time
//     splits into chunks like phase_init's: per-chunk composed maps, a carry over the chunks, an apply pass.
// All arithmetic is float64 whatever the magnitude's dtype; the running phase is reduced to [-pi, pi] after every
// addition.  No FFT is involved, so every n_fft works.
//
// Kernels (one CTA of NT threads per (signal, chunk); a thread owns P = ceil(F / NT) consecutive bins):
//   pghi_max_kernel<T>         per-signal max of the magnitude (threshold tol * max)
//   pghi_frames_kernel<T, 1>   compose the per-frame maps of a chunk (all chunks but the last)
//   pghi_carry_kernel          running phase at the start of every chunk, sequentially over the chunks
//   pghi_frames_kernel<T, 0>   recompute the per-frame maps, integrate from the chunk's start, write mag * e^{i phi}
//   pghi_stream_kernel<T>      the stream mode (frames_body<T, 2>): one CTA per signal finalises the frames of one
//                              push from the state of the last one, with the causal threshold (DESIGN.md section 3.7.1)
#include <limits.h>
#include <math.h>

#include <algorithm>

#include "specinv_common.cuh"

namespace specinv {
namespace pghi {

constexpr int NT = 256;
constexpr int NW = NT / 32;
constexpr int MIN_CHUNK = 32;          // frames per chunk at least
constexpr int SMS = 148;               // B200
constexpr double PI = 3.14159265358979323846;
constexpr double TWO_PI = 2 * PI;
constexpr double INV_TWO_PI = 0.15915494309189533576888;

enum : unsigned char { NONE = 0, ROOT = 1, LEFT = 2, RIGHT = 3 };

struct Params {
    int B, F, T, M, hop, chunks, chunk_len;
    long long sb, sf, st;              // element strides of the (B, F, T) magnitude
    double tol, K0, K1, K2;            // K0 = 2 pi c / M, K1 = a M / gamma, K2 = gamma / (M a)
    size_t cta_bytes;                  // per-CTA working set (shared memory, or `scratch` when it does not fit)
};

__device__ __forceinline__ double wrap(double x) { return fma(-rint(x * INV_TWO_PI), TWO_PI, x); }

// x -> min(hi, max(lo, x)) with lo <= hi.  `then(a, b)` applies a first.
template <typename T> struct Clamp { T lo, hi; };
template <typename T> __device__ __forceinline__ Clamp<T> then(Clamp<T> a, Clamp<T> b) {
    return {fmin(b.hi, fmax(b.lo, a.lo)), fmin(b.hi, fmax(b.lo, a.hi))};
}
template <typename T> __device__ __forceinline__ T at(Clamp<T> f, T x) { return fmin(f.hi, fmax(f.lo, x)); }

// Both reach scans in one: the widest path from a time source (A, B) and the island's max on one side (PL, PR).
template <typename T> struct Reach { Clamp<T> w, mx; };
template <typename T> __device__ __forceinline__ Reach<T> then(Reach<T> a, Reach<T> b) {
    return {then(a.w, b.w), then(a.mx, b.mx)};
}
template <typename T> __device__ __forceinline__ Reach<T> ident(Reach<T>*) {
    return {{T(-INFINITY), T(INFINITY)}, {T(-INFINITY), T(INFINITY)}};
}
template <typename T> __device__ __forceinline__ Reach<T> shfl_up(Reach<T> v, int d) {
    return {{__shfl_up_sync(~0u, v.w.lo, d), __shfl_up_sync(~0u, v.w.hi, d)},
            {__shfl_up_sync(~0u, v.mx.lo, d), __shfl_up_sync(~0u, v.mx.hi, d)}};
}
template <typename T> __device__ __forceinline__ Reach<T> shfl_down(Reach<T> v, int d) {
    return {{__shfl_down_sync(~0u, v.w.lo, d), __shfl_down_sync(~0u, v.w.hi, d)},
            {__shfl_down_sync(~0u, v.mx.lo, d), __shfl_down_sync(~0u, v.mx.hi, d)}};
}

// Segmented sum along a run: `reset` starts a run at root g with offset c, otherwise c is added.
struct Seg { int reset, g; double c; };
__device__ __forceinline__ Seg then(Seg a, Seg b) { return b.reset ? b : Seg{a.reset, a.g, wrap(a.c + b.c)}; }
__device__ __forceinline__ Seg ident(Seg*) { return {0, -1, 0.0}; }
__device__ __forceinline__ Seg shfl_up(Seg v, int d) {
    return {__shfl_up_sync(~0u, v.reset, d), __shfl_up_sync(~0u, v.g, d), __shfl_up_sync(~0u, v.c, d)};
}
__device__ __forceinline__ Seg shfl_down(Seg v, int d) {
    return {__shfl_down_sync(~0u, v.reset, d), __shfl_down_sync(~0u, v.g, d), __shfl_down_sync(~0u, v.c, d)};
}

// Exclusive block scan in both directions at once: f <- composition over the threads below, b <- over the threads
// above (highest first).  wf / wb: NW entries of shared memory owned by this scan.
template <typename V>
__device__ __forceinline__ void block_scan2(V& f, V& b, V* wf, V* wb) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    V fi = f, bi = b;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const V fu = shfl_up(fi, d), bd = shfl_down(bi, d);
        if (lane >= d) fi = then(fu, fi);
        if (lane + d < 32) bi = then(bd, bi);
    }
    if (lane == 31) wf[w] = fi;
    if (lane == 0) wb[w] = bi;
    __syncthreads();
    V pf = ident((V*)nullptr), pb = ident((V*)nullptr);
    for (int k = 0; k < w; ++k) pf = then(pf, wf[k]);
    for (int k = NW - 1; k > w; --k) pb = then(pb, wb[k]);
    V ef = shfl_up(fi, 1), eb = shfl_down(bi, 1);
    if (lane == 0) ef = ident((V*)nullptr);
    if (lane == 31) eb = ident((V*)nullptr);
    f = then(pf, ef);
    b = then(pb, eb);
}

// The per-CTA working set, in dynamic shared memory or, for large F, in the CTA's slice of the workspace.
template <typename T> struct Work {
    double* s;              // [3][F] log(max(mag, thr)), ring over frames n-1, n, n+1
    double* ph[2];          // [F] running phase (apply) or composed offsets (compose), ping-pong
    int* g[2];              // [F] composed sources (compose)
    T* mag;                 // [3][F] magnitudes, same ring
    T* lw;                  // [F] left reach A
    T* lmx;                 // [F] island max left of the bin
    unsigned char* ch;      // [F] choice
};

__host__ __device__ inline size_t al16(size_t v) { return (v + 15) & ~(size_t)15; }

template <typename T> __host__ __device__ inline size_t work_bytes(int F, Work<T>* w, char* base) {
    size_t o = 0;
    auto take = [&](size_t n) { char* p = base + o; o = al16(o + n); return p; };
    char* s = take(3 * (size_t)F * 8);
    char* p0 = take((size_t)F * 8); char* p1 = take((size_t)F * 8);
    char* g0 = take((size_t)F * 4); char* g1 = take((size_t)F * 4);
    char* mg = take(3 * (size_t)F * sizeof(T));
    char* lw = take((size_t)F * sizeof(T)); char* lm = take((size_t)F * sizeof(T));
    char* ch = take((size_t)F);
    if (w) {
        w->s = (double*)s; w->ph[0] = (double*)p0; w->ph[1] = (double*)p1; w->g[0] = (int*)g0; w->g[1] = (int*)g1;
        w->mag = (T*)mg; w->lw = (T*)lw; w->lmx = (T*)lm; w->ch = (unsigned char*)ch;
    }
    return o;
}

template <typename T>
__global__ void __launch_bounds__(NT) pghi_max_kernel(Params p, const T* __restrict__ mag,
                                                      unsigned long long* __restrict__ maxbits) {
    const int b = blockIdx.y;
    const T* mb = mag + (long long)b * p.sb;
    double mx = 0.0;                   // magnitudes are >= 0; NaN never wins a comparison
    for (int t = blockIdx.x; t < p.T; t += gridDim.x)
        for (int m = threadIdx.x; m < p.F; m += NT) {
            const double v = (double)__ldg(mb + (long long)m * p.sf + (long long)t * p.st);
            if (v > mx) mx = v;
        }
#pragma unroll
    for (int d = 16; d; d >>= 1) mx = fmax(mx, __shfl_xor_sync(~0u, mx, d));
    __shared__ double red[NW];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < NW; ++k) mx = fmax(mx, red[k]);
        // non-negative doubles order like their bit patterns
        if (mx > 0.0) atomicMax(maxbits + b, (unsigned long long)__double_as_longlong(mx));
    }
}

// One call of the stream mode (MODE 2, pghi_stream_kernel): the magnitude rows are frames frame0 + r, r < p.T - frame0
// (p.T is the end of the frames seen so far); frames [first, first + n_fin) are finalised.  state: StreamHead, then
// the running phase [F] (StreamState); out: [B][n_fin][F].
struct Stream { int frame0, first, n_fin; };
struct StreamHead { double max; long long count; };      // running max of the frames read, frames final so far

__host__ __device__ inline size_t stream_row_bytes(int F) { return al16(sizeof(StreamHead) + (size_t)F * 8); }

// Block-wide max; every thread gets it.  red: NW doubles, free until the next __syncthreads.
__device__ __forceinline__ double block_max(double v, double* red) {
#pragma unroll
    for (int d = 16; d; d >>= 1) v = fmax(v, __shfl_xor_sync(~0u, v, d));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    for (int k = 0; k < NW; ++k) v = fmax(v, red[k]);
    return v;
}

// MODE 0: apply (write mag * e^{i phi} for the chunk's frames); MODE 1: compose the chunk's per-frame maps;
// MODE 2: apply for a stream, with the causal threshold thr_n = tol * max(frames 0 .. n + 1) (DESIGN.md section 3.7.1).
template <typename T, int MODE>
__device__ __forceinline__ void frames_body(Params p, const T* __restrict__ mag,
                                            const unsigned long long* __restrict__ maxbits,
                                            const double* __restrict__ phi_start, int* __restrict__ map_g,
                                            double* __restrict__ map_c, cx_t<T>* __restrict__ out,
                                            char* __restrict__ scratch, Stream sm, char* __restrict__ state) {
    extern __shared__ __align__(16) char smem[];
    __shared__ Reach<T> wrf[NW], wrb[NW];
    __shared__ Seg wsf[NW], wsb[NW];
    const int F = p.F, tid = threadIdx.x;
    const int per_signal = MODE == 2 ? 1 : MODE ? p.chunks - 1 : p.chunks;
    const int b = blockIdx.x / per_signal, chunk = blockIdx.x % per_signal;
    const int ta = MODE == 2 ? sm.first : chunk * p.chunk_len;
    const int tb = MODE == 2 ? sm.first + sm.n_fin : min(p.T, ta + p.chunk_len);
    Work<T> wk;
    work_bytes<T>(F, &wk, scratch ? scratch + (size_t)blockIdx.x * p.cta_bytes : smem);
    const T* mb = mag + (long long)b * p.sb;
    StreamHead* head = nullptr;
    double* st_phase = nullptr;
    double runmax = 0.0;
    __shared__ double red[MODE == 2 ? NW : 1];
    if (MODE == 2) {
        head = (StreamHead*)(state + (size_t)b * stream_row_bytes(F));
        st_phase = (double*)(head + 1);
        if (ta > 0) {
            if (head->count != ta) {           // not this stream's next call: refuse visibly, leave the state
                for (int i = tid; i < sm.n_fin * F; i += NT)
                    out[(long long)b * sm.n_fin * F + i] = mk<T>(T(NAN), T(NAN));
                return;
            }
            runmax = head->max;
        }
    }
    double thr = MODE == 2 ? 0.0 : p.tol * __longlong_as_double((long long)maxbits[b]);
    const int P = (F + NT - 1) / NT, lo = min(F, tid * P), hi = min(F, lo + P);
    const long long chunk_row = ((long long)b * p.chunks + chunk) * F;

    // ring slot of frame n: frames ta-1, ta, ta+1 are slots 0, 1, 2
    auto slot = [&](int n) { return (n - ta + 1) % 3; };
    auto load = [&](int n) {
        const int r = slot(n);
        for (int m = tid; m < F; m += NT) {
            const T v = __ldg(mb + (long long)m * p.sf + (long long)n * p.st);
            wk.mag[r * F + m] = v;
            wk.s[r * F + m] = log(fmax((double)v, thr));
        }
    };
    // stream mode: the magnitudes first (their max moves the threshold), the logs once the threshold is known
    auto load_mag = [&](int n) {
        const int r = slot(n);
        double mx = 0.0;                   // magnitudes are >= 0; NaN never wins a comparison
        for (int m = tid; m < F; m += NT) {
            const T v = __ldg(mb + (long long)m * p.sf + (long long)(n - sm.frame0) * p.st);
            wk.mag[r * F + m] = v;
            if ((double)v > mx) mx = (double)v;
        }
        return mx;
    };
    auto relog = [&](int n) {              // own bins only: the same threads wrote them in load_mag
        const int r = slot(n);
        for (int m = tid; m < F; m += NT) wk.s[r * F + m] = log(fmax((double)wk.mag[r * F + m], thr));
    };
    // ping-pong: the phase (apply) or the composed map (compose) up to frame n-1, and the one being built
    double *ph0 = wk.ph[0], *ph1 = wk.ph[1];
    int *g0 = wk.g[0], *g1 = wk.g[1];
    for (int m = tid; m < F; m += NT) {
        if (MODE == 2) ph0[m] = ta > 0 ? st_phase[m] : 0.0;
        else if (MODE) { g0[m] = m; ph0[m] = 0.0; }
        else ph0[m] = p.chunks > 1 ? phi_start[chunk_row + m] : 0.0;
    }
    if (MODE == 2) {
        double mx = load_mag(ta);
        if (ta > 0) mx = fmax(mx, load_mag(ta - 1));
        runmax = block_max(fmax(runmax, mx), red);
        thr = p.tol * runmax;
        if (ta > 0) relog(ta - 1);
        relog(ta);
    } else {
        if (ta > 0) load(ta - 1);
        load(ta);
    }
    auto write_out = [&](int n, const double* ph) {
        const T* mg = wk.mag + slot(n) * F;
        cx_t<T>* o = MODE == 2 ? out + ((long long)b * sm.n_fin + (n - ta)) * F : out + ((long long)b * p.T + n) * F;
        for (int m = tid; m < F; m += NT) {
            double sn, cs;
            sincos(ph[m], &sn, &cs);
            const double v = (double)mg[m];
            o[m] = mk<T>((T)(v * cs), (T)(v * sn));
        }
    };

    for (int n = ta; n < tb; ++n) {
        if (MODE != 1 && n > ta) write_out(n - 1, ph0);
        if (MODE == 2) {
            // thr_n: fold frame n+1 into the running max; the ring's logs change only when the threshold does
            const double mx = block_max(fmax(runmax, n + 1 < p.T ? load_mag(n + 1) : 0.0), red);
            if (mx != runmax) {
                runmax = mx;
                thr = p.tol * runmax;
                if (n > 0) relog(n - 1);
                relog(n);
            }
            if (n + 1 < p.T) relog(n + 1);
        } else if (n + 1 < p.T) {
            load(n + 1);
        }
        __syncthreads();
        const T* mp = wk.mag + slot(n - 1) * F;      // not read in frame 0
        const T* mc = wk.mag + slot(n) * F;
        const double* sp = wk.s + slot(n - 1) * F;
        const double* sc = wk.s + slot(n) * F;
        const double* sn = wk.s + slot(n + 1) * F;   // read only when n + 1 < T
        const bool has_prev = n > 0, dn_on = n >= 1 && n + 1 < p.T;

        auto sig = [&](int j) { return (double)mc[j] > thr; };
        auto src = [&](int j) {                       // time source S: mag[j, n-1] where both bins are significant
            return (has_prev && (double)mp[j] > thr && sig(j)) ? mp[j] : T(-1);
        };
        auto trans = [&](int j) -> Reach<T> {        // the step from bin j to its neighbour
            if (!sig(j)) return {{T(-1), T(-1)}, {T(-1), T(-1)}};
            const T v = mc[j];
            return {{fmin(src(j), v), v}, {v, T(INFINITY)}};
        };
        auto dm = [&](const double* s, int j) { return (j >= 1 && j + 2 <= F) ? 0.5 * (s[j + 1] - s[j - 1]) : 0.0; };
        auto dnn = [&](int j) { return dn_on ? 0.5 * (sn[j] - sp[j]) : 0.0; };
        auto fstep = [&](int j) { return p.K0 - p.K2 * (0.5 * (dnn(j) + dnn(j + 1))); };    // bin j -> j + 1
        auto root_c = [&](int j) {
            if (!has_prev) return 0.0;
            const double base = TWO_PI * (double)(((long long)j * p.hop) % p.M) / (double)p.M;
            return base + p.K1 * (0.5 * (dm(sp, j) + dm(sc, j)));
        };

        // 1. reach scans: A (left), B (right) and the island's max on either side
        Reach<T> rf = ident((Reach<T>*)nullptr), rb = rf;
        for (int j = lo; j < hi; ++j) rf = then(rf, trans(j));
        for (int j = hi - 1; j >= lo; --j) rb = then(rb, trans(j));
        block_scan2(rf, rb, wrf, wrb);
        for (int j = lo; j < hi; ++j) {
            wk.lw[j] = at(rf.w, T(-1));
            wk.lmx[j] = at(rf.mx, T(-1));
            rf = then(rf, trans(j));
        }
        for (int j = hi - 1; j >= lo; --j) {
            const T B = at(rb.w, T(-1)), PR = at(rb.mx, T(-1));
            unsigned char c = NONE;
            if (sig(j)) {
                const T S = src(j), A = wk.lw[j], PL = wk.lmx[j], v = mc[j];
                const T W = fmax(S, fmax(A, B));
                if (W >= T(0)) c = S == W ? ROOT : A == W ? LEFT : RIGHT;
                else c = (v > PL && v >= PR) ? ROOT : (PL >= v && PL >= PR) ? LEFT : RIGHT;   // seeded at its max
            }
            wk.ch[j] = c;
            rb = then(rb, trans(j));
        }

        // 2. offsets along the runs: forward for roots and left-reached bins, backward for right-reached ones
        auto elf = [&](int j) -> Seg {
            const unsigned char c = wk.ch[j];
            if (c == LEFT) return {0, -1, fstep(j - 1)};
            if (c == ROOT) return {1, j, root_c(j)};
            return {1, -1, 0.0};
        };
        auto elb = [&](int j) -> Seg {
            const unsigned char c = wk.ch[j];
            if (c == RIGHT) return {0, -1, -fstep(j)};
            if (c == ROOT) return {1, j, root_c(j)};
            return {1, -1, 0.0};
        };
        Seg sf = ident((Seg*)nullptr), sb = sf;
        for (int j = lo; j < hi; ++j) sf = then(sf, elf(j));
        for (int j = hi - 1; j >= lo; --j) sb = then(sb, elb(j));
        block_scan2(sf, sb, wsf, wsb);
        auto put = [&](int j, Seg v) {
            if (MODE) {
                g1[j] = v.g < 0 ? -1 : g0[v.g];
                ph1[j] = v.g < 0 ? v.c : wrap(ph0[v.g] + v.c);
            } else {
                ph1[j] = v.g < 0 ? v.c : wrap(ph0[v.g] + v.c);
            }
        };
        for (int j = lo; j < hi; ++j) {
            sf = then(sf, elf(j));
            const unsigned char c = wk.ch[j];
            if (c == ROOT || c == LEFT) put(j, sf);
            else if (c == NONE) put(j, Seg{1, -1, 0.0});
        }
        for (int j = hi - 1; j >= lo; --j) {
            sb = then(sb, elb(j));
            if (wk.ch[j] == RIGHT) put(j, sb);
        }
        __syncthreads();
        { double* t = ph0; ph0 = ph1; ph1 = t; }
        { int* t = g0; g0 = g1; g1 = t; }
    }
    if (MODE == 2) {
        if (tb > ta) write_out(tb - 1, ph0);
        for (int m = tid; m < F; m += NT) st_phase[m] = ph0[m];
        if (tid == 0) *head = StreamHead{runmax, (long long)tb};
    } else if (MODE) {
        for (int m = tid; m < F; m += NT) {
            map_g[chunk_row + m] = g0[m];
            map_c[chunk_row + m] = ph0[m];
        }
    } else {
        write_out(tb - 1, ph0);
    }
}

template <typename T, int MODE>
__global__ void __launch_bounds__(NT) pghi_frames_kernel(Params p, const T* __restrict__ mag,
                                                         const unsigned long long* __restrict__ maxbits,
                                                         const double* __restrict__ phi_start, int* __restrict__ map_g,
                                                         double* __restrict__ map_c, cx_t<T>* __restrict__ out,
                                                         char* __restrict__ scratch) {
    frames_body<T, MODE>(p, mag, maxbits, phi_start, map_g, map_c, out, scratch, Stream{}, nullptr);
}

// One CTA per signal: finalise frames [sm.first, sm.first + sm.n_fin) of a stream (specinv_pghi_stream).
template <typename T>
__global__ void __launch_bounds__(NT) pghi_stream_kernel(Params p, const T* __restrict__ mag, Stream sm,
                                                         char* __restrict__ state, cx_t<T>* __restrict__ out,
                                                         char* __restrict__ scratch) {
    frames_body<T, 2>(p, mag, nullptr, nullptr, nullptr, nullptr, out, scratch, sm, state);
}

// phi_start[b][k] = the running phase of frame k * chunk_len - 1 (zero for k = 0), through the composed maps.
__global__ void __launch_bounds__(NT) pghi_carry_kernel(Params p, const int* __restrict__ map_g,
                                                        const double* __restrict__ map_c, double* phi_start) {
    const long long row0 = (long long)blockIdx.x * p.chunks * p.F;
    for (int m = threadIdx.x; m < p.F; m += NT) phi_start[row0 + m] = 0.0;
    for (int k = 0; k + 1 < p.chunks; ++k) {
        __syncthreads();
        const long long r = row0 + (long long)k * p.F;
        for (int m = threadIdx.x; m < p.F; m += NT) {
            const int g = map_g[r + m];
            const double c = map_c[r + m];
            phi_start[r + p.F + m] = g < 0 ? c : wrap(phi_start[r + g] + c);
        }
    }
}

struct Layout {
    int chunks, chunk_len;
    bool global_work;
    size_t cta_bytes, off_maps_g, off_maps_c, off_phi, off_scratch, total;
};

// Whether a CTA's working set (cta_bytes) exceeds the current device's shared memory and lives in global memory.
// static_extra: static shared memory of the kernel beyond the scan buffers (the stream mode's block max).
template <typename T> static int global_work(int F, size_t static_extra, size_t* cta_bytes, bool* global) {
    *cta_bytes = work_bytes<T>(F, nullptr, nullptr);
    int dev = 0, smem_optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return (int)e;
    const size_t static_smem = 2 * NW * (sizeof(Reach<T>) + sizeof(Seg)) + static_extra;
    *global = *cta_bytes + static_smem > (size_t)smem_optin;
    return 0;
}

template <typename T> static int layout(int B, int F, int T_, Layout* L) {
    int rc = global_work<T>(F, 0, &L->cta_bytes, &L->global_work);
    if (rc) return rc;
    cudaError_t e;
    int per_sm = 1;
    if (!L->global_work) {
        e = cudaFuncSetAttribute(pghi_frames_kernel<T, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L->cta_bytes);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(pghi_frames_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)L->cta_bytes);
        if (e == cudaSuccess)
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pghi_frames_kernel<T, 0>, NT, L->cta_bytes);
        if (e != cudaSuccess) return (int)e;
    } else {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pghi_frames_kernel<T, 0>, NT, 0);
        if (e != cudaSuccess) return (int)e;
    }
    // split time only when the signals leave more than half of the resident CTA slots idle; the split runs the
    // per-frame structure twice (compose, apply) plus the carry
    const long long slots = (long long)SMS * (per_sm > 0 ? per_sm : 1);
    long long chunks = 1;
    if (2LL * B < slots) chunks = (slots + B - 1) / B;
    if (chunks > T_ / MIN_CHUNK) chunks = T_ / MIN_CHUNK;
    if (chunks < 1) chunks = 1;
    L->chunk_len = (int)((T_ + chunks - 1) / chunks);
    L->chunks = (int)((T_ + L->chunk_len - 1) / L->chunk_len);
    const size_t rows = (size_t)B * L->chunks * F;
    size_t o = al16((size_t)B * 8);
    L->off_maps_g = o; if (L->chunks > 1) o = al16(o + rows * 4);
    L->off_maps_c = o; if (L->chunks > 1) o = al16(o + rows * 8);
    L->off_phi = o;    if (L->chunks > 1) o = al16(o + rows * 8);
    L->off_scratch = o; if (L->global_work) o += (size_t)B * L->chunks * L->cta_bytes;
    L->total = o;
    return 0;
}

template <typename T>
static int run(Params p, const void* mag, void* out, char* ws, size_t ws_bytes, cudaStream_t st) {
    Layout L;
    int rc = layout<T>(p.B, p.F, p.T, &L);
    if (rc) return rc;
    if (ws_bytes < L.total) return SPECINV_ERR_INVALID;
    if ((long long)p.B * L.chunks > INT_MAX) return SPECINV_ERR_UNSUPPORTED;
    p.chunks = L.chunks;
    p.chunk_len = L.chunk_len;
    p.cta_bytes = L.cta_bytes;
    auto* maxbits = (unsigned long long*)ws;
    int* map_g = (int*)(ws + L.off_maps_g);
    double* map_c = (double*)(ws + L.off_maps_c);
    double* phi = (double*)(ws + L.off_phi);
    char* scratch = L.global_work ? ws + L.off_scratch : nullptr;
    const size_t dyn = L.global_work ? 0 : L.cta_bytes;
    const T* m = (const T*)mag;
    cudaError_t e = cudaMemsetAsync(maxbits, 0, (size_t)p.B * 8, st);
    if (e != cudaSuccess) return (int)e;
    const int gx = (int)std::min<long long>(p.T, std::max<long long>(1, (SMS * 8 + p.B - 1) / p.B));
    pghi_max_kernel<T><<<dim3(gx, p.B), NT, 0, st>>>(p, m, maxbits);
    if (L.chunks > 1) {
        pghi_frames_kernel<T, 1><<<p.B * (L.chunks - 1), NT, dyn, st>>>(p, m, maxbits, nullptr, map_g, map_c, nullptr,
                                                                           scratch);
        pghi_carry_kernel<<<p.B, NT, 0, st>>>(p, map_g, map_c, phi);
    }
    pghi_frames_kernel<T, 0><<<p.B * L.chunks, NT, dyn, st>>>(p, m, maxbits, phi, nullptr, nullptr, (cx_t<T>*)out,
                                                                 scratch);
    return (int)cudaGetLastError();
}

static bool valid_sizes(int dtype, int batch, int n_bins, int64_t n_frames) {
    return (dtype == SPECINV_F32 || dtype == SPECINV_F64) && batch >= 1 && batch <= 65535 && n_bins >= 2 &&
           n_frames >= 1 && n_frames <= INT_MAX;
}

// Stream state: [batch] rows of StreamHead + running phase, then, when the working set does not fit in shared memory,
// [batch] CTA working sets.
template <typename T> static int stream_state_bytes(int B, int F, size_t* bytes, size_t* cta_bytes, bool* global) {
    const int rc = global_work<T>(F, NW * sizeof(double), cta_bytes, global);
    if (rc) return rc;
    *bytes = (size_t)B * stream_row_bytes(F) + (*global ? (size_t)B * *cta_bytes : 0);
    return 0;
}

template <typename T>
static int run_stream(Params p, const void* mag, Stream sm, char* state, size_t state_bytes, void* out,
                      cudaStream_t st) {
    size_t need = 0;
    bool global = false;
    int rc = stream_state_bytes<T>(p.B, p.F, &need, &p.cta_bytes, &global);
    if (rc) return rc;
    if (state_bytes < need) return SPECINV_ERR_INVALID;
    if (sm.n_fin == 0) return SPECINV_OK;
    char* scratch = global ? state + (size_t)p.B * stream_row_bytes(p.F) : nullptr;
    const size_t dyn = global ? 0 : p.cta_bytes;
    if (!global) {
        const cudaError_t e = cudaFuncSetAttribute(pghi_stream_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)dyn);
        if (e != cudaSuccess) return (int)e;
    }
    pghi_stream_kernel<T><<<p.B, NT, dyn, st>>>(p, (const T*)mag, sm, state, (cx_t<T>*)out, scratch);
    return (int)cudaGetLastError();
}

static bool valid_analysis(int n_bins, int n_fft, int hop, int win_length, double gamma, double tol) {
    return n_fft >= 2 && n_fft / 2 + 1 == n_bins && hop >= 1 && win_length >= 1 && win_length <= n_fft &&
           gamma > 0.0 && gamma < INFINITY && tol > 0.0 && tol < 1.0;
}

static Params analysis_params(int batch, int n_bins, int n_fft, int hop, int win_length, double gamma, double tol) {
    Params p{};
    p.B = batch; p.F = n_bins; p.M = n_fft; p.hop = hop;
    p.tol = tol;
    const double c = (n_fft - win_length) / 2 + win_length / 2.0;      // window centre inside the frame
    p.K0 = 2 * PI * c / n_fft;
    p.K1 = (double)hop * n_fft / gamma;
    p.K2 = gamma / ((double)n_fft * hop);
    return p;
}

}  // namespace pghi
}  // namespace specinv

extern "C" {

int specinv_pghi_workspace_bytes(int dtype, int batch, int n_bins, int64_t n_frames, size_t* bytes) {
    using namespace specinv::pghi;
    if (!bytes || !valid_sizes(dtype, batch, n_bins, n_frames)) return SPECINV_ERR_INVALID;
    Layout L;
    const int rc = dtype == SPECINV_F64 ? layout<double>(batch, n_bins, (int)n_frames, &L)
                                        : layout<float>(batch, n_bins, (int)n_frames, &L);
    if (rc) return rc;
    *bytes = L.total;
    return SPECINV_OK;
}

int specinv_pghi(int dtype, const void* mag, int64_t sb, int64_t sf, int64_t st, void* out, int batch, int n_bins,
                 int64_t n_frames, int n_fft, int hop, int win_length, double gamma, double tol, void* workspace,
                 size_t workspace_bytes, void* stream) {
    using namespace specinv::pghi;
    if (!valid_sizes(dtype, batch, n_bins, n_frames) || !mag || !out || !workspace) return SPECINV_ERR_INVALID;
    if (!valid_analysis(n_bins, n_fft, hop, win_length, gamma, tol)) return SPECINV_ERR_INVALID;
    Params p = analysis_params(batch, n_bins, n_fft, hop, win_length, gamma, tol);
    p.T = (int)n_frames;
    p.sb = sb; p.sf = sf; p.st = st;
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == SPECINV_F64 ? run<double>(p, mag, out, (char*)workspace, workspace_bytes, s)
                                : run<float>(p, mag, out, (char*)workspace, workspace_bytes, s);
}

int specinv_pghi_stream_state_bytes(int dtype, int batch, int n_bins, size_t* bytes) {
    using namespace specinv::pghi;
    if (!bytes || !valid_sizes(dtype, batch, n_bins, 1)) return SPECINV_ERR_INVALID;
    size_t cta = 0;
    bool global = false;
    return dtype == SPECINV_F64 ? stream_state_bytes<double>(batch, n_bins, bytes, &cta, &global)
                                : stream_state_bytes<float>(batch, n_bins, bytes, &cta, &global);
}

int specinv_pghi_stream(int dtype, const void* mag, int64_t sb, int64_t sf, int64_t st, int frame0, int n_rows,
                        int n_final, int final, void* state, size_t state_bytes, void* out, int batch, int n_bins,
                        int n_fft, int hop, int win_length, double gamma, double tol, void* stream) {
    using namespace specinv::pghi;
    if (!valid_sizes(dtype, batch, n_bins, n_rows) || !mag || !state || (n_final > 0 && !out)) return SPECINV_ERR_INVALID;
    if (!valid_analysis(n_bins, n_fft, hop, win_length, gamma, tol)) return SPECINV_ERR_INVALID;
    // rows: the frame before the first one finalised (unless that is frame 0), the n_final frames, and one frame of
    // look-ahead unless `final`
    const int ahead = final ? 0 : 1;
    if ((final != 0 && final != 1) || frame0 < 0 || n_final < 0 || n_rows - n_final - ahead < 0 ||
        (long long)frame0 + n_rows > INT_MAX)
        return SPECINV_ERR_INVALID;
    const int first = frame0 + n_rows - n_final - ahead;
    if (first > 0 && first - 1 < frame0) return SPECINV_ERR_INVALID;
    Params p = analysis_params(batch, n_bins, n_fft, hop, win_length, gamma, tol);
    p.T = frame0 + n_rows;
    p.chunks = 1;
    p.sb = sb; p.sf = sf; p.st = st;
    const Stream sm{frame0, first, n_final};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == SPECINV_F64 ? run_stream<double>(p, mag, sm, (char*)state, state_bytes, out, s)
                                : run_stream<float>(p, mag, sm, (char*)state, state_bytes, out, s);
}

}  // extern "C"
