// Argument block and point-wise stage shared by the generic tile kernels (specinv_generic.cu: radix-2^2 and direct
// DFT; specinv_generic_mr.cu: mixed radix).
#pragma once

#include "specinv_common.cuh"

namespace specinv {

// OP_GLR: fast Griffin-Lim with the momentum on the previous rebuilt spectrum (torchaudio.functional.griffinlim):
// state out = s, projection of s - lr * s_prev
enum { OP_STFT = 0, OP_ISTFT = 1, OP_GL = 2, OP_ADMM = 3, OP_GLR = 4 };

struct TileArgs {
    const void* x_in;
    void* x_out;
    const void* s0_in_main;  const void* s0_in_nyq;   // GL: q_in   ADMM: X_in   ISTFT: spectrum
    void* s0_out_main;       void* s0_out_nyq;        // GL: q_out  ADMM: X_out  STFT: spectrum
    const void* s1_in_main;  const void* s1_in_nyq;   // ADMM: U_in
    void* s1_out_main;       void* s1_out_nyq;        // ADMM: U_out
    const void* mag_main;    const void* mag_nyq;
    const void* tw; const void* twr; const void* wa; const void* ws; const void* inv_env;
    double* sums;
    double coef;       // GL: lr = alpha/(1+alpha)   ADMM: rho
    Dims dm;
    int tile_frames;   // owned frames per tile
    int Mp;            // padded complex elements per frame in shared memory
};

// Addresses of the bins of one (signal, frame) row.  NYQ = false: the caller guarantees kk != M (every (k, M-k) pair
// but k = 0), so the onesided layout's separate Nyquist array never enters the address arithmetic.
template <typename T, bool NYQ = true>
struct BinIO {
    const TileArgs& a;
    long long fr;     // b*T + t
    long long roff;   // fr * row: element offset of the frame's main row
    __device__ BinIO(const TileArgs& a_, long long fr_) : a(a_), fr(fr_), roff(fr_ * a_.dm.row) {}
    __device__ __forceinline__ cx_t<T> ldc(const void* main, const void* nyq, int kk) const {
        // read-only path (ld.global.nc): the inputs are never written by the launch (ping-pong state), and the
        // compiler may then batch the loads of unrolled iterations ahead of the stores
        if (NYQ && a.dm.onesided && kk == a.dm.M) return __ldg((const cx_t<T>*)nyq + fr);
        return __ldg((const cx_t<T>*)main + roff + kk);
    }
    __device__ __forceinline__ void stc(void* main, void* nyq, int kk, cx_t<T> v) const {
        if (NYQ && a.dm.onesided && kk == a.dm.M) ((cx_t<T>*)nyq)[fr] = v;
        else ((cx_t<T>*)main)[roff + kk] = v;
    }
    __device__ __forceinline__ T ldm(int kk) const {
        if (NYQ && a.dm.onesided && kk == a.dm.M) return __ldg((const T*)a.mag_nyq + fr);
        return __ldg((const T*)a.mag_main + roff + kk);
    }
};

// Point-wise stage for one frequency bin, split into its global loads (`bin_load`: issued early / batched by the
// callers that pipeline) and the arithmetic + stores (`bin_apply`).  s = STFT bin of the current signal estimate;
// bin_apply returns the spectrum value that goes into the inverse transform.
template <typename T>
struct BinIn {
    cx_t<T> s0, s1;   // GL: q_prev / ADMM: X, U / ISTFT: spectrum
    T m;              // target magnitude
};

template <typename T, int OP, typename IO>
__device__ __forceinline__ BinIn<T> bin_load(const TileArgs& a, const IO& io, int kk) {
    BinIn<T> in;
    in.s0 = mk<T>(T(0), T(0)); in.s1 = in.s0; in.m = T(0);
    if constexpr (OP == OP_ISTFT) {
        in.s0 = io.ldc(a.s0_in_main, a.s0_in_nyq, kk);
    } else if constexpr (OP == OP_GL || OP == OP_GLR) {
        in.m = io.ldm(kk);
        if (a.s0_in_main != nullptr) in.s0 = io.ldc(a.s0_in_main, a.s0_in_nyq, kk);
    } else if constexpr (OP == OP_ADMM) {
        in.s0 = io.ldc(a.s0_in_main, a.s0_in_nyq, kk);
        in.s1 = io.ldc(a.s1_in_main, a.s1_in_nyq, kk);
        in.m = io.ldm(kk);
    }
    return in;
}

template <typename T, int OP, typename IO>
__device__ __forceinline__ cx_t<T> bin_apply(const TileArgs& a, const IO& io, int kk, cx_t<T> s, const BinIn<T>& in,
                                             bool owned, bool want_sums, T& dsum, T& esum) {
    if constexpr (OP == OP_STFT) {
        io.stc(a.s0_out_main, a.s0_out_nyq, kk, s);
        return s;
    } else if constexpr (OP == OP_ISTFT) {
        return in.s0;
    } else if constexpr (OP == OP_GL || OP == OP_GLR) {
        // methods.py:243-247 (OP_GLR: torchaudio's griffinlim, the state is s itself)
        const T lr = (T)a.coef;
        const bool momentum = a.s0_in_main != nullptr;     // NULL state: plain Griffin-Lim (lr == 0), q_n = s
        const T m = in.m;
        if constexpr (OP == OP_GLR) {       // the state is s: store it before q is formed (fewer live registers)
            if (owned && momentum) io.stc(a.s0_out_main, a.s0_out_nyq, kk, s);
        }
        cx_t<T> q = s;
        if (momentum) q = mk<T>(s.x - in.s0.x * lr, s.y - in.s0.y * lr);
        if (owned) {
            if (OP == OP_GL && momentum) io.stc(a.s0_out_main, a.s0_out_nyq, kk, q);
            if (want_sums) {
                T r = fast_sqrt(s.x * s.x + s.y * s.y);
                dsum += (r - m) * (r - m);
                esum += r * r;
            }
        }
        return project<T>(q, m);
    } else {
        // methods.py:467-475 with Y = X + U
        const T rho = (T)a.coef;
        const T inv = T(1) / (T(1) + rho);
        const cx_t<T> X = in.s0, U = in.s1;
        const T m = in.m;
        cx_t<T> Z = mk<T>((rho * (X.x + U.x) + s.x) * inv, (rho * (X.y + U.y) + s.y) * inv);
        cx_t<T> Un = mk<T>(U.x + X.x - Z.x, U.y + X.y - Z.y);
        cx_t<T> Xn = project<T>(mk<T>(Z.x - Un.x, Z.y - Un.y), m);
        if (owned) {
            io.stc(a.s0_out_main, a.s0_out_nyq, kk, Xn);
            io.stc(a.s1_out_main, a.s1_out_nyq, kk, Un);
            if (want_sums) {
                T r = fast_sqrt(s.x * s.x + s.y * s.y);
                dsum += (r - m) * (r - m);
                esum += r * r;
            }
        }
        return mk<T>(Xn.x + Un.x, Xn.y + Un.y);
    }
}

template <typename T, int OP, typename IO>
__device__ __forceinline__ cx_t<T> bin_update(const TileArgs& a, const IO& io, int kk, cx_t<T> s,
                                              bool owned, bool want_sums, T& dsum, T& esum) {
    const BinIn<T> in = bin_load<T, OP>(a, io, kk);
    return bin_apply<T, OP>(a, io, kk, s, in, owned, want_sums, dsum, esum);
}

// implemented in specinv_generic_mr.cu: SPECINV_ERR_UNSUPPORTED when M = n_fft / 2 has a prime factor > 13
int mr_tile_launch(int dtype, int op, TileArgs& a, cudaStream_t st);

}  // namespace specinv
