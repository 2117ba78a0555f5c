// Per-lane building blocks of the "16 values per lane" fused iteration kernels (onesided, fp32, hop = n_fft/4):
//   LANES =  32: n_fft = 1024, hop =  256 -- one warp per frame        (M = 512  = 8 x 8 x 8)
//   LANES =  64: n_fft = 2048, hop =  512 -- two warps per frame       (M = 1024 = 8 x 16 x 8)
//   LANES = 128: n_fft = 4096, hop = 1024 -- four warps per frame      (M = 2048 = 16 x 16 x 8)
//
// A frame's real FFT of N points is a complex FFT of M = N/2 = R1 x R2 x 8 points done by LANES lanes holding
// 16 complex values each, in three passes with two exchanges through shared memory per direction.  With
// n = 8 R2 a + 8 b + c and k = ka + R1 kb + R1 R2 kc:
//   pass 1 : lane l owns z[LANES i + l], i = 0..15: 16/R1 FFTs of R1 points over a, times W_M^((8 b + c) ka)
//                                                                              -- exchange E1 (ka, b, c) --
//   pass 2 : lane l owns (ka = (l >> 3) + (LANES / 8) r, c = l & 7), r < 16/R2: FFTs of R2 points over b,
//            times W_(8 R2)^(c kb)                                             -- exchange E2 (k1, c) --
//   pass 3 : lane l owns the residue classes k1 = ka + R1 kb in {l, 2 LANES - l} ({0, LANES} for l = 0): two
//            FFT8 over c -> Zh[k1 + 2 LANES kc].
// Class 2 LANES - l is the mirror (k -> M - k) of class l, so every (Z[k], Z[M-k]) pair of the real-FFT
// post/pre-processing lives in ONE thread: projection and momentum / ADMM update run in registers on the FFT
// outputs; for a fixed kc consecutive lanes touch consecutive bins (coalesced rows of q / mag).  The inverse
// runs the passes backwards.
// A hop is 4 of a lane's 16 sample pairs (i -> i + 4): overlap-add is a per-thread shift-accumulate and the
// input ring is thread-private.
//
// 16 complex values per lane keep the kernels under 168 registers (12 free-running warps per SM, no lockstep)
// and the fully unrolled frame body (~28 KB) inside the instruction cache.
//
// Everything is __host__ __device__: tests/host_emu runs the exact index logic on the CPU.
#pragma once

#include "fft_regs.cuh"

namespace specinv {
namespace wfast {

// OP_ISTFT: stand-alone inverse transform + overlap-add (methods.py:233); OP_GLP: plain Griffin-Lim (alpha = 0:
// q_n = STFT(x_{n-1}), so no momentum state is read or written); OP_GLR: fast Griffin-Lim with the momentum taken on
// the previous REBUILT spectrum (torchaudio.functional.griffinlim): the state is s = STFT(x_{n-1}) itself, the
// projection gets s - m s_prev.  Same traffic as OP_GL, only the stored value differs.
enum { OP_GL = 0, OP_ADMM = 1, OP_ISTFT = 2, OP_GLP = 3, OP_GLR = 4 };

// complex products on the packed FP32x2 pipe (fft_regs.cuh): 2 instructions each
SPX_HD float2 cmulf(float2 a, float2 b) { return cmul2(a, b); }
SPX_HD float2 cmulcf(float2 a, float2 b) { return cmulc2(a, b); }     // a*conj(b)

#ifdef __CUDA_ARCH__
__device__ __forceinline__ float approx_sqrt(float v) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
__device__ __forceinline__ float approx_rsqrt(float v) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
#else
inline float approx_sqrt(float v) { return sqrtf(v); }
inline float approx_rsqrt(float v) { return 1.0f / sqrtf(v); }
#endif

// real-FFT post-process of one (P = Zh[k], Q = Zh[M-k]) pair, Zh = Z/2 (the 1/2 is folded into the analysis
// window):  s[k], s[M-k] of the N-point real transform; w = W_N^k
SPX_HD void post_pair(float2 P, float2 Q, float2 w, float2& sP, float2& sQ) {
    const float2 E = P + f2(Q.x, -Q.y);                 // (er, ei)   = P + conj(Q)
    const float2 O = f2(P.y, -P.x) + f2(Q.y, Q.x);      // (orr, oi)  = -i (P - conj(Q))
    const float2 WO = cmul2(O, w);                      // (wor, woi)
    sP = E + WO;
    const float2 D = E - WO;
    sQ = f2(D.x, -D.y);                                 // (er - wor, woi - ei)
}
// (wc = conj(w) from a table, or nullptr-equivalent HC = false: computed on the fly)
template <bool HC>
SPX_HD void post_pair_t(float2 P, float2 Q, float2 w, float2 wc, float2& sP, float2& sQ) {
    const float2 E = P + f2(Q.x, -Q.y);
    const float2 O = f2(P.y, -P.x) + f2(Q.y, Q.x);
    const float2 WO = HC ? cmul2t(O, w, wc) : cmul2(O, w);
    sP = E + WO;
    const float2 D = E - WO;
    sQ = f2(D.x, -D.y);
}
template <bool HC>
SPX_HD void pre_pair_t(float2 hP, float2 hQ, float2 w, float2 wc, float2& P, float2& Q) {
    const float2 A = hP + f2(hQ.x, -hQ.y);
    const float2 D = hP - f2(hQ.x, -hQ.y);
    const float2 G = HC ? cmulc2t(D, w, wc) : cmulc2(D, w);
    P = A + f2(-G.y, G.x);
    const float2 R = A - f2(-G.y, G.x);
    Q = f2(R.x, -R.y);
}
// inverse pre-process: (h[k], h[M-k]) -> (Z'[k], Z'[M-k]), the inputs of the M-point inverse complex FFT
SPX_HD void pre_pair(float2 hP, float2 hQ, float2 w, float2& P, float2& Q) {
    const float2 A = hP + f2(hQ.x, -hQ.y);              // (Ar, Ai) = hP + conj(hQ)
    const float2 D = hP - f2(hQ.x, -hQ.y);              // (Dr, Di) = hP - conj(hQ)
    const float2 G = cmulc2(D, w);                      // (Gr, Gi) = D * conj(w)
    P = A + f2(-G.y, G.x);                              // (Ar - Gi, Ai + Gr) = A + i G
    const float2 R = A - f2(-G.y, G.x);                 // (Ar + Gi, Ai - Gr)
    Q = f2(R.x, -R.y);                                  // (Ar + Gi, Gr - Ai)
}

constexpr int V = 16;            // complex values per lane (8 for the n_fft = 512 variant: template parameter VV)

template <int LANES, int VV = V>
struct Cfg {
    static_assert(LANES == 32 || LANES == 64 || LANES == 128, "LANES");
    static_assert(VV == 16 || (VV == 8 && LANES == 32), "values per lane");
    static constexpr int M = VV * LANES;          // complex FFT size = bins in a main row
    static constexpr int N = 2 * M;               // n_fft
    static constexpr int HOP = N / 4;             // samples
    static constexpr int RC = VV / 2;             // radix of pass 3 = values per residue class (8; 4 when VV = 8)
    static constexpr int LOGRC = RC == 8 ? 3 : 2;
    static constexpr int R1 = LANES == 128 ? 16 : 8;
    static constexpr int R2 = M / (R1 * RC);      // 8, 16, 16 (VV = 16); 8 (VV = 8)
    static constexpr int S1 = VV / R1;            // pass-1 transforms per lane
    static constexpr int S2 = VV / R2;            // pass-2 transforms per lane
};

template <int R, bool INV> SPX_HD void fft_small(float2* t) {
    if constexpr (R == 4) fft4<INV>(t[0], t[1], t[2], t[3]);
    else if constexpr (R == 8) fft8<INV>(t);
    else fft16<INV>(t);
}

// ---- exchange addressing (float2 units), XOR-swizzled 16-byte columns, no padding --------------------------
// E1: rows (ka, c) -> RC ka + c of R2 float2; E2: rows k1 of RC float2.  The swizzle makes both the 128-bit row
// accesses (8 consecutive rows per quarter-warp) and the 64-bit scattered accesses conflict free
// (tests/host_emu/test_warp_core.cu counts the wavefronts of every access).
// GRP = 4: E1 of the 8-values-per-lane variant, whose rows come in groups of RC = 4 (the scattered side varies c in
// the low two row bits), needs the two swizzle bits the other way round.
template <int RLEN, int GRP = 8> SPX_HD int ex_swz(int row) {
    if constexpr (RLEN == 4) return (row >> 2) & 1;
    else if constexpr (RLEN == 8 && GRP == 4) return (((row >> 1) & 1) << 1) | ((row >> 2) & 1);
    else if constexpr (RLEN == 8) return (row >> 1) & 3;
    else return row & 7;
}
template <int RLEN, int GRP = 8> SPX_HD int ex_addr(int row, int col) {
    return RLEN * row + 2 * (((col >> 1) ^ ex_swz<RLEN, GRP>(row)) & (RLEN / 2 - 1)) + (col & 1);
}
// 128-bit access: elements (row, 2 p) and (row, 2 p + 1)
template <int RLEN, int GRP = 8> SPX_HD int ex_addr4(int row, int p) {
    return RLEN * row + 2 * ((p ^ ex_swz<RLEN, GRP>(row)) & (RLEN / 2 - 1));
}

template <int LANES> SPX_HD int class_b(int l) { return l == 0 ? LANES : 2 * LANES - l; }
// bin of the P element of pair slot j (the Q element is bin M - kP); lane 0 slot 0 is the special
// DC / Nyquist / bin-M/2 slot
template <int LANES, int VV = V> SPX_HD int slot_bin_rt(int l, int j) {
    constexpr int H = VV / 4;
    return l != 0 ? l + 2 * LANES * j : (j < H ? 2 * LANES * j : LANES + 2 * LANES * (j - H));
}

// Per-lane constant tables (the kernel keeps them in tensor memory, the host emulation in arrays)
template <int LANES, int VV = V>
struct LaneTables {
    float2 wa[VV];                    // 0.5 * analysis window pairs (w[2 LANES i + 2 l], w[2 LANES i + 2 l + 1])
    float2 ws[VV];                    // synthesis window pairs (already scaled by 1/N or N^-1/2)
    float2 tw1[VV];                   // [R1 s + ka]  W_M^((l + LANES s) ka)
    float2 tw2[Cfg<LANES, VV>::R2];   // [kb]         W_(RC R2)^((l & (RC-1)) kb)
    float2 twr[VV / 2];               // [j]          W_N^(slot_bin(l, j))
};

// ---- forward ---------------------------------------------------------------------------------------------
// v[i] = windowed z[LANES i + l] on entry
template <int LANES, int VV = V, bool HC = false>
SPX_HD void fwd_pass1(int l, float2* v, const float2* tw1, float2* e1, const float2* tw1c = nullptr) {
    using C = Cfg<LANES, VV>;
    const int c = l & (C::RC - 1);
    static_for<C::S1>([&](auto sc) {
        constexpr int s = decltype(sc)::value;
        float2 t[C::R1];
        static_for<C::R1>([&](auto ac) { constexpr int a = decltype(ac)::value; t[a] = v[C::S1 * a + s]; });
        fft_small<C::R1, false>(t);
        const int b = (l + LANES * s) >> C::LOGRC;
        static_for<C::R1>([&](auto kc) {
            constexpr int ka = decltype(kc)::value;
            const float2 y = ka == 0 ? t[0] : (HC ? cmul2t(t[ka], tw1[C::R1 * s + ka], tw1c[C::R1 * s + ka]) : cmulf(t[ka], tw1[C::R1 * s + ka]));
            e1[ex_addr<C::R2, C::RC>(C::RC * ka + c, b)] = y;
        });
    });
}

template <int LANES, int VV = V, bool HC = false>
SPX_HD void fwd_pass2(int l, const float2* e1, const float2* tw2, float2* e2, const float2* tw2c = nullptr) {
    using C = Cfg<LANES, VV>;
    const int c = l & (C::RC - 1);
    static_for<C::S2>([&](auto rc) {
        constexpr int r = decltype(rc)::value;
        const int ka = (l >> C::LOGRC) + (LANES / C::RC) * r;
        float2 t[C::R2];
        static_for<C::R2 / 2>([&](auto pc) {
            constexpr int p = decltype(pc)::value;
            const float4 q = *reinterpret_cast<const float4*>(e1 + ex_addr4<C::R2, C::RC>(C::RC * ka + c, p));
            t[2 * p] = f2(q.x, q.y); t[2 * p + 1] = f2(q.z, q.w);
        });
        fft_small<C::R2, false>(t);
        static_for<C::R2>([&](auto kc) {
            constexpr int kb = decltype(kc)::value;
            const float2 y = kb == 0 ? t[0] : (HC ? cmul2t(t[kb], tw2[kb], tw2c[kb]) : cmulf(t[kb], tw2[kb]));
            e2[ex_addr<C::RC>(ka + C::R1 * kb, c)] = y;
        });
    });
}

// A[kc] = Zh[l + 2 LANES kc], B[kc] = Zh[class_b(l) + 2 LANES kc]
template <int LANES, int VV = V>
SPX_HD void fwd_pass3(int l, const float2* e2, float2* A, float2* B) {
    constexpr int RC = VV / 2;
    const int ra = l, rb = class_b<LANES>(l);
    static_for<RC / 2>([&](auto pc) {
        constexpr int p = decltype(pc)::value;
        const float4 qa = *reinterpret_cast<const float4*>(e2 + ex_addr4<RC>(ra, p));
        const float4 qb = *reinterpret_cast<const float4*>(e2 + ex_addr4<RC>(rb, p));
        A[2 * p] = f2(qa.x, qa.y); A[2 * p + 1] = f2(qa.z, qa.w);
        B[2 * p] = f2(qb.x, qb.y); B[2 * p + 1] = f2(qb.z, qb.w);
    });
    fft_small<RC, false>(A);
    fft_small<RC, false>(B);
}

// ---- point-wise stage ------------------------------------------------------------------------------------
// q * mag / (|q| + 1e-16) (methods.py:246-247) with ONE special-function op: mag * rsqrt(|q|^2 + 1e-32).  The two
// agree to rounding unless |q| ~ 1e-16 (where both give q * mag * ~1e16), and |q| = 0 gives 0, not NaN.
SPX_HD float2 project_rsq(float2 q, float mag) {
    const float s = mag * approx_rsqrt(q.x * q.x + (q.y * q.y + 1e-32f));
    return smul2(q, s);
}

// One bin: s = STFT bin of the current estimate.  Returns the value fed to the inverse transform.
template <int OP, bool SUMS>
SPX_HD float2 bin_update(float2 s, float2 a0, float2 a1, float m, float coef, float coef2, float2& o0, float2& o1,
                         float& dsum, float& esum) {
    if constexpr (SUMS) {
        const float r = approx_sqrt(s.x * s.x + s.y * s.y);
        dsum += (r - m) * (r - m);
        esum += r * r;
    }
    if constexpr (OP == OP_GLP) {
        return project_rsq(s, m);
    } else if constexpr (OP == OP_GL) {
        const float2 q = pfma(f2(-coef, -coef), a0, s);             // s - lr * q_prev
        o0 = q;
        return project_rsq(q, m);
    } else if constexpr (OP == OP_GLR) {
        o0 = s;                                                     // state: the rebuilt spectrum
        return project_rsq(pfma(f2(-coef, -coef), a0, s), m);       // s - m * s_prev
    } else {
        const float rho = coef, inv = coef2;
        const float2 XU = a0 + a1;
        const float2 Z = smul2(pfma(f2(rho, rho), XU, s), inv);      // (rho (X + U) + s) / (1 + rho)
        const float2 Un = XU - Z;
        const float2 Xn = project_rsq(Z - Un, m);
        o0 = Xn; o1 = Un;
        return Xn + Un;
    }
}

// Pair processing with the point-wise update, in place: on return A / B hold the inputs of the inverse
// pass 3.  (dsum, esum) += this lane's share of sum (|s|-mag)^2, sum |s|^2.
// `io` gives access to the state of the lane's bins, element e = 2 j (the P bin of slot j) or 2 j + 1 (the Q
// bin; lane 0 slot 0: bins 0 and M/2), e = -1: the Nyquist bin (lane 0 only):
//     float2 io.s0(e), io.s1(e); float io.mag(e); void io.put(e, o0, o1)
// so that values are fetched right where they are used (no block of 48 live registers).
template <int OP, bool SUMS, int VV = V, bool HC = false, typename IO>
SPX_HD void pointwise(int l, float2* A, float2* B, const float2* twr, IO& io, float coef, float coef2, float& dsum,
                      float& esum, const float2* twrc = nullptr) {
    constexpr int RC = VV / 2, H = RC / 2;      // pair slots per lane; lane 0 pairs inside its two classes
    const bool l0 = l == 0;
    auto upd = [&](auto ec, float2 sv) {
        constexpr int e = decltype(ec)::value;
        float2 o0 = f2(0.f, 0.f), o1 = f2(0.f, 0.f);
        const float2 h = bin_update<OP, SUMS>(sv, OP == OP_GLP ? f2(0.f, 0.f) : io.s0(e),
                                              OP == OP_ADMM ? io.s1(e) : f2(0.f, 0.f), io.mag(e), coef, coef2, o0, o1, dsum, esum);
        if constexpr (OP != OP_GLP) io.put(e, o0, o1);
        return h;
    };
    // slot 0
    if (l0) {
        // lane 0: A[0] = Zh[0] -> DC and Nyquist (both real), A[H] = Zh[M/2] -> bin M/2 = conj(Z[M/2])
        const float2 z0 = A[0], z4 = A[H];
        const float2 h0 = upd(std::integral_constant<int, 0>{}, f2(2.f * (z0.x + z0.y), 0.f));
        const float2 hM = upd(std::integral_constant<int, -1>{}, f2(2.f * (z0.x - z0.y), 0.f));
        const float2 h4 = upd(std::integral_constant<int, 1>{}, f2(2.f * z4.x, -2.f * z4.y));
        A[0] = f2(h0.x + hM.x, h0.x - hM.x);        // C2R ignores Im(DC), Im(Nyquist)
        A[H] = f2(2.f * h4.x, -2.f * h4.y);
    } else {
        float2 sP, sQ, P, Q;
        const float2 w = twr[0], wc = HC ? twrc[0] : w;
        post_pair_t<HC>(A[0], B[RC - 1], w, wc, sP, sQ);
        const float2 hP = upd(std::integral_constant<int, 0>{}, sP);
        const float2 hQ = upd(std::integral_constant<int, 1>{}, sQ);
        pre_pair_t<HC>(hP, hQ, w, wc, P, Q);
        A[0] = P; B[RC - 1] = Q;
    }
    // slots 1..RC-1.  general lanes: (A[j], B[RC-1-j]); lane 0, j < H: (A[j], A[RC-j]); lane 0, j >= H:
    // (B[j-H], B[RC-1-(j-H)])
    static_for<RC - 1>([&](auto jc) {
        constexpr int j = decltype(jc)::value + 1;
        float2 P, Q;
        if constexpr (j < H) { P = A[j]; Q = l0 ? A[RC - j] : B[RC - 1 - j]; }
        else { P = l0 ? B[j - H] : A[j]; Q = l0 ? B[RC - 1 - (j - H)] : B[RC - 1 - j]; }
        const float2 w = twr[j], wc = HC ? twrc[j] : w;
        float2 sP, sQ;
        post_pair_t<HC>(P, Q, w, wc, sP, sQ);
        const float2 hP = upd(std::integral_constant<int, 2 * j>{}, sP);
        const float2 hQ = upd(std::integral_constant<int, 2 * j + 1>{}, sQ);
        pre_pair_t<HC>(hP, hQ, w, wc, P, Q);
        if constexpr (j < H) { A[j] = P; if (l0) A[RC - j] = Q; else B[RC - 1 - j] = Q; }
        else { if (l0) { B[j - H] = P; B[RC - 1 - (j - H)] = Q; } else { A[j] = P; B[RC - 1 - j] = Q; } }
    });
}

// Stand-alone inverse transform (ISTFT): the given spectrum h replaces the point-wise stage; on return A / B hold
// the inputs of the inverse pass 3.  `io.s0(e)` as above (e = -1: the Nyquist bin).
template <int VV = V, bool HC = false, typename IO>
SPX_HD void spectrum_pairs(int l, float2* A, float2* B, const float2* twr, IO& io, const float2* twrc = nullptr) {
    constexpr int RC = VV / 2, H = RC / 2;
    const bool l0 = l == 0;
    if (l0) {
        const float2 h0 = io.s0(0), hM = io.s0(-1), h4 = io.s0(1);
        A[0] = f2(h0.x + hM.x, h0.x - hM.x);        // C2R ignores Im(DC), Im(Nyquist)
        A[H] = f2(2.f * h4.x, -2.f * h4.y);
    } else {
        pre_pair_t<HC>(io.s0(0), io.s0(1), twr[0], HC ? twrc[0] : twr[0], A[0], B[RC - 1]);
    }
    static_for<RC - 1>([&](auto jc) {
        constexpr int j = decltype(jc)::value + 1;
        float2 P, Q;
        pre_pair_t<HC>(io.s0(2 * j), io.s0(2 * j + 1), twr[j], HC ? twrc[j] : twr[j], P, Q);
        if constexpr (j < H) { A[j] = P; if (l0) A[RC - j] = Q; else B[RC - 1 - j] = Q; }
        else { if (l0) { B[j - H] = P; B[RC - 1 - (j - H)] = Q; } else { A[j] = P; B[RC - 1 - j] = Q; } }
    });
}

// ---- inverse ---------------------------------------------------------------------------------------------
template <int LANES, int VV = V>
SPX_HD void inv_pass3(int l, float2* A, float2* B, float2* e2) {
    constexpr int RC = VV / 2;
    fft_small<RC, true>(A);       // A[c] = Y2'[class a, c]
    fft_small<RC, true>(B);
    const int ra = l, rb = class_b<LANES>(l);
    static_for<RC / 2>([&](auto pc) {
        constexpr int p = decltype(pc)::value;
        *reinterpret_cast<float4*>(e2 + ex_addr4<RC>(ra, p)) = make_float4(A[2 * p].x, A[2 * p].y, A[2 * p + 1].x, A[2 * p + 1].y);
        *reinterpret_cast<float4*>(e2 + ex_addr4<RC>(rb, p)) = make_float4(B[2 * p].x, B[2 * p].y, B[2 * p + 1].x, B[2 * p + 1].y);
    });
}

template <int LANES, int VV = V, bool HC = false>
SPX_HD void inv_pass2(int l, const float2* e2, const float2* tw2, float2* e1, const float2* tw2c = nullptr) {
    using C = Cfg<LANES, VV>;
    const int c = l & (C::RC - 1);
    static_for<C::S2>([&](auto rc) {
        constexpr int r = decltype(rc)::value;
        const int ka = (l >> C::LOGRC) + (LANES / C::RC) * r;
        float2 t[C::R2];
        static_for<C::R2>([&](auto kc) {
            constexpr int kb = decltype(kc)::value;
            const float2 y = e2[ex_addr<C::RC>(ka + C::R1 * kb, c)];
            t[kb] = kb == 0 ? y : (HC ? cmulc2t(y, tw2[kb], tw2c[kb]) : cmulcf(y, tw2[kb]));
        });
        fft_small<C::R2, true>(t);   // t[b] = Y1'[ka, b, c] (before the pass-1 twiddle)
        static_for<C::R2 / 2>([&](auto pc) {
            constexpr int p = decltype(pc)::value;
            *reinterpret_cast<float4*>(e1 + ex_addr4<C::R2, C::RC>(C::RC * ka + c, p)) =
                make_float4(t[2 * p].x, t[2 * p].y, t[2 * p + 1].x, t[2 * p + 1].y);
        });
    });
}

// v[i] = z'[LANES i + l] (unscaled)
template <int LANES, int VV = V, bool HC = false>
SPX_HD void inv_pass1(int l, const float2* e1, const float2* tw1, float2* v, const float2* tw1c = nullptr) {
    using C = Cfg<LANES, VV>;
    const int c = l & (C::RC - 1);
    static_for<C::S1>([&](auto sc) {
        constexpr int s = decltype(sc)::value;
        const int b = (l + LANES * s) >> C::LOGRC;
        float2 t[C::R1];
        static_for<C::R1>([&](auto kc) {
            constexpr int ka = decltype(kc)::value;
            const float2 y = e1[ex_addr<C::R2, C::RC>(C::RC * ka + c, b)];
            t[ka] = ka == 0 ? y : (HC ? cmulc2t(y, tw1[C::R1 * s + ka], tw1c[C::R1 * s + ka]) : cmulcf(y, tw1[C::R1 * s + ka]));
        });
        fft_small<C::R1, true>(t);
        static_for<C::R1>([&](auto ac) { constexpr int a = decltype(ac)::value; v[C::S1 * a + s] = t[a]; });
    });
}

}  // namespace wfast
}  // namespace specinv
