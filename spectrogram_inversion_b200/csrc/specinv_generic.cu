// Generic (any power-of-two n_fft, any hop, every torch.stft option the reference forwards)
// fused tile kernels: STFT, ISTFT, one Griffin-Lim iteration, one ADMM iteration.
//
// One CTA owns a tile of consecutive frames of one signal and the output samples
// [t0*hop, t1*hop) of the padded signal.  It (re)computes the K = ceil(N/hop)-1 frames before
// the tile as a halo so that the overlap-add of its output range needs no other CTA: no
// atomics, deterministic, and the whole iteration
//     frame+window -> real FFT -> point-wise update/projection -> inverse real FFT
//     -> windowed overlap-add -> 1/envelope
// stays in shared memory.  The real FFT of length N is an N/2-point complex FFT done in place:
// forward decimation-in-frequency (natural -> bit-reversed), the point-wise stage works directly
// on bit-reversed positions, inverse decimation-in-time (bit-reversed -> natural), so no
// reordering pass is ever needed.  Two radix-2 stages are fused per pass (radix-2^2).
//
// Replaces, per iteration, torch.stft + ~8 point-wise kernels + fft.irfft + conv_transpose1d with
// a dense diag(window) weight of the reference (methods.py:241-248, :464-477, :127-132).
#include <cstdlib>

#include "specinv_common.cuh"
#include "generic_tile.cuh"
#include "generic_fft.cuh"

namespace specinv {

template <typename T, int OP>
__global__ void __launch_bounds__(1024) tile_kernel(const TileArgs a) {
    using C = cx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* wb = reinterpret_cast<C*>(smem_raw);

    const Dims& dm = a.dm;
    const int M = dm.M, N = dm.N, hop = dm.hop, Mp = a.Mp;
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * a.tile_frames;
    const int t1 = min(dm.T, t0 + a.tile_frames);
    const int f0 = (OP == OP_STFT) ? t0 : max(0, t0 - dm.K);
    const int nfr = t1 - f0;
    const int tid = threadIdx.x, NT = blockDim.x;

    const C* tw = (const C*)a.tw;
    const C* twr = (const C*)a.twr;
    const T* wa = (const T*)a.wa;
    const T* ws = (const T*)a.ws;

    // ---- A: frame + analysis window: z[n] = x[2n] w[2n] + i x[2n+1] w[2n+1] ---------------
    if constexpr (OP != OP_ISTFT) {
        const T* x = (const T*)a.x_in + (long long)b * dm.L;
        for (int idx = tid; idx < nfr * M; idx += NT) {
            const int f = idx / M, n = idx - f * M;
            const long long pp = (long long)(f0 + f) * hop + 2 * n;
            const long long i0 = pad_index(pp, dm.P, dm.L, dm.pad_mode);
            const long long i1 = pad_index(pp + 1, dm.P, dm.L, dm.pad_mode);
            const T v0 = i0 >= 0 ? x[i0] : T(0);
            const T v1 = i1 >= 0 ? x[i1] : T(0);
            wb[f * Mp + padidx(n)] = mk<T>(v0 * wa[2 * n], v1 * wa[2 * n + 1]);
        }
        __syncthreads();

        // ---- B: forward DIF passes (natural -> bit-reversed) ------------------------------------
        fft_forward_inplace<T>(wb, nfr, M, Mp, tw);
    }

    // ---- C: real-FFT post-process, point-wise update, inverse pre-process (pairs k, M-k) ----
    T dsum = T(0), esum = T(0);
    const bool want_sums = a.sums != nullptr;
    {
        const int npair = M / 2 + 1;
        const int sh = 32 - dm.logM;
        for (int idx = tid; idx < nfr * npair; idx += NT) {
            const int f = idx / npair, k = idx - f * npair;
            const int t = f0 + f;
            const bool owned = t >= t0;
            C* v = wb + f * Mp;
            const int kA = k, kB = M - k;
            const int pA = padidx((int)(__brev((unsigned)kA) >> sh));
            const int pB = padidx((int)(__brev((unsigned)(kB & (M - 1))) >> sh));
            const C w = twr[k];
            C sA = mk<T>(T(0), T(0)), sB = sA;
            if constexpr (OP != OP_ISTFT) {
                rfft_post_pair<T>(v[pA], v[pB], w, sA, sB);
            }
            const BinIO<T> io(a, (long long)b * dm.T + t);
            C hA, hB;
            if (dm.onesided) {
                hA = bin_update<T, OP>(a, io, kA, sA, owned, want_sums, dsum, esum);
                hB = (kB != kA) ? bin_update<T, OP>(a, io, kB, sB, owned, want_sums, dsum, esum) : hA;
            } else {
                // two-sided: bins kA, kB and their mirrors N-kA, N-kB (= conj of the real-input STFT);
                // ifft(...).real (methods.py:145-146) == irfft of the Hermitian part (p[k]+conj p[N-k])/2
                hA = bin_update<T, OP>(a, io, kA, sA, owned, want_sums, dsum, esum);
                if (kA != 0) {
                    C m = bin_update<T, OP>(a, io, N - kA, mk<T>(sA.x, -sA.y), owned, want_sums, dsum, esum);
                    hA = mk<T>(T(0.5) * (hA.x + m.x), T(0.5) * (hA.y - m.y));
                }
                if (kB != kA) {
                    hB = bin_update<T, OP>(a, io, kB, sB, owned, want_sums, dsum, esum);
                    if (kB != M) {
                        C m = bin_update<T, OP>(a, io, N - kB, mk<T>(sB.x, -sB.y), owned, want_sums, dsum, esum);
                        hB = mk<T>(T(0.5) * (hB.x + m.x), T(0.5) * (hB.y - m.y));
                    }
                } else {
                    hB = hA;
                }
            }
            if constexpr (OP != OP_STFT) {
                if (k == 0) { hA.y = T(0); hB.y = T(0); }  // C2R ignores Im(DC), Im(Nyquist)
                C zA, zB;
                irfft_pre_pair<T>(hA, hB, w, zA, zB);
                v[pA] = zA;
                if (kB != kA && k != 0) v[pB] = zB;
            }
        }
    }

    if constexpr (OP == OP_GL || OP == OP_GLR || OP == OP_ADMM) {
        if (want_sums) {   // fused metric epilogue: block reduce, one double atomic pair per CTA
            __shared__ double red[2][32];
            double d = (double)dsum, e = (double)esum;
            for (int o = 16; o > 0; o >>= 1) {
                d += __shfl_xor_sync(0xffffffffu, d, o);
                e += __shfl_xor_sync(0xffffffffu, e, o);
            }
            if ((tid & 31) == 0) { red[0][tid >> 5] = d; red[1][tid >> 5] = e; }
            __syncthreads();
            if (tid == 0) {
                double dd = 0, ee = 0;
                for (int i = 0; i < (NT >> 5); ++i) { dd += red[0][i]; ee += red[1][i]; }
                atomicAdd(a.sums, dd);
                atomicAdd(a.sums + 1, ee);
            }
        }
    }
    if constexpr (OP == OP_STFT) return;
    __syncthreads();

    // ---- D: inverse DIT passes (bit-reversed -> natural), conj twiddles ------------------------
    fft_inverse_inplace<T>(wb, nfr, M, dm.logM, Mp, tw);

    // ---- E: windowed overlap-add of the owned output range (gather), times 1/envelope --------
    {
        const long long o0 = (long long)t0 * hop;
        const long long o1 = (t1 == dm.T) ? dm.Lp : (long long)t1 * hop;
        T* xo = (T*)a.x_out + (long long)b * dm.L;
        const T* ienv = (const T*)a.inv_env;
        const T* wbf = reinterpret_cast<const T*>(wb);
        for (long long pp = o0 + tid; pp < o1; pp += NT) {
            const long long m = pp - dm.P;
            if (m < 0 || m >= dm.L) continue;
            int tlo = pp >= N ? (int)((pp - N) / hop) + 1 : 0;
            if (tlo < f0) tlo = f0;
            int thi = (int)(pp / hop);
            if (thi > t1 - 1) thi = t1 - 1;
            T acc = T(0);
            for (int t = tlo; t <= thi; ++t) {
                const int i = (int)(pp - (long long)t * hop);
                acc += wbf[2 * ((t - f0) * Mp + padidx(i >> 1)) + (i & 1)] * ws[i];
            }
            xo[m] = acc * ienv[m];
        }
    }
}

// ------------------------------------------------------------------------------------------
// Any n_fft the mixed-radix kernels (specinv_generic_mr.cu) do not take -- a half with a prime factor > 13, or an ODD
// n_fft (two-sided spectra only: the reference infers n_fft = bin count, methods.py:65-68) --: the same tile structure
// with the transforms done as direct DFTs on the W_N table of the plan.  O(N^2) per frame instead of O(N log N) -- a coverage path (about 4x the generic FFT kernel's time at
// N = 400), never a fallback to another library.  Shared memory per frame: N time samples and N/2+1 bins.
//   forward : s[k] = sum_n fr[n] W_N^(kn), k <= N/2               (fr = frame * analysis window)
//   inverse : x[n] = Re h[0] + (-1)^n Re h[N/2] + 2 sum_{0<k<N/2} Re(h[k] conj(W_N^(kn)))   (C2R, unnormalised:
//             the synthesis window carries 1/N or N^-1/2 like in the FFT kernels)
// ------------------------------------------------------------------------------------------
template <typename T, int OP>
__global__ void __launch_bounds__(512) dft_tile_kernel(const TileArgs a) {
    using C = cx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Dims& dm = a.dm;
    const int N = dm.N, H = dm.M + 1, hop = dm.hop;
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * a.tile_frames;
    const int t1 = min(dm.T, t0 + a.tile_frames);
    const int f0 = (OP == OP_STFT) ? t0 : max(0, t0 - dm.K);
    const int nfr = t1 - f0;
    const int tid = threadIdx.x, NT = blockDim.x;
    C* hb = reinterpret_cast<C*>(smem_raw);                          // [frames][H] half spectra
    T* fb = reinterpret_cast<T*>(hb + (size_t)(a.tile_frames + dm.K) * H);   // [frames][N] time frames
    const C* __restrict__ tw = (const C*)a.tw;                       // W_N^j = (cos, -sin)(2 pi j / N)
    const T* wa = (const T*)a.wa;
    const T* ws = (const T*)a.ws;

    T dsum = T(0), esum = T(0);
    const bool want_sums = a.sums != nullptr;
    if constexpr (OP != OP_ISTFT) {
        const T* x = (const T*)a.x_in + (long long)b * dm.L;
        for (int idx = tid; idx < nfr * N; idx += NT) {
            const int f = idx / N, n = idx - f * N;
            const long long i0 = pad_index((long long)(f0 + f) * hop + n, dm.P, dm.L, dm.pad_mode);
            fb[idx] = (i0 >= 0 ? x[i0] : T(0)) * wa[n];
        }
        __syncthreads();
    }
    // ---- forward DFT of every half-spectrum bin + point-wise stage
    for (int idx = tid; idx < nfr * H; idx += NT) {
        const int f = idx / H, k = idx - f * H;
        const int t = f0 + f;
        const bool owned = t >= t0;
        C s = mk<T>(T(0), T(0));
        if constexpr (OP != OP_ISTFT) {
            const T* fr = fb + (size_t)f * N;
            T sr = T(0), si = T(0);
            int j = 0;                                               // (k n) mod N
            for (int n = 0; n < N; ++n) {
                const C w = tw[j];
                sr += fr[n] * w.x; si += fr[n] * w.y;
                j += k; if (j >= N) j -= N;
            }
            s = mk<T>(sr, si);
        }
        const BinIO<T> io(a, (long long)b * dm.T + t);
        C h = bin_update<T, OP>(a, io, k, s, owned, want_sums, dsum, esum);
        if (!dm.onesided && k != 0 && (k != dm.M || (N & 1))) {
            // two-sided: the mirrored bin N-k holds conj(s) of the real-input STFT; ifft(...).real (methods.py:145-146)
            // is the C2R transform of the Hermitian part (p[k] + conj p[N-k]) / 2  (odd N: no Nyquist bin, k = M = (N-1)/2
            // has a mirror like every other bin)
            const C m = bin_update<T, OP>(a, io, N - k, mk<T>(s.x, -s.y), owned, want_sums, dsum, esum);
            h = mk<T>(T(0.5) * (h.x + m.x), T(0.5) * (h.y - m.y));
        }
        hb[idx] = h;
    }
    if constexpr (OP == OP_GL || OP == OP_GLR || OP == OP_ADMM) {
        if (want_sums) {
            __shared__ double red[2][32];
            double d = (double)dsum, e = (double)esum;
            for (int o = 16; o > 0; o >>= 1) {
                d += __shfl_xor_sync(0xffffffffu, d, o);
                e += __shfl_xor_sync(0xffffffffu, e, o);
            }
            if ((tid & 31) == 0) { red[0][tid >> 5] = d; red[1][tid >> 5] = e; }
            __syncthreads();
            if (tid == 0) {
                double dd = 0, ee = 0;
                for (int i = 0; i < (NT >> 5); ++i) { dd += red[0][i]; ee += red[1][i]; }
                atomicAdd(a.sums, dd);
                atomicAdd(a.sums + 1, ee);
            }
        }
    }
    if constexpr (OP == OP_STFT) return;
    __syncthreads();
    // ---- inverse (C2R) DFT of every sample
    for (int idx = tid; idx < nfr * N; idx += NT) {
        const int f = idx / N, n = idx - f * N;
        const C* h = hb + (size_t)f * H;
        const bool oddN = N & 1;
        T acc = oddN ? h[0].x : h[0].x + ((n & 1) ? -h[dm.M].x : h[dm.M].x);
        T part = T(0);
        int j = n;                                                   // (k n) mod N for k = 1
        const int kend = oddN ? dm.M + 1 : dm.M;
        for (int k = 1; k < kend; ++k) {
            const C w = tw[j];
            part += h[k].x * w.x + h[k].y * w.y;                     // Re(h conj(W))
            j += n; if (j >= N) j -= N;
        }
        fb[idx] = acc + T(2) * part;
    }
    __syncthreads();
    // ---- windowed overlap-add of the owned output range (gather), times 1/envelope
    {
        const long long o0 = (long long)t0 * hop;
        const long long o1 = (t1 == dm.T) ? dm.Lp : (long long)t1 * hop;
        T* xo = (T*)a.x_out + (long long)b * dm.L;
        const T* ienv = (const T*)a.inv_env;
        for (long long pp = o0 + tid; pp < o1; pp += NT) {
            const long long m = pp - dm.P;
            if (m < 0 || m >= dm.L) continue;
            int tlo = pp >= N ? (int)((pp - N) / hop) + 1 : 0;
            if (tlo < f0) tlo = f0;
            int thi = (int)(pp / hop);
            if (thi > t1 - 1) thi = t1 - 1;
            T acc = T(0);
            for (int t = tlo; t <= thi; ++t) {
                const int i = (int)(pp - (long long)t * hop);
                acc += fb[(size_t)(t - f0) * N + i] * ws[i];
            }
            xo[m] = acc * ienv[m];
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int g_smem_optin = -1;

static int smem_optin() {
    if (g_smem_optin < 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 0;
        g_smem_optin = v;
    }
    return g_smem_optin;
}

template <typename T, int OP>
static int launch_dft_tile(TileArgs& a, cudaStream_t st) {
    const Dims& dm = a.dm;
    const size_t frame_bytes = ((size_t)dm.N + 2 * (size_t)(dm.M + 1)) * sizeof(T);
    const int halo = (OP == OP_STFT) ? 0 : dm.K;
    const int optin = smem_optin();
    if (optin <= 0) return SPECINV_ERR_NO_DEVICE;
    const size_t big = (size_t)optin - 1024;
    const size_t budget = big < (size_t)100 * 1024 ? big : (size_t)100 * 1024;
    int cap = (int)(budget / frame_bytes);
    if (cap - halo < (halo > 1 ? 2 * halo : 2)) cap = (int)(big / frame_bytes);
    int owned = cap - halo;
    if (owned < 1) return SPECINV_ERR_UNSUPPORTED;
    if (owned > dm.T) owned = dm.T;
    while (owned > 4 * (halo > 0 ? halo : 1) && (long long)dm.B * ((dm.T + owned - 1) / owned) < 2 * 148) owned = (owned + 1) / 2;
    a.tile_frames = owned;
    // (the kernel places the time frames behind tile_frames + K half spectra whatever the op)
    const size_t smem = (size_t)(owned + dm.K) * frame_bytes;
    if (smem > big) return SPECINV_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(dft_tile_kernel<T, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((dm.T + owned - 1) / owned, dm.B);
    if (grid.y > 65535) return SPECINV_ERR_UNSUPPORTED;
    dft_tile_kernel<T, OP><<<grid, 512, smem, st>>>(a);
    return (int)cudaGetLastError();
}

template <typename T, int OP>
static int launch_tile(TileArgs& a, cudaStream_t st) {
    const Dims& dm = a.dm;
    // the mixed-radix team kernel (specinv_generic_mr.cu) serves every size whose half factors into 2 .. 13;
    // SPECINV_GENERIC_MR=0 keeps the radix-2^2 CTA-wide kernel / the direct DFT (A/B timing, tests of those kernels)
    // (read per launch, like SPECINV_FORCE_GENERIC: tests switch it inside one process)
    const char* mr_env = getenv("SPECINV_GENERIC_MR");
    if (!(mr_env && mr_env[0] == '0')) {
        const int rc = mr_tile_launch(sizeof(T) == 8 ? SPECINV_F64 : SPECINV_F32, OP, a, st);
        if (rc != SPECINV_ERR_UNSUPPORTED) return rc;
    }
    if (!dm.pow2) return launch_dft_tile<T, OP>(a, st);
    const int Mp = dm.M + (dm.M >> 4);
    const size_t frame_bytes = (size_t)Mp * 2 * sizeof(T);
    const int halo = (OP == OP_STFT) ? 0 : dm.K;
    const int optin = smem_optin();
    if (optin <= 0) return SPECINV_ERR_NO_DEVICE;
    const size_t big = (size_t)optin - 1024;        // static smem of the reduction + slack
    size_t budget = big < (size_t)100 * 1024 ? big : (size_t)100 * 1024;   // 2 CTAs / SM when possible
    int cap = (int)(budget / frame_bytes);
    if (cap - halo < (halo > 1 ? 2 * halo : 2)) cap = (int)(big / frame_bytes);  // poor owned/halo ratio: one fat CTA
    int owned = cap - halo;
    if (owned < 1) return SPECINV_ERR_UNSUPPORTED;  // hop too small for this n_fft: halo does not fit
    if (owned > dm.T) owned = dm.T;
    // small problems: prefer enough tiles to cover the 148 SMs
    while (owned > 4 * (halo > 0 ? halo : 1) && (long long)dm.B * ((dm.T + owned - 1) / owned) < 2 * 148) owned = (owned + 1) / 2;
    a.tile_frames = owned;
    a.Mp = Mp;
    const size_t smem = (size_t)(owned + halo) * frame_bytes;
    cudaError_t e = cudaFuncSetAttribute(tile_kernel<T, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((dm.T + owned - 1) / owned, dm.B);
    if (grid.y > 65535) return SPECINV_ERR_UNSUPPORTED;
    // threads per CTA: enough to give every thread a few butterflies per pass
    const long long bf = (long long)(owned + halo) * (dm.M >> 2);     // radix-4 butterflies per pass
    const int threads = bf >= 4096 ? 1024 : bf >= 1024 ? 512 : 256;
    tile_kernel<T, OP><<<grid, threads, smem, st>>>(a);
    return (int)cudaGetLastError();
}

static void fill_plan(TileArgs& a, const Dims& dm, int dtype, const void* plan) {
    const PlanLayout pl = plan_layout(dm, dtype);
    const char* p = (const char*)plan;
    a.tw = p + pl.tw; a.twr = p + pl.twr; a.wa = p + pl.wa; a.ws = p + pl.ws; a.inv_env = p + pl.inv_env;
    a.dm = dm;
}

template <int OP>
static int dispatch(int dtype, TileArgs& a, cudaStream_t st) {
    return dtype == SPECINV_F64 ? launch_tile<double, OP>(a, st) : launch_tile<float, OP>(a, st);
}

int generic_stft(const specinv_desc* d, const void* plan, const void* x, void* main_out, void* nyq_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !x || !main_out || (dm.onesided && !nyq_out)) return SPECINV_ERR_INVALID;
    TileArgs a{}; fill_plan(a, dm, d->dtype, plan);
    a.x_in = x; a.s0_out_main = main_out; a.s0_out_nyq = nyq_out;
    return dispatch<OP_STFT>(d->dtype, a, (cudaStream_t)stream);
}

int generic_istft(const specinv_desc* d, const void* plan, const void* main_in, const void* nyq_in, void* x_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !x_out || !main_in || (dm.onesided && !nyq_in)) return SPECINV_ERR_INVALID;
    TileArgs a{}; fill_plan(a, dm, d->dtype, plan);
    a.x_out = x_out; a.s0_in_main = main_in; a.s0_in_nyq = nyq_in;
    return dispatch<OP_ISTFT>(d->dtype, a, (cudaStream_t)stream);
}

// rebuilt = false: specinv_gl_iter (OP_GL); true: specinv_gl_rebuilt_iter (OP_GLR, the state is the rebuilt spectrum)
static int generic_momentum_iter(bool rebuilt, const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                                 const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                                 const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !x_in || !x_out || !mag_main || x_in == x_out) return SPECINV_ERR_INVALID;
    if (!q_in_main != !q_out_main || (!q_in_main && lr != 0.0)) return SPECINV_ERR_INVALID;
    if (q_in_main && q_in_main == q_out_main) return SPECINV_ERR_INVALID;
    if (dm.onesided && (!mag_nyq || (q_in_main && (!q_in_nyq || !q_out_nyq)))) return SPECINV_ERR_INVALID;
    TileArgs a{}; fill_plan(a, dm, d->dtype, plan);
    a.x_in = x_in; a.x_out = x_out;
    a.s0_in_main = q_in_main; a.s0_in_nyq = q_in_nyq; a.s0_out_main = q_out_main; a.s0_out_nyq = q_out_nyq;
    a.mag_main = mag_main; a.mag_nyq = mag_nyq; a.coef = lr; a.sums = sums;
    // without state both ops are plain Griffin-Lim: one kernel serves them
    if (rebuilt && q_in_main) return dispatch<OP_GLR>(d->dtype, a, (cudaStream_t)stream);
    return dispatch<OP_GL>(d->dtype, a, (cudaStream_t)stream);
}

int generic_gl_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                    const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                    const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream) {
    return generic_momentum_iter(false, d, plan, x_in, x_out, q_in_main, q_in_nyq, q_out_main, q_out_nyq, mag_main,
                                 mag_nyq, lr, sums, stream);
}

int generic_gl_rebuilt_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                            const void* s_in_main, const void* s_in_nyq, void* s_out_main, void* s_out_nyq,
                            const void* mag_main, const void* mag_nyq, double m, double* sums, void* stream) {
    return generic_momentum_iter(true, d, plan, x_in, x_out, s_in_main, s_in_nyq, s_out_main, s_out_nyq, mag_main,
                                 mag_nyq, m, sums, stream);
}

int generic_admm_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                      const void* X_in_main, const void* X_in_nyq, const void* U_in_main, const void* U_in_nyq,
                      void* X_out_main, void* X_out_nyq, void* U_out_main, void* U_out_nyq,
                      const void* mag_main, const void* mag_nyq, double rho, double* sums, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !x_in || !x_out || !X_in_main || !U_in_main || !X_out_main || !U_out_main || !mag_main) return SPECINV_ERR_INVALID;
    if (dm.onesided && (!X_in_nyq || !U_in_nyq || !X_out_nyq || !U_out_nyq || !mag_nyq)) return SPECINV_ERR_INVALID;
    if (x_in == x_out || X_in_main == X_out_main || U_in_main == U_out_main) return SPECINV_ERR_INVALID;
    TileArgs a{}; fill_plan(a, dm, d->dtype, plan);
    a.x_in = x_in; a.x_out = x_out;
    a.s0_in_main = X_in_main; a.s0_in_nyq = X_in_nyq; a.s0_out_main = X_out_main; a.s0_out_nyq = X_out_nyq;
    a.s1_in_main = U_in_main; a.s1_in_nyq = U_in_nyq; a.s1_out_main = U_out_main; a.s1_out_nyq = U_out_nyq;
    a.mag_main = mag_main; a.mag_nyq = mag_nyq; a.coef = rho; a.sums = sums;
    return dispatch<OP_ADMM>(d->dtype, a, (cudaStream_t)stream);
}

}  // namespace specinv
