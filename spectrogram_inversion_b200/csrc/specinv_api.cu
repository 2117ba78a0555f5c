// extern "C" entry points of libspecinv_b200.so (see include/specinv_b200.h), the plan
// initialisation kernels, layout conversion and the standalone metric reduction.
#include <atomic>
#include <cstdlib>

#include "specinv_common.cuh"

namespace specinv {

// ---------------------------------------------------------------- PDL guard (see specinv_common.cuh)
static const uintptr_t kNoStream = ~(uintptr_t)0;
static std::atomic<uintptr_t> g_tables_last_on{kNoStream};   // stream whose latest library launch wrote plan tables
void note_tables_launch(cudaStream_t st) { g_tables_last_on.store((uintptr_t)st, std::memory_order_release); }
void note_other_launch(cudaStream_t st) {
    uintptr_t expect = (uintptr_t)st;                        // only the same stream's mark is cleared
    g_tables_last_on.compare_exchange_strong(expect, kNoStream, std::memory_order_acq_rel);
}
bool pdl_prologue_safe(cudaStream_t st) {
    uintptr_t expect = (uintptr_t)st;
    return !g_tables_last_on.compare_exchange_strong(expect, kNoStream, std::memory_order_acq_rel);
}

// implemented in specinv_generic.cu
int generic_stft(const specinv_desc*, const void*, const void*, void*, void*, void*);
int generic_istft(const specinv_desc*, const void*, const void*, const void*, void*, void*);
int generic_gl_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, void*, void*,
                    const void*, const void*, double, double*, void*);
int generic_gl_rebuilt_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, void*, void*,
                            const void*, const void*, double, double*, void*);
int generic_admm_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, const void*,
                      const void*, void*, void*, void*, void*, const void*, const void*, double, double*, void*);
// implemented in specinv_fastw.cu (the specialised kernels); return SPECINV_ERR_UNSUPPORTED when not applicable

int fastw_gl_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, void*, void*,
                  const void*, const void*, double, double*, void*);
int fastw_gl_rebuilt_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, void*, void*,
                          const void*, const void*, double, double*, void*);
int fastw_admm_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, const void*,
                    const void*, void*, void*, void*, void*, const void*, const void*, double, double*, void*);
int fastw_istft(const specinv_desc*, const void*, const void*, const void*, void*, void*);
int fastw_gl_plain_iter(const specinv_desc*, const void*, const void*, void*, const void*, const void*, double*, void*);

// SPECINV_FORCE_GENERIC=1 routes everything through the generic tile kernels (testing / A-B timing)
static bool force_generic() {
    const char* e = getenv("SPECINV_FORCE_GENERIC");
    return e && e[0] == '1';
}

// ---------------------------------------------------------------- plan
template <typename T>
__global__ void plan_tables_kernel(int N, int M, int pow2, int normalized, const T* __restrict__ window,
                                   cx_t<T>* tw, cx_t<T>* twr, T* wa, T* ws) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (pow2 ? i < M : i < N) {
        double s, c;
        sincospi(2.0 * i / (pow2 ? M : N), &s, &c);
        tw[i] = mk<T>((T)c, (T)(-s));
    }
    if (i <= M / 2) {
        double s, c;
        sincospi(2.0 * i / N, &s, &c);
        twr[i] = mk<T>((T)c, (T)(-s));
    }
    if (i < N) {
        // forward: 1 (or N^-1/2 when normalized); inverse: 1/N (or N^-1/2), methods.py:143
        const double fs = normalized ? rsqrt((double)N) : 1.0;
        const double is = normalized ? rsqrt((double)N) : 1.0 / N;
        wa[i] = (T)((double)window[i] * fs);
        ws[i] = (T)((double)window[i] * is);
    }
}

// env[m] = sum_t w^2[m + P - t*hop]  (methods.py:129-131), inv_env = 1/env without epsilon.
// frame_offset / total_frames: the plan describes frames [frame_offset, frame_offset + T) of a longer signal
// with total_frames frames (frame-range sharding); the envelope then also counts the neighbours' frames.
template <typename T>
__global__ void plan_envelope_kernel(Dims dm, long long frame_offset, long long total_frames,
                                     const T* __restrict__ window, T* env, T* inv_env) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= dm.L) return;
    const long long pp = m + dm.P + frame_offset * dm.hop;
    long long tlo = pp >= dm.N ? (pp - dm.N) / dm.hop + 1 : 0;
    long long thi = pp / dm.hop;
    if (thi > total_frames - 1) thi = total_frames - 1;
    T acc = T(0);
    for (long long t = tlo; t <= thi; ++t) {
        const T w = window[pp - t * dm.hop];
        acc += w * w;
    }
    env[m] = acc;
    inv_env[m] = T(1) / acc;
}

// 1/envelope of samples [x0, x0 + len) of a signal of `total` frames (total < 0: not known yet, only samples whose
// covering frames have all been seen are asked for), read from a plan of T0 = dm.T frames.  The envelope kernel above
// sums w^2 over the covering frames in ascending order, so a sample's value depends only on (m + P) mod hop and on
// whether its frame range is clipped by the first or by the last frame: the head of the signal is the plan's head,
// the tail (total >= T0) the plan's tail, and every interior sample equals the plan's interior sample at the same
// phase.  T0 must satisfy (T0 - 1) * hop >= n_fft unless total == T0.
template <typename T>
__global__ void inv_env_window_kernel(Dims dm, const T* __restrict__ inv_env, long long x0, long long len,
                                      long long total, T* __restrict__ out) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= len) return;
    const long long pp = x0 + j + dm.P;                       // position in the padded signal
    long long q;
    if (total == dm.T) q = pp;
    else if (total >= 0 && pp >= total * dm.hop) q = pp - (total - dm.T) * dm.hop;   // clipped by the last frame
    else if (pp < dm.N) q = pp;                                                       // clipped by the first frame
    else q = dm.N + (pp - dm.N) % dm.hop;                                             // interior
    out[j] = inv_env[q - dm.P];
}

template <typename T>
static int plan_init_t(const Dims& dm, const specinv_desc* d, const void* window, void* plan, long long frame_offset,
                       long long total_frames, cudaStream_t st) {
    const PlanLayout pl = plan_layout(dm, d->dtype);
    char* p = (char*)plan;
    const int n = dm.N;
    plan_tables_kernel<T><<<(n + 255) / 256, 256, 0, st>>>(dm.N, dm.M, dm.pow2, d->normalized, (const T*)window,
                                                           (cx_t<T>*)(p + pl.tw), (cx_t<T>*)(p + pl.twr),
                                                           (T*)(p + pl.wa), (T*)(p + pl.ws));
    note_tables_launch(st);       // an iteration kernel launched right behind this one must not overlap it
    plan_envelope_kernel<T><<<(unsigned)((dm.L + 255) / 256), 256, 0, st>>>(dm, frame_offset, total_frames,
                                                                            (const T*)window, (T*)(p + pl.env),
                                                                            (T*)(p + pl.inv_env));
    note_other_launch(st);        // the envelope kernel does not touch the tables: overlap behind it is safe
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- layout conversion
// 32x32 tile transpose between the reference's (batch, freq, time) tensor (arbitrary element
// strides) and the split frame-major layout.  TO_INTERNAL: coalesced along the smaller of the two
// source strides when reading, along freq when writing.
template <typename V, bool TO_INTERNAL>
__global__ void convert_kernel(Dims dm, int F, V* main, V* nyq, V* ext, long long sb, long long sf, long long st) {
    __shared__ V tile[32][33];
    const int b = blockIdx.z;
    const int fbase = blockIdx.x * 32, tbase = blockIdx.y * 32;
    const bool time_fast = st <= sf;   // which external index should follow threadIdx.x
    auto internal = [&](int f, int t) -> V* {
        const long long fr = (long long)b * dm.T + t;
        if (dm.onesided && f == dm.M) return nyq + fr;
        return main + fr * dm.row + f;
    };
    if (TO_INTERNAL) {
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int f = time_fast ? fbase + j : fbase + threadIdx.x;
            const int t = time_fast ? tbase + threadIdx.x : tbase + j;
            if (f < F && t < dm.T) {
                const V v = ext[b * sb + f * sf + t * st];
                if (time_fast) tile[j][threadIdx.x] = v; else tile[threadIdx.x][j] = v;
            }
        }
        __syncthreads();
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int f = fbase + threadIdx.x, t = tbase + j;
            if (f < F && t < dm.T) *internal(f, t) = tile[threadIdx.x][j];
        }
    } else {
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int f = fbase + threadIdx.x, t = tbase + j;
            if (f < F && t < dm.T) tile[threadIdx.x][j] = *internal(f, t);
        }
        __syncthreads();
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int f = time_fast ? fbase + j : fbase + threadIdx.x;
            const int t = time_fast ? tbase + threadIdx.x : tbase + j;
            if (f < F && t < dm.T) ext[b * sb + f * sf + t * st] = time_fast ? tile[j][threadIdx.x] : tile[threadIdx.x][j];
        }
    }
}

// The external tensor is frame-major itself (frequency stride 1: what torch.stft returns and what `abs()` of it keeps):
// no transpose, every (signal, frame) row of F bins is one contiguous run on both sides -- a warp copies a row with
// coalesced accesses (main <- the first `row` bins, nyq <- the last one when onesided).
template <typename V, bool TO_INTERNAL>
__global__ void __launch_bounds__(256) rowcopy_kernel(Dims dm, int F, V* __restrict__ main, V* __restrict__ nyq,
                                                      V* __restrict__ ext, long long sb, long long st) {
    const int lane = threadIdx.x & 31;
    const long long rows = (long long)dm.B * dm.T;
    const long long wstride = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += wstride) {
        const long long b = r / dm.T, t = r - b * dm.T;
        V* e = ext + b * sb + t * st;
        V* m = main + r * dm.row;
#pragma unroll 4
        for (int k = lane; k < dm.row; k += 32) {
            if (TO_INTERNAL) m[k] = e[k]; else e[k] = m[k];
        }
        if (dm.onesided && lane == 0) {
            if (TO_INTERNAL) nyq[r] = e[dm.M]; else e[dm.M] = nyq[r];
        }
    }
}

template <typename V, bool TO_INTERNAL>
static int convert(const Dims& dm, V* main, V* nyq, V* ext, long long sb, long long sf, long long st, cudaStream_t s) {
    const int F = dm.onesided ? dm.M + 1 : dm.N;
    if (sf == 1) {
        const long long rows = (long long)dm.B * dm.T;
        long long blocks = (rows + 7) / 8;                       // 8 warps per block, one row per warp and trip
        if (blocks > 148 * 32) blocks = 148 * 32;
        rowcopy_kernel<V, TO_INTERNAL><<<(unsigned)blocks, 256, 0, s>>>(dm, F, main, nyq, ext, sb, st);
        return (int)cudaGetLastError();
    }
    dim3 grid((F + 31) / 32, (dm.T + 31) / 32, dm.B), block(32, 8);
    if (grid.y > 65535 || grid.z > 65535) return SPECINV_ERR_UNSUPPORTED;
    convert_kernel<V, TO_INTERNAL><<<grid, block, 0, s>>>(dm, F, main, nyq, ext, sb, sf, st);
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- metric sums
template <typename T>
__global__ void metric_sums_kernel(const T* __restrict__ a, const T* __restrict__ b, long long n, double* out3) {
    double d = 0, e = 0, g = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double x = (double)a[i], y = (double)b[i];
        d += (x - y) * (x - y); e += x * x; g += y * y;
    }
    __shared__ double red[3][8];
    for (int o = 16; o > 0; o >>= 1) {
        d += __shfl_xor_sync(0xffffffffu, d, o);
        e += __shfl_xor_sync(0xffffffffu, e, o);
        g += __shfl_xor_sync(0xffffffffu, g, o);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = d; red[1][threadIdx.x >> 5] = e; red[2][threadIdx.x >> 5] = g; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[threadIdx.x][i];
        atomicAdd(out3 + threadIdx.x, s);
    }
}

// ---------------------------------------------------------------- frame-range sharding helpers
// out[b][i] = left[b][i] + right[b][i] on a (rows x n) strided view: both neighbours add the two partial
// overlap-add sums of the shared (n_fft - hop)-sample region in the SAME order, so they hold bit-identical values.
template <typename T>
__global__ void halo_sum_kernel(const T* __restrict__ left, long long ld_left, const T* __restrict__ right,
                                long long ld_right, T* out, long long ld_out, int rows, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (i < n && b < rows) out[b * ld_out + i] = left[b * ld_left + i] + right[b * ld_right + i];
}

// Re-create the centre padding of the global signal inside a rank-local padded buffer (the reference
// re-pads x at every torch.stft call, methods.py:241).  x holds padded samples [off, off + len) of every row.
template <typename T>
__global__ void fill_padding_kernel(T* x, long long ld, int rows, long long off, long long len, int P, long long L,
                                    int pad_mode) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // 0 .. 2P-1: left pad then right pad
    const int b = blockIdx.y;
    if (j >= 2LL * P || b >= rows) return;
    const long long pp = j < P ? j : P + L + (j - P);        // global padded index of a padding sample
    if (pp < off || pp >= off + len) return;
    const long long src = pad_index(pp, P, L, pad_mode);     // index into the unpadded global signal, or -1
    T v = T(0);
    if (src >= 0) {
        const long long sl = src + P - off;                   // local position of the source sample
        if (sl < 0 || sl >= len) return;                      // source lives on another rank (circular): caller forbids
        v = x[b * ld + sl];
    }
    x[b * ld + (pp - off)] = v;
}

}  // namespace specinv

namespace specinv {
template <typename T>
__global__ void fill_ones_kernel(T* a, T* b, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { a[i] = T(1); b[i] = T(1); }
}

}  // namespace specinv

using namespace specinv;

extern "C" {

int specinv_abi_version(void) { return SPECINV_ABI_VERSION; }

const char* specinv_error_string(int code) {
    switch (code) {
        case SPECINV_OK: return "ok";
        case SPECINV_ERR_INVALID: return "invalid argument";
        case SPECINV_ERR_UNSUPPORTED: return "configuration not supported by the sm_100a kernels";
        case SPECINV_ERR_NO_DEVICE: return "no usable CUDA device";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int specinv_signal_length(const specinv_desc* d, int64_t* length) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!length) return SPECINV_ERR_INVALID;
    *length = dm.L;
    return SPECINV_OK;
}

int specinv_plan_bytes(const specinv_desc* d, size_t* bytes) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!bytes) return SPECINV_ERR_INVALID;
    *bytes = plan_layout(dm, d->dtype).total;
    return SPECINV_OK;
}

int specinv_plan_init(const specinv_desc* d, const void* window, void* plan, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!window || !plan) return SPECINV_ERR_INVALID;
    return d->dtype == SPECINV_F64 ? plan_init_t<double>(dm, d, window, plan, 0, dm.T, (cudaStream_t)stream)
                                   : plan_init_t<float>(dm, d, window, plan, 0, dm.T, (cudaStream_t)stream);
}

int specinv_plan_init_ranged(const specinv_desc* d, const void* window, void* plan, int64_t frame_offset,
                             int64_t total_frames, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!window || !plan || d->center) return SPECINV_ERR_INVALID;   // a frame range is described un-centred
    if (frame_offset < 0 || frame_offset + dm.T > total_frames) return SPECINV_ERR_INVALID;
    return d->dtype == SPECINV_F64
               ? plan_init_t<double>(dm, d, window, plan, frame_offset, total_frames, (cudaStream_t)stream)
               : plan_init_t<float>(dm, d, window, plan, frame_offset, total_frames, (cudaStream_t)stream);
}

int specinv_plan_envelope(const specinv_desc* d, const void* plan, void* env_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || !env_out) return SPECINV_ERR_INVALID;
    const PlanLayout pl = plan_layout(dm, d->dtype);
    const size_t es = d->dtype == SPECINV_F64 ? 8 : 4;
    return (int)cudaMemcpyAsync(env_out, (const char*)plan + pl.env, (size_t)dm.L * es, cudaMemcpyDeviceToDevice,
                                (cudaStream_t)stream);
}

int specinv_plan_inv_env_window(const specinv_desc* d, const void* plan, int64_t x0, int64_t len,
                                int64_t total_frames, void* out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan || (len > 0 && !out) || x0 < 0 || len < 0) return SPECINV_ERR_INVALID;
    if (total_frames != dm.T) {
        if (total_frames >= 0 && total_frames < dm.T) return SPECINV_ERR_INVALID;    // use a plan of total_frames
        if ((long long)(dm.T - 1) * dm.hop < dm.N) return SPECINV_ERR_INVALID;       // head and tail would overlap
        if (total_frames >= 0 && x0 + len > (total_frames - 1) * dm.hop + dm.N - 2LL * dm.P) return SPECINV_ERR_INVALID;
    } else if (x0 + len > dm.L) {
        return SPECINV_ERR_INVALID;
    }
    if (len == 0) return SPECINV_OK;
    const PlanLayout pl = plan_layout(dm, d->dtype);
    const unsigned blocks = (unsigned)((len + 255) / 256);
    if (d->dtype == SPECINV_F64)
        inv_env_window_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>(
            dm, (const double*)((const char*)plan + pl.inv_env), x0, len, total_frames, (double*)out);
    else
        inv_env_window_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>(
            dm, (const float*)((const char*)plan + pl.inv_env), x0, len, total_frames, (float*)out);
    return (int)cudaGetLastError();
}

int specinv_plan_unit_envelope(const specinv_desc* d, void* plan, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!plan) return SPECINV_ERR_INVALID;
    const PlanLayout pl = plan_layout(dm, d->dtype);
    char* p = (char*)plan;
    const unsigned blocks = (unsigned)((dm.L + 255) / 256);
    if (d->dtype == SPECINV_F64)
        fill_ones_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((double*)(p + pl.env), (double*)(p + pl.inv_env), dm.L);
    else
        fill_ones_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((float*)(p + pl.env), (float*)(p + pl.inv_env), dm.L);
    return (int)cudaGetLastError();
}

int specinv_pack_complex(const specinv_desc* d, const void* spec, int64_t sb, int64_t sf, int64_t st,
                         void* main_out, void* nyq_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!spec || !main_out || (dm.onesided && !nyq_out)) return SPECINV_ERR_INVALID;
    if (d->dtype == SPECINV_F64)
        return convert<double2, true>(dm, (double2*)main_out, (double2*)nyq_out, (double2*)spec, sb, sf, st, (cudaStream_t)stream);
    return convert<float2, true>(dm, (float2*)main_out, (float2*)nyq_out, (float2*)spec, sb, sf, st, (cudaStream_t)stream);
}

int specinv_pack_real(const specinv_desc* d, const void* mag, int64_t sb, int64_t sf, int64_t st,
                      void* main_out, void* nyq_out, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!mag || !main_out || (dm.onesided && !nyq_out)) return SPECINV_ERR_INVALID;
    if (d->dtype == SPECINV_F64)
        return convert<double, true>(dm, (double*)main_out, (double*)nyq_out, (double*)mag, sb, sf, st, (cudaStream_t)stream);
    return convert<float, true>(dm, (float*)main_out, (float*)nyq_out, (float*)mag, sb, sf, st, (cudaStream_t)stream);
}

int specinv_unpack_complex(const specinv_desc* d, const void* main_in, const void* nyq_in,
                           void* spec_out, int64_t sb, int64_t sf, int64_t st, void* stream) {
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    if (!spec_out || !main_in || (dm.onesided && !nyq_in)) return SPECINV_ERR_INVALID;
    if (d->dtype == SPECINV_F64)
        return convert<double2, false>(dm, (double2*)main_in, (double2*)nyq_in, (double2*)spec_out, sb, sf, st, (cudaStream_t)stream);
    return convert<float2, false>(dm, (float2*)main_in, (float2*)nyq_in, (float2*)spec_out, sb, sf, st, (cudaStream_t)stream);
}

int specinv_stft(const specinv_desc* d, const void* plan, const void* x, void* main_out, void* nyq_out, void* stream) {
    return generic_stft(d, plan, x, main_out, nyq_out, stream);
}

int specinv_istft(const specinv_desc* d, const void* plan, const void* main_in, const void* nyq_in, void* x_out,
                  void* stream) {
    if (d && plan && main_in && x_out && !force_generic()) {
        const int rw = fastw_istft(d, plan, main_in, nyq_in, x_out, stream);
        if (rw != SPECINV_ERR_UNSUPPORTED) return rw;
    }
    return generic_istft(d, plan, main_in, nyq_in, x_out, stream);
}

int specinv_gl_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                    const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                    const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream) {
    if (!d || !plan || !x_in || !x_out || !mag_main || x_in == x_out) return SPECINV_ERR_INVALID;
    if (!q_in_main && !q_out_main) {
        // plain Griffin-Lim: with lr == 0 the momentum state is neither needed nor produced
        if (lr != 0.0 || q_in_nyq || q_out_nyq) return SPECINV_ERR_INVALID;
        if (!force_generic() && d->onesided && mag_nyq) {
            const int rc = fastw_gl_plain_iter(d, plan, x_in, x_out, mag_main, mag_nyq, sums, stream);
            if (rc != SPECINV_ERR_UNSUPPORTED) return rc;
        }
        return generic_gl_iter(d, plan, x_in, x_out, nullptr, nullptr, nullptr, nullptr, mag_main, mag_nyq, 0.0, sums, stream);
    }
    if (!q_in_main || !q_out_main || q_in_main == q_out_main) return SPECINV_ERR_INVALID;
    if (!force_generic() && d->onesided && q_in_nyq && q_out_nyq && mag_nyq) {
        const int rc = fastw_gl_iter(d, plan, x_in, x_out, q_in_main, q_in_nyq, q_out_main, q_out_nyq, mag_main, mag_nyq,
                                     lr, sums, stream);
        if (rc != SPECINV_ERR_UNSUPPORTED) return rc;
    }
    return generic_gl_iter(d, plan, x_in, x_out, q_in_main, q_in_nyq, q_out_main, q_out_nyq, mag_main, mag_nyq, lr,
                           sums, stream);
}

int specinv_gl_rebuilt_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                            const void* s_in_main, const void* s_in_nyq, void* s_out_main, void* s_out_nyq,
                            const void* mag_main, const void* mag_nyq, double m, double* sums, void* stream) {
    // without state (m == 0) the update is plain Griffin-Lim, exactly what specinv_gl_iter runs then
    if (!s_in_main && !s_out_main)
        return specinv_gl_iter(d, plan, x_in, x_out, nullptr, s_in_nyq, nullptr, s_out_nyq, mag_main, mag_nyq, m, sums,
                               stream);
    if (!d || !plan || !x_in || !x_out || !mag_main || x_in == x_out) return SPECINV_ERR_INVALID;
    if (!s_in_main || !s_out_main || s_in_main == s_out_main) return SPECINV_ERR_INVALID;
    if (!force_generic() && d->onesided && s_in_nyq && s_out_nyq && mag_nyq) {
        const int rc = fastw_gl_rebuilt_iter(d, plan, x_in, x_out, s_in_main, s_in_nyq, s_out_main, s_out_nyq, mag_main,
                                             mag_nyq, m, sums, stream);
        if (rc != SPECINV_ERR_UNSUPPORTED) return rc;
    }
    return generic_gl_rebuilt_iter(d, plan, x_in, x_out, s_in_main, s_in_nyq, s_out_main, s_out_nyq, mag_main, mag_nyq, m,
                                   sums, stream);
}

int specinv_admm_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                      const void* X_in_main, const void* X_in_nyq, const void* U_in_main, const void* U_in_nyq,
                      void* X_out_main, void* X_out_nyq, void* U_out_main, void* U_out_nyq,
                      const void* mag_main, const void* mag_nyq, double rho, double* sums, void* stream) {
    if (!d || !plan || !x_in || !x_out || !X_in_main || !U_in_main || !X_out_main || !U_out_main || !mag_main)
        return SPECINV_ERR_INVALID;
    if (x_in == x_out || X_in_main == X_out_main || U_in_main == U_out_main) return SPECINV_ERR_INVALID;
    if (!force_generic() && d->onesided && X_in_nyq && U_in_nyq && X_out_nyq && U_out_nyq && mag_nyq) {
        const int rc = fastw_admm_iter(d, plan, x_in, x_out, X_in_main, X_in_nyq, U_in_main, U_in_nyq, X_out_main,
                                       X_out_nyq, U_out_main, U_out_nyq, mag_main, mag_nyq, rho, sums, stream);
        if (rc != SPECINV_ERR_UNSUPPORTED) return rc;
    }
    return generic_admm_iter(d, plan, x_in, x_out, X_in_main, X_in_nyq, U_in_main, U_in_nyq, X_out_main, X_out_nyq,
                             U_out_main, U_out_nyq, mag_main, mag_nyq, rho, sums, stream);
}

int specinv_halo_sum(int dtype, const void* left, int64_t ld_left, const void* right, int64_t ld_right, void* out,
                     int64_t ld_out, int rows, int64_t n, void* stream) {
    if (!left || !right || !out || rows < 1 || n < 1) return SPECINV_ERR_INVALID;
    dim3 grid((unsigned)((n + 255) / 256), rows);
    if (dtype == SPECINV_F64)
        halo_sum_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>((const double*)left, ld_left, (const double*)right,
                                                                         ld_right, (double*)out, ld_out, rows, n);
    else if (dtype == SPECINV_F32)
        halo_sum_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)left, ld_left, (const float*)right,
                                                                        ld_right, (float*)out, ld_out, rows, n);
    else return SPECINV_ERR_INVALID;
    return (int)cudaGetLastError();
}

int specinv_fill_padding(int dtype, void* x, int64_t ld, int rows, int64_t padded_offset, int64_t local_len, int pad,
                         int64_t signal_len, int pad_mode, void* stream) {
    if (!x || rows < 1 || pad < 0 || local_len < 1 || signal_len < 1) return SPECINV_ERR_INVALID;
    if (pad == 0) return SPECINV_OK;
    // an interior range of a frame-sharded signal holds no padding sample at all: nothing to launch
    if (padded_offset >= pad && padded_offset + local_len <= pad + signal_len) return SPECINV_OK;
    // A buffer that holds padding samples must also hold their sources: reflect padding mirrors sample P + k onto
    // P - k (and L + P - 1 - k onto L + P - 1 + k), so an edge range needs 2 * pad + 1 samples; otherwise the kernel
    // would have to leave stale padding behind (the source lives on the neighbouring rank).
    if (pad_mode == SPECINV_PAD_REFLECT) {
        const long long end = padded_offset + local_len;                       // buffer = padded samples [offset, end)
        const bool has_left = padded_offset < pad, has_right = end > pad + signal_len;
        // farthest sources: of the first left-pad sample in the buffer (2 pad - offset) and of the last right-pad one
        if (has_left && 2LL * pad - padded_offset >= end) return SPECINV_ERR_INVALID;
        if (has_right && 2LL * signal_len - 2 + 2LL * pad - (end - 1) < padded_offset) return SPECINV_ERR_INVALID;
    }
    if (pad_mode == SPECINV_PAD_CIRCULAR && (padded_offset > 0 || padded_offset + local_len < signal_len + 2LL * pad))
        return SPECINV_ERR_UNSUPPORTED;   // wraps around the whole signal: single-range buffers only
    dim3 grid((unsigned)((2LL * pad + 255) / 256), rows);
    if (dtype == SPECINV_F64)
        fill_padding_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>((double*)x, ld, rows, padded_offset, local_len,
                                                                             pad, signal_len, pad_mode);
    else if (dtype == SPECINV_F32)
        fill_padding_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((float*)x, ld, rows, padded_offset, local_len,
                                                                            pad, signal_len, pad_mode);
    else return SPECINV_ERR_INVALID;
    return (int)cudaGetLastError();
}

int specinv_metric_sums(int dtype, const void* a, const void* b, int64_t n, double* out3, void* stream) {
    if (!a || !b || !out3 || n < 0) return SPECINV_ERR_INVALID;
    if (dtype != SPECINV_F32 && dtype != SPECINV_F64) return SPECINV_ERR_INVALID;
    if (n == 0) return SPECINV_OK;
    long long blocks = (n + 256 * 8 - 1) / (256 * 8);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (dtype == SPECINV_F64)
        metric_sums_kernel<double><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const double*)a, (const double*)b, n, out3);
    else
        metric_sums_kernel<float><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const float*)a, (const float*)b, n, out3);
    return (int)cudaGetLastError();
}

}  // extern "C"
