/*
 * specinv_b200 -- C ABI of the B200-native (sm_100a) iterative STFT/ISTFT
 * phase-retrieval hot path: Griffin-Lim / fast Griffin-Lim, ADMM, RTISI-LA and the
 * spectral metrics of torch_specinv 0.2.1.
 *
 * The reference (yoyololicon/spectrogram-inversion) is pure Python on top of
 * PyTorch ops and has no FFI of its own; the boundary it offers is its Python
 * signatures (torch_specinv/methods.py:193, :273, :415; metrics.py:4,17,32).  This
 * header is the C level directly below them: every entry point replaces the
 * PyTorch-op sequence of one reference code region (cited per function) with
 * hand-written CUDA kernels.  INTEGRATION.md shows the ctypes binding a maintainer
 * of the reference would add.
 *
 * Conventions
 *  - plain C, no torch types; every pointer is a DEVICE pointer unless the name
 *    ends in _host; the caller owns and allocates every buffer;
 *  - every call is asynchronous on the given CUDA stream (a cudaStream_t passed
 *    as void*); nothing synchronises, nothing allocates, no global state;
 *  - return value: 0 = ok, negative = SPECINV_ERR_*, positive = cudaError_t;
 *  - real type is float (SPECINV_F32) or double (SPECINV_F64); complex values are
 *    interleaved (re, im) pairs of that type.
 *
 * Internal ("split, frame-major") spectrum layout used by all kernels
 *    main : [batch][n_frames][row]  complex, row = n_fft/2 (onesided) or n_fft
 *    nyq  : [batch][n_frames]       complex, the k = n_fft/2 bin (onesided only)
 *  magnitudes use the same two arrays with real elements.  Splitting the Nyquist
 *  bin off keeps every frame row 16-byte aligned (n_fft/2 * 8 B) for vector / bulk
 *  loads; specinv_pack_* / specinv_unpack_* convert from / to the reference's
 *  strided (batch, freq, time) tensors.
 */
#ifndef SPECINV_B200_H
#define SPECINV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPECINV_ABI_VERSION 1

enum {
    SPECINV_OK = 0,
    SPECINV_ERR_INVALID = -1,      /* bad argument (null pointer, n_fft out of range, ...) */
    SPECINV_ERR_UNSUPPORTED = -2,  /* valid in the reference but not implemented by these kernels */
    SPECINV_ERR_NO_DEVICE = -3     /* no sm_100 device / kernel image not loadable */
};

enum { SPECINV_F32 = 0, SPECINV_F64 = 1 };

/* torch.stft pad_mode (methods.py:38) */
enum { SPECINV_PAD_REFLECT = 0, SPECINV_PAD_CONSTANT = 1, SPECINV_PAD_REPLICATE = 2, SPECINV_PAD_CIRCULAR = 3 };

/* Normalised STFT description == the output of the reference's _args_helper
 * (methods.py:21-91) plus the problem size. */
typedef struct specinv_desc {
    int32_t n_fft;       /* 16..8192; odd only with onesided = 0 (RTISI-LA: even, n_fft/2 must factor into 2 .. 13) */
    int32_t hop;         /* hop_length, 1..n_fft */
    int32_t n_frames;    /* T */
    int32_t batch;       /* B */
    int32_t center;      /* 0/1 (methods.py:37) */
    int32_t pad_mode;    /* SPECINV_PAD_* (only used when center) */
    int32_t normalized;  /* 0/1: N^-1/2 on both transforms (methods.py:143) */
    int32_t onesided;    /* 0/1 (methods.py:59-68) */
    int32_t dtype;       /* SPECINV_F32 / SPECINV_F64 */
    int32_t reserved[7]; /* must be zero */
} specinv_desc;

int specinv_abi_version(void);
const char* specinv_error_string(int code);

/* Output length of the overlap-add, (T-1)*hop + n_fft - 2*pad  (methods.py:127-128,148). */
int specinv_signal_length(const specinv_desc* d, int64_t* length);

/* ---- plan: twiddles, scaled analysis/synthesis windows, 1/envelope ------------------
 * Replaces _get_ola_weight (methods.py:94-96) and the one-shot envelope
 * conv_transpose1d (methods.py:129-131).  `window` is the n_fft-long window already
 * zero-padded by the host exactly like methods.py:79-83.  inv_env = 1/sum_t w^2 with NO
 * epsilon: a zero envelope gives inf, like the reference's division (methods.py:132). */
int specinv_plan_bytes(const specinv_desc* d, size_t* bytes);
int specinv_plan_init(const specinv_desc* d, const void* window, void* plan, void* stream);
/* Frame-range sharding of one long signal: the plan describes frames [frame_offset, frame_offset + T)
 * of a signal with total_frames frames, un-centred (d->center must be 0; the caller keeps the centre
 * padding inside its local buffer); the envelope counts the neighbouring ranks' frames too, so
 * partial overlap-add sums of two ranks can simply be added. */
int specinv_plan_init_ranged(const specinv_desc* d, const void* window, void* plan, int64_t frame_offset,
                             int64_t total_frames, void* stream);
/* copies the length-L envelope (not its inverse) out of the plan */
int specinv_plan_envelope(const specinv_desc* d, const void* plan, void* env_out, void* stream);
/* replaces the plan's envelope by 1: specinv_istft then returns the plain windowed overlap-add (no
 * normalisation), which is what the adjoint of torch.stft needs (autograd of methods.py:241). */
int specinv_plan_unit_envelope(const specinv_desc* d, void* plan, void* stream);

/* ---- layout conversion (strides in ELEMENTS of the (batch, freq, time) tensor) ---------- */
int specinv_pack_complex(const specinv_desc* d, const void* spec, int64_t sb, int64_t sf, int64_t st,
                         void* main_out, void* nyq_out, void* stream);
int specinv_pack_real(const specinv_desc* d, const void* mag, int64_t sb, int64_t sf, int64_t st,
                      void* main_out, void* nyq_out, void* stream);
int specinv_unpack_complex(const specinv_desc* d, const void* main_in, const void* nyq_in,
                           void* spec_out, int64_t sb, int64_t sf, int64_t st, void* stream);

/* ---- one-shot setup on the split layout ---------------------------------------------------------
 * specinv_phase_init : phase_init, methods.py:572-615 (magnitude -> complex start C = mag*exp(i*phi)),
 *                      one fused pass instead of ~15 full-tensor ops; hop / n_fft come from the desc.
 * specinv_spec_abs   : target magnitude |C| of a complex initial estimate, methods.py:110. */
int specinv_phase_init(const specinv_desc* d, const void* mag_main, const void* mag_nyq, void* c_main, void* c_nyq,
                       void* stream);
/* phase_in / phase_out (nullable): B*F doubles, the running phase before / after this frame range */
int specinv_phase_init_ex(const specinv_desc* d, const void* mag_main, const void* mag_nyq, void* c_main, void* c_nyq,
                          const double* phase_in, double* phase_out, void* stream);
int specinv_spec_abs(const specinv_desc* d, const void* c_main, const void* c_nyq, void* mag_main, void* mag_nyq,
                     void* stream);

/* ---- primitives ---------------------------------------------------------------------------
 * specinv_stft  : torch.stft as called at methods.py:241, :464  (x (B,L) -> spectrum)
 * specinv_istft : _istft, methods.py:135-150 (spectrum -> x (B,L)), envelope from the plan */
int specinv_stft(const specinv_desc* d, const void* plan, const void* x, void* main_out, void* nyq_out,
                 void* stream);
int specinv_istft(const specinv_desc* d, const void* plan, const void* main_in, const void* nyq_in,
                  void* x_out, void* stream);

/* ---- fused iterations ---------------------------------------------------------------------
 * specinv_gl_iter : one closure call of griffin_lim, methods.py:237-250:
 *      s = STFT(x_in); q_out = s - lr*q_in; x_out = ISTFT(q_out*mag/(|q_out|+1e-16))
 *   q_in/q_out and x_in/x_out must not alias (neighbouring tiles re-read the old state).
 *   Plain Griffin-Lim (alpha = 0, so lr = 0 and q_out == s): pass all four q pointers as NULL and the
 *   momentum state is neither read nor written (4 instead of 20 bytes of traffic per bin).
 *   sums (may be NULL): two doubles to which sum (|s|-mag)^2 and sum |s|^2 over all
 *   B*F*T bins are ADDED (the fused metric epilogue for methods.py:181-182).
 * specinv_admm_iter : one closure call of ADMM, methods.py:458-483 with Y == X + U:
 *      R = STFT(x_in); Z = (rho*(X+U)+R)/(1+rho); U' = U+X-Z; X' = proj(Z-U'); x_out = ISTFT(X'+U') */
int specinv_gl_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                    const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                    const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream);
/* specinv_gl_rebuilt_iter : one loop pass of torchaudio.functional.griffinlim, whose fast Griffin-Lim takes the
 *   momentum on the previous REBUILT spectrum instead of the previous momentum spectrum:
 *      s = STFT(x_in); s_out = s; a = s - m*s_in; x_out = ISTFT(mag*a/(|a|+1e-16))      (m = momentum/(1+momentum))
 *   Arguments, aliasing rules, the NULL-state plain Griffin-Lim case (all four s pointers NULL, m = 0: the same kernel
 *   as specinv_gl_iter's) and `sums` as for specinv_gl_iter.  A zero s_in makes the first pass s_out = s, a = s. */
int specinv_gl_rebuilt_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                            const void* s_in_main, const void* s_in_nyq, void* s_out_main, void* s_out_nyq,
                            const void* mag_main, const void* mag_nyq, double m, double* sums, void* stream);
int specinv_admm_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                      const void* X_in_main, const void* X_in_nyq, const void* U_in_main, const void* U_in_nyq,
                      void* X_out_main, void* X_out_nyq, void* U_out_main, void* U_out_nyq,
                      const void* mag_main, const void* mag_nyq, double rho, double* sums, void* stream);

/* ---- RTISI-LA ---------------------------------------------------------------------------------
 * The whole of RTISI_LA's loops and final overlap-add, methods.py:353-408, as one persistent kernel
 * (one CTA per signal, all sliding state on chip).  `window` is the padded n_fft window (as for
 * specinv_plan_init), synth_coeff = hop / (window . window) (methods.py:318), look_ahead < 0 means
 * (n_fft-1)/hop (methods.py:322-324), `scratch` holds 2*n_fft reals (asym_window1/2, methods.py:326-336). */
int specinv_rtisi_la(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                     const void* mag_nyq, void* x_out, void* scratch, int look_ahead, int asymmetric_window,
                     int max_iter, double alpha, double synth_coeff, void* stream);

/* The same run cut at outer-step boundaries (the `for i in range(steps + look_ahead)` loop, methods.py:363): outer
 * steps [step_begin, step_end) of the T + look_ahead steps, each with its max_iter inner iterations, its commit and
 * its block of x_out.  `state` (specinv_rtisi_state_bytes, caller-owned device memory) receives the sliding state
 * before step step_end when step_end < T + look_ahead and provides it when step_begin > 0; per signal, in the real
 * type of the run:
 *   frames [LA+1][n_fft]   active frames, oldest first, as the kernels hold them: the un-normalised inverse FFT
 *                          (= irfft frame of methods.py:398 times n_fft, or times n_fft^1/2 when `normalized`)
 *   pre    [LA+1][F] cplx  momentum spectra of the active frames (methods.py:392; index LA is not used: zero)
 *   kept   [K][n_fft]      kept frames, oldest first, already multiplied by window * synth_coeff (methods.py:365-368)
 *   carry  [n_fft]         overlap-add of the committed frames * window beyond the samples already written (:407)
 * Running [0, s) and [s, T + LA) with the state in between gives bit-identical x_out to one run: this is how the
 * Python layer shows the reference's per-step progress bar (methods.py:362,400), and what the per-step parity tests
 * feed with the oracle's state. */
int specinv_rtisi_state_bytes(const specinv_desc* d, int look_ahead, size_t* bytes);
int specinv_rtisi_la_steps(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                           const void* mag_nyq, void* x_out, void* scratch, int look_ahead, int asymmetric_window,
                           int max_iter, double alpha, double synth_coeff, int step_begin, int step_end, void* state,
                           void* stream);

/* Streaming RTISI-LA: the same outer steps on magnitude frames that arrive a few at a time, with windows of frames and
 * samples instead of whole-signal buffers, so neither the final frame count T nor the output length L is needed
 * before the last call.  d->n_frames = frames received so far (the total when `final`); pad_mode is not used.
 *   magnitudes  mag_main [B][n_rows][row], mag_nyq [B][n_rows]: row r of a signal is frame frame0 + r.  The rows must
 *               reach from max(0, step_begin - LA) -- a resume re-reads the LA older active frames -- to the newest
 *               frame the steps read, min(step_end, n_frames) - 1; frame0 <= max(0, step_begin - LA).
 *   x_out       [B][x_len]: column c of a signal is output sample x0 + c.  The window must be exactly the samples
 *               these steps finish: the commit of step i finishes [(i-LA)*hop - P, (i-LA+1)*hop - P) (P = n_fft/2 when
 *               centred, else 0; clamped at 0), and a final call also finishes everything up to L = (n_frames-1)*hop
 *               + n_fft - 2P.  Without `final` the window is not clamped at L: samples past L(n_frames) are final as
 *               values but belong to the signal only if more frames follow (the caller holds them back).
 *   inv_env     [x_len]: 1/envelope of samples [x0, x0 + x_len) (specinv_plan_inv_env_window).
 *   plan        any plan of this n_fft / hop / window / normalized / onesided / dtype: only its T-independent
 *               tables are read.
 *   steps       [step_begin, step_end): step i reads frame i, so step_end <= n_frames without `final` and
 *               step_end <= n_frames + LA with it.  Only the final call may be empty (step_begin == step_end ==
 *               n_frames + LA, look_ahead = 0): it releases the carry the commit of frame n_frames-1 left behind.
 *   final       0/1: n_frames is the total; frames past it have zero magnitude (methods.py:339), the commit of frame
 *               n_frames-1 flushes the whole carry and no state is saved after step n_frames + LA.
 *   state       as for specinv_rtisi_la_steps (its bytes do not depend on n_frames); always required.
 * Every argument is checked before any launch (SPECINV_ERR_INVALID).  The kernel is chosen as for specinv_rtisi_la,
 * and the concatenated windows of any sequence of calls are bit-identical to one specinv_rtisi_la run. */
int specinv_rtisi_la_stream(const specinv_desc* d, const void* plan, const void* window, const void* mag_main,
                            const void* mag_nyq, int frame0, int n_rows, void* x_out, const void* inv_env, int64_t x0,
                            int64_t x_len, void* scratch, int look_ahead, int asymmetric_window, int max_iter,
                            double alpha, double synth_coeff, int step_begin, int step_end, int final, void* state,
                            void* stream);
/* out[j] = 1/envelope of sample x0 + j of a signal with total_frames frames (< 0: not known yet; then only samples
 * whose covering frames all exist may be asked for), gathered from a plan of d->n_frames = T0 frames.  The envelope
 * sums w^2 over the covering frames in ascending order, so a sample's value depends only on (m + P) mod hop and on
 * which end clips its frame range: head, interior and tail of any signal are bitwise equal to the plan's.  Needs
 * (T0 - 1) * hop >= n_fft, and total_frames >= T0 or < 0; total_frames == T0 reads the plan as it is. */
int specinv_plan_inv_env_window(const specinv_desc* d, const void* plan, int64_t x0, int64_t len,
                                int64_t total_frames, void* out, void* stream);

/* ---- frame-range sharding helpers (single long signal over several GPUs) --------------------------
 * specinv_halo_sum    : out = left + right over rows x n strided views -- the per-iteration combination of
 *                       the two partial overlap-add sums of the (n_fft - hop)-sample region two neighbouring
 *                       ranks share (each rank receives the other's partial by NVLink P2P / NCCL send-recv).
 * specinv_fill_padding: re-creates the centre padding (torch.stft pad_mode) of the GLOBAL signal inside a
 *                       rank-local padded buffer holding padded samples [padded_offset, padded_offset+local_len). */
int specinv_halo_sum(int dtype, const void* left, int64_t ld_left, const void* right, int64_t ld_right, void* out,
                     int64_t ld_out, int rows, int64_t n, void* stream);
int specinv_fill_padding(int dtype, void* x, int64_t ld, int rows, int64_t padded_offset, int64_t local_len, int pad,
                         int64_t signal_len, int pad_mode, void* stream);

/* The same exchange as ONE kernel over NVLink peer memory (no NCCL call, no host synchronisation): every rank owns
 * a receive area of specinv_halo_area_bytes() allocated by specinv_ipc_alloc (cudaMalloc + cudaIpcGetMemHandle, 64-byte
 * handle to hand to the neighbours through any channel) and maps its neighbours' areas with specinv_ipc_open.
 * specinv_halo_exchange pushes this rank's partial sums of the first / last `ov` samples of every row of x into the
 * left / right neighbour's area (NULL: no neighbour), raises their flags to `seq` (1, 2, 3, ... per exchange), waits
 * for its own flags and adds left partial + right partial in place.  The wait is bounded (SPECINV_P2P_TIMEOUT_MS,
 * default 10000): after a timeout the kernel records the exchange number in the area's status word and this and all
 * later exchanges return without adding; specinv_halo_status copies that word to the host (synchronising `stream`):
 * 0 = every exchange so far found its neighbour. */
size_t specinv_halo_area_bytes(int dtype, int rows, int64_t ov);
int specinv_ipc_alloc(size_t bytes, void** dptr, void* handle64);
int specinv_ipc_open(const void* handle64, void** dptr);
int specinv_ipc_close(void* dptr);
int specinv_ipc_free(void* dptr);
int specinv_halo_exchange(int dtype, void* x, int64_t ld, int rows, int64_t local_len, int64_t ov, void* recv_self,
                          void* recv_left_peer, void* recv_right_peer, uint32_t seq, void* stream);
int specinv_halo_status(int dtype, const void* recv_self, int rows, int64_t ov, uint32_t* status, void* stream);

/* ---- small problems: a whole run of fast Griffin-Lim iterations in ONE persistent kernel ---------------------
 * (csrc/specinv_resident.cu; replaces n_iters calls of specinv_gl_iter, i.e. n_iters passes of the closure
 * methods.py:237-250 under the loop methods.py:178-190).  When B * T frames fit the shared memory of the SMs
 * (hop = n_fft/4, n_fft 1024 / 2048 / 4096, fp32, onesided, not circular padding, at most one signal per SM) the
 * momentum spectra, magnitudes and signal stay on chip for all iterations; HBM sees the state once in, once out.
 *   specinv_gl_run_workspace_bytes: SPECINV_ERR_UNSUPPORTED when the problem does not fit -- use specinv_gl_iter.
 *   specinv_gl_run: iterations iter0 .. iter0 + n_iters - 1; those with (i % eva_iter) == eva_iter - 1 add their
 *     metric sums (as specinv_gl_iter's `sums`) to sums[2 k], sums[2 k + 1], k = 0, 1, ... in order (sums == NULL:
 *     no evaluation).  q_in / q_out and x_in / x_out may alias.  `workspace` (16-byte aligned, caller-owned, device)
 *     carries the neighbour exchange of the CTAs; nothing is allocated, nothing synchronises.
 *   specinv_gl_run_status: 0, or the iteration at which a CTA timed out waiting for a neighbour
 *     (SPECINV_RESIDENT_TIMEOUT_MS, default 5000; the result is then invalid).  Synchronises `stream`. */
int specinv_gl_run_workspace_bytes(const specinv_desc* d, size_t* bytes);
int specinv_gl_run(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                   const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                   const void* mag_main, const void* mag_nyq, double lr, int n_iters, int iter0, int eva_iter,
                   double* sums, void* workspace, void* stream);
int specinv_gl_run_status(const specinv_desc* d, const void* workspace, uint32_t* status, void* stream);

/* ---- torchaudio's InverseMelScale (csrc/specinv_mel.cu, spectrogram_inversion_b200.torchaudio_compat) -----------
 * out[b, f, t] = relu(sum_j P[f, j] * mel[b, j, t]) for f in [f_lo, f_hi), and 0 for every other f (no multiply).
 *   P    [n_stft][n_mels] row-major: pinv(fb^T), the minimum-norm least-squares operator of the mel filterbank; its
 *        rows outside [f_lo, f_hi) must be zero (bins no filter covers).  Not read when f_lo == f_hi.
 *   mel  [batch][n_mels][n_frames] contiguous;  out [batch][n_stft][n_frames] contiguous (torchaudio's layout).
 * relu is torch.relu's: NaN stays NaN.  Any n_stft >= 1, n_mels >= 1 (the kernel tiles over n_mels); FFMA in fp32,
 * DFMA in fp64, summed over j in ascending order.  Every argument is checked before any launch (SPECINV_ERR_INVALID:
 * dtype, sizes, 0 <= f_lo <= f_hi <= n_stft, NULL pointers); n_frames == 0 launches nothing. */
int specinv_mel_inverse(int dtype, const void* P, int n_stft, int n_mels, int f_lo, int f_hi, const void* mel,
                        void* out, int batch, int64_t n_frames, void* stream);

/* ---- metrics (metrics.py:4-43, F.mse_loss at methods.py:182) ---------------------------------
 * out[0] += sum (a-b)^2, out[1] += sum a^2, out[2] += sum b^2 over n contiguous reals. */
int specinv_metric_sums(int dtype, const void* a, const void* b, int64_t n, double* out3, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPECINV_B200_H */
