// Entry points of the specialised fused kernels (specinv_fastw_kernel.cuh) and the hop = n_fft/4 instances; the
// hop = n_fft/2 and n_fft/8 instances live in specinv_fastw_ov2.cu / specinv_fastw_ov8.cu.
#include "specinv_fastw_kernel.cuh"

namespace specinv {
namespace wfast {
SPECINV_FASTW_DEFINE_LAUNCH(4)

static int launch_op(int op, const WArgs& a, const specinv_desc* d, cudaStream_t st) {
    switch (d->n_fft / d->hop) {
        case 2: return fastw_launch_ov2(op, a, d->n_fft, st);
        case 4: return fastw_launch_ov4(op, a, d->n_fft, st);
        case 8: return fastw_launch_ov8(op, a, d->n_fft, st);
        default: return SPECINV_ERR_UNSUPPORTED;
    }
}
}  // namespace wfast

static bool fastw_applicable(const specinv_desc* d) {
    return d->dtype == SPECINV_F32 && d->onesided &&
           (d->hop * 2 == d->n_fft || d->hop * 4 == d->n_fft || d->hop * 8 == d->n_fft) &&
           (d->n_fft == 512 || d->n_fft == 1024 || d->n_fft == 2048 || d->n_fft == 4096);
}

static void fill_common(wfast::WArgs& a, const Dims& dm, const specinv_desc* d, const void* plan) {
    const PlanLayout pl = plan_layout(dm, d->dtype);
    const char* p = (const char*)plan;
    a.tw = (const float2*)(p + pl.tw); a.twr = (const float2*)(p + pl.twr);
    a.wa = (const float*)(p + pl.wa); a.ws = (const float*)(p + pl.ws); a.inv_env = (const float*)(p + pl.inv_env);
    a.B = dm.B; a.T = dm.T; a.P = dm.P; a.pad_mode = dm.pad_mode; a.L = dm.L;
}

// Return SPECINV_ERR_UNSUPPORTED when the shape is not one these kernels are specialised for.
// op = OP_GL (state q = s - lr q_prev) or OP_GLR (state = the rebuilt spectrum s, the projection gets s - lr s_prev).
static int fastw_momentum_iter(int op, const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                               const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                               const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream) {
    if (!fastw_applicable(d)) return SPECINV_ERR_UNSUPPORTED;
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    wfast::WArgs a{};
    fill_common(a, dm, d, plan);
    a.x_in = (const float*)x_in; a.x_out = (float*)x_out;
    a.s0_in = (const float2*)q_in_main; a.s0_in_nyq = (const float2*)q_in_nyq;
    a.s0_out = (float2*)q_out_main; a.s0_out_nyq = (float2*)q_out_nyq;
    a.mag = (const float*)mag_main; a.mag_nyq = (const float*)mag_nyq;
    a.coef = (float)lr; a.sums = sums;
    return wfast::launch_op(op, a, d, (cudaStream_t)stream);
}

int fastw_gl_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                  const void* q_in_main, const void* q_in_nyq, void* q_out_main, void* q_out_nyq,
                  const void* mag_main, const void* mag_nyq, double lr, double* sums, void* stream) {
    return fastw_momentum_iter(wfast::OP_GL, d, plan, x_in, x_out, q_in_main, q_in_nyq, q_out_main, q_out_nyq, mag_main,
                               mag_nyq, lr, sums, stream);
}

int fastw_gl_rebuilt_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                          const void* s_in_main, const void* s_in_nyq, void* s_out_main, void* s_out_nyq,
                          const void* mag_main, const void* mag_nyq, double m, double* sums, void* stream) {
    return fastw_momentum_iter(wfast::OP_GLR, d, plan, x_in, x_out, s_in_main, s_in_nyq, s_out_main, s_out_nyq,
                               mag_main, mag_nyq, m, sums, stream);
}

// Plain Griffin-Lim (alpha = 0, methods.py:243 with lr = 0): x_out = ISTFT(proj(STFT(x_in))), no momentum state.
int fastw_gl_plain_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out, const void* mag_main,
                        const void* mag_nyq, double* sums, void* stream) {
    if (!fastw_applicable(d)) return SPECINV_ERR_UNSUPPORTED;
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    wfast::WArgs a{};
    fill_common(a, dm, d, plan);
    a.x_in = (const float*)x_in; a.x_out = (float*)x_out;
    a.mag = (const float*)mag_main; a.mag_nyq = (const float*)mag_nyq;
    a.sums = sums;
    return wfast::launch_op(wfast::OP_GLP, a, d, (cudaStream_t)stream);
}

// x_out = ISTFT(spectrum) (methods.py:135-150) with the same kernel: inverse half of the frame pipeline only.
int fastw_istft(const specinv_desc* d, const void* plan, const void* main_in, const void* nyq_in, void* x_out,
                void* stream) {
    if (!fastw_applicable(d) || !nyq_in) return SPECINV_ERR_UNSUPPORTED;
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    wfast::WArgs a{};
    fill_common(a, dm, d, plan);
    a.x_out = (float*)x_out;
    a.s0_in = (const float2*)main_in; a.s0_in_nyq = (const float2*)nyq_in;
    return wfast::launch_op(wfast::OP_ISTFT, a, d, (cudaStream_t)stream);
}

int fastw_admm_iter(const specinv_desc* d, const void* plan, const void* x_in, void* x_out,
                    const void* X_in_main, const void* X_in_nyq, const void* U_in_main, const void* U_in_nyq,
                    void* X_out_main, void* X_out_nyq, void* U_out_main, void* U_out_nyq,
                    const void* mag_main, const void* mag_nyq, double rho, double* sums, void* stream) {
    if (!fastw_applicable(d)) return SPECINV_ERR_UNSUPPORTED;
    Dims dm; int rc = make_dims(d, &dm); if (rc) return rc;
    wfast::WArgs a{};
    fill_common(a, dm, d, plan);
    a.x_in = (const float*)x_in; a.x_out = (float*)x_out;
    a.s0_in = (const float2*)X_in_main; a.s0_in_nyq = (const float2*)X_in_nyq;
    a.s0_out = (float2*)X_out_main; a.s0_out_nyq = (float2*)X_out_nyq;
    a.s1_in = (const float2*)U_in_main; a.s1_in_nyq = (const float2*)U_in_nyq;
    a.s1_out = (float2*)U_out_main; a.s1_out_nyq = (float2*)U_out_nyq;
    a.mag = (const float*)mag_main; a.mag_nyq = (const float*)mag_nyq;
    a.coef = (float)rho; a.coef2 = (float)(1.0 / (1.0 + rho)); a.sums = sums;
    return wfast::launch_op(wfast::OP_ADMM, a, d, (cudaStream_t)stream);
}

}  // namespace specinv
