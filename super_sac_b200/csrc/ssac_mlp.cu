// C-ABI dispatch for the ensemble MLP entry points (see include/ssac_b200.h).
#include <cstring>

#include "ssac_mlp.cuh"

namespace ssac {
int mlp_forward_simt(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                     const float* b3, const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx,
                     int64_t x_gs, int B, float* h1, float* h2, float* y, cudaStream_t s, int impl, const HeadEpi* epi,
                     int phase, int keep_hidden);
int mlp_forward_rows(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                     const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx, int B, float* y,
                     cudaStream_t s);
void set_fused_forward(int on);
int get_fused_forward();
int mlp_backward_pre(const float* W2, const float* W3, int G, int H, int B, const float* h1, const float* h2, float* ws, int u_async,
                     cudaStream_t s, int impl);
int mlp_backward_post(const float* W3, int G, int D, int H, const float* x, int64_t ldx, int64_t x_gs, int B, const float* h1,
                      const float* h2, const float* dq, float* ws, float* gW1, float* gb1, float* gW2, float* gb2,
                      float* gW3, float* gb3, cudaStream_t s, int impl);
int mlp_backward_dact(const float* W1, const float* W2, const float* W3, int G, int D, int H, int col0, int A, int B,
                      const float* h1, const float* h2, const float* dq, float* da, float* ws, cudaStream_t s, int impl);
void set_overlap(int on);
int get_overlap();
int mlp_backward_simt(const float* W1, const float* W2, const float* W3, const int32_t* net_index, int G, int D, int H,
                      int O, const float* x, int64_t ldx, int64_t x_gs, int B, const float* h1, const float* h2,
                      const float* dy, const float* dh2_extra, float extra_scale, float* gW1, float* gb1, float* gW2,
                      float* gb2, float* gW3, float* gb3, int accumulate, float* dx, int64_t lddx, float* ws,
                      cudaStream_t s, int impl);
}  // namespace ssac

using namespace ssac;

static int g_default_impl = 2;  // tcgen05 3xTF32 tensor-core path

extern "C" {

int ssac_default_mlp_impl(void) { return g_default_impl; }
int ssac_set_default_mlp_impl(int impl) {
  if (impl != 1 && impl != 2) return fail(SSAC_E_BADARG, "ssac_set_default_mlp_impl: impl must be 1 (fp32 FFMA) or 2 (tcgen05 3xTF32)");
  g_default_impl = impl;
  return 0;
}

int ssac_set_fused_forward(int on) { set_fused_forward(on); return 0; }
int ssac_get_fused_forward(void) { return get_fused_forward(); }
int ssac_set_overlap(int on) { set_overlap(on); return 0; }
int ssac_get_overlap(void) { return get_overlap(); }

int ssac_mlp_forward(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                     const float* b3, const int32_t* net_index_dev, int G, int D, int H, int O, const float* x_dev,
                     int64_t ldx, int64_t x_gs, int B, float* h1_dev, float* h2_dev, int keep_hidden, float* y_dev,
                     int impl, void* stream) {
  SSAC_REQUIRE(W1 && b1 && W2 && b2 && W3 && b3 && x_dev && y_dev, "ssac_mlp_forward: null pointer");
  SSAC_REQUIRE(G > 0 && D > 0 && H > 0 && O > 0 && B > 0 && ldx >= D, "ssac_mlp_forward: bad sizes");
  if (impl == 0) impl = ssac_default_mlp_impl();
  if (impl == 1 || impl == 2)
    return mlp_forward_simt(W1, b1, W2, b2, W3, b3, net_index_dev, G, D, H, O, x_dev, ldx, x_gs, B, h1_dev, h2_dev,
                            y_dev, (cudaStream_t)stream, impl, nullptr, 0, keep_hidden);
  if (impl == 3) {
    SSAC_REQUIRE(!keep_hidden && x_gs == 0, "ssac_mlp_forward: impl 3 is forward-only on a shared batch");
    return mlp_forward_rows(W1, b1, W2, b2, W3, b3, net_index_dev, G, D, H, O, x_dev, ldx, B, y_dev, (cudaStream_t)stream);
  }
  return fail(SSAC_E_UNSUPPORTED, "ssac_mlp_forward: unknown impl");
}

int ssac_actor_forward_sample(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                              const float* b3, int D, int H, int A, int deterministic, const float* x_dev, int64_t ldx,
                              int B, float* h1_dev, float* h2_dev, int keep_hidden, float* out_dev, const float* eps_dev,
                              const float* noise_dev, float sigma, float clip, float log_std_lo, float log_std_hi,
                              float* a_dev, int64_t lda, float* logp_dev, float* tanh_out_dev, int impl, void* stream) {
  SSAC_REQUIRE(W1 && b1 && W2 && b2 && W3 && b3 && x_dev && out_dev && a_dev && h1_dev && h2_dev,
               "ssac_actor_forward_sample: null pointer");
  SSAC_REQUIRE(D > 0 && H > 0 && A > 0 && A <= 16 && B > 0 && ldx >= D && lda >= A, "ssac_actor_forward_sample: bad sizes");
  SSAC_REQUIRE(deterministic || eps_dev, "ssac_actor_forward_sample: a stochastic actor needs eps");
  if (impl == 0) impl = ssac_default_mlp_impl();
  HeadEpi e;
  memset(&e, 0, sizeof(e));
  e.kind = deterministic ? 2 : 1;
  e.eps = eps_dev; e.noise = noise_dev; e.sigma = sigma; e.clip = clip; e.lo = log_std_lo; e.hi = log_std_hi;
  e.a = a_dev; e.lda = lda; e.logp = logp_dev; e.tanh_out = tanh_out_dev; e.A = A;
  return mlp_forward_simt(W1, b1, W2, b2, W3, b3, nullptr, 1, D, H, deterministic ? A : 2 * A, x_dev, ldx, 0, B, h1_dev,
                          h2_dev, out_dev, (cudaStream_t)stream, impl, &e, 0, keep_hidden);
}

int ssac_critic_forward_loss(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                             const float* b3, int N, int D, int H, const float* x_dev, int64_t ldx, int B,
                             float* h1_dev, float* h2_dev, float* q_dev, const float* y_dev, const float* w_dev,
                             const float* imp_dev, const float* popart_dev, int pop, int E, int n_total, float* dq_dev,
                             float* loss_dev, int phase, const float* qt_dev, int M, const float* logp_dev,
                             const float* log_alpha_dev, const float* r_dev, const float* d_dev, double gamma,
                             float* y_out_dev, float* td_logs_dev, int impl, void* stream) {
  SSAC_REQUIRE(W1 && b1 && W2 && b2 && W3 && b3 && x_dev && h1_dev && h2_dev &&
                   (phase == 1 || (q_dev && (y_dev || qt_dev) && dq_dev)),
               "ssac_critic_forward_loss: null pointer");
  SSAC_REQUIRE(N > 0 && D > 0 && H > 0 && B > 0 && E > 0 && ldx >= D, "ssac_critic_forward_loss: bad sizes");
  SSAC_REQUIRE(!qt_dev || (phase == 2 && M > 0 && r_dev && d_dev && !(popart_dev && pop)),
               "ssac_critic_forward_loss: the in-place TD target needs phase 2, M > 0, r, d and no PopArt");
  if (impl == 0) impl = ssac_default_mlp_impl();
  HeadEpi e;
  memset(&e, 0, sizeof(e));
  e.kind = 3;
  e.y = y_dev; e.w = w_dev; e.imp = imp_dev; e.popart = popart_dev; e.pop = pop;
  e.inv_count = 1.f / ((float)B * (float)E * (float)(n_total > 0 ? n_total : N));
  e.dq = dq_dev; e.loss = loss_dev;
  e.qt = qt_dev; e.M = M; e.logp_t = logp_dev; e.log_alpha = log_alpha_dev; e.r = r_dev; e.d = d_dev; e.gamma = (float)gamma;
  e.y_out = y_out_dev; e.td_logs = td_logs_dev;
  return mlp_forward_simt(W1, b1, W2, b2, W3, b3, nullptr, N, D, H, 1, x_dev, ldx, 0, B, h1_dev, h2_dev, q_dev,
                          (cudaStream_t)stream, impl, &e, phase, 1);
}

int64_t ssac_mlp_backward_ws(int G, int B, int H) { return 2 * (int64_t)G * B * H; }

int ssac_mlp_backward(const float* W1, const float* W2, const float* W3, const int32_t* net_index_dev, int G, int D,
                      int H, int O, const float* x_dev, int64_t ldx, int64_t x_gs, int B, const float* h1_dev,
                      const float* h2_dev, const float* dy_dev, const float* dh2_extra_dev, float extra_scale,
                      float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3, int accumulate,
                      float* dx_dev, int64_t lddx, float* ws_dev, int impl, void* stream) {
  SSAC_REQUIRE(W1 && W2 && W3 && x_dev && h1_dev && h2_dev, "ssac_mlp_backward: null pointer");
  SSAC_REQUIRE(G > 0 && D > 0 && H > 0 && O > 0 && B > 0 && ldx >= D, "ssac_mlp_backward: bad sizes");
  SSAC_REQUIRE(!dx_dev || lddx >= D, "ssac_mlp_backward: lddx < D");
  if (impl == 0) impl = ssac_default_mlp_impl();
  if (impl == 1 || impl == 2)
    return mlp_backward_simt(W1, W2, W3, net_index_dev, G, D, H, O, x_dev, ldx, x_gs, B, h1_dev, h2_dev, dy_dev,
                             dh2_extra_dev, extra_scale, gW1, gb1, gW2, gb2, gW3, gb3, accumulate, dx_dev, lddx,
                             ws_dev, (cudaStream_t)stream, impl);
  return fail(SSAC_E_UNSUPPORTED, "ssac_mlp_backward: unknown impl");
}

int ssac_mlp_backward_pre(const float* W2, const float* W3, int G, int H, int B, const float* h1_dev, const float* h2_dev,
                          float* ws_dev, int u_async, int impl, void* stream) {
  SSAC_REQUIRE(W2 && W3 && h1_dev && h2_dev && ws_dev, "ssac_mlp_backward_pre: null pointer");
  SSAC_REQUIRE(G > 0 && H > 0 && B > 0, "ssac_mlp_backward_pre: bad sizes");
  if (impl == 0) impl = ssac_default_mlp_impl();
  if (impl != 2) return fail(SSAC_E_UNSUPPORTED, "ssac_mlp_backward_pre: the split backward exists for impl 2 (tcgen05) only");
  return mlp_backward_pre(W2, W3, G, H, B, h1_dev, h2_dev, ws_dev, u_async, (cudaStream_t)stream, impl);
}

int ssac_mlp_backward_post(const float* W3, int G, int D, int H, const float* x_dev, int64_t ldx, int64_t x_gs, int B,
                           const float* h1_dev, const float* h2_dev, const float* dq_dev, float* ws_dev, float* gW1,
                           float* gb1, float* gW2, float* gb2, float* gW3, float* gb3, int impl, void* stream) {
  SSAC_REQUIRE(W3 && x_dev && h1_dev && h2_dev && dq_dev && ws_dev && gW1 && gb1 && gW2 && gb2 && gW3 && gb3,
               "ssac_mlp_backward_post: null pointer");
  SSAC_REQUIRE(G > 0 && D > 0 && H > 0 && B > 0 && ldx >= D, "ssac_mlp_backward_post: bad sizes");
  if (impl == 0) impl = ssac_default_mlp_impl();
  if (impl != 2) return fail(SSAC_E_UNSUPPORTED, "ssac_mlp_backward_post: the split backward exists for impl 2 (tcgen05) only");
  return mlp_backward_post(W3, G, D, H, x_dev, ldx, x_gs, B, h1_dev, h2_dev, dq_dev, ws_dev, gW1, gb1, gW2, gb2, gW3, gb3,
                           (cudaStream_t)stream, impl);
}

int ssac_mlp_backward_dact(const float* W1, const float* W2, const float* W3, int G, int D, int H, int col0, int A, int B,
                           const float* h1_dev, const float* h2_dev, const float* dq_dev, float* da_dev, float* ws_dev,
                           int impl, void* stream) {
  SSAC_REQUIRE(W1 && W2 && W3 && h1_dev && h2_dev && dq_dev && da_dev && ws_dev, "ssac_mlp_backward_dact: null pointer");
  SSAC_REQUIRE(G > 0 && D > 0 && H > 0 && B > 0, "ssac_mlp_backward_dact: bad sizes");
  if (impl == 0) impl = ssac_default_mlp_impl();
  if (impl != 1 && impl != 2) return fail(SSAC_E_UNSUPPORTED, "ssac_mlp_backward_dact: unknown impl");
  return mlp_backward_dact(W1, W2, W3, G, D, H, col0, A, B, h1_dev, h2_dev, dq_dev, da_dev, ws_dev, (cudaStream_t)stream, impl);
}

}  // extern "C"
