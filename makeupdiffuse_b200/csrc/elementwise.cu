// Probes, the fused DDIM / PLMS / DPM-Solver update (+CFG) kernels, the fused DDPM step, layout conversion and the small elementwise kernels.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>

#include "common.cuh"

namespace mkd {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  char tmp[sizeof(g_err)];  // an argument may be mkd_last_error() itself (a decline reason quoted by the next message)
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tmp, sizeof(tmp), fmt, ap);
  va_end(ap);
  memcpy(g_err, tmp, sizeof(g_err));
}
bool pdl_enabled() {
  // on: 6.97 -> 6.74 ms per UNet+ControlNet step (round 2; it measured slightly negative in round 1, before the launch
  // count fell and the GEMM prologues grew a cluster rendezvous)
  static const int v = debug_switch("MKD_PDL", 1);
  return v == 1;
}
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace mkd
using namespace mkd;

extern "C" long long mkd_launch_count(void) { return mkd::g_launches.load(std::memory_order_relaxed); }
extern "C" int mkd_abi_version(void) { return MKD_ABI_VERSION; }
extern "C" int mkd_compiled_arch(void) { return 100; }
extern "C" const char* mkd_last_error(void) { return mkd::g_err; }
extern "C" int mkd_device_ok(int device) {
  cudaDeviceProp p;
  cudaError_t e = cudaGetDeviceProperties(&p, device);
  MKD_REQUIRE(e == cudaSuccess, MKD_E_CUDA, "cudaGetDeviceProperties(%d): %s", device, cudaGetErrorString(e));
  MKD_REQUIRE(p.major == 10 && p.minor == 0, MKD_E_ARCH,
              "device %d is sm_%d%d; libmkd_b200 is built for sm_100a (B200) only and has no fallback", device,
              p.major, p.minor);
  return MKD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// DDIM update.  Latents are tiny (4096 floats per 256^2 sample): the point of the kernel is ONE launch
// instead of ~12 ATen kernels + 4 torch.full + a cat/chunk per step, and exact fp32 op-by-op rounding.
// ---------------------------------------------------------------------------------------------------------
__global__ void ddim_update_kernel(const float* __restrict__ x, const float* __restrict__ eps, int cfg,
                                   float cfg_scale, const float* __restrict__ noise, float s1m, float sqrt_at,
                                   float sqrt_ap, float dirc, float sigma, float temp, float* __restrict__ x_prev,
                                   float* __restrict__ pred_x0, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float e = eps[i];
    if (cfg) {
      float ec = eps[n + i];
      e = __fadd_rn(e, __fmul_rn(cfg_scale, __fsub_rn(ec, e)));  // e_u + s * (e_c - e_u)   cddim.py:40
    }
    float xv = x[i];
    float p0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(s1m, e)), sqrt_at);  // cddim.py:63
    float xp = __fadd_rn(__fmul_rn(sqrt_ap, p0), __fmul_rn(dirc, e));  // cddim.py:74,78
    if (noise) xp = __fadd_rn(xp, __fmul_rn(__fmul_rn(sigma, noise[i]), temp));  // cddim.py:75,78
    if (pred_x0) pred_x0[i] = p0;
    x_prev[i] = xp;
  }
}

// The same update writing x_prev into the gather buffers of up to 8 ranks (peer memory mapped over NVLink): the final
// step of a batch-sharded run produces its slice of the all-gathered result directly in every rank's buffer, so the
// path's only collective needs no separate launch (a signal barrier between the ranks follows on the host side).
struct PeerPtrs {
  float* p[8];
};
template <int NP>
__global__ void ddim_update_peers_kernel(const float* __restrict__ x, const float* __restrict__ eps, int cfg,
                                         float cfg_scale, const float* __restrict__ noise, float s1m, float sqrt_at,
                                         float sqrt_ap, float dirc, float sigma, float temp, PeerPtrs out,
                                         float* __restrict__ pred_x0, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float e = eps[i];
    if (cfg) {
      float ec = eps[n + i];
      e = __fadd_rn(e, __fmul_rn(cfg_scale, __fsub_rn(ec, e)));
    }
    float xv = x[i];
    float p0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(s1m, e)), sqrt_at);
    float xp = __fadd_rn(__fmul_rn(sqrt_ap, p0), __fmul_rn(dirc, e));
    if (noise) xp = __fadd_rn(xp, __fmul_rn(__fmul_rn(sigma, noise[i]), temp));
    if (pred_x0) pred_x0[i] = p0;
#pragma unroll
    for (int r = 0; r < NP; ++r) out.p[r][i] = xp;
  }
}

extern "C" int mkd_ddim_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, const float* noise,
                                     float sqrt_one_minus_at, float sqrt_at, float sqrt_a_prev, float dir_coef,
                                     float sigma_t, float temperature, float* const* x_prev_peers, int n_peers,
                                     float* pred_x0, int64_t n, mkd_stream_t stream) {
  MKD_REQUIRE(x && eps && x_prev_peers && n >= 0, MKD_E_INVALID, "ddim_update_peers: null pointer or negative n");
  MKD_REQUIRE(n_peers >= 1 && n_peers <= 8, MKD_E_INVALID, "ddim_update_peers: n_peers=%d must be 1..8 (one box)", n_peers);
  PeerPtrs pp;
  for (int r = 0; r < 8; ++r) pp.p[r] = r < n_peers ? x_prev_peers[r] : nullptr;  // host array of device pointers
  for (int r = 0; r < n_peers; ++r) MKD_REQUIRE(pp.p[r] != nullptr, MKD_E_INVALID, "ddim_update_peers: null peer pointer %d", r);
  if (n == 0) return MKD_OK;
  int threads = 256;
  int blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t st = (cudaStream_t)stream;
#define MKD_PEERS_CASE(NP)                                                                                              \
  case NP:                                                                                                              \
    MKD_LAUNCH_OK(launch_pdl(ddim_update_peers_kernel<NP>, dim3(blocks), dim3(threads), 0, st, x, eps, cfg, cfg_scale,  \
                             noise, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef, sigma_t, temperature, pp,        \
                             pred_x0, n));                                                                              \
    break;
  switch (n_peers) {
    MKD_PEERS_CASE(1) MKD_PEERS_CASE(2) MKD_PEERS_CASE(3) MKD_PEERS_CASE(4)
    MKD_PEERS_CASE(5) MKD_PEERS_CASE(6) MKD_PEERS_CASE(7) MKD_PEERS_CASE(8)
  }
#undef MKD_PEERS_CASE
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

extern "C" int mkd_ddim_update(const float* x, const float* eps, int cfg, float cfg_scale, const float* noise,
                               float sqrt_one_minus_at, float sqrt_at, float sqrt_a_prev, float dir_coef,
                               float sigma_t, float temperature, float* x_prev, float* pred_x0, int64_t n,
                               mkd_stream_t stream) {
  MKD_REQUIRE(x && eps && x_prev && n >= 0, MKD_E_INVALID, "ddim_update: null pointer or negative n");
  if (n == 0) return MKD_OK;
  int threads = 256;
  int blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  MKD_LAUNCH_OK(launch_pdl(ddim_update_kernel, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, eps, cfg, cfg_scale, noise, sqrt_one_minus_at,
                                                                   sqrt_at, sqrt_a_prev, dir_coef, sigma_t,
                                                                   temperature, x_prev, pred_x0, n));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// PLMS update (upstream ldm/models/diffusion/plms.py p_sample_plms): the CFG combine, the store of e_t into the
// sampler's history ring, the Adams-Bashforth combination e' of up to four eps and the DDIM update on e', in one pass.
// e_store / h1..h3 / x / x_prev carry no __restrict__: the header allows e_store == h3 and x_prev == x, and each thread
// reads every input element before it stores its own.  Torch on CUDA evaluates `t / k` with a CPU-scalar k as
// t * fl(1 / k) (ATen div_true_kernel_cuda), so the divisors 2, 12 and 24 are applied as products with those reciprocals.
// ---------------------------------------------------------------------------------------------------------
template <int NP>
__global__ void plms_update_kernel(const float* x, const float* __restrict__ eps, int cfg, float cfg_scale, float* e_store,
                                   int mode, const float* h1, const float* h2, const float* h3, float s1m, float sqrt_at,
                                   float sqrt_ap, float dirc, PeerPtrs out, float* pred_x0, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float e = eps[i];
    if (cfg) e = __fadd_rn(e, __fmul_rn(cfg_scale, __fsub_rn(eps[n + i], e)));  // e_u + s * (e_c - e_u)   plms.py get_model_output
    float ep = e;
    if (mode == 1) {  // pseudo improved Euler: (e_t + e_next) / 2, e_t from the history
      ep = __fmul_rn(__fadd_rn(h1[i], e), 0.5f);
    } else if (mode == 2) {  // (3 e_t - o[-1]) / 2
      ep = __fmul_rn(__fsub_rn(__fmul_rn(3.0f, e), h1[i]), 0.5f);
    } else if (mode == 3) {  // (23 e_t - 16 o[-1] + 5 o[-2]) / 12
      ep = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(23.0f, e), __fmul_rn(16.0f, h1[i])), __fmul_rn(5.0f, h2[i])), 1.0f / 12.0f);
    } else if (mode == 4) {  // (55 e_t - 59 o[-1] + 37 o[-2] - 9 o[-3]) / 24
      float s = __fsub_rn(__fmul_rn(55.0f, e), __fmul_rn(59.0f, h1[i]));
      s = __fsub_rn(__fadd_rn(s, __fmul_rn(37.0f, h2[i])), __fmul_rn(9.0f, h3[i]));
      ep = __fmul_rn(s, 1.0f / 24.0f);
    }
    float p0 = __fdiv_rn(__fsub_rn(x[i], __fmul_rn(s1m, ep)), sqrt_at);  // get_x_prev_and_pred_x0 (= cddim.py:63,74,78)
    float xp = __fadd_rn(__fmul_rn(sqrt_ap, p0), __fmul_rn(dirc, ep));
    if (e_store) e_store[i] = e;
    if (pred_x0) pred_x0[i] = p0;
#pragma unroll
    for (int r = 0; r < NP; ++r) out.p[r][i] = xp;
  }
}

static int plms_launch(const float* x, const float* eps, int cfg, float cfg_scale, float* e_store, int mode, const float* h1,
                       const float* h2, const float* h3, float s1m, float sqrt_at, float sqrt_ap, float dirc,
                       const PeerPtrs& pp, int n_peers, float* pred_x0, int64_t n, mkd_stream_t stream, const char* who) {
  MKD_REQUIRE(x && eps && n >= 0, MKD_E_INVALID, "%s: null pointer or negative n", who);
  MKD_REQUIRE(mode >= 0 && mode <= 4, MKD_E_INVALID, "%s: mode=%d must be 0..4", who, mode);
  MKD_REQUIRE((mode < 1 || h1) && (mode < 3 || h2) && (mode < 4 || h3), MKD_E_INVALID,
              "%s: mode %d needs %d history pointer(s)", who, mode, mode <= 2 ? 1 : mode - 1);
  for (int r = 0; r < n_peers; ++r) MKD_REQUIRE(pp.p[r] != nullptr, MKD_E_INVALID, "%s: null x_prev pointer %d", who, r);
  if (n == 0) return MKD_OK;
  int threads = 256;
  int blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t st = (cudaStream_t)stream;
#define MKD_PLMS_CASE(NP)                                                                                               \
  case NP:                                                                                                              \
    MKD_LAUNCH_OK(launch_pdl(plms_update_kernel<NP>, dim3(blocks), dim3(threads), 0, st, x, eps, cfg, cfg_scale, e_store, \
                             mode, h1, h2, h3, s1m, sqrt_at, sqrt_ap, dirc, pp, pred_x0, n));                           \
    break;
  switch (n_peers) {
    MKD_PLMS_CASE(1) MKD_PLMS_CASE(2) MKD_PLMS_CASE(3) MKD_PLMS_CASE(4)
    MKD_PLMS_CASE(5) MKD_PLMS_CASE(6) MKD_PLMS_CASE(7) MKD_PLMS_CASE(8)
  }
#undef MKD_PLMS_CASE
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

extern "C" int mkd_plms_update(const float* x, const float* eps, int cfg, float cfg_scale, float* e_store, int mode,
                               const float* h1, const float* h2, const float* h3, float sqrt_one_minus_at, float sqrt_at,
                               float sqrt_a_prev, float dir_coef, float* x_prev, float* pred_x0, int64_t n,
                               mkd_stream_t stream) {
  PeerPtrs pp = {};
  pp.p[0] = x_prev;
  return plms_launch(x, eps, cfg, cfg_scale, e_store, mode, h1, h2, h3, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef,
                     pp, 1, pred_x0, n, stream, "plms_update");
}

extern "C" int mkd_plms_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, float* e_store, int mode,
                                     const float* h1, const float* h2, const float* h3, float sqrt_one_minus_at,
                                     float sqrt_at, float sqrt_a_prev, float dir_coef, float* const* x_prev_peers,
                                     int n_peers, float* pred_x0, int64_t n, mkd_stream_t stream) {
  MKD_REQUIRE(x_prev_peers, MKD_E_INVALID, "plms_update_peers: null peer array");
  MKD_REQUIRE(n_peers >= 1 && n_peers <= 8, MKD_E_INVALID, "plms_update_peers: n_peers=%d must be 1..8 (one box)", n_peers);
  PeerPtrs pp = {};
  for (int r = 0; r < n_peers; ++r) pp.p[r] = x_prev_peers[r];  // host array of device pointers
  return plms_launch(x, eps, cfg, cfg_scale, e_store, mode, h1, h2, h3, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef,
                     pp, n_peers, pred_x0, n, stream, "plms_update_peers");
}

// ---------------------------------------------------------------------------------------------------------
// DPM-Solver++ multistep update (upstream dpm_solver.py, predict_x0=True, solver_type 'dpm_solver'): the CFG combine,
// the data prediction m_k at the evaluated time, its store into the sampler's two-slot ring and the order-1 or order-2
// step to the next time, in one pass.  x / x_prev carry no __restrict__ (the header allows x_prev == x); each thread reads
// every input element before it stores its own.  The data prediction is a true division by alpha_s, as upstream's
// tensor / tensor; every other scalar arrives precomputed from upstream's torch expressions.
// ---------------------------------------------------------------------------------------------------------
template <int NP>
__global__ void dpm_update_kernel(const float* x, const float* __restrict__ eps, int cfg, float cfg_scale, float alpha_s,
                                  float sigma_s, float* __restrict__ m_store, int order, const float* __restrict__ m_prev,
                                  float ratio, float phi, float half_phi, float inv_r0, PeerPtrs out, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float e = eps[i];
    if (cfg) e = __fadd_rn(e, __fmul_rn(cfg_scale, __fsub_rn(eps[n + i], e)));  // noise_uncond + s * (noise - noise_uncond)
    float xv = x[i];
    float m = __fdiv_rn(__fsub_rn(xv, __fmul_rn(sigma_s, e)), alpha_s);  // data_prediction_fn
    float xp = __fsub_rn(__fmul_rn(ratio, xv), __fmul_rn(phi, m));       // (sigma_t / sigma_s) x - (alpha_t phi) m_k
    if (order == 2) {
      float d = __fmul_rn(inv_r0, __fsub_rn(m, m_prev[i]));            // D1_0 = (1 / r0) (m_k - m_{k-1})
      xp = __fsub_rn(xp, __fmul_rn(half_phi, d));                      //   - (0.5 alpha_t phi) D1_0
    }
    if (m_store) m_store[i] = m;
#pragma unroll
    for (int r = 0; r < NP; ++r) out.p[r][i] = xp;
  }
}

static int dpm_launch(const float* x, const float* eps, int cfg, float cfg_scale, float alpha_s, float sigma_s,
                      float* m_store, int order, const float* m_prev, float ratio, float phi, float half_phi, float inv_r0,
                      const PeerPtrs& pp, int n_peers, int64_t n, mkd_stream_t stream, const char* who) {
  MKD_REQUIRE(x && eps && n >= 0, MKD_E_INVALID, "%s: null pointer or negative n", who);
  MKD_REQUIRE(order == 1 || order == 2, MKD_E_INVALID, "%s: order=%d must be 1 or 2", who, order);
  MKD_REQUIRE(order == 1 || m_prev, MKD_E_INVALID, "%s: order 2 needs m_prev", who);
  for (int r = 0; r < n_peers; ++r) MKD_REQUIRE(pp.p[r] != nullptr, MKD_E_INVALID, "%s: null x_prev pointer %d", who, r);
  if (n == 0) return MKD_OK;
  int threads = 256;
  int blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t st = (cudaStream_t)stream;
#define MKD_DPM_CASE(NP)                                                                                                \
  case NP:                                                                                                              \
    MKD_LAUNCH_OK(launch_pdl(dpm_update_kernel<NP>, dim3(blocks), dim3(threads), 0, st, x, eps, cfg, cfg_scale, alpha_s, \
                             sigma_s, m_store, order, m_prev, ratio, phi, half_phi, inv_r0, pp, n));                    \
    break;
  switch (n_peers) {
    MKD_DPM_CASE(1) MKD_DPM_CASE(2) MKD_DPM_CASE(3) MKD_DPM_CASE(4)
    MKD_DPM_CASE(5) MKD_DPM_CASE(6) MKD_DPM_CASE(7) MKD_DPM_CASE(8)
  }
#undef MKD_DPM_CASE
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

extern "C" int mkd_dpm_update(const float* x, const float* eps, int cfg, float cfg_scale, float alpha_s, float sigma_s,
                              float* m_store, int order, const float* m_prev, float sigma_ratio, float phi, float half_phi,
                              float inv_r0, float* x_prev, int64_t n, mkd_stream_t stream) {
  PeerPtrs pp = {};
  pp.p[0] = x_prev;
  return dpm_launch(x, eps, cfg, cfg_scale, alpha_s, sigma_s, m_store, order, m_prev, sigma_ratio, phi, half_phi, inv_r0,
                    pp, 1, n, stream, "dpm_update");
}

extern "C" int mkd_dpm_update_peers(const float* x, const float* eps, int cfg, float cfg_scale, float alpha_s,
                                    float sigma_s, float* m_store, int order, const float* m_prev, float sigma_ratio,
                                    float phi, float half_phi, float inv_r0, float* const* x_prev_peers, int n_peers,
                                    int64_t n, mkd_stream_t stream) {
  MKD_REQUIRE(x_prev_peers, MKD_E_INVALID, "dpm_update_peers: null peer array");
  MKD_REQUIRE(n_peers >= 1 && n_peers <= 8, MKD_E_INVALID, "dpm_update_peers: n_peers=%d must be 1..8 (one box)", n_peers);
  PeerPtrs pp = {};
  for (int r = 0; r < n_peers; ++r) pp.p[r] = x_prev_peers[r];  // host array of device pointers
  return dpm_launch(x, eps, cfg, cfg_scale, alpha_s, sigma_s, m_store, order, m_prev, sigma_ratio, phi, half_phi, inv_r0,
                    pp, n_peers, n, stream, "dpm_update_peers");
}

// ---------------------------------------------------------------------------------------------------------
// DDPM ancestral step (upstream ddpm.py p_sample after its model call): predict_start_from_noise, the optional clamp,
// q_posterior's mean and the noise term, in one pass.  Every row reads its own timestep from the device vector t and
// its five coefficients from fp32 device tables indexed by it, so the launch is graph-capturable and rows may carry
// different t.  x / x_prev carry no __restrict__ (the header allows x_prev == x); each thread reads every input element
// before it stores its own.  A t outside [0, T) yields NaN for that row rather than an out-of-bounds read.
// ---------------------------------------------------------------------------------------------------------
struct DdpmTables {
  const float* sqrt_recip_ac;
  const float* sqrt_recipm1_ac;
  const float* coef1;
  const float* coef2;
  const float* sigma;
};

template <int NP>
__global__ void ddpm_update_kernel(const float* x, const float* __restrict__ eps, const int64_t* __restrict__ t,
                                   int64_t per_row, DdpmTables tb, int T, int clip, const float* __restrict__ noise,
                                   float temp, float* __restrict__ x0_out, PeerPtrs out, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t tr = t[i / per_row];
    const float xv = x[i], e = eps[i], nz = noise[i];
    float xr = __int_as_float(0x7fffffff), xp = xr;
    if (tr >= 0 && tr < T) {
      xr = __fsub_rn(__fmul_rn(tb.sqrt_recip_ac[tr], xv), __fmul_rn(tb.sqrt_recipm1_ac[tr], e));  // x_recon
      if (clip) xr = xr < -1.f ? -1.f : (xr > 1.f ? 1.f : xr);                                    // clamp_(-1, 1), NaN kept
      const float mean = __fadd_rn(__fmul_rn(tb.coef1[tr], xr), __fmul_rn(tb.coef2[tr], xv));     // q_posterior mean
      const float s = tr == 0 ? 0.f : tb.sigma[tr];  // nonzero_mask * exp(0.5 * log_variance): the mask is exact
      xp = __fadd_rn(mean, __fmul_rn(s, __fmul_rn(nz, temp)));  // mean + (mask * sigma) * (noise * temperature)
    }
    if (x0_out) x0_out[i] = xr;
#pragma unroll
    for (int r = 0; r < NP; ++r) out.p[r][i] = xp;
  }
}

static int ddpm_launch(const float* x, const float* eps, const int64_t* t, int B, const DdpmTables& tb, int T, int clip,
                       const float* noise, float temperature, float* x0_out, const PeerPtrs& pp, int n_peers, int64_t n,
                       mkd_stream_t stream, const char* who) {
  MKD_REQUIRE(x && eps && t && noise && n >= 0, MKD_E_INVALID, "%s: null pointer or negative n", who);
  MKD_REQUIRE(tb.sqrt_recip_ac && tb.sqrt_recipm1_ac && tb.coef1 && tb.coef2 && tb.sigma && T > 0, MKD_E_INVALID,
              "%s: null table or T=%d", who, T);
  MKD_REQUIRE(B >= 1 && n % B == 0, MKD_E_INVALID, "%s: n=%lld is not B=%d rows of equal size", who, (long long)n, B);
  for (int r = 0; r < n_peers; ++r) MKD_REQUIRE(pp.p[r] != nullptr, MKD_E_INVALID, "%s: null x_prev pointer %d", who, r);
  if (n == 0) return MKD_OK;
  int threads = 256;
  int blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t per_row = n / B;
#define MKD_DDPM_CASE(NP)                                                                                              \
  case NP:                                                                                                             \
    MKD_LAUNCH_OK(launch_pdl(ddpm_update_kernel<NP>, dim3(blocks), dim3(threads), 0, st, x, eps, t, per_row, tb, T,  \
                             clip, noise, temperature, x0_out, pp, n));                                               \
    break;
  switch (n_peers) {
    MKD_DDPM_CASE(1) MKD_DDPM_CASE(2) MKD_DDPM_CASE(3) MKD_DDPM_CASE(4)
    MKD_DDPM_CASE(5) MKD_DDPM_CASE(6) MKD_DDPM_CASE(7) MKD_DDPM_CASE(8)
  }
#undef MKD_DDPM_CASE
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

extern "C" int mkd_ddpm_update(const float* x, const float* eps, const int64_t* t, int B, const float* sqrt_recip_ac,
                               const float* sqrt_recipm1_ac, const float* coef1, const float* coef2, const float* sigma,
                               int T, int clip, const float* noise, float temperature, float* x0_out, float* x_prev,
                               int64_t n, mkd_stream_t stream) {
  PeerPtrs pp = {};
  pp.p[0] = x_prev;
  DdpmTables tb = {sqrt_recip_ac, sqrt_recipm1_ac, coef1, coef2, sigma};
  return ddpm_launch(x, eps, t, B, tb, T, clip, noise, temperature, x0_out, pp, 1, n, stream, "ddpm_update");
}

extern "C" int mkd_ddpm_update_peers(const float* x, const float* eps, const int64_t* t, int B,
                                     const float* sqrt_recip_ac, const float* sqrt_recipm1_ac, const float* coef1,
                                     const float* coef2, const float* sigma, int T, int clip, const float* noise,
                                     float temperature, float* x0_out, float* const* x_prev_peers, int n_peers,
                                     int64_t n, mkd_stream_t stream) {
  MKD_REQUIRE(x_prev_peers, MKD_E_INVALID, "ddpm_update_peers: null peer array");
  MKD_REQUIRE(n_peers >= 1 && n_peers <= 8, MKD_E_INVALID, "ddpm_update_peers: n_peers=%d must be 1..8 (one box)",
              n_peers);
  PeerPtrs pp = {};
  for (int r = 0; r < n_peers; ++r) pp.p[r] = x_prev_peers[r];  // host array of device pointers
  DdpmTables tb = {sqrt_recip_ac, sqrt_recipm1_ac, coef1, coef2, sigma};
  return ddpm_launch(x, eps, t, B, tb, T, clip, noise, temperature, x0_out, pp, n_peers, n, stream,
                     "ddpm_update_peers");
}

// ---------------------------------------------------------------------------------------------------------
// NCHW fp32 <-> NHWC T through a 32x32 smem transpose tile (coalesced on both sides).
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, T* __restrict__ dst, int C, int HW, int ld) {
  pdl_wait();
  __shared__ float tile[32][33];
  int n = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int c = c0 + j, p = p0 + threadIdx.x;
    tile[j][threadIdx.x] = (c < C && p < HW) ? src[((int64_t)n * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int p = p0 + j, c = c0 + threadIdx.x;
    if (p < HW && c < C) dst[((int64_t)n * HW + p) * ld + c] = from_f<T>(tile[threadIdx.x][j]);
  }
}
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ src, float* __restrict__ dst, int C, int HW, int ld) {
  pdl_wait();
  __shared__ float tile[32][33];
  int n = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int p = p0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (p < HW && c < C) ? to_f(src[((int64_t)n * HW + p) * ld + c]) : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int c = c0 + j, p = p0 + threadIdx.x;
    if (c < C && p < HW) dst[((int64_t)n * C + c) * HW + p] = tile[threadIdx.x][j];
  }
}

extern "C" int mkd_nchw_to_nhwc(const float* src, void* dst, int dtype, int N, int C, int H, int W, int ld_dst,
                                mkd_stream_t stream) {
  MKD_REQUIRE(src && dst && N > 0 && C > 0 && H > 0 && W > 0 && ld_dst >= C, MKD_E_INVALID, "nchw_to_nhwc: bad args");
  MKD_REQUIRE(N <= 65535, MKD_E_INVALID, "nchw_to_nhwc: N too large");
  dim3 grid((H * W + 31) / 32, (C + 31) / 32, N), block(32, 8);
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(nchw_to_nhwc_kernel<bf16>, dim3(grid), dim3(block), 0, (cudaStream_t)stream, src, (bf16*)dst, C, H * W, ld_dst));
  else
    MKD_LAUNCH_OK(launch_pdl(nchw_to_nhwc_kernel<float>, dim3(grid), dim3(block), 0, (cudaStream_t)stream, src, (float*)dst, C, H * W, ld_dst));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}
extern "C" int mkd_nhwc_to_nchw(const void* src, float* dst, int dtype, int N, int C, int H, int W, int ld_src,
                                mkd_stream_t stream) {
  MKD_REQUIRE(src && dst && N > 0 && C > 0 && H > 0 && W > 0 && ld_src >= C, MKD_E_INVALID, "nhwc_to_nchw: bad args");
  MKD_REQUIRE(N <= 65535, MKD_E_INVALID, "nhwc_to_nchw: N too large");
  dim3 grid((H * W + 31) / 32, (C + 31) / 32, N), block(32, 8);
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(nhwc_to_nchw_kernel<bf16>, dim3(grid), dim3(block), 0, (cudaStream_t)stream, (const bf16*)src, dst, C, H * W, ld_src));
  else
    MKD_LAUNCH_OK(launch_pdl(nhwc_to_nchw_kernel<float>, dim3(grid), dim3(block), 0, (cudaStream_t)stream, (const float*)src, dst, C, H * W, ld_src));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void timestep_embedding_kernel(const int64_t* __restrict__ t, T* __restrict__ out, int B, int dim,
                                          float neg_log_mp) {
  pdl_wait();
  int half = dim / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * half; i += gridDim.x * blockDim.x) {
    int b = i / half, k = i % half;
    float f = expf(neg_log_mp * (float)k / (float)half);
    float a = (float)t[b] * f;
    out[(int64_t)b * dim + k] = from_f<T>(cosf(a));
    out[(int64_t)b * dim + half + k] = from_f<T>(sinf(a));
    if ((dim & 1) && k == 0) out[(int64_t)b * dim + dim - 1] = from_f<T>(0.f);
  }
}
extern "C" int mkd_timestep_embedding(const int64_t* t, void* out, int dtype, int B, int dim, float max_period,
                                      mkd_stream_t stream) {
  MKD_REQUIRE(t && out && B > 0 && dim >= 2, MKD_E_INVALID, "timestep_embedding: bad args");
  int n = B * (dim / 2), threads = 128, blocks = (n + threads - 1) / threads;
  float nl = -logf(max_period);
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(timestep_embedding_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, t, (bf16*)out, B, dim, nl));
  else
    MKD_LAUNCH_OK(launch_pdl(timestep_embedding_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, t, (float*)out, B, dim, nl));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// fp32 timesteps (DPM-Solver's fractional model times): upstream's t.float() * freqs with t as given.  The body is the
// int64 kernel's with (float)t[b] already a float, so integer t below 2^24 give the same bits.
template <typename T>
__global__ void timestep_embedding_f32_kernel(const float* __restrict__ t, T* __restrict__ out, int B, int dim,
                                              float neg_log_mp) {
  pdl_wait();
  int half = dim / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * half; i += gridDim.x * blockDim.x) {
    int b = i / half, k = i % half;
    float f = expf(neg_log_mp * (float)k / (float)half);
    float a = t[b] * f;
    out[(int64_t)b * dim + k] = from_f<T>(cosf(a));
    out[(int64_t)b * dim + half + k] = from_f<T>(sinf(a));
    if ((dim & 1) && k == 0) out[(int64_t)b * dim + dim - 1] = from_f<T>(0.f);
  }
}
extern "C" int mkd_timestep_embedding_f32(const float* t, void* out, int dtype, int B, int dim, float max_period,
                                          mkd_stream_t stream) {
  MKD_REQUIRE(t && out && B > 0 && dim >= 2, MKD_E_INVALID, "timestep_embedding_f32: bad args");
  int n = B * (dim / 2), threads = 128, blocks = (n + threads - 1) / threads;
  float nl = -logf(max_period);
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(timestep_embedding_f32_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, t, (bf16*)out, B, dim, nl));
  else
    MKD_LAUNCH_OK(launch_pdl(timestep_embedding_f32_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, t, (float*)out, B, dim, nl));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void silu_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = from_f<T>(silu_f(to_f(x[i])));
}
extern "C" int mkd_silu(const void* x, void* y, int dtype, int64_t n, mkd_stream_t stream) {
  MKD_REQUIRE(x && y && n >= 0, MKD_E_INVALID, "silu: bad args");
  if (n == 0) return MKD_OK;
  int threads = 256, blocks = (int)((n + threads - 1) / threads);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(silu_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const bf16*)x, (bf16*)y, n));
  else
    MKD_LAUNCH_OK(launch_pdl(silu_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const float*)x, (float*)y, n));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// GEGLU, 8 channels per thread (16-byte bf16 vectors).
template <typename T>
__global__ void geglu_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t M, int inner, int ldx, int ldy) {
  pdl_wait();
  int vpr = inner / 8;
  int64_t total = M * vpr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t m = i / vpr;
    int c = (int)(i % vpr) * 8;
    float a[8], g[8];
    load8(x + m * ldx + c, a);
    load8(x + m * ldx + inner + c, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] *= gelu_erf_f(g[j]);
    store8(y + m * ldy + c, a);
  }
}
extern "C" int mkd_geglu(const void* x, void* y, int dtype, int64_t M, int inner, int ldx, int ldy,
                         mkd_stream_t stream) {
  MKD_REQUIRE(x && y && M > 0 && inner > 0, MKD_E_INVALID, "geglu: bad args");
  MKD_REQUIRE(inner % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && aligned16(x) && aligned16(y), MKD_E_ALIGN,
              "geglu: inner/ld must be multiples of 8 and pointers 16B aligned");
  int64_t total = M * (inner / 8);
  int threads = 256, blocks = (int)((total + threads - 1) / threads);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(geglu_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const bf16*)x, (bf16*)y, M, inner, ldx, ldy));
  else
    MKD_LAUNCH_OK(launch_pdl(geglu_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const float*)x, (float*)y, M, inner, ldx, ldy));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

template <typename T>
__global__ void add_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ y, int64_t M, int C,
                           int lda, int ldb, int ldy) {
  pdl_wait();
  int vpr = C / 8;
  int64_t total = M * vpr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t m = i / vpr;
    int c = (int)(i % vpr) * 8;
    float u[8], v[8];
    load8(a + m * lda + c, u);
    load8(b + m * ldb + c, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) u[j] += v[j];
    store8(y + m * ldy + c, u);
  }
}
extern "C" int mkd_add(const void* a, const void* b, void* y, int dtype, int64_t M, int C, int lda, int ldb, int ldy,
                       mkd_stream_t stream) {
  MKD_REQUIRE(a && b && y && M > 0 && C > 0, MKD_E_INVALID, "add: bad args");
  MKD_REQUIRE(C % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldy % 8 == 0 && aligned16(a) && aligned16(b) && aligned16(y),
              MKD_E_ALIGN, "add: C/ld must be multiples of 8 and pointers 16B aligned");
  int64_t total = M * (C / 8);
  int threads = 256, blocks = (int)((total + threads - 1) / threads);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (dtype == MKD_BF16)
    MKD_LAUNCH_OK(launch_pdl(add_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const bf16*)a, (const bf16*)b, (bf16*)y, M, C, lda, ldb, ldy));
  else
    MKD_LAUNCH_OK(launch_pdl(add_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, (const float*)a, (const float*)b, (float*)y, M, C, lda, ldb, ldy));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// ---- token + position embedding of the CLIP text encoder (once per prompt) ------------------------------------------
// out[b * T + t, :] = tok_emb[ids[b * T + t], :] + pos_emb[t, :]   (fp32 tables, fp32 out; C % 4 == 0)
namespace {
__global__ void embed_tokens_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tok, const float* __restrict__ pos,
                                    float* __restrict__ out, int rows, int T, int C, int vocab, int ld_out) {
  pdl_wait();
  const int vpr = C / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)rows * vpr; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / vpr), c = (int)(i % vpr) * 4;
    int64_t id = ids[r];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);  // (the host wrapper rejects out-of-range ids; never read out of bounds)
    const float4 a = *reinterpret_cast<const float4*>(tok + id * C + c);
    const float4 b = *reinterpret_cast<const float4*>(pos + (int64_t)(r % T) * C + c);
    *reinterpret_cast<float4*>(out + (int64_t)r * ld_out + c) = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}
}  // namespace

extern "C" int mkd_embed_tokens(const int64_t* ids, const float* tok_emb, const float* pos_emb, float* out, int B, int T,
                                int C, int vocab, int ld_out, mkd_stream_t stream) {
  MKD_REQUIRE(ids && tok_emb && pos_emb && out && B > 0 && T > 0 && C > 0 && vocab > 0, MKD_E_INVALID, "embed_tokens: bad args");
  MKD_REQUIRE(C % 4 == 0 && ld_out % 4 == 0 && ld_out >= C && aligned16(tok_emb) && aligned16(pos_emb) && aligned16(out), MKD_E_ALIGN,
              "embed_tokens: C / ld_out must be multiples of 4, pointers 16B aligned");
  const int64_t n = (int64_t)B * T * (C / 4);
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  MKD_LAUNCH_OK(launch_pdl(embed_tokens_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, ids, tok_emb, pos_emb, out, B * T, T, C,
                           vocab, ld_out));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}

// ---- test-harness output (SURVEY.md 8(f) rank 4): diffusion_makeup.py:344-358 `save_local` -------------------------
// torchvision.utils.make_grid(images, nrow, padding = 2, pad_value = 0) -> optional clamp to [-1, 1] (test_step,
// :340-341) -> (x + 1) / 2 -> CHW to HWC -> (x * 255).astype(uint8) (truncation), as ONE pass writing the uint8 grid the
// PNG encoder takes: the device -> host copy shrinks 4x and no fp32 grid exists.  The fp32 operations are the
// reference's, in its order, so the bytes are identical.  C == 1 images are replicated to 3 channels like make_grid.
namespace {
__global__ void image_grid_u8_kernel(const float* __restrict__ src, unsigned char* __restrict__ dst, int N, int C, int H, int W,
                                     int xmaps, int pad, int GH, int GW, int clamp, int rescale) {
  pdl_wait();
  const int64_t total = (int64_t)GH * GW * 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % 3), gx = (int)((i / 3) % GW), gy = (int)(i / (3 * (int64_t)GW));
    const int cy = gy / (H + pad), cx = gx / (W + pad);
    const int y = gy - cy * (H + pad) - pad, x = gx - cx * (W + pad) - pad;
    const int k = cy * xmaps + cx;
    float v = 0.f;  // pad_value
    if (y >= 0 && x >= 0 && cx < xmaps && k < N && y < H && x < W) {
      v = src[(((int64_t)k * C + (C == 1 ? 0 : c)) * H + y) * W + x];
      if (clamp) v = fminf(fmaxf(v, -1.0f), 1.0f);
    }
    if (rescale) v = (v + 1.0f) / 2.0f;
    v = v * 255.0f;
    // numpy's float32 -> uint8 cast of in-range values truncates toward zero; out-of-range input (no clamp) wraps
    // through int on the reference's platform, which this mirrors for the representable range
    dst[i] = (unsigned char)(int)v;
  }
}
}  // namespace

extern "C" int mkd_image_grid_u8(const float* images, unsigned char* grid, int N, int C, int H, int W, int nrow, int padding,
                                 int clamp, int rescale, mkd_stream_t stream) {
  MKD_REQUIRE(images && grid && N > 0 && (C == 1 || C == 3) && H > 0 && W > 0 && nrow > 0 && padding >= 0, MKD_E_INVALID,
              "image_grid_u8: bad args (C must be 1 or 3)");
  if (N == 1) padding = 0;  // make_grid returns a single image as it is, without the padding frame
  const int xmaps = nrow < N ? nrow : N, ymaps = (N + xmaps - 1) / xmaps;
  const int GH = (H + padding) * ymaps + padding, GW = (W + padding) * xmaps + padding;
  const int64_t total = (int64_t)GH * GW * 3;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  MKD_LAUNCH_OK(launch_pdl(image_grid_u8_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, images, grid, N, C, H, W, xmaps, padding,
                           GH, GW, clamp, rescale));
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}
