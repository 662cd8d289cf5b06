// Generic implicit-GEMM convolution (CUDA cores, fp32 accumulate).  It serves
//   (1) the fp32 check mode (dtype == MKD_F32) — the whole network at 1e-4 against the oracle,
//   (2) shapes the tcgen05 kernel does not take: C or K not tileable (conv_in 4->320, out 320->4, the hint block's
//       6/16/32/96-channel layers), stride-2 / upsampling convs, tiny-M linears (timestep MLP, emb_layers).
// The hot shapes of the bf16 path go to gemm_tcgen05.cu; mkd_conv2d_path() reports which kernel a descriptor gets.
//
// Tiling: 64 output pixels x 64 output channels per CTA, K chunks of 16, 256 threads x (4x4) micro-tiles.
#include "common.cuh"
using namespace mkd;

namespace {
constexpr int BM = 64, BN = 64, BK = 16;

struct ConvP {
  int N, H, W, C, K, R, S, stride, pad, up;
  int P, Q;      // output spatial
  int Hin, Win;  // logical (post-upsample) input spatial
  int ldx, ldy, ldr, lde;
  int Ktot;      // R*S*C
  int M;         // N*P*Q
  int Kout;      // stored output channels (K or K/2 for GEGLU)
  int gb;        // geglu block
  int act;
  float alpha;
  int res_f32, ldy32;
  float* y32;
};

template <typename T, bool GEGLU>
__global__ void __launch_bounds__(256) conv_generic_kernel(ConvP p, const T* __restrict__ x, const T* __restrict__ w,
                                                           T* __restrict__ y, const float* __restrict__ bias,
                                                           const T* __restrict__ emb, const void* __restrict__ res) {
  pdl_wait();
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[GEGLU ? 2 : 1][BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;

  // A loader: row lr, 4 consecutive k starting at lk
  const int lr = tid / 4, lk = (tid % 4) * 4;
  const int m = m0 + lr;
  const bool mvalid = m < p.M;
  int pn = 0, pp = 0, pq = 0;
  if (mvalid) {
    pn = m / (p.P * p.Q);
    int rem = m % (p.P * p.Q);
    pp = rem / p.Q;
    pq = rem % p.Q;
  }
  // B loader: weight row(s) for tile column lr
  const int oc = n0 + lr;  // output channel (stored index)
  int wrow0 = oc, wrow1 = 0;
  if (GEGLU) {
    wrow0 = (oc / p.gb) * 2 * p.gb + oc % p.gb;
    wrow1 = wrow0 + p.gb;
  }
  const bool nvalid = oc < p.Kout;

  float acc[GEGLU ? 2 : 1][4][4];
#pragma unroll
  for (int g = 0; g < (GEGLU ? 2 : 1); ++g)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[g][i][j] = 0.f;

  for (int k0 = 0; k0 < p.Ktot; k0 += BK) {
    // ---- stage A (im2col gather) ----
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int k = k0 + lk + j;
      float v = 0.f;
      if (mvalid && k < p.Ktot) {
        int tap = k / p.C, c = k - tap * p.C;
        int r = tap / p.S, s = tap - r * p.S;
        int ih = pp * p.stride - p.pad + r, iw = pq * p.stride - p.pad + s;
        if (ih >= 0 && ih < p.Hin && iw >= 0 && iw < p.Win) {
          if (p.up) {
            ih >>= 1;
            iw >>= 1;
          }
          v = to_f(x[((int64_t)(pn * p.H + ih) * p.W + iw) * p.ldx + c]);
        }
      }
      As[lk + j][lr] = v;
    }
    // ---- stage B (weights) ----
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int k = k0 + lk + j;
      bool ok = nvalid && k < p.Ktot;
      Bs[0][lk + j][lr] = ok ? to_f(w[(int64_t)wrow0 * p.Ktot + k]) : 0.f;
      if (GEGLU) Bs[1][lk + j][lr] = ok ? to_f(w[(int64_t)wrow1 * p.Ktot + k]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[4], b[4];
      *reinterpret_cast<float4*>(a) = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(&Bs[0][kk][tx * 4]);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[0][i][j] = fmaf(a[i], b[j], acc[0][i][j]);
      if (GEGLU) {
        *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(&Bs[1][kk][tx * 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[GEGLU ? 1 : 0][i][j] = fmaf(a[i], b[j], acc[GEGLU ? 1 : 0][i][j]);
      }
    }
    __syncthreads();
  }

  // ---- epilogue ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int mm = m0 + ty * 4 + i;
    if (mm >= p.M) continue;
    int nimg = mm / (p.P * p.Q);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int o = n0 + tx * 4 + j;
      if (o >= p.Kout) continue;
      float v;
      if (GEGLU) {
        int r0 = (o / p.gb) * 2 * p.gb + o % p.gb, r1 = r0 + p.gb;
        float a = acc[0][i][j] + (bias ? bias[r0] : 0.f);
        float g = acc[GEGLU ? 1 : 0][i][j] + (bias ? bias[r1] : 0.f);
        v = a * gelu_erf_f(g);
      } else {
        v = acc[0][i][j];
        if (bias) v += bias[o];
        if (emb) v += to_f(emb[(int64_t)nimg * p.lde + o]);
        v *= p.alpha;
        if (res)
          v += p.res_f32 ? static_cast<const float*>(res)[(int64_t)mm * p.ldr + o]
                         : to_f(static_cast<const T*>(res)[(int64_t)mm * p.ldr + o]);
        if (p.act == MKD_ACT_SILU) v = silu_f(v);
      }
      if (p.y32) p.y32[(int64_t)mm * p.ldy32 + o] = v;
      if (y) y[(int64_t)mm * p.ldy + o] = from_f<T>(v);
    }
  }
}
}  // namespace

namespace mkd {
int conv2d_generic(const mkd_conv_desc* d, cudaStream_t stream) {
  MKD_REQUIRE(d->stats == nullptr, MKD_E_INVALID, "conv2d: fused GroupNorm statistics need the tcgen05 path (%s)", mkd_last_error());
  ConvP p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.C = d->C; p.K = d->K; p.R = d->R; p.S = d->S;
  p.stride = d->stride; p.pad = d->pad; p.up = d->upsample ? 1 : 0;
  p.Hin = p.up ? 2 * d->H : d->H;
  p.Win = p.up ? 2 * d->W : d->W;
  p.P = (p.Hin + 2 * p.pad + d->pad_hi_extra - p.R) / p.stride + 1;  // (the kernel bounds-checks every tap)
  p.Q = (p.Win + 2 * p.pad + d->pad_hi_extra - p.S) / p.stride + 1;
  p.ldx = d->ldx; p.ldy = d->ldy; p.ldr = d->ldr; p.lde = d->lde;
  p.Ktot = p.R * p.S * p.C;
  p.M = p.N * p.P * p.Q;
  p.act = d->act;
  p.gb = d->geglu_block > 0 ? d->geglu_block : 1;
  p.Kout = d->act == MKD_ACT_GEGLU ? d->K / 2 : d->K;
  p.alpha = d->alpha;
  p.res_f32 = d->residual_dtype == MKD_F32 ? 1 : 0;
  p.y32 = d->y32;
  p.ldy32 = d->ldy32;
  dim3 grid((p.M + BM - 1) / BM, (p.Kout + BN - 1) / BN);
  MKD_REQUIRE(grid.y <= 65535, MKD_E_INVALID, "conv2d: K too large");
  const bool geglu = d->act == MKD_ACT_GEGLU;
  if (d->dtype == MKD_BF16) {
    if (geglu)
      MKD_LAUNCH_OK(launch_pdl(conv_generic_kernel<bf16, true>, dim3(grid), dim3(256), 0, stream, p, (const bf16*)d->x, (const bf16*)d->w, (bf16*)d->y,
                                                                d->bias, (const bf16*)d->emb, d->residual));
    else
      MKD_LAUNCH_OK(launch_pdl(conv_generic_kernel<bf16, false>, dim3(grid), dim3(256), 0, stream, p, (const bf16*)d->x, (const bf16*)d->w, (bf16*)d->y,
                                                                 d->bias, (const bf16*)d->emb, d->residual));
  } else {
    if (geglu)
      MKD_LAUNCH_OK(launch_pdl(conv_generic_kernel<float, true>, dim3(grid), dim3(256), 0, stream, p, (const float*)d->x, (const float*)d->w,
                                                                 (float*)d->y, d->bias, (const float*)d->emb,
                                                                 d->residual));
    else
      MKD_LAUNCH_OK(launch_pdl(conv_generic_kernel<float, false>, dim3(grid), dim3(256), 0, stream, p, (const float*)d->x, (const float*)d->w,
                                                                  (float*)d->y, d->bias, (const float*)d->emb,
                                                                  d->residual));
  }
  MKD_CHECK_LAUNCH();
  return MKD_OK;
}
}  // namespace mkd

static int validate(const mkd_conv_desc* d) {
  MKD_REQUIRE(d != nullptr, MKD_E_INVALID, "conv2d: null descriptor");
  MKD_REQUIRE(d->dtype == MKD_BF16 || d->dtype == MKD_F32, MKD_E_INVALID, "conv2d: bad dtype %d", d->dtype);
  MKD_REQUIRE(d->x && d->w && (d->y || d->y32), MKD_E_INVALID, "conv2d: null x/w/y");
  MKD_REQUIRE(d->residual_dtype == MKD_BF16 || d->residual_dtype == MKD_F32, MKD_E_INVALID, "conv2d: bad residual_dtype");
  MKD_REQUIRE(!d->residual || d->dtype == MKD_BF16 || d->residual_dtype == MKD_F32, MKD_E_INVALID,
              "conv2d: an fp32 conv takes an fp32 residual");
  MKD_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->C > 0 && d->K > 0 && d->R > 0 && d->S > 0 && d->stride > 0 &&
                  d->pad >= 0 && d->pad_hi_extra >= 0 && d->pad_hi_extra <= 1,
              MKD_E_INVALID, "conv2d: non-positive dimension");
  MKD_REQUIRE(d->ldx >= d->C, MKD_E_INVALID, "conv2d: ldx %d < C %d", d->ldx, d->C);
  const int kout = d->act == MKD_ACT_GEGLU ? d->K / 2 : d->K;
  MKD_REQUIRE(!d->y || d->ldy >= kout, MKD_E_INVALID, "conv2d: ldy %d < output channels %d", d->ldy, kout);
  MKD_REQUIRE(!d->y32 || d->ldy32 >= kout, MKD_E_INVALID, "conv2d: ldy32 %d < output channels %d", d->ldy32, kout);
  MKD_REQUIRE(!d->residual || d->ldr >= kout, MKD_E_INVALID, "conv2d: ldr too small");
  MKD_REQUIRE(!d->emb || d->lde >= kout, MKD_E_INVALID, "conv2d: lde too small");
  MKD_REQUIRE(d->act >= MKD_ACT_NONE && d->act <= MKD_ACT_GEGLU, MKD_E_INVALID, "conv2d: bad act");
  if (d->x2) {
    MKD_REQUIRE(d->C2 > 0 && d->ldx2 >= d->C2, MKD_E_INVALID, "conv2d: x2 term needs C2 > 0 and ldx2 >= C2");
    MKD_REQUIRE(d->dtype == MKD_BF16 && d->stride == 1 && !d->upsample && d->act != MKD_ACT_GEGLU && d->path != MKD_PATH_GENERIC &&
                    d->path != MKD_PATH_TCGEN05_SINGLE,
                MKD_E_INVALID, "conv2d: the x2 term is bf16, stride 1, no upsample / GEGLU, tensor-core CTA-pair kernel only");
  }
  MKD_REQUIRE(d->wgroups >= 0 && d->wgroups <= 2, MKD_E_INVALID, "conv2d: wgroups must be 0, 1 or 2");
  if (d->wgroups == 2)
    MKD_REQUIRE(d->dtype == MKD_BF16 && d->path != MKD_PATH_GENERIC && d->path != MKD_PATH_TCGEN05_SINGLE && d->N % 2 == 0, MKD_E_INVALID,
                "conv2d: weight groups are bf16, even batch, tensor-core CTA-pair kernel only");
  if (d->gn_y) {
    MKD_REQUIRE(d->dtype == MKD_BF16 && d->act == MKD_ACT_NONE && d->gn_groups > 0 && d->K % d->gn_groups == 0 &&
                    (d->K / d->gn_groups) % 8 == 0 && d->gn_gamma && d->gn_beta && d->gn_ld >= d->K && d->path != MKD_PATH_GENERIC &&
                    d->path != MKD_PATH_TCGEN05_SINGLE && d->stride == 1 && !d->upsample && !d->stats,
                MKD_E_INVALID, "conv2d: the GroupNorm tail is bf16, act NONE, whole vectors of 8 channels per group, stride 1, CTA-pair kernel only");
  }
  if (d->act == MKD_ACT_GEGLU) {
    MKD_REQUIRE(d->K % 2 == 0 && d->geglu_block > 0 && (d->K / 2) % d->geglu_block == 0, MKD_E_INVALID,
                "conv2d: GEGLU needs K even and K/2 %% geglu_block == 0");
    MKD_REQUIRE(!d->emb && !d->residual && d->alpha == 1.0f, MKD_E_INVALID, "conv2d: GEGLU excludes emb/residual/alpha");
  }
  const int Hin = d->upsample ? 2 * d->H : d->H, Win = d->upsample ? 2 * d->W : d->W;
  MKD_REQUIRE(Hin + 2 * d->pad + d->pad_hi_extra >= d->R && Win + 2 * d->pad + d->pad_hi_extra >= d->S, MKD_E_INVALID,
              "conv2d: filter larger than input");
  MKD_REQUIRE((int64_t)d->N * Hin * Win < (1ll << 31), MKD_E_INVALID, "conv2d: too many pixels");
  MKD_REQUIRE(d->path >= MKD_PATH_AUTO && d->path <= MKD_PATH_TCGEN05_PAIR, MKD_E_INVALID, "conv2d: bad path");
  return MKD_OK;
}

extern "C" int mkd_conv2d_path(const mkd_conv_desc* d) {
  int rc = validate(d);
  if (rc) return rc;
  if (d->path == MKD_PATH_GENERIC) return MKD_PATH_GENERIC;
  bool ok = mkd::conv2d_tcgen05_supported(d);
  if ((d->x2 || d->wgroups == 2 || d->gn_y) && !ok) return MKD_E_INVALID;  // no other kernel takes the second term: the caller issues the two layers separately
  if (d->path >= MKD_PATH_TCGEN05) {  // forced tensor-core kernel (either of the two)
    if (!ok) return MKD_E_INVALID;  // conv2d_tcgen05_supported() left the reason in mkd_last_error()
    return MKD_PATH_TCGEN05;
  }
  return ok ? MKD_PATH_TCGEN05 : MKD_PATH_GENERIC;
}

extern "C" int mkd_conv2d(const mkd_conv_desc* d, mkd_stream_t stream) {
  int path = mkd_conv2d_path(d);
  if (path < 0) return path;
  if (path == MKD_PATH_TCGEN05) return mkd::conv2d_tcgen05(d, (cudaStream_t)stream);
  return mkd::conv2d_generic(d, (cudaStream_t)stream);
}
