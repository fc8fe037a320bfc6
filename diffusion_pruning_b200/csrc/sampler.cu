// Scheduler steps of the sampling loop beyond DDIM eta 0: classifier-free guidance with the diffusers guidance rescale,
// stochastic DDIM and DPM-Solver++ (1 / 2M), as one fused elementwise pass per step. The per-step scalars come from
// sampling.sampler_plan (float64 on the host); the kernels only apply
//   x_out = c_x x + c_0 x0 + c_h x0_hist + c_e eps + c_n noise.
// The rescale needs per-sample standard deviations of the guided and the text prediction: cfg_pred_stats writes fixed-order
// fp64 partial sums (no atomics, as in norm.cu, so a sampling pass is bit-reproducible) and every thread of the step
// kernel reduces its sample's partials in chunk order. For inpainting the step kernel is instantiated with the mask blend
// (aptp_cfg_sampler_step_masked), which resets the known region in the same pass.
#include "common.cuh"
#include "../../include/aptp_sm100.h"

namespace aptp {

constexpr int kStatChunks = APTP_SAMPLER_STAT_CHUNKS;

// One expression in both kernels, so the statistics describe exactly the m the step kernel forms.
__device__ __forceinline__ float cfg_combine(float pu, float pc, float guidance) { return fmaf(guidance, pc - pu, pu); }

// grid (kStatChunks, batch): block (c, b) sums elements [c nv / C, (c + 1) nv / C) of sample b, nv = float4 per sample.
__global__ void __launch_bounds__(256) cfg_pred_stats_kernel(const float4* __restrict__ pred, long long nv, int batch,
                                                             float guidance, double* __restrict__ partials) {
  const int c = blockIdx.x, b = blockIdx.y;
  const long long beg = nv * c / kStatChunks, end = nv * (c + 1) / kStatChunks;
  const float4* pu = pred + (long long)b * nv;
  const float4* pc = pred + ((long long)batch + b) * nv;
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long v = beg + threadIdx.x; v < end; v += blockDim.x) {
    const float4 u = pu[v], t = pc[v];
    const float tu[4] = {u.x, u.y, u.z, u.w}, tc[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double mt = tc[k], m = cfg_combine(tu[k], tc[k], guidance);
      s[0] += mt;
      s[1] += mt * mt;
      s[2] += m;
      s[3] += m * m;
    }
  }
  __shared__ double red[8][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    if (lane == 0) red[warp][k] = s[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w][threadIdx.x];
    partials[((long long)b * kStatChunks + c) * 4 + threadIdx.x] = t;
  }
}

// rescale * std(m_text) / std(m) + (1 - rescale): diffusers rescale_noise_cfg folded into one factor on m.
__device__ __forceinline__ float rescale_factor(const double* __restrict__ partials, int b, long long n, float rescale) {
  const double* p = partials + (long long)b * kStatChunks * 4;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int c = 0; c < kStatChunks; ++c) {
    s0 += p[4 * c + 0];
    s1 += p[4 * c + 1];
    s2 += p[4 * c + 2];
    s3 += p[4 * c + 3];
  }
  const double nn = (double)n;
  const double var_text = (s1 - s0 * s0 / nn) / (nn - 1.0), var_cfg = (s3 - s2 * s2 / nn) / (nn - 1.0);
  const double r = rescale;
  return (float)(r * (sqrt(var_text) / sqrt(var_cfg)) + (1.0 - r));
}

// The inpainting blend's operands (kBlend only): the known region, re-noised to the next timestep, replaces x_step
// where the mask is 0.
struct BlendArgs {
  const float4* image;
  const float* mask;        // [batch][plane], broadcast over the channels
  const float4* init_noise;
  long long plane;
  float a_next, s_next;
};

// mask values of the 4 elements of float4 i of sample b (j0 = its first element within the sample). When the plane
// size is a multiple of 4 they sit in one plane row and come as one float4; otherwise the float4 may straddle two
// channel planes and every element is indexed on its own.
__device__ __forceinline__ void load_mask4(const BlendArgs& bl, int b, long long j0, float m[4]) {
  const float* mb = bl.mask + b * bl.plane;
  if ((bl.plane & 3) == 0) {
    const float4 m4 = *reinterpret_cast<const float4*>(mb + j0 % bl.plane);
    m[0] = m4.x, m[1] = m4.y, m[2] = m4.z, m[3] = m4.w;
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) m[e] = mb[(j0 + e) % bl.plane];
  }
}

// (1 - m) proper + m x_step with proper = a_next image + s_next init_noise: m = 0 gives proper and m = 1 gives x_step
// bit for bit (the other product is a signed zero), and a_next = 1, s_next = 0 gives proper = image bit for bit.
__device__ __forceinline__ float blend(float m, float x_step, float img, float n0, float a_next, float s_next) {
  const float proper = fmaf(a_next, img, s_next * n0);
  return fmaf(m, x_step, (1.f - m) * proper);
}

template <bool kBlend>
__global__ void __launch_bounds__(256) cfg_sampler_step_kernel(
    const float4* __restrict__ pred, const float4* __restrict__ x, float4* __restrict__ x_out, long long nv, int batch,
    float guidance, float rescale, const double* __restrict__ partials, AptpSamplerCoeffs k, const float4* hist_in,
    float4* hist_out, const float* __restrict__ noise, long long noise_ld, int v_prediction, BlendArgs bl) {
  const long long total = nv * batch;
  int cur_b = -1;
  float scale = 1.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / nv);
    if (partials != nullptr && b != cur_b) {
      scale = rescale_factor(partials, b, nv * 4, rescale);
      cur_b = b;
    }
    const float4 u4 = pred[i], c4 = pred[total + i], x4 = x[i];
    float4 h4 = make_float4(0.f, 0.f, 0.f, 0.f), z4 = h4;
    if (hist_in != nullptr) h4 = hist_in[i];
    if (noise != nullptr) z4 = *reinterpret_cast<const float4*>(noise + b * noise_ld + (i - b * nv) * 4);
    const float pu[4] = {u4.x, u4.y, u4.z, u4.w}, pc[4] = {c4.x, c4.y, c4.z, c4.w};
    const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, hs[4] = {h4.x, h4.y, h4.z, h4.w}, zs[4] = {z4.x, z4.y, z4.z, z4.w};
    float o[4], x0s[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float m = cfg_combine(pu[e], pc[e], guidance);
      if (partials != nullptr) m *= scale;
      float x0, eps;
      if (v_prediction) {
        x0 = k.sa * xs[e] - k.sb * m;
        eps = k.sa * m + k.sb * xs[e];
      } else {
        eps = m;
        x0 = (xs[e] - k.sb * m) / k.sa;
      }
      x0s[e] = x0;
      o[e] = k.c_x * xs[e] + k.c_0 * x0 + k.c_h * hs[e] + k.c_e * eps + k.c_n * zs[e];
    }
    if constexpr (kBlend) {
      const float4 i4 = bl.image[i], n4 = bl.init_noise[i];
      const float is[4] = {i4.x, i4.y, i4.z, i4.w}, ns[4] = {n4.x, n4.y, n4.z, n4.w};
      float m[4];
      load_mask4(bl, b, (i - b * nv) * 4, m);
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = blend(m[e], o[e], is[e], ns[e], bl.a_next, bl.s_next);
    }
    x_out[i] = make_float4(o[0], o[1], o[2], o[3]);
    if (hist_out != nullptr) hist_out[i] = make_float4(x0s[0], x0s[1], x0s[2], x0s[3]);
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace aptp

using namespace aptp;

extern "C" int aptp_cfg_pred_stats(const float* pred, int64_t n_per_sample, int32_t batch, float guidance,
                                   double* partials, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  APTP_REQUIRE(pred && partials, "aptp_cfg_pred_stats: null pointer");
  APTP_REQUIRE(n_per_sample > 1 && n_per_sample % 4 == 0 && batch >= 0,
               "aptp_cfg_pred_stats: n_per_sample must be a multiple of 4 and > 1 (got %lld), batch >= 0",
               (long long)n_per_sample);
  APTP_REQUIRE(aligned16(pred), "aptp_cfg_pred_stats: pred must be 16-byte aligned");
  if (batch == 0) return APTP_OK;
  cfg_pred_stats_kernel<<<dim3(kStatChunks, batch), 256, 0, stream>>>(reinterpret_cast<const float4*>(pred),
                                                                       n_per_sample / 4, batch, guidance, partials);
  APTP_CUDA_CHECK(cudaGetLastError());
  return APTP_OK;
}

template <bool kBlend>
static int sampler_step(const char* name, const float* pred, const float* x, float* x_out, int64_t n_per_sample,
                        int32_t batch, float guidance, float rescale, const double* partials,
                        const AptpSamplerCoeffs* coeffs, const float* x0_hist_in, float* x0_hist_out, const float* noise,
                        int64_t noise_ld, int32_t v_prediction, const BlendArgs& bl, cudaStream_t stream) {
  APTP_REQUIRE(pred && x && x_out && coeffs, "%s: null pointer", name);
  APTP_REQUIRE(x_out != x, "%s: x_out must not alias x", name);
  APTP_REQUIRE(n_per_sample > 0 && n_per_sample % 4 == 0 && batch >= 0,
               "%s: n_per_sample must be a positive multiple of 4 (got %lld), batch >= 0", name,
               (long long)n_per_sample);
  APTP_REQUIRE(!partials || n_per_sample > 1, "%s: rescale needs n_per_sample > 1", name);
  APTP_REQUIRE(coeffs->c_h == 0.f || x0_hist_in, "%s: c_h != 0 needs x0_hist_in", name);
  APTP_REQUIRE(coeffs->c_n == 0.f || noise, "%s: c_n != 0 needs noise", name);
  APTP_REQUIRE(!noise || (noise_ld >= n_per_sample && noise_ld % 4 == 0),
               "%s: noise_ld must be a multiple of 4 and >= n_per_sample", name);
  APTP_REQUIRE(aligned16(pred) && aligned16(x) && aligned16(x_out) && aligned16(x0_hist_in) && aligned16(x0_hist_out) &&
                   aligned16(noise),
               "%s: pointers must be 16-byte aligned", name);
  if (batch == 0) return APTP_OK;
  const long long nv = n_per_sample / 4;
  long long blocks = (nv * batch + 255) / 256, cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cfg_sampler_step_kernel<kBlend><<<(unsigned)blocks, 256, 0, stream>>>(
      reinterpret_cast<const float4*>(pred), reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(x_out), nv,
      batch, guidance, rescale, partials, *coeffs, reinterpret_cast<const float4*>(x0_hist_in),
      reinterpret_cast<float4*>(x0_hist_out), noise, noise_ld, v_prediction, bl);
  APTP_CUDA_CHECK(cudaGetLastError());
  return APTP_OK;
}

extern "C" int aptp_cfg_sampler_step(const float* pred, const float* x, float* x_out, int64_t n_per_sample,
                                     int32_t batch, float guidance, float rescale, const double* partials,
                                     const AptpSamplerCoeffs* coeffs, const float* x0_hist_in, float* x0_hist_out,
                                     const float* noise, int64_t noise_ld, int32_t v_prediction, void* stream_) {
  return sampler_step<false>("aptp_cfg_sampler_step", pred, x, x_out, n_per_sample, batch, guidance, rescale, partials,
                             coeffs, x0_hist_in, x0_hist_out, noise, noise_ld, v_prediction, BlendArgs{},
                             reinterpret_cast<cudaStream_t>(stream_));
}

extern "C" int aptp_cfg_sampler_step_masked(const float* pred, const float* x, float* x_out, int64_t n_per_sample,
                                            int32_t batch, float guidance, float rescale, const double* partials,
                                            const AptpSamplerCoeffs* coeffs, const float* x0_hist_in,
                                            float* x0_hist_out, const float* noise, int64_t noise_ld,
                                            int32_t v_prediction, const float* image, const float* mask,
                                            int64_t plane_size, const float* init_noise, float a_next, float s_next,
                                            void* stream_) {
  APTP_REQUIRE(image && mask && init_noise, "aptp_cfg_sampler_step_masked: null pointer");
  APTP_REQUIRE(plane_size > 0 && n_per_sample % plane_size == 0,
               "aptp_cfg_sampler_step_masked: plane_size (%lld) must divide n_per_sample (%lld)",
               (long long)plane_size, (long long)n_per_sample);
  APTP_REQUIRE(aligned16(image) && aligned16(mask) && aligned16(init_noise),
               "aptp_cfg_sampler_step_masked: pointers must be 16-byte aligned");
  APTP_REQUIRE(image != x_out && init_noise != x_out && mask != x_out && image != x0_hist_out &&
                   init_noise != x0_hist_out && mask != x0_hist_out,
               "aptp_cfg_sampler_step_masked: image / mask / init_noise must not alias an output");
  const BlendArgs bl{reinterpret_cast<const float4*>(image), mask, reinterpret_cast<const float4*>(init_noise),
                     (long long)plane_size, a_next, s_next};
  return sampler_step<true>("aptp_cfg_sampler_step_masked", pred, x, x_out, n_per_sample, batch, guidance, rescale,
                            partials, coeffs, x0_hist_in, x0_hist_out, noise, noise_ld, v_prediction, bl,
                            reinterpret_cast<cudaStream_t>(stream_));
}
