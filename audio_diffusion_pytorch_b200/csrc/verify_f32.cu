// fp32 VERIFICATION MODE (B200UNet.verify_fp32): the same launch program, packed-weight layouts,
// folds and fusion algebra as the bf16 tensor-core path, executed with fp32 storage and fp32
// arithmetic by deliberately simple CUDA-core kernels (one thread per output, no tiling, exact
// SiLU / GELU / exp).  It exists to check the PROGRAM -- weight packing, LayerNorm folds, phase-folded
// upsample convs, the concatenated conditioning GEMM, guidance combine, sampler update -- against
// the reference at fp32 tolerance (rtol 1e-3 / atol 1e-4), which the bf16 storage of the fast
// path cannot show.  Not a performance path: ~100x slower than the tcgen05 kernels.
// Entry points mirror their bf16 counterparts argument for argument (a/w/out/residual/h are fp32).
#include "common.cuh"
#include "ptx.cuh"

namespace adp {

__device__ __forceinline__ float silu_exact(float z) { return z / (1.f + expf(-z)); }
__device__ __forceinline__ float gelu_exact(float z) { return 0.5f * z * (1.f + erff(z * 0.70710678118654752f)); }

// out[b,t,p*n_valid+n] = (sum_slot sum_k a[b,t+off(p,slot),k] * w[p*n_pad+n, slot*c_in+k] + bias[n])
//                        * gate[b,n] + residual[b,t,p*n_valid+n]          (include/adp_b200.h)
__global__ void __launch_bounds__(256)
f32_conv_gemm_kernel(const adp_conv_gemm_args a) {
  pdl_launch_dependents();
  pdl_wait();
  const float* A = static_cast<const float*>(a.a);
  const float* W = static_cast<const float*>(a.w);
  const float* R = static_cast<const float*>(a.residual);
  float* O = static_cast<float*>(a.out);
  const int64_t per_row = static_cast<int64_t>(a.phases) * a.n_valid;
  const int64_t total = static_cast<int64_t>(a.B) * a.T * per_row;
  const int ldg = a.ld_gate > 0 ? a.ld_gate : a.n_valid;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = i / per_row;
    const int col = static_cast<int>(i - row * per_row);
    const int p = col / a.n_valid, n = col - p * a.n_valid;
    const int b = static_cast<int>(row / a.T), t = static_cast<int>(row - static_cast<int64_t>(b) * a.T);
    int slots, off0;
    if (a.up_factor > 1) {
      if (p == 0) { slots = 2; off0 = -1; }
      else if (p == a.up_factor - 1) { slots = 2; off0 = 0; }
      else { slots = 1; off0 = 0; }
    } else {
      slots = a.ntaps; off0 = a.tap_off[0];
    }
    const float* wr = W + (static_cast<int64_t>(p) * a.n_pad + n) * a.k_total;
    float acc = 0.f;
    for (int s = 0; s < slots; ++s) {
      const int tt = t + (a.up_factor > 1 ? off0 + s : a.tap_off[s]);
      if (tt < 0 || tt >= a.T) continue;               // conv zero padding
      const float* ar = A + (static_cast<int64_t>(b) * a.T + tt) * a.lda;
      const float* ws = wr + static_cast<int64_t>(s) * a.c_in;
      float part = 0.f;
      for (int k = 0; k < a.c_in; ++k) part = fmaf(ar[k], ws[k], part);
      acc += part;
    }
    if (a.bias) acc += a.bias[n];
    if (a.gate) acc *= a.gate[static_cast<int64_t>(b) * ldg + n];
    const int64_t oidx = row * a.ldo + col;
    if (R) acc += R[oidx];
    O[oidx] = acc;
  }
}

// per-(b, group) sum / sum of squares -> fp64 bins (accumulating).  grid (chunks, B)
__global__ void __launch_bounds__(256)
f32_gn_stats_kernel(const float* __restrict__ x, double* __restrict__ stats, int T, int C, int groups) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double s_bins[2 * 64];
  if (threadIdx.x < 128) s_bins[threadIdx.x] = 0.0;
  __syncthreads();
  const int b = blockIdx.y, gsz = C / groups;
  const int64_t n = static_cast<int64_t>(T) * C;
  const float* xb = x + static_cast<int64_t>(b) * n;
  int cur = -1;
  double s = 0.0, q = 0.0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(i % C) / gsz;
    if (g != cur) {
      if (cur >= 0) { atomicAdd(&s_bins[2 * cur], s); atomicAdd(&s_bins[2 * cur + 1], q); }
      cur = g; s = 0.0; q = 0.0;
    }
    const double v = xb[i];
    s += v; q += v * v;
  }
  if (cur >= 0) { atomicAdd(&s_bins[2 * cur], s); atomicAdd(&s_bins[2 * cur + 1], q); }
  __syncthreads();
  if (threadIdx.x < 2 * groups && s_bins[threadIdx.x] != 0.0)
    atomicAdd(stats + static_cast<int64_t>(b) * 2 * groups + threadIdx.x, s_bins[threadIdx.x]);
}

__global__ void __launch_bounds__(256)
f32_gn_silu_kernel(const float* __restrict__ x, float* __restrict__ y, const double* __restrict__ stats,
                   const float* __restrict__ gamma, const float* __restrict__ beta, int B, int T, int C,
                   int groups, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  const int gsz = C / groups;
  const int64_t total = static_cast<int64_t>(B) * T * C;
  const double inv_n = 1.0 / (static_cast<double>(gsz) * T);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int b = static_cast<int>(i / (static_cast<int64_t>(T) * C));
    const double* st = stats + (static_cast<int64_t>(b) * groups + c / gsz) * 2;
    const double mean = st[0] * inv_n;
    const double var = fmax(st[1] * inv_n - mean * mean, 0.0);
    const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float z = (x[i] - static_cast<float>(mean)) * rstd * gamma[c] + beta[c];
    y[i] = silu_exact(z);
  }
}

// one warp per row: y = LN(x; eps) * (1 + scale) + shift, optionally y2 = LN(y; eps2)
__global__ void __launch_bounds__(256)
f32_ln_film_kernel(const float* __restrict__ x, float* __restrict__ y, float* __restrict__ y2,
                   const float* __restrict__ ss, int ss_stride, int B, int T, int C, float eps, float eps2) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t rows = static_cast<int64_t>(B) * T;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5); r < rows;
       r += static_cast<int64_t>(gridDim.x) * 8) {
    const float* xr = x + r * C;
    const float* sc = ss ? ss + (r / T) * ss_stride : nullptr;
    float m = 0.f;
    for (int c = lane; c < C; c += 32) m += xr[c];
    m = warp_sum(m) / C;
    float v = 0.f;
    for (int c = lane; c < C; c += 32) { const float d = xr[c] - m; v += d * d; }
    const float rstd = rsqrtf(warp_sum(v) / C + eps);
    float m2 = 0.f;
    for (int c = lane; c < C; c += 32) {
      float o = (xr[c] - m) * rstd;
      if (sc) o = o * (1.f + sc[c]) + sc[C + c];
      y[r * C + c] = o;
      m2 += o;
    }
    if (y2) {
      m2 = warp_sum(m2) / C;
      float v2 = 0.f;
      for (int c = lane; c < C; c += 32) { const float d = y[r * C + c] - m2; v2 += d * d; }
      const float rstd2 = rsqrtf(warp_sum(v2) / C + eps2);
      for (int c = lane; c < C; c += 32) y2[r * C + c] = (y[r * C + c] - m2) * rstd2;
    }
  }
}

// softmax(q k^T * scale) v, head dim 64; one thread per (b, head, query), online softmax
__global__ void __launch_bounds__(128)
f32_attention_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     float* __restrict__ o, int B, int H, int Tq, int Tk, int ldq, int ldk, int ldv, int ldo,
                     float scale) {
  pdl_launch_dependents();
  pdl_wait();
  const int64_t total = static_cast<int64_t>(B) * H * Tq;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int tq = static_cast<int>(i % Tq);
    const int h = static_cast<int>((i / Tq) % H);
    const int b = static_cast<int>(i / (static_cast<int64_t>(Tq) * H));
    const float* qr = q + (static_cast<int64_t>(b) * Tq + tq) * ldq + h * 64;
    float qv[64], acc[64];
#pragma unroll
    for (int d = 0; d < 64; ++d) { qv[d] = qr[d] * scale; acc[d] = 0.f; }
    float mx = -INFINITY, l = 0.f;
    for (int j = 0; j < Tk; ++j) {
      const float* kr = k + (static_cast<int64_t>(b) * Tk + j) * ldk + h * 64;
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < 64; ++d) s = fmaf(qv[d], kr[d], s);
      const float mn = fmaxf(mx, s);
      const float corr = expf(mx - mn), pj = expf(s - mn);
      l = l * corr + pj;
      const float* vr = v + (static_cast<int64_t>(b) * Tk + j) * ldv + h * 64;
#pragma unroll
      for (int d = 0; d < 64; ++d) acc[d] = acc[d] * corr + pj * vr[d];
      mx = mn;
    }
    float* orow = o + (static_cast<int64_t>(b) * Tq + tq) * ldo + h * 64;
    const float inv = 1.f / l;
#pragma unroll
    for (int d = 0; d < 64; ++d) orow[d] = acc[d] * inv;
  }
}

// y[b, n] = act_out( sum_k act_in(x[b, k]) * w[n, k] + bias[n] )
__global__ void __launch_bounds__(256)
f32_linear_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                  float* __restrict__ y, int B, int K, int N, int ldx, int ldw, int ldy, int in_act,
                  int out_act) {
  pdl_launch_dependents();
  pdl_wait();
  const int total = B * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / N, n = i - b * N;
    float acc = 0.f;
    for (int k = 0; k < K; ++k) {
      float xv = x[static_cast<int64_t>(b) * ldx + k];
      if (in_act == ADP_ACT_GELU) xv = gelu_exact(xv);
      else if (in_act == ADP_ACT_SILU) xv = silu_exact(xv);
      acc = fmaf(xv, w[static_cast<int64_t>(n) * ldw + k], acc);
    }
    if (bias) acc += bias[n];
    if (out_act == ADP_ACT_GELU) acc = gelu_exact(acc);
    else if (out_act == ADP_ACT_SILU) acc = silu_exact(acc);
    y[static_cast<int64_t>(b) * ldy + n] = acc;
  }
}

__global__ void __launch_bounds__(256)
f32_silu_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n) {
  pdl_launch_dependents();
  pdl_wait();
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    y[i] = silu_exact(x[i]);
}

// Downsample conv of level 0: out[b, to, c] = bias[c] + sum_{ci, j} w[c][ci][j] * in[b, ci, to*f + j],
// in = cat([x, append]); out fp32 channels-last
__global__ void __launch_bounds__(256) f32_stem_in_kernel(const adp_stem_in_args a) {
  pdl_launch_dependents();
  pdl_wait();
  const int cin = a.cx + a.ca, To = a.T / a.f;
  float* out = static_cast<float*>(a.out);
  const int64_t total = static_cast<int64_t>(a.B) * To * a.c0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % a.c0);
    const int to = static_cast<int>((i / a.c0) % To);
    const int b = static_cast<int>(i / (static_cast<int64_t>(a.c0) * To));
    float acc = a.bias ? a.bias[c] : 0.f;
    for (int ci = 0; ci < cin; ++ci)
      for (int j = 0; j < a.f; ++j) {
        const int64_t tt = static_cast<int64_t>(to) * a.f + j;
        const float xv = ci < a.cx ? a.x[(static_cast<int64_t>(b) * a.cx + ci) * a.T + tt]
                                   : a.append[(static_cast<int64_t>(b) * a.ca + (ci - a.cx)) * a.T + tt];
        acc = fmaf(xv, a.w[(static_cast<int64_t>(c) * cin + ci) * a.f + j], acc);
      }
    out[i] = acc;
  }
}

// Level-0 output: v = skip + gate * (conv3(nearest-upsample(h)) + bias), guidance combine, sampler
// update -- the semantics of stem_out_kernel (stem.cu) with h in fp32
__device__ __forceinline__ float f32_stem_branch(const adp_stem_out_args& a, const float* hb, int o, int t) {
  float y = a.bias ? a.bias[o] : 0.f;
  for (int k = 0; k < 3; ++k) {
    const int idx = t + k - 1;
    if (idx < 0 || idx >= a.T) continue;
    const float* row = hb + static_cast<int64_t>(idx / a.f) * a.c0;
    for (int c = 0; c < a.c0; ++c) y = fmaf(row[c], a.w[(static_cast<int64_t>(o) * a.c0 + c) * 3 + k], y);
  }
  return y;
}

__global__ void __launch_bounds__(256) f32_stem_out_kernel(const adp_stem_out_args a) {
  pdl_launch_dependents();
  pdl_wait();
  const int ldg = a.ld_gate > 0 ? a.ld_gate : a.co;
  const int cin = a.cx + a.ca, Tl = a.T / a.f;
  const float* h = static_cast<const float*>(a.h);
  const int64_t total = static_cast<int64_t>(a.B) * a.T;
  // one thread per (batch, position): every input channel is read before any output channel is
  // written (x_next may alias x)
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int t = static_cast<int>(i % a.T);
    const int b = static_cast<int>(i / a.T);
    float xin[8];
    for (int c = 0; c < 8; ++c) {
      xin[c] = 0.f;
      if (c < a.cx) xin[c] = a.x[(static_cast<int64_t>(b) * a.cx + c) * a.T + t];
      else if (c < cin) xin[c] = a.append[(static_cast<int64_t>(b) * a.ca + (c - a.cx)) * a.T + t];
    }
    for (int o = 0; o < a.co; ++o) {
      float skip;
      if (a.w_adapt) {
        skip = a.b_adapt ? a.b_adapt[o] : 0.f;
        for (int c = 0; c < cin; ++c) skip = fmaf(xin[c], a.w_adapt[o * cin + c], skip);
      } else {
        skip = xin[o];
      }
      float v = skip + a.gate[static_cast<int64_t>(b) * ldg + o] *
                           f32_stem_branch(a, h + static_cast<int64_t>(b) * Tl * a.c0, o, t);
      if (a.cfg) {
        const float vm = skip + a.gate[static_cast<int64_t>(b + a.B) * ldg + o] *
                                    f32_stem_branch(a, h + static_cast<int64_t>(b + a.B) * Tl * a.c0, o, t);
        v = vm + (v - vm) * a.cfg_scale;
      }
      const int64_t oidx = (static_cast<int64_t>(b) * a.co + o) * a.T + t;
      if (a.v_out) a.v_out[oidx] = v;
      if (a.x_next) {
        const float a0 = a.ab[0], b0 = a.ab[1], a1 = a.ab[2], b1 = a.ab[3];
        a.x_next[oidx] = a1 * (a0 * xin[o] - b0 * v) + b1 * (b0 * xin[o] + a0 * v);
      }
    }
  }
}

static int f32_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  if (g < 1) g = 1;
  if (g > 148 * 16) g = 148 * 16;
  return static_cast<int>(g);
}

}  // namespace adp

using namespace adp;

extern "C" int adp_f32_conv_gemm(const adp_conv_gemm_args* args, adp_stream_t stream) {
  ADP_CHECK(args && args->a && args->w && args->out, "adp_f32_conv_gemm: null pointer");
  const adp_conv_gemm_args& a = *args;
  ADP_CHECK(a.B > 0 && a.T > 0 && a.c_in > 0 && a.n_valid > 0 && a.phases >= 1, "adp_f32_conv_gemm: bad sizes");
  ADP_CHECK(!a.stats, "adp_f32_conv_gemm: statistics are a separate pass");
  ADP_CHECK(a.up_factor <= 1 || a.phases == a.up_factor, "adp_f32_conv_gemm: phases != up_factor");
  ADP_CHECK(a.up_factor > 1 || (a.ntaps >= 1 && a.ntaps <= 3 && a.phases == 1), "adp_f32_conv_gemm: taps");
  ADP_CUDA(launch_k(f32_conv_gemm_kernel, dim3(f32_grid(static_cast<int64_t>(a.B) * a.T * a.phases * a.n_valid)),
                    dim3(256), (size_t)0, as_stream(stream), a));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_gn_stats(const float* x, double* stats, int B, int T, int C, int groups,
                                adp_stream_t stream) {
  ADP_CHECK(x && stats && B > 0 && B <= 65535 && T > 0 && C > 0 && groups > 0 && groups <= 64 && C % groups == 0,
            "adp_f32_gn_stats: bad args");
  int gx = f32_grid(static_cast<int64_t>(T) * C);
  if (gx > 148 * 4) gx = 148 * 4;
  ADP_CUDA(launch_k(f32_gn_stats_kernel, dim3(gx, B), dim3(256), (size_t)0, as_stream(stream), x, stats, T, C,
                    groups));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_gn_silu(const float* x, float* y, const double* stats, const float* gamma,
                               const float* beta, int B, int T, int C, int groups, float eps,
                               adp_stream_t stream) {
  ADP_CHECK(x && y && stats && gamma && beta && B > 0 && T > 0 && C > 0 && groups > 0 && C % groups == 0,
            "adp_f32_gn_silu: bad args");
  ADP_CUDA(launch_k(f32_gn_silu_kernel, dim3(f32_grid(static_cast<int64_t>(B) * T * C)), dim3(256), (size_t)0,
                    as_stream(stream), x, y, stats, gamma, beta, B, T, C, groups, eps));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_ln_film(const float* x, float* y, float* y2, const float* scale_shift, int ss_stride,
                               int B, int T, int C, float eps, float eps2, adp_stream_t stream) {
  ADP_CHECK(x && y && B > 0 && T > 0 && C > 0, "adp_f32_ln_film: bad args");
  ADP_CUDA(launch_k(f32_ln_film_kernel, dim3(f32_grid(static_cast<int64_t>(B) * T * 32)), dim3(256), (size_t)0,
                    as_stream(stream), x, y, y2, scale_shift, ss_stride, B, T, C, eps, eps2));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_attention(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq,
                                 int Tk, int ldq, int ldk, int ldv, int ldo, float scale, adp_stream_t stream) {
  ADP_CHECK(q && k && v && o && B > 0 && H > 0 && Tq > 0 && Tk > 0, "adp_f32_attention: bad args");
  int64_t n = static_cast<int64_t>(B) * H * Tq;
  int64_t g = (n + 127) / 128;
  if (g > 148 * 16) g = 148 * 16;
  ADP_CUDA(launch_k(f32_attention_kernel, dim3(static_cast<int>(g)), dim3(128), (size_t)0, as_stream(stream), q, k,
                    v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo, scale));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_linear(const float* x, const float* w, const float* bias, float* y, int B, int K, int N,
                              int ldx, int ldw, int ldy, int in_act, int out_act, adp_stream_t stream) {
  ADP_CHECK(x && w && y && B > 0 && K > 0 && N > 0, "adp_f32_linear: bad args");
  ADP_CUDA(launch_k(f32_linear_kernel, dim3(f32_grid(static_cast<int64_t>(B) * N)), dim3(256), (size_t)0,
                    as_stream(stream), x, w, bias, y, B, K, N, ldx, ldw, ldy, in_act, out_act));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_silu(const float* x, float* y, int64_t n, adp_stream_t stream) {
  ADP_CHECK(x && y && n > 0, "adp_f32_silu: bad args");
  ADP_CUDA(launch_k(f32_silu_kernel, dim3(f32_grid(n)), dim3(256), (size_t)0, as_stream(stream), x, y, n));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_stem_in(const adp_stem_in_args* args, adp_stream_t stream) {
  ADP_CHECK(args && args->x && args->w && args->out, "adp_f32_stem_in: null pointer");
  const adp_stem_in_args& a = *args;
  ADP_CHECK(!a.noise && !a.stats, "adp_f32_stem_in: noising / statistics are not part of the verification mode");
  ADP_CHECK(a.f >= 1 && a.T % a.f == 0 && (a.ca == 0) == (a.append == nullptr), "adp_f32_stem_in: bad args");
  ADP_CUDA(launch_k(f32_stem_in_kernel, dim3(f32_grid(static_cast<int64_t>(a.B) * (a.T / a.f) * a.c0)), dim3(256),
                    (size_t)0, as_stream(stream), a));
  ADP_LAUNCH_CHECK();
  return 0;
}

extern "C" int adp_f32_stem_out(const adp_stem_out_args* args, adp_stream_t stream) {
  ADP_CHECK(args && args->h && args->x && args->w && args->gate, "adp_f32_stem_out: null pointer");
  const adp_stem_out_args& a = *args;
  ADP_CHECK(!a.noise && !a.loss_sum && !a.dv, "adp_f32_stem_out: the fused loss is not part of the verification mode");
  ADP_CHECK(a.w_adapt || a.cx + a.ca == a.co, "adp_f32_stem_out: identity skip needs cx+ca == co");
  ADP_CHECK(!a.x_next || a.ab, "adp_f32_stem_out: x_next needs ab");
  ADP_CHECK(a.f >= 1 && a.T % a.f == 0 && (a.ca == 0) == (a.append == nullptr), "adp_f32_stem_out: bad args");
  ADP_CHECK(a.cx + a.ca <= 8 && a.co <= a.cx, "adp_f32_stem_out: in <= 8 channels, out <= x channels");
  ADP_CUDA(launch_k(f32_stem_out_kernel, dim3(f32_grid(static_cast<int64_t>(a.B) * a.T)), dim3(256),
                    (size_t)0, as_stream(stream), a));
  ADP_LAUNCH_CHECK();
  return 0;
}
