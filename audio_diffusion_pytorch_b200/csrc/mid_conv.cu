// adp_narrow_conv for C = 32 and C = 64: one kernel per ConvBlock of the thin, long levels
// (README config: [8, 65536, 32] and [8, 16384, 64] activations).
//
// These levels are HBM-bound: a conv3 is only 6*C flop per byte moved.  The three-kernel path
// (adp_gn_silu -> adp_conv_gemm -> adp_ln_film) streams the level's tensor through HBM five to
// seven times and its 128 x C tcgen05 tiles are dominated by per-tile barrier / drain overheads
// (profiles/r1_gemm_skeleton_v5.txt).  Here GroupNorm-apply + SiLU happens while rows are staged
// into smem, the conv is a [rows x 3C] x [3C x C] GEMM on mma.sync.m16n8k16 (A fragments by
// ldmatrix over overlapping row windows: tap k of row t is smem row t + k; weights as bf16 in
// smem), and bias, residual, LayerNorm + FiLM and the next GroupNorm's statistics are applied
// to the accumulator fragments: x (+ residual) is read once, y written once.
//   * persistent blocks over row tiles of one batch element; the next tile's rows are
//     prefetched into registers before the current tile is computed; smem double buffered
//   * smem rows padded by 16 bytes so ldmatrix (8 rows x 16 B) and the 4-byte residual reads
//     in accumulator layout are bank-conflict free
//   * SiLU with one MUFU op (tanh.approx); operands enter the tensor core as bf16 exactly like
//     on the tcgen05 path of the wider levels
#include "common.cuh"
#include "ptx.cuh"

namespace adp {

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0,
                                               uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// 256 threads per block, 2 blocks per SM (128 x 4 half-size tiles measured no faster end to end,
// DESIGN.md section 8)
template <int C>
struct MidCfg {
  static constexpr int NTH = 256;                      // threads per block
  static constexpr int TB = C == 32 ? 256 : 128;       // rows per tile
  static constexpr int TPR = NTH / TB;                 // staging threads per row
  static constexpr int RPW = TB / (NTH / 32);          // rows per warp in the MMA phase
  static constexpr int RS = C * 2 + 16;                // padded smem row stride of s_x (bytes)
  static constexpr int WS = 3 * C * 2 + 16;            // padded stride of one W row (n) in smem
  static constexpr int MB = RPW / 16;                  // m16 blocks per warp
  static constexpr int NT = C / 8;                     // n8 tiles
  static constexpr int OS = C + 4;                     // padded fp32 row stride of s_o (floats)
  static constexpr int LPR = C / 8;                    // epilogue lanes per row (8 channels each)
  static constexpr int ER = TB * LPR / NTH;            // epilogue rows per thread
  static constexpr int X_BYTES = (TB + 2) * RS;
  static constexpr int O_BYTES = TB * OS * 4;
  static constexpr int W_BYTES = C * WS;
  static constexpr int SMEM = X_BYTES + O_BYTES + W_BYTES;
};

// Per tile: (1) the prefetched rows are activated (GroupNorm + SiLU) into s_x; (2) the next
// tile's rows and this tile's residual rows are requested; (3) conv3 as an mma.sync GEMM over
// overlapping row windows of s_x; (4) the fp32 accumulators go to s_o in row-major order and
// (5) the row-wise epilogue (bias is already in the accumulator; + residual, LayerNorm + FiLM,
// statistics) runs with ONE thread per 8 consecutive channels of a row: 16-byte residual loads
// and output stores, FiLM coefficients of the thread's 8 channels in registers, 3 shuffles per
// reduction.  (The first version ran the epilogue in the accumulator-fragment layout: 4-byte
// stores, 4-byte shared-memory residual reads and a shuffle chain per fragment row made the
// kernel issue/latency bound at 15-40 % of HBM bandwidth, profiles/r2_ncu_mid_conv64.txt.)
template <int C>
__global__ void __launch_bounds__(256, 2) mid_conv_kernel(const adp_narrow_conv_args a) {
  using Cfg = MidCfg<C>;
  constexpr int NTH = Cfg::NTH, TB = Cfg::TB, TPR = Cfg::TPR, RS = Cfg::RS, WS = Cfg::WS, MB = Cfg::MB, NT = Cfg::NT;
  constexpr int OS = Cfg::OS, LPR = Cfg::LPR, ER = Cfg::ER, RPW = Cfg::RPW;
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* s_x = smem;                                          // [TB+2][RS] activated rows t0-1 .. t0+TB
  float* s_o = reinterpret_cast<float*>(smem + Cfg::X_BYTES);   // [TB][OS]   conv output (fp32)
  uint8_t* s_w = smem + Cfg::X_BYTES + Cfg::O_BYTES;            // [C][WS]    W[n][k = tap*C + ci] bf16
  __shared__ __align__(16) float s_ga[C], s_de[C];   // GroupNorm a, d per channel
  __shared__ __align__(16) float s_sc[C], s_sh[C];   // FiLM 1+scale, shift
  __shared__ float s_bias[C];
  __shared__ float s_stats[2 * 64];
  const int b = blockIdx.y;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, q = lane & 3;
  const bool has_res = a.residual != nullptr, has_film = a.scale_shift != nullptr;

  if (tid < 128) s_stats[tid] = 0.f;
  if (a.w_packed) {            // bf16 [C][3C] image prepared by the host: straight 16-byte copy
    constexpr int VPRW = 3 * C * 2 / 16;             // 16-byte vectors per W row
    const uint4* wp = static_cast<const uint4*>(a.w_packed);
    for (int i = tid; i < C * VPRW; i += NTH) {
      const int co = i / VPRW, v = i - co * VPRW;
      *reinterpret_cast<uint4*>(s_w + co * WS + v * 16) = __ldg(wp + i);
    }
  } else {                     // PyTorch fp32 [co][ci][tap] -> [co][tap*C + ci]
    for (int pidx = tid; pidx < C * C; pidx += NTH) {
      const int co = pidx / C, ci = pidx % C;
      const float* src = a.w + static_cast<size_t>(pidx) * 3;
#pragma unroll
      for (int tap = 0; tap < 3; ++tap)
        *reinterpret_cast<__nv_bfloat16*>(s_w + co * WS + (tap * C + ci) * 2) = __float2bfloat16(src[tap]);
    }
  }
  if (tid < C) {
    const int c = tid;
    const int gsz = C / a.groups, gi = c / gsz;
    const double inv_n = 1.0 / (static_cast<double>(gsz) * a.T);
    const double sm = a.stats_in[(static_cast<size_t>(b) * a.groups + gi) * 2];
    const double sq = a.stats_in[(static_cast<size_t>(b) * a.groups + gi) * 2 + 1];
    const double mean = sm * inv_n;
    const float var = fmaxf(static_cast<float>(sq * inv_n - mean * mean), 0.f);
    const float ga = a.gamma[c] * rsqrtf(var + a.gn_eps);
    s_ga[c] = ga;
    s_de[c] = a.beta[c] - static_cast<float>(mean) * ga;
    s_bias[c] = a.bias ? a.bias[c] : 0.f;
    const float* ss = has_film ? a.scale_shift + static_cast<size_t>(b) * a.ss_stride : nullptr;
    s_sc[c] = has_film ? 1.f + ss[c] : 1.f;
    s_sh[c] = has_film ? ss[C + c] : 0.f;
  }
  __syncthreads();

  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(a.x) + static_cast<size_t>(b) * a.T * C;
  const __nv_bfloat16* rb =
      has_res ? static_cast<const __nv_bfloat16*>(a.residual) + static_cast<size_t>(b) * a.T * C : nullptr;
  __nv_bfloat16* yb = static_cast<__nv_bfloat16*>(a.y) + static_cast<size_t>(b) * a.T * C;
  const int n_tiles = (a.T + TB - 1) / TB;

  // staging: thread -> (row, 32-channel part); 4 x 16 bytes each
  const int srow = tid / TPR, spart = tid % TPR;
  // epilogue: thread -> 8 channels [8*el, 8*el+8) of rows erow0 + i*(256/LPR)
  const int el = tid % LPR, erow0 = tid / LPR;
  float fsc[8], fsh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { fsc[j] = s_sc[el * 8 + j]; fsh[j] = s_sh[el * 8 + j]; }

  auto load_tile = [&](int tile, uint4 (&xr)[4], uint4 (&hr)[4]) {
    const int t0 = tile * TB;
    const int t = t0 + srow;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      xr[i] = make_uint4(0, 0, 0, 0);
      hr[i] = make_uint4(0, 0, 0, 0);
    }
    if (t < a.T) {
      const uint4* p = reinterpret_cast<const uint4*>(xb + static_cast<size_t>(t) * C + spart * 32);
#pragma unroll
      for (int i = 0; i < 4; ++i) xr[i] = __ldg(p + i);
    }
    if (tid < 2 * TPR) {        // halo rows t0-1 (first TPR threads) and t0+TB (next TPR)
      const int th = tid < TPR ? t0 - 1 : t0 + TB;
      if (th >= 0 && th < a.T) {
        const uint4* p = reinterpret_cast<const uint4*>(xb + static_cast<size_t>(th) * C + (tid % TPR) * 32);
#pragma unroll
        for (int i = 0; i < 4; ++i) hr[i] = __ldg(p + i);
      }
    }
  };
  auto activate = [&](const uint4& u, int c8, bool valid) {   // channels c8 .. c8+7 of the part
    if (!valid) return make_uint4(0, 0, 0, 0);                // conv zero padding
    // coefficients of the thread's part from smem (all threads of a part read the same words)
    const float4 a0 = *reinterpret_cast<const float4*>(&s_ga[spart * 32 + c8]);
    const float4 a1 = *reinterpret_cast<const float4*>(&s_ga[spart * 32 + c8 + 4]);
    const float4 d0 = *reinterpret_cast<const float4*>(&s_de[spart * 32 + c8]);
    const float4 d1 = *reinterpret_cast<const float4*>(&s_de[spart * 32 + c8 + 4]);
    const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
    uint4 o;
    o.x = pack_bf16(silu_fast(f0.x * a0.x + d0.x), silu_fast(f0.y * a0.y + d0.y));
    o.y = pack_bf16(silu_fast(f1.x * a0.z + d0.z), silu_fast(f1.y * a0.w + d0.w));
    o.z = pack_bf16(silu_fast(f2.x * a1.x + d1.x), silu_fast(f2.y * a1.y + d1.y));
    o.w = pack_bf16(silu_fast(f3.x * a1.z + d1.z), silu_fast(f3.y * a1.w + d1.w));
    return o;
  };

  // statistics of the thread's 8 channels: two halves of 4 (a half never straddles a group)
  float st_s[2] = {0.f, 0.f}, st_q[2] = {0.f, 0.f};

  int tile = blockIdx.x;
  uint4 xr[4], hr[4];
  if (tile < n_tiles) load_tile(tile, xr, hr);
  const uint32_t w_base = smem_u32(s_w);
  const uint32_t x_base = smem_u32(s_x);
  for (; tile < n_tiles; tile += gridDim.x) {
    const int t0 = tile * TB;
    {
      const bool valid = t0 + srow < a.T;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<uint4*>(s_x + (srow + 1) * RS + spart * 64 + i * 16) = activate(xr[i], i * 8, valid);
      if (tid < 2 * TPR) {
        const int th = tid < TPR ? t0 - 1 : t0 + TB;
        const bool hv = th >= 0 && th < a.T;
        uint8_t* dst = s_x + (tid < TPR ? 0 : TB + 1) * RS + (tid % TPR) * 64;
        // the halo thread's part is (tid % TPR), whose coefficients this thread holds only if it
        // equals spart: true by construction (tid % TPR == spart)
#pragma unroll
        for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(dst + i * 16) = activate(hr[i], i * 8, hv);
      }
    }
    if (tile + gridDim.x < n_tiles) load_tile(tile + gridDim.x, xr, hr);   // prefetch
    // residual rows of this tile in the epilogue's mapping, in flight during the MMAs
    uint4 res[ER];
    if (has_res) {
#pragma unroll
      for (int i = 0; i < ER; ++i) {
        const int t = t0 + erow0 + i * (NTH / LPR);
        res[i] = make_uint4(0, 0, 0, 0);
        if (t < a.T) res[i] = __ldg(reinterpret_cast<const uint4*>(rb + static_cast<size_t>(t) * C + el * 8));
      }
    }
    __syncthreads();        // s_x complete; every thread has left the previous tile's epilogue (s_o)

    float acc[MB][NT][4];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb)
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        acc[mb][j][0] = s_bias[8 * j + 2 * q]; acc[mb][j][1] = s_bias[8 * j + 2 * q + 1];
        acc[mb][j][2] = acc[mb][j][0]; acc[mb][j][3] = acc[mb][j][1];
      }
#pragma unroll
    for (int tap = 0; tap < 3; ++tap) {
#pragma unroll
      for (int c16 = 0; c16 < C / 16; ++c16) {
        uint32_t af[MB][4];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
          const int r0 = warp * RPW + mb * 16;
          // matrices: (rows 0-7, k 0-7) (rows 8-15, k 0-7) (rows 0-7, k 8-15) (rows 8-15, k 8-15)
          ldsm_x4(x_base + static_cast<uint32_t>(r0 + (lane & 7) + ((lane >> 3) & 1) * 8 + tap) * RS +
                      (c16 * 16 + ((lane >> 4) & 1) * 8) * 2, af[mb]);
        }
#pragma unroll
        for (int np = 0; np < NT / 2; ++np) {
          uint32_t bf[4];
          // matrices: (n 0-7, k 0-7) (n 0-7, k 8-15) (n 8-15, k 0-7) (n 8-15, k 8-15)
          ldsm_x4(w_base + static_cast<uint32_t>(np * 16 + (lane & 7) + ((lane >> 4) & 1) * 8) * WS +
                      (tap * C + c16 * 16 + ((lane >> 3) & 1) * 8) * 2, bf);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) {
            mma_bf16_16816(acc[mb][2 * np], af[mb], bf[0], bf[1]);
            mma_bf16_16816(acc[mb][2 * np + 1], af[mb], bf[2], bf[3]);
          }
        }
      }
    }
    // accumulator fragments -> row-major fp32 tile: lane (g, q) owns rows g / g+8, channels 8j+2q, +1
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) {
      const int r = warp * RPW + mb * 16 + g;
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        *reinterpret_cast<float2*>(s_o + r * OS + 8 * j + 2 * q) = make_float2(acc[mb][j][0], acc[mb][j][1]);
        *reinterpret_cast<float2*>(s_o + (r + 8) * OS + 8 * j + 2 * q) = make_float2(acc[mb][j][2], acc[mb][j][3]);
      }
    }
    __syncthreads();        // s_o complete (and every warp is done reading s_x)

    // row-wise epilogue: this thread's 8 channels of ER rows
#pragma unroll
    for (int i = 0; i < ER; ++i) {
      const int rl = erow0 + i * (NTH / LPR);
      const int t = t0 + rl;
      const float4 o0 = *reinterpret_cast<const float4*>(s_o + rl * OS + el * 8);
      const float4 o1 = *reinterpret_cast<const float4*>(s_o + rl * OS + el * 8 + 4);
      float y[8] = {o0.x, o0.y, o0.z, o0.w, o1.x, o1.y, o1.z, o1.w};
      if (has_res) {
        const float2 r0 = unpack_bf16(res[i].x), r1 = unpack_bf16(res[i].y);
        const float2 r2 = unpack_bf16(res[i].z), r3 = unpack_bf16(res[i].w);
        y[0] += r0.x; y[1] += r0.y; y[2] += r1.x; y[3] += r1.y;
        y[4] += r2.x; y[5] += r2.y; y[6] += r3.x; y[7] += r3.y;
      }
      if (has_film) {   // following ModulationItem: LayerNorm over C (no affine) + FiLM
        float m = ((y[0] + y[1]) + (y[2] + y[3])) + ((y[4] + y[5]) + (y[6] + y[7]));
#pragma unroll
        for (int o = LPR >> 1; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
        m *= (1.f / C);
        float v = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) { y[j] -= m; v += y[j] * y[j]; }
#pragma unroll
        for (int o = LPR >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const float rstd = rsqrtf(v * (1.f / C) + a.ln_eps);
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = y[j] * rstd * fsc[j] + fsh[j];
      }
      uint4 ov;
      ov.x = pack_bf16(y[0], y[1]); ov.y = pack_bf16(y[2], y[3]);
      ov.z = pack_bf16(y[4], y[5]); ov.w = pack_bf16(y[6], y[7]);
      if (t < a.T) {
        *reinterpret_cast<uint4*>(yb + static_cast<size_t>(t) * C + el * 8) = ov;
        const float2 q0 = unpack_bf16(ov.x), q1 = unpack_bf16(ov.y);   // statistics of the ROUNDED values
        const float2 q2 = unpack_bf16(ov.z), q3 = unpack_bf16(ov.w);
        st_s[0] += (q0.x + q0.y) + (q1.x + q1.y);
        st_q[0] += (q0.x * q0.x + q0.y * q0.y) + (q1.x * q1.x + q1.y * q1.y);
        st_s[1] += (q2.x + q2.y) + (q3.x + q3.y);
        st_q[1] += (q2.x * q2.x + q2.y * q2.y) + (q3.x * q3.x + q3.y * q3.y);
      }
    }
  }
  if (a.stats_out) {
    const int gsz = C / a.groups;
    // lanes el, el+LPR, ... of a warp hold the same channels: fold, then one atomic per (warp, half)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) {
        st_s[hf] += __shfl_xor_sync(0xffffffffu, st_s[hf], o);
        st_q[hf] += __shfl_xor_sync(0xffffffffu, st_q[hf], o);
      }
      if (lane < LPR) {
        const int gi = (el * 8 + hf * 4) / gsz;
        atomicAdd(&s_stats[2 * gi], st_s[hf]);
        atomicAdd(&s_stats[2 * gi + 1], st_q[hf]);
      }
    }
    __syncthreads();
    if (tid < 2 * a.groups && s_stats[tid] != 0.f)
      atomicAdd(a.stats_out + static_cast<size_t>(b) * 2 * a.groups + tid, static_cast<double>(s_stats[tid]));
  }
}

template <int C>
static int launch_mid(const adp_narrow_conv_args& a, cudaStream_t stream) {
  using Cfg = MidCfg<C>;
  static SmemAttrCache smem_cache;
  ADP_CUDA(ensure_dyn_smem(mid_conv_kernel<C>, (size_t)Cfg::SMEM, smem_cache));
  int dev = 0, sms = 148, occ = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mid_conv_kernel<C>, Cfg::NTH, Cfg::SMEM) != cudaSuccess ||
      occ < 1)
    occ = 1;
  const int n_tiles = (a.T + Cfg::TB - 1) / Cfg::TB;
  int gx = (occ * sms) / a.B;               // one wave of persistent blocks
  if (gx < 1) gx = 1;
  if (gx > n_tiles) gx = n_tiles;
  ADP_CUDA(launch_k(mid_conv_kernel<C>, dim3(gx, a.B), dim3(Cfg::NTH), (size_t)Cfg::SMEM, stream, a));
  return 0;
}

int mid_conv(const adp_narrow_conv_args& a, cudaStream_t stream) {
  if (a.C == 32) return launch_mid<32>(a, stream);
  if (a.C == 64) return launch_mid<64>(a, stream);
  return set_error("adp_narrow_conv: C=%d is not built (8, 32, 64)", a.C);
}

}  // namespace adp
