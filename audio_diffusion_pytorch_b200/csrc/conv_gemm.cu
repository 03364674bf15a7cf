// adp_conv_gemm: persistent shifted-tap GEMM on tcgen05 (see include/adp_b200.h).
//
// GEMM view (swapped w.r.t. the usual conv-as-GEMM so that one accumulator ROW is one time
// position): D[m = time position, n = output channel] = sum_{tap,k} A[m + off(tap), k] * W[n, tap, k]
//   A: channels-last activations -> K-major operand.  ONE TMA box of (128 + span) rows per
//      64-channel chunk serves all taps: tap j is the same smem tile read through a UMMA
//      descriptor whose start address is advanced by j rows (the 128B swizzle is a function of
//      the absolute smem address, so row-shifted starts need no re-layout).  Rows outside
//      [0,T) are zero-filled by TMA = the conv's zero padding.
//   W: packed weights [N][taps*C_in] -> K-major operand.
//   A pipeline stage = KC chunks x {A box, one W box per tap} behind ONE full/empty mbarrier
//      pair, so the single-thread issue loops pay one barrier round trip per KC*taps*4 MMAs.
//   D: fp32 in TMEM, 128 lanes x BN columns, DOUBLE buffered: the epilogue of tile i drains
//      buffer i&1 while the MMAs of tile i+1 fill the other one.
// Persistent: each CTA owns a contiguous range of tiles (n fastest).  Warp roles (192 threads):
// warp 0 TMA producer + TMEM allocator, warp 1 MMA issuer, warps 2-5 epilogue (TMEM lane
// quarter = warp & 3).  The epilogue prefetches the residual rows of its tile into registers
// while the tile's MMAs still run, and keeps GroupNorm partial sums in thread-private smem
// slots (no shuffles / atomics per tile; one reduction per batch change).
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace adp {

// adp_debug_set(2, 1): the weights are not written by the preceding kernels, so the producer may
// fetch them before griddepcontrol.wait (set while an inference graph is captured)
int g_early_w = 0;

constexpr int kBM = 128;
constexpr int kMaxStages = 8;
constexpr int kMaxGroups = 8;      // GroupNorm groups handled by the fused statistics

struct Gemm2Params {
  __nv_bfloat16* out;
  const __nv_bfloat16* residual;
  const float* bias;
  const float* gate;
  double* stats;
  int B, T, tiles_per_batch, c_in, ldo;
  int n_pad, n_valid;
  int ntaps, tap_off0, up_factor;
  int groups, group_size, group_shift;   // group_shift >= 0: group = ch >> shift
  int out_fp32, ld_gate;
  int n_tiles_n, total_tiles, tiles_per_cta;
  int a_rows;            // rows per A box = 128 + tap span
  int kc;                // 64-channel chunks per stage
  int k_stages;          // stages per tile = (c_in / BK) / kc
  int n_stages;          // ring depth
  int a_sub_bytes, w_sub_bytes, stage_bytes, max_taps;
  int early_w;           // weights may be fetched before griddepcontrol.wait
};

struct TileInfo {
  int b, t0, n0, phase, ch0, ntaps, min_off;
};

__device__ __forceinline__ TileInfo tile_info(const Gemm2Params& p, int tile, int BN) {
  TileInfo ti;
  const int m_tile = tile / p.n_tiles_n;
  const int n_tile = tile - m_tile * p.n_tiles_n;
  ti.b = m_tile / p.tiles_per_batch;
  ti.t0 = (m_tile - ti.b * p.tiles_per_batch) * kBM;
  ti.n0 = n_tile * BN;
  ti.phase = ti.n0 / p.n_pad;
  ti.ch0 = ti.n0 - ti.phase * p.n_pad;
  if (p.up_factor > 1) {   // nearest-upsample + conv3: taps collapse per output phase
    if (ti.phase == 0) { ti.ntaps = 2; ti.min_off = -1; }
    else if (ti.phase == p.up_factor - 1) { ti.ntaps = 2; ti.min_off = 0; }
    else { ti.ntaps = 1; ti.min_off = 0; }
  } else {
    ti.ntaps = p.ntaps;
    ti.min_off = p.tap_off0;
  }
  return ti;
}

// thread-private GroupNorm partial sums: slot (value v of group g, epilogue thread et)
template <int NET>      // NET = epilogue threads per CTA
struct StatSlots {
  float* base;   // [2*kMaxGroups][NET]
  int et;
  int cur_g;
  float s, q;
  __device__ __forceinline__ void flush() {
    if (cur_g >= 0) {
      base[(2 * cur_g) * NET + et] += s;
      base[(2 * cur_g + 1) * NET + et] += q;
    }
    s = 0.f; q = 0.f;
  }
  __device__ __forceinline__ void add(float v, int g) {
    if (g != cur_g) { flush(); cur_g = g; }
    s += v; q += v * v;
  }
};

// GroupNorm partial sums for group sizes that are neither >= 8 nor 4 (never the case in the
// reference configurations): straight into the thread-private slots, one element at a time.
static __device__ __noinline__ void stats_generic(float* slots, int net, int et, int ch, int shift,
                                                  int gsize, float v0, float v1, float v2, float v3,
                                                  float v4, float v5, float v6, float v7) {
  const float v[8] = {v0, v1, v2, v3, v4, v5, v6, v7};
  for (int i = 0; i < 8; ++i) {
    const int g = shift >= 0 ? (ch + i) >> shift : (ch + i) / gsize;
    slots[(2 * g) * net + et] += v[i];
    slots[(2 * g + 1) * net + et] += v[i] * v[i];
  }
}

// EW = epilogue warps: 4 (one per TMEM lane quarter) or, for the long-K shapes that run one CTA
// per SM with <= one tile per CTA (nothing to overlap the drain with), 8: two warps per lane
// quarter, each draining half of the tile's columns.
template <int BN, int SW, int EW>
__global__ void __launch_bounds__(64 + 32 * EW, EW == 8 ? 1 : (BN <= 64 ? 3 : (BN <= 128 ? 2 : 1)))
conv_gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                  const Gemm2Params p) {
  constexpr int BK = SW / 2;
  constexpr int ACC_COLS = BN < 32 ? 32 : BN;     // TMEM columns per accumulator buffer
  constexpr int CH = BN < 32 ? 16 : 32;           // epilogue column chunk
  constexpr uint32_t kWTapBytes = BN * SW;        // bytes one W box writes
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
  __shared__ uint64_t acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;
  constexpr int NET = 32 * EW;                    // epilogue threads
  constexpr int BNW = BN / (EW / 4);              // columns drained by one epilogue warp
  static_assert(EW == 4 || BNW >= 32, "8 epilogue warps need >= 32 columns per warp");
  __shared__ float s_part[2 * kMaxGroups * NET];
  // per-tile bias / gate of the BN output columns, double buffered like the accumulators:
  // staged while the tile's MMAs run so the drain never waits on a global load
  __shared__ __align__(16) float s_bias[2][BN < 32 ? 32 : BN];
  __shared__ __align__(16) float s_gate[2][BN < 32 ? 32 : BN];

  pdl_launch_dependents();
  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* ring = smem_raw + ((1024u - (raw & 1023u)) & 1023u);

  const int tile_begin = blockIdx.x * p.tiles_per_cta;
  int tile_end = tile_begin + p.tiles_per_cta;
  if (tile_end > p.total_tiles) tile_end = p.total_tiles;

  for (int i = threadIdx.x; i < 2 * kMaxGroups * NET; i += blockDim.x) s_part[i] = 0.f;
  if (warp == 0) {
    tmem_alloc(&tmem_slot, 2 * ACC_COLS);
    tmem_relinquish();
  } else if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.n_stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], EW); }
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_slot, 0);   // warp-uniform for ptxas
  // Programmatic dependent launch: this kernel may have started while its predecessor still
  // runs.  Activations / statistics / conditioning come from the predecessor, so every role
  // that reads them calls griddepcontrol.wait first.  The WEIGHTS do not (p.early_w, set by the
  // host only while it captures an inference graph): the producer puts the weight boxes of the
  // first ring stages in flight BEFORE waiting, taking the first-load latency off the
  // critical path of the many short GEMMs that follow an elementwise kernel.
  if (warp == 0) {
    // ---------------------------------------------------------------------- TMA producer
    {
      const uint32_t a_bytes = static_cast<uint32_t>(p.a_rows) * SW;
      const int total_it = (tile_end - tile_begin) * p.k_stages;
      int early = 0;
      if (p.early_w) {
        early = total_it < p.n_stages ? total_it : p.n_stages;
        if (elect_one()) {
          int tile = tile_begin, ks = 0;
          for (int it = 0; it < early; ++it) {          // stage `it` of the (still empty) ring
            const TileInfo ti = tile_info(p, tile, BN);
            uint8_t* st = ring + it * p.stage_bytes;
            const uint32_t tx_it = static_cast<uint32_t>(p.kc) * (a_bytes + ti.ntaps * kWTapBytes);
            mbar_arrive_expect_tx(&full_bar[it], tx_it);
            for (int c = 0; c < p.kc; ++c) {
              const int k0 = (ks * p.kc + c) * BK;
              uint8_t* wdst = st + p.kc * p.a_sub_bytes + c * p.max_taps * p.w_sub_bytes;
              for (int tap = 0; tap < ti.ntaps; ++tap)
                tma_load_2d(wdst + tap * p.w_sub_bytes, &tmW, &full_bar[it], tap * p.c_in + k0, ti.n0);
            }
            if (++ks == p.k_stages) { ks = 0; ++tile; }
          }
        }
        __syncwarp();
      }
      pdl_wait();
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const TileInfo ti = tile_info(p, tile, BN);
        const uint32_t tx = static_cast<uint32_t>(p.kc) * (a_bytes + ti.ntaps * kWTapBytes);
        for (int ks = 0; ks < p.k_stages; ++ks, ++it) {
          const bool armed = it < early;                 // barrier armed + weights already issued
          if (!armed) mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* st = ring + s * p.stage_bytes;
          if (elect_one()) {
            if (!armed) mbar_arrive_expect_tx(&full_bar[s], tx);
            for (int c = 0; c < p.kc; ++c) {
              const int k0 = (ks * p.kc + c) * BK;
              tma_load_3d(st + c * p.a_sub_bytes, &tmA, &full_bar[s], k0, ti.t0 + ti.min_off, ti.b);
              if (armed) continue;
              uint8_t* wdst = st + p.kc * p.a_sub_bytes + c * p.max_taps * p.w_sub_bytes;
              for (int tap = 0; tap < ti.ntaps; ++tap)
                tma_load_2d(wdst + tap * p.w_sub_bytes, &tmW, &full_bar[s], tap * p.c_in + k0, ti.n0);
            }
          }
          __syncwarp();
          if (++s == p.n_stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16(kBM, BN, 0, 0);
    // descriptor of the ring base; byte offsets are added to the 14-bit address field
    const uint64_t desc0 = umma_desc_kmajor<SW>(smem_u32(ring));
    const uint32_t stage_u = static_cast<uint32_t>(p.stage_bytes) >> 4;
    const uint32_t a_sub_u = static_cast<uint32_t>(p.a_sub_bytes) >> 4;
    const uint32_t w_sub_u = static_cast<uint32_t>(p.w_sub_bytes) >> 4;
    const uint32_t w_base_u = static_cast<uint32_t>(p.kc) * a_sub_u;
    int s = 0;
    uint32_t ph = 0, j = 0;
    for (int tile = tile_begin; tile < tile_end; ++tile, ++j) {
      const TileInfo ti = tile_info(p, tile, BN);
      const uint32_t buf = j & 1;
      mbar_wait(&acc_empty[buf], ((j >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * ACC_COLS;
      uint32_t accumulate = 0;
      for (int ks = 0; ks < p.k_stages; ++ks) {
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        if (elect_one()) {        // ONE elected thread issues the whole stage and its commit
          const uint64_t sdesc = desc0 + static_cast<uint64_t>(s * stage_u);
          for (int c = 0; c < p.kc; ++c) {
            const uint64_t adesc = sdesc + c * a_sub_u;
            const uint64_t wdesc = sdesc + w_base_u + c * p.max_taps * w_sub_u;
            for (int tap = 0; tap < ti.ntaps; ++tap) {
#pragma unroll
              for (int kk = 0; kk < BK / 16; ++kk) {
                umma_bf16(d_tmem, adesc + ((tap * SW + kk * 32) >> 4),
                          wdesc + tap * w_sub_u + ((kk * 32) >> 4), idesc, accumulate);
                accumulate = 1;
              }
            }
          }
          umma_commit(&empty_bar[s]);
          if (ks == p.k_stages - 1) umma_commit(&acc_full[buf]);
        }
        accumulate = 1;
        __syncwarp();
        if (++s == p.n_stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp < 2 + EW) {
    // -------------------------------------------------------------------------- epilogue
    pdl_wait();
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const bool do_stats = p.stats != nullptr;
    const int et = threadIdx.x - 64;        // 0..NET-1 among epilogue threads
    const int cbeg = ((warp - 2) >> 2) * BNW;   // first tile column of this warp
    StatSlots<NET> acc{s_part, et, -1, 0.f, 0.f};
    int cur_b = -1;
    uint32_t j = 0;

    auto publish_stats = [&](int b_done) {   // all 128 epilogue threads
      acc.flush();
      acc.cur_g = -1;
      named_bar_sync(1, NET);
      for (int r2 = warp - 2; r2 < 2 * p.groups; r2 += EW) {     // one warp per row of slots
        const float* rowp = s_part + r2 * NET + lane;
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < EW; ++i) tot += rowp[32 * i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane == 0 && tot != 0.f)
          atomicAdd(p.stats + static_cast<size_t>(b_done) * 2 * p.groups + r2,
                    static_cast<double>(tot));
      }
      named_bar_sync(1, NET);
      for (int g2 = 0; g2 < 2 * p.groups; ++g2) s_part[g2 * NET + et] = 0.f;
    };

    for (int tile = tile_begin; tile < tile_end; ++tile, ++j) {
      const TileInfo ti = tile_info(p, tile, BN);
      const uint32_t buf = j & 1;
      const int t = ti.t0 + row;
      const bool row_ok = t < p.T;
      const size_t row_off = (static_cast<size_t>(ti.b) * p.T + (row_ok ? t : 0)) * p.ldo +
                             static_cast<size_t>(ti.phase) * p.n_valid;
      if (do_stats && ti.b != cur_b) {
        if (cur_b >= 0) publish_stats(cur_b);
        cur_b = ti.b;
      }
      // residual rows of this tile -> registers, while the tile's MMAs are still running
      uint4 res[BNW / 8];
      if (p.residual) {
#pragma unroll
        for (int i = 0; i < BNW / 8; ++i) {
          const int ch = ti.ch0 + cbeg + i * 8;
          res[i] = make_uint4(0, 0, 0, 0);
          if (row_ok && ch < p.n_valid)
            res[i] = __ldg(reinterpret_cast<const uint4*>(p.residual + row_off + ch));
        }
      }
      for (int c = et; c < BN; c += NET) {
        const int ch = ti.ch0 + c;
        const bool ok = ch < p.n_valid;
        s_bias[buf][c] = (p.bias && ok) ? __ldg(p.bias + ch) : 0.f;
        s_gate[buf][c] = (p.gate && ok) ? __ldg(p.gate + static_cast<size_t>(ti.b) * p.ld_gate + ch) : 1.f;
      }
      named_bar_sync(2, NET);     // staging visible to all epilogue warps
      mbar_wait(&acc_full[buf], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + buf * ACC_COLS + lane_addr;
      // Specialised drains for the shapes the network launches (bias, optional residual and
      // statistics with >= 8-channel groups, every column valid): the generic loop below pays
      // ~25 instructions of run-time flag tests per 8-channel vector, and the drain of a
      // short-K tile is issue/fetch bound.
      auto drain_fast = [&](auto res_c, auto st_c) {
        constexpr bool RES = decltype(res_c)::value;
        constexpr bool ST = decltype(st_c)::value;
#pragma unroll
        for (int cc = 0; cc < BNW; cc += CH) {
          const int c0 = cbeg + cc;
          uint32_t r[CH];
          if constexpr (CH == 16) tmem_ld16(taddr + c0, r);
          else tmem_ld32(taddr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int v8 = 0; v8 < CH / 8; ++v8) {
            const int ch = ti.ch0 + c0 + v8 * 8;
            const float4 b0 = *reinterpret_cast<const float4*>(&s_bias[buf][c0 + v8 * 8]);
            const float4 b1 = *reinterpret_cast<const float4*>(&s_bias[buf][c0 + v8 * 8 + 4]);
            float v[8];
            v[0] = __uint_as_float(r[v8 * 8 + 0]) + b0.x; v[1] = __uint_as_float(r[v8 * 8 + 1]) + b0.y;
            v[2] = __uint_as_float(r[v8 * 8 + 2]) + b0.z; v[3] = __uint_as_float(r[v8 * 8 + 3]) + b0.w;
            v[4] = __uint_as_float(r[v8 * 8 + 4]) + b1.x; v[5] = __uint_as_float(r[v8 * 8 + 5]) + b1.y;
            v[6] = __uint_as_float(r[v8 * 8 + 6]) + b1.z; v[7] = __uint_as_float(r[v8 * 8 + 7]) + b1.w;
            if constexpr (RES) {
              const uint4 rr = res[(cc + v8 * 8) / 8];
              const float2 r0 = unpack_bf16(rr.x), r1 = unpack_bf16(rr.y);
              const float2 r2 = unpack_bf16(rr.z), r3 = unpack_bf16(rr.w);
              v[0] += r0.x; v[1] += r0.y; v[2] += r1.x; v[3] += r1.y;
              v[4] += r2.x; v[5] += r2.y; v[6] += r3.x; v[7] += r3.y;
            }
            uint4 o;
            o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]);
            o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
            if (row_ok) {
              *reinterpret_cast<uint4*>(p.out + row_off + ch) = o;
              if constexpr (ST) {      // statistics of the ROUNDED values the next layer reads
                const float2 q0 = unpack_bf16(o.x), q1 = unpack_bf16(o.y);
                const float2 q2 = unpack_bf16(o.z), q3 = unpack_bf16(o.w);
                const float s8 = ((q0.x + q0.y) + (q1.x + q1.y)) + ((q2.x + q2.y) + (q3.x + q3.y));
                const float q8 = ((q0.x * q0.x + q0.y * q0.y) + (q1.x * q1.x + q1.y * q1.y)) +
                                 ((q2.x * q2.x + q2.y * q2.y) + (q3.x * q3.x + q3.y * q3.y));
                const int g = ch >> p.group_shift;
                if (g != acc.cur_g) { acc.flush(); acc.cur_g = g; }
                acc.s += s8; acc.q += q8;
              }
            }
          }
        }
      };
      const bool fast = !p.gate && !p.out_fp32 && ti.ch0 + cbeg + BNW <= p.n_valid &&
                        (!do_stats || p.group_shift >= 3);
      if (fast) {
        if (p.residual) {
          if (do_stats) drain_fast(std::true_type{}, std::true_type{});
          else drain_fast(std::true_type{}, std::false_type{});
        } else {
          if (do_stats) drain_fast(std::false_type{}, std::true_type{});
          else drain_fast(std::false_type{}, std::false_type{});
        }
      }
#pragma unroll
      for (int cc = 0; cc < BNW; cc += CH) {
        if (fast) break;
        const int c0 = cbeg + cc;
        uint32_t r[CH];
        if constexpr (CH == 16) tmem_ld16(taddr + c0, r);
        else tmem_ld32(taddr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int v8 = 0; v8 < CH / 8; ++v8) {
          const int ch = ti.ch0 + c0 + v8 * 8;
          if (ch >= p.n_valid) continue;           // padded columns (uniform)
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[v8 * 8 + i]);
          {
            const float4 b0 = *reinterpret_cast<const float4*>(&s_bias[buf][c0 + v8 * 8]);
            const float4 b1 = *reinterpret_cast<const float4*>(&s_bias[buf][c0 + v8 * 8 + 4]);
            v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
            v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
          }
          if (p.gate) {
            const float4 g0 = *reinterpret_cast<const float4*>(&s_gate[buf][c0 + v8 * 8]);
            const float4 g1 = *reinterpret_cast<const float4*>(&s_gate[buf][c0 + v8 * 8 + 4]);
            v[0] *= g0.x; v[1] *= g0.y; v[2] *= g0.z; v[3] *= g0.w;
            v[4] *= g1.x; v[5] *= g1.y; v[6] *= g1.z; v[7] *= g1.w;
          }
          if (p.out_fp32) {
            if (row_ok) {
              float* op = reinterpret_cast<float*>(p.out) + row_off + ch;
              *reinterpret_cast<float4*>(op) = make_float4(v[0], v[1], v[2], v[3]);
              *reinterpret_cast<float4*>(op + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
            continue;
          }
          if (row_ok) {
            if (p.residual) {
              const uint4 rr = res[(cc + v8 * 8) / 8];
              const float2 r0 = unpack_bf16(rr.x), r1 = unpack_bf16(rr.y);
              const float2 r2 = unpack_bf16(rr.z), r3 = unpack_bf16(rr.w);
              v[0] += r0.x; v[1] += r0.y; v[2] += r1.x; v[3] += r1.y;
              v[4] += r2.x; v[5] += r2.y; v[6] += r3.x; v[7] += r3.y;
            }
            uint4 o;
            o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]);
            o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
            *reinterpret_cast<uint4*>(p.out + row_off + ch) = o;
            if (do_stats) {  // statistics of the ROUNDED values the next layer will read
              const float2 q0 = unpack_bf16(o.x), q1 = unpack_bf16(o.y);
              const float2 q2 = unpack_bf16(o.z), q3 = unpack_bf16(o.w);
              v[0] = q0.x; v[1] = q0.y; v[2] = q1.x; v[3] = q1.y;
              v[4] = q2.x; v[5] = q2.y; v[6] = q3.x; v[7] = q3.y;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.f;
          }
          if (do_stats) {
            if (p.group_shift >= 3) {          // the whole 8-vector lies in one group
              float s8 = 0.f, q8 = 0.f;
#pragma unroll
              for (int i = 0; i < 8; ++i) { s8 += v[i]; q8 += v[i] * v[i]; }
              const int g = ch >> p.group_shift;
              if (g != acc.cur_g) { acc.flush(); acc.cur_g = g; }
              acc.s += s8; acc.q += q8;
            } else if (p.group_shift == 2) {   // 4-channel groups: the vector spans g and g + 1
              const int g = ch >> 2;
              float* lo = s_part + (2 * g) * NET + et;
              lo[0] += (v[0] + v[1]) + (v[2] + v[3]);
              lo[NET] += (v[0] * v[0] + v[1] * v[1]) + (v[2] * v[2] + v[3] * v[3]);
              lo[2 * NET] += (v[4] + v[5]) + (v[6] + v[7]);
              lo[3 * NET] += (v[4] * v[4] + v[5] * v[5]) + (v[6] * v[6] + v[7] * v[7]);
            } else {
              // rare group sizes: out of line, or this code is unrolled BN/8 times into the
              // drain loop and the epilogue stalls on instruction fetch
              stats_generic(s_part, NET, et, ch, p.group_shift, p.group_size, v[0], v[1], v[2], v[3],
                            v[4], v[5], v[6], v[7]);
            }
          }
        }
      }
      // accumulator buffer drained -> hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
    if (do_stats && cur_b >= 0) publish_stats(cur_b);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem_base, 2 * ACC_COLS);
  }
}

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// EW = 4 picks the CTAs per SM from the shape and may hand over to the 8-drain-warp variant,
// which always runs one CTA per SM.
template <int BN, int SW, int EW = 4>
static int launch_gemm2(const adp_conv_gemm_args& a, cudaStream_t stream) {
  constexpr int BK = SW / 2;
  const int tiles_per_batch = (a.T + kBM - 1) / kBM;
  const bool up = a.up_factor > 1;
  const int max_taps = up ? 2 : a.ntaps;
  const int span = up ? 1 : a.ntaps - 1;
  const int a_rows = kBM + span;
  const int k_chunks = a.c_in / BK;

  Gemm2Params p;
  p.a_sub_bytes = (a_rows * SW + 1023) / 1024 * 1024;
  p.w_sub_bytes = (BN * SW + 1023) / 1024 * 1024;
  p.max_taps = max_taps;
  const int chunk_bytes = p.a_sub_bytes + max_taps * p.w_sub_bytes;

  auto budget_of = [](int o) {
    return (o == 1 ? (EW == 8 ? 204 : 196) : (o == 2 ? 96 : 60)) * 1024;   // 227 KB - static - 1 KB
  };  // <= 11 KB static smem/CTA
  // CTAs per SM: the epilogue (4 warps per CTA) is the critical resource of short-K tiles, so
  // those run 2-3 CTAs per SM; long-K tiles want deep rings of fat stages instead.
  int occ = 1;
  if constexpr (EW == 4) {
    const int w_iters = k_chunks * max_taps;
    if (BN <= 64 && w_iters <= 8) occ = 3;
    else if (BN <= 128 && w_iters <= 12) occ = 2;
    const int tmem_occ = 512 / (2 * (BN < 32 ? 32 : BN));
    if (occ > tmem_occ) occ = tmem_occ;
    while (occ > 1 && budget_of(occ) < 2 * chunk_bytes) --occ;   // need >= 2 stages in the ring
    if constexpr (BN >= 64) {
      // at most ~two tiles per SM: little or nothing overlaps the drain -> one CTA per SM with
      // 8 drain warps (also when 2 CTAs/SM were possible but every SM gets <= one tile anyway)
      const long total = (long)a.B * tiles_per_batch * (a.phases * a.n_pad / BN);
      if ((occ == 1 && total <= 2L * num_sms()) || total <= (long)num_sms())
        return launch_gemm2<BN, SW, 8>(a, stream);
    }
  }
  const int budget = budget_of(occ);
  // chunks per stage: amortise one mbarrier round trip over >= 8 MMAs where smem allows
  int kc = 1;
  while (kc * 2 <= 4 && k_chunks % (kc * 2) == 0 && kc * max_taps * (BK / 16) < 8 &&
         2 * (kc * 2) * chunk_bytes <= budget)
    kc *= 2;
  p.kc = kc;
  p.k_stages = k_chunks / kc;
  p.stage_bytes = kc * chunk_bytes;
  int n_stages = budget / p.stage_bytes;
  if (n_stages > kMaxStages) n_stages = kMaxStages;
  if (n_stages < 2)
    return set_error("adp_conv_gemm: stage of %d bytes does not fit (BN=%d)", p.stage_bytes, BN);
  p.n_stages = n_stages;
  const size_t smem = static_cast<size_t>(n_stages) * p.stage_bytes + 1024;

  CUtensorMap tmA, tmW;
  {
    const uint64_t dims[3] = {(uint64_t)a.c_in, (uint64_t)a.T, (uint64_t)a.B};
    const uint64_t strides[2] = {(uint64_t)a.lda * 2, (uint64_t)a.T * a.lda * 2};
    const uint32_t box[3] = {(uint32_t)BK, (uint32_t)a_rows, 1};
    if (int e = make_tmap_bf16(&tmA, a.a, 3, dims, strides, box, SW)) return e;
  }
  {
    const uint64_t dims[2] = {(uint64_t)a.k_total, (uint64_t)a.phases * a.n_pad};
    const uint64_t strides[1] = {(uint64_t)a.k_total * 2};
    const uint32_t box[2] = {(uint32_t)BK, (uint32_t)BN};
    if (int e = make_tmap_bf16(&tmW, a.w, 2, dims, strides, box, SW)) return e;
  }

  static SmemAttrCache smem_cache;
  ADP_CUDA(ensure_dyn_smem(conv_gemm2_kernel<BN, SW, EW>, smem, smem_cache));

  p.out = static_cast<__nv_bfloat16*>(a.out);
  p.residual = static_cast<const __nv_bfloat16*>(a.residual);
  p.bias = a.bias;
  p.gate = a.gate;
  p.stats = a.stats;
  p.B = a.B;
  p.T = a.T;
  p.tiles_per_batch = tiles_per_batch;
  p.c_in = a.c_in;
  p.ldo = a.ldo;
  p.n_pad = a.n_pad;
  p.n_valid = a.n_valid;
  p.ntaps = a.ntaps;
  p.tap_off0 = a.tap_off[0];
  p.up_factor = a.up_factor;
  p.groups = a.stats ? a.groups : 0;
  p.group_size = a.stats ? a.n_valid / a.groups : 1;
  p.group_shift = -1;
  for (int sft = 0; sft < 16; ++sft)
    if ((1 << sft) == p.group_size) p.group_shift = sft;
  p.out_fp32 = a.out_fp32;
  p.ld_gate = a.ld_gate > 0 ? a.ld_gate : a.n_valid;
  p.n_tiles_n = a.phases * a.n_pad / BN;
  p.total_tiles = a.B * tiles_per_batch * p.n_tiles_n;
  p.a_rows = a_rows;
  p.early_w = g_early_w;

  const int slots = occ * num_sms();
  int grid = p.total_tiles < slots ? p.total_tiles : slots;
  p.tiles_per_cta = (p.total_tiles + grid - 1) / grid;
  grid = (p.total_tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  ADP_CUDA(launch_k(conv_gemm2_kernel<BN, SW, EW>, dim3(grid), dim3(64 + 32 * EW), smem, stream, tmA, tmW, p));
  ADP_LAUNCH_CHECK();
  return 0;
}

template <int SW>
static int dispatch_bn2(const adp_conv_gemm_args& a, int bn, cudaStream_t s) {
  switch (bn) {
    case 16: return launch_gemm2<16, SW>(a, s);
    case 32: return launch_gemm2<32, SW>(a, s);
    case 64: return launch_gemm2<64, SW>(a, s);
    case 128: return launch_gemm2<128, SW>(a, s);
    case 256: return launch_gemm2<256, SW>(a, s);
  }
  return set_error("adp_conv_gemm: unsupported N tile %d", bn);
}

}  // namespace adp

extern "C" int adp_debug_set(int key, int value) {
  switch (key) {
    case 2: adp::g_early_w = value; return 0;
    case 6: adp::g_pdl = value; return 0;
  }
  return adp::set_error("adp_debug_set: bad key %d (2 = early weight fetch, 6 = PDL)", key);
}

extern "C" int adp_conv_gemm(const adp_conv_gemm_args* args, adp_stream_t stream) {
  using namespace adp;
  ADP_CHECK(args != nullptr, "adp_conv_gemm: null args");
  const adp_conv_gemm_args& a = *args;
  ADP_CHECK(a.a && a.w && a.out, "adp_conv_gemm: null a/w/out");
  ADP_CHECK(a.B > 0 && a.T > 0, "adp_conv_gemm: bad B=%d T=%d", a.B, a.T);
  ADP_CHECK(a.c_in >= 16 && a.c_in % 16 == 0, "adp_conv_gemm: c_in=%d must be a multiple of 16",
            a.c_in);
  ADP_CHECK(a.lda % 8 == 0 && a.ldo % 8 == 0 && a.k_total % 8 == 0 && a.lda >= a.c_in,
            "adp_conv_gemm: pitches lda=%d ldo=%d k_total=%d must be multiples of 8", a.lda, a.ldo,
            a.k_total);
  ADP_CHECK(a.n_valid > 0 && a.n_valid % 8 == 0 && a.n_valid <= a.n_pad && a.n_pad % 16 == 0,
            "adp_conv_gemm: n_valid=%d n_pad=%d", a.n_valid, a.n_pad);
  ADP_CHECK(a.phases >= 1, "adp_conv_gemm: phases=%d", a.phases);
  ADP_CHECK(a.ld_gate % 4 == 0, "adp_conv_gemm: ld_gate=%d must be a multiple of 4", a.ld_gate);
  if (a.up_factor > 1) {
    ADP_CHECK(a.phases == a.up_factor, "adp_conv_gemm: phases (%d) != up_factor (%d)", a.phases,
              a.up_factor);
    ADP_CHECK(a.k_total >= 2 * a.c_in, "adp_conv_gemm: upsample weights need 2 tap slots");
  } else {
    ADP_CHECK(a.ntaps >= 1 && a.ntaps <= 3 && a.phases == 1, "adp_conv_gemm: ntaps=%d phases=%d",
              a.ntaps, a.phases);
    ADP_CHECK(a.k_total >= a.ntaps * a.c_in, "adp_conv_gemm: k_total too small");
    for (int i = 1; i < a.ntaps; ++i)
      ADP_CHECK(a.tap_off[i] == a.tap_off[i - 1] + 1,
                "adp_conv_gemm: tap offsets must be consecutive and ascending");
  }
  if (a.out_fp32) {
    ADP_CHECK(!a.residual && !a.stats, "adp_conv_gemm: out_fp32 excludes residual/stats");
  }
  if (a.stats) {
    ADP_CHECK(a.groups > 0 && a.groups <= kMaxGroups && a.n_valid % a.groups == 0,
              "adp_conv_gemm: groups=%d n_valid=%d (fused statistics handle <= %d groups)",
              a.groups, a.n_valid, kMaxGroups);
  }
  // N tile: persistent CTAs take care of SM fill; prefer 128 (W traffic dominates either way
  // and two accumulator buffers of 128 columns leave room for 2 CTAs/SM on short-K shapes)
  int bn = a.block_n;
  if (bn == 0) {
    const long m_tiles = (long)a.B * ((a.T + kBM - 1) / kBM);
    bn = 16;
    for (int cand = 128; cand >= 16; cand >>= 1) {
      if (a.n_pad % cand) continue;
      const long tiles = m_tiles * (a.phases * a.n_pad / cand);
      if (tiles >= 96 || cand <= 64) { bn = cand; break; }
    }
  }
  ADP_CHECK(a.n_pad % bn == 0, "adp_conv_gemm: N tile %d does not divide n_pad %d", bn, a.n_pad);
  cudaStream_t s = as_stream(stream);
  if (a.c_in % 64 == 0) return dispatch_bn2<128>(a, bn, s);
  if (a.c_in % 32 == 0) return dispatch_bn2<64>(a, bn, s);
  return dispatch_bn2<32>(a, bn, s);
}
