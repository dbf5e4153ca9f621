// Row-wise HBM-bound kernels of the conformer trunk on the packed [M, 512] layout:
//   K-ln        nn.LayerNorm(512, eps 1e-5)                       Gconform.py:57-63 (norm1..norm5)
//   K-boundhead norm5 + cutheard Linear(512, 1) + sigmoid         Gconform.py:63,135,137-138
//   K-dwconv    depthwise Conv1d(k=31, pad 15) + BatchNorm1d(eval) + SiLU, per-clip zero halo
//                                                                 base_conv.py:66-68
// Roofline: HBM.  LN reads 2 KB and writes 1-3 KB per row; dwconv reads/writes 1 KB + 1 KB per row.
#include "host_common.h"
#include "sm100_ptx.cuh"

#include "../../include/some_b200.h"

namespace some {

constexpr int D = SOME_DIM;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct LnParams {
  const float* x[2];
  const float* gamma[2];
  const float* beta[2];
  __nv_bfloat16* out_bf16[2];
  float* out_f32[2];
  int M;
};

// one warp per row: lane holds columns {128 i + 4 lane .. +3}, i < 4 (coalesced float4)
__device__ __forceinline__ void ln_load(const float* __restrict__ xr, int lane, float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float4 t = *reinterpret_cast<const float4*>(xr + 128 * i + 4 * lane);
    v[4 * i] = t.x, v[4 * i + 1] = t.y, v[4 * i + 2] = t.z, v[4 * i + 3] = t.w;
  }
}
__device__ __forceinline__ void ln_normalise(const float (&v)[16], const float* __restrict__ gamma,
                                             const float* __restrict__ beta, int lane, float (&y)[16]) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += v[i];
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float d = v[i] - mean;
    q = fmaf(d, d, q);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + 1e-5f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + 128 * i + 4 * lane));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + 128 * i + 4 * lane));
    y[4 * i + 0] = fmaf((v[4 * i + 0] - mean) * rstd, g.x, b.x);
    y[4 * i + 1] = fmaf((v[4 * i + 1] - mean) * rstd, g.y, b.y);
    y[4 * i + 2] = fmaf((v[4 * i + 2] - mean) * rstd, g.z, b.z);
    y[4 * i + 3] = fmaf((v[4 * i + 3] - mean) * rstd, g.w, b.w);
  }
}
__device__ __forceinline__ void ln_row(const float* __restrict__ xr, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, int lane, float (&y)[16]) {
  float v[16];
  ln_load(xr, lane, v);
  ln_normalise(v, gamma, beta, lane, y);
}
__device__ __forceinline__ void ln_store(const LnParams& p, int grp, int row, int lane, const float (&y)[16]) {
  if (p.out_f32[grp] != nullptr) {
    float* o = p.out_f32[grp] + (size_t)row * D;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(o + 128 * i + 4 * lane) = make_float4(y[4 * i], y[4 * i + 1], y[4 * i + 2], y[4 * i + 3]);
  }
  if (p.out_bf16[grp] != nullptr) {
    __nv_bfloat16* o = p.out_bf16[grp] + (size_t)row * D;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<uint2*>(o + 128 * i + 4 * lane) =
          make_uint2(pack_bf16x2(y[4 * i], y[4 * i + 1]), pack_bf16x2(y[4 * i + 2], y[4 * i + 3]));
  }
}

// Each warp streams LN_RPW rows per pass with all their loads issued up front (128 B per lane in flight): the kernel is a
// pure HBM stream and memory-level parallelism is what sets its bandwidth.
constexpr int LN_RPW = 2;
__global__ void __launch_bounds__(256) layernorm_kernel(const LnParams p) {
  const int grp = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * LN_RPW;
  griddep_launch();   // programmatic dependent launch (host_common.h)
  griddep_wait();
  if (row0 >= p.M) return;
  float v[LN_RPW][16];
#pragma unroll
  for (int r = 0; r < LN_RPW; ++r)
    if (row0 + r < p.M) ln_load(p.x[grp] + (size_t)(row0 + r) * D, lane, v[r]);
#pragma unroll
  for (int r = 0; r < LN_RPW; ++r) {
    if (row0 + r < p.M) {
      float y[16];
      ln_normalise(v[r], p.gamma[grp], p.beta[grp], lane, y);
      ln_store(p, grp, row0 + r, lane, y);
    }
  }
}

// K-rowstats: bf16(x) and the full-row (sum x, sum x^2) in slot 0 of ln_stats, for a residual stream that no producer GEMM
// has written yet (the input projection in front of block 0): the LayerNorm-folded consumer GEMMs then treat it like any
// other producer output (some_gemm, SOME_EPI_LN_*; ln_parts = 1).  Same streaming structure as layernorm_kernel.
struct RowStatsParams {
  const float* x[2];
  __nv_bfloat16* out_bf16[2];
  float* stats[2];
  int M;
};
__global__ void __launch_bounds__(256) row_stats_kernel(const RowStatsParams p) {
  const int grp = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * LN_RPW;
  if (row0 >= p.M) return;
  float v[LN_RPW][16];
#pragma unroll
  for (int r = 0; r < LN_RPW; ++r)
    if (row0 + r < p.M) ln_load(p.x[grp] + (size_t)(row0 + r) * D, lane, v[r]);
#pragma unroll
  for (int r = 0; r < LN_RPW; ++r) {
    if (row0 + r < p.M) {
      float s = 0.f, q = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        s += v[r][i];
        q = fmaf(v[r][i], v[r][i], q);
      }
      s = warp_sum(s);
      q = warp_sum(q);
      __nv_bfloat16* o = p.out_bf16[grp] + (size_t)(row0 + r) * D;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<uint2*>(o + 128 * i + 4 * lane) =
            make_uint2(pack_bf16x2(v[r][4 * i], v[r][4 * i + 1]), pack_bf16x2(v[r][4 * i + 2], v[r][4 * i + 3]));
      if (lane == 0)
        reinterpret_cast<float2*>(p.stats[grp])[(size_t)(row0 + r) * SOME_LN_SLOTS] = make_float2(s, q);
    }
  }
}

// K-colmeans (calibration only, load time): column means of a GEMM's (effective) A operand.  A block owns 128 columns; its
// 8 thread rows stride over the rows and their partial sums are added in a fixed order, so the means (and the bias
// corrections derived from them) are the same in every run.
__global__ void __launch_bounds__(128 * 8)
col_means_kernel(const __nv_bfloat16* __restrict__ a, int M, int K, int lda, const float* __restrict__ stats, int parts,
                 float inv_m, float* __restrict__ out) {
  __shared__ float part[8][128];
  const int k = blockIdx.x * 128 + threadIdx.x;
  float acc = 0.f;
  for (int row = threadIdx.y; row < M && k < K; row += 8) {
    float v = __bfloat162float(a[(size_t)row * lda + k]);
    if (stats != nullptr) {
      float s = 0.f, q = 0.f;
      const float2* st = reinterpret_cast<const float2*>(stats) + (size_t)row * SOME_LN_SLOTS;
      for (int i = 0; i < parts; ++i) s += st[i].x, q += st[i].y;
      const float mean = s / K;
      const float var = fmaxf(q / K - mean * mean, 0.f);
      v = (v - mean) * rsqrtf(var + 1e-5f);
    }
    acc += v;
  }
  part[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && k < K) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += part[i][threadIdx.x];
    out[k] = s * inv_m;
  }
}

__global__ void __launch_bounds__(256)
bound_head_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                  const float* __restrict__ w, float bias, int M, float* __restrict__ bounds) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  griddep_launch();
  griddep_wait();
  if (row >= M) return;
  float y[16];
  ln_row(x + (size_t)row * D, gamma, beta, lane, y);
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 ww = __ldg(reinterpret_cast<const float4*>(w + 128 * i + 4 * lane));
    dot = fmaf(y[4 * i], ww.x, dot);
    dot = fmaf(y[4 * i + 1], ww.y, dot);
    dot = fmaf(y[4 * i + 2], ww.z, dot);
    dot = fmaf(y[4 * i + 3], ww.w, dot);
  }
  dot = warp_sum(dot) + bias;
  if (lane == 0) bounds[row] = 1.0f / (1.0f + expf(-dot));
}

// ---------------------------------------------------------------------------------------------------
// Depthwise conv.  Work item = one 128-frame tile of one clip x 64 channels (tiles never span clips; frames outside
// the clip read as zero).  Persistent CTAs: a CTA keeps ONE channel block for its whole life, so the 31 x 2 BN-folded
// taps of each thread are loaded into registers once, and it walks over frame tiles with a cp.async double buffer
// (the (128 + 30) x 64 bf16 window of the next tile streams in while the current one is computed).  Each thread owns a
// channel pair and 16 consecutive frames: 16 packed-f32x2 accumulators, the 46 input rows stream through once
// (row-major accumulation, fully unrolled, no per-tap predicates).
constexpr int DW_T = 128;     // frames per tile
constexpr int DW_C = 64;      // channels per CTA
constexpr int DW_FR = 16;     // frames per thread
constexpr int DW_HALO = 15;
constexpr int DW_ROWS = DW_T + 2 * DW_HALO;
constexpr int DW_TILE_BYTES = DW_ROWS * DW_C * 2;

struct DwParams {
  const __nv_bfloat16* x[2];
  const float* w[2];  // [31][512]
  const float* b[2];  // [512]
  __nv_bfloat16* out[2];
  const int32_t* cu_frames;
  int tiles_per_clip;
  int num_tiles;      // tiles_per_clip * B
  int ctas_per_cb;    // CTAs sharing one (channel block, group)
};

__global__ void __launch_bounds__(256) dwconv_kernel(const DwParams p) {
  __shared__ __align__(16) __nv_bfloat16 tile[2][DW_ROWS * DW_C];
  const int grp = blockIdx.z;
  const int c0 = blockIdx.y * DW_C;
  const __nv_bfloat16* __restrict__ x = p.x[grp];
  __nv_bfloat16* __restrict__ out = p.out[grp];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = c0 + 2 * lane;

  auto tile_rows = [&](int t, int& clip_begin, int& clip_end, int& row0) -> bool {
    const int clip = t / p.tiles_per_clip;
    clip_begin = p.cu_frames[clip];
    clip_end = p.cu_frames[clip + 1];
    row0 = clip_begin + (t - clip * p.tiles_per_clip) * DW_T;
    return row0 < clip_end;
  };
  auto prefetch = [&](int t, int buf) {  // rows [row0 - 15, row0 + 128 + 15) x 64 channels, 8 x 16 B per row
    int clip_begin, clip_end, row0;
    if (!tile_rows(t, clip_begin, clip_end, row0)) return;
    const uint32_t dst0 = smem_u32(&tile[buf][0]);
    for (int i = threadIdx.x; i < DW_ROWS * 8; i += 256) {
      const int r = i >> 3, ch = i & 7;
      const int grow = row0 - DW_HALO + r;
      const bool ok = grow >= clip_begin && grow < clip_end;
      const int sz = ok ? 16 : 0;  // src-size 0 => zero fill (the per-clip zero padding of the conv)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (r * DW_C + ch * 8) * 2),
                   "l"(x + (size_t)(ok ? grow : clip_begin) * D + c0 + ch * 8), "r"(sz)
                   : "memory");
    }
  };

  // Packed fp32x2 FMAs (sm_100 FFMA2): {a[c], a[c+1]} += {w[c], w[c+1]} * {x[c], x[c+1]} in ONE instruction per lane.
  uint64_t w[SOME_CONV_K];
#pragma unroll
  for (int k = 0; k < SOME_CONV_K; ++k) w[k] = __ldg(reinterpret_cast<const unsigned long long*>(p.w[grp] + k * D + c));
  const uint64_t bb = __ldg(reinterpret_cast<const unsigned long long*>(p.b[grp] + c));
  griddep_launch();   // programmatic dependent launch: the taps (weights) are loaded, activations only after the wait
  griddep_wait();

  int t = blockIdx.x, buf = 0;
  if (t < p.num_tiles) prefetch(t, 0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (; t < p.num_tiles; t += p.ctas_per_cb, buf ^= 1) {
    if (t + p.ctas_per_cb < p.num_tiles) prefetch(t + p.ctas_per_cb, buf ^ 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();
    int clip_begin, clip_end, row0;
    if (tile_rows(t, clip_begin, clip_end, row0)) {
      uint64_t a[DW_FR];
#pragma unroll
      for (int f = 0; f < DW_FR; ++f) a[f] = bb;
      const int f0 = warp * DW_FR;  // first output frame (tile-relative) of this thread
      const __nv_bfloat16* tb = &tile[buf][0];
#pragma unroll
      for (int r = 0; r < DW_FR + SOME_CONV_K - 1; ++r) {
        const uint32_t xb = *reinterpret_cast<const uint32_t*>(tb + (f0 + r) * DW_C + 2 * lane);  // bf16x2
        // bf16 -> f32 is a 16-bit shift: {lo, hi} as packed f32x2
        const uint64_t xv = (static_cast<uint64_t>(xb & 0xffff0000u) << 32) | static_cast<uint64_t>(xb << 16);
#pragma unroll
        for (int f = 0; f < DW_FR; ++f) {
          const int k = r - f;  // tap index: output frame f reads tile rows f .. f + 30
          if (k >= 0 && k < SOME_CONV_K) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a[f]) : "l"(w[k]), "l"(xv));
        }
      }
#pragma unroll
      for (int f = 0; f < DW_FR; ++f) {
        const int grow = row0 + f0 + f;
        if (grow < clip_end) {
          const float a0 = __uint_as_float(static_cast<uint32_t>(a[f])), a1 = __uint_as_float(static_cast<uint32_t>(a[f] >> 32));
          *reinterpret_cast<uint32_t*>(out + (size_t)grow * D + c) = pack_bf16x2(silu_fast(a0), silu_fast(a1));
        }
      }
    }
    __syncthreads();  // everyone is done with tile[buf] before the prefetch of the iteration after next refills it
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

}  // namespace some

using namespace some;

extern "C" int some_layernorm(const some_ln_args* a, cudaStream_t stream) {
  SOME_REQUIRE(a != nullptr && (a->groups == 1 || a->groups == 2), "some_layernorm: bad args");
  if (a->M <= 0) return 0;
  LnParams p;
  for (int g = 0; g < 2; ++g) {
    const int s = g < a->groups ? g : 0;
    SOME_REQUIRE(a->x[s] && a->gamma[s] && a->beta[s], "some_layernorm: null input in group %d", s);
    SOME_REQUIRE(a->out_bf16[s] || a->out_f32[s], "some_layernorm: no output in group %d", s);
    p.x[g] = a->x[s], p.gamma[g] = a->gamma[s], p.beta[g] = a->beta[s];
    p.out_bf16[g] = reinterpret_cast<__nv_bfloat16*>(a->out_bf16[s]);
    p.out_f32[g] = a->out_f32[s];
  }
  p.M = a->M;
  dim3 grid((a->M + 8 * LN_RPW - 1) / (8 * LN_RPW), a->groups);
  launch_pdl(layernorm_kernel, grid, dim3(256), 0, stream, p);
  return check_launch("some_layernorm");
}

extern "C" int some_row_stats(const some_rowstats_args* a, cudaStream_t stream) {
  SOME_REQUIRE(a != nullptr && (a->groups == 1 || a->groups == 2), "some_row_stats: bad args");
  if (a->M <= 0) return 0;
  RowStatsParams p;
  for (int g = 0; g < 2; ++g) {
    const int s = g < a->groups ? g : 0;
    SOME_REQUIRE(a->x[s] && a->out_bf16[s] && a->ln_stats[s], "some_row_stats: null pointer in group %d", s);
    p.x[g] = a->x[s];
    p.out_bf16[g] = reinterpret_cast<__nv_bfloat16*>(a->out_bf16[s]);
    p.stats[g] = a->ln_stats[s];
  }
  p.M = a->M;
  dim3 grid((a->M + 8 * LN_RPW - 1) / (8 * LN_RPW), a->groups);
  row_stats_kernel<<<grid, 256, 0, stream>>>(p);
  return check_launch("some_row_stats");
}

extern "C" int some_col_means(const uint16_t* a, int M, int K, int lda, const float* ln_stats, int ln_parts, float* out,
                              cudaStream_t stream) {
  SOME_REQUIRE(a != nullptr && out != nullptr && M > 0 && K > 0 && K <= SOME_CALIB_K, "some_col_means: bad arguments");
  SOME_REQUIRE(ln_stats == nullptr || (ln_parts >= 1 && ln_parts <= SOME_LN_SLOTS), "some_col_means: bad ln_parts");
  col_means_kernel<<<(K + 127) / 128, dim3(128, 8), 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(a), M, K, lda,
                                                                  ln_stats, ln_parts, 1.0f / M, out);
  return check_launch("some_col_means");
}

extern "C" int some_bound_head(const float* x, const float* gamma, const float* beta, const float* w, float bias,
                               int M, float* bounds, cudaStream_t stream) {
  SOME_REQUIRE(x && gamma && beta && w && bounds, "some_bound_head: null pointer");
  if (M <= 0) return 0;
  launch_pdl(bound_head_kernel, dim3((M + 7) / 8), dim3(256), 0, stream, x, gamma, beta, w, bias, M, bounds);
  return check_launch("some_bound_head");
}

extern "C" int some_dwconv_bn_silu(const some_dwconv_args* a, cudaStream_t stream) {
  SOME_REQUIRE(a != nullptr && (a->groups == 1 || a->groups == 2), "some_dwconv_bn_silu: bad args");
  if (a->B <= 0 || a->max_frames <= 0) return 0;
  SOME_REQUIRE(a->cu_frames != nullptr, "some_dwconv_bn_silu: null cu_frames");
  DwParams p;
  for (int g = 0; g < 2; ++g) {
    const int s = g < a->groups ? g : 0;
    SOME_REQUIRE(a->x[s] && a->w[s] && a->b[s] && a->out[s], "some_dwconv_bn_silu: null pointer in group %d", s);
    p.x[g] = reinterpret_cast<const __nv_bfloat16*>(a->x[s]);
    p.w[g] = a->w[s], p.b[g] = a->b[s];
    p.out[g] = reinterpret_cast<__nv_bfloat16*>(a->out[s]);
  }
  p.cu_frames = a->cu_frames;
  p.tiles_per_clip = (a->max_frames + DW_T - 1) / DW_T;
  const long long nt = 1ll * p.tiles_per_clip * a->B;
  SOME_REQUIRE(nt < (1ll << 31), "some_dwconv_bn_silu: too many tiles");
  p.num_tiles = static_cast<int>(nt);
  // persistent grid: 2 CTAs per SM in total (register-limited occupancy), split evenly over the (channel block, group) pairs
  int per_cb = (2 * num_sms()) / ((D / DW_C) * a->groups);   // floor: every CTA resident in the first (only) wave
  if (per_cb < 1) per_cb = 1;
  p.ctas_per_cb = static_cast<int>(nt < per_cb ? nt : per_cb);
  dim3 grid(p.ctas_per_cb, D / DW_C, a->groups);
  launch_pdl(dwconv_kernel, grid, dim3(256), 0, stream, p);
  return check_launch("some_dwconv_bn_silu");
}
