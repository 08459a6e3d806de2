// tcgen05 GEMM for sm_100a:  C = epilogue(A · Wᵀ),  A:(M,K) bf16, W:(N,K) bf16 (nn.Linear layout), fp32 accumulate in TMEM.
//
// Persistent, warp-specialised:
//   warp 0      TMA producer   (one elected lane; cp.async.bulk.tensor 2D, 128B swizzle, STAGES-deep mbarrier ring)
//   warp 1      MMA issuer     (one lane issues tcgen05.mma cta_group::1 128xBNx16; owns the TMEM allocation)
//   warps 2..5  epilogue       (tcgen05.ld 32x32b: thread == accumulator row; bias / GELU / LayerScale / residual /
//                               per-head RMSNorm + RoPE; 16-byte global stores)
// Two TMEM accumulator buffers (2 x BN columns) let the epilogue of tile i overlap the main loop of tile i+1.
// Tiles are visited n-fastest so the CTAs of one wave share A rows through L2 and W stays L2-resident.
#include <cstdlib>
#include "common.cuh"
#include "ptx.cuh"
#include "../../include/actionmesh_b200.h"

namespace amb {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one swizzle-128B row

struct GemmParams {
  int M, N, K;
  int k_split_blocks;  // k-blocks >= this come from the second A source (INT_MAX: single source)
  void* C;
  long long ldc;
  int c_fp32;
  const float* bias;
  const void* residual;
  long long ldr;
  int res_fp32;
  int act;
  const float* col_scale;
  int grp_rows, grp_stride, row_off;
  int norm_cols, norm_seg;
  const float* norm_w0;
  const float* norm_w1;
  float norm_eps;
  int rope_cols;
  const float* rope_cos;
  const float* rope_sin;
  int rope_rows_per_pos;
  void* C2;        // optional bf16 copy of the output
  long long ldc2;
};

// Exact (erf) GELU, x·Φ(x), as the reference's FeedForward uses (diffusers GELU, approximate="none").  Φ(-|x|) =
// ½·erfc(|x|/√2) through Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7): one MUFU.RCP, one MUFU.EX2 and six FMAs instead of
// libdevice erff's two divergent branches (~28 instructions); the absolute error of the result (4.2e-7 over |x| <= 12) is
// that of the fp32 erf formula itself (4.5e-7).  The FF1 epilogue was instruction-bound on this function.
__device__ __forceinline__ float gelu_erf(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f * 0.70710678118654752440f, ax, 1.0f)));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = ex2_approx(ax * ax * (-0.5f * 1.4426950408889634f));
  const float q = 0.5f * (p * t) * e;  // Φ(-|x|)
  return x * (x >= 0.0f ? 1.0f - q : q);
}

template <int BN, int STAGES>
struct GemmSmem {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 4) * 8 + 16 + 1024;  // + alignment slack
};

// store 8 consecutive output columns of one row (values already final)
__device__ __forceinline__ void store8(void* C, int c_fp32, long long off, const float* v) {
  if (c_fp32) {
    float4* p = reinterpret_cast<float4*>(reinterpret_cast<float*>(C) + off);
    p[0] = make_float4(v[0], v[1], v[2], v[3]);
    p[1] = make_float4(v[4], v[5], v[6], v[7]);
  } else {
    uint4 o;
    o.x = pack_bf16(v[0], v[1]);
    o.y = pack_bf16(v[2], v[3]);
    o.z = pack_bf16(v[4], v[5]);
    o.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(C) + off) = o;
  }
}
__device__ __forceinline__ void load8_residual(const void* R, int r_fp32, long long off, float* r) {
  if (r_fp32) {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(R) + off);
    float4 a = p[0], b = p[1];
    r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
  } else {
    uint4 raw = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(R) + off);
    float2 f0 = unpack_bf16(raw.x), f1 = unpack_bf16(raw.y), f2 = unpack_bf16(raw.z), f3 = unpack_bf16(raw.w);
    r[0] = f0.x; r[1] = f0.y; r[2] = f1.x; r[3] = f1.y; r[4] = f2.x; r[5] = f2.y; r[6] = f3.x; r[7] = f3.y;
  }
}

// raw residual words of 32 consecutive columns (8 x 16 bytes of fp32, or 4 x 16 bytes of bf16): issued one chunk ahead of
// their use so that the global-load latency hides behind the TMEM read, the math and the stores of the previous chunk
struct Res32 {
  uint4 w[8];
};
__device__ __forceinline__ void load_res32(const GemmParams& p, long long drow, int col, Res32& r) {
  if (p.res_fp32) {
    const uint4* q = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.residual) + drow * p.ldr + col);
#pragma unroll
    for (int i = 0; i < 8; ++i) r.w[i] = q[i];
  } else {
    const uint4* q = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.residual) + drow * p.ldr + col);
#pragma unroll
    for (int i = 0; i < 4; ++i) r.w[i] = q[i];
  }
}
__device__ __forceinline__ void add_res32(const GemmParams& p, const Res32& r, float* v) {
  if (p.res_fp32) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[4 * i] += __uint_as_float(r.w[i].x);
      v[4 * i + 1] += __uint_as_float(r.w[i].y);
      v[4 * i + 2] += __uint_as_float(r.w[i].z);
      v[4 * i + 3] += __uint_as_float(r.w[i].w);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f0 = unpack_bf16(r.w[i].x), f1 = unpack_bf16(r.w[i].y), f2 = unpack_bf16(r.w[i].z), f3 = unpack_bf16(r.w[i].w);
      v[8 * i] += f0.x; v[8 * i + 1] += f0.y; v[8 * i + 2] += f1.x; v[8 * i + 3] += f1.y;
      v[8 * i + 4] += f2.x; v[8 * i + 5] += f2.y; v[8 * i + 6] += f3.x; v[8 * i + 7] += f3.y;
    }
  }
}

// bias -> activation -> column scale -> residual -> store, for `NV` (multiple of 8) consecutive columns starting at col
template <int NV>
__device__ __forceinline__ void finish_and_store(const GemmParams& p, float* v, long long drow, int col, bool valid,
                                                 const Res32* res = nullptr) {
  if (p.bias) {
#pragma unroll
    for (int j = 0; j < NV; j += 4) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col + j));
      v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
    }
  }
  if (p.act == 1) {
#pragma unroll
    for (int j = 0; j < NV; ++j) v[j] = gelu_erf(v[j]);
  }
  if (p.col_scale) {
#pragma unroll
    for (int j = 0; j < NV; j += 4) {
      const float4 s = __ldg(reinterpret_cast<const float4*>(p.col_scale + col + j));
      v[j] *= s.x; v[j + 1] *= s.y; v[j + 2] *= s.z; v[j + 3] *= s.w;
    }
  }
  if (!valid) return;
  if (res != nullptr && NV == 32) {  // residual words were loaded a chunk ahead
    add_res32(p, *res, v);
#pragma unroll
    for (int j = 0; j < NV; j += 8) store8(p.C, p.c_fp32, drow * p.ldc + col + j, v + j);
    if (p.C2) {
#pragma unroll
      for (int j = 0; j < NV; j += 8) store8(p.C2, 0, drow * p.ldc2 + col + j, v + j);
    }
    return;
  }
#pragma unroll
  for (int j = 0; j < NV; j += 8) {
    if (p.residual) {
      float r[8];
      load8_residual(p.residual, p.res_fp32, drow * p.ldr + col + j, r);
#pragma unroll
      for (int t = 0; t < 8; ++t) v[j + t] += r[t];
    }
    store8(p.C, p.c_fp32, drow * p.ldc + col + j, v + j);
    if (p.C2) store8(p.C2, 0, drow * p.ldc2 + col + j, v + j);
  }
}

// Epilogue of one 128 x BN accumulator tile held in TMEM (thread == row): bias / GELU / LayerScale / residual, or the
// per-head RMSNorm (+RoPE) path, then 16-byte global stores.  Shared by the 1-CTA and the 2-CTA kernels.
template <int BN>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, uint32_t taddr, int n0, int row, long long drow,
                                              bool valid, int c_begin = 0, int c_end = BN) {
  if (n0 < (p.norm_cols > p.rope_cols ? p.norm_cols : p.rope_cols)) {
    // ---- per-head RMSNorm and/or RoPE: one head = 128 accumulator columns, all owned by this thread ----
    if constexpr (BN % 128 == 0) {
#pragma unroll 1
      for (int hc = c_begin; hc < c_end; hc += 128) {
        const int col0 = n0 + hc;
        // Two passes over the head's 128 accumulator columns, 32 at a time (TMEM re-reads are cheap, registers are not:
        // 10 warps are budgeted as 12, i.e. 168 registers per thread): sum of squares first, then scale / rotate / store.
        float rs = 1.0f;
        const bool do_norm = col0 < p.norm_cols, do_rope = col0 < p.rope_cols;
        if (do_norm) {
          float ss = 0.f;
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            float v[32];
            tmem_ld_x32f(taddr + hc + c * 32, v);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; ++j) ss += v[j] * v[j];
          }
          rs = rsqrtf(ss * (1.0f / 128.0f) + p.norm_eps);
        }
        const float* w = (col0 < p.norm_seg) ? p.norm_w0 : p.norm_w1;
        const int pos = (valid ? row : 0) / p.rope_rows_per_pos;
        const float* cs = p.rope_cos + (long long)pos * 64;
        const float* sn = p.rope_sin + (long long)pos * 64;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          float v[32];
          tmem_ld_x32f(taddr + hc + c * 32, v);
          tmem_wait_ld();
          if (do_norm) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 ww = __ldg(reinterpret_cast<const float4*>(w + c * 32 + j));
              v[j] *= rs * ww.x; v[j + 1] *= rs * ww.y; v[j + 2] *= rs * ww.z; v[j + 3] *= rs * ww.w;
            }
          }
          if (do_rope) {  // interleaved pairs (2i, 2i+1) rotate by angle i of the row's position: 16 angles per 32 columns
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const float4 c4 = __ldg(reinterpret_cast<const float4*>(cs + c * 16 + j));
              const float4 s4 = __ldg(reinterpret_cast<const float4*>(sn + c * 16 + j));
              float a, b;
              a = v[2 * j + 0]; b = v[2 * j + 1]; v[2 * j + 0] = a * c4.x - b * s4.x; v[2 * j + 1] = b * c4.x + a * s4.x;
              a = v[2 * j + 2]; b = v[2 * j + 3]; v[2 * j + 2] = a * c4.y - b * s4.y; v[2 * j + 3] = b * c4.y + a * s4.y;
              a = v[2 * j + 4]; b = v[2 * j + 5]; v[2 * j + 4] = a * c4.z - b * s4.z; v[2 * j + 5] = b * c4.z + a * s4.z;
              a = v[2 * j + 6]; b = v[2 * j + 7]; v[2 * j + 6] = a * c4.w - b * s4.w; v[2 * j + 7] = b * c4.w + a * s4.w;
            }
          }
          if (!do_norm && !do_rope && p.bias) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + c * 32 + j));
              v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
            }
          }
          if (valid) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) store8(p.C, p.c_fp32, drow * p.ldc + col0 + c * 32 + j, v + j);
          }
        }
      }
    }
  } else {
    // ---- plain epilogue in 32-column chunks; the residual words of chunk c+1 are in flight while chunk c is processed ----
    const bool pre = p.residual != nullptr && valid;
    Res32 rcur, rnext;
    if (pre) load_res32(p, drow, n0 + c_begin, rcur);
#pragma unroll 1
    for (int c = c_begin; c < c_end; c += 32) {
      float v[32];
      tmem_ld_x32f(taddr + c, v);
      if (pre && c + 32 < c_end) load_res32(p, drow, n0 + c + 32, rnext);
      tmem_wait_ld();
      finish_and_store<32>(p, v, drow, n0 + c, valid, pre ? &rcur : nullptr);
      rcur = rnext;
    }
  }
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(192, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                 const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  using L = GemmSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFFSET);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform: role code stays on the uniform datapath
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(&tmem_full[a], 1);
        mbar_init(&tmem_empty[a], 128);
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_n_tiles = p.N / BN;
  const int num_m_tiles = (p.M + BM - 1) / BM;
  const int num_tiles = num_n_tiles * num_m_tiles;
  const int num_kb = p.K / BK;

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged; one elected lane issues) =====================
    int s = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (tile / num_n_tiles) * BM;
      const int n0 = (tile % num_n_tiles) * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[s], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full_bar[s], L::STAGE_BYTES);
          uint8_t* sa = smem + s * L::STAGE_BYTES;
          uint8_t* sb = sa + L::A_BYTES;
          if (kb < p.k_split_blocks) tma_load_2d(sa, &tmA, &full_bar[s], kb * BK, m0, kEvictNormal);
          else tma_load_2d(sa, &tmA2, &full_bar[s], (kb - p.k_split_blocks) * BK, m0, kEvictNormal);
          tma_load_2d(sb, &tmB, &full_bar[s], kb * BK, n0, kEvictLast);
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp converged; descriptors live in uniform registers) =====================
    constexpr uint32_t idesc = make_idesc_bf16(BM, BN, 0, 0);
    int s = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[s], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * L::STAGE_BYTES);
        const uint64_t adesc = make_desc_kmajor_sw128(a_addr);
        const uint64_t bdesc = make_desc_kmajor_sw128(a_addr + L::A_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)  // +32 B per UMMA_K step == +2 in the descriptor's (addr >> 4) field
            mma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          tc_commit(&empty_bar[s]);  // smem slot reusable once these MMAs have read it
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; phase ^= 1; }
      }
      if (elect_one()) tc_commit(&tmem_full[acc]);  // accumulator complete
      __syncwarp();
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int quarter = warp & 3;  // TMEM lane quarter this warp may access
    const int row_in_tile = quarter * 32 + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m0 = (tile / num_n_tiles) * BM;
      const int n0 = (tile % num_n_tiles) * BN;
      const int row = m0 + row_in_tile;
      const bool valid = row < p.M;
      long long drow = row;
      if (p.grp_rows > 0) drow = (long long)(row / p.grp_rows) * p.grp_stride + (row % p.grp_rows) + p.row_off;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
      epilogue_tile<BN>(p, taddr, n0, row, drow, valid);
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}


static GemmParams make_params(const amb_gemm_args* a) {
  GemmParams p;
  p.M = a->m; p.N = a->n; p.K = a->k;
  p.k_split_blocks = a->a2 ? a->k_split / BK : 0x7fffffff;
  p.C = a->c; p.ldc = a->ldc; p.c_fp32 = a->c_fp32;
  p.bias = a->bias;
  p.residual = a->residual; p.ldr = a->ldr; p.res_fp32 = a->res_fp32;
  p.act = a->act;
  p.col_scale = a->col_scale;
  p.grp_rows = a->grp_rows; p.grp_stride = a->grp_stride; p.row_off = a->row_off;
  p.norm_cols = a->norm_cols; p.norm_seg = a->norm_seg;
  p.norm_w0 = a->norm_w0; p.norm_w1 = a->norm_w1 ? a->norm_w1 : a->norm_w0;
  p.norm_eps = a->norm_eps;
  p.rope_cols = a->rope_cols; p.rope_cos = a->rope_cos; p.rope_sin = a->rope_sin;
  p.rope_rows_per_pos = a->rope_rows_per_pos > 0 ? a->rope_rows_per_pos : 1;
  p.C2 = a->c2; p.ldc2 = a->ldc2;

  return p;
}

// =====================================================================================================================
// 2-CTA variant (tcgen05 cta_group::2): a cluster of two CTAs on one TPC computes a 256 x 256 output tile.  Each CTA
// stages its own 128 rows of A and HALF of the W tile (128 of the 256 output columns' rows), so per k-block it moves
// 32 KB instead of 48 KB through TMA / shared memory for the same MMA work — the single-CTA kernel is bound by
// shared-memory bandwidth (MMA operand reads + TMA writes), not by the tensor pipe.  The leader CTA issues one
// 256 x 256 x 16 MMA per UMMA_K step that reads both CTAs' shared memory and writes each CTA's 128 accumulator rows into
// its own TMEM.  Barriers: `full` lives in the leader (both CTAs' TMA bytes are credited to it), `empty` / `tmem_full`
// are signalled in both CTAs by multicast commits, `tmem_empty` collects both epilogues in the leader.
// =====================================================================================================================
template <int STAGES>
struct Gemm2Smem {
  static constexpr int A_BYTES = BM * BK * 2;        // 16 KB: my 128 rows of A
  static constexpr int B_BYTES = 128 * BK * 2;       // 16 KB: my half of the 256-row W tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 4) * 8 + 16 + 1024;
};

constexpr int GEMM2_THREADS = 320;  // TMA warp, MMA warp, 8 epilogue warps (lane quarter x column half)

template <int STAGES>
// (10 warps are budgeted as 12 by the register allocator: at most 168 registers per thread)
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM2_THREADS, 1)
gemm2_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                  const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  using L = Gemm2Smem<STAGES>;
  constexpr int BN = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFFSET);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;      // [2] (leader's copy is the live one: 16 warp arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = (rank == 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(&tmem_full[a], 1);
        mbar_init(&tmem_empty[a], 16);  // one arrival per epilogue warp of both CTAs
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_pair(tmem_slot, 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_n_tiles = p.N / BN;
  const int num_m_pairs = (p.M + 2 * BM - 1) / (2 * BM);
  const int num_tiles = num_n_tiles * num_m_pairs;
  const int num_kb = p.K / BK;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    int s = 0;
    uint32_t phase = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      const int m0 = (tile / num_n_tiles) * (2 * BM) + rank * BM;
      const int nb = (tile % num_n_tiles) * BN + rank * 128;  // my half of the W tile rows
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[s], phase ^ 1);
        if (elect_one()) {
          if (leader) mbar_expect_tx(&full_bar[s], 2 * L::STAGE_BYTES);  // bytes of BOTH CTAs land on the leader's barrier
          uint8_t* sa = smem + s * L::STAGE_BYTES;
          uint8_t* sb = sa + L::A_BYTES;
          if (kb < p.k_split_blocks) tma_load_2d_pair(sa, &tmA, &full_bar[s], kb * BK, m0, kEvictNormal);
          else tma_load_2d_pair(sa, &tmA2, &full_bar[s], (kb - p.k_split_blocks) * BK, m0, kEvictNormal);
          tma_load_2d_pair(sb, &tmB, &full_bar[s], kb * BK, nb, kEvictLast);
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===================== MMA issuer (leader CTA only) =====================
      constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, 0, 0);
      int s = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[s], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * L::STAGE_BYTES);
          const uint64_t adesc = make_desc_kmajor_sw128(a_addr);
          const uint64_t bdesc = make_desc_kmajor_sw128(a_addr + L::A_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma_ss_pair(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
            tc_commit_pair(&empty_bar[s]);
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; phase ^= 1; }
        }
        if (elect_one()) tc_commit_pair(&tmem_full[acc]);
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue (warps 2..9 of both CTAs; each CTA owns its 128 accumulator rows; a warp owns the 32
    // rows of its TMEM lane quarter and one 128-column half of the tile) =====================
    const int quarter = warp & 3;
    const int chalf = (warp - 2) >> 2;
    const int row_in_tile = quarter * 32 + lane;
    int it = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m0 = (tile / num_n_tiles) * (2 * BM) + rank * BM;
      const int n0 = (tile % num_n_tiles) * BN;
      const int row = m0 + row_in_tile;
      const bool valid = row < p.M;
      long long drow = row;
      if (p.grp_rows > 0) drow = (long long)(row / p.grp_rows) * p.grp_stride + (row % p.grp_rows) + p.row_off;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
      epilogue_tile<BN>(p, taddr, n0, row, drow, valid, chalf * 128, chalf * 128 + 128);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tmem_empty[acc]);
        else mbar_arrive_remote(&tmem_empty[acc], 0);
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();  // no CTA of the pair may free TMEM / exit while its peer still uses shared memory or TMEM
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

template <int STAGES>
static int launch_gemm2(const amb_gemm_args* a, cudaStream_t stream) {
  using L = Gemm2Smem<STAGES>;
  CUtensorMap tmA, tmA2, tmB;
  const int k1 = (a->a2 != nullptr) ? a->k_split : a->k;
  {
    uint64_t dims[2] = {(uint64_t)k1, (uint64_t)a->m};
    uint64_t str[1] = {(uint64_t)a->lda * 2};
    uint32_t box[2] = {BK, BM};
    int r = encode_tmap_bf16(&tmA, a->a, 2, dims, str, box);
    if (r) return r;
  }
  if (a->a2) {
    uint64_t dims[2] = {(uint64_t)(a->k - a->k_split), (uint64_t)a->m};
    uint64_t str[1] = {(uint64_t)a->lda2 * 2};
    uint32_t box[2] = {BK, BM};
    int r = encode_tmap_bf16(&tmA2, a->a2, 2, dims, str, box);
    if (r) return r;
  } else {
    tmA2 = tmA;
  }
  {
    uint64_t dims[2] = {(uint64_t)a->k, (uint64_t)a->n};
    uint64_t str[1] = {(uint64_t)a->ldw * 2};
    uint32_t box[2] = {BK, 128};
    int r = encode_tmap_bf16(&tmB, a->w, 2, dims, str, box);
    if (r) return r;
  }
  GemmParams p = make_params(a);
  auto kern = gemm2_bf16_kernel<STAGES>;
  {
    int r = ensure_smem_optin(kern, L::TOTAL);
    if (r) return r;
  }
  const int num_tiles = (a->n / 256) * ((a->m + 2 * BM - 1) / (2 * BM));
  int clusters = num_sms() / 2;
  if (clusters > num_tiles) clusters = num_tiles;
  kern<<<2 * clusters, GEMM2_THREADS, L::TOTAL, stream>>>(tmA, tmA2, tmB, p);  // cluster dims are compiled in (__cluster_dims__)
  AMB_CHECK_CUDA(cudaGetLastError());
  return AMB_OK;
}

template <int BN, int STAGES>
static int launch_gemm(const amb_gemm_args* a, cudaStream_t stream) {
  using L = GemmSmem<BN, STAGES>;
  CUtensorMap tmA, tmA2, tmB;
  const int k1 = (a->a2 != nullptr) ? a->k_split : a->k;
  {
    uint64_t dims[2] = {(uint64_t)k1, (uint64_t)a->m};
    uint64_t str[1] = {(uint64_t)a->lda * 2};
    uint32_t box[2] = {BK, BM};
    int r = encode_tmap_bf16(&tmA, a->a, 2, dims, str, box);
    if (r) return r;
  }
  if (a->a2) {
    uint64_t dims[2] = {(uint64_t)(a->k - a->k_split), (uint64_t)a->m};
    uint64_t str[1] = {(uint64_t)a->lda2 * 2};
    uint32_t box[2] = {BK, BM};
    int r = encode_tmap_bf16(&tmA2, a->a2, 2, dims, str, box);
    if (r) return r;
  } else {
    tmA2 = tmA;
  }
  {
    uint64_t dims[2] = {(uint64_t)a->k, (uint64_t)a->n};
    uint64_t str[1] = {(uint64_t)a->ldw * 2};
    uint32_t box[2] = {BK, BN};
    int r = encode_tmap_bf16(&tmB, a->w, 2, dims, str, box);
    if (r) return r;
  }
  GemmParams p = make_params(a);
  auto kern = gemm_bf16_kernel<BN, STAGES>;
  {
    int r = ensure_smem_optin(kern, L::TOTAL);
    if (r) return r;
  }
  const int num_tiles = (a->n / BN) * ((a->m + BM - 1) / BM);
  int grid = num_sms();
  if (grid > num_tiles) grid = num_tiles;
  kern<<<grid, 192, L::TOTAL, stream>>>(tmA, tmA2, tmB, p);
  AMB_CHECK_CUDA(cudaGetLastError());
  return AMB_OK;
}

}  // namespace amb

using namespace amb;

extern "C" int amb_gemm_bf16(const amb_gemm_args* a, amb_stream_t stream) {
  AMB_CHECK_ARG(a && a->a && a->w && a->c, "gemm: null pointer");
  AMB_CHECK_ARG(a->m > 0 && a->n > 0 && a->k > 0, "gemm: bad shape m=%d n=%d k=%d", a->m, a->n, a->k);
  AMB_CHECK_ARG(a->k % BK == 0, "gemm: k=%d must be a multiple of %d", a->k, BK);
  AMB_CHECK_ARG(a->n % 64 == 0, "gemm: n=%d must be a multiple of 64", a->n);
  AMB_CHECK_ARG(a->lda % 8 == 0 && a->ldw % 8 == 0 && a->ldc % 8 == 0, "gemm: lda/ldw/ldc must be multiples of 8 elements");
  AMB_CHECK_ARG(!a->a2 || (a->k_split > 0 && a->k_split < a->k && a->k_split % BK == 0 && a->lda2 % 8 == 0),
                "gemm: bad k_split %d", a->k_split);
  AMB_CHECK_ARG(!a->residual || a->ldr % 8 == 0, "gemm: ldr must be a multiple of 8");
  AMB_CHECK_ARG(a->act == 0 || a->act == 1, "gemm: unknown activation %d", a->act);
  AMB_CHECK_ARG(!a->c2 || a->ldc2 % 8 == 0, "gemm: ldc2 must be a multiple of 8");
  // the epilogue moves 8 columns (bf16) or 4 columns (fp32) per 16-byte access, starting from these base pointers
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  AMB_CHECK_ARG(al16(a->c) && al16(a->c2) && al16(a->residual) && al16(a->bias) && al16(a->col_scale),
                "gemm: c/c2/residual/bias/col_scale must be 16-byte aligned");
  AMB_CHECK_ARG(al16(a->norm_w0) && al16(a->norm_w1) && al16(a->rope_cos) && al16(a->rope_sin),
                "gemm: norm weights and rope tables must be 16-byte aligned");
  if (a->norm_cols > 0 || a->rope_cols > 0) {
    AMB_CHECK_ARG(a->n % 128 == 0 && a->norm_cols % 128 == 0 && a->rope_cols % 128 == 0,
                  "gemm: head epilogue needs n, norm_cols, rope_cols multiples of 128");
    AMB_CHECK_ARG(a->norm_cols == 0 || (a->norm_w0 && a->norm_seg % 128 == 0), "gemm: norm weights / norm_seg (multiple of 128) required");
    AMB_CHECK_ARG(a->rope_cols == 0 || (a->rope_cos && a->rope_sin), "gemm: rope tables required");
    AMB_CHECK_ARG(!a->residual && a->act == 0 && !a->col_scale && !a->c2, "gemm: head epilogue excludes residual/activation/col_scale/c2");
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (a->n % 256 == 0 && a->m >= 256) return launch_gemm2<6>(a, s);  // CTA pairs, 256 x 256 tiles
  if (a->n % 256 == 0) return launch_gemm<256, 4>(a, s);
  if (a->n % 128 == 0) return launch_gemm<128, 6>(a, s);
  return launch_gemm<64, 8>(a, s);
}
