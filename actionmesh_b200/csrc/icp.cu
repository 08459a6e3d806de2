// Gradient ICP of the ActionBench metrics on the GPU (SURVEY 8(f) rank 4, DESIGN §12).
//
// Replaces actionbench/icp.py:53-112 (gradient_icp): for each of F problems (prediction / ground-truth cloud pairs) and
// each of the 24 canonical starts R_init[r], Adam minimises the Chamfer loss (pytorch3d chamfer_distance, point means of
// squared distances, both directions) of x_i = (s ⊙ p_i) @ R + T over (r6d, T, s), R = R_init[r] @ rot6d(r6d).
//
// One iteration is two launches and no host work:
//  - icp_search_kernel: both nearest-neighbour directions of all F x 24 (problem, start) pairs.  Exact difference-form
//    squared distances, ties to the lowest index.  "A" blocks take 32 prediction points x 24 starts (a warp per 6 starts,
//    one shared-memory ground-truth point serves 6 queries held in registers); "B" blocks take 512 ground-truth points of
//    one start (4 per thread) against the transformed prediction, which is computed while it is staged into shared
//    memory.  The transformed clouds never reach global memory.  Each block reduces its queries' loss and gradient to the
//    13 sums loss, G = Σ g, M = Σ p ⊗ g (p untransformed, g the loss gradient on the moving point) with warp butterflies
//    and writes them to its own slot: no atomics, so the sums are deterministic and independent of F.
//  - icp_update_kernel: one warp per problem, a lane per start.  Sums the block slots in a fixed order, backpropagates
//    dT = G, dR = diag(s) M, ds[a] = Σ_b R[a][b] M[a][b] through R_init @ rot6d(·), takes torch's single-tensor Adam step
//    and keeps the best result exactly as icp.py:99-106 does (see amb_gradient_icp in the header).
#include <cfloat>
#include <cstddef>

#include "common.cuh"
#include "../../include/actionmesh_b200.h"

namespace amb {

constexpr int ICP_STARTS = 24;
constexpr int ICP_THREADS = 128;
constexpr int ICP_TILE = 512;                 // points per shared-memory tile
constexpr int ICP_A_PTS = 32;                 // prediction points per A block (a warp each group of starts)
constexpr int ICP_A_GRP = ICP_STARTS / 4;     // starts per thread in an A block
constexpr int ICP_B_PER = 4;                  // ground-truth points per thread in a B block
constexpr int ICP_B_PTS = ICP_THREADS * ICP_B_PER;
constexpr int ICP_NSUM = 13;                  // loss, G[3], M[3][3]
constexpr int ICP_NPAR = 12;                  // r6d[6], T[3], s[3]

struct IcpLayout {
  int n_a, n_b_per_start, n_slots;  // block counts per problem
  size_t partial, params, rot, m, v, total;  // float offsets into the workspace
};

static IcpLayout icp_layout(int n_problems, int n_pred, int n_gt) {
  IcpLayout L;
  L.n_a = (n_pred + ICP_A_PTS - 1) / ICP_A_PTS;
  L.n_b_per_start = (n_gt + ICP_B_PTS - 1) / ICP_B_PTS;
  L.n_slots = L.n_a + L.n_b_per_start;
  const size_t ps = (size_t)n_problems * ICP_STARTS;
  L.partial = 0;
  L.params = L.partial + ps * L.n_slots * ICP_NSUM;
  L.rot = L.params + ps * ICP_NPAR;
  L.m = L.rot + ps * 9;
  L.v = L.m + ps * ICP_NPAR;
  L.total = L.v + ps * ICP_NPAR;
  return L;
}

// R = R_init @ rot6d(d6) (pytorch3d rotation_6d_to_matrix: Gram-Schmidt with F.normalize's eps 1e-12, rows b1, b2, b1 x b2)
__device__ void rot6d_forward(const float* d6, const float* Ri, float* R) {
  const float* a1 = d6;
  const float* a2 = d6 + 3;
  const float n1 = fmaxf(sqrtf(a1[0] * a1[0] + a1[1] * a1[1] + a1[2] * a1[2]), 1e-12f);
  float b[3][3];
  for (int k = 0; k < 3; ++k) b[0][k] = a1[k] / n1;
  const float c = b[0][0] * a2[0] + b[0][1] * a2[1] + b[0][2] * a2[2];
  float u[3];
  for (int k = 0; k < 3; ++k) u[k] = a2[k] - c * b[0][k];
  const float n2 = fmaxf(sqrtf(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]), 1e-12f);
  for (int k = 0; k < 3; ++k) b[1][k] = u[k] / n2;
  b[2][0] = b[0][1] * b[1][2] - b[0][2] * b[1][1];
  b[2][1] = b[0][2] * b[1][0] - b[0][0] * b[1][2];
  b[2][2] = b[0][0] * b[1][1] - b[0][1] * b[1][0];
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 3; ++k) R[3 * a + k] = Ri[3 * a] * b[0][k] + Ri[3 * a + 1] * b[1][k] + Ri[3 * a + 2] * b[2][k];
}

__device__ inline void cross3(const float* a, const float* b, float* o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

// Gradient of the loss w.r.t. d6 given dL/dR for R = R_init @ rot6d(d6).
__device__ void rot6d_backward(const float* d6, const float* Ri, const float* dR, float* dd6) {
  const float* a1 = d6;
  const float* a2 = d6 + 3;
  const float l1 = sqrtf(a1[0] * a1[0] + a1[1] * a1[1] + a1[2] * a1[2]);
  const float n1 = fmaxf(l1, 1e-12f);
  float b1[3], u[3], b2[3];
  for (int k = 0; k < 3; ++k) b1[k] = a1[k] / n1;
  const float c = b1[0] * a2[0] + b1[1] * a2[1] + b1[2] * a2[2];
  for (int k = 0; k < 3; ++k) u[k] = a2[k] - c * b1[k];
  const float l2 = sqrtf(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  const float n2 = fmaxf(l2, 1e-12f);
  for (int k = 0; k < 3; ++k) b2[k] = u[k] / n2;
  // dL/dR6 = R_init^T dL/dR; rows are the gradients of b1, b2, b3
  float g[3][3];
  for (int c6 = 0; c6 < 3; ++c6)
    for (int k = 0; k < 3; ++k) g[c6][k] = Ri[c6] * dR[k] + Ri[3 + c6] * dR[3 + k] + Ri[6 + c6] * dR[6 + k];
  float t[3];
  cross3(b2, g[2], t);  // b3 = b1 x b2
  for (int k = 0; k < 3; ++k) g[0][k] += t[k];
  cross3(g[2], b1, t);
  for (int k = 0; k < 3; ++k) g[1][k] += t[k];
  // b2 = normalize(u)
  float du[3];
  if (l2 > 1e-12f) {
    const float dot = b2[0] * g[1][0] + b2[1] * g[1][1] + b2[2] * g[1][2];
    for (int k = 0; k < 3; ++k) du[k] = (g[1][k] - b2[k] * dot) / l2;
  } else {
    for (int k = 0; k < 3; ++k) du[k] = g[1][k] / 1e-12f;
  }
  // u = a2 - (b1 . a2) b1
  const float dub1 = du[0] * b1[0] + du[1] * b1[1] + du[2] * b1[2];
  for (int k = 0; k < 3; ++k) {
    dd6[3 + k] = du[k] - dub1 * b1[k];
    g[0][k] += -c * du[k] - dub1 * a2[k];
  }
  // b1 = normalize(a1)
  if (l1 > 1e-12f) {
    const float dot = b1[0] * g[0][0] + b1[1] * g[0][1] + b1[2] * g[0][2];
    for (int k = 0; k < 3; ++k) dd6[k] = (g[0][k] - b1[k] * dot) / l1;
  } else {
    for (int k = 0; k < 3; ++k) dd6[k] = g[0][k] / 1e-12f;
  }
}

// x = (s ⊙ p) @ R + T
__device__ inline void icp_xform(const float* R, const float* T, const float* s, float p0, float p1, float p2, float& x0,
                                 float& x1, float& x2) {
  const float q0 = s[0] * p0, q1 = s[1] * p1, q2 = s[2] * p2;
  x0 = fmaf(q2, R[6], fmaf(q1, R[3], q0 * R[0])) + T[0];
  x1 = fmaf(q2, R[7], fmaf(q1, R[4], q0 * R[1])) + T[1];
  x2 = fmaf(q2, R[8], fmaf(q1, R[5], q0 * R[2])) + T[2];
}

__device__ inline float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Adds one query's contribution (loss d2 * inv_n, gradient g on the moving point, untransformed moving point p).
__device__ inline void icp_accum(float* acc, float d2, float inv_n, float xm0, float xm1, float xm2, float y0, float y1,
                                 float y2, float p0, float p1, float p2) {
  const float g0 = 2.f * (xm0 - y0) * inv_n, g1 = 2.f * (xm1 - y1) * inv_n, g2 = 2.f * (xm2 - y2) * inv_n;
  acc[0] += d2 * inv_n;
  acc[1] += g0;
  acc[2] += g1;
  acc[3] += g2;
  acc[4] += p0 * g0;
  acc[5] += p0 * g1;
  acc[6] += p0 * g2;
  acc[7] += p1 * g0;
  acc[8] += p1 * g1;
  acc[9] += p1 * g2;
  acc[10] += p2 * g0;
  acc[11] += p2 * g1;
  acc[12] += p2 * g2;
}

// grid: (n_a + 24 * n_b_per_start, F); blocks [0, n_a) are A blocks, the rest B blocks (start-major).
__global__ void __launch_bounds__(ICP_THREADS) icp_search_kernel(const float* __restrict__ pred, int n_pred,
                                                                 const float* __restrict__ gt, int n_gt,
                                                                 const float* __restrict__ params,
                                                                 const float* __restrict__ rot, int n_a, int n_bps,
                                                                 float* __restrict__ partial) {
  __shared__ float sx[ICP_TILE], sy[ICP_TILE], sz[ICP_TILE];
  __shared__ float sR[ICP_STARTS][9], sT[ICP_STARTS][3], sS[ICP_STARTS][3];
  __shared__ float sred[ICP_THREADS / 32][ICP_NSUM];
  const int f = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_slots = n_a + n_bps;
  pred += (size_t)f * n_pred * 3;
  gt += (size_t)f * n_gt * 3;
  for (int i = tid; i < ICP_STARTS * 9; i += ICP_THREADS) sR[i / 9][i % 9] = rot[(size_t)f * ICP_STARTS * 9 + i];
  for (int i = tid; i < ICP_STARTS * 3; i += ICP_THREADS) {
    const float* pp = params + ((size_t)f * ICP_STARTS + i / 3) * ICP_NPAR;
    sT[i / 3][i % 3] = pp[6 + i % 3];
    sS[i / 3][i % 3] = pp[9 + i % 3];
  }
  __syncthreads();

  if (blockIdx.x < n_a) {
    // ---- pred -> gt: a thread holds one prediction point under ICP_A_GRP starts; the gt tile is shared by all of them
    const int i = blockIdx.x * ICP_A_PTS + lane;
    const int r0 = warp * ICP_A_GRP;
    const bool live = i < n_pred;
    float p0 = 0.f, p1 = 0.f, p2 = 0.f;
    if (live) {
      p0 = pred[3 * i];
      p1 = pred[3 * i + 1];
      p2 = pred[3 * i + 2];
    }
    float x0[ICP_A_GRP], x1[ICP_A_GRP], x2[ICP_A_GRP], bd[ICP_A_GRP];
    int bi[ICP_A_GRP];
#pragma unroll
    for (int k = 0; k < ICP_A_GRP; ++k) {
      icp_xform(sR[r0 + k], sT[r0 + k], sS[r0 + k], p0, p1, p2, x0[k], x1[k], x2[k]);
      bd[k] = INFINITY;
      bi[k] = 0;
    }
    for (int t0 = 0; t0 < n_gt; t0 += ICP_TILE) {
      const int cnt = min(ICP_TILE, n_gt - t0);
      __syncthreads();
      for (int j = tid; j < cnt; j += ICP_THREADS) {
        sx[j] = gt[3 * (t0 + j)];
        sy[j] = gt[3 * (t0 + j) + 1];
        sz[j] = gt[3 * (t0 + j) + 2];
      }
      __syncthreads();
#pragma unroll 2
      for (int j = 0; j < cnt; ++j) {
        const float y0 = sx[j], y1 = sy[j], y2 = sz[j];
#pragma unroll
        for (int k = 0; k < ICP_A_GRP; ++k) {
          const float dx = x0[k] - y0, dy = x1[k] - y1, dz = x2[k] - y2;
          const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
          if (d < bd[k]) {
            bd[k] = d;
            bi[k] = t0 + j;
          }
        }
      }
    }
    const float inv_n = 1.f / (float)n_pred;
#pragma unroll
    for (int k = 0; k < ICP_A_GRP; ++k) {
      float acc[ICP_NSUM];
#pragma unroll
      for (int c = 0; c < ICP_NSUM; ++c) acc[c] = 0.f;
      if (live) {
        const int j = bi[k];
        icp_accum(acc, bd[k], inv_n, x0[k], x1[k], x2[k], gt[3 * j], gt[3 * j + 1], gt[3 * j + 2], p0, p1, p2);
      }
      float* out = partial + (((size_t)f * ICP_STARTS + r0 + k) * n_slots + blockIdx.x) * ICP_NSUM;
#pragma unroll
      for (int c = 0; c < ICP_NSUM; ++c) {
        const float v = warp_sum(acc[c]);
        if (lane == 0) out[c] = v;
      }
    }
  } else {
    // ---- gt -> pred: a thread holds ICP_B_PER gt points of start r; the prediction is transformed while staged
    const int b = blockIdx.x - n_a;
    const int r = b / n_bps, chunk = b % n_bps;
    const float* R = sR[r];
    const float* T = sT[r];
    const float* S = sS[r];
    float y0[ICP_B_PER], y1[ICP_B_PER], y2[ICP_B_PER], bd[ICP_B_PER];
    int bi[ICP_B_PER];
#pragma unroll
    for (int k = 0; k < ICP_B_PER; ++k) {
      const int j = chunk * ICP_B_PTS + k * ICP_THREADS + tid;
      y0[k] = y1[k] = y2[k] = 0.f;
      if (j < n_gt) {
        y0[k] = gt[3 * j];
        y1[k] = gt[3 * j + 1];
        y2[k] = gt[3 * j + 2];
      }
      bd[k] = INFINITY;
      bi[k] = 0;
    }
    for (int t0 = 0; t0 < n_pred; t0 += ICP_TILE) {
      const int cnt = min(ICP_TILE, n_pred - t0);
      __syncthreads();
      for (int i = tid; i < cnt; i += ICP_THREADS) {
        float a0, a1, a2;
        icp_xform(R, T, S, pred[3 * (t0 + i)], pred[3 * (t0 + i) + 1], pred[3 * (t0 + i) + 2], a0, a1, a2);
        sx[i] = a0;
        sy[i] = a1;
        sz[i] = a2;
      }
      __syncthreads();
#pragma unroll 2
      for (int i = 0; i < cnt; ++i) {
        const float a0 = sx[i], a1 = sy[i], a2 = sz[i];
#pragma unroll
        for (int k = 0; k < ICP_B_PER; ++k) {
          const float dx = y0[k] - a0, dy = y1[k] - a1, dz = y2[k] - a2;
          const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
          if (d < bd[k]) {
            bd[k] = d;
            bi[k] = t0 + i;
          }
        }
      }
    }
    const float inv_n = 1.f / (float)n_gt;
    float acc[ICP_NSUM];
#pragma unroll
    for (int c = 0; c < ICP_NSUM; ++c) acc[c] = 0.f;
#pragma unroll
    for (int k = 0; k < ICP_B_PER; ++k) {
      const int j = chunk * ICP_B_PTS + k * ICP_THREADS + tid;
      if (j < n_gt) {
        const int i = bi[k];
        const float p0 = pred[3 * i], p1 = pred[3 * i + 1], p2 = pred[3 * i + 2];
        float a0, a1, a2;
        icp_xform(R, T, S, p0, p1, p2, a0, a1, a2);
        icp_accum(acc, bd[k], inv_n, a0, a1, a2, y0[k], y1[k], y2[k], p0, p1, p2);
      }
    }
#pragma unroll
    for (int c = 0; c < ICP_NSUM; ++c) {
      const float v = warp_sum(acc[c]);
      if (lane == 0) sred[warp][c] = v;
    }
    __syncthreads();
    if (tid < ICP_NSUM) {
      float v = sred[0][tid];
      for (int w = 1; w < ICP_THREADS / 32; ++w) v += sred[w][tid];
      partial[(((size_t)f * ICP_STARTS + r) * n_slots + n_a + chunk) * ICP_NSUM + tid] = v;
    }
  }
}

// One thread per (problem, start): parameters from params_in (NULL: the reference's initial values), moments zeroed,
// R = R_init @ rot6d(r6d).
__global__ void icp_prepare_kernel(const float* __restrict__ params_in, const float* __restrict__ r_init, int n,
                                   float* __restrict__ params, float* __restrict__ rot, float* __restrict__ m,
                                   float* __restrict__ v) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const float init[ICP_NPAR] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f, 1.f, 1.f, 1.f};
  float* p = params + (size_t)t * ICP_NPAR;
  for (int k = 0; k < ICP_NPAR; ++k) {
    p[k] = params_in ? params_in[(size_t)t * ICP_NPAR + k] : init[k];
    m[(size_t)t * ICP_NPAR + k] = 0.f;
    v[(size_t)t * ICP_NPAR + k] = 0.f;
  }
  rot6d_forward(p, r_init + (t % ICP_STARTS) * 9, rot + (size_t)t * 9);
}

struct IcpStep {
  int it;                    // 0-based iteration (index into the tables)
  const float* step_size;    // lr / (1 - beta1^t), t = it + 1
  const float* bc2_sqrt;     // sqrt(1 - beta2^t)
  float* best_rot;           // (F, 9)
  float* best_t;             // (F, 3)
  float* best_s;             // (F, 3)
  float* best_loss;          // (F)
  int32_t* best_start;       // (F)
  float* trace;              // (n_iter, F, 24) or NULL
};

// grid F, one warp: lane r < 24 owns start r.  do_step == 0: write loss and gradient (no 1/24, no step) and stop.
__global__ void __launch_bounds__(32) icp_update_kernel(const float* __restrict__ partial, int n_slots,
                                                        const float* __restrict__ r_init, float* __restrict__ params,
                                                        float* __restrict__ rot, float* __restrict__ m,
                                                        float* __restrict__ v, int do_step, IcpStep st,
                                                        float* __restrict__ out_loss, float* __restrict__ out_grad) {
  const int f = blockIdx.x, r = threadIdx.x;
  const int nF = gridDim.x;
  const bool live = r < ICP_STARTS;
  float loss = INFINITY;
  float grad[ICP_NPAR];
  const size_t ps = (size_t)f * ICP_STARTS + (live ? r : 0);
  float* p = params + ps * ICP_NPAR;
  float* R = rot + ps * 9;
  if (live) {
    float sum[ICP_NSUM];
    for (int c = 0; c < ICP_NSUM; ++c) sum[c] = 0.f;
    const float* src = partial + ps * n_slots * ICP_NSUM;
    for (int b = 0; b < n_slots; ++b)
      for (int c = 0; c < ICP_NSUM; ++c) sum[c] += src[(size_t)b * ICP_NSUM + c];
    loss = sum[0];
    const float* M = sum + 4;
    float dR[9];
    for (int a = 0; a < 3; ++a) {
      grad[9 + a] = R[3 * a] * M[3 * a] + R[3 * a + 1] * M[3 * a + 1] + R[3 * a + 2] * M[3 * a + 2];
      for (int c = 0; c < 3; ++c) dR[3 * a + c] = p[9 + a] * M[3 * a + c];
    }
    for (int c = 0; c < 3; ++c) grad[6 + c] = sum[1 + c];
    rot6d_backward(p, r_init + r * 9, dR, grad);
  }
  if (!do_step) {
    if (live) {
      out_loss[ps] = loss;
      for (int k = 0; k < ICP_NPAR; ++k) out_grad[ps * ICP_NPAR + k] = grad[k];
    }
    return;
  }
  // first index of the minimum over starts (torch's min(0)); lanes >= 24 hold +inf
  float bl = loss;
  int bs = live ? r : ICP_STARTS;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ol = __shfl_xor_sync(0xffffffffu, bl, o);
    const int os = __shfl_xor_sync(0xffffffffu, bs, o);
    if (ol < bl || (ol == bl && os < bs)) {
      bl = ol;
      bs = os;
    }
  }
  if (!live) return;
  if (st.trace) st.trace[((size_t)st.it * nF + f) * ICP_STARTS + r] = loss;
  const bool improves = bs == r && bl < st.best_loss[f];  // strict <, as `min_loss.item() < best_loss`
  if (improves)
    for (int k = 0; k < 9; ++k) st.best_rot[f * 9 + k] = R[k];  // the R that produced the loss
  // torch single-tensor Adam (betas 0.9/0.999, eps 1e-8) on loss.mean(): gradients carry the 1/24
  const float step_size = st.step_size[st.it], bc2 = st.bc2_sqrt[st.it];
  float* mm = m + ps * ICP_NPAR;
  float* vv = v + ps * ICP_NPAR;
  const float inv_starts = 1.f / (float)ICP_STARTS;
  for (int k = 0; k < ICP_NPAR; ++k) {
    const float g = grad[k] * inv_starts;
    const float mk = mm[k] + 0.1f * (g - mm[k]);
    const float vk = vv[k] * 0.999f + 0.001f * g * g;
    mm[k] = mk;
    vv[k] = vk;
    p[k] = p[k] - step_size * (mk / (sqrtf(vk) / bc2 + 1e-8f));
  }
  rot6d_forward(p, r_init + r * 9, R);
  if (improves) {
    for (int k = 0; k < 3; ++k) {
      st.best_t[f * 3 + k] = p[6 + k];  // T and s after opt.step(), as the reference clones them
      st.best_s[f * 3 + k] = p[9 + k];
    }
    st.best_loss[f] = bl;
    st.best_start[f] = r;
  }
}

__global__ void icp_best_init_kernel(float* best_loss, int32_t* best_start, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    best_loss[i] = INFINITY;
    best_start[i] = -1;
  }
}

__global__ void transform_points_kernel(const float* __restrict__ pts, int n_problems, int n_points,
                                        const float* __restrict__ R, const float* __restrict__ T,
                                        const float* __restrict__ s, float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n_problems * n_points) return;
  const int f = (int)(i / n_points);
  const float* Rf = R + f * 9;
  const float* sf = s + f * 3;
  const float* Tf = T + f * 3;
  const float p0 = pts[3 * i], p1 = pts[3 * i + 1], p2 = pts[3 * i + 2];
  // Scale(s).compose(Rotate(R), Translate(T)): p @ (diag(s) R) + T
  for (int c = 0; c < 3; ++c)
    out[3 * i + c] = fmaf(p2, sf[2] * Rf[6 + c], fmaf(p1, sf[1] * Rf[3 + c], p0 * (sf[0] * Rf[c]))) + Tf[c];
}

static int icp_check(const float* pred, const float* gt, int n_problems, int n_pred, int n_gt, const float* r_init,
                     void* workspace, size_t workspace_bytes, const char* what) {
  AMB_CHECK_ARG(pred && gt && r_init && workspace, "%s: null pointer", what);
  AMB_CHECK_ARG(n_problems > 0 && n_pred > 0 && n_gt > 0, "%s: empty cloud or no problems (F=%d, P_pred=%d, P_gt=%d)",
                what, n_problems, n_pred, n_gt);
  AMB_CHECK_ARG(n_problems <= 65535, "%s: at most 65535 problems per call", what);
  const IcpLayout L = icp_layout(n_problems, n_pred, n_gt);
  AMB_CHECK_ARG(workspace_bytes >= L.total * sizeof(float), "%s: workspace of %zu bytes < %zu required", what,
                workspace_bytes, L.total * sizeof(float));
  return AMB_OK;
}

static int icp_search(const float* pred, const float* gt, int F, int n_pred, int n_gt, float* ws, const IcpLayout& L,
                      cudaStream_t s) {
  const dim3 grid(L.n_a + ICP_STARTS * L.n_b_per_start, F);
  icp_search_kernel<<<grid, ICP_THREADS, 0, s>>>(pred, n_pred, gt, n_gt, ws + L.params, ws + L.rot, L.n_a,
                                                 L.n_b_per_start, ws + L.partial);
  AMB_CHECK_CUDA(cudaGetLastError());
  return AMB_OK;
}

}  // namespace amb

using namespace amb;

extern "C" int amb_icp_workspace_bytes(int n_problems, int n_pred, int n_gt, size_t* bytes) {
  AMB_CHECK_ARG(bytes, "icp_workspace_bytes: null pointer");
  AMB_CHECK_ARG(n_problems > 0 && n_pred > 0 && n_gt > 0, "icp_workspace_bytes: bad counts");
  *bytes = icp_layout(n_problems, n_pred, n_gt).total * sizeof(float);
  return AMB_OK;
}

extern "C" int amb_icp_chamfer_grad(const float* pred, const float* gt, int n_problems, int n_pred, int n_gt,
                                    const float* r_init, const float* params, void* workspace, size_t workspace_bytes,
                                    float* out_loss, float* out_grad, amb_stream_t stream) {
  if (int rc = icp_check(pred, gt, n_problems, n_pred, n_gt, r_init, workspace, workspace_bytes, "icp_chamfer_grad"))
    return rc;
  AMB_CHECK_ARG(params && out_loss && out_grad, "icp_chamfer_grad: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  const IcpLayout L = icp_layout(n_problems, n_pred, n_gt);
  float* ws = static_cast<float*>(workspace);
  const int n = n_problems * ICP_STARTS;
  icp_prepare_kernel<<<(n + 127) / 128, 128, 0, s>>>(params, r_init, n, ws + L.params, ws + L.rot, ws + L.m, ws + L.v);
  AMB_CHECK_CUDA(cudaGetLastError());
  if (int rc = icp_search(pred, gt, n_problems, n_pred, n_gt, ws, L, s)) return rc;
  icp_update_kernel<<<n_problems, 32, 0, s>>>(ws + L.partial, L.n_slots, r_init, ws + L.params, ws + L.rot, ws + L.m,
                                              ws + L.v, 0, IcpStep{}, out_loss, out_grad);
  AMB_CHECK_CUDA(cudaGetLastError());
  return AMB_OK;
}

extern "C" int amb_gradient_icp(const float* pred, const float* gt, int n_problems, int n_pred, int n_gt,
                                const float* r_init, int n_iter, const float* step_size, const float* bc2_sqrt,
                                void* workspace, size_t workspace_bytes, float* out_rot, float* out_t, float* out_s,
                                float* out_loss, int32_t* out_start, float* loss_trace, amb_stream_t stream) {
  if (int rc = icp_check(pred, gt, n_problems, n_pred, n_gt, r_init, workspace, workspace_bytes, "gradient_icp"))
    return rc;
  AMB_CHECK_ARG(step_size && bc2_sqrt && out_rot && out_t && out_s && out_loss && out_start,
                "gradient_icp: null pointer");
  AMB_CHECK_ARG(n_iter > 0, "gradient_icp: n_iter must be positive (got %d)", n_iter);
  cudaStream_t s = (cudaStream_t)stream;
  const IcpLayout L = icp_layout(n_problems, n_pred, n_gt);
  float* ws = static_cast<float*>(workspace);
  const int n = n_problems * ICP_STARTS;
  icp_prepare_kernel<<<(n + 127) / 128, 128, 0, s>>>(nullptr, r_init, n, ws + L.params, ws + L.rot, ws + L.m, ws + L.v);
  AMB_CHECK_CUDA(cudaGetLastError());
  icp_best_init_kernel<<<(n_problems + 127) / 128, 128, 0, s>>>(out_loss, out_start, n_problems);
  AMB_CHECK_CUDA(cudaGetLastError());
  IcpStep st{0, step_size, bc2_sqrt, out_rot, out_t, out_s, out_loss, out_start, loss_trace};
  for (int it = 0; it < n_iter; ++it) {
    if (int rc = icp_search(pred, gt, n_problems, n_pred, n_gt, ws, L, s)) return rc;
    st.it = it;
    icp_update_kernel<<<n_problems, 32, 0, s>>>(ws + L.partial, L.n_slots, r_init, ws + L.params, ws + L.rot, ws + L.m,
                                                ws + L.v, 1, st, nullptr, nullptr);
    AMB_CHECK_CUDA(cudaGetLastError());
  }
  return AMB_OK;
}

extern "C" int amb_transform_points(const float* points, int n_problems, int n_points, const float* rot,
                                    const float* t, const float* s, float* out, amb_stream_t stream) {
  AMB_CHECK_ARG(points && rot && t && s && out, "transform_points: null pointer");
  AMB_CHECK_ARG(n_problems >= 0 && n_points >= 0, "transform_points: bad counts");
  const size_t n = (size_t)n_problems * n_points;
  if (n == 0) return AMB_OK;
  transform_points_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(points, n_problems, n_points,
                                                                                        rot, t, s, out);
  AMB_CHECK_CUDA(cudaGetLastError());
  return AMB_OK;
}
