// Loss reductions (HBM-bound, vectorised, coalesced) for the distillation step:
//   * multi-pair MSE in ONE launch (GeneralDistill.py:60-82: ~50 MSELoss launches per step in the reference);
//   * row-wise softmax cross-entropy with ignore_index / label smoothing (eff_bert.py:1263-1302,1699-1702; xvlm.py:479-483);
//   * soft-target KL (GeneralDistill.py:84-89) and dense soft-label CE (ITC with idx, xvlm.py:404-416);
//   * L2 row normalisation (xvlm.py:375-382) and device-side ITM hard-negative sampling (xvlm.py:422-455).
#include "evlm_common.cuh"
#include "../../include/evlm.h"
#include <atomic>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;

// ------------------------------------------------------------------------------------------------ multi-pair MSE
__device__ __forceinline__ float4 ld4_any(const void* p, int dtype, int64_t i) {
  if (dtype == EVLM_BF16) {
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p) + i);
    const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i);
}
__device__ __forceinline__ float ld1_any(const void* p, int dtype, int64_t i) {
  return dtype == EVLM_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]) : reinterpret_cast<const float*>(p)[i];
}

// 1-D grid; every block walks every pair with a grid stride, so pairs of very different sizes (ViT attention maps: 60M
// elements, text attention maps: 2M) load all SMs evenly; four independent 16-byte loads per tensor are in flight per thread.
__global__ void __launch_bounds__(256) mse_pairs_fwd_kernel(const evlm_mse_pair* __restrict__ pairs, int npairs, float* __restrict__ out) {
  __shared__ float red[32];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  for (int pi = 0; pi < npairs; ++pi) {
    const evlm_mse_pair pr = pairs[pi];
    const int64_t n4 = pr.n >> 2;
    const bool vec = ((reinterpret_cast<uintptr_t>(pr.s) & 15) == 0) && ((reinterpret_cast<uintptr_t>(pr.t) & 15) == 0);
    float acc = 0.f;
    if (vec && pr.rowdot != nullptr && (pr.row_len & 3) == 0 && pr.row_len > 0 && pr.n % pr.row_len == 0) {
      // attention map whose gradient will be formed INSIDE the attention backward (evlm_attn_args.dp_kd_coef): besides the squared
      // error, leave the per-row sums  sum_j (s_ij - t_ij) s_ij  (unscaled) — the softmax backward needs them and both maps are in
      // registers here.  A WARP walks whole rows (two at a time, every lane a float4 column of both): one shuffle reduction and one
      // plain store per row, no atomics, no per-element row arithmetic.
      const int lane = threadIdx.x & 31;
      const int64_t rl4 = pr.row_len >> 2, nrows = pr.n / pr.row_len;
      const int64_t warp0 = tid >> 5, nwarps = stride >> 5;
      for (int64_t r0 = warp0; r0 < nrows; r0 += 2 * nwarps) {
        const int64_t r1 = r0 + nwarps;
        const bool two = r1 < nrows;
        float dot0 = 0.f, dot1 = 0.f;
        for (int64_t c = lane; c < rl4; c += 64) {
          const bool second = c + 32 < rl4;
          float4 a[4], b[4];
          a[0] = ld4_any(pr.s, pr.s_dtype, (r0 * rl4 + c) * 4);
          b[0] = ld4_any(pr.t, pr.t_dtype, (r0 * rl4 + c) * 4);
          if (second) {
            a[1] = ld4_any(pr.s, pr.s_dtype, (r0 * rl4 + c + 32) * 4);
            b[1] = ld4_any(pr.t, pr.t_dtype, (r0 * rl4 + c + 32) * 4);
          }
          if (two) {
            a[2] = ld4_any(pr.s, pr.s_dtype, (r1 * rl4 + c) * 4);
            b[2] = ld4_any(pr.t, pr.t_dtype, (r1 * rl4 + c) * 4);
            if (second) {
              a[3] = ld4_any(pr.s, pr.s_dtype, (r1 * rl4 + c + 32) * 4);
              b[3] = ld4_any(pr.t, pr.t_dtype, (r1 * rl4 + c + 32) * 4);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if ((u & 1) && !second) continue;
            if ((u & 2) && !two) continue;
            const float d0 = a[u].x - b[u].x, d1 = a[u].y - b[u].y, d2 = a[u].z - b[u].z, d3 = a[u].w - b[u].w;
            acc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
            const float dt = d0 * a[u].x + d1 * a[u].y + d2 * a[u].z + d3 * a[u].w;
            if (u & 2) dot1 += dt;
            else dot0 += dt;
          }
        }
        dot0 = warp_sum(dot0);
        if (two) dot1 = warp_sum(dot1);
        if (lane == 0) {
          pr.rowdot[r0] = dot0;
          if (two) pr.rowdot[r1] = dot1;
        }
      }
    } else if (vec && pr.rowdot == nullptr) {
      int64_t i = tid;
      for (; i + 3 * stride < n4; i += 4 * stride) {
        float4 a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          a[u] = ld4_any(pr.s, pr.s_dtype, (i + u * stride) * 4);
          b[u] = ld4_any(pr.t, pr.t_dtype, (i + u * stride) * 4);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float d0 = a[u].x - b[u].x, d1 = a[u].y - b[u].y, d2 = a[u].z - b[u].z, d3 = a[u].w - b[u].w;
          acc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        }
      }
      for (; i < n4; i += stride) {
        const float4 a = ld4_any(pr.s, pr.s_dtype, i * 4), b = ld4_any(pr.t, pr.t_dtype, i * 4);
        const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
        acc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
      }
      for (int64_t j = n4 * 4 + tid; j < pr.n; j += stride) {
        const float d = ld1_any(pr.s, pr.s_dtype, j) - ld1_any(pr.t, pr.t_dtype, j);
        acc += d * d;
      }
    } else {
      // unaligned maps (or rows the warp-per-row loop cannot take) that want the row sums leave them one atomic per element, as the
      // backward's scalar path does
      for (int64_t j = tid; j < pr.n; j += stride) {
        const float a = ld1_any(pr.s, pr.s_dtype, j);
        const float d = a - ld1_any(pr.t, pr.t_dtype, j);
        acc += d * d;
        if (pr.rowdot != nullptr) atomicAdd(pr.rowdot + j / pr.row_len, d * a);
      }
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) atomicAdd(out + pi, acc * (pr.scale / (float)pr.n));
  }
}

__global__ void __launch_bounds__(256) mse_pairs_bwd_kernel(const evlm_mse_pair* __restrict__ pairs, int npairs, const float* __restrict__ dout) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  for (int pi = 0; pi < npairs; ++pi) {
    const evlm_mse_pair pr = pairs[pi];
    if (pr.ds == nullptr) continue;
    float* ds = reinterpret_cast<float*>(pr.ds);
    const float k = dout[pi] * pr.scale * 2.f / (float)pr.n;
    const int64_t n4 = pr.n >> 2;
    const bool vec = ((reinterpret_cast<uintptr_t>(pr.s) & 15) == 0) && ((reinterpret_cast<uintptr_t>(pr.t) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(ds) & 15) == 0);
    if (vec && pr.rowdot != nullptr) {
      // attention map: besides ds, the per-row dot products sum_j ds_ij s_ij.  A warp covers 32 consecutive float4 (128 elements):
      // at most TWO rows when row_len >= 128 elements... in general the lanes of a warp fall into runs of equal row index; the run
      // heads are found with a shuffle and every run leaves as one atomicAdd.
      const int lane = threadIdx.x & 31;
      const int64_t rl4 = pr.row_len >> 2;
      const int64_t n4r = (n4 + 31) & ~(int64_t)31;        // every lane of a warp takes part in the shuffles
      constexpr int U = 2;                                 // independent float4 pairs in flight per thread and iteration
      for (int64_t i0 = tid; i0 < n4r; i0 += U * stride) {
        float4 a[U], b[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t i = i0 + u * stride;
          ok[u] = i < n4;
          if (ok[u]) {
            a[u] = ld4_any(pr.s, pr.s_dtype, i * 4);
            b[u] = ld4_any(pr.t, pr.t_dtype, i * 4);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t i = i0 + u * stride;
          if (i >= n4r) break;                             // (warp-uniform: n4r and the strides are multiples of 32)
          float dot = 0.f;
          int64_t row = -1;
          if (ok[u]) {
            const float4 d = make_float4(k * (a[u].x - b[u].x), k * (a[u].y - b[u].y), k * (a[u].z - b[u].z), k * (a[u].w - b[u].w));
            *reinterpret_cast<float4*>(ds + i * 4) = d;
            dot = d.x * a[u].x + d.y * a[u].y + d.z * a[u].z + d.w * a[u].w;
            row = n4r < 0xffffffffLL ? (int64_t)((uint32_t)i / (uint32_t)rl4) : i / rl4;     // (a 64-bit division costs ~40 instructions)
          }
          // segmented suffix sums: lane l ends up with the sum over the lanes >= l of its run of equal rows
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_down_sync(0xffffffffu, dot, o);
            const int64_t r2 = __shfl_down_sync(0xffffffffu, row, o);
            if (lane + o < 32 && r2 == row) dot += v;
          }
          const int64_t rprev = __shfl_up_sync(0xffffffffu, row, 1);
          if (ok[u] && (lane == 0 || rprev != row)) atomicAdd(pr.rowdot + row, dot);
        }
      }
    } else if (vec) {
      int64_t i = tid;
      for (; i + 3 * stride < n4; i += 4 * stride) {
        float4 a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          a[u] = ld4_any(pr.s, pr.s_dtype, (i + u * stride) * 4);
          b[u] = ld4_any(pr.t, pr.t_dtype, (i + u * stride) * 4);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          *reinterpret_cast<float4*>(ds + (i + u * stride) * 4) =
              make_float4(k * (a[u].x - b[u].x), k * (a[u].y - b[u].y), k * (a[u].z - b[u].z), k * (a[u].w - b[u].w));
      }
      for (; i < n4; i += stride) {
        const float4 a = ld4_any(pr.s, pr.s_dtype, i * 4), b = ld4_any(pr.t, pr.t_dtype, i * 4);
        *reinterpret_cast<float4*>(ds + i * 4) = make_float4(k * (a.x - b.x), k * (a.y - b.y), k * (a.z - b.z), k * (a.w - b.w));
      }
      for (int64_t j = n4 * 4 + tid; j < pr.n; j += stride) ds[j] = k * (ld1_any(pr.s, pr.s_dtype, j) - ld1_any(pr.t, pr.t_dtype, j));
    } else {
      for (int64_t j = tid; j < pr.n; j += stride) {
        const float a = ld1_any(pr.s, pr.s_dtype, j);
        const float d = k * (a - ld1_any(pr.t, pr.t_dtype, j));
        ds[j] = d;
        if (pr.rowdot != nullptr) atomicAdd(pr.rowdot + j / pr.row_len, d * a);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ row softmax statistics
// block per row: returns (max, log-sum-exp) of x[0..V) * inv_temp.
// ONE pass over the row (online max / sum per thread, 8 values in flight per thread through 8-byte loads), then one block-wide
// combine: the row statistics are HBM-bound, and a 30522-wide fp32 row read twice with dependent scalar loads ran at ~1.3 TB/s.
__device__ __forceinline__ void row_lse(const float* __restrict__ x, int V, float inv_temp, float* red, float& mx, float& lse) {
  float m = -INFINITY, s = 0.f;
  auto fold8 = [&](const float (&v)[8]) {
    float bm = fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7])));
    if (bm > m) {
      s *= __expf(m - bm);     // m = -inf on the first batch: exp(-inf) = 0 and s is 0 anyway
      m = bm;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) s += __expf(v[u] - m);
  };
  int done = 0;
  if ((reinterpret_cast<uintptr_t>(x) & 7) == 0) {
    const float2* x2 = reinterpret_cast<const float2*>(x);
    const int n2 = V >> 1;
    int i = threadIdx.x;
    for (; i + 3 * (int)blockDim.x < n2; i += 4 * blockDim.x) {
      const float2 a = x2[i], b = x2[i + blockDim.x], c = x2[i + 2 * blockDim.x], d = x2[i + 3 * blockDim.x];
      const float v[8] = {a.x * inv_temp, a.y * inv_temp, b.x * inv_temp, b.y * inv_temp, c.x * inv_temp, c.y * inv_temp, d.x * inv_temp, d.y * inv_temp};
      fold8(v);
    }
    for (; i < n2; i += blockDim.x) {
      const float2 a = x2[i];
      const float lo = a.x * inv_temp, hi = a.y * inv_temp;
      const float bm = fmaxf(lo, hi);
      if (bm > m) {
        s *= __expf(m - bm);
        m = bm;
      }
      s += __expf(lo - m) + __expf(hi - m);
    }
    done = n2 * 2;
  }
  for (int v = done + threadIdx.x; v < V; v += blockDim.x) {
    const float xv = x[v] * inv_temp;
    if (xv > m) {
      s *= __expf(m - xv);
      m = xv;
    }
    s += __expf(xv - m);
  }
  const float mb = block_max(m, red);
  s = block_sum(m == -INFINITY ? 0.f : s * __expf(m - mb), red);
  mx = mb;
  lse = mb + logf(s);
}

__global__ void __launch_bounds__(256) xent_fwd_kernel(const float* __restrict__ logits, int64_t ld, int V, const int64_t* __restrict__ labels,
                                                       int64_t ignore_index, float ls, float* __restrict__ loss_rows, float* __restrict__ lse_o) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const float* x = logits + r * ld;
  float mx, lse;
  row_lse(x, V, 1.f, red, mx, lse);
  const int64_t lab = labels[r];
  float sumx = 0.f;
  if (ls > 0.f) {
    for (int v = threadIdx.x; v < V; v += blockDim.x) sumx += x[v];
    sumx = block_sum(sumx, red);
  }
  if (threadIdx.x == 0) {
    if (lse_o) lse_o[r] = lse;
    float loss = 0.f;
    if (lab != ignore_index) {
      // -(1-ls) * logp[lab] - ls/V * sum_v logp[v]   with the label itself getting (1-ls) instead of ls/V (scatter_, :1291-1292)
      const float logp_lab = x[lab] - lse;
      if (ls > 0.f) {
        const float neg = ls / (float)V;
        const float sum_logp = sumx - (float)V * lse;
        loss = -((1.f - ls) * logp_lab + neg * (sum_logp - logp_lab));
      } else {
        loss = -logp_lab;
      }
    }
    loss_rows[r] = loss;
  }
}

__global__ void __launch_bounds__(256) xent_bwd_kernel(const float* __restrict__ logits, int64_t ld, int V, const int64_t* __restrict__ labels,
                                                       int64_t ignore_index, float ls, const float* __restrict__ lse, const float* __restrict__ g_rows,
                                                       float* __restrict__ dl, int64_t ld_d, int accumulate) {
  const int64_t r = blockIdx.x;
  const float* x = logits + r * ld;
  float* d = dl + r * ld_d;
  const int64_t lab = labels[r];
  const float g = (lab == ignore_index) ? 0.f : g_rows[r];
  const float l = lse[r];
  const float neg = ls > 0.f ? ls / (float)V : 0.f;
  // d loss / d x_v = sum_target * softmax_v - target_v ; sum_target = (1-ls) + neg*(V-1)
  const float tsum = ls > 0.f ? (1.f - ls) + neg * (float)(V - 1) : 1.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float p = __expf(x[v] - l);
    const float tgt = (v == lab) ? (1.f - ls) : neg;
    const float val = g * (tsum * p - tgt);
    d[v] = accumulate ? d[v] + val : val;
  }
}

__global__ void __launch_bounds__(256) kl_fwd_kernel(const float* __restrict__ s, const float* __restrict__ t, int64_t ld_s, int64_t ld_t, int V,
                                                     float inv_temp, float* __restrict__ kl_rows, float* __restrict__ lse_s_o,
                                                     float* __restrict__ lse_t_o) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const float* xs = s + r * ld_s;
  const float* xt = t + r * ld_t;
  float ms, ls_, mt, lt;
  row_lse(xs, V, inv_temp, red, ms, ls_);
  row_lse(xt, V, inv_temp, red, mt, lt);
  float acc = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float lpt = xt[v] * inv_temp - lt;
    const float lps = xs[v] * inv_temp - ls_;
    const float pt = __expf(lpt);
    acc += pt > 0.f ? pt * (lpt - lps) : 0.f;   // KLDivLoss: 0 where target == 0
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) {
    kl_rows[r] = acc;
    if (lse_s_o) lse_s_o[r] = ls_;
    if (lse_t_o) lse_t_o[r] = lt;
  }
}
// d kl_row / d s_v = inv_temp * (softmax(s/T)_v - softmax(t/T)_v)
__global__ void __launch_bounds__(256) kl_bwd_kernel(const float* __restrict__ s, const float* __restrict__ t, int64_t ld_s, int64_t ld_t, int V,
                                                     float inv_temp, const float* __restrict__ lse_s, const float* __restrict__ lse_t,
                                                     const float* __restrict__ g_rows, float* __restrict__ dl, int64_t ld_d, int accumulate) {
  const int64_t r = blockIdx.x;
  const float* xs = s + r * ld_s;
  const float* xt = t + r * ld_t;
  float* d = dl + r * ld_d;
  const float g = g_rows[r] * inv_temp, a = lse_s[r], b = lse_t[r];
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float val = g * (__expf(xs[v] * inv_temp - a) - __expf(xt[v] * inv_temp - b));
    d[v] = accumulate ? d[v] + val : val;
  }
}

__global__ void __launch_bounds__(256) soft_xent_fwd_kernel(const float* __restrict__ logits, int64_t ld, const float* __restrict__ labels,
                                                            int64_t ld_l, int V, float* __restrict__ loss_rows, float* __restrict__ lse_o) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const float* x = logits + r * ld;
  const float* y = labels + r * ld_l;
  float mx, lse;
  row_lse(x, V, 1.f, red, mx, lse);
  float acc = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) acc += y[v] * (x[v] - lse);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) {
    loss_rows[r] = -acc;
    if (lse_o) lse_o[r] = lse;
  }
}
// d/dx_v = (sum_u y_u) softmax_v - y_v
__global__ void __launch_bounds__(256) soft_xent_bwd_kernel(const float* __restrict__ logits, int64_t ld, const float* __restrict__ labels,
                                                            int64_t ld_l, int V, const float* __restrict__ lse, const float* __restrict__ g_rows,
                                                            float* __restrict__ dl, int64_t ld_d, int accumulate) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const float* x = logits + r * ld;
  const float* y = labels + r * ld_l;
  float* d = dl + r * ld_d;
  float ys = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) ys += y[v];
  ys = block_sum(ys, red);
  const float g = g_rows[r], l = lse[r];
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float val = g * (ys * __expf(x[v] - l) - y[v]);
    d[v] = accumulate ? d[v] + val : val;
  }
}

__global__ void __launch_bounds__(256) reduce_sum_kernel(const float* __restrict__ x, int64_t n, float scale, float* __restrict__ out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) acc += x[i];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) atomicAdd(out, acc * scale);
}

// ------------------------------------------------------------------------------------------------ L2 normalise (warp per row)
__global__ void l2norm_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, float* __restrict__ inv_norm, int64_t rows, int D) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  float s = 0.f;
  for (int c = lane; c < D; c += 32) { const float v = x[r * D + c]; s += v * v; }
  s = warp_sum(s);
  const float inv = 1.f / fmaxf(sqrtf(s), 1e-12f);  // F.normalize eps
  for (int c = lane; c < D; c += 32) y[r * D + c] = x[r * D + c] * inv;
  if (lane == 0 && inv_norm) inv_norm[r] = inv;
}
// dx = inv * (dy - y * <dy, y>)
__global__ void l2norm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ inv_norm,
                                  float* __restrict__ dx, int64_t rows, int D) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  float s = 0.f;
  for (int c = lane; c < D; c += 32) s += dy[r * D + c] * y[r * D + c];
  s = warp_sum(s);
  const float inv = inv_norm[r];
  for (int c = lane; c < D; c += 32) dx[r * D + c] = inv * (dy[r * D + c] - y[r * D + c] * s);
}

// ------------------------------------------------------------------------------------------------ ITM negative sampling
// One warp per row b: w_j = softmax(sim[b,:])_j + 1e-5, zeroed where j == b (idx == NULL) or idx[j] == idx[b];
// inverse-CDF draw with u[b].  Sequential prefix over <= a few thousand entries: negligible.
__global__ void itm_sample_kernel(const float* __restrict__ sim, int64_t ld, const int64_t* __restrict__ idx, const float* __restrict__ u,
                                  int64_t* __restrict__ neg, int B) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* x = sim + (int64_t)b * ld;
  float m = -INFINITY;
  for (int j = lane; j < B; j += 32) m = fmaxf(m, x[j]);
  m = warp_max(m);
  float s = 0.f;
  for (int j = lane; j < B; j += 32) s += __expf(x[j] - m);
  s = warp_sum(s);
  const int64_t my = idx ? idx[b] : 0;
  float tot = 0.f;
  for (int j = lane; j < B; j += 32) {
    const bool ex = idx ? (idx[j] == my) : (j == b);
    tot += ex ? 0.f : (__expf(x[j] - m) / s + 1e-5f);
  }
  tot = warp_sum(tot);
  if (lane == 0) {
    const float target = u[b] * tot;
    float c = 0.f;
    int pick = -1, last_ok = -1;
    for (int j = 0; j < B; ++j) {
      const bool ex = idx ? (idx[j] == my) : (j == b);
      if (ex) continue;
      last_ok = j;
      c += __expf(x[j] - m) / s + 1e-5f;
      if (c > target) { pick = j; break; }
    }
    if (pick < 0) pick = last_ok >= 0 ? last_ok : b;
    neg[b] = pick;
  }
}

static inline unsigned grid_for(int64_t n, int threads, int64_t cap = 148 * 8) {
  int64_t b = (n + threads - 1) / threads;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}
}  // namespace evlm
using namespace evlm;
#define ST(s) reinterpret_cast<cudaStream_t>(s)
#define COUNT(n) g_launch_count.fetch_add(n, std::memory_order_relaxed)

extern "C" int evlm_mse_pairs_fwd(const evlm_mse_pair* pairs_dev, int npairs, float* out, void* stream) {
  if (!pairs_dev || npairs <= 0 || !out) return EVLM_EINVAL;
  cudaMemsetAsync(out, 0, npairs * sizeof(float), ST(stream));
  mse_pairs_fwd_kernel<<<148 * 6, 256, 0, ST(stream)>>>(pairs_dev, npairs, out);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_mse_pairs_bwd(const evlm_mse_pair* pairs_dev, int npairs, const float* dout, void* stream) {
  if (!pairs_dev || npairs <= 0 || !dout) return EVLM_EINVAL;
  mse_pairs_bwd_kernel<<<148 * 6, 256, 0, ST(stream)>>>(pairs_dev, npairs, dout);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_xent_fwd(const float* logits, int64_t ld, int64_t rows, int V, const int64_t* labels, int64_t ignore_index,
                             float label_smoothing, float* loss_rows, float* lse, void* stream) {
  if (!logits || !labels || !loss_rows || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  xent_fwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(logits, ld, V, labels, ignore_index, label_smoothing, loss_rows, lse);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_xent_bwd(const float* logits, int64_t ld, int64_t rows, int V, const int64_t* labels, int64_t ignore_index,
                             float label_smoothing, const float* lse, const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate,
                             void* stream) {
  if (!logits || !labels || !lse || !g_rows || !dlogits || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  xent_bwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(logits, ld, V, labels, ignore_index, label_smoothing, lse, g_rows, dlogits, ld_d, accumulate);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_kl_fwd(const float* s_logits, const float* t_logits, int64_t ld_s, int64_t ld_t, int64_t rows, int V, float inv_temp,
                           float* kl_rows, float* lse_s, float* lse_t, void* stream) {
  if (!s_logits || !t_logits || !kl_rows || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  kl_fwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(s_logits, t_logits, ld_s, ld_t, V, inv_temp, kl_rows, lse_s, lse_t);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_kl_bwd(const float* s_logits, const float* t_logits, int64_t ld_s, int64_t ld_t, int64_t rows, int V, float inv_temp,
                           const float* lse_s, const float* lse_t, const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate,
                           void* stream) {
  if (!s_logits || !t_logits || !lse_s || !lse_t || !g_rows || !dlogits || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  kl_bwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(s_logits, t_logits, ld_s, ld_t, V, inv_temp, lse_s, lse_t, g_rows, dlogits, ld_d, accumulate);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_soft_xent_fwd(const float* logits, int64_t ld, const float* labels, int64_t ld_l, int64_t rows, int V, float* loss_rows,
                                  float* lse, void* stream) {
  if (!logits || !labels || !loss_rows || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  soft_xent_fwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(logits, ld, labels, ld_l, V, loss_rows, lse);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_soft_xent_bwd(const float* logits, int64_t ld, const float* labels, int64_t ld_l, int64_t rows, int V, const float* lse,
                                  const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate, void* stream) {
  if (!logits || !labels || !lse || !g_rows || !dlogits || rows < 0 || V <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  soft_xent_bwd_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(logits, ld, labels, ld_l, V, lse, g_rows, dlogits, ld_d, accumulate);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_reduce_sum(const float* x, int64_t n, float scale, float* out, int32_t accumulate, void* stream) {
  if (!x || !out || n < 0) return EVLM_EINVAL;
  if (!accumulate) cudaMemsetAsync(out, 0, sizeof(float), ST(stream));
  if (n == 0) return EVLM_OK;
  reduce_sum_kernel<<<grid_for(n, 256, 148 * 4), 256, 0, ST(stream)>>>(x, n, scale, out);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_l2norm_fwd(const float* x, float* y, float* inv_norm, int64_t rows, int D, void* stream) {
  if (!x || !y || rows < 0 || D <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  l2norm_fwd_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, ST(stream)>>>(x, y, inv_norm, rows, D);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_l2norm_bwd(const float* dy, const float* y, const float* inv_norm, float* dx, int64_t rows, int D, void* stream) {
  if (!dy || !y || !inv_norm || !dx || rows < 0 || D <= 0) return EVLM_EINVAL;
  if (rows == 0) return EVLM_OK;
  l2norm_bwd_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, ST(stream)>>>(dy, y, inv_norm, dx, rows, D);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
extern "C" int evlm_itm_sample_neg(const float* sim, int64_t ld, const int64_t* idx, const float* u, int64_t* neg_out, int B, void* stream) {
  if (!sim || !u || !neg_out || B <= 1) return EVLM_EINVAL;
  itm_sample_kernel<<<(B + 3) / 4, 128, 0, ST(stream)>>>(sim, ld, idx, u, neg_out, B);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
