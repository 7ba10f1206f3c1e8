// SPADE+Style normalisation / modulation and InstanceNorm kernels (HBM-bound; NHWC bf16, fp32/fp64 statistics).
// One 16-byte vector (8 channels) per thread access, fully coalesced along the channel axis; per-channel
// partial sums live in registers, are combined across the block through shared memory and leave the block as one
// fp64 atomic per channel (so E[x^2]-E[x]^2 is formed without cancellation trouble).
#include "common.cuh"

namespace {

constexpr int NT = 256;

template <int ACT>
__device__ __forceinline__ float act_t(float v) {
  if (ACT == S2E_ACT_LRELU) return fmaxf(v, 0.2f * v);
  if (ACT == S2E_ACT_RELU) return fmaxf(v, 0.f);
  return v;
}

// ---------------------------------------------------------------- per-channel sum / sum of squares
// grid = (chunks, G) ; G = B when per_sample else 1 (then the chunk range spans all samples)
// Statistics are accumulated on SHIFTED data: sum (x - p), sum (x - p)^2 with the pivot p[c] = the group's first pixel.  The raw
// moments E[x^2] - E[x]^2 lose (mean / sigma)^2 of their relative precision to cancellation when they are built from fp32
// per-thread partial sums; with a pivot that is a sample of the channel the loss is ((p - mean) / sigma)^2, i.e. O(1).
// acc layout per group: [sum (x-p)][sum (x-p)^2][p], doubles.
__global__ void __launch_bounds__(NT) stats_kernel(const bf16* __restrict__ x, int HW, int C, long long pix_total,
                                                   int per_sample, double* __restrict__ acc) {
  extern __shared__ float red[];  // [lanes][ncg][8]
  const int g = blockIdx.y;
  const long long span = per_sample ? HW : pix_total;
  const long long base = per_sample ? (long long)g * HW : 0;
  const long long chunk = (span + gridDim.x - 1) / gridDim.x;
  const long long b0 = base + (long long)blockIdx.x * chunk;
  const long long b1 = min(base + span, b0 + chunk);
  const int cg = C >> 3;
  const int tid = threadIdx.x;
  double* out = acc + (size_t)g * 3 * C;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = tid % ncg, my_lane = tid / ncg;
    const int c = (cg0 + my_cg) * 8;
    float pv[8], a0[8], a1[8];
    unpack8(*reinterpret_cast<const bf16x8*>(x + base * C + c), pv);
    if (blockIdx.x == 0 && my_lane == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) out[2 * (size_t)C + c + j] = (double)pv[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) a0[j] = a1[j] = 0.f;
    auto eat = [&](const bf16x8& v) {
      float f[8];
      unpack8(v, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = f[j] - pv[j];
        a0[j] += d;
        a1[j] = fmaf(d, d, a1[j]);
      }
    };
    if (my_lane < lanes) {
      long long p = b0 + my_lane;
      for (; p + 3LL * lanes < b1; p += 4LL * lanes) {
        bf16x8 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = ld_stream8(x + (p + (long long)i * lanes) * C + c);
#pragma unroll
        for (int i = 0; i < 4; ++i) eat(v[i]);
      }
      for (; p < b1; p += lanes) eat(ld_stream8(x + p * C + c));
    }
#pragma unroll 1
    for (int a = 0; a < 2; ++a) {
      __syncthreads();
      if (my_lane < lanes) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[(my_lane * ncg + my_cg) * 8 + j] = a == 0 ? a0[j] : a1[j];
      }
      __syncthreads();
      for (int idx = tid; idx < ncg * 8; idx += NT) {
        float sum = 0.f;
        for (int l = 0; l < lanes; ++l) sum += red[l * ncg * 8 + idx];
        atomicAdd(out + (size_t)a * C + cg0 * 8 + idx, (double)sum);
      }
    }
  }
}

// in_scale (optional, one value per `group` consecutive statistic groups): statistics are those of x * in_scale without
// the product ever being formed: mean stays that of x, rstd' = s / sqrt(var * s^2 + eps), so (x - mean) * rstd' == norm(s x).
// count_dev (optional): the element count lives on the device (statistics merged across ranks, s2e_norm_merge); then
// count = count_dev[0] and count_unbiased = count_dev[0] * count_unbiased (the host passes the up-sampling factor).
__global__ void finalize_kernel(const double* __restrict__ acc, int G, int C, double count, float eps, float* mean,
                                float* rstd, float* running_mean, float* running_var, float momentum,
                                long long* nbt, const float* __restrict__ in_scale, int group, double count_unbiased,
                                const double* __restrict__ count_dev = nullptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && nbt) *nbt += 1;
  if (i >= G * C) return;
  if (count_dev) {
    count = count_dev[0];
    count_unbiased *= count;
  }
  const int g = i / C, c = i % C;
  const double s = acc[(size_t)g * 3 * C + c], ss = acc[(size_t)g * 3 * C + C + c], pivot = acc[(size_t)g * 3 * C + 2 * (size_t)C + c];
  const double ms = s / count;          // mean of the shifted data
  const double m = pivot + ms;
  double var = ss / count - ms * ms;
  if (var < 0) var = 0;
  mean[i] = (float)m;
  const double sc = in_scale ? (double)in_scale[g / group] : 1.0;
  rstd[i] = (float)(sc / sqrt(var * sc * sc + (double)eps));
  if (running_mean && g == 0) {
    const double cu = count_unbiased > 0 ? count_unbiased : count;   // element count BatchNorm sees (x4 when the statistics
    const double unb = cu > 1 ? var * cu / (cu - 1) : var;           // come from the source of a nearest-2x up-sampling)
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
  }
}

// Statistics of several ranks (or batch shards) combined into one record: rec[r] = [sum (x-p_r)][sum (x-p_r)^2][p_r] (C each,
// the acc format of stats_kernel) followed by the element count n_r.  Chan et al.'s pairwise update in rank order,
//   mean_r = p_r + s_r / n_r,  M2_r = ss_r - s_r^2 / n_r,  delta = mean_r - mean,
//   mean += delta n_r / (n + n_r),  M2 += M2_r + delta^2 n n_r / (n + n_r),
// never forms raw moments, so a channel whose mean is large against its spread, or shards whose means differ by many
// sigma, lose no precision.  Output in the acc format (pivot = global mean, sum (x - p) = 0, sum (x - p)^2 = M2) and the
// total count.  Empty shards (n_r = 0) are skipped.
__global__ void merge_kernel(const double* __restrict__ rec, int world, int C, double* __restrict__ acc,
                             double* __restrict__ count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const size_t stride = 3 * (size_t)C + 1;
  double n = 0, mean = 0, m2 = 0;
  for (int r = 0; r < world; ++r) {
    const double* q = rec + r * stride;
    const double nr = q[3 * (size_t)C];
    if (nr <= 0) continue;
    const double s = q[c], ss = q[C + c];
    const double mr = q[2 * (size_t)C + c] + s / nr;
    const double m2r = fmax(ss - s * s / nr, 0.0);
    const double tot = n + nr, d = mr - mean;
    mean = n == 0 ? mr : mean + d * (nr / tot);
    m2 = n == 0 ? m2r : m2 + m2r + d * d * (n * nr / tot);
    n = tot;
  }
  acc[c] = 0.0;
  acc[C + c] = m2;
  acc[2 * (size_t)C + c] = mean;
  if (c == 0) *count = n;
}

// Pixel index of x for output pixel q of sample b.  up_w == 0: x has the output's resolution.  up_w = W of the output:
// x is the (H/2, W/2) tensor the block input was nearest-2x up-sampled from (generator.py:50,86-93); the up-sampled copy
// is never materialised, the kernels read the source through this index map.
__device__ __forceinline__ long long x_pixel(int b, long long q, int HW, int up_w) {
  if (!up_w) return (long long)b * HW + q;
  const unsigned qq = (unsigned)q, uw = (unsigned)up_w;   // q < HW < 2^31: 32-bit division
  const unsigned h = qq / uw, w = qq - h * uw;
  return (long long)b * (HW >> 2) + (long long)((h >> 1) * (uw >> 1) + (w >> 1));
}

// bit j = (o[j] > 0): the activation mask of 8 channels in one byte
__device__ __forceinline__ uint8_t sign_bits8(const float* o) {
  uint32_t m = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) m |= (o[j] > 0.f ? 1u : 0u) << j;
  return (uint8_t)m;
}

// constants of the fused gamma|beta-convolution epilogue (conv_tc.cu): par[b][0..3][c]
__global__ void spade_params_kernel(const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ style,
                                    int B, int C, int per_sample, float* __restrict__ par) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i % C;
  const int so = per_sample ? b * C : 0;
  const float rs = rstd[so + c];
  float* o = par + (size_t)b * 4 * C + c;
  o[0] = rs;
  o[C] = -mean[so + c] * rs;
  o[2 * C] = style ? 1.f + style[(size_t)b * 2 * C + c] : 0.f;   // style == NULL: plain SPADE, no style term
  o[3 * C] = style ? style[(size_t)b * 2 * C + C + c] : 0.f;
}

// ---------------------------------------------------------------- SPADE+Style forward (elementwise, 8 B/elem)
// grid = (unit chunks, B).  A thread owns one 8-channel group: its per-channel constants (mean, rstd, style, with the output
// scale folded in) live in registers, then it streams pixels: 3 x 16-byte loads + 1 x 16-byte store per pixel.
//   out = act( t (1 + gamma) + os beta + v ),   t = os (x - mu) rs,   v = os (x (1 + s0) + s1)      (os = 1/2; plain SPADE: os = 1, v = 0)
// UP (nearest-2x up-sampled input): a thread walks SOURCE pixels, so x, t and v are formed once per four output pixels.
// amask (optional): one bit per element, set where out > 0 -- all the backward pass needs of `out` (16x fewer bytes).
template <int ACT, bool UP>
__global__ void __launch_bounds__(NT) spade_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ gb,
                                                       const float* __restrict__ style, const float* __restrict__ mean,
                                                       const float* __restrict__ rstd, int HW, int C, int per_sample,
                                                       bf16* __restrict__ out, uint8_t* __restrict__ amask, int W) {
  const int b = blockIdx.y;
  const int units = UP ? (HW >> 2) : HW;
  const long long chunk = ((long long)units + gridDim.x - 1) / gridDim.x;
  const long long q0 = (long long)blockIdx.x * chunk;
  const long long q1 = min((long long)units, q0 + chunk);
  const int cg = C >> 3;
  const float* mu_b = mean + (per_sample ? b * C : 0);
  const float* rs_b = rstd + (per_sample ? b * C : 0);
  const float* st_b = style ? style + (size_t)b * 2 * C : nullptr;
  const float os = style ? 0.5f : 1.0f;
  const long long base = (long long)b * HW;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = threadIdx.x % ncg, my_lane = threadIdx.x / ncg;
    if (my_lane >= lanes) continue;
    const int c = (cg0 + my_cg) * 8;
    const int mcol = cg0 + my_cg;
    float kA[8], kB[8], kC[8], kD[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float rs = rs_b[c + j];
      kA[j] = os * rs;
      kB[j] = -os * mu_b[c + j] * rs;
      kC[j] = st_b ? os * (1.f + st_b[c + j]) : 0.f;
      kD[j] = st_b ? os * st_b[C + c + j] : 0.f;
    }
    auto emit = [&](long long p, const float* t, const float* v, const bf16x8& vg, const bf16x8& vb) {
      float gf[8], bf_[8], o[8];
      unpack8(vg, gf);
      unpack8(vb, bf_);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = act_t<ACT>(fmaf(t[j], gf[j], t[j]) + fmaf(os, bf_[j], v[j]));
      st_stream8(out + p * C + c, pack8(o));
      if (amask) amask[p * cg + mcol] = sign_bits8(o);
    };
    if (UP) {
      const unsigned Ws = (unsigned)W >> 1;
      for (long long u = q0 + my_lane; u < q1; u += lanes) {
        const unsigned uu = (unsigned)u;
        const unsigned hs = uu / Ws, ws = uu - hs * Ws;
        const long long p00 = base + (long long)(2u * hs) * W + 2u * ws;
        const long long pk[4] = {p00, p00 + 1, p00 + W, p00 + W + 1};
        const bf16x8 vx = ld_stream8(x + ((long long)b * units + u) * C + c);
        bf16x8 vg[4], vb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          vg[k] = ld_stream8(gb + pk[k] * 2 * C + c);
          vb[k] = ld_stream8(gb + pk[k] * 2 * C + C + c);
        }
        float xf[8], t[8], v[8];
        unpack8(vx, xf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          t[j] = fmaf(xf[j], kA[j], kB[j]);
          v[j] = fmaf(xf[j], kC[j], kD[j]);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) emit(pk[k], t, v, vg[k], vb[k]);
      }
    } else {
      auto one = [&](long long p, const bf16x8& vx, const bf16x8& vg, const bf16x8& vb) {
        float xf[8], t[8], v[8];
        unpack8(vx, xf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          t[j] = fmaf(xf[j], kA[j], kB[j]);
          v[j] = fmaf(xf[j], kC[j], kD[j]);
        }
        emit(p, t, v, vg, vb);
      };
      long long q = q0 + my_lane;
      for (; q + lanes < q1; q += 2 * lanes) {      // two pixels in flight
        const long long pA = base + q, pB = base + q + lanes;
        const bf16x8 xa = ld_stream8(x + pA * C + c), xb = ld_stream8(x + pB * C + c);
        const bf16x8 ga = ld_stream8(gb + pA * 2 * C + c), gbb = ld_stream8(gb + pB * 2 * C + c);
        const bf16x8 ba = ld_stream8(gb + pA * 2 * C + C + c), bb = ld_stream8(gb + pB * 2 * C + C + c);
        one(pA, xa, ga, ba);
        one(pB, xb, gbb, bb);
      }
      for (; q < q1; q += lanes) {
        const long long p = base + q;
        one(p, ld_stream8(x + p * C + c), ld_stream8(gb + p * 2 * C + c), ld_stream8(gb + p * 2 * C + C + c));
      }
    }
  }
}

// ---------------------------------------------------------------- SPADE+Style backward
// Notation: g = os * dout * act'(out) (os = 1/2 with the style half, 1 for plain SPADE), xh = (x - mu) * rs,
// dxh = g * (1 + gamma).  BatchNorm / InstanceNorm backward needs m1 = mean(dxh), m2 = mean(dxh * xh) first:
//   pass 1 (reduce): per (sample, channel) raw moments  T1 = sum g, T2 = sum g x, T3 = sum g gamma, T4 = sum g gamma x
//                    -- no per-channel constants in the hot loop; everything else is linear in them (fold kernel)
//   fold           : S1 = sum dxh = T1 + T3,  S2 = sum dxh xh = rs (T2 + T4) + E (T1 + T3),  E = -mu rs,
//                    dstyle = (T2, T1),  sum dgamma = rs T2 + E T1,  sum dbeta = T1,  m1, m2
//   pass 2 (apply) : dx = g (rs (1 + gamma) + s0') + x (-rs^2 m2) + (rs^2 m2 mu - rs m1),  dgamma = g (x rs + E),  dbeta = g
// Nearest-2x up-sampled input (UP): a thread walks SOURCE pixels; the four output pixels of a source pixel share x, so x is
// loaded once, and pass 2 adds their four dx on the spot: the gradient leaves at the source resolution (the adjoint of the
// up-sampling costs no pass of its own and the full-resolution dx is never written).
template <int ACT>
__device__ __forceinline__ float gate(uint32_t mbits, int j, float os, float osn) {
  if (ACT == S2E_ACT_NONE) return os;
  return ((mbits >> j) & 1u) ? os : osn;
}

// block_channel_reduce with U units (pixels / source pixels) per loop trip, their loads free to overlap
template <int NACC, int U, typename F>
__device__ __forceinline__ void block_channel_reduce_u(int C, long long u_begin, long long u_end, double* out /*[NACC][C]*/, F&& body) {
  extern __shared__ float red[];
  const int cg = C >> 3;
  const int tid = threadIdx.x;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = tid % ncg, my_lane = tid / ncg;
    float acc[NACC][8];
#pragma unroll
    for (int a = 0; a < NACC; ++a)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[a][j] = 0.f;
    if (my_lane < lanes) {
      long long p = u_begin + my_lane;
      for (; p + (long long)(U - 1) * lanes < u_end; p += (long long)U * lanes) {
#pragma unroll
        for (int i = 0; i < U; ++i) body(p + (long long)i * lanes, (cg0 + my_cg) * 8, acc);
      }
      for (; p < u_end; p += lanes) body(p, (cg0 + my_cg) * 8, acc);
    }
    for (int a = 0; a < NACC; ++a) {
      __syncthreads();
      if (my_lane < lanes) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[(my_lane * ncg + my_cg) * 8 + j] = acc[a][j];
      }
      __syncthreads();
      for (int idx = tid; idx < ncg * 8; idx += NT) {
        float sum = 0.f;
        for (int l = 0; l < lanes; ++l) sum += red[l * ncg * 8 + idx];
        atomicAdd(out + (size_t)a * C + cg0 * 8 + idx, (double)sum);
      }
    }
  }
}

// pass 1.  racc[b][0..3][C] += T1..T4 (row 4 unused).  W = output width (UP only).
template <int ACT, bool UP>
__global__ void __launch_bounds__(NT) spade_bwd_reduce_kernel(const bf16* __restrict__ dout, const uint8_t* __restrict__ amask,
                                                              const bf16* __restrict__ x, const bf16* __restrict__ gb, int HW, int C,
                                                              double* __restrict__ racc, int W, int gstride, float os) {
  const int b = blockIdx.y;
  const int units = UP ? (HW >> 2) : HW;
  const long long chunk = ((long long)units + gridDim.x - 1) / gridDim.x;
  const long long u0 = (long long)blockIdx.x * chunk;
  const long long u1 = min((long long)units, u0 + chunk);
  const float osn = ACT == S2E_ACT_LRELU ? 0.2f * os : 0.f;
  const int cgs = C >> 3;
  const long long base = (long long)b * HW;
  auto body = [&](long long u, int c, float(*a)[8]) {
    if (UP) {
      const unsigned Ws = (unsigned)W >> 1, uu = (unsigned)u;
      const unsigned hs = uu / Ws, ws = uu - hs * Ws;
      const long long p00 = base + (long long)(2u * hs) * W + 2u * ws;
      const long long pk[4] = {p00, p00 + 1, p00 + W, p00 + W + 1};
      bf16x8 vd[4], vg[4];
      uint32_t mb[4];
      const bf16x8 vx = ld_stream8(x + ((long long)b * units + u) * C + c);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        vd[k] = ld_stream8(dout + pk[k] * C + c);
        vg[k] = ld_stream8(gb + pk[k] * gstride + c);
        mb[k] = ACT != S2E_ACT_NONE ? (uint32_t)amask[pk[k] * cgs + (c >> 3)] : 0xffu;
      }
      float xf[8], G[8], GG[8];
      unpack8(vx, xf);
#pragma unroll
      for (int j = 0; j < 8; ++j) G[j] = GG[j] = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float df[8], gf[8];
        unpack8(vd[k], df);
        unpack8(vg[k], gf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float g = df[j] * gate<ACT>(mb[k], j, os, osn);
          G[j] += g;
          GG[j] = fmaf(g, gf[j], GG[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        a[0][j] += G[j];
        a[1][j] = fmaf(G[j], xf[j], a[1][j]);
        a[2][j] += GG[j];
        a[3][j] = fmaf(GG[j], xf[j], a[3][j]);
      }
    } else {
      const long long p = base + u;
      const bf16x8 vd = ld_stream8(dout + p * C + c), vx = ld_stream8(x + p * C + c), vg = ld_stream8(gb + p * gstride + c);
      const uint32_t mbits = ACT != S2E_ACT_NONE ? (uint32_t)amask[p * cgs + (c >> 3)] : 0xffu;
      float df[8], xf[8], gf[8];
      unpack8(vd, df);
      unpack8(vx, xf);
      unpack8(vg, gf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float g = df[j] * gate<ACT>(mbits, j, os, osn);
        const float gg = g * gf[j];
        a[0][j] += g;
        a[1][j] = fmaf(g, xf[j], a[1][j]);
        a[2][j] += gg;
        a[3][j] = fmaf(gg, xf[j], a[3][j]);
      }
    }
  };
  block_channel_reduce_u<4, UP ? 1 : 4>(C, u0, u1, racc + (size_t)b * 5 * C, body);
}

// fold: raw moments -> per-sample statistics m1 / m2 (float [B][2][C]) or, for batch statistics, the per-channel sums
// S1 = sum dxh, S2 = sum dxh xh and their element count (double [2][C] + 1: `sums`, turned into m1 / m2 by the apply pass,
// so that ranks sharing batch statistics can add their sums in between), dstyle [B][2C] and, optionally, chsum [3][C] =
// per-channel sums over the whole batch of dgamma, dbeta and dx.  The last one needs no extra pass: the normalisation part
// of dx sums to zero over the pixels its statistics were taken from, so sum dx = sum_b (1 + s0[b]) * T1[b].  With
// statistics shared across ranks that holds over the global batch only; a rank's sum is then off by its share of the
// normalisation part, but the bias gradients it feeds are summed across ranks before use, and the shares cancel there.
__global__ void spade_style_bwd_fold_kernel(const double* __restrict__ racc, int B, int C, int per_sample, int frozen, double count,
                                            const float* __restrict__ style, const float* __restrict__ mean,
                                            const float* __restrict__ rstd, float* __restrict__ m12, double* __restrict__ sums,
                                            float* __restrict__ dstyle, float* __restrict__ chsum) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i % C;
  const double* r = racc + (size_t)b * 5 * C;
  if (dstyle) {
    dstyle[(size_t)b * 2 * C + c] = (float)r[C + c];        // d s0 = sum g x
    dstyle[(size_t)b * 2 * C + C + c] = (float)r[c];        // d s1 = sum g
  }
  if (per_sample) {
    const double rs = (double)rstd[(size_t)b * C + c], E = -(double)mean[(size_t)b * C + c] * rs;
    const double s1 = r[c] + r[2 * C + c];
    const double s2 = rs * (r[C + c] + r[3 * C + c]) + E * s1;
    m12[(size_t)b * 2 * C + c] = frozen ? 0.f : (float)(s1 / count);
    m12[(size_t)b * 2 * C + C + c] = frozen ? 0.f : (float)(s2 / count);
  }
  if (b == 0 && (!per_sample || chsum)) {
    double s1 = 0, s2 = 0, sg = 0, sb = 0, sx = 0;
    for (int bb = 0; bb < B; ++bb) {
      const double* q = racc + (size_t)bb * 5 * C;
      const int so = per_sample ? bb * C : 0;
      const double rs = (double)rstd[so + c], E = -(double)mean[so + c] * rs;
      const double t1 = q[c], t2 = q[C + c], t3 = q[2 * C + c], t4 = q[3 * C + c];
      s1 += t1 + t3;
      s2 += rs * (t2 + t4) + E * (t1 + t3);
      sb += t1;
      sg += rs * t2 + E * t1;
      if (style) sx += (1.0 + (double)style[(size_t)bb * 2 * C + c]) * t1;
    }
    if (!per_sample) {
      sums[c] = s1;
      sums[C + c] = s2;
      if (c == 0) sums[2 * (size_t)C] = count;
    }
    if (chsum) {
      chsum[c] = (float)sg;
      chsum[C + c] = (float)sb;
      // frozen statistics: the normalisation part of dx no longer sums to zero: sum dx = sum rstd dxh + (1 + s0) sum g
      chsum[2 * C + c] = (float)sx;
    }
  }
}

// pass 2.  dx: [B][HW][C], or with UP the gradient w.r.t. the half-resolution source [B][HW/4][C] (2x2 sums folded in).
template <int ACT, bool UP>
__global__ void __launch_bounds__(NT) spade_bwd_apply_kernel(const bf16* __restrict__ dout, const uint8_t* __restrict__ amask,
                                                             const bf16* __restrict__ x, const bf16* __restrict__ gb,
                                                             const float* __restrict__ style, const float* __restrict__ mean,
                                                             const float* __restrict__ rstd, const float* __restrict__ m12,
                                                             const double* __restrict__ sums, int frozen, int HW,
                                                             int C, int per_sample, bf16* __restrict__ dx, int dx_acc,
                                                             bf16* __restrict__ dgb, int W, int gstride) {
  const int b = blockIdx.y;
  const int units = UP ? (HW >> 2) : HW;
  const long long chunk = ((long long)units + gridDim.x - 1) / gridDim.x;
  const long long q0 = (long long)blockIdx.x * chunk;
  const long long q1 = min((long long)units, q0 + chunk);
  const int cg = C >> 3;
  const int so = per_sample ? b * C : 0;
  const float* m1p = m12 + (per_sample ? (size_t)b * 2 * C : 0);
  const float* s0p = style ? style + (size_t)b * 2 * C : nullptr;
  const float os = style ? 0.5f : 1.0f;
  const float osn = ACT == S2E_ACT_LRELU ? 0.2f * os : 0.f;
  const long long base = (long long)b * HW;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = threadIdx.x % ncg, my_lane = threadIdx.x / ncg;
    if (my_lane >= lanes) continue;
    const int c = (cg0 + my_cg) * 8;
    const int mcol = cg0 + my_cg;
    float kA[8], kR[8], kC[8], kD[8], kE[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float m1, m2;
      if (per_sample) {
        m1 = m1p[c + j];
        m2 = m1p[C + c + j];
      } else {    // batch statistics: from this batch's sums, or those of all ranks added together
        m1 = frozen ? 0.f : (float)(sums[c + j] / sums[2 * (size_t)C]);
        m2 = frozen ? 0.f : (float)(sums[C + c + j] / sums[2 * (size_t)C]);
      }
      const float rs = rstd[so + c + j], mu = mean[so + c + j];
      kR[j] = rs;
      kA[j] = rs + (s0p ? 1.f + s0p[c + j] : 0.f);
      kC[j] = -rs * rs * m2;
      kD[j] = rs * rs * m2 * mu - rs * m1;
      kE[j] = -mu * rs;
    }
    if (UP) {
      const unsigned Ws = (unsigned)W >> 1;
      for (long long u = q0 + my_lane; u < q1; u += lanes) {
        const unsigned uu = (unsigned)u;
        const unsigned hs = uu / Ws, ws = uu - hs * Ws;
        const long long p00 = base + (long long)(2u * hs) * W + 2u * ws;
        const long long pk[4] = {p00, p00 + 1, p00 + W, p00 + W + 1};
        const long long ps = ((long long)b * units + u) * C + c;
        bf16x8 vd[4], vg[4];
        uint32_t mb[4];
        const bf16x8 vx = ld_stream8(x + ps);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          vd[k] = ld_stream8(dout + pk[k] * C + c);
          vg[k] = ld_stream8(gb + pk[k] * gstride + c);
          mb[k] = ACT != S2E_ACT_NONE ? (uint32_t)amask[pk[k] * cg + mcol] : 0xffu;
        }
        float xf[8], xh[8], acc[8];
        unpack8(vx, xf);
        if (dx_acc) {
          unpack8(*reinterpret_cast<const bf16x8*>(dx + ps), acc);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xh[j] = fmaf(xf[j], kR[j], kE[j]);
          acc[j] = fmaf(4.f, fmaf(xf[j], kC[j], kD[j]), acc[j]);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float df[8], gf[8], odg[8], odb[8];
          unpack8(vd[k], df);
          unpack8(vg[k], gf);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float g = df[j] * gate<ACT>(mb[k], j, os, osn);
            acc[j] = fmaf(g, fmaf(kR[j], gf[j], kA[j]), acc[j]);
            odg[j] = g * xh[j];
            odb[j] = g;
          }
          st_stream8(dgb + pk[k] * 2 * C + c, pack8(odg));
          st_stream8(dgb + pk[k] * 2 * C + C + c, pack8(odb));
        }
        *reinterpret_cast<bf16x8*>(dx + ps) = pack8(acc);
      }
    } else {
      // two pixels per iteration: all six 16-byte loads are issued before the first use
      auto finish = [&](long long p, const bf16x8& vd, const bf16x8& vx, const bf16x8& vg, uint32_t mbits) {
        float df[8], xf[8], gf[8], odx[8], odg[8], odb[8], prev[8];
        if (dx_acc) unpack8(*reinterpret_cast<const bf16x8*>(dx + p * C + c), prev);
        unpack8(vd, df);
        unpack8(vx, xf);
        unpack8(vg, gf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float g = df[j] * gate<ACT>(mbits, j, os, osn);
          float d = fmaf(g, fmaf(kR[j], gf[j], kA[j]), fmaf(xf[j], kC[j], kD[j]));
          if (dx_acc) d += prev[j];
          odx[j] = d;
          odg[j] = g * fmaf(xf[j], kR[j], kE[j]);
          odb[j] = g;
        }
        *reinterpret_cast<bf16x8*>(dx + p * C + c) = pack8(odx);
        st_stream8(dgb + p * 2 * C + c, pack8(odg));
        st_stream8(dgb + p * 2 * C + C + c, pack8(odb));
      };
      long long q = q0 + my_lane;
      for (; q + lanes < q1; q += 2 * lanes) {
        const long long pA = base + q, pB = base + q + lanes;
        const bf16x8 da = ld_stream8(dout + pA * C + c), db = ld_stream8(dout + pB * C + c);
        const bf16x8 xa = ld_stream8(x + pA * C + c), xb = ld_stream8(x + pB * C + c);
        const bf16x8 ga = ld_stream8(gb + pA * gstride + c), gb2 = ld_stream8(gb + pB * gstride + c);
        const uint32_t ma = ACT != S2E_ACT_NONE ? (uint32_t)amask[pA * cg + mcol] : 0xffu;
        const uint32_t mb = ACT != S2E_ACT_NONE ? (uint32_t)amask[pB * cg + mcol] : 0xffu;
        finish(pA, da, xa, ga, ma);
        finish(pB, db, xb, gb2, mb);
      }
      for (; q < q1; q += lanes) {
        const long long p = base + q;
        const uint32_t mbits = ACT != S2E_ACT_NONE ? (uint32_t)amask[p * cg + mcol] : 0xffu;
        finish(p, ld_stream8(dout + p * C + c), ld_stream8(x + p * C + c), ld_stream8(gb + p * gstride + c), mbits);
      }
    }
  }
}

// ---------------------------------------------------------------- InstanceNorm (+act)
// same streaming structure as the SPADE kernels: grid (pixel chunks, B), per-channel constants in registers
// PAIR: the batch holds [fake ; real] halves of a discriminator feature (pix2pix_model.py:328-338) and the block normalises
// sample b AND sample b + pair_off; the feature-matching term sum |y_fake - y_real| (pix2pix_model.py:233-241, on the values as
// rounded to bf16) is reduced on the way and added to *pair_l1 -- no pass of its own over the feature map.
template <bool PAIR>
__global__ void __launch_bounds__(NT) instnorm_apply_kernel(const bf16* __restrict__ x, const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, int HW, int C, int act,
                                                            bf16* __restrict__ y, int pair_off, float* __restrict__ pair_l1) {
  const int b = blockIdx.y;
  const long long chunk = ((long long)HW + gridDim.x - 1) / gridDim.x;
  const long long q0 = (long long)blockIdx.x * chunk;
  const long long q1 = min((long long)HW, q0 + chunk);
  const int cg = C >> 3;
  float l1 = 0.f;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = threadIdx.x % ncg, my_lane = threadIdx.x / ncg;
    if (my_lane >= lanes) continue;
    const int c = (cg0 + my_cg) * 8;
    float ka[8], kb[8], ka2[8], kb2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      ka[j] = rstd[(size_t)b * C + c + j];
      kb[j] = -mean[(size_t)b * C + c + j] * ka[j];
      if (PAIR) {
        ka2[j] = rstd[(size_t)(b + pair_off) * C + c + j];
        kb2[j] = -mean[(size_t)(b + pair_off) * C + c + j] * ka2[j];
      }
    }
    const long long base = (long long)b * HW, base2 = (long long)(b + pair_off) * HW;
    auto emit = [&](long long p, const bf16x8& v) {
      float f[8], o[8];
      unpack8(v, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = act_apply(fmaf(f[j], ka[j], kb[j]), act);
      st_stream8(y + p * C + c, pack8(o));
    };
    auto emit2 = [&](long long q, const bf16x8& v, const bf16x8& v2) {
      float f[8], f2[8], o[8], o2[8];
      unpack8(v, f);
      unpack8(v2, f2);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = act_apply(fmaf(f[j], ka[j], kb[j]), act);
        o2[j] = act_apply(fmaf(f2[j], ka2[j], kb2[j]), act);
      }
      const bf16x8 r = pack8(o), r2 = pack8(o2);
      st_stream8(y + (base + q) * C + c, r);
      st_stream8(y + (base2 + q) * C + c, r2);
      unpack8(r, o);
      unpack8(r2, o2);
#pragma unroll
      for (int j = 0; j < 8; ++j) l1 += fabsf(o[j] - o2[j]);
    };
    long long q = q0 + my_lane;
    if (PAIR) {
      for (; q + lanes < q1; q += 2LL * lanes) {   // two pixels of both samples in flight
        const bf16x8 a0 = ld_stream8(x + (base + q) * C + c), a1 = ld_stream8(x + (base2 + q) * C + c);
        const bf16x8 c0 = ld_stream8(x + (base + q + lanes) * C + c), c1 = ld_stream8(x + (base2 + q + lanes) * C + c);
        emit2(q, a0, a1);
        emit2(q + lanes, c0, c1);
      }
      for (; q < q1; q += lanes) emit2(q, ld_stream8(x + (base + q) * C + c), ld_stream8(x + (base2 + q) * C + c));
    } else {
      for (; q + 3LL * lanes < q1; q += 4LL * lanes) {   // four 16-byte loads in flight per thread
        bf16x8 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = ld_stream8(x + (base + q + (long long)i * lanes) * C + c);
#pragma unroll
        for (int i = 0; i < 4; ++i) emit(base + q + (long long)i * lanes, v[i]);
      }
      for (; q < q1; q += lanes) emit(base + q, ld_stream8(x + (base + q) * C + c));
    }
  }
  if (PAIR) {   // every thread arrives here (the `continue` above only skips channel passes)
    __shared__ float red[NT / 32];
    l1 = warp_sum(l1);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = l1;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < NT / 32; ++i) t += red[i];
      atomicAdd(pair_l1, t);
    }
  }
}

// Backward, rewritten in round 2e like the SPADE kernels (section 4.2 of DESIGN.md).  The round-1 kernels read y only for
// the sign of the activation (a third of the reduce pass's bytes) and fetched mean / rstd per ELEMENT through __ldg inside the
// generic reduction helper (16 extra loads per 16-byte data load).  Now: the sign is that of fmaf(x, rstd, -mean*rstd) --
// the very expression the forward kernel rounds to y, so the mask is bit-identical -- per-channel constants live in
// registers, four pixels (eight 16-byte loads) are in flight per thread, and the apply pass uses folded constants:
//   g = dy * act'(v),  v = x*ka + kb            reduce:  S1 = sum g,  S2 = ka * sum g (x - mu)   ( = sum g * xhat )
//   dx = rstd (g - m1 - xhat m2) = g*ka + x*kc + kd,   kc = -ka^2 m2,  kd = -ka (m1 + kb m2)
// Bytes per element: reduce 4 (dy, x), apply 6 (dy, x in, dx out); before 6 and 8.
template <int ACT>
__device__ __forceinline__ float in_gate(float d, float v) {
  if (ACT == S2E_ACT_LRELU) return v > 0.f ? d : 0.2f * d;
  if (ACT == S2E_ACT_RELU) return v > 0.f ? d : 0.f;
  return d;
}

template <int ACT>
__global__ void __launch_bounds__(NT) instnorm_bwd_reduce_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                                 const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                 int HW, int C, double* __restrict__ racc) {
  extern __shared__ float red[];  // [lanes][ncg][8]
  const int b = blockIdx.y;
  const long long chunk = ((long long)HW + gridDim.x - 1) / gridDim.x;
  const long long base = (long long)b * HW;
  const long long q0 = (long long)blockIdx.x * chunk;
  const long long q1 = min((long long)HW, q0 + chunk);
  const int cg = C >> 3;
  const int tid = threadIdx.x;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = tid % ncg, my_lane = tid / ncg;
    const int c = (cg0 + my_cg) * 8;
    float ka[8], kb[8], mu[8], a0[8], a1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      ka[j] = rstd[(size_t)b * C + c + j];
      mu[j] = mean[(size_t)b * C + c + j];
      kb[j] = -mu[j] * ka[j];
      a0[j] = a1[j] = 0.f;
    }
    auto eat = [&](const bf16x8& vd, const bf16x8& vx) {
      float df[8], xf[8];
      unpack8(vd, df);
      unpack8(vx, xf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float g = in_gate<ACT>(df[j], fmaf(xf[j], ka[j], kb[j]));
        a0[j] += g;
        a1[j] = fmaf(g, xf[j] - mu[j], a1[j]);
      }
    };
    if (my_lane < lanes) {
      long long q = q0 + my_lane;
      for (; q + 3LL * lanes < q1; q += 4LL * lanes) {
        bf16x8 vd[4], vx[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          vd[i] = ld_stream8(dy + (base + q + (long long)i * lanes) * C + c);
          vx[i] = ld_stream8(x + (base + q + (long long)i * lanes) * C + c);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) eat(vd[i], vx[i]);
      }
      for (; q < q1; q += lanes) eat(ld_stream8(dy + (base + q) * C + c), ld_stream8(x + (base + q) * C + c));
    }
    // combine the pixel lanes through shared memory, one atomic per channel and block
#pragma unroll 1
    for (int a = 0; a < 2; ++a) {
      __syncthreads();
      if (my_lane < lanes) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[(my_lane * ncg + my_cg) * 8 + j] = a == 0 ? a0[j] : a1[j];
      }
      __syncthreads();
      for (int idx = tid; idx < ncg * 8; idx += NT) {
        float sum = 0.f;
        for (int l = 0; l < lanes; ++l) sum += red[l * ncg * 8 + idx];
        const int ch = cg0 * 8 + idx;
        if (a == 1) sum *= rstd[(size_t)b * C + ch];
        atomicAdd(racc + (size_t)b * 2 * C + (size_t)a * C + ch, (double)sum);
      }
    }
  }
}

template <int ACT>
__global__ void __launch_bounds__(NT) instnorm_bwd_apply_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                                const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                const double* __restrict__ racc, int HW, int C, bf16* __restrict__ dx) {
  const int b = blockIdx.y;
  const long long chunk = ((long long)HW + gridDim.x - 1) / gridDim.x;
  const long long q0 = (long long)blockIdx.x * chunk;
  const long long q1 = min((long long)HW, q0 + chunk);
  const int cg = C >> 3;
  const float inv = 1.f / (float)HW;
  for (int cg0 = 0; cg0 < cg; cg0 += NT) {
    const int ncg = min(NT, cg - cg0);
    const int lanes = NT / ncg;
    const int my_cg = threadIdx.x % ncg, my_lane = threadIdx.x / ncg;
    if (my_lane >= lanes) continue;
    const int c = (cg0 + my_cg) * 8;
    float ka[8], kb[8], kc[8], kd[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      ka[j] = rstd[(size_t)b * C + c + j];
      kb[j] = -mean[(size_t)b * C + c + j] * ka[j];
      const float m1 = (float)racc[(size_t)b * 2 * C + c + j] * inv;
      const float m2 = (float)racc[(size_t)b * 2 * C + C + c + j] * inv;
      kc[j] = -ka[j] * ka[j] * m2;
      kd[j] = -ka[j] * fmaf(kb[j], m2, m1);
    }
    const long long base = (long long)b * HW;
    auto emit = [&](long long p, const bf16x8& vd, const bf16x8& vx) {
      float df[8], xf[8], o[8];
      unpack8(vd, df);
      unpack8(vx, xf);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float g = in_gate<ACT>(df[j], fmaf(xf[j], ka[j], kb[j]));
        o[j] = fmaf(g, ka[j], fmaf(xf[j], kc[j], kd[j]));
      }
      st_stream8(dx + p * C + c, pack8(o));
    };
    long long q = q0 + my_lane;
    for (; q + 3LL * lanes < q1; q += 4LL * lanes) {
      bf16x8 vd[4], vx[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        vd[i] = ld_stream8(dy + (base + q + (long long)i * lanes) * C + c);
        vx[i] = ld_stream8(x + (base + q + (long long)i * lanes) * C + c);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) emit(base + q + (long long)i * lanes, vd[i], vx[i]);
    }
    for (; q < q1; q += lanes) emit(base + q, ld_stream8(dy + (base + q) * C + c), ld_stream8(x + (base + q) * C + c));
  }
}

// pixel chunks per sample for the streaming elementwise kernels: ~16 resident blocks per SM in total, and at least
// 8 pixels per pixel-lane so the per-thread constant setup is amortised
int ew_chunks(int HW, int B, int C) {
  const int ncg = (C >> 3) < NT ? (C >> 3) : NT;
  const int lanes = NT / ncg;
  long long want = ((long long)s2e_num_sms() * 16 + B - 1) / B;
  long long maxc = ((long long)HW + 8LL * lanes - 1) / (8LL * lanes);
  if (want > maxc) want = maxc;
  return (int)(want < 1 ? 1 : want);
}
int red_chunks(long long pixels, int G, int blocks_per_sm = 4) {
  // aim for `blocks_per_sm` resident blocks per SM overall (one full wave), at least 64 pixels per block
  long long want = blocks_per_sm == 4 ? ((long long)s2e_num_sms() * 4 + G - 1) / G : ((long long)s2e_num_sms() * blocks_per_sm) / G;
  long long maxc = (pixels + 63) / 64;
  if (want > maxc) want = maxc;
  return (int)(want < 1 ? 1 : want);
}
size_t red_smem(int C) {
  int ncg = (C >> 3) < NT ? (C >> 3) : NT;
  int lanes = NT / ncg;
  return (size_t)lanes * ncg * 8 * sizeof(float);
}

}  // namespace

extern "C" {

int s2e_norm_stats(const void* x, int B, int HW, int C, int per_sample, double* acc, void* stream) {
  S2E_REQUIRE(C % 8 == 0 && C >= 8, "norm_stats needs C %% 8 == 0 (C=%d)", C);
  cudaStream_t st = (cudaStream_t)stream;
  const int G = per_sample ? B : 1;
  S2E_CHECK_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * G * 3 * C, st));   // [sum (x-p)][sum (x-p)^2][pivot p] per group
  if ((long long)B * HW == 0) return S2E_OK;    // an empty batch (shard): zero sums, no pivot pixel to read
  const long long span = per_sample ? HW : (long long)B * HW;
  dim3 grid(red_chunks(span, G), G);
  stats_kernel<<<grid, NT, red_smem(C), st>>>((const bf16*)x, HW, C, (long long)B * HW, per_sample, acc);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_norm_finalize(const double* acc, int G, int C, double count, double count_unbiased, float eps, float* mean,
                      float* rstd, float* running_mean, float* running_var, float momentum, int64_t* nbt, void* stream) {
  finalize_kernel<<<ceil_div(G * C, 256), 256, 0, (cudaStream_t)stream>>>(acc, G, C, count, eps, mean, rstd, running_mean,
                                                                           running_var, momentum, (long long*)nbt, nullptr, 1,
                                                                           count_unbiased);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_norm_merge(const double* records, int world, int C, double* acc, double* count, void* stream) {
  S2E_REQUIRE(world >= 1 && C >= 1, "norm_merge: bad world %d / C %d", world, C);
  merge_kernel<<<ceil_div(C, 256), 256, 0, (cudaStream_t)stream>>>(records, world, C, acc, count);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_norm_finalize_merged(const double* acc, const double* count, int C, double unbiased_factor, float eps, float* mean,
                             float* rstd, float* running_mean, float* running_var, float momentum, int64_t* nbt, void* stream) {
  finalize_kernel<<<ceil_div(C, 256), 256, 0, (cudaStream_t)stream>>>(acc, 1, C, 0.0, eps, mean, rstd, running_mean, running_var,
                                                                      momentum, (long long*)nbt, nullptr, 1, unbiased_factor,
                                                                      count);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

// c[b] = (eps / is_b) * sum_{n in sample b, c} S2[n][c] * rstd'[n][c]^2   (one block per sample)
__global__ void sn_corr_coef_kernel(const double* __restrict__ racc, const float* __restrict__ rstd, const float* __restrict__ inv_sigma,
                                    int C, int group, float eps, float* __restrict__ coef) {
  const int b = blockIdx.x;
  float acc = 0.f;
  for (int i = threadIdx.x; i < group * C; i += blockDim.x) {
    const int n = b * group + i / C, c = i % C;
    const float r = rstd[(size_t)n * C + c];
    acc += (float)racc[(size_t)n * 2 * C + C + c] * r * r;
  }
  __shared__ float sh[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) coef[b] = eps / inv_sigma[b] * v;
  }
}
// dW[co][k] = - sum_b coef[b] * U[b][co] * V[b][k]
__global__ void sn_corr_apply_kernel(const float* __restrict__ coef, const float* __restrict__ U, const float* __restrict__ V, int Bn,
                                     int Cout, int K, float* __restrict__ dw) {
  const long long n = (long long)Cout * K;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i / K), k = (int)(i % K);
    float acc = 0.f;
    for (int b = 0; b < Bn; ++b) acc = fmaf(coef[b] * U[(size_t)b * Cout + co], V[(size_t)b * K + k], acc);
    dw[i] = -acc;
  }
}

int s2e_spade_params(const float* mean, const float* rstd, const float* style, int B, int C, int per_sample, float* par,
                     void* stream) {
  if (B * C == 0) return S2E_OK;
  spade_params_kernel<<<ceil_div(B * C, 256), 256, 0, (cudaStream_t)stream>>>(mean, rstd, style, B, C, per_sample, par);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_spade_style_fwd(const void* x, const void* gb, const float* style, const float* mean, const float* rstd, int B,
                        int HW, int C, int per_sample, int act, void* out, uint8_t* act_mask, int up_w, void* stream) {
  S2E_REQUIRE(C % 8 == 0, "spade_style_fwd needs C %% 8 == 0 (C=%d)", C);
  S2E_REQUIRE(up_w == 0 || (up_w % 2 == 0 && HW % up_w == 0 && (HW / up_w) % 2 == 0), "spade_style_fwd: bad up-sampled width %d", up_w);
  if ((long long)B * HW == 0) return S2E_OK;
  dim3 grid(ew_chunks(up_w ? HW / 4 : HW, B, C), B);
#define S2E_SPADE_FWD(ACT_, UP_)                                                                                          \
  spade_fwd_kernel<ACT_, UP_><<<grid, NT, 0, (cudaStream_t)stream>>>((const bf16*)x, (const bf16*)gb, style, mean, rstd, HW, C, \
                                                                     per_sample, (bf16*)out, act_mask, up_w)
  if (up_w) {
    if (act == S2E_ACT_LRELU) S2E_SPADE_FWD(S2E_ACT_LRELU, true);
    else if (act == S2E_ACT_RELU) S2E_SPADE_FWD(S2E_ACT_RELU, true);
    else S2E_SPADE_FWD(S2E_ACT_NONE, true);
  } else {
    if (act == S2E_ACT_LRELU) S2E_SPADE_FWD(S2E_ACT_LRELU, false);
    else if (act == S2E_ACT_RELU) S2E_SPADE_FWD(S2E_ACT_RELU, false);
    else S2E_SPADE_FWD(S2E_ACT_NONE, false);
  }
#undef S2E_SPADE_FWD
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

// ACT_ / UP_ dispatch of the SPADE+Style backward kernels
#define S2E_SPADE_BWD_DISPATCH(M)                        \
  do {                                                   \
    if (up_w) {                                          \
      if (act == S2E_ACT_LRELU) M(S2E_ACT_LRELU, true);  \
      else if (act == S2E_ACT_RELU) M(S2E_ACT_RELU, true); \
      else M(S2E_ACT_NONE, true);                        \
    } else {                                             \
      if (act == S2E_ACT_LRELU) M(S2E_ACT_LRELU, false); \
      else if (act == S2E_ACT_RELU) M(S2E_ACT_RELU, false); \
      else M(S2E_ACT_NONE, false);                       \
    }                                                    \
  } while (0)

static int spade_bwd_check(const uint8_t* act_mask, const float* style, const float* dstyle, int HW, int C, int act, int up_w,
                           int gb_stride) {
  S2E_REQUIRE(C % 8 == 0, "spade_style_bwd needs C %% 8 == 0 (C=%d)", C);
  S2E_REQUIRE(up_w == 0 || (up_w % 2 == 0 && HW % up_w == 0 && (HW / up_w) % 2 == 0), "spade_style_bwd: bad up-sampled width %d", up_w);
  S2E_REQUIRE(act == S2E_ACT_NONE || act_mask, "spade_style_bwd: the activation mask written by the forward pass is required");
  const int gstride = gb_stride > 0 ? gb_stride : 2 * C;
  S2E_REQUIRE(gstride >= C && gstride % 8 == 0, "spade_style_bwd: bad gamma stride %d", gstride);
  S2E_REQUIRE(style || !dstyle, "spade_style_bwd: plain SPADE (style == NULL) has no style gradient");
  return S2E_OK;
}

int s2e_spade_style_bwd_reduce(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                               const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act,
                               double* racc, double* sums, float* dstyle, float* chsum, int up_w, int gb_stride, void* stream) {
  S2E_REQUIRE((per_sample & 1) || sums, "spade_style_bwd_reduce: batch statistics need the `sums` buffer");
  cudaStream_t st = (cudaStream_t)stream;
  if ((long long)B * HW == 0) {   // an empty shard (its tensors may be NULL) adds nothing to the sums of its peers
    if (!(per_sample & 1)) S2E_CHECK_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C + 1), st));
    return S2E_OK;
  }
  int rc = spade_bwd_check(act_mask, style, dstyle, HW, C, act, up_w, gb_stride);
  if (rc) return rc;
  // racc: double [B][5][C] followed by float m12 [B][2][C]
  S2E_CHECK_CUDA(cudaMemsetAsync(racc, 0, sizeof(double) * B * 5 * C, st));
  float* m12 = (float*)(racc + (size_t)B * 5 * C);
  // per_sample bit 1: the statistics are constants (BatchNorm in eval mode: running statistics) -- no m1 / m2 terms
  const int frozen = (per_sample >> 1) & 1;
  per_sample &= 1;
  const int gstride = gb_stride > 0 ? gb_stride : 2 * C;
  const float os = style ? 0.5f : 1.0f;
  const int units = up_w ? HW / 4 : HW;     // source pixels when the up-sampling is folded in
  const double count = per_sample ? (double)HW : (double)B * HW;
#define S2E_SPADE_BWD_REDUCE(ACT_, UP_)                                                                                       \
  do {                                                                                                                        \
    /* the reduce pass runs as exactly ONE wave of resident blocks (its register count differs per instantiation) */        \
    int nb = 2;                                                                                                               \
    S2E_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, spade_bwd_reduce_kernel<ACT_, UP_>, NT, red_smem(C)));  \
    dim3 grid(red_chunks(units, B, nb < 1 ? 1 : (nb > 3 ? 3 : nb)), B);                                                       \
    spade_bwd_reduce_kernel<ACT_, UP_><<<grid, NT, red_smem(C), st>>>((const bf16*)dout, act_mask, (const bf16*)x, (const bf16*)gb, \
                                                                      HW, C, racc, up_w, gstride, os);                        \
    S2E_LAUNCH_CHECK();                                                                                                       \
  } while (0)
  S2E_SPADE_BWD_DISPATCH(S2E_SPADE_BWD_REDUCE);
#undef S2E_SPADE_BWD_REDUCE
  spade_style_bwd_fold_kernel<<<ceil_div(B * C, 256), 256, 0, st>>>(racc, B, C, per_sample, frozen, count, style, mean, rstd, m12,
                                                                    sums, dstyle, chsum);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_spade_style_bwd_apply(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                              const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act,
                              const double* racc, const double* sums, void* dx, int dx_accumulate, void* dgb, int up_w,
                              int gb_stride, void* stream) {
  if ((long long)B * HW == 0) return S2E_OK;
  int rc = spade_bwd_check(act_mask, style, nullptr, HW, C, act, up_w, gb_stride);
  if (rc) return rc;
  S2E_REQUIRE((per_sample & 1) || sums, "spade_style_bwd_apply: batch statistics need the `sums` buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const float* m12 = (const float*)(racc + (size_t)B * 5 * C);
  const int frozen = (per_sample >> 1) & 1;
  per_sample &= 1;
  const int gstride = gb_stride > 0 ? gb_stride : 2 * C;
  const int units = up_w ? HW / 4 : HW;
  dim3 grid2(ew_chunks(units, B, C), B);
#define S2E_SPADE_BWD_APPLY(ACT_, UP_)                                                                                        \
  spade_bwd_apply_kernel<ACT_, UP_><<<grid2, NT, 0, st>>>((const bf16*)dout, act_mask, (const bf16*)x, (const bf16*)gb, style, \
                                                          mean, rstd, m12, sums, frozen, HW, C, per_sample, (bf16*)dx,        \
                                                          dx_accumulate, (bf16*)dgb, up_w, gstride)
  S2E_SPADE_BWD_DISPATCH(S2E_SPADE_BWD_APPLY);
#undef S2E_SPADE_BWD_APPLY
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_spade_style_bwd(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                        const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act, double* racc,
                        void* dx, int dx_accumulate, void* dgb, float* dstyle, float* chsum, int up_w, int gb_stride,
                        void* stream) {
  // racc: double [B][5][C], float m12 [B][2][C], then the batch-statistics sums, double [2][C] + 1
  double* sums = racc + (size_t)B * 5 * C + (size_t)B * C;
  int rc = s2e_spade_style_bwd_reduce(dout, act_mask, x, gb, style, mean, rstd, B, HW, C, per_sample, act, racc, sums, dstyle,
                                      chsum, up_w, gb_stride, stream);
  if (rc) return rc;
  return s2e_spade_style_bwd_apply(dout, act_mask, x, gb, style, mean, rstd, B, HW, C, per_sample, act, racc, sums, dx,
                                   dx_accumulate, dgb, up_w, gb_stride, stream);
}
#undef S2E_SPADE_BWD_DISPATCH

int s2e_sn_in_correction(const double* racc, const float* rstd, const float* inv_sigma, int Bn, int group, int C, float eps,
                         const float* U, const float* V, int K, float* coef, float* dw, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  sn_corr_coef_kernel<<<Bn, 256, 0, st>>>(racc, rstd, inv_sigma, C, group, eps, coef);
  S2E_LAUNCH_CHECK();
  const long long n = (long long)C * K;
  long long g = (n + 255) / 256;
  if (g > (long long)s2e_num_sms() * 16) g = (long long)s2e_num_sms() * 16;
  sn_corr_apply_kernel<<<(unsigned)g, 256, 0, st>>>(coef, U, V, Bn, C, K, dw);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_instnorm_fwd(const void* x, int B, int HW, int C, int act, float eps, const float* in_scale, int group, double* acc,
                     float* mean, float* rstd, void* y, float* pair_l1, void* stream) {
  S2E_REQUIRE(!pair_l1 || B % 2 == 0, "instnorm_fwd: the fake / real pair sum needs an even batch (B = %d)", B);
  int rc = s2e_norm_stats(x, B, HW, C, 1, acc, stream);
  if (rc) return rc;
  finalize_kernel<<<ceil_div(B * C, 256), 256, 0, (cudaStream_t)stream>>>(acc, B, C, (double)HW, eps, mean, rstd, nullptr, nullptr,
                                                                           0.f, nullptr, in_scale, group > 0 ? group : 1, 0.0);
  S2E_LAUNCH_CHECK();
  if (pair_l1) {
    dim3 grid(ew_chunks(HW, B / 2, C), B / 2);
    instnorm_apply_kernel<true><<<grid, NT, 0, (cudaStream_t)stream>>>((const bf16*)x, mean, rstd, HW, C, act, (bf16*)y, B / 2, pair_l1);
  } else {
    dim3 grid(ew_chunks(HW, B, C), B);
    instnorm_apply_kernel<false><<<grid, NT, 0, (cudaStream_t)stream>>>((const bf16*)x, mean, rstd, HW, C, act, (bf16*)y, 0, nullptr);
  }
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_instnorm_bwd(const void* dy, const void* y, const void* x, const float* mean, const float* rstd, int B, int HW,
                     int C, int act, double* racc, void* dx, void* stream) {
  S2E_REQUIRE(C % 8 == 0, "instnorm_bwd needs C %% 8 == 0 (C=%d)", C);
  cudaStream_t st = (cudaStream_t)stream;
  S2E_CHECK_CUDA(cudaMemsetAsync(racc, 0, sizeof(double) * B * 2 * C, st));
  dim3 grid(red_chunks(HW, B), B), grid2(ew_chunks(HW, B, C), B);
  const bf16 *d_ = (const bf16*)dy, *x_ = (const bf16*)x;
  (void)y;   // the activation's sign is recomputed from x (same expression as the forward pass): y is not read any more
#define S2E_IN_BWD(ACT_)                                                                                             \
  instnorm_bwd_reduce_kernel<ACT_><<<grid, NT, red_smem(C), st>>>(d_, x_, mean, rstd, HW, C, racc);                  \
  S2E_LAUNCH_CHECK();                                                                                                \
  instnorm_bwd_apply_kernel<ACT_><<<grid2, NT, 0, st>>>(d_, x_, mean, rstd, racc, HW, C, (bf16*)dx);
  if (act == S2E_ACT_LRELU) { S2E_IN_BWD(S2E_ACT_LRELU) }
  else if (act == S2E_ACT_RELU) { S2E_IN_BWD(S2E_ACT_RELU) }
  else { S2E_IN_BWD(S2E_ACT_NONE) }
#undef S2E_IN_BWD
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

}  // extern "C"
