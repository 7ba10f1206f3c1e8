// Integer path, layout, weight packing, spectral norm, resampling, small linear layers, losses, Adam.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>

#include <type_traits>

#include "common.cuh"

// ------------------------------------------------------------------------------------------ host state
static thread_local char g_err[512] = "";
static int g_debug[8] = {0, 0, 0, 0, 0, 0, 0, 0};

void s2e_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int s2e_num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}
int s2e_debug_get(int key) { return (key >= 0 && key < 8) ? g_debug[key] : 0; }

int s2e_tapconv_fwd_tc(const s2e_conv_t*, const void*, const void*, const float*, const float*, void*, cudaStream_t);
int s2e_tapconv_wgrad_tc(const s2e_conv_t*, const void*, const void*, float*, cudaStream_t);
int s2e_tapconv_fwd_simt(const s2e_conv_t*, const void*, const void*, const float*, const float*, void*, cudaStream_t);
int s2e_tapconv_wgrad_simt(const s2e_conv_t*, const void*, const void*, float*, cudaStream_t);

namespace {

constexpr int NT = 256;
inline int grid1d(long long n, int per = NT) {
  long long g = (n + per - 1) / per;
  const long long cap = (long long)s2e_num_sms() * 32;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}
#define GRID_STRIDE(i, n) for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (long long)gridDim.x * blockDim.x)

__device__ __forceinline__ float block_sum(float v) {
  __shared__ float sh[32];
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.f;
  if (w == 0) v = warp_sum(v);
  return v;  // valid in thread 0
}

inline int floor_div(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

// ------------------------------------------------------------------------------------------ integer path
__global__ void onehot_kernel(const long long* __restrict__ label, long long HW, int nc, long long n, float* __restrict__ out) {
  GRID_STRIDE(i, n) {
    const long long hw = i % HW;
    const int c = (int)((i / HW) % nc);
    const long long b = i / (HW * nc);
    out[i] = (label[b * HW + hw] == c) ? 1.0f : 0.0f;
  }
}

__global__ void seg_nearest_kernel(const float* __restrict__ seg, int C, int Hs, int Ws, int Hd, int Wd, int Cpad, float sh,
                                   float sw, long long n, bf16* __restrict__ out) {
  GRID_STRIDE(i, n) {
    const int c = (int)(i % Cpad);
    long long p = i / Cpad;
    const int wd = (int)(p % Wd);
    p /= Wd;
    const int hd = (int)(p % Hd);
    const int b = (int)(p / Hd);
    float v = 0.f;
    if (c < C) {
      const int hs = min((int)floorf(hd * sh), Hs - 1);
      const int ws = min((int)floorf(wd * sw), Ws - 1);
      v = seg[(((long long)b * C + c) * Hs + hs) * Ws + ws];
    }
    out[i] = __float2bfloat16(v);
  }
}

// nearest resize + 3x3 im2col of a thin NCHW fp32 map into 64 bf16 channels per pixel: channel (r*3+s)*C + c holds
// seg[b][c][src(h+r-1)][src(w+s-1)] (zero outside the resized map and for channels >= 9*C).
__global__ void seg_im2col_kernel(const float* __restrict__ seg, int C, int Hs, int Ws, int Hd, int Wd, float sh, float sw,
                                  long long n, bf16* __restrict__ out) {
  GRID_STRIDE(i, n) {  // one thread per (pixel, 8-channel chunk)
    const int ch = (int)(i & 7);
    long long p = i >> 3;
    const int wd = (int)(p % Wd);
    p /= Wd;
    const int hd = (int)(p % Hd);
    const int b = (int)(p / Hd);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = ch * 8 + j;
      float val = k >= 62 ? 1.f : 0.f;   // two constant-one channels: carry the bias (hi + lo part) through the GEMM
      if (k < 9 * C) {
        const int t = k / C, c = k - t * C;
        const int h = hd + t / 3 - 1, w = wd + t % 3 - 1;
        if (h >= 0 && h < Hd && w >= 0 && w < Wd) {
          const int hs = min((int)floorf(h * sh), Hs - 1);
          const int ws = min((int)floorf(w * sw), Ws - 1);
          val = seg[(((long long)b * C + c) * Hs + hs) * Ws + ws];
        }
      }
      v[j] = val;
    }
    *reinterpret_cast<bf16x8*>(out + i * 8) = pack8(v);
  }
}
// C == 4 (the OpenEDS segmap): one thread per pixel gathers its 3x3 neighbourhood (36 values, neighbouring threads
// share cache lines) and writes the whole 128-byte im2col row; two taps fill one 16-byte chunk.
__global__ void seg_im2col_c4_kernel(const float* __restrict__ seg, int Hs, int Ws, int Hd, int Wd, float sh, float sw,
                                     long long npix, bf16* __restrict__ out) {
  GRID_STRIDE(p, npix) {
    const int wd = (int)(p % Wd);
    long long r0 = p / Wd;
    const int hd = (int)(r0 % Hd);
    const int b = (int)(r0 / Hd);
    const float* sb = seg + (long long)b * 4 * Hs * Ws;
    const long long plane = (long long)Hs * Ws;
    int hs[3], ws[3];
    bool hv[3], wv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int h = hd + k - 1, w = wd + k - 1;
      hv[k] = h >= 0 && h < Hd;
      wv[k] = w >= 0 && w < Wd;
      hs[k] = min((int)floorf((hv[k] ? h : 0) * sh), Hs - 1);
      ws[k] = min((int)floorf((wv[k] ? w : 0) * sw), Ws - 1);
    }
    float v[40];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const bool ok = hv[t / 3] && wv[t % 3];
      const float* q = sb + (long long)hs[t / 3] * Ws + ws[t % 3];
#pragma unroll
      for (int c = 0; c < 4; ++c) v[t * 4 + c] = ok ? q[c * plane] : 0.f;
    }
    v[36] = v[37] = v[38] = v[39] = 0.f;
    bf16* o = out + p * 64;
#pragma unroll
    for (int ch = 0; ch < 5; ++ch) st_stream8(o + ch * 8, pack8(v + ch * 8));
    const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float one[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f, 1.f};   // channels 62, 63 = 1: the bias columns of the GEMM
    st_stream8(o + 40, pack8(z));
    st_stream8(o + 48, pack8(z));
    st_stream8(o + 56, pack8(one));
  }
}
// OIHW (Cout, C, 3, 3) fp32 -> bf16 [Cout][64] with k = (r*3+s)*C + c   (and the adjoint for the weight gradient)
__global__ void pack_im2col_kernel(const float* __restrict__ w, int Cout, int C, bf16* __restrict__ out) {
  GRID_STRIDE(i, (long long)Cout * 64) {
    const int k = (int)(i & 63), co = (int)(i >> 6);
    float v = 0.f;
    if (k < 9 * C) {
      const int t = k / C, c = k - t * C;
      v = w[((long long)co * C + c) * 9 + t];
    }
    out[i] = __float2bfloat16(v);
  }
}
__global__ void unpack_im2col_kernel(const float* __restrict__ dwp, int Cout, int C, float* __restrict__ dw, float* __restrict__ db) {
  GRID_STRIDE(i, (long long)Cout * C * 9) {
    const int t = (int)(i % 9);
    const long long r = i / 9;
    const int c = (int)(r % C), co = (int)(r / C);
    dw[i] = dwp[(long long)co * 64 + t * C + c];
    if (db && t == 0 && c == 0) db[co] = dwp[(long long)co * 64 + 63];   // gradient of the bias column
  }
}
// layout
__global__ void nchw2nhwc_kernel(const float* __restrict__ x, int C, int H, int W, long long n, bf16* __restrict__ y) {
  GRID_STRIDE(i, n) {
    const int c = (int)(i % C);
    long long p = i / C;
    const int w = (int)(p % W);
    p /= W;
    const int h = (int)(p % H);
    const long long b = p / H;
    y[i] = __float2bfloat16(x[((b * C + c) * H + h) * W + w]);
  }
}
__global__ void nhwc2nchw_kernel(const bf16* __restrict__ x, int C, int H, int W, long long n, float* __restrict__ y) {
  GRID_STRIDE(i, n) {
    const int w = (int)(i % W);
    long long p = i / W;
    const int h = (int)(p % H);
    p /= H;
    const int c = (int)(p % C);
    const long long b = p / C;
    y[i] = __bfloat162float(x[((b * H + h) * W + w) * C + c]);
  }
}

// ------------------------------------------------------------------------------------------ weight packing
struct PackGeom {
  int Cout, Cin, kh, kw, stride, pad;
  int Ctot, co_off;  // several OIHW tensors may be packed side by side along Cout (gamma | beta)
  int CinPad;        // packed input-channel count (>= Cin; extra channels carry zero weights)
  int amin, bmin, na, nb;  // stride-2 tap grid
};

__global__ void pack_weight_kernel(const float* __restrict__ w, PackGeom g, int transposed, long long n, bf16* __restrict__ out) {
  const int CinP = g.stride == 2 ? 4 * g.CinPad : g.CinPad;
  GRID_STRIDE(i, n) {
    int cp, co;
    long long r0 = i;
    if (transposed) {
      co = (int)(r0 % g.Cout);
      r0 /= g.Cout;
      cp = (int)(r0 % CinP);
      r0 /= CinP;
    } else {
      cp = (int)(r0 % CinP);
      r0 /= CinP;
      co = (int)(r0 % g.Cout);
      r0 /= g.Cout;
    }
    const int t = (int)r0;
    const long long oidx = transposed ? ((long long)t * CinP + cp) * g.Ctot + g.co_off + co
                                      : ((long long)t * g.Ctot + g.co_off + co) * CinP + cp;
    int r, s, ci;
    if (g.stride == 1) {
      r = t / g.kw;
      s = t % g.kw;
      ci = cp;
    } else {
      const int a = g.amin + t / g.nb, b = g.bmin + t % g.nb;
      const int ph = cp / g.CinPad;
      ci = cp % g.CinPad;
      r = 2 * a + (ph >> 1) + g.pad;
      s = 2 * b + (ph & 1) + g.pad;
    }
    float v = 0.f;
    if (ci < g.Cin && r >= 0 && r < g.kh && s >= 0 && s < g.kw) v = w[(((long long)co * g.Cin + ci) * g.kh + r) * g.kw + s];
    out[oidx] = __float2bfloat16(v);
  }
}

__device__ __forceinline__ long long packed_index(const PackGeom& g, int co, int ci, int r, int s) {
  co += g.co_off;
  if (g.stride == 1) return ((long long)(r * g.kw + s) * g.Ctot + co) * g.CinPad + ci;
  const int rr = r - g.pad, ss = s - g.pad;
  const int i = ((rr % 2) + 2) % 2, j = ((ss % 2) + 2) % 2;
  const int a = (rr - i) / 2, b = (ss - j) / 2;
  const int t = (a - g.amin) * g.nb + (b - g.bmin);
  return ((long long)t * g.Ctot + co) * (4 * g.CinPad) + (i * 2 + j) * g.CinPad + ci;
}

__global__ void wgrad_dot_kernel(const float* __restrict__ dwp, const float* __restrict__ w, PackGeom g, long long n, float* dot) {
  float acc = 0.f;
  GRID_STRIDE(i, n) {
    const int s = (int)(i % g.kw);
    long long r0 = i / g.kw;
    const int r = (int)(r0 % g.kh);
    r0 /= g.kh;
    const int ci = (int)(r0 % g.Cin);
    const int co = (int)(r0 / g.Cin);
    acc = fmaf(dwp[packed_index(g, co, ci, r, s)], w[i], acc);
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(dot, acc);
}

__global__ void unpack_wgrad_kernel(const float* __restrict__ dwp, PackGeom g, const float* __restrict__ u, const float* __restrict__ v,
                                    const float* __restrict__ inv_sigma, const float* __restrict__ dot, long long n, int accumulate,
                                    float* __restrict__ dw) {
  const float is = inv_sigma ? *inv_sigma : 1.f;
  const float dt = u ? *dot : 0.f;
  const int kk = g.kh * g.kw;
  GRID_STRIDE(i, n) {
    const int s = (int)(i % g.kw);
    long long r0 = i / g.kw;
    const int r = (int)(r0 % g.kh);
    r0 /= g.kh;
    const int ci = (int)(r0 % g.Cin);
    const int co = (int)(r0 / g.Cin);
    float gval = dwp[packed_index(g, co, ci, r, s)];
    if (u) gval = is * (gval - is * dt * u[co] * v[ci * kk + r * g.kw + s]);
    dw[i] = accumulate ? dw[i] + gval : gval;
  }
}

// Multi-tensor packing: one launch re-packs every weight an optimizer step touched.  A thread owns one (co, ci) pair,
// reads its kh*kw contiguous master values once and scatters them to their tap-major slots; lanes run along the
// contiguous axis of the OUTPUT (ci, or co for the transposed layout) so the 2-byte stores coalesce.  Slots that no
// (r, s) maps to (stride-2 phase padding, cin_pad columns, im2col columns >= 9C) are never written: the destination
// must have been zero-filled once, when it was allocated.
constexpr int PACK_MAX_JOBS = 40;
struct PackJob {
  const float* w;
  const float* bias;
  bf16* out;
  PackGeom g;
  int transposed, im2col;
  int blk0;
};
struct PackTable {
  int n;
  PackJob j[PACK_MAX_JOBS];
};
__global__ void __launch_bounds__(256) pack_weight_multi_kernel(const __grid_constant__ PackTable t) {
  int k = 0;
  while (k + 1 < t.n && (int)blockIdx.x >= t.j[k + 1].blk0) ++k;
  const PackJob& J = t.j[k];
  const PackGeom& g = J.g;
  const long long q = (long long)(blockIdx.x - J.blk0) * 256 + threadIdx.x;
  if (q >= (long long)g.Cout * g.Cin) return;
  int co, ci;
  if (J.transposed) {
    co = (int)(q % g.Cout);
    ci = (int)(q / g.Cout);
  } else {
    ci = (int)(q % g.Cin);
    co = (int)(q / g.Cin);
  }
  const int kk = g.kh * g.kw;
  const float* src = J.w + ((long long)co * g.Cin + ci) * kk;
  if (J.im2col) {  // [Cout][64], k = (r*3+s)*C + c ; columns 62, 63 = bias (multiply the constant-one channels)
    for (int tt = 0; tt < 9; ++tt) J.out[(long long)co * 64 + tt * g.Cin + ci] = __float2bfloat16(src[tt]);
    if (J.bias && ci == 0) {  // bias = hi + lo in two bf16 columns (2^-17 relative precision instead of 2^-9)
      const float bv = J.bias[co];
      const bf16 hi = __float2bfloat16(bv);
      J.out[(long long)co * 64 + 63] = hi;
      J.out[(long long)co * 64 + 62] = __float2bfloat16(bv - __bfloat162float(hi));
    }
    return;
  }
  const int CinP = g.stride == 2 ? 4 * g.CinPad : g.CinPad;
  for (int r = 0; r < g.kh; ++r) {
    for (int s2 = 0; s2 < g.kw; ++s2) {
      int tt, cp;
      if (g.stride == 1) {
        tt = r * g.kw + s2;
        cp = ci;
      } else {
        const int rr = r - g.pad, ss = s2 - g.pad;
        const int i = ((rr % 2) + 2) % 2, jj = ((ss % 2) + 2) % 2;
        const int a = (rr - i) / 2, b = (ss - jj) / 2;
        tt = (a - g.amin) * g.nb + (b - g.bmin);
        cp = (i * 2 + jj) * g.CinPad + ci;
      }
      const long long o = J.transposed ? ((long long)tt * CinP + cp) * g.Ctot + g.co_off + co
                                       : ((long long)tt * g.Ctot + g.co_off + co) * CinP + cp;
      J.out[o] = __float2bfloat16(src[r * g.kw + s2]);
    }
  }
}

// ------------------------------------------------------------------------------------------ spectral norm
// One power iteration of torch.nn.utils.spectral_norm for a whole TABLE of layers per launch (the layers of a network
// are independent: each iteration depends on its own W, u, v only).  Four launches per iteration regardless of the
// number of layers:  (1) part[chunk][c] = sum_{r in chunk} W[r][c] u[r]   (2) v = normalize(sum_chunk part)
// (3) s[r] = W[r][:] . v   (4) u = normalize(s), 1/sigma = 1 / (u . s).   Partials are combined in a fixed order, no
// floating-point atomics: the iteration is bitwise reproducible and independent of how layers are grouped in a table.
constexpr int SN_MAX_JOBS = 32;
constexpr int SN_RCHUNK = 64;
struct SnJob {
  const float* w;
  float *u, *v, *inv, *scratch, *ucopy, *vcopy;
  int rows, cols;
  int blk_a, blk_c;  // first block of this job in kernels (1) and (3)
};
struct SnTable {
  int n, it;  // it = iteration number (selects inv[it], ucopy + it*rows, vcopy + it*cols)
  SnJob j[SN_MAX_JOBS];
};
__device__ __forceinline__ int sn_find_a(const SnTable& t, int blk) {
  int k = 0;
  while (k + 1 < t.n && blk >= t.j[k + 1].blk_a) ++k;
  return k;
}
__device__ __forceinline__ int sn_find_c(const SnTable& t, int blk) {
  int k = 0;
  while (k + 1 < t.n && blk >= t.j[k + 1].blk_c) ++k;
  return k;
}
// (1): 128 threads; block = (128 columns) x (one 64-row chunk)
__global__ void __launch_bounds__(128) sn_wt_u_multi_kernel(const __grid_constant__ SnTable t) {
  const int k = sn_find_a(t, blockIdx.x);
  const SnJob& J = t.j[k];
  const int local = blockIdx.x - J.blk_a;
  const int cblocks = (J.cols + 127) >> 7;
  const int chunk = local / cblocks, cb = local - chunk * cblocks;
  const int c = cb * 128 + threadIdx.x;
  __shared__ float su[SN_RCHUNK];
  const int r0 = chunk * SN_RCHUNK, r1 = min(J.rows, r0 + SN_RCHUNK);
  if (threadIdx.x < r1 - r0) su[threadIdx.x] = J.u[r0 + threadIdx.x];
  __syncthreads();
  if (c >= J.cols) return;
  const float* w = J.w + (long long)r0 * J.cols + c;
  float acc = 0.f;
  int r = 0;
  const int nr = r1 - r0;
  for (; r + 8 <= nr; r += 8) {  // 8 independent loads in flight per thread
    float wv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) wv[q] = w[(long long)(r + q) * J.cols];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc = fmaf(wv[q], su[r + q], acc);
  }
  for (; r < nr; ++r) acc = fmaf(w[(long long)r * J.cols], su[r], acc);
  float* part = J.scratch + J.cols + J.rows;
  part[(long long)chunk * J.cols + c] = acc;
}
// (2) / (4): one block per job.  which = 0: v <- normalize(sum of partials);  1: u <- normalize(s), inv_sigma
__global__ void __launch_bounds__(1024) sn_normalize_multi_kernel(const __grid_constant__ SnTable t, int which) {
  const SnJob& J = t.j[blockIdx.x];
  const int n = which ? J.rows : J.cols;
  const int nparts = which ? 1 : (J.rows + SN_RCHUNK - 1) / SN_RCHUNK;
  const float* raw = which ? J.scratch + J.cols : J.scratch + J.cols + J.rows;
  float* outv = which ? J.u : J.v;
  float* copy = which ? (J.ucopy ? J.ucopy + (long long)t.it * J.rows : nullptr)
                      : (J.vcopy ? J.vcopy + (long long)t.it * J.cols : nullptr);
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float v = 0.f;
    for (int q = 0; q < nparts; ++q) v += raw[(long long)q * n + i];
    outv[i] = v;  // staged un-normalised; rescaled below by the same thread
    acc = fmaf(v, v, acc);
  }
  __shared__ float s_norm;
  acc = block_sum(acc);
  if (threadIdx.x == 0) s_norm = acc;
  __syncthreads();
  const float nsq = s_norm;
  const float denom = fmaxf(sqrtf(nsq), 1e-12f);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = outv[i] / denom;
    outv[i] = v;
    if (copy) copy[i] = v;
  }
  // sigma = u . (W v) = ||Wv||^2 / max(||Wv||, eps)
  if (which && threadIdx.x == 0) J.inv[t.it] = 1.f / (nsq / denom);
}
// (3): one warp per row, 8 rows per block; the row is read with 4 independent (vector) loads in flight per lane
__global__ void __launch_bounds__(256) sn_w_v_multi_kernel(const __grid_constant__ SnTable t) {
  const int k = sn_find_c(t, blockIdx.x);
  const SnJob& J = t.j[k];
  const int r = (blockIdx.x - J.blk_c) * 8 + (threadIdx.x >> 5);
  if (r >= J.rows) return;
  const int lane = threadIdx.x & 31;
  const float* w = J.w + (long long)r * J.cols;
  const float* v = J.v;
  float acc = 0.f;
  if ((J.cols & 3) == 0) {
    const float4* w4 = reinterpret_cast<const float4*>(w);
    const float4* v4 = reinterpret_cast<const float4*>(v);
    const int n4 = J.cols >> 2;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int c = lane;
    for (; c + 96 < n4; c += 128) {
      const float4 x0 = w4[c], x1 = w4[c + 32], x2 = w4[c + 64], x3 = w4[c + 96];
      const float4 y0 = v4[c], y1 = v4[c + 32], y2 = v4[c + 64], y3 = v4[c + 96];
      a0 = fmaf(x0.x, y0.x, fmaf(x0.y, y0.y, fmaf(x0.z, y0.z, fmaf(x0.w, y0.w, a0))));
      a1 = fmaf(x1.x, y1.x, fmaf(x1.y, y1.y, fmaf(x1.z, y1.z, fmaf(x1.w, y1.w, a1))));
      a2 = fmaf(x2.x, y2.x, fmaf(x2.y, y2.y, fmaf(x2.z, y2.z, fmaf(x2.w, y2.w, a2))));
      a3 = fmaf(x3.x, y3.x, fmaf(x3.y, y3.y, fmaf(x3.z, y3.z, fmaf(x3.w, y3.w, a3))));
    }
    for (; c < n4; c += 32) {
      const float4 x0 = w4[c], y0 = v4[c];
      a0 = fmaf(x0.x, y0.x, fmaf(x0.y, y0.y, fmaf(x0.z, y0.z, fmaf(x0.w, y0.w, a0))));
    }
    acc = (a0 + a1) + (a2 + a3);
  } else {
    for (int c = lane; c < J.cols; c += 32) acc = fmaf(w[c], v[c], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) J.scratch[J.cols + r] = acc;
}
// evaluation mode (no buffer update): inv_sigma = 1 / (u . (W v)); one block per job
__global__ void __launch_bounds__(1024) sn_dot_multi_kernel(const __grid_constant__ SnTable t) {
  const SnJob& J = t.j[blockIdx.x];
  const float* s = J.scratch + J.cols;
  float acc = 0.f;
  for (int i = threadIdx.x; i < J.rows; i += blockDim.x) acc = fmaf(J.u[i], s[i], acc);
  acc = block_sum(acc);
  if (threadIdx.x == 0) J.inv[t.it] = 1.f / acc;
}

// ------------------------------------------------------------------------------------------ space <-> depth
// VEC = 8: one 16-byte vector of 8 channels per thread (C % 8 == 0); VEC = 1: scalar fallback.  32-bit index math.
template <int VEC>
__global__ void s2d_kernel(const bf16* __restrict__ x, int H, int W, int C, int H2, int W2, unsigned n, bf16* __restrict__ y) {
  const unsigned CV = (unsigned)(C / VEC);
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {  // output [B][H2][W2][4][CV]
    const unsigned c = i % CV;
    unsigned p = i / CV;
    const unsigned ph = p & 3u;
    p >>= 2;
    const unsigned w2 = p % (unsigned)W2;
    p /= (unsigned)W2;
    const unsigned h2 = p % (unsigned)H2;
    const unsigned b = p / (unsigned)H2;
    const int h = 2 * (int)h2 + (int)(ph >> 1), w = 2 * (int)w2 + (int)(ph & 1);
    const bool in = h < H && w < W;
    const long long src = ((((long long)b * H + h) * W + w) * CV + c) * VEC;
    if (VEC == 8) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (in) v = *reinterpret_cast<const uint4*>(x + src);
      *reinterpret_cast<uint4*>(y + (long long)i * 8) = v;
    } else {
      y[i] = in ? x[src] : __float2bfloat16(0.f);
    }
  }
}
template <int VEC>
__global__ void d2s_kernel(const bf16* __restrict__ dy, int H, int W, int C, int H2, int W2, unsigned n, bf16* __restrict__ dx) {
  const unsigned CV = (unsigned)(C / VEC);
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {  // dx [B][H][W][CV]
    const unsigned c = i % CV;
    unsigned p = i / CV;
    const unsigned w = p % (unsigned)W;
    p /= (unsigned)W;
    const unsigned h = p % (unsigned)H;
    const unsigned b = p / (unsigned)H;
    const unsigned ph = (h & 1u) * 2u + (w & 1u);
    const long long src = (((((long long)b * H2 + (h >> 1)) * W2 + (w >> 1)) * 4 + ph) * CV + c) * VEC;
    if (VEC == 8)
      *reinterpret_cast<uint4*>(dx + (long long)i * 8) = *reinterpret_cast<const uint4*>(dy + src);
    else
      dx[i] = dy[src];
  }
}

// ------------------------------------------------------------------------------------------ resampling
__global__ void upsample2x_fwd_kernel(const bf16* __restrict__ x, int H, int W, int C8, long long n, bf16* __restrict__ y) {
  GRID_STRIDE(i, n) {  // over output vectors [B][2H][2W][C8]
    const int c = (int)(i % C8);
    long long p = i / C8;
    const int w = (int)(p % (2 * W));
    p /= 2 * W;
    const int h = (int)(p % (2 * H));
    const long long b = p / (2 * H);
    const uint4 v = *reinterpret_cast<const uint4*>(x + (((b * H + (h >> 1)) * W + (w >> 1)) * C8 + c) * 8);
    *reinterpret_cast<uint4*>(y + i * 8) = v;
  }
}
__global__ void upsample2x_bwd_kernel(const bf16* __restrict__ dy, int H, int W, int C8, long long n, bf16* __restrict__ dx) {
  GRID_STRIDE(i, n) {  // over input vectors [B][H][W][C8]
    const int c = (int)(i % C8);
    long long p = i / C8;
    const int w = (int)(p % W);
    p /= W;
    const int h = (int)(p % H);
    const long long b = p / H;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, f[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long src = (((b * 2 * H + 2 * h + (q >> 1)) * 2 * W + 2 * w + (q & 1)) * C8 + c) * 8;
      unpack8(*reinterpret_cast<const bf16x8*>(dy + src), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    *reinterpret_cast<bf16x8*>(dx + i * 8) = pack8(acc);
  }
}

__global__ void avgpool_fwd_kernel(const bf16* __restrict__ x, int H, int W, int C, int Ho, int Wo, long long n, bf16* __restrict__ y) {
  GRID_STRIDE(i, n) {
    const int c = (int)(i % C);
    long long p = i / C;
    const int wo = (int)(p % Wo);
    p /= Wo;
    const int ho = (int)(p % Ho);
    const long long b = p / Ho;
    float acc = 0.f;
    int cnt = 0;
    for (int dh = -1; dh <= 1; ++dh)
      for (int dw = -1; dw <= 1; ++dw) {
        const int h = 2 * ho + dh, w = 2 * wo + dw;
        if (h >= 0 && h < H && w >= 0 && w < W) {
          acc += __bfloat162float(x[((b * H + h) * W + w) * C + c]);
          ++cnt;
        }
      }
    y[i] = __float2bfloat16(acc / (float)cnt);
  }
}
// 8 channels per thread (C % 8 == 0), 32-bit index math
__global__ void avgpool_fwd_vec_kernel(const bf16* __restrict__ x, int H, int W, int C8, int Ho, int Wo, unsigned n, bf16* __restrict__ y) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned c = i % (unsigned)C8;
    unsigned p = i / (unsigned)C8;
    const int wo = (int)(p % (unsigned)Wo);
    p /= (unsigned)Wo;
    const int ho = (int)(p % (unsigned)Ho);
    const unsigned b = p / (unsigned)Ho;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, f[8];
    int cnt = 0;
#pragma unroll
    for (int dh = -1; dh <= 1; ++dh)
#pragma unroll
      for (int dw = -1; dw <= 1; ++dw) {
        const int h = 2 * ho + dh, w = 2 * wo + dw;
        if (h >= 0 && h < H && w >= 0 && w < W) {
          unpack8(*reinterpret_cast<const bf16x8*>(x + ((((long long)b * H + h) * W + w) * C8 + c) * 8), f);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] += f[j];
          ++cnt;
        }
      }
    const float inv = 1.f / (float)cnt;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] *= inv;
    *reinterpret_cast<bf16x8*>(y + (long long)i * 8) = pack8(acc);
  }
}
__device__ __forceinline__ int pool_cnt(int o, int L) {  // valid taps of window o along a length-L axis
  int c = 0;
  for (int d = -1; d <= 1; ++d) c += (2 * o + d >= 0 && 2 * o + d < L);
  return c;
}
__global__ void avgpool_bwd_vec_kernel(const bf16* __restrict__ dy, int H, int W, int C8, int Ho, int Wo, unsigned n, bf16* __restrict__ dx);
__global__ void avgpool_bwd_kernel(const bf16* __restrict__ dy, int H, int W, int C, int Ho, int Wo, long long n, bf16* __restrict__ dx) {
  GRID_STRIDE(i, n) {
    const int c = (int)(i % C);
    long long p = i / C;
    const int w = (int)(p % W);
    p /= W;
    const int h = (int)(p % H);
    const long long b = p / H;
    float acc = 0.f;
    for (int ho = (h) / 2; ho <= (h + 1) / 2; ++ho) {
      if (ho < 0 || ho >= Ho) continue;
      for (int wo = (w) / 2; wo <= (w + 1) / 2; ++wo) {
        if (wo < 0 || wo >= Wo) continue;
        acc += __bfloat162float(dy[((b * Ho + ho) * Wo + wo) * C + c]) / (float)(pool_cnt(ho, H) * pool_cnt(wo, W));
      }
    }
    dx[i] = __float2bfloat16(acc);
  }
}

__global__ void avgpool_bwd_vec_kernel(const bf16* __restrict__ dy, int H, int W, int C8, int Ho, int Wo, unsigned n, bf16* __restrict__ dx) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned c = i % (unsigned)C8;
    unsigned p = i / (unsigned)C8;
    const int w = (int)(p % (unsigned)W);
    p /= (unsigned)W;
    const int h = (int)(p % (unsigned)H);
    const unsigned b = p / (unsigned)H;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, f[8];
    for (int ho = h / 2; ho <= (h + 1) / 2; ++ho) {
      if (ho >= Ho) continue;
      for (int wo = w / 2; wo <= (w + 1) / 2; ++wo) {
        if (wo >= Wo) continue;
        const float sc = 1.f / (float)(pool_cnt(ho, H) * pool_cnt(wo, W));
        unpack8(*reinterpret_cast<const bf16x8*>(dy + ((((long long)b * Ho + ho) * Wo + wo) * C8 + c) * 8), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(f[j], sc, acc[j]);
      }
    }
    *reinterpret_cast<bf16x8*>(dx + (long long)i * 8) = pack8(acc);
  }
}

__device__ __forceinline__ void bilin_src(int d, float scale, int in, int* i0, int* i1, float* l1) {
  float s = ((float)d + 0.5f) * scale - 0.5f;
  if (s < 0.f) s = 0.f;
  int a = (int)s;
  if (a > in - 1) a = in - 1;
  *i0 = a;
  *i1 = a + ((a < in - 1) ? 1 : 0);
  *l1 = s - (float)a;
}
__global__ void bilinear_fwd_kernel(const float* __restrict__ x, int Hs, int Ws, int Hd, int Wd, float sh, float sw, long long n,
                                    bf16* __restrict__ y) {
  GRID_STRIDE(i, n) {
    const int wd = (int)(i % Wd);
    long long p = i / Wd;
    const int hd = (int)(p % Hd);
    const long long nn = p / Hd;
    int h0, h1, w0, w1;
    float lh, lw;
    bilin_src(hd, sh, Hs, &h0, &h1, &lh);
    bilin_src(wd, sw, Ws, &w0, &w1, &lw);
    const float* src = x + nn * Hs * Ws;
    const float v = (1.f - lh) * ((1.f - lw) * src[h0 * Ws + w0] + lw * src[h0 * Ws + w1]) +
                    lh * ((1.f - lw) * src[h1 * Ws + w0] + lw * src[h1 * Ws + w1]);
    y[i] = __float2bfloat16(v);
  }
}
__global__ void bilinear_bwd_kernel(const bf16* __restrict__ dy, int Hs, int Ws, int Hd, int Wd, float sh, float sw, long long n,
                                    float* __restrict__ dx) {
  GRID_STRIDE(i, n) {
    const int wd = (int)(i % Wd);
    long long p = i / Wd;
    const int hd = (int)(p % Hd);
    const long long nn = p / Hd;
    int h0, h1, w0, w1;
    float lh, lw;
    bilin_src(hd, sh, Hs, &h0, &h1, &lh);
    bilin_src(wd, sw, Ws, &w0, &w1, &lw);
    const float g = __bfloat162float(dy[i]);
    float* dst = dx + nn * Hs * Ws;
    atomicAdd(dst + h0 * Ws + w0, g * (1.f - lh) * (1.f - lw));
    atomicAdd(dst + h0 * Ws + w1, g * (1.f - lh) * lw);
    atomicAdd(dst + h1 * Ws + w0, g * lh * (1.f - lw));
    atomicAdd(dst + h1 * Ws + w1, g * lh * lw);
  }
}

// one thread per pixel of the (2B, H, W) batch: nc + 1 coalesced fp32 reads, Cpad bf16 written as 16-byte vectors
__global__ void make_d_input_kernel(const float* __restrict__ seg, const float* __restrict__ fake, const float* __restrict__ real, int B,
                                    int nc, long long HW, int Cpad, long long npix, bf16* __restrict__ out) {
  GRID_STRIDE(p, npix) {
    const long long hw = p % HW;
    const int b2 = (int)(p / HW);
    const int b = b2 % B;
    const float* sp = seg + (long long)b * nc * HW + hw;
    const float img = (b2 < B ? fake : real)[(long long)b * HW + hw];
    bf16* o = out + p * Cpad;
    if ((Cpad & 7) == 0) {
      for (int c0 = 0; c0 < Cpad; c0 += 8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c = c0 + j;
          v[j] = c < nc ? sp[(long long)c * HW] : (c == nc ? img : 0.f);
        }
        st_stream8(o + c0, pack8(v));
      }
    } else {
      for (int c = 0; c < Cpad; ++c) o[c] = __float2bfloat16(c < nc ? sp[(long long)c * HW] : (c == nc ? img : 0.f));
    }
  }
}
__global__ void d_input_grad_kernel(const bf16* __restrict__ dxin, int nc, int Cpad, long long n, float* __restrict__ dfake) {
  GRID_STRIDE(i, n) dfake[i] = __bfloat162float(dxin[i * Cpad + nc]);
}

// ------------------------------------------------------------------------------------------ differentiable augmentation
// DiffAugment (Zhao et al., NeurIPS 2020) of the D input; the formulas and the record layout are in the header.
// Philox4x32-10 (Salmon et al., SC'11), the generator of curand / Random123: 10 rounds, the key bumped between rounds.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k.x += 0x9E3779B9u;
      k.y += 0xBB67AE85u;
    }
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}
__device__ __forceinline__ float da_unit(unsigned r) { return (float)(r >> 8) * (1.f / 16777216.f); }
__device__ __forceinline__ int da_below(unsigned r, int n) { return (int)(((unsigned long long)r * (unsigned)n) >> 32); }

// Box-Muller in fp64 on two words, u = ((r >> 8) + 0.5) 2^-24 > 0 so that log(u) is finite
__device__ __forceinline__ double2 da_normal2(unsigned ru, unsigned rv) {
  const double u = ((double)(ru >> 8) + 0.5) * (1.0 / 16777216.0), v = ((double)(rv >> 8) + 0.5) * (1.0 / 16777216.0);
  const double r = sqrt(-2.0 * log(u));
  double sn, cs;
  sincospi(2.0 * v, &sn, &cs);
  return make_double2(r * cs, r * sn);
}

// the geometric record of one sample (s2e_diffaug_draw_geom's formulas in the header): M in fp64, rounded once to fp32
__device__ void da_draw_geom(uint4 c, uint2 key, uint4 r2, double p, int H, int W, float* __restrict__ m, int& bits) {
  c.w = 3u;
  const uint4 r3 = philox4x32_10(c, key);
  c.w = 4u;
  const uint4 r4 = philox4x32_10(c, key);
  c.w = 5u;
  const uint4 r5 = philox4x32_10(c, key);
  const double p_rot = 1.0 - sqrt(fmax(1.0 - p, 0.0));
  const bool mirror = (double)da_unit(r2.y) < p && (double)da_unit(r2.z) < 0.5;
  const bool g_s = (double)da_unit(r2.w) < p, g_r1 = (double)da_unit(r3.x) < p_rot, g_a = (double)da_unit(r3.y) < p;
  const bool g_r2 = (double)da_unit(r3.z) < p_rot, g_t = (double)da_unit(r3.w) < p;
  const double2 n01 = da_normal2(r4.x, r4.y), n23 = da_normal2(r5.x, r5.y);
  const double is = g_s ? exp2(-0.2 * n01.x) : 1.0, ia = g_a ? exp2(-0.2 * n01.y) : 1.0;
  const double t1 = g_r1 ? 2.0 * (double)da_unit(r4.z) - 1.0 : 0.0, t2 = g_r2 ? 2.0 * (double)da_unit(r4.w) - 1.0 : 0.0;
  double s1, c1, s2, c2;
  sincospi(t1, &s1, &c1);
  sincospi(t2, &s2, &c2);
  // A = F S(1/s) R(-th1) diag(1/a, a) R(-th2), R(-t) = [[cos t, sin t], [-sin t, cos t]]
  const double b00 = c1 * ia, b01 = s1 / ia, b10 = -s1 * ia, b11 = c1 / ia;          // R(-th1) diag(1/a, a)
  const double f = mirror ? -is : is;
  const double a00 = f * (b00 * c2 - b01 * s2), a01 = f * (b00 * s2 + b01 * c2);
  const double a10 = is * (b10 * c2 - b11 * s2), a11 = is * (b10 * s2 + b11 * c2);
  const double dx = g_t ? -0.125 * n23.x * (double)W : 0.0, dy = g_t ? -0.125 * n23.y * (double)H : 0.0;
  m[0] = (float)a00;
  m[1] = (float)a01;
  m[2] = (float)(a00 * dx + a01 * dy);
  m[3] = (float)a10;
  m[4] = (float)a11;
  m[5] = (float)(a10 * dx + a11 * dy);
  m[6] = m[7] = 0.f;
  bits = (mirror ? S2E_DIFFAUG_XFLIP : 0) | ((g_s || g_r1 || g_a || g_r2 || g_t) ? S2E_DIFFAUG_GEOMETRIC : 0);
}

// one block: thread t writes the records of samples t, t + 256, ... from the counter it read, then thread 0 advances it.
// GATE (s2e_diffaug_draw_p): also the per-op gates, unit(r6 | r7 | r8) < p in fp64, from block 1's spare words and block 2
// GEOM (s2e_diffaug_draw_geom, with GATE): also the mirror and geometric records and bits, from blocks 2 to 5
template <bool GATE, bool GEOM = false>
__global__ void __launch_bounds__(256) diffaug_draw_kernel(long long* state, int B, long long index_offset, int H, int W,
                                                           float* __restrict__ rec, const double* __restrict__ prob,
                                                           int* __restrict__ opmask, float* __restrict__ geom = nullptr) {
  const unsigned long long seed = (unsigned long long)state[0], ctr = (unsigned long long)state[1];
  const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  const int sx = (H + 4) / 8, sy = (W + 4) / 8;    // int(H / 8 + 0.5)
  const int cx = (H + 1) / 2, cy = (W + 1) / 2;    // int(H / 2 + 0.5)
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const unsigned idx = (unsigned)(index_offset + b);
    const uint4 r0 = philox4x32_10(make_uint4(idx, (unsigned)ctr, (unsigned)(ctr >> 32), 0u), key);
    const uint4 r1 = philox4x32_10(make_uint4(idx, (unsigned)ctr, (unsigned)(ctr >> 32), 1u), key);
    float* o = rec + (long long)b * S2E_DIFFAUG_RECORD;
    o[0] = da_unit(r0.x);
    o[1] = da_unit(r0.y);
    o[2] = (float)(da_below(r0.z, 2 * sx + 1) - sx);
    o[3] = (float)(da_below(r0.w, 2 * sy + 1) - sy);
    o[4] = (float)da_below(r1.x, H + 1 - cx % 2);
    o[5] = (float)da_below(r1.y, W + 1 - cy % 2);
    if (GATE) {
      const uint4 r2 = philox4x32_10(make_uint4(idx, (unsigned)ctr, (unsigned)(ctr >> 32), 2u), key);
      const double pr = *prob;
      int bits = ((double)da_unit(r1.z) < pr ? S2E_DIFFAUG_COLOR : 0) | ((double)da_unit(r1.w) < pr ? S2E_DIFFAUG_TRANSLATION : 0) |
                 ((double)da_unit(r2.x) < pr ? S2E_DIFFAUG_CUTOUT : 0);
      if constexpr (GEOM) {
        int gbits;
        da_draw_geom(make_uint4(idx, (unsigned)ctr, (unsigned)(ctr >> 32), 0u), key, r2, pr, H, W,
                     geom + (long long)b * S2E_DIFFAUG_GEOM_RECORD, gbits);
        bits |= gbits;
      }
      opmask[b] = bits;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) state[1] = (long long)(ctr + 1);
}

__device__ __forceinline__ double block_sum_f64(double v) {
  __shared__ double sh[32];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sh[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.0;
  if (w == 0)
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;  // valid in thread 0
}

// per-image means for contrast: block b2 reduces fake[b2] (b2 < B) or real[b2 - B] in fp64
__global__ void __launch_bounds__(1024) diffaug_means_kernel(const float* __restrict__ fake, const float* __restrict__ real, int B,
                                                             long long HW, float* __restrict__ means) {
  const int b2 = blockIdx.x;
  const float* x = (b2 < B ? fake : real) + (long long)(b2 % B) * HW;
  double s0 = 0.0, s1 = 0.0;
  long long i = threadIdx.x;
  for (; i + blockDim.x < HW; i += 2 * blockDim.x) {
    s0 += (double)x[i];
    s1 += (double)x[i + blockDim.x];
  }
  if (i < HW) s0 += (double)x[i];
  const double s = block_sum_f64(s0 + s1);
  if (threadIdx.x == 0) means[b2] = (float)(s / (double)HW);
}

// is output pixel (i, j) of a sample with record r outside its cutout rectangle?
__device__ __forceinline__ bool da_not_cut(int i, int j, int H, int W, const float* r, int policy) {
  if (policy & S2E_DIFFAUG_CUTOUT) {
    const int cx = (H + 1) / 2, cy = (W + 1) / 2;
    const int x0 = (int)r[4] - cx / 2, y0 = (int)r[5] - cy / 2;
    if (i >= x0 && i < x0 + cx && j >= y0 && j < y0 + cy) return false;
  }
  return true;
}

// reflection of a tap index into [0, n), n >= 2: torch's 'reflect' padding, repeated
__device__ __forceinline__ int da_fold(int k, int n) {
  const int m = 2 * (n - 1);
  int q = k % m;
  if (q < 0) q += m;
  return q < n ? q : m - q;
}
// the source point of warped-image position (si, sj) in pixel coordinates, fp32 without contraction (the header's X, Y)
__device__ __forceinline__ void da_warp(const float* m, int si, int sj, int H, int W, float& X, float& Y) {
  const float hx = 0.5f * (float)(W - 1), hy = 0.5f * (float)(H - 1);
  const float xc = __fsub_rn((float)sj, hx), yc = __fsub_rn((float)si, hy);
  X = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], xc), __fmul_rn(m[1], yc)), m[2]), hx);
  Y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[3], xc), __fmul_rn(m[4], yc)), m[5]), hy);
}
// sample b's M for its policy: s2e_diffaug_draw_geom folds the mirror into row 0 whenever the coin applied it, so a policy
// without XFLIP negates that row back (exact)
__device__ __forceinline__ void da_load_m(const float* __restrict__ geom, int b, int policy, int mask, float* m) {
  const float* g = geom + (long long)b * S2E_DIFFAUG_GEOM_RECORD;
  const float f = ((mask & S2E_DIFFAUG_XFLIP) && !(policy & S2E_DIFFAUG_XFLIP)) ? -1.f : 1.f;
  m[0] = f * __ldg(g);
  m[1] = f * __ldg(g + 1);
  m[2] = f * __ldg(g + 2);
  m[3] = __ldg(g + 3);
  m[4] = __ldg(g + 4);
  m[5] = __ldg(g + 5);
}

// make_d_input_kernel with the augmentation applied while gathering: one thread per output pixel of the (2B, H, W) batch.
// MASKED: sample b applies policy & opmask[b] (s2e_diffaug_draw_p's gates)
// GEOM (with MASKED): also XFLIP / GEOMETRIC with geom's matrices (s2e_diffaug_draw_geom)
template <bool COLOR, bool MASKED = false, bool GEOM = false>
__global__ void make_d_input_aug_kernel(const float* __restrict__ seg, const float* __restrict__ fake, const float* __restrict__ real,
                                        int B, int nc, int H, int W, int Cpad, long long npix, const float* __restrict__ rec,
                                        const float* __restrict__ means, int policy_all, bf16* __restrict__ out,
                                        const int* __restrict__ opmask = nullptr, const float* __restrict__ geom = nullptr) {
  const long long HW = (long long)H * W;
  GRID_STRIDE(p, npix) {
    const long long hw = p % HW;
    const int b2 = (int)(p / HW);
    const int b = b2 % B;
    const int policy = MASKED ? policy_all & __ldg(opmask + b) : policy_all;
    const float* r = rec + (long long)b * S2E_DIFFAUG_RECORD;
    const int i = (int)(hw / W), j = (int)(hw % W);
    int si = i, sj = j;
    if (policy & S2E_DIFFAUG_TRANSLATION) {
      si += (int)__ldg(r + 2);
      sj += (int)__ldg(r + 3);
    }
    const bool keep = si >= 0 && si < H && sj >= 0 && sj < W && da_not_cut(i, j, H, W, r, policy);
    long long shw = keep ? (long long)si * W + sj : 0;
    float img = 0.f;
    bool warped = false;
    if constexpr (GEOM) {
      if (keep && (policy & S2E_DIFFAUG_GEOMETRIC)) {   // labels at the nearest tap, the image bilinear, taps reflected
        float m[6], X, Y;
        da_load_m(geom, b, policy, __ldg(opmask + b), m);
        da_warp(m, si, sj, H, W, X, Y);
        shw = (long long)da_fold((int)floorf(Y + 0.5f), H) * W + da_fold((int)floorf(X + 0.5f), W);
        const float x0 = floorf(X), y0 = floorf(Y), fx = X - x0, fy = Y - y0;
        const int c0 = da_fold((int)x0, W), c1 = da_fold((int)x0 + 1, W);
        const float* row0 = (b2 < B ? fake : real) + (long long)b * HW + (long long)da_fold((int)y0, H) * W;
        const float* row1 = (b2 < B ? fake : real) + (long long)b * HW + (long long)da_fold((int)y0 + 1, H) * W;
        img = (1.f - fy) * ((1.f - fx) * row0[c0] + fx * row0[c1]) + fy * ((1.f - fx) * row1[c0] + fx * row1[c1]);
        warped = true;
      } else if (keep && (policy & S2E_DIFFAUG_XFLIP)) {
        shw = (long long)si * W + (W - 1 - sj);
      }
    }
    const float* sp = seg + (long long)b * nc * HW + shw;
    if (keep) {
      if (!warped) img = (b2 < B ? fake : real)[(long long)b * HW + shw];
      if (COLOR && (!MASKED || (policy & S2E_DIFFAUG_COLOR))) {   // brightness, then contrast around the brightened image's mean
                                                                  // (saturation: identity on 1 channel)
        const float br = __ldg(r) - 0.5f, ct = __ldg(r + 1) + 0.5f;
        const float mb = __ldg(means + b2) + br;
        img = (img + br - mb) * ct + mb;
      }
    }
    bf16* o = out + p * Cpad;
    if ((Cpad & 7) == 0) {
      for (int c0 = 0; c0 < Cpad; c0 += 8) {
        float v[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int c = c0 + jj;
          v[jj] = c < nc ? (keep ? sp[(long long)c * HW] : 0.f) : (c == nc ? img : 0.f);
        }
        st_stream8(o + c0, pack8(v));
      }
    } else {
      for (int c = 0; c < Cpad; ++c) o[c] = __float2bfloat16(c < nc ? (keep ? sp[(long long)c * HW] : 0.f) : (c == nc ? img : 0.f));
    }
  }
}

// g'(b, i, j): the gradient of output channel nc at the pixel that read source (i, j), 0 if none did
__device__ __forceinline__ float da_grad_gather(const bf16* __restrict__ dxin, int nc, int Cpad, int H, int W, int b, int i, int j,
                                                const float* r, int policy) {
  int oi = i, oj = j;
  if (policy & S2E_DIFFAUG_TRANSLATION) {
    oi -= (int)__ldg(r + 2);
    oj -= (int)__ldg(r + 3);
  }
  if (oi < 0 || oi >= H || oj < 0 || oj >= W || !da_not_cut(oi, oj, H, W, r, policy)) return 0.f;
  return __bfloat162float(dxin[(((long long)b * H + oi) * W + oj) * Cpad + nc]);
}
// contrast's adjoint needs sum(g') per sample: block b reduces it in fp64 (MASKED: only where the sample's colour gate passed)
template <bool MASKED = false>
__global__ void __launch_bounds__(1024) d_input_grad_aug_sum_kernel(const bf16* __restrict__ dxin, int nc, int Cpad, int H, int W,
                                                                    const float* __restrict__ rec, int policy_all, double* __restrict__ sums,
                                                                    const int* __restrict__ opmask = nullptr) {
  const int b = blockIdx.x;
  const int policy = MASKED ? policy_all & __ldg(opmask + b) : policy_all;
  if (MASKED && !(policy & S2E_DIFFAUG_COLOR)) return;    // block-uniform: the apply kernel passes this sample's gradient through
  const float* r = rec + (long long)b * S2E_DIFFAUG_RECORD;
  double s = 0.0;
  for (long long hw = threadIdx.x; hw < (long long)H * W; hw += blockDim.x)
    s += (double)da_grad_gather(dxin, nc, Cpad, H, W, b, (int)(hw / W), (int)(hw % W), r, policy);
  s = block_sum_f64(s);
  if (threadIdx.x == 0) sums[b] = s;
}
// the unfolded images k = s0 + 2 t (n-1), s0 in {s, -s} (once when s is 0 or n-1), that lie in [lo, hi]: callback f(k)
template <class Fn>
__device__ __forceinline__ void da_for_images(int s, int n, double lo, double hi, Fn&& f) {
  const int period = 2 * (n - 1);
  for (int fam = 0; fam < ((s == 0 || s == n - 1) ? 1 : 2); ++fam) {
    const int s0 = fam ? -s : s;
    const int t0 = (int)ceil((lo - s0) / period), t1 = (int)floor((hi - s0) / period);
    for (int t = t0; t <= t1; ++t) f(s0 + t * period);
  }
}
// Warp^T(h) at source pixel (sr, sc) of sample b: every (warped-image position, bilinear tap) pair whose folded tap is
// (sr, sc), summed in a fixed order.  The boxes only bound the search; the forward's own fp32 taps decide.
__device__ float da_warp_adjoint(const bf16* __restrict__ dxin, int nc, int Cpad, int H, int W, int b, int sr, int sc,
                                 const float* r, int policy, const float* m) {
  const double hx = 0.5 * (W - 1), hy = 0.5 * (H - 1);
  const double m0 = m[0], m1 = m[1], m2 = m[2], m3 = m[3], m4 = m[4], m5 = m[5];
  // reach: the taps of M (output rect), widened
  const double ex = fabs(m0) * hx + fabs(m1) * hy, ey = fabs(m3) * hx + fabs(m4) * hy;
  const double xlo = m2 + hx - ex - 2.0, xhi = m2 + hx + ex + 2.0, ylo = m5 + hy - ey - 2.0, yhi = m5 + hy + ey + 2.0;
  const double det = m0 * m4 - m1 * m3;
  const double i00 = m4 / det, i01 = -m1 / det, i10 = -m3 / det, i11 = m0 / det;
  const double bx = fabs(i00) + fabs(i01) + 1.0, by = fabs(i10) + fabs(i11) + 1.0;    // M^-1 ([-1, 1]^2), + 1 pixel
  float acc = 0.f;
  da_for_images(sr, H, ylo, yhi, [&](int R) {
    da_for_images(sc, W, xlo, xhi, [&](int C) {
      const double px = C - hx - m2, py = R - hy - m5;
      const double qx = i00 * px + i01 * py + hx, qy = i10 * px + i11 * py + hy;
      const int j0 = max(0, (int)ceil(qx - bx)), j1 = min(W - 1, (int)floor(qx + bx));
      const int q0 = max(0, (int)ceil(qy - by)), q1 = min(H - 1, (int)floor(qy + by));
      for (int qi = q0; qi <= q1; ++qi)
        for (int qj = j0; qj <= j1; ++qj) {
          float X, Y;
          da_warp(m, qi, qj, H, W, X, Y);
          const float x0 = floorf(X), y0 = floorf(Y);
          const int dx = C - (int)x0, dy = R - (int)y0;
          if ((unsigned)dx > 1u || (unsigned)dy > 1u) continue;
          const float fx = X - x0, fy = Y - y0;
          const float w = (dy ? fy : 1.f - fy) * (dx ? fx : 1.f - fx);
          acc = fmaf(w, da_grad_gather(dxin, nc, Cpad, H, W, b, qi, qj, r, policy), acc);
        }
    });
  });
  return acc;
}

template <bool COLOR, bool MASKED = false, bool GEOM = false>
__global__ void d_input_grad_aug_kernel(const bf16* __restrict__ dxin, int B, int nc, int Cpad, int H, int W, const float* __restrict__ rec,
                                        int policy_all, const double* __restrict__ sums, float* __restrict__ dfake,
                                        const int* __restrict__ opmask = nullptr, const float* __restrict__ geom = nullptr) {
  const long long HW = (long long)H * W;
  GRID_STRIDE(p, (long long)B * HW) {
    const int b = (int)(p / HW);
    const long long hw = p % HW;
    const int policy = MASKED ? policy_all & __ldg(opmask + b) : policy_all;
    const float* r = rec + (long long)b * S2E_DIFFAUG_RECORD;
    float g;
    if constexpr (GEOM) {
      const int i = (int)(hw / W), j = (int)(hw % W);
      if (policy & S2E_DIFFAUG_GEOMETRIC) {
        float m[6];
        da_load_m(geom, b, policy, __ldg(opmask + b), m);
        g = da_warp_adjoint(dxin, nc, Cpad, H, W, b, i, j, r, policy, m);
      } else {
        g = da_grad_gather(dxin, nc, Cpad, H, W, b, i, (policy & S2E_DIFFAUG_XFLIP) ? W - 1 - j : j, r, policy);
      }
    } else {
      g = da_grad_gather(dxin, nc, Cpad, H, W, b, (int)(hw / W), (int)(hw % W), r, policy);
    }
    if (COLOR && (!MASKED || (policy & S2E_DIFFAUG_COLOR))) {   // dfake = c g' + (1 - c) mean(g'); a gated-off sample passes g' through
      const float ct = __ldg(r + 1) + 0.5f;
      g = fmaf(ct, g, (1.f - ct) * (float)(__ldg(sums + b) / (double)HW));
    }
    dfake[p] = g;
  }
}

// ADA's controller (Karras et al., NeurIPS 2020), one thread: the formulas are in the header next to s2e_ada_update
__global__ void ada_update_kernel(const double* __restrict__ stat, int num_D, double* __restrict__ acc, int* __restrict__ pos,
                                  double* __restrict__ p, double target, double kimg, int interval) {
  const int n = 2 * num_D + 1;
  for (int k = 0; k < n; ++k) acc[k] += stat[k];
  const int q = *pos + 1;
  if (q < interval) {
    *pos = q;
    return;
  }
  double r = 0.0;
  for (int i = 0; i < num_D; ++i) r += acc[2 * i] / acc[2 * i + 1];
  r /= (double)num_D;
  const double sgn = (double)((r > target) - (r < target));
  p[0] = fmin(fmax(p[0] + sgn * acc[2 * num_D] / (kimg * 1000.0), 0.0), 1.0);
  acc[n] = r;
  for (int k = 0; k < n; ++k) acc[k] = 0.0;
  *pos = 0;
}

// ------------------------------------------------------------------------------------------ elementwise
__global__ void add_kernel(const bf16* __restrict__ a, const bf16* __restrict__ b, long long nvec, long long n, bf16* __restrict__ y) {
  GRID_STRIDE(i, nvec) {
    float fa[8], fb[8];
    unpack8(*reinterpret_cast<const bf16x8*>(a + i * 8), fa);
    unpack8(*reinterpret_cast<const bf16x8*>(b + i * 8), fb);
#pragma unroll
    for (int j = 0; j < 8; ++j) fa[j] += fb[j];
    *reinterpret_cast<bf16x8*>(y + i * 8) = pack8(fa);
  }
  if (blockIdx.x == 0)
    for (long long i = nvec * 8 + threadIdx.x; i < n; i += blockDim.x)
      y[i] = __float2bfloat16(__bfloat162float(a[i]) + __bfloat162float(b[i]));
}
__global__ void act_fwd_kernel(const bf16* __restrict__ x, long long n, int act, bf16* __restrict__ y) {
  GRID_STRIDE(i, n) y[i] = __float2bfloat16(act_apply(__bfloat162float(x[i]), act));
}
__global__ void act_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ y, long long n, int act, bf16* __restrict__ dx) {
  GRID_STRIDE(i, n) {
    const float o = __bfloat162float(y[i]);
    float g = __bfloat162float(dy[i]);
    if (act == S2E_ACT_LRELU) g *= (o > 0.f ? 1.f : 0.2f);
    if (act == S2E_ACT_RELU) g *= (o > 0.f ? 1.f : 0.f);
    dx[i] = __float2bfloat16(g);
  }
}
__global__ void tanh_fwd_kernel(const bf16* __restrict__ x, long long n, float* __restrict__ y) {
  GRID_STRIDE(i, n) y[i] = tanhf(__bfloat162float(x[i]));
}
__global__ void tanh_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, long long n, bf16* __restrict__ dx) {
  GRID_STRIDE(i, n) dx[i] = __float2bfloat16(dy[i] * (1.f - y[i] * y[i]));
}
__global__ void fill_kernel(float* p, long long n, float v) { GRID_STRIDE(i, n) p[i] = v; }

// ------------------------------------------------------------------------------------------ small linear layers
__device__ __forceinline__ float lin_x(const void* x, int m, int k, int K, int hw) {
  if (hw <= 0) return ((const float*)x)[(long long)m * K + k];
  const int Cc = K / hw, c = k / hw, s = k % hw;  // flattened NCHW index k = c*hw + s ; stored NHWC
  const float v = __bfloat162float(((const bf16*)x)[((long long)m * hw + s) * Cc + c]);
  return v > 0.f ? v : 0.2f * v;
}
__global__ void linear_fwd_kernel(const void* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b, int M, int N,
                                  int K, int act, int hw, float* __restrict__ y) {
  const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (o >= M * N) return;
  const int lane = threadIdx.x & 31, m = o / N, n = o % N;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc = fmaf(lin_x(x, m, k, K, hw), w[(long long)n * K + k], acc);
  acc = warp_sum(acc);
  if (lane == 0) y[o] = act_apply(acc + (b ? b[n] : 0.f), act);
}
__device__ __forceinline__ float lin_dpre(const float* dy, const float* y, int idx, int act) {
  float g = dy[idx];
  if (act == S2E_ACT_LRELU) g *= (y[idx] > 0.f ? 1.f : 0.2f);
  if (act == S2E_ACT_RELU) g *= (y[idx] > 0.f ? 1.f : 0.f);
  return g;
}
__global__ void linear_bwd_dx_kernel(const float* __restrict__ dy, const float* __restrict__ y, const void* __restrict__ x,
                                     const float* __restrict__ w, int M, int N, int K, int act, int hw, void* __restrict__ dx) {
  GRID_STRIDE(i, (long long)M * K) {
    const int m = (int)(i / K), k = (int)(i % K);
    float acc = 0.f;
    for (int n = 0; n < N; ++n) acc = fmaf(lin_dpre(dy, y, m * N + n, act), w[(long long)n * K + k], acc);
    if (hw <= 0) {
      ((float*)dx)[i] = acc;
    } else {
      const int Cc = K / hw, c = k / hw, s = k % hw;
      const long long xi = ((long long)m * hw + s) * Cc + c;
      const float xv = __bfloat162float(((const bf16*)x)[xi]);
      ((bf16*)dx)[xi] = __float2bfloat16(acc * (xv > 0.f ? 1.f : 0.2f));
    }
  }
}
template <int KMAX>
__global__ void __launch_bounds__(256) linear_bwd_dx_smallk_kernel(const float* __restrict__ dy, const float* __restrict__ y,
                                                                    const float* __restrict__ w, int N, int K, int act,
                                                                    float* __restrict__ dx) {
  __shared__ float red[8][KMAX];
  const int m = blockIdx.x;
  float acc[KMAX];
#pragma unroll
  for (int k = 0; k < KMAX; ++k) acc[k] = 0.f;
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    const float g = lin_dpre(dy, y, m * N + n, act);
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
      if (k < K) acc[k] = fmaf(g, w[(long long)n * K + k], acc[k]);
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const float v = warp_sum(acc[k]);
    if (lane == 0) red[wid][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    float v = 0.f;
    for (int i = 0; i < 8; ++i) v += red[i][threadIdx.x];
    dx[(long long)m * K + threadIdx.x] = v;
  }
}

__global__ void linear_bwd_dw_kernel(const float* __restrict__ dy, const float* __restrict__ y, const void* __restrict__ x, int M, int N,
                                     int K, int act, int hw, float* __restrict__ dw, float* __restrict__ db) {
  GRID_STRIDE(i, (long long)N * K) {
    const int n = (int)(i / K), k = (int)(i % K);
    float acc = 0.f, accb = 0.f;
    for (int m = 0; m < M; ++m) {
      const float g = lin_dpre(dy, y, m * N + n, act);
      acc = fmaf(g, lin_x(x, m, k, K, hw), acc);
      accb += g;
    }
    dw[i] = acc;
    if (k == 0 && db) db[n] = accb;
  }
}

// ------------------------------------------------------------------------------------------ losses
__device__ __forceinline__ float ld_any(const void* p, long long i, int f32) {
  return f32 ? ((const float*)p)[i] : __bfloat162float(((const bf16*)p)[i]);
}
__device__ __forceinline__ float loss_value(float a, float b, int kind, float target) {
  switch (kind) {
    case S2E_RED_SUM: return a;
    case S2E_RED_HINGE_REAL: return fminf(a - 1.f, 0.f);
    case S2E_RED_HINGE_FAKE: return fminf(-a - 1.f, 0.f);
    case S2E_RED_LS: return (a - target) * (a - target);
    case S2E_RED_BCE: return fmaxf(a, 0.f) - a * target + log1pf(expf(-fabsf(a)));   // BCE with logits, stable form
    case S2E_RED_L1: return fabsf(a - b);
    case S2E_RED_SIGN: return (float)((a > 0.f) - (a < 0.f));
    default: return (a - b) * (a - b);
  }
}
__device__ __forceinline__ float loss_grad(float a, float b, int kind, float target) {
  switch (kind) {
    case S2E_RED_SUM: return 1.f;
    case S2E_RED_HINGE_REAL: return (a - 1.f < 0.f) ? 1.f : 0.f;
    case S2E_RED_HINGE_FAKE: return (-a - 1.f < 0.f) ? -1.f : 0.f;
    case S2E_RED_LS: return 2.f * (a - target);
    case S2E_RED_BCE: return 1.f / (1.f + expf(-a)) - target;
    case S2E_RED_L1: {
      const float df = a - b;
      return df > 0.f ? 1.f : (df < 0.f ? -1.f : 0.f);
    }
    case S2E_RED_SIGN: return 0.f;
    default: return 2.f * (a - b);
  }
}
// bf16 tensors whose pointers are 16-byte aligned take the 8-wide path (the feature-matching loss runs over the big
// discriminator features); everything else (fp32 images, ragged tails) goes element by element.
__global__ void reduce_loss_kernel(const void* __restrict__ x, const void* __restrict__ y, long long n, int f32, int kind, float coef,
                                   float target, int vec, float* out) {
  float acc = 0.f;
  const bool two = (kind == S2E_RED_L1 || kind == S2E_RED_L2);
  const long long nv = vec ? n >> 3 : 0;
  GRID_STRIDE(i, nv) {
    float a[8], b[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    unpack8(ld_stream8((const bf16*)x + i * 8), a);
    if (two) unpack8(ld_stream8((const bf16*)y + i * 8), b);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc += loss_value(a[j], b[j], kind, target);
  }
  for (long long i = nv * 8 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc += loss_value(ld_any(x, i, f32), two ? ld_any(y, i, f32) : 0.f, kind, target);
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(out, acc * coef);
}
__global__ void reduce_loss_bwd_kernel(const void* __restrict__ x, const void* __restrict__ y, long long n, int f32, int kind, float coef,
                                       float target, int vec, const float* __restrict__ gout, void* __restrict__ dx, int accumulate) {
  const float g0 = gout[0] * coef;
  const bool two = (kind == S2E_RED_L1 || kind == S2E_RED_L2);
  const long long nv = vec ? n >> 3 : 0;
  GRID_STRIDE(i, nv) {
    float a[8], b[8] = {0, 0, 0, 0, 0, 0, 0, 0}, o[8], prev[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    unpack8(ld_stream8((const bf16*)x + i * 8), a);
    if (two) unpack8(ld_stream8((const bf16*)y + i * 8), b);
    if (accumulate) unpack8(*reinterpret_cast<const bf16x8*>((bf16*)dx + i * 8), prev);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = prev[j] + g0 * loss_grad(a[j], b[j], kind, target);
    *reinterpret_cast<bf16x8*>((bf16*)dx + i * 8) = pack8(o);
  }
  for (long long i = nv * 8 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float d = g0 * loss_grad(ld_any(x, i, f32), two ? ld_any(y, i, f32) : 0.f, kind, target);
    if (f32) {
      float* o = (float*)dx;
      o[i] = accumulate ? o[i] + d : d;
    } else {
      bf16* o = (bf16*)dx;
      o[i] = __float2bfloat16(accumulate ? __bfloat162float(o[i]) + d : d);
    }
  }
}

// state[0] = step count, state[1] = lr, state[2] = lr / (1 - b1^step), state[3] = sqrt(1 - b2^step)
__global__ void adam_prepare_kernel(float* state, float b1, float b2) {
  const float step = state[0] + 1.f;
  state[0] = step;
  state[2] = state[1] / (1.f - powf(b1, step));
  state[3] = sqrtf(1.f - powf(b2, step));
}
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                            const float* __restrict__ state, float b1, float b2, float eps, float wd) {
  const float step_size = state[2], bc2_sqrt = state[3];
  GRID_STRIDE(i, n) {
    float gi = g[i];
    if (wd != 0.f) gi = fmaf(wd, p[i], gi);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= step_size * (mi / denom);
  }
}

// Multi-tensor Adam: a block owns one 4096-element chunk of one tensor of the table (float4 path when the chunk is
// full; every pointer comes from the caching allocator, i.e. is at least 16-byte aligned).
constexpr int ADAM_MAX_TENSORS = 48;
constexpr int ADAM_CHUNK = 4096;
struct AdamTable {
  int nt;
  float* p[ADAM_MAX_TENSORS];
  const float* g[ADAM_MAX_TENSORS];
  float* m[ADAM_MAX_TENSORS];
  float* v[ADAM_MAX_TENSORS];
  long long n[ADAM_MAX_TENSORS];
  int blk0[ADAM_MAX_TENSORS];
};
// the EMA instantiation: e[k] is the moving average of p[k], decay the user's beta (the ramp is applied on the device)
struct AdamEmaTable : AdamTable {
  float* e[ADAM_MAX_TENSORS];
  float decay;
};
__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float b1, float b2, float eps, float wd,
                                         float step_size, float bc2_sqrt) {
  if (wd != 0.f) g = fmaf(wd, p, g);
  m = b1 * m + (1.f - b1) * g;
  v = b2 * v + (1.f - b2) * g * g;
  const float denom = sqrtf(v) / bc2_sqrt + eps;
  p -= step_size * (m / denom);
}
// EMA = true: after the Adam update, e <- fmaf(beta_t, e - p, p) with the new p, where beta_t = min(decay, (1+t)/(10+t))
// and t = state[0], the step count s2e_adam_prepare just advanced (so a CUDA-graph replay ramps correctly).
template <bool EMA>
__global__ void __launch_bounds__(256) adam_multi_kernel(const __grid_constant__ std::conditional_t<EMA, AdamEmaTable, AdamTable> t,
                                                         const float* __restrict__ state, float b1, float b2, float eps, float wd) {
  int k = 0;
  while (k + 1 < t.nt && (int)blockIdx.x >= t.blk0[k + 1]) ++k;
  const long long off = (long long)(blockIdx.x - t.blk0[k]) * ADAM_CHUNK;
  const long long left = t.n[k] - off;
  float* __restrict__ p = t.p[k] + off;
  const float* __restrict__ g = t.g[k] + off;
  float* __restrict__ m = t.m[k] + off;
  float* __restrict__ v = t.v[k] + off;
  const float step_size = state[2], bc2_sqrt = state[3];
  float* __restrict__ ema = nullptr;
  float bt = 0.f;
  if constexpr (EMA) {
    ema = t.e[k] + off;
    bt = fminf(t.decay, (1.f + state[0]) / (10.f + state[0]));
  }
  const bool aligned = ((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)m) | ((uintptr_t)v) | ((uintptr_t)ema)) & 15) == 0;
  if (left >= ADAM_CHUNK && aligned) {
#pragma unroll
    for (int i = 0; i < ADAM_CHUNK / (256 * 4); ++i) {
      const int e = (i * 256 + threadIdx.x) * 4;
      float4 pv = *reinterpret_cast<float4*>(p + e);
      const float4 gv = *reinterpret_cast<const float4*>(g + e);
      float4 mv = *reinterpret_cast<float4*>(m + e);
      float4 vv = *reinterpret_cast<float4*>(v + e);
      adam_one(pv.x, gv.x, mv.x, vv.x, b1, b2, eps, wd, step_size, bc2_sqrt);
      adam_one(pv.y, gv.y, mv.y, vv.y, b1, b2, eps, wd, step_size, bc2_sqrt);
      adam_one(pv.z, gv.z, mv.z, vv.z, b1, b2, eps, wd, step_size, bc2_sqrt);
      adam_one(pv.w, gv.w, mv.w, vv.w, b1, b2, eps, wd, step_size, bc2_sqrt);
      *reinterpret_cast<float4*>(p + e) = pv;
      *reinterpret_cast<float4*>(m + e) = mv;
      *reinterpret_cast<float4*>(v + e) = vv;
      if constexpr (EMA) {
        float4 ev = *reinterpret_cast<float4*>(ema + e);
        ev.x = fmaf(bt, ev.x - pv.x, pv.x);
        ev.y = fmaf(bt, ev.y - pv.y, pv.y);
        ev.z = fmaf(bt, ev.z - pv.z, pv.z);
        ev.w = fmaf(bt, ev.w - pv.w, pv.w);
        *reinterpret_cast<float4*>(ema + e) = ev;
      }
    }
  } else {
    const int cnt = (int)(left < ADAM_CHUNK ? left : ADAM_CHUNK);
    for (int e = threadIdx.x; e < cnt; e += 256) {
      float pv = p[e], mv = m[e], vv = v[e];
      adam_one(pv, g[e], mv, vv, b1, b2, eps, wd, step_size, bc2_sqrt);
      p[e] = pv;
      m[e] = mv;
      v[e] = vv;
      if constexpr (EMA) ema[e] = fmaf(bt, ema[e] - pv, pv);
    }
  }
}

// Multi-tensor byte copy (the EMA nets' buffers): a block owns one COPY_CHUNK-byte chunk of one row of the table, moved
// in 16-byte words when both ends are 16-byte aligned.
constexpr int COPY_MAX_ROWS = 48;
constexpr int COPY_CHUNK = 16384;
struct CopyTable {
  int nr;
  void* dst[COPY_MAX_ROWS];
  const void* src[COPY_MAX_ROWS];
  long long nbytes[COPY_MAX_ROWS];
  int blk0[COPY_MAX_ROWS];
};
__global__ void __launch_bounds__(256) copy_multi_kernel(const __grid_constant__ CopyTable t) {
  int k = 0;
  while (k + 1 < t.nr && (int)blockIdx.x >= t.blk0[k + 1]) ++k;
  const long long off = (long long)(blockIdx.x - t.blk0[k]) * COPY_CHUNK;
  const int cnt = (int)(t.nbytes[k] - off < COPY_CHUNK ? t.nbytes[k] - off : COPY_CHUNK);
  unsigned char* d = (unsigned char*)t.dst[k] + off;
  const unsigned char* s = (const unsigned char*)t.src[k] + off;
  int head = 0;
  if (((((uintptr_t)d) | ((uintptr_t)s)) & 15) == 0) {
    head = cnt & ~15;
    for (int i = threadIdx.x * 16; i < head; i += 256 * 16)
      *reinterpret_cast<uint4*>(d + i) = *reinterpret_cast<const uint4*>(s + i);
  }
  for (int i = head + threadIdx.x; i < cnt; i += 256) d[i] = s[i];
}

PackGeom make_pack_geom(int Cout, int Cin, int kh, int kw, int stride, int pad, int Ctot = 0, int co_off = 0, int cin_pad = 0) {
  PackGeom g;
  g.CinPad = cin_pad > Cin ? cin_pad : Cin;
  g.Ctot = Ctot > 0 ? Ctot : Cout;
  g.co_off = co_off;
  g.Cout = Cout;
  g.Cin = Cin;
  g.kh = kh;
  g.kw = kw;
  g.stride = stride;
  g.pad = pad;
  g.amin = floor_div(-pad, 2);
  g.bmin = floor_div(-pad, 2);
  g.na = floor_div(kh - 1 - pad, 2) - g.amin + 1;
  g.nb = floor_div(kw - 1 - pad, 2) - g.bmin + 1;
  return g;
}

}  // namespace

// ========================================================================================== C ABI
extern "C" {

const char* s2e_last_error(void) { return g_err; }
int s2e_abi_version(void) { return 1; }
int s2e_debug_set(int key, int value) {
  if (key < 0 || key >= 8) return S2E_ERR_ARG;
  g_debug[key] = value;
  return S2E_OK;
}

int s2e_tapconv_fwd(const s2e_conv_t* d, const void* x, const void* wp, const float* bias, const float* scale, void* y,
                    int impl, void* stream) {
  S2E_REQUIRE(d && d->ntaps >= 1 && d->ntaps <= S2E_MAX_TAPS, "tapconv_fwd: bad tap count");
  if (impl == S2E_IMPL_SIMT || g_debug[1]) return s2e_tapconv_fwd_simt(d, x, wp, bias, scale, y, (cudaStream_t)stream);
  return s2e_tapconv_fwd_tc(d, x, wp, bias, scale, y, (cudaStream_t)stream);
}
int s2e_tapconv_wgrad(const s2e_conv_t* d, const void* x, const void* dy, float* dwp, int impl, void* stream) {
  S2E_REQUIRE(d && d->ntaps >= 1 && d->ntaps <= S2E_MAX_TAPS, "tapconv_wgrad: bad tap count");
  if (impl == S2E_IMPL_SIMT || g_debug[1]) return s2e_tapconv_wgrad_simt(d, x, dy, dwp, (cudaStream_t)stream);
  return s2e_tapconv_wgrad_tc(d, x, dy, dwp, (cudaStream_t)stream);
}

int s2e_onehot_nchw(const int64_t* label, int B, int H, int W, int nc, float* out, void* stream) {
  const long long n = (long long)B * nc * H * W;
  if (!n) return S2E_OK;
  onehot_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const long long*)label, (long long)H * W, nc, n, out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_seg_nearest_nhwc(const float* seg, int B, int C, int Hs, int Ws, int Hd, int Wd, int Cpad, void* out, void* stream) {
  S2E_REQUIRE(Cpad >= C, "seg_nearest: Cpad < C");
  const long long n = (long long)B * Hd * Wd * Cpad;
  if (!n) return S2E_OK;
  const float sh = (float)Hs / (float)Hd, sw = (float)Ws / (float)Wd;
  seg_nearest_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(seg, C, Hs, Ws, Hd, Wd, Cpad, sh, sw, n, (bf16*)out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_seg_im2col3x3(const float* seg, int B, int C, int Hs, int Ws, int Hd, int Wd, void* out, void* stream) {
  S2E_REQUIRE(9 * C <= 62, "seg_im2col3x3: 9*C + the two constant-one channels must fit 64 channels (C=%d)", C);
  const long long n = (long long)B * Hd * Wd * 8;
  if (!n) return S2E_OK;
  if (C == 4)
    seg_im2col_c4_kernel<<<grid1d(n / 8, 128), 128, 0, (cudaStream_t)stream>>>(seg, Hs, Ws, Hd, Wd, (float)Hs / (float)Hd,
                                                                              (float)Ws / (float)Wd, n / 8, (bf16*)out);
  else
    seg_im2col_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(seg, C, Hs, Ws, Hd, Wd, (float)Hs / (float)Hd, (float)Ws / (float)Wd,
                                                                  n, (bf16*)out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_pack_weight_im2col3x3(const float* w, int Cout, int C, void* out, void* stream) {
  S2E_REQUIRE(9 * C <= 64, "pack_weight_im2col3x3: 9*C must fit 64 channels");
  pack_im2col_kernel<<<grid1d((long long)Cout * 64), NT, 0, (cudaStream_t)stream>>>(w, Cout, C, (bf16*)out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_unpack_wgrad_im2col3x3(const float* dwp, int Cout, int C, float* dw, float* db, void* stream) {
  unpack_im2col_kernel<<<grid1d((long long)Cout * C * 9), NT, 0, (cudaStream_t)stream>>>(dwp, Cout, C, dw, db);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_nchw_f32_to_nhwc_bf16(const float* x, int B, int C, int H, int W, void* y, void* stream) {
  const long long n = (long long)B * C * H * W;
  if (!n) return S2E_OK;
  nchw2nhwc_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(x, C, H, W, n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_nhwc_bf16_to_nchw_f32(const void* x, int B, int C, int H, int W, float* y, void* stream) {
  const long long n = (long long)B * C * H * W;
  if (!n) return S2E_OK;
  nhwc2nchw_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, C, H, W, n, y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_packed_taps(int kh, int kw, int stride, int pad, int* ntaps, int* dy, int* dx) {
  S2E_REQUIRE(stride == 1 || stride == 2, "packed_taps: stride must be 1 or 2");
  PackGeom g = make_pack_geom(1, 1, kh, kw, stride, pad);
  int n = 0;
  if (stride == 1) {
    for (int r = 0; r < kh; ++r)
      for (int s = 0; s < kw; ++s) {
        if (n >= S2E_MAX_TAPS) return S2E_ERR_UNSUPPORTED;
        dy[n] = r - pad;
        dx[n] = s - pad;
        ++n;
      }
  } else {
    for (int a = 0; a < g.na; ++a)
      for (int b = 0; b < g.nb; ++b) {
        if (n >= S2E_MAX_TAPS) return S2E_ERR_UNSUPPORTED;
        dy[n] = g.amin + a;
        dx[n] = g.bmin + b;
        ++n;
      }
  }
  *ntaps = n;
  return S2E_OK;
}
int s2e_pack_weight(const float* w, int Cout, int Cin, int kh, int kw, int stride, int pad, int transposed, int Cout_total,
                    int co_offset, int cin_pad, void* out, void* stream) {
  S2E_REQUIRE(stride == 1 || stride == 2, "pack_weight: stride must be 1 or 2");
  PackGeom g = make_pack_geom(Cout, Cin, kh, kw, stride, pad, Cout_total, co_offset, cin_pad);
  const int T = stride == 1 ? kh * kw : g.na * g.nb;
  const long long n = (long long)T * Cout * (stride == 2 ? 4 * g.CinPad : g.CinPad);
  pack_weight_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(w, g, transposed, n, (bf16*)out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_unpack_wgrad(const float* dwp, int Cout, int Cin, int kh, int kw, int stride, int pad, int Cout_total, int co_offset,
                     int cin_pad, const float* w_orig, const float* u, const float* v, const float* inv_sigma, float* dot,
                     float* dw, int accumulate, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  PackGeom g = make_pack_geom(Cout, Cin, kh, kw, stride, pad, Cout_total, co_offset, cin_pad);
  const long long n = (long long)Cout * Cin * kh * kw;
  if (u) {
    S2E_REQUIRE(v && inv_sigma && dot && w_orig, "unpack_wgrad: spectral args incomplete");
    S2E_CHECK_CUDA(cudaMemsetAsync(dot, 0, sizeof(float), st));
    wgrad_dot_kernel<<<grid1d(n), NT, 0, st>>>(dwp, w_orig, g, n, dot);
    S2E_LAUNCH_CHECK();
  }
  unpack_wgrad_kernel<<<grid1d(n), NT, 0, st>>>(dwp, g, u, v, inv_sigma, dot, n, accumulate, dw);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_spectral_power_iter_multi(const s2e_sn_job_t* jobs, int n_jobs, int update, int n_iters, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  S2E_REQUIRE(n_jobs >= 0 && n_iters >= 1, "spectral_power_iter_multi: bad counts");
  for (int base = 0; base < n_jobs; base += SN_MAX_JOBS) {
    SnTable t;
    t.n = n_jobs - base < SN_MAX_JOBS ? n_jobs - base : SN_MAX_JOBS;
    int blk_a = 0, blk_c = 0;
    for (int k = 0; k < t.n; ++k) {
      const s2e_sn_job_t& s = jobs[base + k];
      S2E_REQUIRE(s.w && s.u && s.v && s.inv_sigma && s.scratch && s.rows > 0 && s.cols > 0, "spectral_power_iter_multi: job %d incomplete", base + k);
      SnJob& J = t.j[k];
      J.w = s.w; J.u = s.u; J.v = s.v; J.inv = s.inv_sigma; J.scratch = s.scratch; J.ucopy = s.u_copy; J.vcopy = s.v_copy;
      J.rows = s.rows; J.cols = s.cols;
      J.blk_a = blk_a; J.blk_c = blk_c;
      blk_a += ceil_div(s.cols, 128) * ceil_div(s.rows, SN_RCHUNK);
      blk_c += ceil_div(s.rows, 8);
    }
    for (int it = 0; it < n_iters; ++it) {
      t.it = it;
      if (update) {
        sn_wt_u_multi_kernel<<<blk_a, 128, 0, st>>>(t);
        sn_normalize_multi_kernel<<<t.n, 1024, 0, st>>>(t, 0);
        sn_w_v_multi_kernel<<<blk_c, 256, 0, st>>>(t);
        sn_normalize_multi_kernel<<<t.n, 1024, 0, st>>>(t, 1);
      } else {
        sn_w_v_multi_kernel<<<blk_c, 256, 0, st>>>(t);
        sn_dot_multi_kernel<<<t.n, 1024, 0, st>>>(t);
      }
      S2E_LAUNCH_CHECK();
    }
  }
  return S2E_OK;
}
int s2e_spectral_power_iter(const float* w, int rows, int cols, float* u, float* v, float* inv_sigma, float* scratch,
                            int update, float* u_copy, float* v_copy, void* stream) {
  s2e_sn_job_t j;
  j.w = w; j.u = u; j.v = v; j.inv_sigma = inv_sigma; j.scratch = scratch; j.u_copy = u_copy; j.v_copy = v_copy;
  j.rows = rows; j.cols = cols;
  return s2e_spectral_power_iter_multi(&j, 1, update, 1, stream);
}

int s2e_space_to_depth(const void* x, int B, int H, int W, int C, void* y, void* stream) {
  const int H2 = (H + 1) / 2, W2 = (W + 1) / 2;
  const int vec = (C % 8 == 0) ? 8 : 1;
  const long long n = (long long)B * H2 * W2 * 4 * (C / vec);
  if (!n) return S2E_OK;
  S2E_REQUIRE(n < (1LL << 31), "space_to_depth: tensor too large for 32-bit indexing");
  if (vec == 8)
    s2d_kernel<8><<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, H, W, C, H2, W2, (unsigned)n, (bf16*)y);
  else
    s2d_kernel<1><<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, H, W, C, H2, W2, (unsigned)n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_depth_to_space(const void* dy, int B, int H, int W, int C, void* dx, void* stream) {
  const int H2 = (H + 1) / 2, W2 = (W + 1) / 2;
  const int vec = (C % 8 == 0) ? 8 : 1;
  const long long n = (long long)B * H * W * (C / vec);
  if (!n) return S2E_OK;
  S2E_REQUIRE(n < (1LL << 31), "depth_to_space: tensor too large for 32-bit indexing");
  if (vec == 8)
    d2s_kernel<8><<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, H, W, C, H2, W2, (unsigned)n, (bf16*)dx);
  else
    d2s_kernel<1><<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, H, W, C, H2, W2, (unsigned)n, (bf16*)dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_upsample2x_fwd(const void* x, int B, int H, int W, int C, void* y, void* stream) {
  S2E_REQUIRE(C % 8 == 0, "upsample2x needs C %% 8 == 0");
  const long long n = (long long)B * 4 * H * W * (C / 8);
  if (!n) return S2E_OK;
  upsample2x_fwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, H, W, C / 8, n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_upsample2x_bwd(const void* dy, int B, int H, int W, int C, void* dx, void* stream) {
  S2E_REQUIRE(C % 8 == 0, "upsample2x needs C %% 8 == 0");
  const long long n = (long long)B * H * W * (C / 8);
  if (!n) return S2E_OK;
  upsample2x_bwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, H, W, C / 8, n, (bf16*)dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_add(const void* a, const void* b, long long n, void* y, void* stream) {
  if (!n) return S2E_OK;
  S2E_REQUIRE((((uintptr_t)a | (uintptr_t)b | (uintptr_t)y) & 15) == 0, "add: pointers must be 16B aligned");
  add_kernel<<<grid1d(n / 8 + 1), NT, 0, (cudaStream_t)stream>>>((const bf16*)a, (const bf16*)b, n / 8, n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_act_fwd(const void* x, long long n, int act, void* y, void* stream) {
  if (!n) return S2E_OK;
  act_fwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, n, act, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_act_bwd(const void* dy, const void* y, long long n, int act, void* dx, void* stream) {
  if (!n) return S2E_OK;
  act_bwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, (const bf16*)y, n, act, (bf16*)dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_avgpool3s2_fwd(const void* x, int B, int H, int W, int C, void* y, void* stream) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long n = (long long)B * Ho * Wo * C;
  if (!n) return S2E_OK;
  if (C % 8 == 0 && n / 8 < (1LL << 31))
    avgpool_fwd_vec_kernel<<<grid1d(n / 8), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, H, W, C / 8, Ho, Wo, (unsigned)(n / 8), (bf16*)y);
  else
    avgpool_fwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, H, W, C, Ho, Wo, n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_avgpool3s2_bwd(const void* dy, int B, int H, int W, int C, void* dx, void* stream) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long n = (long long)B * H * W * C;
  if (!n) return S2E_OK;
  if (C % 8 == 0 && n / 8 < (1LL << 31))
    avgpool_bwd_vec_kernel<<<grid1d(n / 8), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, H, W, C / 8, Ho, Wo, (unsigned)(n / 8), (bf16*)dx);
  else
    avgpool_bwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dy, H, W, C, Ho, Wo, n, (bf16*)dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_bilinear_fwd(const float* x, int N, int Hs, int Ws, int Hd, int Wd, void* y, void* stream) {
  const long long n = (long long)N * Hd * Wd;
  if (!n) return S2E_OK;
  bilinear_fwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(x, Hs, Ws, Hd, Wd, (float)Hs / Hd, (float)Ws / Wd, n, (bf16*)y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_bilinear_bwd(const void* dy, int N, int Hs, int Ws, int Hd, int Wd, float* dx, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = (long long)N * Hd * Wd;
  S2E_CHECK_CUDA(cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)N * Hs * Ws, st));
  if (!n) return S2E_OK;
  bilinear_bwd_kernel<<<grid1d(n), NT, 0, st>>>((const bf16*)dy, Hs, Ws, Hd, Wd, (float)Hs / Hd, (float)Ws / Wd, n, dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_make_d_input(const float* seg, const float* fake, const float* real, int B, int nc, int H, int W, int Cpad,
                     void* out, void* stream) {
  S2E_REQUIRE(Cpad > nc, "make_d_input: Cpad must exceed nc");
  const long long n = (long long)2 * B * H * W * Cpad;
  if (!n) return S2E_OK;
  const long long npix = 2LL * B * H * W;
  make_d_input_kernel<<<grid1d(npix), NT, 0, (cudaStream_t)stream>>>(seg, fake, real, B, nc, (long long)H * W, Cpad, npix, (bf16*)out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_d_input_grad(const void* dxin, int B, int nc, int H, int W, int Cpad, float* dfake, void* stream) {
  const long long n = (long long)B * H * W;
  if (!n) return S2E_OK;
  d_input_grad_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)dxin, nc, Cpad, n, dfake);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_diffaug_draw(int64_t* state, int B, long long index_offset, int H, int W, float* params_out, void* stream) {
  S2E_REQUIRE(state && B >= 0 && H > 0 && W > 0 && index_offset >= 0, "diffaug_draw: bad arguments");
  S2E_REQUIRE(index_offset + B <= (1LL << 32), "diffaug_draw: sample indices must fit in 32 bits");
  S2E_REQUIRE(B == 0 || params_out, "diffaug_draw: params_out is null");
  diffaug_draw_kernel<false><<<1, 256, 0, (cudaStream_t)stream>>>((long long*)state, B, index_offset, H, W, params_out, nullptr, nullptr);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_diffaug_draw_p(int64_t* state, const double* p, int B, long long index_offset, int H, int W, float* params_out, int* opmask_out,
                       void* stream) {
  S2E_REQUIRE(state && p && B >= 0 && H > 0 && W > 0 && index_offset >= 0, "diffaug_draw_p: bad arguments");
  S2E_REQUIRE(index_offset + B <= (1LL << 32), "diffaug_draw_p: sample indices must fit in 32 bits");
  S2E_REQUIRE(B == 0 || (params_out && opmask_out), "diffaug_draw_p: params_out / opmask_out is null");
  diffaug_draw_kernel<true><<<1, 256, 0, (cudaStream_t)stream>>>((long long*)state, B, index_offset, H, W, params_out, p, opmask_out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_diffaug_means(const float* fake, const float* real, int B, int H, int W, float* means_out, void* stream) {
  S2E_REQUIRE(B >= 0 && H > 0 && W > 0, "diffaug_means: bad arguments");
  if (!B) return S2E_OK;
  diffaug_means_kernel<<<2 * B, 1024, 0, (cudaStream_t)stream>>>(fake, real, B, (long long)H * W, means_out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_make_d_input_aug(const float* seg, const float* fake, const float* real, int B, int nc, int H, int W, int Cpad,
                         const float* params, const float* means, int policy, void* out, void* stream) {
  S2E_REQUIRE(Cpad > nc, "make_d_input_aug: Cpad must exceed nc");
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL) == 0, "make_d_input_aug: unknown policy bits %#x", policy);
  S2E_REQUIRE(params && (means || !(policy & S2E_DIFFAUG_COLOR)), "make_d_input_aug: params / means missing");
  const long long npix = 2LL * B * H * W;
  if (!npix) return S2E_OK;
  auto k = (policy & S2E_DIFFAUG_COLOR) ? make_d_input_aug_kernel<true> : make_d_input_aug_kernel<false>;
  k<<<grid1d(npix), NT, 0, (cudaStream_t)stream>>>(seg, fake, real, B, nc, H, W, Cpad, npix, params, means, policy, (bf16*)out, nullptr,
                                                   nullptr);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_d_input_grad_aug(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                         double* scratch, float* dfake, void* stream) {
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL) == 0, "d_input_grad_aug: unknown policy bits %#x", policy);
  S2E_REQUIRE(params && (scratch || !(policy & S2E_DIFFAUG_COLOR)), "d_input_grad_aug: params / scratch missing");
  const long long n = (long long)B * H * W;
  if (!n) return S2E_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (policy & S2E_DIFFAUG_COLOR) {
    d_input_grad_aug_sum_kernel<<<B, 1024, 0, st>>>((const bf16*)dxin, nc, Cpad, H, W, params, policy, scratch);
    S2E_LAUNCH_CHECK();
    d_input_grad_aug_kernel<true><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, scratch, dfake);
  } else {
    d_input_grad_aug_kernel<false><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, nullptr, dfake);
  }
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_make_d_input_aug_masked(const float* seg, const float* fake, const float* real, int B, int nc, int H, int W, int Cpad,
                                const float* params, const float* means, int policy, const int* opmask, void* out, void* stream) {
  S2E_REQUIRE(Cpad > nc, "make_d_input_aug_masked: Cpad must exceed nc");
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL) == 0, "make_d_input_aug_masked: unknown policy bits %#x", policy);
  S2E_REQUIRE(params && opmask && (means || !(policy & S2E_DIFFAUG_COLOR)), "make_d_input_aug_masked: params / opmask / means missing");
  const long long npix = 2LL * B * H * W;
  if (!npix) return S2E_OK;
  auto k = (policy & S2E_DIFFAUG_COLOR) ? make_d_input_aug_kernel<true, true> : make_d_input_aug_kernel<false, true>;
  k<<<grid1d(npix), NT, 0, (cudaStream_t)stream>>>(seg, fake, real, B, nc, H, W, Cpad, npix, params, means, policy, (bf16*)out, opmask,
                                                   nullptr);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_d_input_grad_aug_masked(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                                const int* opmask, double* scratch, float* dfake, void* stream) {
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL) == 0, "d_input_grad_aug_masked: unknown policy bits %#x", policy);
  S2E_REQUIRE(params && opmask && (scratch || !(policy & S2E_DIFFAUG_COLOR)), "d_input_grad_aug_masked: params / opmask / scratch missing");
  const long long n = (long long)B * H * W;
  if (!n) return S2E_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (policy & S2E_DIFFAUG_COLOR) {
    d_input_grad_aug_sum_kernel<true><<<B, 1024, 0, st>>>((const bf16*)dxin, nc, Cpad, H, W, params, policy, scratch, opmask);
    S2E_LAUNCH_CHECK();
    d_input_grad_aug_kernel<true, true><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, scratch, dfake,
                                                                  opmask);
  } else {
    d_input_grad_aug_kernel<false, true><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, nullptr, dfake,
                                                                   opmask);
  }
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_diffaug_draw_geom(int64_t* state, const double* p, int B, long long index_offset, int H, int W, float* params_out,
                          float* geom_out, int* opmask_out, void* stream) {
  S2E_REQUIRE(state && p && B >= 0 && H > 0 && W > 0 && index_offset >= 0, "diffaug_draw_geom: bad arguments");
  S2E_REQUIRE(index_offset + B <= (1LL << 32), "diffaug_draw_geom: sample indices must fit in 32 bits");
  S2E_REQUIRE(B == 0 || (params_out && geom_out && opmask_out), "diffaug_draw_geom: params_out / geom_out / opmask_out is null");
  diffaug_draw_kernel<true, true><<<1, 256, 0, (cudaStream_t)stream>>>((long long*)state, B, index_offset, H, W, params_out, p,
                                                                        opmask_out, geom_out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_make_d_input_aug_geom(const float* seg, const float* fake, const float* real, int B, int nc, int H, int W, int Cpad,
                              const float* params, const float* means, int policy, const int* opmask, const float* geom, void* out,
                              void* stream) {
  S2E_REQUIRE(Cpad > nc, "make_d_input_aug_geom: Cpad must exceed nc");
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL_GEOM) == 0, "make_d_input_aug_geom: unknown policy bits %#x", policy);
  S2E_REQUIRE(!(policy & S2E_DIFFAUG_GEOMETRIC) || (H >= 2 && W >= 2), "make_d_input_aug_geom: geometric needs H, W >= 2");
  S2E_REQUIRE(params && opmask && geom && (means || !(policy & S2E_DIFFAUG_COLOR)),
              "make_d_input_aug_geom: params / opmask / geom / means missing");
  const long long npix = 2LL * B * H * W;
  if (!npix) return S2E_OK;
  auto k = (policy & S2E_DIFFAUG_COLOR) ? make_d_input_aug_kernel<true, true, true> : make_d_input_aug_kernel<false, true, true>;
  k<<<grid1d(npix), NT, 0, (cudaStream_t)stream>>>(seg, fake, real, B, nc, H, W, Cpad, npix, params, means, policy, (bf16*)out, opmask,
                                                   geom);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_d_input_grad_aug_geom(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                              const int* opmask, const float* geom, double* scratch, float* dfake, void* stream) {
  S2E_REQUIRE((policy & ~S2E_DIFFAUG_ALL_GEOM) == 0, "d_input_grad_aug_geom: unknown policy bits %#x", policy);
  S2E_REQUIRE(!(policy & S2E_DIFFAUG_GEOMETRIC) || (H >= 2 && W >= 2), "d_input_grad_aug_geom: geometric needs H, W >= 2");
  S2E_REQUIRE(params && opmask && geom && (scratch || !(policy & S2E_DIFFAUG_COLOR)),
              "d_input_grad_aug_geom: params / opmask / geom / scratch missing");
  const long long n = (long long)B * H * W;
  if (!n) return S2E_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (policy & S2E_DIFFAUG_COLOR) {
    d_input_grad_aug_sum_kernel<true><<<B, 1024, 0, st>>>((const bf16*)dxin, nc, Cpad, H, W, params, policy, scratch, opmask);
    S2E_LAUNCH_CHECK();
    d_input_grad_aug_kernel<true, true, true><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, scratch,
                                                                        dfake, opmask, geom);
  } else {
    d_input_grad_aug_kernel<false, true, true><<<grid1d(n), NT, 0, st>>>((const bf16*)dxin, B, nc, Cpad, H, W, params, policy, nullptr,
                                                                         dfake, opmask, geom);
  }
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_ada_update(const double* step_stat, int num_D, double* acc, int* pos, double* p, double target, double kimg, int interval,
                   void* stream) {
  S2E_REQUIRE(step_stat && acc && pos && p && num_D >= 1 && interval >= 1 && kimg > 0.0, "ada_update: bad arguments");
  ada_update_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_stat, num_D, acc, pos, p, target, kimg, interval);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_tanh_fwd(const void* x, long long n, float* y, void* stream) {
  if (!n) return S2E_OK;
  tanh_fwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>((const bf16*)x, n, y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_tanh_bwd(const float* dy, const float* y, long long n, void* dx, void* stream) {
  if (!n) return S2E_OK;
  tanh_bwd_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(dy, y, n, (bf16*)dx);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_linear_fwd(const void* x, const float* w, const float* b, int M, int N, int K, int act, int in_nhwc_hw, float* y,
                   void* stream) {
  S2E_REQUIRE(in_nhwc_hw <= 0 || K % in_nhwc_hw == 0, "linear_fwd: K must be a multiple of hw");
  const long long threads = (long long)M * N * 32;
  if (!threads) return S2E_OK;
  linear_fwd_kernel<<<(unsigned)ceil_div_ll(threads, 256), 256, 0, (cudaStream_t)stream>>>(x, w, b, M, N, K, act, in_nhwc_hw, y);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_linear_bwd(const float* dy, const float* y, const void* x, const float* w, int M, int N, int K, int act,
                   int in_nhwc_hw, void* dx, float* dw, float* db, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (dx) {
    if (in_nhwc_hw <= 0 && K <= 32 && N >= 256)
      linear_bwd_dx_smallk_kernel<32><<<M, 256, 0, st>>>(dy, y, w, N, K, act, (float*)dx);
    else
      linear_bwd_dx_kernel<<<grid1d((long long)M * K), NT, 0, st>>>(dy, y, x, w, M, N, K, act, in_nhwc_hw, dx);
    S2E_LAUNCH_CHECK();
  }
  if (dw) {
    linear_bwd_dw_kernel<<<grid1d((long long)N * K), NT, 0, st>>>(dy, y, x, M, N, K, act, in_nhwc_hw, dw, db);
    S2E_LAUNCH_CHECK();
  }
  return S2E_OK;
}

int s2e_reduce_loss(const void* x, const void* y, long long n, int x_is_f32, int kind, float coef, float target, float* out,
                    int accumulate, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!accumulate) S2E_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float), st));
  if (!n) return S2E_OK;
  int g = grid1d(n, NT * 8);
  const int vec = !x_is_f32 && (((uintptr_t)x | (uintptr_t)y) & 15) == 0;
  reduce_loss_kernel<<<g, NT, 0, st>>>(x, y, n, x_is_f32, kind, coef, target, vec, out);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_reduce_loss_bwd(const void* x, const void* y, long long n, int x_is_f32, int kind, float coef, float target,
                        const float* gout, void* dx, int accumulate, void* stream) {
  if (!n) return S2E_OK;
  const int vec = !x_is_f32 && (((uintptr_t)x | (uintptr_t)y | (uintptr_t)dx) & 15) == 0;
  reduce_loss_bwd_kernel<<<grid1d(vec ? (n + 7) / 8 : n), NT, 0, (cudaStream_t)stream>>>(x, y, n, x_is_f32, kind, coef, target, vec, gout, dx,
                                                                                       accumulate);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_adam_prepare(float* state, float beta1, float beta2, void* stream) {
  adam_prepare_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state, beta1, beta2);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* state, float beta1, float beta2,
                  float eps, float weight_decay, void* stream) {
  if (!n) return S2E_OK;
  adam_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(p, g, m, v, n, state, beta1, beta2, eps, weight_decay);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}
int s2e_adam_multi(int n_tensors, float* const* p, const float* const* g, float* const* m, float* const* v,
                   const long long* n, const float* state, float beta1, float beta2, float eps, float weight_decay,
                   void* stream) {
  S2E_REQUIRE(n_tensors >= 0 && state, "adam_multi: bad arguments");
  for (int base = 0; base < n_tensors;) {
    AdamTable t;
    t.nt = 0;
    int blocks = 0;
    while (base < n_tensors && t.nt < ADAM_MAX_TENSORS) {
      if (n[base] > 0) {
        S2E_REQUIRE(p[base] && g[base] && m[base] && v[base], "adam_multi: tensor %d has a null pointer", base);
        const int k = t.nt++;
        t.p[k] = p[base];
        t.g[k] = g[base];
        t.m[k] = m[base];
        t.v[k] = v[base];
        t.n[k] = n[base];
        t.blk0[k] = blocks;
        blocks += (int)ceil_div_ll(n[base], ADAM_CHUNK);
      }
      ++base;
    }
    if (t.nt == 0) break;
    adam_multi_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(t, state, beta1, beta2, eps, weight_decay);
    S2E_LAUNCH_CHECK();
  }
  return S2E_OK;
}
int s2e_adam_multi_ema(int n_tensors, float* const* p, const float* const* g, float* const* m, float* const* v,
                       const long long* n, const float* state, float beta1, float beta2, float eps, float weight_decay,
                       float* const* ema, float ema_decay, void* stream) {
  S2E_REQUIRE(n_tensors >= 0 && state && ema, "adam_multi_ema: bad arguments");
  S2E_REQUIRE(ema_decay >= 0.f && ema_decay < 1.f, "adam_multi_ema: ema_decay %g is outside [0, 1)", (double)ema_decay);
  for (int base = 0; base < n_tensors;) {
    AdamEmaTable t;
    t.nt = 0;
    t.decay = ema_decay;
    int blocks = 0;
    while (base < n_tensors && t.nt < ADAM_MAX_TENSORS) {
      if (n[base] > 0) {
        S2E_REQUIRE(p[base] && g[base] && m[base] && v[base] && ema[base], "adam_multi_ema: tensor %d has a null pointer", base);
        const int k = t.nt++;
        t.p[k] = p[base];
        t.g[k] = g[base];
        t.m[k] = m[base];
        t.v[k] = v[base];
        t.e[k] = ema[base];
        t.n[k] = n[base];
        t.blk0[k] = blocks;
        blocks += (int)ceil_div_ll(n[base], ADAM_CHUNK);
      }
      ++base;
    }
    if (t.nt == 0) break;
    adam_multi_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(t, state, beta1, beta2, eps, weight_decay);
    S2E_LAUNCH_CHECK();
  }
  return S2E_OK;
}
int s2e_copy_multi(int n_rows, void* const* dst, const void* const* src, const long long* nbytes, void* stream) {
  S2E_REQUIRE(n_rows >= 0, "copy_multi: bad row count");
  for (int base = 0; base < n_rows;) {
    CopyTable t;
    t.nr = 0;
    int blocks = 0;
    while (base < n_rows && t.nr < COPY_MAX_ROWS) {
      if (nbytes[base] > 0) {
        S2E_REQUIRE(dst[base] && src[base], "copy_multi: row %d has a null pointer", base);
        const int k = t.nr++;
        t.dst[k] = dst[base];
        t.src[k] = src[base];
        t.nbytes[k] = nbytes[base];
        t.blk0[k] = blocks;
        blocks += (int)ceil_div_ll(nbytes[base], COPY_CHUNK);
      }
      ++base;
    }
    if (t.nr == 0) break;
    copy_multi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(t);
    S2E_LAUNCH_CHECK();
  }
  return S2E_OK;
}
int s2e_pack_weight_multi(const s2e_pack_job_t* jobs, int n_jobs, void* stream) {
  S2E_REQUIRE(n_jobs >= 0, "pack_weight_multi: bad job count");
  for (int base = 0; base < n_jobs; base += PACK_MAX_JOBS) {
    PackTable t;
    t.n = n_jobs - base < PACK_MAX_JOBS ? n_jobs - base : PACK_MAX_JOBS;
    int blocks = 0;
    for (int k = 0; k < t.n; ++k) {
      const s2e_pack_job_t& s = jobs[base + k];
      S2E_REQUIRE(s.w_oihw && s.out_bf16 && s.Cout > 0 && s.Cin > 0, "pack_weight_multi: job %d incomplete", base + k);
      PackJob& J = t.j[k];
      J.w = s.w_oihw;
      J.bias = s.im2col3x3 ? s.bias : nullptr;
      J.out = (bf16*)s.out_bf16;
      J.im2col = s.im2col3x3;
      J.transposed = s.transposed;
      if (s.im2col3x3) {
        S2E_REQUIRE(9 * s.Cin <= 62, "pack_weight_multi: im2col3x3 needs 9*C <= 62");
        J.g = make_pack_geom(s.Cout, s.Cin, 3, 3, 1, 1);
        J.transposed = 0;
      } else {
        S2E_REQUIRE(s.stride == 1 || s.stride == 2, "pack_weight_multi: stride must be 1 or 2");
        J.g = make_pack_geom(s.Cout, s.Cin, s.kh, s.kw, s.stride, s.pad, s.Cout_total, s.co_offset, s.cin_pad);
      }
      J.blk0 = blocks;
      blocks += (int)ceil_div_ll((long long)s.Cout * s.Cin, 256);
    }
    pack_weight_multi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(t);
    S2E_LAUNCH_CHECK();
  }
  return S2E_OK;
}
int s2e_fill_f32(float* p, long long n, float value, void* stream) {
  if (!n) return S2E_OK;
  fill_kernel<<<grid1d(n), NT, 0, (cudaStream_t)stream>>>(p, n, value);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

}  // extern "C"
