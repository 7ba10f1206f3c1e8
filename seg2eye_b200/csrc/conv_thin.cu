// "Thin" tap-convolutions: one side has only a handful of channels (the 4-class segmap, the 5-channel D input, the
// 1-channel image / PatchGAN logit).  These layers are < 1.5 % of the step's FLOPs but K or N is 1..36, so they are
// bandwidth-bound CUDA-core work, not tensor-core work (SURVEY 8(d)).  Same contract as s2e_tapconv_{fwd,wgrad}.
//   K1 thin input  : y[p][co]  = act(scale * sum_t sum_cs x[p+t][cs] W[t][co][cs] + b)      (mlp_shared, G.fc, D model0,
//                                                                                            E layer0, dgrad of conv_img/model4)
//   K2 thin output : y[p][cs]  = act(scale * sum_t sum_ci x[p+t][ci] W[t][cs][ci] + b)      (conv_img, D model4, dgrad of D model0)
//   K3 thin wgrad  : dW[t][co][ci] += sum_p dy[p][co] x[p+t][ci]  with either Cin or Cout thin
#include "common.cuh"

namespace {

struct ThinGeom {
  int B, Hi, Wi, Cin, Ho, Wo, Cout, ntaps, act, in_act;
  int dy[S2E_MAX_TAPS], dx[S2E_MAX_TAPS];
};

constexpr int K1_CO_TILE = 256;  // couts per block (weights staged in smem as float)

// ------------------------------------------------------------------------------------------------ K1
// thread = 8 couts x 4 consecutive output pixels of one row: each weight vector read from shared memory feeds four
// pixels (the kernel is FMA-bound instead of shared-memory-bound); coordinates are decoded once per quad.
constexpr int K1_PX = 4;
template <int CS4>  // CS4 = 1: Cin == 4 (one 8-byte load per pixel-tap); 0: generic Cin <= 32
__global__ void __launch_bounds__(256) thin_in_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                          const float* __restrict__ bias, const float* __restrict__ scale,
                                                          bf16* __restrict__ y, const ThinGeom g, int quads_per_row, long long nquads,
                                                          const bf16* __restrict__ mask, float mask_slope) {
  // mask (optional, shaped like y): where mask <= 0 the output is multiplied by mask_slope (fused [Leaky]ReLU backward)
  extern __shared__ float ws[];  // [T][Cs][cot]  (cot = couts of this block)
  const int co0 = blockIdx.y * K1_CO_TILE;
  const int cot = min(K1_CO_TILE, g.Cout - co0);
  const int Cs = g.Cin;
  for (int i = threadIdx.x; i < g.ntaps * Cs * cot; i += blockDim.x) {
    const int co = i % cot, r = i / cot, cs = r % Cs, t = r / Cs;
    ws[i] = __bfloat162float(wp[((long long)t * g.Cout + co0 + co) * Cs + cs]);
  }
  __syncthreads();
  const int ncog = cot >> 3;
  const float sc = scale ? __ldg(scale) : 1.f;
  const unsigned nwork = (unsigned)(nquads * ncog);   // host guarantees < 2^31
  for (unsigned v = blockIdx.x * blockDim.x + threadIdx.x; v < nwork; v += gridDim.x * blockDim.x) {
    const unsigned q = v / (unsigned)ncog;
    const int cog = (int)(v - q * ncog);
    const int qw = (int)(q % (unsigned)quads_per_row);
    const unsigned r = q / (unsigned)quads_per_row;
    const int ho = (int)(r % (unsigned)g.Ho);
    const int b = (int)(r / (unsigned)g.Ho);
    const int wo0 = qw * K1_PX;
    float acc[K1_PX][8];
#pragma unroll
    for (int i = 0; i < K1_PX; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int t = 0; t < g.ntaps; ++t) {
      const int hi = ho + g.dy[t];
      if (hi < 0 || hi >= g.Hi) continue;
      const bf16* xrow = x + ((long long)b * g.Hi + hi) * g.Wi * Cs;
      const float* wt = ws + (size_t)t * Cs * cot + cog * 8;
      const int wbase = wo0 + g.dx[t];
      if (CS4) {
        float xv[K1_PX][4];
#pragma unroll
        for (int i = 0; i < K1_PX; ++i) {
          const int wi = wbase + i;
          uint2 raw = make_uint2(0u, 0u);
          if (wi >= 0 && wi < g.Wi) raw = *reinterpret_cast<const uint2*>(xrow + (long long)wi * 4);
          const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
          const float2 c = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
          xv[i][0] = a.x; xv[i][1] = a.y; xv[i][2] = c.x; xv[i][3] = c.y;
        }
#pragma unroll
        for (int cs = 0; cs < 4; ++cs) {
          const float4 w0 = *reinterpret_cast<const float4*>(wt + (size_t)cs * cot);
          const float4 w1 = *reinterpret_cast<const float4*>(wt + (size_t)cs * cot + 4);
#pragma unroll
          for (int i = 0; i < K1_PX; ++i) {
            const float xx = xv[i][cs];
            acc[i][0] = fmaf(xx, w0.x, acc[i][0]); acc[i][1] = fmaf(xx, w0.y, acc[i][1]);
            acc[i][2] = fmaf(xx, w0.z, acc[i][2]); acc[i][3] = fmaf(xx, w0.w, acc[i][3]);
            acc[i][4] = fmaf(xx, w1.x, acc[i][4]); acc[i][5] = fmaf(xx, w1.y, acc[i][5]);
            acc[i][6] = fmaf(xx, w1.z, acc[i][6]); acc[i][7] = fmaf(xx, w1.w, acc[i][7]);
          }
        }
      } else {
        for (int cs = 0; cs < Cs; ++cs) {
          const float4 w0 = *reinterpret_cast<const float4*>(wt + (size_t)cs * cot);
          const float4 w1 = *reinterpret_cast<const float4*>(wt + (size_t)cs * cot + 4);
#pragma unroll
          for (int i = 0; i < K1_PX; ++i) {
            const int wi = wbase + i;
            const float xx = (wi >= 0 && wi < g.Wi) ? __bfloat162float(xrow[(long long)wi * Cs + cs]) : 0.f;
            acc[i][0] = fmaf(xx, w0.x, acc[i][0]); acc[i][1] = fmaf(xx, w0.y, acc[i][1]);
            acc[i][2] = fmaf(xx, w0.z, acc[i][2]); acc[i][3] = fmaf(xx, w0.w, acc[i][3]);
            acc[i][4] = fmaf(xx, w1.x, acc[i][4]); acc[i][5] = fmaf(xx, w1.y, acc[i][5]);
            acc[i][6] = fmaf(xx, w1.z, acc[i][6]); acc[i][7] = fmaf(xx, w1.w, acc[i][7]);
          }
        }
      }
    }
    const int cbase = co0 + cog * 8;
    float bv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bv[j] = bias ? __ldg(bias + cbase + j) : 0.f;
    bf16* yrow = y + (((long long)b * g.Ho + ho) * g.Wo) * g.Cout + cbase;
#pragma unroll
    for (int i = 0; i < K1_PX; ++i) {
      if (wo0 + i < g.Wo) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = act_apply(acc[i][j] * sc + bv[j], g.act);
        if (mask) {
          float mf[8];
          unpack8(ld_stream8(mask + (yrow - y) + (long long)(wo0 + i) * g.Cout), mf);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] *= (mf[j] > 0.f ? 1.f : mask_slope);
        }
        st_stream8(yrow + (long long)(wo0 + i) * g.Cout, pack8(o));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ K2
// LPP lanes cooperate on one output pixel, each owning 16-byte channel chunks of the wide input.
template <int CS_MAX>
__global__ void __launch_bounds__(256) thin_out_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                           const float* __restrict__ bias, const float* __restrict__ scale,
                                                           bf16* __restrict__ y, const ThinGeom g, long long P, int lpp) {
  extern __shared__ float ws[];  // [T][Cs][Cin]
  const int Cs = g.Cout, Cin = g.Cin;
  for (int i = threadIdx.x; i < g.ntaps * Cs * Cin; i += blockDim.x) ws[i] = __bfloat162float(wp[i]);
  __syncthreads();
  const int nchunk = Cin >> 3;
  const int sub = threadIdx.x % lpp;
  const unsigned gpix = (blockIdx.x * blockDim.x + threadIdx.x) / (unsigned)lpp;
  const unsigned gstride = gridDim.x * blockDim.x / (unsigned)lpp;
  const unsigned Pu = (unsigned)P, Pend = ((Pu + gstride - 1) / gstride) * gstride;   // host guarantees P < 2^31
  const float sc = scale ? __ldg(scale) : 1.f;
  for (unsigned p = gpix; p < Pend; p += gstride) {  // uniform trip count per warp
    const bool pv = p < Pu;
    unsigned pp = pv ? p : 0u;
    const int wo = (int)(pp % (unsigned)g.Wo);
    pp /= (unsigned)g.Wo;
    const int ho = (int)(pp % (unsigned)g.Ho);
    const int b = (int)(pp / (unsigned)g.Ho);
    float acc[CS_MAX];
#pragma unroll
    for (int c = 0; c < CS_MAX; ++c) acc[c] = 0.f;
    if (pv) {
      for (int t = 0; t < g.ntaps; ++t) {
        const int hi = ho + g.dy[t], wi = wo + g.dx[t];
        if (hi < 0 || hi >= g.Hi || wi < 0 || wi >= g.Wi) continue;
        const bf16* xp = x + (((long long)b * g.Hi + hi) * g.Wi + wi) * Cin;
        for (int ch = sub; ch < nchunk; ch += lpp) {
          float xf[8];
          unpack8(*reinterpret_cast<const bf16x8*>(xp + ch * 8), xf);
#pragma unroll
          for (int c = 0; c < CS_MAX; ++c) {
            if (c < Cs) {
              const float* wt = ws + ((size_t)t * Cs + c) * Cin + ch * 8;
              const float4 w0 = *reinterpret_cast<const float4*>(wt);
              const float4 w1 = *reinterpret_cast<const float4*>(wt + 4);
              acc[c] += xf[0] * w0.x + xf[1] * w0.y + xf[2] * w0.z + xf[3] * w0.w + xf[4] * w1.x + xf[5] * w1.y +
                        xf[6] * w1.z + xf[7] * w1.w;
            }
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < CS_MAX; ++c) {
      if (c < Cs) {
        float v = acc[c];
        for (int o = lpp >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (pv && sub == 0) y[(long long)p * Cs + c] = __float2bfloat16(act_apply(v * sc + (bias ? __ldg(bias + c) : 0.f), g.act));
      }
    }
  }
}

// K2 fast path for a single output channel (conv_img 64->1, PatchGAN head): lane = one 8-channel chunk of one pixel,
// its tap weights live in registers (TMAX*8 floats), LPP lanes are reduced with shuffles; a warp walks a contiguous
// range of output pixels with incrementally updated coordinates.
template <int TMAX, int LPP>
__global__ void __launch_bounds__(256) thin_out1_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                            const float* __restrict__ bias, const float* __restrict__ scale,
                                                            bf16* __restrict__ y, const ThinGeom g, long long P, long long pix_per_warp) {
  constexpr int PPW = 32 / LPP;  // pixels processed per warp iteration
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPP, slot = lane / LPP;
  const long long gwarp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  float wreg[TMAX][8];
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (t < g.ntaps) unpack8(*reinterpret_cast<const bf16x8*>(wp + (long long)t * g.Cin + sub * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) wreg[t][j] = f[j];
  }
  const float sc = scale ? __ldg(scale) : 1.f;
  const float bv = bias ? __ldg(bias) : 0.f;
  const long long p0 = gwarp * pix_per_warp;
  const long long p1 = min(P, p0 + pix_per_warp);
  if (p0 >= p1) return;
  // this lane's pixel coordinates, advanced by PPW pixels per iteration without divisions
  unsigned pp0 = (unsigned)min(p0 + slot, P - 1);
  int wo = (int)(pp0 % (unsigned)g.Wo);
  pp0 /= (unsigned)g.Wo;
  int ho = (int)(pp0 % (unsigned)g.Ho);
  int b = (int)(pp0 / (unsigned)g.Ho);
  for (long long pb = p0; pb < p1; pb += PPW) {
    const long long p = pb + slot;
    const bool pv = p < p1;
    // issue every tap's 16-byte load first (clamped address, validity folded into a 0/1 factor): no branches between
    // the loads, so all of them are in flight together
    bf16x8 xv[TMAX];
    float valid[TMAX];
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
      const int hi = ho + g.dy[t], wi = wo + g.dx[t];
      const bool ok = pv && t < g.ntaps && hi >= 0 && hi < g.Hi && wi >= 0 && wi < g.Wi;
      const int hc = min(max(hi, 0), g.Hi - 1), wc = min(max(wi, 0), g.Wi - 1), bc = min(b, g.B - 1);
      valid[t] = ok ? 1.f : 0.f;
      xv[t] = *reinterpret_cast<const bf16x8*>(x + (((long long)bc * g.Hi + hc) * g.Wi + wc) * g.Cin + sub * 8);
    }
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
      float xf[8], part = 0.f;
      unpack8(xv[t], xf);
#pragma unroll
      for (int j = 0; j < 8; ++j) part = fmaf(xf[j], wreg[t][j], part);
      acc = fmaf(part, valid[t], acc);
    }
#pragma unroll
    for (int o = LPP >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (pv && sub == 0) y[p] = __float2bfloat16(act_apply(acc * sc + bv, g.act));
    wo += PPW;
    while (wo >= g.Wo) {
      wo -= g.Wo;
      if (++ho == g.Ho) {
        ho = 0;
        ++b;
      }
    }
  }
}

// K2 tiled variant for conv_img (64 -> 1, 3x3, stride 1): every input pixel is read from global memory ONCE per tile
// (plus a one-pixel halo) instead of once per tap.  Phase 0: the whole halo tile is staged in shared memory with
// cp.async (every 16-byte chunk in flight at once; out-of-image pixels are zero-filled).  Phase 1: 8 lanes per input
// pixel form the nine per-tap dot products d[pixel][t] = x[pixel] . W[t] (tap weights in registers) and park them in
// shared memory.  Phase 2: one thread per output pixel adds its nine neighbours' entries
// y[p] = sum_t d[p + tap_t][t].
constexpr int T1_TW = 32, T1_TH = 8, T1_HW = T1_TW + 2, T1_NHP = (T1_TH + 2) * T1_HW;
constexpr int T1_MT = (T1_NHP + 15) / 16;      // 16-pixel row blocks of the halo tile (the last one is partly padding)
constexpr int T1_XP = 72;                      // pixel pitch of the staged tile in bf16: 144 bytes, so that the 16-byte fragment
                                               // loads of eight consecutive pixels fall into different banks
constexpr int T1_SMEM = T1_MT * 16 * T1_XP * 2 + T1_NHP * 9 * 4;

// ---- warp-level bf16 MMA (mma.sync m16n8k16, fp32 accumulate) for the single-image-channel layers.  These layers are GEMMs
// with N (or M, or K) = 9 taps: far too thin for a 128-row tcgen05 tile, and on the CUDA cores they were bound by instruction
// issue (ncu, round 2e: 352 M / 415 M / 439 M warp instructions for forward / data gradient / weight gradient of conv_img at
// B16 640x384, 0.44 / 0.59 / 0.70 ms against 0.1 - 0.2 ms of DRAM time).  One mma.sync replaces 128 FMAs + their unpacking.
// Fragment layout (PTX ISA, m16n8k16 .bf16): g = lane / 4, t = lane % 4;
//   A (16 x 16, row): a0 = (row g, k 2t..2t+1), a1 = (row g+8, same k), a2 = (row g, k 2t+8..2t+9), a3 = (row g+8, k 2t+8..)
//   B (16 x 8, col):  b0 = (k 2t..2t+1, col g), b1 = (k 2t+8..2t+9, col g);   C: c0,c1 = (row g, cols 2t, 2t+1), c2,c3 = (row g+8, ..)
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// max(v, 0) / min(v, 0) on a bf16 pair: leaky_relu(x) . w = max(x,0) . w + 0.2 * (min(x,0) . w) -- both operands exact in bf16,
// the factor 0.2 is applied to the fp32 accumulator (rounding 0.2 * x to bf16 first would cost 2^-9 on every negative input)
__device__ __forceinline__ uint32_t bf2_pos(uint32_t v) {
  const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&v), __float2bfloat162_rn(0.f));
  return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t bf2_neg(uint32_t v) {
  const __nv_bfloat162 r = __hmin2(*reinterpret_cast<const __nv_bfloat162*>(&v), __float2bfloat162_rn(0.f));
  return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t pack_bf16_bits(bf16 lo, bf16 hi) {
  return (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
}
__device__ __forceinline__ float in_act_slope(int in_act) { return in_act == S2E_ACT_LRELU ? 0.2f : 0.f; }

__global__ void __launch_bounds__(256, 3) thin_out1_tile_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                                const float* __restrict__ bias, const float* __restrict__ scale,
                                                                bf16* __restrict__ y, const ThinGeom g, int tiles_w, int tiles_h,
                                                                float* __restrict__ img_out, const float* __restrict__ img_target,
                                                                float* __restrict__ img_sums) {
  // img_out != NULL: the image head of the generator (generator.py:97-99): tanh is applied to the fp32 accumulator and the
  // result is written as fp32 (no bf16 rounding of the pre-activation); with img_target the block also adds its partial
  // sums of |fake - target| and (fake - target)^2 to img_sums[0..1] (the L1 / L2 image losses, pix2pix_model.py:197-208)
  extern __shared__ __align__(16) uint8_t t1_smem[];
  bf16* xs = reinterpret_cast<bf16*>(t1_smem);                               // [T1_MT * 16][T1_XP]  (64 channels + 16 bytes of padding)
  float* d = reinterpret_cast<float*>(t1_smem + T1_MT * 16 * T1_XP * 2);     // [T1_NHP][9]
  int tile = blockIdx.x;
  const int tw_idx = tile % tiles_w;
  tile /= tiles_w;
  const int th_idx = tile % tiles_h;
  const int b = tile / tiles_h;
  const int h0 = th_idx * T1_TH - 1, w0 = tw_idx * T1_TW - 1;
  const bf16* xb = x + (long long)b * g.Hi * g.Wi * 64;
  for (int i = threadIdx.x; i < T1_NHP * 8; i += 256) {
    const int hp = i >> 3, ch = i & 7;
    const int hh = hp / T1_HW, ww = hp - hh * T1_HW;
    const int hi = h0 + hh, wi = w0 + ww;
    const bool ok = hi >= 0 && hi < g.Hi && wi >= 0 && wi < g.Wi;
    const bf16* src = ok ? xb + ((long long)hi * g.Wi + wi) * 64 + ch * 8 : xb;
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(xs + hp * T1_XP + ch * 8);
    const int nbytes = ok ? 16 : 0;   // src-size 0 => the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  // Phase 1 as a GEMM on mma.sync: d[pixel][tap] = act(x[pixel]) . W[tap] with M = 16 halo pixels per row block, N = 16 taps
  // (two 8-wide halves, nine live), K = 64 channels (four steps).  Lane (g, t) reads the 32 bytes [16t, 16t+16) of pixels g and
  // g + 8 as its A fragments: k index 2t+e of step s is physical channel 16t + 4s + e, k index 8+2t+e is channel 16t + 4s + 2 + e
  // (any bijection works for a dot product, the B fragments below use the same one).
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  uint32_t wb[2][4][2];   // [tap half][k step][b0 | b1], loaded while the tile is in flight
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int tap = h * 8 + fg;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const bf16* wsrc = wp + (long long)tap * 64 + 16 * ft + 4 * ks;
      wb[h][ks][0] = tap < g.ntaps ? *reinterpret_cast<const uint32_t*>(wsrc) : 0u;
      wb[h][ks][1] = tap < g.ntaps ? *reinterpret_cast<const uint32_t*>(wsrc + 2) : 0u;
    }
  }
  const float nslope = in_act_slope(g.in_act);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  for (int mt = warp; mt < T1_MT; mt += 8) {
    const int rowA = mt * 16 + fg, rowB = rowA + 8;
    const uint4 xa0 = *reinterpret_cast<const uint4*>(xs + rowA * T1_XP + 16 * ft), xa1 = *reinterpret_cast<const uint4*>(xs + rowA * T1_XP + 16 * ft + 8);
    const uint4 xb0 = *reinterpret_cast<const uint4*>(xs + rowB * T1_XP + 16 * ft), xb1 = *reinterpret_cast<const uint4*>(xs + rowB * T1_XP + 16 * ft + 8);
    const uint32_t wa[8] = {xa0.x, xa0.y, xa0.z, xa0.w, xa1.x, xa1.y, xa1.z, xa1.w};
    const uint32_t wbw[8] = {xb0.x, xb0.y, xb0.z, xb0.w, xb1.x, xb1.y, xb1.z, xb1.w};
    float accp[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, accn[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t a0 = wa[2 * ks], a2 = wa[2 * ks + 1], a1 = wbw[2 * ks], a3 = wbw[2 * ks + 1];
      if (g.in_act == S2E_ACT_NONE) {
#pragma unroll
        for (int h = 0; h < 2; ++h) mma16816(accp[h], a0, a1, a2, a3, wb[h][ks][0], wb[h][ks][1]);
      } else {
        const uint32_t p0 = bf2_pos(a0), p1 = bf2_pos(a1), p2 = bf2_pos(a2), p3 = bf2_pos(a3);
#pragma unroll
        for (int h = 0; h < 2; ++h) mma16816(accp[h], p0, p1, p2, p3, wb[h][ks][0], wb[h][ks][1]);
        if (g.in_act == S2E_ACT_LRELU) {
          const uint32_t n0 = bf2_neg(a0), n1 = bf2_neg(a1), n2 = bf2_neg(a2), n3 = bf2_neg(a3);
#pragma unroll
          for (int h = 0; h < 2; ++h) mma16816(accn[h], n0, n1, n2, n3, wb[h][ks][0], wb[h][ks][1]);
        }
      }
    }
    // c0, c1 = (pixel rowA, taps 2t, 2t+1), c2, c3 = (pixel rowB, same taps); second half: tap 8 sits in column 0 (t == 0)
    if (rowA < T1_NHP) {
      d[rowA * 9 + 2 * ft] = fmaf(nslope, accn[0][0], accp[0][0]);
      d[rowA * 9 + 2 * ft + 1] = fmaf(nslope, accn[0][1], accp[0][1]);
      if (ft == 0) d[rowA * 9 + 8] = fmaf(nslope, accn[1][0], accp[1][0]);
    }
    if (rowB < T1_NHP) {
      d[rowB * 9 + 2 * ft] = fmaf(nslope, accn[0][2], accp[0][2]);
      d[rowB * 9 + 2 * ft + 1] = fmaf(nslope, accn[0][3], accp[0][3]);
      if (ft == 0) d[rowB * 9 + 8] = fmaf(nslope, accn[1][2], accp[1][2]);
    }
  }
  __syncthreads();
  const int th = threadIdx.x >> 5, tw = threadIdx.x & 31;
  const int ho = th_idx * T1_TH + th, wo = tw_idx * T1_TW + tw;
  float l1 = 0.f, l2 = 0.f;
  if (ho < g.Ho && wo < g.Wo) {
    float acc = 0.f;
    for (int t = 0; t < g.ntaps; ++t) acc += d[((th + 1 + g.dy[t]) * T1_HW + (tw + 1 + g.dx[t])) * 9 + t];
    const float sc = scale ? __ldg(scale) : 1.f;
    const float bv = bias ? __ldg(bias) : 0.f;
    const float v = act_apply(acc * sc + bv, g.act);
    const long long idx = ((long long)b * g.Ho + ho) * g.Wo + wo;
    if (img_out) {
      const float tv = tanhf(v);
      img_out[idx] = tv;
      if (img_target) {
        const float df = tv - __ldg(img_target + idx);
        l1 = fabsf(df);
        l2 = df * df;
      }
    } else {
      y[idx] = __float2bfloat16(v);
    }
  }
  if (img_out && img_target) {   // block-uniform branch
    __shared__ float red[2][8];
    l1 = warp_sum(l1);
    l2 = warp_sum(l2);
    if ((threadIdx.x & 31) == 0) {
      red[0][threadIdx.x >> 5] = l1;
      red[1][threadIdx.x >> 5] = l2;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
      atomicAdd(img_sums + threadIdx.x, t);
    }
  }
}

// ---- conv_img's data gradient (generator.py:97-99 backward): a 1 -> 64 channel tap convolution,
//   y[q][c] = m(q, c) * scale * sum_t x1[q + tap_t] * W[t][c],   m = 1 or mask_slope where the mask tensor is <= 0,
// as one mma.sync k-step per 16 pixels: A[pixel][tap] is gathered from a staged (TH+2) x (TW+2) tile of the one-channel
// input, B[tap][c] are the weights, and the logical column (n-tile j, col 2t+e) is physical channel 16t + 2j + e, so that a
// lane ends up with 16 CONTIGUOUS channels of pixels g and g + 8 (two 16-byte stores each, the mask read the same way).
constexpr int IG_TW = 32, IG_TH = 8, IG_PW = IG_TW + 2;
__global__ void __launch_bounds__(256) img_dgrad_mma_kernel(const bf16* __restrict__ x1, const bf16* __restrict__ wp,
                                                            const float* __restrict__ bias, const float* __restrict__ scale,
                                                            bf16* __restrict__ y, const ThinGeom g, int tiles_w, int tiles_h,
                                                            const bf16* __restrict__ mask, float mask_slope) {
  __shared__ bf16 xt[(IG_TH + 2) * IG_PW];
  int tile = blockIdx.x;
  const int tw_idx = tile % tiles_w;
  tile /= tiles_w;
  const int th_idx = tile % tiles_h;
  const int b = tile / tiles_h;
  const int h0 = th_idx * IG_TH, w0 = tw_idx * IG_TW;
  const bf16* xb = x1 + (long long)b * g.Hi * g.Wi;
  for (int i = threadIdx.x; i < (IG_TH + 2) * IG_PW; i += 256) {
    const int r = i / IG_PW, c = i - r * IG_PW;
    const int hi = h0 + r - 1, wi = w0 + c - 1;
    xt[i] = (hi >= 0 && hi < g.Hi && wi >= 0 && wi < g.Wi) ? xb[(long long)hi * g.Wi + wi] : __float2bfloat16(0.f);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  // B fragments: b0 = (taps 2t, 2t+1; column g), b1 = (taps 2t+8, 2t+9; column g); column g of n-tile j = channel 16(g/2) + 2j + (g&1)
  uint32_t wb[8][2];
  int off[3];   // staged-tile offsets of taps 2t, 2t+1 and 8 relative to the pixel itself
  {
    const int t0 = 2 * ft, t1 = 2 * ft + 1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = 16 * (fg >> 1) + 2 * j + (fg & 1);
      const bf16 z = __float2bfloat16(0.f);
      wb[j][0] = pack_bf16_bits(t0 < g.ntaps ? wp[t0 * 64 + ch] : z, t1 < g.ntaps ? wp[t1 * 64 + ch] : z);
      wb[j][1] = (ft == 0 && 8 < g.ntaps) ? pack_bf16_bits(wp[8 * 64 + ch], z) : 0u;
    }
    off[0] = t0 < g.ntaps ? g.dy[t0] * IG_PW + g.dx[t0] : 0;
    off[1] = t1 < g.ntaps ? g.dy[t1] * IG_PW + g.dx[t1] : 0;
    off[2] = 8 < g.ntaps ? g.dy[8] * IG_PW + g.dx[8] : 0;
  }
  const float sc = scale ? __ldg(scale) : 1.f;
  __syncthreads();
  // 16 row blocks of 16 pixels (tile row r = mt / 2, columns (mt & 1) * 16 ..): two per warp
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int mt = warp * 2 + it;
    const int r = mt >> 1, c0 = (mt & 1) * 16;
    const int pA = (r + 1) * IG_PW + c0 + fg + 1, pB = pA + 8;   // pixels g and g + 8 of the block, in the staged tile
    const uint32_t a0 = pack_bf16_bits(xt[pA + off[0]], xt[pA + off[1]]);
    const uint32_t a1 = pack_bf16_bits(xt[pB + off[0]], xt[pB + off[1]]);
    const uint32_t a2 = ft == 0 ? pack_bf16_bits(xt[pA + off[2]], __float2bfloat16(0.f)) : 0u;
    const uint32_t a3 = ft == 0 ? pack_bf16_bits(xt[pB + off[2]], __float2bfloat16(0.f)) : 0u;
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
      mma16816(acc[j], a0, a1, a2, a3, wb[j][0], wb[j][1]);
    }
    const int ho = h0 + r;
#pragma unroll
    for (int half = 0; half < 2; ++half) {   // pixel g (c0, c1 of every n-tile), then pixel g + 8 (c2, c3)
      const int wo = w0 + c0 + fg + 8 * half;
      if (ho >= g.Ho || wo >= g.Wo) continue;
      const long long pix = ((long long)b * g.Ho + ho) * g.Wo + wo;
      float o[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[2 * j] = acc[j][2 * half] * sc;
        o[2 * j + 1] = acc[j][2 * half + 1] * sc;
      }
      if (bias) {
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] += __ldg(bias + 16 * ft + e);
      }
#pragma unroll
      for (int e = 0; e < 16; ++e) o[e] = act_apply(o[e], g.act);
      if (mask) {
        float mf[16];
        unpack8(ld_stream8(mask + pix * 64 + 16 * ft), mf);
        unpack8(ld_stream8(mask + pix * 64 + 16 * ft + 8), mf + 8);
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] *= (mf[e] > 0.f ? 1.f : mask_slope);
      }
      st_stream8(y + pix * 64 + 16 * ft, pack8(o));
      st_stream8(y + pix * 64 + 16 * ft + 8, pack8(o + 8));
    }
  }
}

// ---- conv_img's weight gradient: dW[t][c] += sum_q act(x[q][c]) * dy1[q - tap_t]  (one output channel, 64 input channels) with
// M = 16 taps (nine live), N = 64 channels, K = pixels: per 16 consecutive pixels of a row one k-step.  A^T is gathered from a
// staged (TH+2) x (TW+2) tile of the one-channel gradient; for B a lane reads the 16 bytes [8g, 8g+8) of pixels 2t, 2t+1, 2t+8,
// 2t+9 (column g of n-tile j = channel 8g + j) and pairs the two pixels of a k pair with byte permutes.  Persistent blocks keep
// the 9 x 64 result in registers over all their tiles and reduce it once (shared-memory atomics, then one global atomic per value).
constexpr int IW_TW = 128, IW_TH = 8, IW_PW = IW_TW + 2;
__global__ void __launch_bounds__(256) img_wgrad_mma_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy1,
                                                            float* __restrict__ dwp, const ThinGeom g, int tiles_w, int tiles_h,
                                                            int num_tiles) {
  __shared__ bf16 dt[(IW_TH + 2) * IW_PW];
  __shared__ float red[9 * 64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  // staged-tile offsets: A^T[tap][pixel q] = dy1[q - tap]
  const int offg = fg < g.ntaps ? -(g.dy[fg] * IW_PW + g.dx[fg]) : 0;
  const int off8 = 8 < g.ntaps ? -(g.dy[8] * IW_PW + g.dx[8]) : 0;
  const bool live_g = fg < g.ntaps, live_8 = fg == 0 && 8 < g.ntaps;
  float accp[8][4], accn[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) accp[j][e] = accn[j][e] = 0.f;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    int tt = tile;
    const int tw_idx = tt % tiles_w;
    tt /= tiles_w;
    const int th_idx = tt % tiles_h;
    const int b = tt / tiles_h;
    const int h0 = th_idx * IW_TH, w0 = tw_idx * IW_TW;
    const bf16* db = dy1 + (long long)b * g.Ho * g.Wo;
    __syncthreads();   // the previous tile's fragments have been read
    for (int i = threadIdx.x; i < (IW_TH + 2) * IW_PW; i += 256) {
      const int r = i / IW_PW, c = i - r * IW_PW;
      const int ho = h0 + r - 1, wo = w0 + c - 1;
      dt[i] = (ho >= 0 && ho < g.Ho && wo >= 0 && wo < g.Wo) ? db[(long long)ho * g.Wo + wo] : __float2bfloat16(0.f);
    }
    __syncthreads();
    const int hi = h0 + warp;            // one tile row per warp
    if (hi >= g.Hi) continue;
    const bf16* xrow = x + (((long long)b * g.Hi + hi) * g.Wi) * 64 + 8 * fg;
#pragma unroll 2
    for (int kb = 0; kb < IW_TW / 16; ++kb) {
      const int c0 = kb * 16;
      if (w0 + c0 >= g.Wi) break;   // warp-uniform
      // B: pixels 2t, 2t+1, 2t+8, 2t+9 of this block, channels [8g, 8g+8)
      uint4 xv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int wi = w0 + c0 + 2 * ft + (i & 1) + 8 * (i >> 1);
        xv[i] = wi < g.Wi ? __ldg(reinterpret_cast<const uint4*>(xrow + (long long)wi * 64)) : make_uint4(0u, 0u, 0u, 0u);
      }
      // A^T: (tap g | tap 8; pixels 2t, 2t+1 | 2t+8, 2t+9)
      const int pq = (warp + 1) * IW_PW + c0 + 2 * ft + 1;
      const uint32_t a0 = live_g ? pack_bf16_bits(dt[pq + offg], dt[pq + 1 + offg]) : 0u;
      const uint32_t a2 = live_g ? pack_bf16_bits(dt[pq + 8 + offg], dt[pq + 9 + offg]) : 0u;
      const uint32_t a1 = live_8 ? pack_bf16_bits(dt[pq + off8], dt[pq + 1 + off8]) : 0u;
      const uint32_t a3 = live_8 ? pack_bf16_bits(dt[pq + 8 + off8], dt[pq + 9 + off8]) : 0u;
      const uint32_t w[4][4] = {{xv[0].x, xv[0].y, xv[0].z, xv[0].w}, {xv[1].x, xv[1].y, xv[1].z, xv[1].w},
                                {xv[2].x, xv[2].y, xv[2].z, xv[2].w}, {xv[3].x, xv[3].y, xv[3].z, xv[3].w}};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t sel = (j & 1) ? 0x7632u : 0x5410u;   // channel 8g + j of two pixels -> one k pair (low half = first pixel)
        const uint32_t b0 = __byte_perm(w[0][j >> 1], w[1][j >> 1], sel), b1 = __byte_perm(w[2][j >> 1], w[3][j >> 1], sel);
        if (g.in_act == S2E_ACT_NONE) {
          mma16816(accp[j], a0, a1, a2, a3, b0, b1);
        } else {
          mma16816(accp[j], a0, a1, a2, a3, bf2_pos(b0), bf2_pos(b1));
          if (g.in_act == S2E_ACT_LRELU) mma16816(accn[j], a0, a1, a2, a3, bf2_neg(b0), bf2_neg(b1));
        }
      }
    }
  }
  // c0, c1 = (tap g, columns 2t, 2t+1 of n-tile j = channels 8(2t) + j, 8(2t+1) + j); c2, c3 = the same for tap g + 8
  for (int i = threadIdx.x; i < 9 * 64; i += 256) red[i] = 0.f;
  __syncthreads();
  const float nslope = in_act_slope(g.in_act);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (live_g) {
      atomicAdd(&red[fg * 64 + 16 * ft + j], fmaf(nslope, accn[j][0], accp[j][0]));
      atomicAdd(&red[fg * 64 + 16 * ft + 8 + j], fmaf(nslope, accn[j][1], accp[j][1]));
    }
    if (live_8) {
      atomicAdd(&red[8 * 64 + 16 * ft + j], fmaf(nslope, accn[j][2], accp[j][2]));
      atomicAdd(&red[8 * 64 + 16 * ft + 8 + j], fmaf(nslope, accn[j][3], accp[j][3]));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < g.ntaps * 64; i += 256) atomicAdd(dwp + i, red[i]);
}

// PatchGAN logit head (discriminator.py:38: Cin = 8*ndf -> 1, 4x4, stride 1, pad 2; K = 8192) in "tap-channel" form:
//   y[p] = sum_t D[p + tap_t][t],   D[q][t] = x[q] . W[t]        (a 1x1 convolution Cin -> 16 tap channels + a gather)
// so the input is read ONCE, not once per tap.  head_dots_kernel forms D in fp32 on the CUDA cores (2 * 16 * Cin FLOPs per
// pixel: FMA-bound at ~30 us for B32 82x50x512, where zero-padding the single output channel to a 64-wide tensor-core tile
// moved 16 taps x the whole input through shared memory: 0.21 ms): one warp per four pixels, each lane owns NCH 8-channel
// chunks of the pixel (the pixel row is one coalesced read), tap weights come from shared memory as conflict-free
// 16-byte loads and feed four pixels; the 64 lane-partial sums are combined with a halving butterfly (62 shuffles, not 320).
// head_gather_kernel adds the taps' entries, scale, bias, activation.  Backward (ops.HeadConvFn): head_scatter_kernel builds
// G[q][t] = dy[q - tap_t] (64 channels, 16 live), and dx = G . W, dW = G^T . x are 1x1 convolutions on the tcgen05 kernels.
constexpr int HD_THREADS = 128;
template <int NCH>
__global__ void __launch_bounds__(HD_THREADS) head_dots_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                               float* __restrict__ D, int Cin, int ntaps, long long P) {
  extern __shared__ __align__(16) float hd_ws[];          // [16 taps][NCH][2 halves][32 lanes][4]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 16 * NCH * 256; i += HD_THREADS) {
    const int e = i & 3, l = (i >> 2) & 31, h = (i >> 7) & 1, r = i >> 8;
    const int ch = r % NCH, t = r / NCH;
    const int c = (ch * 32 + l) * 8 + h * 4 + e;
    hd_ws[i] = (t < ntaps && c < Cin) ? __bfloat162float(wp[(long long)t * Cin + c]) : 0.f;
  }
  __syncthreads();
  const long long ngroups = (P + 3) >> 2;
  for (long long grp = (long long)blockIdx.x * (HD_THREADS / 32) + warp; grp < ngroups; grp += (long long)gridDim.x * (HD_THREADS / 32)) {
    const long long p0 = grp << 2;
    float xf[4][NCH][8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        const int c0 = (ch * 32 + lane) * 8;
        uint4 raw = make_uint4(0u, 0u, 0u, 0u);
        if (p0 + i < P && c0 < Cin) raw = __ldg(reinterpret_cast<const uint4*>(x + (p0 + i) * Cin + c0));
        unpack8(*reinterpret_cast<const bf16x8*>(&raw), xf[i][ch]);
      }
    }
    float v[64];   // v[i * 16 + t]: this lane's share of pixel i, tap t
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      float w[NCH][8];
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        const float4 a = *reinterpret_cast<const float4*>(hd_ws + (((t * NCH + ch) * 2 + 0) * 32 + lane) * 4);
        const float4 c = *reinterpret_cast<const float4*>(hd_ws + (((t * NCH + ch) * 2 + 1) * 32 + lane) * 4);
        w[ch][0] = a.x; w[ch][1] = a.y; w[ch][2] = a.z; w[ch][3] = a.w;
        w[ch][4] = c.x; w[ch][5] = c.y; w[ch][6] = c.z; w[ch][7] = c.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = 0.f;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
          for (int j = 0; j < 8; ++j) a = fmaf(xf[i][ch][j], w[ch][j], a);
        v[i * 16 + t] = a;
      }
    }
    // halving butterfly: after the step with offset o a lane keeps the half of its values selected by its bit o
#pragma unroll
    for (int o = 16, cnt = 64; o >= 1; o >>= 1, cnt >>= 1) {
      const bool upper = (lane & o) != 0;
#pragma unroll
      for (int j = 0; j < cnt / 2; ++j) {
        const float lo = v[j], hi = v[j + cnt / 2];
        const float send = upper ? lo : hi, keep = upper ? hi : lo;
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
    }
    // lane holds values 2*lane, 2*lane + 1: pixel lane >> 3, taps (lane & 7) * 2 + {0, 1}
    const long long p = p0 + (lane >> 3);
    if (p < P) *reinterpret_cast<float2*>(D + p * 16 + (lane & 7) * 2) = make_float2(v[0], v[1]);
  }
}

// gan_sums (nullable, 6 floats, caller-zeroed): the GAN loss reductions over the logits ride in this kernel's epilogue -- the batch
// holds [fake ; real] (pix2pix_model.py:328-338), half h = (b >= half_b), and for each half the kernel adds
//   [3h + 0] += sum y,   [3h + 1] += sum min(y - 1, 0),   [3h + 2] += sum min(-y - 1, 0)      (y as rounded to bf16)
// i.e. the sums behind the hinge / Wasserstein terms of loss.py:58-83 (generator: -mean y_fake; discriminator: -mean min(y_real - 1, 0),
// -mean min(-y_fake - 1, 0)), so those losses need no pass of their own over the logits.
// SIGN (s2e_head_gather_signs): sign_sums[0] += sum sign(y) over the half b >= half_b as well (y as rounded to bf16, sign(0) = 0);
// a block's partial sums of +-1 are integers below 2^24, so the atomics add them exactly in any order
template <bool SIGN = false>
__global__ void __launch_bounds__(256) head_gather_kernel(const float* __restrict__ D, const float* __restrict__ bias,
                                                          const float* __restrict__ scale, bf16* __restrict__ y, const ThinGeom g,
                                                          long long P, float* __restrict__ gan_sums, int half_b,
                                                          float* __restrict__ sign_sums = nullptr) {
  const long long p = (long long)blockIdx.x * 256 + threadIdx.x;
  float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sg = 0.f;
  if (p < P) {
    const int wo = (int)(p % g.Wo);
    const long long r = p / g.Wo;
    const int ho = (int)(r % g.Ho);
    const long long b = r / g.Ho;
    float acc = 0.f;
    for (int t = 0; t < g.ntaps; ++t) {
      const int hi = ho + g.dy[t], wi = wo + g.dx[t];
      if (hi >= 0 && hi < g.Hi && wi >= 0 && wi < g.Wi) acc += __ldg(D + ((b * g.Hi + hi) * g.Wi + wi) * 16 + t);
    }
    const bf16 yb = __float2bfloat16(act_apply(acc * (scale ? __ldg(scale) : 1.f) + (bias ? __ldg(bias) : 0.f), g.act));
    y[p] = yb;
    if (gan_sums) {
      const float v = __bfloat162float(yb);
      const int h = b >= half_b ? 3 : 0;
#pragma unroll
      for (int k = 0; k < 6; ++k) s[k] = 0.f;
      const float t0 = v, t1 = fminf(v - 1.f, 0.f), t2 = fminf(-v - 1.f, 0.f);
      s[0] = h == 0 ? t0 : 0.f; s[1] = h == 0 ? t1 : 0.f; s[2] = h == 0 ? t2 : 0.f;
      s[3] = h == 3 ? t0 : 0.f; s[4] = h == 3 ? t1 : 0.f; s[5] = h == 3 ? t2 : 0.f;
    }
    if (SIGN && b >= half_b) {
      const float v = __bfloat162float(yb);
      sg = (float)((v > 0.f) - (v < 0.f));
    }
  }
  if (gan_sums) {   // kernel-uniform branch
    __shared__ float red[6][8];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const float w = warp_sum(s[k]);
      if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = w;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
      if (t != 0.f) atomicAdd(gan_sums + threadIdx.x, t);
    }
  }
  if (SIGN) {
    __shared__ float red_sg[8];
    const float w = warp_sum(sg);
    if ((threadIdx.x & 31) == 0) red_sg[threadIdx.x >> 5] = w;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red_sg[i];
      if (t != 0.f) atomicAdd(sign_sums, t);
    }
  }
}

// G[q][t] = dy[q - tap_t] for t < ntaps (zero where that output pixel does not exist), zero for the other 64 - ntaps
// channels; thread = one 8-channel chunk of one input pixel
__global__ void __launch_bounds__(256) head_scatter_kernel(const bf16* __restrict__ dy, bf16* __restrict__ G, const ThinGeom g,
                                                           long long nchunks) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= nchunks) return;
  const int ch = (int)(i & 7);
  const long long q = i >> 3;
  const int wi = (int)(q % g.Wi);
  const long long r = q / g.Wi;
  const int hi = (int)(r % g.Hi);
  const long long b = r / g.Hi;
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int t = ch * 8 + j;
    float v = 0.f;
    if (t < g.ntaps) {
      const int ho = hi - g.dy[t], wo = wi - g.dx[t];
      if (ho >= 0 && ho < g.Ho && wo >= 0 && wo < g.Wo) v = __bfloat162float(dy[(b * g.Ho + ho) * g.Wo + wo]);
    }
    f[j] = v;
  }
  *reinterpret_cast<bf16x8*>(G + i * 8) = pack8(f);
}

// ------------------------------------------------------------------------------------------------ K3
// wide tensor A [.., Cw] walked pixel by pixel, thin tensor S [.., Cs] sampled at (pixel + sgn*tap).
// thread = (8-channel chunk of A, one thin channel); acc[T][8] in registers; one atomic per output at the end.
//   thin_x = 1 : A = dy (Cout wide), S = x (Cin thin), S coord = p + tap,  out[t][cw][cs]
//   thin_x = 0 : A = x  (Cin wide),  S = dy (Cout thin), S coord = q - tap, out[t][cs][cw]
template <int TMAX, int MAXT>
__global__ void __launch_bounds__(MAXT) thin_wgrad_kernel(const bf16* __restrict__ A, const bf16* __restrict__ S, float* __restrict__ dwp,
                                                         int Bn, int HA, int WA, int Cw, int HS, int WS, int Cs, const ThinGeom g,
                                                         int thin_x, long long pix_per_block, int nth_pad, int pl_count) {
  // threads = pl_count pixel lanes x nth_pad (>= ncw*Cs, multiple of 32) channel slots; each pixel lane walks its own
  // contiguous slice of the block's pixel range so that small channel counts still fill the block
  const int ncw = Cw >> 3;
  const int slot = threadIdx.x % nth_pad, pl = threadIdx.x / nth_pad;
  const int cw = slot % ncw, cs = slot / ncw;
  const bool active = cs < Cs;
  const long long PA = (long long)Bn * HA * WA;
  const long long b0 = (long long)blockIdx.x * pix_per_block;
  const long long b1 = min(PA, b0 + pix_per_block);
  const long long per_lane = (b1 - b0 + pl_count - 1) / pl_count;
  const long long p0 = min(b1, b0 + (long long)pl * per_lane);
  const long long p1 = min(b1, p0 + per_lane);
  float acc[TMAX][8];
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.f;
  if (active && p0 < p1) {
    const int sgn = thin_x ? 1 : -1;
    int w = (int)(p0 % WA);
    long long r0 = p0 / WA;
    int h = (int)(r0 % HA);
    int b = (int)(r0 / HA);
    int tdy[TMAX], tdx[TMAX];
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
      tdy[t] = t < g.ntaps ? sgn * g.dy[t] : 0;
      tdx[t] = t < g.ntaps ? sgn * g.dx[t] : 0;
    }
    const bf16* ap = A + p0 * Cw + cw * 8;
    for (long long p = p0; p < p1; ++p, ap += Cw) {
      float a[8];
      unpack8(*reinterpret_cast<const bf16x8*>(ap), a);
      if (!thin_x && g.in_act != S2E_ACT_NONE) {   // A is the layer input x: activation applied on load
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = act_apply(a[j], g.in_act);
      }
      const bf16* sb = S + ((long long)b * HS * WS) * Cs + cs;
      float sv[TMAX];
#pragma unroll
      for (int t = 0; t < TMAX; ++t) {   // clamped, branch-free loads: all taps in flight together
        const int hs = h + tdy[t], wss = w + tdx[t];
        const bool ok = t < g.ntaps && hs >= 0 && hs < HS && wss >= 0 && wss < WS;
        const int hc = min(max(hs, 0), HS - 1), wc = min(max(wss, 0), WS - 1);
        float v = __bfloat162float(sb[((long long)hc * WS + wc) * Cs]);
        if (thin_x) v = act_apply(v, g.in_act);      // S is the layer input x
        sv[t] = ok ? v : 0.f;
      }
#pragma unroll
      for (int t = 0; t < TMAX; ++t) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[t][j] = fmaf(a[j], sv[t], acc[t][j]);
      }
      if (++w == WA) {
        w = 0;
        if (++h == HA) {
          h = 0;
          ++b;
        }
      }
    }
  }
  // combine the pixel lanes of the block (lanes that share a warp by shuffles, the rest through shared memory), then
  // one atomic per output element per block
  extern __shared__ float red[];  // [rows][nth_pad] per (t, j) pass
  const bool sub_warp = nth_pad < 32;                      // host guarantees 32 % nth_pad == 0 in that case
  const int rows = sub_warp ? (int)(blockDim.x >> 5) : pl_count;
  const int my_row = sub_warp ? (int)(threadIdx.x >> 5) : pl;
  const bool writer = sub_warp ? (int)(threadIdx.x & 31) < nth_pad : true;
  for (int t = 0; t < g.ntaps; ++t) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = 0.f;
#pragma unroll
      for (int tt = 0; tt < TMAX; ++tt)
        if (tt == t) v = acc[tt][j];
      if (sub_warp)
        for (int o = nth_pad; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      __syncthreads();
      if (writer) red[my_row * nth_pad + slot] = v;
      __syncthreads();
      if (pl == 0 && active) {
        float sum = 0.f;
        for (int l = 0; l < rows; ++l) sum += red[l * nth_pad + slot];
        const int c = cw * 8 + j;
        const long long o = thin_x ? ((long long)t * Cw + c) * Cs + cs : ((long long)t * Cs + cs) * Cw + c;
        atomicAdd(dwp + o, sum);
      }
    }
  }
}

// function attributes are per device: remember which devices were configured (one process may drive several GPUs)
bool first_use_on_device(int* mask) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return true;
  const int bit = 1 << (dev & 31);
  if (*mask & bit) return false;
  *mask |= bit;
  return true;
}

ThinGeom make_thin_geom(const s2e_conv_t* d) {
  ThinGeom g;
  g.B = d->B;
  g.Hi = d->Hi;
  g.Wi = d->Wi;
  g.Cin = d->Cin;
  g.Ho = d->Ho;
  g.Wo = d->Wo;
  g.Cout = d->Cout;
  g.ntaps = d->ntaps;
  g.act = d->act;
  g.in_act = d->in_act;
  for (int i = 0; i < d->ntaps; ++i) {
    g.dy[i] = d->tap_dy[i];
    g.dx[i] = d->tap_dx[i];
  }
  return g;
}

}  // namespace

// returns 1 if handled, 0 if the shape is not "thin", < 0 on error
int s2e_thin_fwd(const s2e_conv_t* d, const void* x, const void* wp, const float* bias, const float* scale, void* y,
                 cudaStream_t stream) {
  const long long P = (long long)d->B * d->Ho * d->Wo;
  if (P == 0) return 1;
  if (P * 32 >= (1LL << 31)) return 0;  // 32-bit index math inside the thin kernels
  ThinGeom g = make_thin_geom(d);
  const bf16* mask = (const bf16*)d->relu_mask;
  // input activation: tiled conv_img kernel only; output mask: thin-input kernel only -- everything else declines
  const bool tile_ok = d->Cout == 1 && d->Cin == 64 && d->ntaps <= 9 && d->Hi == d->Ho && d->Wi == d->Wo;
  if ((d->in_act != S2E_ACT_NONE || d->img_out) && !tile_ok) return 0;
  if (mask && !(d->Cin <= 32 && d->Cout % 8 == 0 && d->Cout >= 8)) return 0;
  bool halo1 = d->ntaps <= 9 && d->Hi == d->Ho && d->Wi == d->Wo;
  for (int t = 0; t < d->ntaps && halo1; ++t) halo1 = d->tap_dy[t] >= -1 && d->tap_dy[t] <= 1 && d->tap_dx[t] >= -1 && d->tap_dx[t] <= 1;
  if (d->Cin == 1 && d->Cout == 64 && halo1 && !s2e_debug_get(7)) {   // conv_img's data gradient: one mma.sync k-step per 16 pixels
    const int tiles_w = ceil_div(d->Wo, IG_TW), tiles_h = ceil_div(d->Ho, IG_TH);
    img_dgrad_mma_kernel<<<(unsigned)(d->B * tiles_h * tiles_w), 256, 0, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g,
                                                                              tiles_w, tiles_h, mask, d->mask_slope);
    S2E_LAUNCH_CHECK();
    return 1;
  }
  if (d->Cin <= 32 && d->Cout % 8 == 0 && d->Cout >= 8) {
    const int cot = d->Cout < K1_CO_TILE ? d->Cout : K1_CO_TILE;
    if (d->Cout % K1_CO_TILE != 0 && d->Cout > K1_CO_TILE) return 0;
    const size_t smem = (size_t)d->ntaps * d->Cin * cot * sizeof(float);
    if (smem > 200 * 1024) return 0;
    static int attr = 0;
    if (first_use_on_device(&attr)) {
      S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_in_fwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_in_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    const int qpr = ceil_div(d->Wo, K1_PX);
    const long long nquads = (long long)d->B * d->Ho * qpr;
    long long work = nquads * (cot / 8);
    long long gx = (work + 255) / 256;
    const long long cap = (long long)s2e_num_sms() * 8;
    if (gx > cap) gx = cap;
    dim3 grid((unsigned)gx, (unsigned)ceil_div(d->Cout, K1_CO_TILE));
    if (d->Cin == 4)
      thin_in_fwd_kernel<1><<<grid, 256, smem, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g, qpr, nquads, mask,
                                                       d->mask_slope);
    else
      thin_in_fwd_kernel<0><<<grid, 256, smem, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g, qpr, nquads, mask,
                                                       d->mask_slope);
    S2E_LAUNCH_CHECK();
    return 1;
  }
  if (d->Cout == 1 && d->Cin == 64 && d->ntaps <= 9 && d->Hi == d->Ho && d->Wi == d->Wo) {
    if (halo1) {
      const int tiles_w = ceil_div(d->Wo, T1_TW), tiles_h = ceil_div(d->Ho, T1_TH);
      static int attr1 = 0;
      if (first_use_on_device(&attr1)) {
        S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_out1_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T1_SMEM));
      }
      thin_out1_tile_kernel<<<(unsigned)(d->B * tiles_h * tiles_w), 256, T1_SMEM, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale,
                                                                                   (bf16*)y, g, tiles_w, tiles_h, d->img_out,
                                                                                   d->img_target, d->img_sums);
      S2E_LAUNCH_CHECK();
      return 1;
    }
  }
  if (d->in_act != S2E_ACT_NONE || d->img_out) return 0;
  if (d->Cout == 1 && d->Cin == 64 && d->ntaps <= 9) {
    const long long warps = (long long)s2e_num_sms() * 32;
    long long ppw = (P + warps - 1) / warps;
    ppw = ((ppw + 3) / 4) * 4;
    if (ppw < 4) ppw = 4;
    const long long nwarps = (P + ppw - 1) / ppw;
    thin_out1_fwd_kernel<9, 8><<<(unsigned)((nwarps * 32 + 255) / 256), 256, 0, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale,
                                                                                        (bf16*)y, g, P, ppw);
    S2E_LAUNCH_CHECK();
    return 1;
  }
  if (d->Cout <= 32 && d->Cin % 8 == 0 && d->Cin >= 8) {
    const size_t smem = (size_t)d->ntaps * d->Cout * d->Cin * sizeof(float);
    if (smem > 200 * 1024) return 0;
    int lpp = 1;
    while (lpp < 32 && lpp * 2 <= d->Cin / 8) lpp *= 2;
    long long gx = (P * lpp + 255) / 256;
    const long long cap = (long long)s2e_num_sms() * 8;
    if (gx > cap) gx = cap;
    static int attr = 0;
    if (first_use_on_device(&attr)) {
      S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_out_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_out_fwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S2E_CHECK_CUDA(cudaFuncSetAttribute(thin_out_fwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    if (d->Cout == 1)
      thin_out_fwd_kernel<1><<<(unsigned)gx, 256, smem, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g, P, lpp);
    else if (d->Cout <= 8)
      thin_out_fwd_kernel<8><<<(unsigned)gx, 256, smem, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g, P, lpp);
    else
      thin_out_fwd_kernel<32><<<(unsigned)gx, 256, smem, stream>>>((const bf16*)x, (const bf16*)wp, bias, scale, (bf16*)y, g, P, lpp);
    S2E_LAUNCH_CHECK();
    return 1;
  }
  return 0;
}

int s2e_thin_wgrad(const s2e_conv_t* d, const void* x, const void* dy, float* dwp, cudaStream_t stream) {
  ThinGeom g = make_thin_geom(d);
  int thin_x;
  if (d->Cin <= 32 && d->Cout % 8 == 0 && (d->Cout / 8) * d->Cin <= 512)
    thin_x = 1;
  else if (d->Cout <= 32 && d->Cin % 8 == 0 && (d->Cin / 8) * d->Cout <= 512)
    thin_x = 0;
  else
    return 0;
  if (d->ntaps > 16) return 0;
  if (!thin_x && d->Cout == 1 && d->Cin == 64 && d->ntaps <= 9 && d->Hi == d->Ho && d->Wi == d->Wo && !s2e_debug_get(7)) {
    bool halo1 = true;
    for (int t = 0; t < d->ntaps; ++t) halo1 = halo1 && d->tap_dy[t] >= -1 && d->tap_dy[t] <= 1 && d->tap_dx[t] >= -1 && d->tap_dx[t] <= 1;
    if (halo1) {   // conv_img's weight gradient on mma.sync
      const int tiles_w = ceil_div(d->Wi, IW_TW), tiles_h = ceil_div(d->Hi, IW_TH);
      const int num_tiles = d->B * tiles_h * tiles_w;
      if (num_tiles == 0) return 1;
      const int grid = num_tiles < 2 * s2e_num_sms() ? num_tiles : 2 * s2e_num_sms();
      img_wgrad_mma_kernel<<<grid, 256, 0, stream>>>((const bf16*)x, (const bf16*)dy, dwp, g, tiles_w, tiles_h, num_tiles);
      S2E_LAUNCH_CHECK();
      return 1;
    }
  }
  const bf16* A = thin_x ? (const bf16*)dy : (const bf16*)x;
  const bf16* S = thin_x ? (const bf16*)x : (const bf16*)dy;
  const int HA = thin_x ? d->Ho : d->Hi, WA = thin_x ? d->Wo : d->Wi, Cw = thin_x ? d->Cout : d->Cin;
  const int HS = thin_x ? d->Hi : d->Ho, WS = thin_x ? d->Wi : d->Wo, Cs = thin_x ? d->Cin : d->Cout;
  const long long PA = (long long)d->B * HA * WA;
  if (PA == 0) return 1;
  // channel slots per pixel lane: exact when they tile a warp (conv_img's weight gradient: 8 slots -> 4 pixel lanes per
  // warp, no idle lanes), otherwise padded to whole warps
  int nth_pad = (Cw / 8) * Cs;
  if (32 % nth_pad != 0) nth_pad = ((nth_pad + 31) / 32) * 32;
  int pl = 256 / nth_pad;
  if (pl < 1) pl = 1;
  if (d->ntaps > 9 && pl * nth_pad > 128) pl = 128 / nth_pad > 0 ? 128 / nth_pad : 1;
  const int threads = pl * nth_pad;
  long long blocks = (long long)s2e_num_sms() * (threads <= 128 ? 8 : (threads <= 256 ? 4 : 2));
  long long ppb = (PA + blocks - 1) / blocks;
  if (ppb < 64LL * pl) ppb = 64LL * pl;
  blocks = (PA + ppb - 1) / ppb;
  const size_t red_bytes = (size_t)threads * sizeof(float);
  if (d->ntaps <= 4)
    thin_wgrad_kernel<4, 512><<<(unsigned)blocks, threads, red_bytes, stream>>>(A, S, dwp, d->B, HA, WA, Cw, HS, WS, Cs, g, thin_x, ppb, nth_pad, pl);
  else if (d->ntaps <= 9)
    thin_wgrad_kernel<9, 512><<<(unsigned)blocks, threads, red_bytes, stream>>>(A, S, dwp, d->B, HA, WA, Cw, HS, WS, Cs, g, thin_x, ppb, nth_pad, pl);
  else if (threads <= 128)
    thin_wgrad_kernel<16, 128><<<(unsigned)blocks, threads, red_bytes, stream>>>(A, S, dwp, d->B, HA, WA, Cw, HS, WS, Cs, g, thin_x, ppb, nth_pad, pl);
  else
    return 0;
  S2E_LAUNCH_CHECK();
  return 1;
}

extern "C" {

int s2e_head_dots(const void* x, const void* wp, long long P, int Cin, int ntaps, float* D, void* stream) {
  S2E_REQUIRE(Cin % 8 == 0 && Cin >= 8 && Cin <= 1024 && ntaps >= 1 && ntaps <= 16, "head_dots: Cin %% 8 == 0, <= 1024, <= 16 taps (Cin=%d taps=%d)", Cin, ntaps);
  if (P == 0) return S2E_OK;
  const int nch = ceil_div(Cin, 256);
  static int attr = 0;
  if (first_use_on_device(&attr)) {
    S2E_CHECK_CUDA(cudaFuncSetAttribute(head_dots_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 4 * 256 * 4));
  }
  long long blocks = ceil_div_ll((P + 3) / 4, HD_THREADS / 32);
  const long long cap = (long long)s2e_num_sms() * 3;      // three resident CTAs per SM (registers): weights are staged once per CTA
  if (blocks > cap) blocks = cap;
  cudaStream_t st = (cudaStream_t)stream;
  if (nch == 1) head_dots_kernel<1><<<(unsigned)blocks, HD_THREADS, 16 * 1 * 256 * 4, st>>>((const bf16*)x, (const bf16*)wp, D, Cin, ntaps, P);
  else if (nch == 2) head_dots_kernel<2><<<(unsigned)blocks, HD_THREADS, 16 * 2 * 256 * 4, st>>>((const bf16*)x, (const bf16*)wp, D, Cin, ntaps, P);
  else head_dots_kernel<4><<<(unsigned)blocks, HD_THREADS, 16 * 4 * 256 * 4, st>>>((const bf16*)x, (const bf16*)wp, D, Cin, ntaps, P);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_head_gather(const s2e_conv_t* d, const float* D, const float* bias, const float* scale, void* y, float* gan_sums, void* stream) {
  S2E_REQUIRE(d && d->Cout == 1 && d->ntaps >= 1 && d->ntaps <= 16, "head_gather: one output channel, <= 16 taps");
  S2E_REQUIRE(!gan_sums || d->B % 2 == 0, "head_gather: the GAN sums need a [fake ; real] batch (B = %d)", d->B);
  const long long P = (long long)d->B * d->Ho * d->Wo;
  if (P == 0) return S2E_OK;
  head_gather_kernel<<<(unsigned)ceil_div_ll(P, 256), 256, 0, (cudaStream_t)stream>>>(D, bias, scale, (bf16*)y, make_thin_geom(d), P, gan_sums,
                                                                                      d->B / 2);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_head_gather_signs(const s2e_conv_t* d, const float* D, const float* bias, const float* scale, void* y, float* gan_sums,
                          float* sign_sums, void* stream) {
  S2E_REQUIRE(d && d->Cout == 1 && d->ntaps >= 1 && d->ntaps <= 16, "head_gather_signs: one output channel, <= 16 taps");
  S2E_REQUIRE(sign_sums && d->B % 2 == 0, "head_gather_signs: the sign sum needs a [fake ; real] batch (B = %d) and a slot", d->B);
  const long long P = (long long)d->B * d->Ho * d->Wo;
  S2E_REQUIRE(P / 2 < (1LL << 24), "head_gather_signs: %lld real-half logits; the fp32 sign sum is exact below 2^24", P / 2);
  if (P == 0) return S2E_OK;
  head_gather_kernel<true><<<(unsigned)ceil_div_ll(P, 256), 256, 0, (cudaStream_t)stream>>>(D, bias, scale, (bf16*)y, make_thin_geom(d), P,
                                                                                            gan_sums, d->B / 2, sign_sums);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

int s2e_head_scatter(const s2e_conv_t* d, const void* dy, void* G, void* stream) {
  S2E_REQUIRE(d && d->Cout == 1 && d->ntaps >= 1 && d->ntaps <= 16, "head_scatter: one output channel, <= 16 taps");
  const long long n = (long long)d->B * d->Hi * d->Wi * 8;
  if (n == 0) return S2E_OK;
  head_scatter_kernel<<<(unsigned)ceil_div_ll(n, 256), 256, 0, (cudaStream_t)stream>>>((const bf16*)dy, (bf16*)G, make_thin_geom(d), n);
  S2E_LAUNCH_CHECK();
  return S2E_OK;
}

}  // extern "C"
