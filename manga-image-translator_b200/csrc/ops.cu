// HBM-bound helper kernels: LayerNorm, fused depthwise-7x7 + LayerNorm, pooling, layout / dtype conversion,
// the LaMa input pack / MPE add / final blend, and the small OCR attention core.
// All operate on NHWC views (channel slice of a wider tensor) with 128-bit accesses along C where aligned.
#include <cuda_bf16.h>
#include <string.h>
#include <stdlib.h>
#include "mitb_internal.h"

namespace mitb {

// fp32 -> bf16 hi / mid operand pair of the tensor-core convs (x ~ hi + mid), same rounding as split4 in tc_common.cuh
__device__ __forceinline__ void split1_bf16(float v, uint16_t& hi, uint16_t& mid) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi = __bfloat16_as_ushort(h);
  mid = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(h)));
}
__device__ __forceinline__ void split4_bf16(const float4 v, uint2& hi, uint2& mid) {
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
  const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&h0), b1 = *reinterpret_cast<const uint32_t*>(&h1);
  const __nv_bfloat162 m0 = __floats2bfloat162_rn(v.x - __uint_as_float(b0 << 16), v.y - __uint_as_float(b0 & 0xffff0000u));
  const __nv_bfloat162 m1 = __floats2bfloat162_rn(v.z - __uint_as_float(b1 << 16), v.w - __uint_as_float(b1 & 0xffff0000u));
  hi = make_uint2(b0, b1);
  mid = make_uint2(*reinterpret_cast<const uint32_t*>(&m0), *reinterpret_cast<const uint32_t*>(&m1));
}

#define LAUNCH_END() do { count_launch(); CUDA_OK(cudaGetLastError()); } while (0)

// ---------------------------------------------------------------------------------------------------
// LayerNorm over C for every pixel (row).  One warp per row, two-pass (mean, then centred variance) in
// registers, C <= 1024 and C % 32 == 0.  Optionally also writes out2 = out + pe[row % T] (the OCR encoder adds
// the positional encoding to q/k only, model_48px_ctc.py:263-266).
template <int PER_LANE>
__global__ void layernorm_kernel(const float* in, int in_cs, int in_coff, float* out, int out_cs, int out_coff,
                                 const float* w, const float* b, float eps, long rows, int C, const float* pe,
                                 float* out2, int out2_cs, int out2_coff, int T, uint16_t* o_hi, uint16_t* o_mid) {
  const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* src = in + row * in_cs + in_coff;
  float v[PER_LANE];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) { int c = lane + 32 * i; v[i] = c < C ? src[c] : 0.f; s += v[i]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) { int c = lane + 32 * i; float d = c < C ? v[i] - mean : 0.f; q += d * d; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / C + eps);
  float* dst = out + row * out_cs + out_coff;
  float* dst2 = out2 ? out2 + row * out2_cs + out2_coff : nullptr;
  const float* per = pe ? pe + (size_t)(row % T) * C : nullptr;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) {
    int c = lane + 32 * i;
    if (c < C) {
      float y = (v[i] - mean) * rstd * w[c] + b[c];
      if (o_hi) { uint16_t hh, mm; split1_bf16(y, hh, mm); o_hi[row * C + c] = hh; o_mid[row * C + c] = mm; }   // consumer conv's operands
      else dst[c] = y;
      if (dst2) dst2[c] = y + per[c];
    }
  }
}

void launch_layernorm(const View& in, const View& out, const float* w, const float* b, float eps, const float* pe,
                      const View* out2, int T, cudaStream_t st, const SplitView* osv) {
  MITB_CHECK(!in.planar && !out.planar, "layernorm expects NHWC views");
  const int C = in.C; const long rows = (long)in.pixels();
  MITB_CHECK(C <= 1024 && out.C == C, "layernorm: C=%d unsupported", C);
  uint16_t* ohi = nullptr; uint16_t* omid = nullptr;
  if (osv && osv->valid()) {
    MITB_CHECK(osv->C == C && osv->Hp == osv->H && osv->Wp == osv->W && (long)osv->N * osv->H * osv->W == rows, "layernorm: split output mismatch");
    ohi = osv->hi; omid = osv->mid;
  }
  const int per = (C + 31) / 32;
  dim3 grid((unsigned)((rows + 7) / 8));
  ProfScope ps("layernorm", 8.0 * rows * C, 8.0 * rows * C, st);
  float* o2 = out2 ? out2->p : nullptr; int o2cs = out2 ? out2->cs : 0, o2off = out2 ? out2->coff : 0;
#define LN_CASE(P) layernorm_kernel<P><<<grid, 256, 0, st>>>(in.p, in.cs, in.coff, out.p, out.cs, out.coff, w, b, eps, rows, C, pe, o2, o2cs, o2off, T, ohi, omid)
  if (per <= 4) LN_CASE(4); else if (per <= 8) LN_CASE(8); else if (per <= 10) LN_CASE(10);
  else if (per <= 16) LN_CASE(16); else LN_CASE(32);
#undef LN_CASE
  LAUNCH_END();
}

// ---------------------------------------------------------------------------------------------------
// ConvNeXt token mixer: depthwise 7x7 (pad 3, bias) immediately followed by LayerNorm over C
// (dbnet_convnext.py:114-122).  blockDim = (C/4, PY): a thread owns 4 channels (one float4) of TX=8 consecutive
// output pixels of one row; the C/4 threads with the same threadIdx.y jointly normalise those 8 pixels.
constexpr int DW_TX = 8;

// ncu (r02, C = 512): the first version of this kernel was bound by instruction issue, not by memory - 31 M warp instructions
// for 9.6 M warp-FMAs: 64-bit address arithmetic and a bounds predicate per input pixel, scalar FMAs.  This version keeps the same
// tiling (same summation order per output: bias, then taps in (dy, dx) order) but runs the taps on the packed fp32x2 pipe (two
// channels per instruction), addresses the input with 32-bit element offsets from one base pointer, and takes a predicate-free
// path for tiles that do not touch the left / right image border (CTA-uniform).
__device__ __forceinline__ void dw_taps(float2 (&acc)[DW_TX][2], const float4 v, const float2 (&wv)[7][2], int j) {
  const float2 lo = make_float2(v.x, v.y), hi = make_float2(v.z, v.w);
#pragma unroll
  for (int dx = 0; dx < 7; ++dx) {
    const int i = j - dx;                    // output pixel fed by input pixel j through tap dx (resolved at compile time)
    if (i >= 0 && i < DW_TX) {
      acc[i][0] = __ffma2_rn(lo, wv[dx][0], acc[i][0]);
      acc[i][1] = __ffma2_rn(hi, wv[dx][1], acc[i][1]);
    }
  }
}

template <int WROW>                  // warps per pixel row = C / 128
__global__ void __launch_bounds__(256, 2) dwconv7_ln_kernel(const float* __restrict__ in, int in_cs, int in_coff, float* __restrict__ out,
                                                            int out_cs, int out_coff, const float* __restrict__ wdw,
                                                            const float* __restrict__ bdw, const float* __restrict__ lnw,
                                                            const float* __restrict__ lnb, float eps, int N, int H, int W, int C,
                                                            uint16_t* __restrict__ o_hi, uint16_t* __restrict__ o_mid) {
  extern __shared__ float red[];                 // [PY][nwarps_per_row][DW_TX]
  const int c = threadIdx.x * 4;
  const int xt = blockIdx.x * DW_TX;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int n = blockIdx.z;
  const bool row_ok = y < H;
  float2 acc[DW_TX][2];
  {
    const float4 bias = __ldg(reinterpret_cast<const float4*>(bdw + c));
#pragma unroll
    for (int i = 0; i < DW_TX; ++i) { acc[i][0] = make_float2(bias.x, bias.y); acc[i][1] = make_float2(bias.z, bias.w); }
  }
  if (row_ok) {
    const bool interior = xt >= 3 && xt + DW_TX + 3 <= W;      // CTA-uniform: no input pixel of this tile is left / right of the image
    const unsigned ucs = (unsigned)in_cs;
    for (int dy = 0; dy < 7; ++dy) {
      const int iy = y + dy - 3;
      if (iy < 0 || iy >= H) continue;
      float2 wv[7][2];
#pragma unroll
      for (int dx = 0; dx < 7; ++dx) {
        const float4 w4 = __ldg(reinterpret_cast<const float4*>(wdw + (unsigned)(dy * 7 + dx) * (unsigned)C + (unsigned)c));
        wv[dx][0] = make_float2(w4.x, w4.y); wv[dx][1] = make_float2(w4.z, w4.w);
      }
      if (interior) {
        const float* rowp = in + ((unsigned)((n * H + iy) * W + xt - 3) * ucs + (unsigned)(in_coff + c));       // host checked: < 2^31 elements
#pragma unroll
        for (int j = 0; j < DW_TX + 6; ++j) dw_taps(acc, __ldg(reinterpret_cast<const float4*>(rowp + (unsigned)j * ucs)), wv, j);
      } else {
        const float* rowp = in + ((unsigned)((n * H + iy) * W) * ucs + (unsigned)(in_coff + c));
#pragma unroll
        for (int j = 0; j < DW_TX + 6; ++j) {
          const int ix = xt + j - 3;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ix >= 0 && ix < W) v = __ldg(reinterpret_cast<const float4*>(rowp + (unsigned)ix * ucs));
          dw_taps(acc, v, wv, j);
        }
      }
    }
  }
  // ---- LayerNorm over C across the threadIdx.x dimension (two-pass: mean, then centred variance).  The eight per-pixel partial
  // sums of a warp are reduced together by a transposed butterfly (9 shuffles instead of 40): after the xor-16/8/4 steps each lane
  // holds ONE pixel's partial (pixel = lane bits 4,3,2), two more steps finish it; lanes with (lane & 3) == 0 publish it.
  const int lane = (threadIdx.y * blockDim.x + threadIdx.x) & 31;
  const int warp_in_row = threadIdx.x >> 5;
  float* myred = red + (size_t)threadIdx.y * WROW * DW_TX;
  float mean[DW_TX], rstd[DW_TX];
  for (int pass = 0; pass < 2; ++pass) {
    float part[DW_TX];
#pragma unroll
    for (int i = 0; i < DW_TX; ++i) {
      if (pass == 0) part[i] = (acc[i][0].x + acc[i][0].y) + (acc[i][1].x + acc[i][1].y);
      else {
        const float a = acc[i][0].x - mean[i], b = acc[i][0].y - mean[i], cc = acc[i][1].x - mean[i], d = acc[i][1].y - mean[i];
        part[i] = (a * a + b * b) + (cc * cc + d * d);
      }
    }
    {
      const bool u16 = lane & 16, u8 = lane & 8, u4 = lane & 4;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float keep = u16 ? part[i + 4] : part[i], give = u16 ? part[i] : part[i + 4];
        part[i] = keep + __shfl_xor_sync(0xffffffffu, give, 16);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float keep = u8 ? part[i + 2] : part[i], give = u8 ? part[i] : part[i + 2];
        part[i] = keep + __shfl_xor_sync(0xffffffffu, give, 8);
      }
      {
        const float keep = u4 ? part[1] : part[0], give = u4 ? part[0] : part[1];
        part[0] = keep + __shfl_xor_sync(0xffffffffu, give, 4);
      }
      part[0] += __shfl_xor_sync(0xffffffffu, part[0], 2);
      part[0] += __shfl_xor_sync(0xffffffffu, part[0], 1);
    }
    __syncthreads();                                           // (pass 1: everyone has read the pass-0 totals)
    if ((lane & 3) == 0) myred[warp_in_row * DW_TX + (lane >> 2)] = part[0];      // pixel index = (bit4, bit3, bit2) = lane >> 2
    __syncthreads();
#pragma unroll
    for (int i = 0; i < DW_TX; ++i) {
      float t = 0.f;
#pragma unroll
      for (int wv = 0; wv < WROW; ++wv) t += myred[wv * DW_TX + i];
      if (pass == 0) mean[i] = t / C; else rstd[i] = rsqrtf(t / C + eps);
    }
  }
  if (!row_ok) return;
  const float4 g = __ldg(reinterpret_cast<const float4*>(lnw + c)), be = __ldg(reinterpret_cast<const float4*>(lnb + c));
  const unsigned opix0 = (unsigned)((n * H + y) * W);
#pragma unroll
  for (int i = 0; i < DW_TX; ++i) {
    const int x = xt + i;
    if (x < W) {
      float4 r;
      r.x = (acc[i][0].x - mean[i]) * rstd[i] * g.x + be.x; r.y = (acc[i][0].y - mean[i]) * rstd[i] * g.y + be.y;
      r.z = (acc[i][1].x - mean[i]) * rstd[i] * g.z + be.z; r.w = (acc[i][1].y - mean[i]) * rstd[i] * g.w + be.w;
      if (o_hi) {                       // the only consumer is the fc1 GEMM: store its bf16 hi / mid operands, dense [pixel][C]
        uint2 hh, mm; split4_bf16(r, hh, mm);
        const unsigned o = (opix0 + (unsigned)x) * (unsigned)C + (unsigned)c;
        *reinterpret_cast<uint2*>(o_hi + o) = hh; *reinterpret_cast<uint2*>(o_mid + o) = mm;
      } else *reinterpret_cast<float4*>(out + ((opix0 + (unsigned)x) * (unsigned)out_cs + (unsigned)(out_coff + c))) = r;
    }
  }
}

void launch_dwconv7_ln(const View& in, const View& out, const float* wdw, const float* bdw, const float* lnw,
                       const float* lnb, float eps, cudaStream_t st, const SplitView* osv) {
  const int C = in.C;
  uint16_t* ohi = nullptr; uint16_t* omid = nullptr;
  if (osv && osv->valid()) {
    MITB_CHECK(osv->C == C && osv->N == in.N && osv->H == in.H && osv->W == in.W && osv->Hp == in.H && osv->Wp == in.W, "dwconv7_ln: split output mismatch");
    ohi = osv->hi; omid = osv->mid;
  }
  MITB_CHECK(C % 128 == 0 && C <= 1024, "dwconv7_ln: C=%d must be a multiple of 128 (<=1024)", C);
  MITB_CHECK(in.cs % 4 == 0 && in.coff % 4 == 0 && out.cs % 4 == 0 && out.coff % 4 == 0, "dwconv7_ln alignment");
  MITB_CHECK((size_t)in.pixels() * (size_t)(in.cs > out.cs ? in.cs : out.cs) < ((size_t)1 << 31) && (size_t)in.pixels() * C < ((size_t)1 << 31),
             "dwconv7_ln: tensor too large for 32-bit element offsets");
  ProfScope ps("dwconv7_ln", (98.0 + 8.0) * in.pixels() * C, 8.0 * in.pixels() * C + 4.0 * 51 * C, st);
  const int tx = C / 4;
  int py = 256 / tx; if (py < 1) py = 1;
  dim3 block(tx, py), grid((in.W + DW_TX - 1) / DW_TX, (in.H + py - 1) / py, in.N);
  const size_t smem = (size_t)py * (tx / 32) * DW_TX * sizeof(float);
#define DW_CASE(R) dwconv7_ln_kernel<R><<<grid, block, smem, st>>>(in.p, in.cs, in.coff, out.p, out.cs, out.coff, wdw, bdw, lnw, lnb, eps, \
                                                                   in.N, in.H, in.W, C, ohi, omid)
  switch (tx / 32) {
    case 1: DW_CASE(1); break;
    case 2: DW_CASE(2); break;
    case 4: DW_CASE(4); break;
    case 8: DW_CASE(8); break;
    default: MITB_CHECK(false, "dwconv7_ln: C=%d (supported: 128, 256, 512, 1024)", C);
  }
#undef DW_CASE
  LAUNCH_END();
}

// ---------------------------------------------------------------------------------------------------
// AvgPool2d: mode 0 = kernel 2 stride 2; mode 1 = kernel 2, stride (2,1), padding (0,1), count_include_pad
// (model_48px_ctc.py:289,295,301) -> out width W+1, zero columns averaged in.
__global__ void avgpool_kernel(const float* in, int in_cs, int in_coff, float* out, int out_cs, int out_coff, int N,
                               int H, int W, int C4, int Ho, int Wo, int mode) {
  const long total = (long)N * Ho * Wo * C4;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4) * 4; long r = i / C4;
    const int ox = (int)(r % Wo); r /= Wo; const int oy = (int)(r % Ho); const int n = (int)(r / Ho);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int iy = oy * 2 + dy;
        const int ix = mode == 0 ? ox * 2 + dx : ox - 1 + dx;
        if (ix >= 0 && ix < W && iy < H) {
          float4 v = __ldg(reinterpret_cast<const float4*>(in + ((size_t)(n * H + iy) * W + ix) * in_cs + in_coff + c));
          s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
      }
    s.x *= 0.25f; s.y *= 0.25f; s.z *= 0.25f; s.w *= 0.25f;
    *reinterpret_cast<float4*>(out + ((size_t)(n * Ho + oy) * Wo + ox) * out_cs + out_coff + c) = s;
  }
}

void launch_avgpool(const View& in, const View& out, int mode, cudaStream_t st) {
  MITB_CHECK(in.C % 4 == 0 && in.cs % 4 == 0 && in.coff % 4 == 0 && out.cs % 4 == 0 && out.coff % 4 == 0, "avgpool alignment");
  const long total = (long)out.N * out.H * out.W * (in.C / 4);
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  avgpool_kernel<<<blocks, 256, 0, st>>>(in.p, in.cs, in.coff, out.p, out.cs, out.coff, in.N, in.H, in.W, in.C / 4,
                                         out.H, out.W, mode);
  LAUNCH_END();
}

// ---------------------------------------------------------------------------------------------------
// layout conversions.  NCHW -> NHWC view (missing channels of the view are zero-filled, e.g. RGB -> 4 channels).
__global__ void nchw_to_nhwc_kernel(const float* src, int N, int C, int H, int W, float* dst, int cs, int coff, int Cv) {
  const long total = (long)N * H * W;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i % ((long)H * W); const int n = (int)(i / ((long)H * W));
    for (int c = 0; c < Cv; ++c)
      dst[i * cs + coff + c] = c < C ? src[((size_t)n * C + c) * H * W + pix] : 0.f;
  }
}
void launch_nchw_to_nhwc(const float* src, int N, int C, int H, int W, const View& dst, cudaStream_t st) {
  const long total = (long)N * H * W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  nchw_to_nhwc_kernel<<<blocks, 256, 0, st>>>(src, N, C, H, W, dst.p, dst.cs, dst.coff, dst.C);
  LAUNCH_END();
}

__global__ void nhwc_to_nchw_kernel(const float* src, int cs, int coff, int N, int C, int H, int W, float* dst) {
  const long total = (long)N * C * H * W;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i % ((long)H * W); long r = i / ((long)H * W); const int c = (int)(r % C); const int n = (int)(r / C);
    dst[i] = src[((size_t)n * H * W + pix) * cs + coff + c];
  }
}
void launch_nhwc_to_nchw(const View& src, float* dst, cudaStream_t st) {
  const long total = (long)src.N * src.C * src.H * src.W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  nhwc_to_nchw_kernel<<<blocks, 256, 0, st>>>(src.p, src.cs, src.coff, src.N, src.C, src.H, src.W, dst);
  LAUNCH_END();
}

// uint8 NHWC image -> fp32 NHWC view with the reference's normalisation:
//   div_first=1: x/127.5 - 1.0   (numpy fp32, dbnet_convnext.py:503: divide, then subtract)
//   div_first=0: (x - 127.5)/127.5 (model_48px_ctc.py:101: subtract, then divide)
__global__ void u8_to_nhwc_kernel(const uint8_t* src, long npix, int C, float* dst, int cs, int coff, int Cv, float mul,
                                  float add, int div_first) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < npix; i += (long)gridDim.x * blockDim.x) {
    for (int c = 0; c < Cv; ++c) {
      float v = 0.f;
      if (c < C) {
        const float x = (float)src[i * C + c];
        v = div_first ? __fsub_rn(__fdiv_rn(x, mul), add) : __fdiv_rn(__fsub_rn(x, add), mul);
      }
      dst[i * cs + coff + c] = v;
    }
  }
}
void launch_u8_to_nhwc(const uint8_t* src, int N, int H, int W, int C, const View& dst, float mul, float add,
                       int div_first, cudaStream_t st) {
  const long npix = (long)N * H * W;
  int blocks = (int)((npix + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  u8_to_nhwc_kernel<<<blocks, 256, 0, st>>>(src, npix, C, dst.p, dst.cs, dst.coff, dst.C, mul, add, div_first);
  LAUNCH_END();
}

__device__ __forceinline__ float act_apply(float v, int act) {
  switch (act) {
    case ACT_RELU: return fmaxf(v, 0.f);
    case ACT_GELU: return 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));
    case ACT_SILU: return v / (1.f + expf(-v));
    case ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    default: return v;
  }
}
__global__ void affine_act_kernel(const float* in, int in_cs, int in_coff, float* out, int out_cs, int out_coff, long npix,
                                  int C, const float* scale, const float* shift, int act) {
  const long total = npix * C;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C); const long pix = i / C;
    float v = in[pix * in_cs + in_coff + c];
    if (scale) v = v * scale[c] + shift[c];
    out[pix * out_cs + out_coff + c] = act_apply(v, act);
  }
}
void launch_affine_act(const View& in, const View& out, const float* scale, const float* shift, int act, cudaStream_t st) {
  const long total = (long)in.pixels() * in.C;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  affine_act_kernel<<<blocks, 256, 0, st>>>(in.p, in.cs, in.coff, out.p, out.cs, out.coff, (long)in.pixels(), in.C, scale, shift, act);
  LAUNCH_END();
}

// ---------------------------------------------------------------------------------------------------
// OCR self-attention core (model_48px_ctc.py:263-269 -> F.multi_head_attention_forward): one CTA per
// (line, head); K and V of that head staged in shared memory (stride hd+1), one warp per query row,
// softmax(q.k / sqrt(hd)) v with no padding mask.
// gridDim.y row blocks per (line, head): each CTA re-stages K/V (L2 resident) and takes every gridDim.y-th group of query rows,
// so the 128 (line, head) pairs of a 16-line chunk fill all 148 SMs several CTAs deep instead of 128 SMs one CTA deep.
__global__ void attention_kernel(const float* qk, const float* v, float* out, int T, int heads, int hd, float scale) {
  extern __shared__ float sm[];
  const int D = heads * hd;
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int ld = hd + 1;
  float* Ks = sm; float* Vs = Ks + (size_t)T * ld;
  float* Ps = Vs + (size_t)T * ld;               // [nwarps][T] probabilities
  float* Qs = Ps + (size_t)(blockDim.x >> 5) * T; // [nwarps][hd]
  for (int i = threadIdx.x; i < T * hd; i += blockDim.x) {
    const int t = i / hd, d = i % hd;
    Ks[t * ld + d] = qk[((size_t)n * T + t) * 2 * D + D + h * hd + d];
    Vs[t * ld + d] = v[((size_t)n * T + t) * D + h * hd + d];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float* P = Ps + (size_t)warp * T; float* Q = Qs + warp * hd;
  for (int t = blockIdx.y * nw + warp; t < T; t += nw * gridDim.y) {
    for (int d = lane; d < hd; d += 32) Q[d] = qk[((size_t)n * T + t) * 2 * D + h * hd + d];
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < T; j += 32) {
      float s = 0.f;
      for (int d = 0; d < hd; ++d) s = fmaf(Q[d], Ks[j * ld + d], s);
      s *= scale; P[j] = s; mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) { float e = expf(P[j] - mx); P[j] = e; sum += e; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    __syncwarp();
    const float inv = 1.f / sum;
    for (int d = lane; d < hd; d += 32) {
      float a = 0.f;
      for (int j = 0; j < T; ++j) a = fmaf(P[j], Vs[j * ld + d], a);
      out[((size_t)n * T + t) * D + h * hd + d] = a * inv;
    }
    __syncwarp();
  }
}

// head_dim = 40 (the OCR encoder, model_48px_ctc.py:432): same decomposition, restructured for instruction count - the generic kernel
// above spends two shared-memory loads per FMA.  K / V rows are padded to 44 floats so that a row is ten aligned LDS.128 (conflict
// free per quarter warp), q lives in registers, the dot products and the P.V accumulation run on the packed fp32x2 pipe, and P.V is
// split over the keys (each lane accumulates its own keys into 40 registers, the 32 partial vectors are summed through shared memory).
constexpr int AT_HD = 40, AT_LD = 44;
__global__ void __launch_bounds__(256) attention40_kernel(const float* __restrict__ qk, const float* __restrict__ v, float* __restrict__ out, int T,
                                                          int heads, float scale) {
  extern __shared__ __align__(16) float sm[];
  const int D = heads * AT_HD;
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ks = sm; float* Vs = Ks + (size_t)T * AT_LD;
  float* Ps = Vs + (size_t)T * AT_LD;                       // [nw][T]
  float* Ob = Ps + (((size_t)nw * T + 3) & ~(size_t)3);     // [nw][32][AT_LD] partial outputs
  for (int i = threadIdx.x; i < T * (AT_HD / 4); i += blockDim.x) {
    const int t = i / (AT_HD / 4), d4 = i % (AT_HD / 4);
    *reinterpret_cast<float4*>(Ks + t * AT_LD + 4 * d4) = __ldg(reinterpret_cast<const float4*>(qk + ((size_t)n * T + t) * 2 * D + D + h * AT_HD) + d4);
    *reinterpret_cast<float4*>(Vs + t * AT_LD + 4 * d4) = __ldg(reinterpret_cast<const float4*>(v + ((size_t)n * T + t) * D + h * AT_HD) + d4);
  }
  __syncthreads();
  float* P = Ps + (size_t)warp * T;
  float* O = Ob + (size_t)warp * 32 * AT_LD;
  for (int t = blockIdx.y * nw + warp; t < T; t += nw * gridDim.y) {
    float2 q[AT_HD / 2];
    {
      const float4* qp = reinterpret_cast<const float4*>(qk + ((size_t)n * T + t) * 2 * D + h * AT_HD);
#pragma unroll
      for (int i = 0; i < AT_HD / 4; ++i) { const float4 a = __ldg(qp + i); q[2 * i] = make_float2(a.x, a.y); q[2 * i + 1] = make_float2(a.z, a.w); }
    }
    float mx = -INFINITY;
    for (int j = lane; j < T; j += 32) {
      const float4* kr = reinterpret_cast<const float4*>(Ks + j * AT_LD);
      float2 s2 = make_float2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < AT_HD / 4; ++i) {
        const float4 a = kr[i];
        s2 = __ffma2_rn(q[2 * i], make_float2(a.x, a.y), s2);
        s2 = __ffma2_rn(q[2 * i + 1], make_float2(a.z, a.w), s2);
      }
      const float s = (s2.x + s2.y) * scale;
      P[j] = s; mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    float2 acc[AT_HD / 2];
#pragma unroll
    for (int i = 0; i < AT_HD / 2; ++i) acc[i] = make_float2(0.f, 0.f);
    for (int j = lane; j < T; j += 32) {                       // this lane's keys: it wrote P[j] itself, no exchange needed yet
      const float e = expf(P[j] - mx);
      sum += e;
      const float4* vr = reinterpret_cast<const float4*>(Vs + j * AT_LD);
#pragma unroll
      for (int i = 0; i < AT_HD / 4; ++i) {
        const float4 a = vr[i];
        acc[2 * i] = __ffma2_rn(make_float2(e, e), make_float2(a.x, a.y), acc[2 * i]);
        acc[2 * i + 1] = __ffma2_rn(make_float2(e, e), make_float2(a.z, a.w), acc[2 * i + 1]);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
#pragma unroll
    for (int i = 0; i < AT_HD / 4; ++i)
      *reinterpret_cast<float4*>(O + lane * AT_LD + 4 * i) = make_float4(acc[2 * i].x, acc[2 * i].y, acc[2 * i + 1].x, acc[2 * i + 1].y);
    __syncwarp();
    const float inv = 1.f / sum;
    for (int d = lane; d < AT_HD; d += 32) {
      float a = 0.f;
#pragma unroll 8
      for (int l = 0; l < 32; ++l) a += O[l * AT_LD + d];
      out[((size_t)n * T + t) * D + h * AT_HD + d] = a * inv;
    }
    __syncwarp();
  }
}

// Sequences whose whole K / V does not fit in shared memory (the OCR reads lines up to T = 2048, the rows of its positional-encoding
// table): K / V of the head stream through shared memory in chunks of AS_TK keys under an online softmax.  Per query row a running max
// m and sum l; when a chunk raises the max, l and the output accumulators are rescaled by exp(m_old - m_new).  Each warp owns AS_R
// consecutive query rows (a CTA covers nw * AS_R rows and streams K / V once for all of them); lane j scores key j of each 32-key group,
// output dimension d lives in lane d % 32, register d / 32.  4-byte loads only, so any alignment; head_dim <= 32 * AS_HDR.
constexpr int AS_TK = 64, AS_R = 4, AS_HDR = 2;
__global__ void __launch_bounds__(256) attention_stream_kernel(const float* __restrict__ qk, const float* __restrict__ v, float* __restrict__ out,
                                                               int T, int heads, int hd, float scale) {
  extern __shared__ float sm[];
  const int D = heads * hd, ld = hd + 1;
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ks = sm; float* Vs = Ks + AS_TK * ld;
  float* Q = Vs + AS_TK * ld + (size_t)warp * AS_R * hd;   // [nw][AS_R][hd]
  const int row0 = (blockIdx.y * nw + warp) * AS_R;
  for (int i = lane; i < AS_R * hd; i += 32) {
    const int t = row0 + i / hd;
    Q[i] = t < T ? qk[((size_t)n * T + t) * 2 * D + h * hd + i % hd] : 0.f;
  }
  float m[AS_R], l[AS_R], acc[AS_R][AS_HDR];
#pragma unroll
  for (int r = 0; r < AS_R; ++r) {
    m[r] = -INFINITY; l[r] = 0.f;
#pragma unroll
    for (int i = 0; i < AS_HDR; ++i) acc[r][i] = 0.f;
  }
  for (int k0 = 0; k0 < T; k0 += AS_TK) {
    const int nk = min(AS_TK, T - k0);
    __syncthreads();                                           // the previous chunk is consumed (and, the first time, Q is staged)
    for (int i = threadIdx.x; i < nk * hd; i += blockDim.x) {
      const int j = i / hd, d = i % hd;
      const size_t row = (size_t)n * T + k0 + j;
      Ks[j * ld + d] = qk[row * 2 * D + D + h * hd + d];
      Vs[j * ld + d] = v[row * D + h * hd + d];
    }
    __syncthreads();
    for (int j0 = 0; j0 < nk; j0 += 32) {
      const int j = j0 + lane;
      float s[AS_R];
#pragma unroll
      for (int r = 0; r < AS_R; ++r) s[r] = 0.f;
      if (j < nk) {
        for (int d = 0; d < hd; ++d) {
          const float kd = Ks[j * ld + d];
#pragma unroll
          for (int r = 0; r < AS_R; ++r) s[r] = fmaf(Q[r * hd + d], kd, s[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < AS_R; ++r) {
        const float sr = j < nk ? s[r] * scale : -INFINITY;
        float cm = sr;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, o));
        const float mn = fmaxf(m[r], cm);                      // finite: lane 0 always holds a key of this group
        const float c = expf(m[r] - mn);                       // 0 on the first group (m = -inf)
        s[r] = expf(sr - mn);                                  // 0 for the lanes past the last key
        l[r] = fmaf(l[r], c, s[r]);                            // per-lane partial sum, reduced at the end
#pragma unroll
        for (int i = 0; i < AS_HDR; ++i) acc[r][i] *= c;
        m[r] = mn;
      }
      const int kn = min(32, nk - j0);
      for (int jj = 0; jj < kn; ++jj) {
        const float* vr = Vs + (j0 + jj) * ld;
        float vd[AS_HDR];
#pragma unroll
        for (int i = 0; i < AS_HDR; ++i) vd[i] = lane + 32 * i < hd ? vr[lane + 32 * i] : 0.f;
#pragma unroll
        for (int r = 0; r < AS_R; ++r) {
          const float p = __shfl_sync(0xffffffffu, s[r], jj);
#pragma unroll
          for (int i = 0; i < AS_HDR; ++i) acc[r][i] = fmaf(p, vd[i], acc[r][i]);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < AS_R; ++r) {
    float sum = l[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const int t = row0 + r;
    if (t >= T) continue;
    const float inv = 1.f / sum;
#pragma unroll
    for (int i = 0; i < AS_HDR; ++i)
      if (lane + 32 * i < hd) out[((size_t)n * T + t) * D + h * hd + lane + 32 * i] = acc[r][i] * inv;
  }
}

void launch_attention(const float* qk, const float* v, float* out, int N, int T, int heads, int hd, cudaStream_t st) {
  if (hd == AT_HD && (((uintptr_t)qk | (uintptr_t)v) & 15) == 0) {
    const int threads = 256, nw = threads / 32;
    const size_t smem = ((size_t)2 * T * AT_LD + (((size_t)nw * T + 3) & ~(size_t)3) + (size_t)nw * 32 * AT_LD) * sizeof(float);
    if (smem <= 200 * 1024) {
      static PerDeviceOnce attr40;
      if (attr40.first()) CUDA_OK(cudaFuncSetAttribute(attention40_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      ProfScope ps("attention", 4.0 * N * heads * (double)T * T * hd, 16.0 * N * T * heads * hd, st);
      int rb = (T + 31) / 32; if (rb > 6) rb = 6; if (rb < 1) rb = 1;
      attention40_kernel<<<dim3(N * heads, rb), threads, smem, st>>>(qk, v, out, T, heads, 1.0f / sqrtf((float)hd));
      LAUNCH_END();
      return;
    }
  }
  const int threads = 256;
  const size_t smem = ((size_t)2 * T * (hd + 1) + (size_t)(threads / 32) * T + (size_t)(threads / 32) * hd) * sizeof(float);
  if (smem > 200 * 1024) {
    MITB_CHECK(hd <= 32 * AS_HDR, "attention: sequence too long (T=%d) for head_dim %d; longer sequences need head_dim <= %d", T, hd,
               32 * AS_HDR);
    const int nw = threads / 32, rows = nw * AS_R;
    MITB_CHECK(N >= 1 && heads >= 1 && (long)N * heads <= INT_MAX && (T + rows - 1) / rows <= 65535, "attention: bad shape n=%d t=%d heads=%d",
               N, T, heads);
    const size_t ssm = ((size_t)2 * AS_TK * (hd + 1) + (size_t)rows * hd) * sizeof(float);   // <= 41.5 KB: no opt-in needed
    ProfScope ps("attention", 4.0 * N * heads * (double)T * T * hd, 16.0 * N * T * heads * hd, st);
    attention_stream_kernel<<<dim3(N * heads, (T + rows - 1) / rows), threads, ssm, st>>>(qk, v, out, T, heads, hd, 1.0f / sqrtf((float)hd));
    LAUNCH_END();
    return;
  }
  static PerDeviceOnce attr_set;
  if (attr_set.first()) CUDA_OK(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  ProfScope ps("attention", 4.0 * N * heads * (double)T * T * hd, 16.0 * N * T * heads * hd, st);
  int rb = (T + 31) / 32; if (rb > 6) rb = 6; if (rb < 1) rb = 1;       // row blocks: >= 4 query rows per warp, <= 6 CTAs per (line, head)
  attention_kernel<<<dim3(N * heads, rb), threads, smem, st>>>(qk, v, out, T, heads, hd, 1.0f / sqrtf((float)hd));
  LAUNCH_END();
}

// ---------------------------------------------------------------------------------------------------
// LaMa glue.  pack: cat(img*(1-mask), mask) NCHW -> NHWC 4 channels (inpainting_lama_mpe.py:604).
__global__ void lama_pack_kernel(const float* img, const float* mask, int N, long HW, float* dst, int cs, int coff, int Cv) {
  const long total = (long)N * HW;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i % HW; const int n = (int)(i / HW);
    const float m = mask[(size_t)n * HW + pix];
    float4 v;
    v.x = img[((size_t)n * 3 + 0) * HW + pix] * (1.f - m);
    v.y = img[((size_t)n * 3 + 1) * HW + pix] * (1.f - m);
    v.z = img[((size_t)n * 3 + 2) * HW + pix] * (1.f - m);
    v.w = m;
    *reinterpret_cast<float4*>(dst + i * cs + coff) = v;
    if (Cv == 8) *reinterpret_cast<float4*>(dst + i * cs + coff + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
void launch_lama_pack_input(const float* img, const float* mask, int N, int H, int W, const View& dst, cudaStream_t st) {
  const long total = (long)N * H * W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  lama_pack_kernel<<<blocks, 256, 0, st>>>(img, mask, N, (long)H * W, dst.p, dst.cs, dst.coff, dst.C);
  LAUNCH_END();
}

// Need maps for the output-sparse LaMa decoder.  need_from_mask: 1 where a hole pixel (mask != 0 / uint8 mask >= 128) lies within
// `radius` (Chebyshev) - the pixels of the last feature map that the final 7x7 conv reads for a hole pixel.  need_pool2: OR over 2x2
// blocks (the logical grid of a stride-2 transposed conv's phases), and that map dilated by 1 (the inputs those phases read).
__global__ void need_from_mask_kernel(const float* mask_f, const uint8_t* mask_u8, int H, int W, int radius, uint8_t* need) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W || y >= H) return;
  int any = 0;
  for (int dy = -radius; dy <= radius && !any; ++dy) {
    const int yy = y + dy; if (yy < 0 || yy >= H) continue;
    for (int dx = -radius; dx <= radius; ++dx) {
      const int xx = x + dx; if (xx < 0 || xx >= W) continue;
      const size_t i = (size_t)yy * W + xx;
      if (mask_f ? mask_f[i] != 0.f : mask_u8[i] >= 128) { any = 1; break; }
    }
  }
  need[(size_t)y * W + x] = (uint8_t)any;
}
__global__ void need_pool2_kernel(const uint8_t* src, int H, int W, uint8_t* pooled) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, h2 = H / 2, w2 = W / 2;
  if (x >= w2 || y >= h2) return;
  const uint8_t* r0 = src + (size_t)(2 * y) * W + 2 * x;
  pooled[(size_t)y * w2 + x] = (uint8_t)((r0[0] | r0[1] | r0[W] | r0[W + 1]) != 0);
}
__global__ void need_dilate1_kernel(const uint8_t* src, int H, int W, uint8_t* dst) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W || y >= H) return;
  int any = 0;
  for (int dy = -1; dy <= 1; ++dy) {
    const int yy = y + dy; if (yy < 0 || yy >= H) continue;
    for (int dx = -1; dx <= 1; ++dx) { const int xx = x + dx; if (xx >= 0 && xx < W) any |= src[(size_t)yy * W + xx]; }
  }
  dst[(size_t)y * W + x] = (uint8_t)(any != 0);
}
void launch_need_from_mask(const float* mask_f, const uint8_t* mask_u8, int H, int W, int radius, uint8_t* need, cudaStream_t st) {
  need_from_mask_kernel<<<dim3((W + 255) / 256, H), 256, 0, st>>>(mask_f, mask_u8, H, W, radius, need);
  LAUNCH_END();
}
void launch_need_pool2(const uint8_t* src, int H, int W, uint8_t* pooled, uint8_t* dilated, cudaStream_t st) {
  MITB_CHECK(H % 2 == 0 && W % 2 == 0, "need_pool2: odd size");
  need_pool2_kernel<<<dim3((W / 2 + 255) / 256, H / 2), 256, 0, st>>>(src, H, W, pooled);
  LAUNCH_END();
  if (dilated) { need_dilate1_kernel<<<dim3((W / 2 + 255) / 256, H / 2), 256, 0, st>>>(pooled, H / 2, W / 2, dilated); LAUNCH_END(); }
}

// blend: out = pred*mask + (1-mask)*img, pred planar NCHW view (inpainting_lama_mpe.py:726)
__global__ void lama_blend_kernel(const float* pred, const float* img, const float* mask, float* out, int N, long HW) {
  const long total = (long)N * 3 * HW;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i % HW; const int n = (int)(i / (3 * HW));
    const float m = mask[(size_t)n * HW + pix];
    out[i] = pred[i] * m + (1.f - m) * img[i];
  }
}
void launch_lama_blend(const View& pred, const float* img, const float* mask, float* out, cudaStream_t st) {
  MITB_CHECK(pred.planar && pred.C == 3 && pred.cs == 3 && pred.coff == 0, "blend expects a planar 3-channel prediction");
  const long total = (long)pred.N * 3 * pred.H * pred.W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  lama_blend_kernel<<<blocks, 256, 0, st>>>(pred.p, img, mask, out, pred.N, (long)pred.H * pred.W);
  LAUNCH_END();
}

// uint8 front/back end of LamaMPEInpainter._infer fused on the device (inpainting_lama_mpe.py:82-92 and :109-117):
//   front: img/255 (fp32 division), mask/255 >= 0.5 -> {0,1}, img *= 1-mask, cat(img*(1-mask), mask) -> NHWC view, + planar mask
//   back : pred*mask + (1-mask)*img -> (x*255).astype(uint8) (truncation) -> optional composite with the original page where
//          the ORIGINAL mask >= 127 (the two thresholds differ at mask value 127, kept as in the reference)
__global__ void lama_pack_u8_kernel(const uint8_t* img, const uint8_t* mask, long npix, float* dst, int cs, int coff, int Cv,
                                    float* maskf) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < npix; i += (long)gridDim.x * blockDim.x) {
    const float m = __fdiv_rn((float)mask[i], 255.f) >= 0.5f ? 1.f : 0.f;
    const float k = 1.f - m;
    float4 v;
    v.x = __fdiv_rn((float)img[i * 3 + 0], 255.f) * k * k;     // premask in _infer (:92) and again in the generator (:604)
    v.y = __fdiv_rn((float)img[i * 3 + 1], 255.f) * k * k;
    v.z = __fdiv_rn((float)img[i * 3 + 2], 255.f) * k * k;
    v.w = m;
    *reinterpret_cast<float4*>(dst + i * cs + coff) = v;
    if (Cv == 8) *reinterpret_cast<float4*>(dst + i * cs + coff + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    maskf[i] = m;
  }
}
void launch_lama_pack_u8(const uint8_t* img, const uint8_t* mask, int H, int W, const View& dst, float* maskf, cudaStream_t st) {
  const long total = (long)H * W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  lama_pack_u8_kernel<<<blocks, 256, 0, st>>>(img, mask, total, dst.p, dst.cs, dst.coff, dst.C, maskf);
  LAUNCH_END();
}

__global__ void lama_blend_u8_kernel(const float* pred, const uint8_t* img, const uint8_t* mask, uint8_t* out, long HW, int composite) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < HW; i += (long)gridDim.x * blockDim.x) {
    const uint8_t mv = mask[i];
    const bool hole = __fdiv_rn((float)mv, 255.f) >= 0.5f;
    const bool keep_orig = composite && mv < 127;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const uint8_t o = img[i * 3 + c];
      const float x = hole ? pred[(size_t)c * HW + i] : __fdiv_rn((float)o, 255.f);
      const uint8_t q = (uint8_t)(int)__fmul_rn(x, 255.f);                 // numpy float32 -> uint8: truncation
      out[i * 3 + c] = keep_orig ? o : q;
    }
  }
}
void launch_lama_blend_u8(const View& pred, const uint8_t* img, const uint8_t* mask, uint8_t* out, int composite, cudaStream_t st) {
  MITB_CHECK(pred.planar && pred.C == 3 && pred.cs == 3 && pred.coff == 0 && pred.N == 1, "blend_u8 expects one planar 3-channel prediction");
  const long total = (long)pred.H * pred.W;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  lama_blend_u8_kernel<<<blocks, 256, 0, st>>>(pred.p, img, mask, out, total, composite);
  LAUNCH_END();
}

// x_l += table[rel_pos]*alpha5 ; x_l += (direct @ W)*alpha6  (inpainting_lama_mpe.py:609-612, 625-632).
// The integer tables may be given at the 256x256 working resolution of load_masked_position_encoding (:751-815); the
// kernel then does its INTER_NEAREST upsampling (sx = min(floor(x * 1/(W/tw)), tw-1), cv2 semantics) and the
// "zero outside the hole" step (:809-813) on the fly instead of materialising 5 full-resolution int planes on the host.
__global__ void mpe_add_kernel(float* x, int cs, int coff, int N, int H, int W, const int* rel_pos, const int* direct, int th,
                               int tw, const float* mask, const float* table, const float* dirw, float a5, float a6) {
  const long npix = (long)N * H * W;
  const long total = npix * 16;                  // 64 channels = 16 float4 per pixel
  const bool lowres = th != H || tw != W;
  const double ify = 1.0 / ((double)H / (double)th), ifx = 1.0 / ((double)W / (double)tw);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i & 15) * 4; const long pix = i >> 4;
    long tpix = pix;
    bool hole = true;
    if (lowres) {
      const int n = (int)(pix / ((long)H * W)); const long r = pix - (long)n * H * W;
      const int y = (int)(r / W), xx = (int)(r - (long)y * W);
      const int sy = min((int)floor((double)y * ify), th - 1), sx = min((int)floor((double)xx * ifx), tw - 1);
      tpix = ((long)n * th + sy) * tw + sx;
      hole = mask[pix] != 0.f;
    }
    const int rp = hole ? rel_pos[tpix] : 0;
    int4 d = make_int4(0, 0, 0, 0);
    if (hole) d = *reinterpret_cast<const int4*>(direct + tpix * 4);
    float4 v = *reinterpret_cast<float4*>(x + pix * cs + coff + c);
    const float4 e = *reinterpret_cast<const float4*>(table + rp * 64 + c);
    const float4 w0 = *reinterpret_cast<const float4*>(dirw + 0 * 64 + c), w1 = *reinterpret_cast<const float4*>(dirw + 1 * 64 + c);
    const float4 w2 = *reinterpret_cast<const float4*>(dirw + 2 * 64 + c), w3 = *reinterpret_cast<const float4*>(dirw + 3 * 64 + c);
    const float d0 = (float)d.x, d1 = (float)d.y, d2 = (float)d.z, d3 = (float)d.w;
    v.x += e.x * a5; v.y += e.y * a5; v.z += e.z * a5; v.w += e.w * a5;
    v.x += (d0 * w0.x + d1 * w1.x + d2 * w2.x + d3 * w3.x) * a6;
    v.y += (d0 * w0.y + d1 * w1.y + d2 * w2.y + d3 * w3.y) * a6;
    v.z += (d0 * w0.z + d1 * w1.z + d2 * w2.z + d3 * w3.z) * a6;
    v.w += (d0 * w0.w + d1 * w1.w + d2 * w2.w + d3 * w3.w) * a6;
    *reinterpret_cast<float4*>(x + pix * cs + coff + c) = v;
  }
}
// ---------------------------------------------------------------------------------------------------
// LamaFourier.load_masked_position_encoding at its 256x256 working resolution (inpainting_lama_mpe.py:763-803) on the device.
// Input: the INTER_AREA-reduced uint8 mask (hole where != 0).  known = (small == 0) is grown by a 3x3 box per step
// (BORDER_REFLECT_101 like cv2.filter2D); a pixel first covered at step i gets pos = i, and direct[k] = 1 when the k-th 2x2 corner
// neighbourhood already touched the known region at that step.  rel_pos = clip(pos, 0, 127) (pos/128*128 is exact in fp32).
// One CTA per image, the whole bitmap ping-pongs in shared memory; ~max-distance iterations of 64 pixels per thread.
constexpr int MPE_N = 256, MPE_T = 1024;
__global__ void __launch_bounds__(MPE_T) mpe_tables_kernel(const uint8_t* small, int* rel_pos, int* direct) {
  extern __shared__ uint8_t mp_sm[];
  uint8_t* A = mp_sm; uint8_t* B = mp_sm + MPE_N * MPE_N;
  const uint8_t* src = small + (size_t)blockIdx.x * MPE_N * MPE_N;
  int* rel = rel_pos + (size_t)blockIdx.x * MPE_N * MPE_N;
  int* dir = direct + (size_t)blockIdx.x * MPE_N * MPE_N * 4;
  int any_known = 0, all_known = 1;
  for (int p = threadIdx.x; p < MPE_N * MPE_N; p += MPE_T) {
    const uint8_t k = src[p] == 0 ? 1 : 0;
    A[p] = k; any_known |= k; all_known &= k;
    rel[p] = 0;
    *reinterpret_cast<int4*>(dir + (size_t)p * 4) = make_int4(0, 0, 0, 0);
  }
  any_known = __syncthreads_or(any_known);
  all_known = __syncthreads_and(all_known);
  if (!any_known) return;                                       // no known pixel: the reference loop never runs, tables stay 0
  auto refl = [](int i) { return i < 0 ? -i : (i >= MPE_N ? 2 * MPE_N - 2 - i : i); };
  int step = 0;
  while (!all_known) {
    ++step;
    int all_now = 1;
    for (int p = threadIdx.x; p < MPE_N * MPE_N; p += MPE_T) {
      const int y = p >> 8, x = p & 255;
      uint8_t g = A[p];
      if (!g) {
        const int ym = refl(y - 1) << 8, y0 = y << 8, yp = refl(y + 1) << 8, xm = refl(x - 1), xp = refl(x + 1);
        const uint8_t a = A[ym + xm], b = A[ym + x], c = A[ym + xp], d = A[y0 + xm], e = A[y0 + xp], f = A[yp + xm], h = A[yp + x], i = A[yp + xp];
        g = a | b | c | d | e | f | h | i;
        if (g) {
          rel[p] = step < 127 ? step : 127;
          *reinterpret_cast<int4*>(dir + (size_t)p * 4) = make_int4((a | b | d) ? 1 : 0, (d | f | h) ? 1 : 0, (b | c | e) ? 1 : 0, (e | h | i) ? 1 : 0);
        }
      }
      B[p] = g; all_now &= g;
    }
    all_known = __syncthreads_and(all_now);
    uint8_t* t = A; A = B; B = t;
  }
}
void launch_mpe_tables(const uint8_t* small, int n, int* rel_pos, int* direct, cudaStream_t st) {
  static PerDeviceOnce attr;
  if (attr.first()) CUDA_OK(cudaFuncSetAttribute(mpe_tables_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * MPE_N * MPE_N));
  mpe_tables_kernel<<<n, MPE_T, 2 * MPE_N * MPE_N, st>>>(small, rel_pos, direct);
  LAUNCH_END();
}

void launch_mpe_add(const View& x, const int* rel_pos, const int* direct, int th, int tw, const float* mask, const float* table,
                    const float* dirw, float a5, float a6, cudaStream_t st) {
  MITB_CHECK(x.C == 64 && x.cs % 4 == 0 && x.coff % 4 == 0, "mpe_add expects the 64-channel stem output");
  const long total = (long)x.pixels() * 16;
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 32) blocks = 148 * 32;
  mpe_add_kernel<<<blocks, 256, 0, st>>>(x.p, x.cs, x.coff, x.N, x.H, x.W, rel_pos, direct, th, tw, mask, table, dirw, a5, a6);
  LAUNCH_END();
}

}  // namespace mitb
