// a1 / a2 / a10: batched letterbox preprocess and plain bilinear resize.
//
// Replaces _TensorRTBaseDetector._preprocess (detector.py:198-264), RKNNDetector._preprocess
// (detector.py:777-839) and utils.downsample (frame_filter.py:53-57) of the reference.
// The interpolation is OpenCV's 8-bit INTER_LINEAR: 11-bit integer tap coefficients per axis,
// horizontal pass in int32, vertical pass ((b0*(S0>>4))>>16 + (b1*(S1>>4))>>16 + 2) >> 2.
//
// (Forcing 7 or 8 CTAs per SM with __launch_bounds__ -- 56 / 48 registers -- measured 3 % / 10 % SLOWER on 32 x 1080p:
// the kernel is not short of warps.)
// Data movement: every CTA owns `rows_per_cta` consecutive output rows of one frame.  Only the
// source rows that carry a non-zero vertical weight are fetched; each is brought into shared
// memory whole by ONE 1-D bulk async copy (cp.async.bulk -> UBLKCP, the TMA engine) tracked by an
// mbarrier, `stages` rows ahead of the row being computed.  Threads then gather their taps from
// shared memory and write planar output rows with 16-byte stores.  Frames whose base / pitch /
// row length are not 16-byte multiples take the same code with a cooperative byte loader.
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <type_traits>

#include "common.cuh"

namespace {

struct PreFrame {
  const uint8_t* src;
  const uint8_t* mask;  // optional ROI mask [src_h, src_w], 0 = outside
  long long pitch;
  int src_h, src_w;
  int xtab, ytab;  // offsets (in 16-byte entries) into the tap arena
  int bulk_ok;     // frame (and mask) rows can be fetched with 16-byte bulk copies
  int out_idx;     // position of this frame in the output batch
  void* out;       // b200va_resize_linear_u8: this frame's own destination buffer (NULL: PreParams::out + out_idx)
};

struct PreParams {
  PreFrame f[B200VA_LAUNCH_FRAMES];
  const int4* tabs;
  void* out;
  int dst_h, dst_w, fmt, rows_per_cta;
  int row_stride, mask_stride, stages, vec_ok;
  int rows_per_stage;  // 1 when no frame of the launch ever needs the second source row
  int keep_pad_rows;   // B200VA_OUT_FLAG_PADS_VALID: full-width pad rows of `out` already hold the pad value
  long long* dbg;      // timing builds: timeline stamps
  const uint8_t* skip; // device-side gates: frames whose flag is non-zero are not letterboxed (indexed by out_idx)
  int pdl_wait;        // launched as a programmatic dependent that must not touch HBM before its primary is done (tick schedule 5)
};
static_assert(sizeof(PreParams) <= 4000, "kernel parameter block too large");

constexpr int kMaxStages = 4;
constexpr int kMaxRowsPerCta = 16;
constexpr int kThreads = 160;  // 4 output pixels per thread -> 640 columns

__device__ __forceinline__ void coop_copy(uint8_t* dst, const uint8_t* src, int bytes) {
  // generic loader for rows that cannot use 16-byte bulk copies
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = __ldg(src + i);
}

// Store 4 pixels (v[j][c]: pixel j, channel c in BGR order, 0..255).  `o` points at the element
// of plane 0 (NCHW) / at the pixel (NHWC); `plane` is the plane stride in elements; `nvalid` is
// how many of the 4 pixels lie inside the row.
template <int FMT>
__device__ __forceinline__ void store_px4(void* o, size_t plane, bool vec_ok, int nvalid, const int (&v)[4][3]) {
  if (FMT == B200VA_OUT_F32_RGB_NCHW) {
    const float k = __int_as_float(0x3B808081);  // float32(1.0/255.0), detector.py:251
#pragma unroll
    for (int pl = 0; pl < 3; ++pl) {
      float* row = (float*)o + pl * plane;
      float r[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) r[j] = __fmul_rn((float)v[j][2 - pl], k);
      if (vec_ok) {
        *reinterpret_cast<float4*>(row) = make_float4(r[0], r[1], r[2], r[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < nvalid) row[j] = r[j];
      }
    }
  } else if (FMT == B200VA_OUT_F16_RGB_NCHW) {
    const float k = 0.0039215087890625f;  // float(float16(1.0/255.0)): NumPy rounds the scalar to half first
#pragma unroll
    for (int pl = 0; pl < 3; ++pl) {
      __half* row = (__half*)o + pl * plane;
      __half r[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) r[j] = __float2half_rn(__fmul_rn((float)v[j][2 - pl], k));
      if (vec_ok) {
        uint2 w;
        w.x = (uint32_t)__half_as_ushort(r[0]) | ((uint32_t)__half_as_ushort(r[1]) << 16);
        w.y = (uint32_t)__half_as_ushort(r[2]) | ((uint32_t)__half_as_ushort(r[3]) << 16);
        *reinterpret_cast<uint2*>(row) = w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < nvalid) row[j] = r[j];
      }
    }
  } else if (FMT == B200VA_OUT_U8_BGR_NCHW) {
#pragma unroll
    for (int pl = 0; pl < 3; ++pl) {
      uint8_t* row = (uint8_t*)o + pl * plane;
      if (vec_ok) {
        *reinterpret_cast<uint32_t*>(row) =
            (uint32_t)v[0][pl] | ((uint32_t)v[1][pl] << 8) | ((uint32_t)v[2][pl] << 16) | ((uint32_t)v[3][pl] << 24);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < nvalid) row[j] = (uint8_t)v[j][pl];
      }
    }
  } else {  // B200VA_OUT_U8_BGR_NHWC
    uint8_t* row = (uint8_t*)o;
    if (vec_ok) {
      uint32_t w0 = (uint32_t)v[0][0] | ((uint32_t)v[0][1] << 8) | ((uint32_t)v[0][2] << 16) | ((uint32_t)v[1][0] << 24);
      uint32_t w1 = (uint32_t)v[1][1] | ((uint32_t)v[1][2] << 8) | ((uint32_t)v[2][0] << 16) | ((uint32_t)v[2][1] << 24);
      uint32_t w2 = (uint32_t)v[2][2] | ((uint32_t)v[3][0] << 8) | ((uint32_t)v[3][1] << 16) | ((uint32_t)v[3][2] << 24);
      uint32_t* q = reinterpret_cast<uint32_t*>(row);
      q[0] = w0;
      q[1] = w1;
      q[2] = w2;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < nvalid) {
          row[3 * j + 0] = (uint8_t)v[j][0];
          row[3 * j + 1] = (uint8_t)v[j][1];
          row[3 * j + 2] = (uint8_t)v[j][2];
        }
    }
  }
}

// Four output pixels of one row from the staged source rows (general two-tap, two-row case).
// The two taps of a pixel are six consecutive bytes of the row (off1 = off0 + 3; where the x axis clamps, off1 = off0
// and a1 = 0, so whatever sits behind off0 + 3 is multiplied by zero).  They are fetched as the three aligned words
// that cover them and lined up with two funnel shifts; per channel one PRMT pairs the tap bytes and one IDP.2A does
// byte * a0 + byte * a1 (the coefficients are at most 2048: two 16-bit halves of one register).  Three word loads
// instead of six byte loads per pixel and row: the byte loads, at a 24- or 48-byte lane stride, kept the shared-memory
// pipe 60-72 % busy with 2- and 4-way bank conflicts.
__device__ __forceinline__ void taps_row(const uint8_t* __restrict__ r, int off0, uint32_t coef, int (&s)[3]) {
  const uint32_t* __restrict__ w = reinterpret_cast<const uint32_t*>(r + (off0 & ~3));
  const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
  const uint32_t sh = (uint32_t)(off0 & 3) * 8u;
  const uint32_t x = __funnelshift_r(w0, w1, sh), y = __funnelshift_r(w1, w2, sh);  // bytes off0 .. off0 + 7
  s[0] = (int)__dp2a_lo(coef, __byte_perm(x, y, 0x0030), 0u);  // (B0, B1)
  s[1] = (int)__dp2a_lo(coef, __byte_perm(x, y, 0x0041), 0u);  // (G0, G1)
  s[2] = (int)__dp2a_lo(coef, __byte_perm(x, y, 0x0052), 0u);  // (R0, R1)
}

template <bool MASK>
__device__ __forceinline__ void px4_general(const TapX (&t)[4], const uint8_t* __restrict__ r0,
                                            const uint8_t* __restrict__ r1, const uint8_t* __restrict__ m0,
                                            const uint8_t* __restrict__ m1, int b0, int b1, int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;  // copyMakeBorder value, detector.py:233-241
      continue;
    }
    int s0[3] = {0, 0, 0}, s1[3] = {0, 0, 0};
    if (b0) {
      int c0 = t[j].a0, c1 = t[j].a1;
      if (MASK) {  // apply_roi zeroes masked source pixels before the resize (pipeline.py:149-154)
        c0 = m0[t[j].mx0 & 0xffff] ? c0 : 0;
        c1 = m0[(unsigned)t[j].mx0 >> 16] ? c1 : 0;
      }
      taps_row(r0, t[j].off0, (uint32_t)c0 | ((uint32_t)c1 << 16), s0);
    }
    if (b1) {
      int c0 = t[j].a0, c1 = t[j].a1;
      if (MASK) {
        c0 = m1[t[j].mx0 & 0xffff] ? c0 : 0;
        c1 = m1[(unsigned)t[j].mx0 >> 16] ? c1 : 0;
      }
      taps_row(r1, t[j].off0, (uint32_t)c0 | ((uint32_t)c1 << 16), s1);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) v[j][c] = (((b0 * (s0[c] >> 4)) >> 16) + ((b1 * (s1[c] >> 4)) >> 16) + 2) >> 2;
  }
}

// Even integer ratios (720p, 1440p and 4K into 640 x 360: ratios 2, 4 and 6): both taps of both axes weigh 1024, and the
// fixed-point formula collapses exactly -- (1024 * (p0 + p1)) >> 4 = 64 (p0 + p1), (1024 * that) >> 16 = p0 + p1 -- to
// the rounded mean of the four source bytes, (p00 + p01 + p10 + p11 + 2) >> 2.  The two tap pixels of a row are lined
// up like in taps_row; a channel's sum is two to four IDP.4A with 0 / 1 byte selectors.  ~28 instructions per pixel
// instead of ~100: on these shapes the general path is bound by instruction issue, not by memory (DESIGN 3.1).
__device__ __forceinline__ void px4_box(const TapX (&t)[4], const uint8_t* __restrict__ r0, const uint8_t* __restrict__ r1,
                                        int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;
      continue;
    }
    const int base = t[j].off0 & ~3;
    const uint32_t sh = (uint32_t)(t[j].off0 & 3) * 8u;
    const uint32_t* __restrict__ w0 = reinterpret_cast<const uint32_t*>(r0 + base);
    const uint32_t* __restrict__ w1 = reinterpret_cast<const uint32_t*>(r1 + base);
    const uint32_t a0 = w0[0], a1 = w0[1], a2 = w0[2], c0 = w1[0], c1 = w1[1], c2 = w1[2];
    const uint32_t x0 = __funnelshift_r(a0, a1, sh), y0 = __funnelshift_r(a1, a2, sh);  // row 0: B0 G0 R0 B1 | G1 R1 . .
    const uint32_t x1 = __funnelshift_r(c0, c1, sh), y1 = __funnelshift_r(c1, c2, sh);  // row 1
    v[j][0] = (int)(__dp4a(x0, 0x01000001u, __dp4a(x1, 0x01000001u, 2u)) >> 2);
    v[j][1] = (int)(__dp4a(x0, 0x00000100u, __dp4a(y0, 0x00000001u, __dp4a(x1, 0x00000100u, __dp4a(y1, 0x00000001u, 2u)))) >> 2);
    v[j][2] = (int)(__dp4a(x0, 0x00010000u, __dp4a(y0, 0x00000100u, __dp4a(x1, 0x00010000u, __dp4a(y1, 0x00000100u, 2u)))) >> 2);
  }
}

// Integer-ratio subsampling (e.g. 1080p -> 640x360): every tap is (2048, 0) on both axes, for which
// the fixed-point formula returns the source byte itself.
template <bool MASK>
__device__ __forceinline__ void px4_identity(const TapX (&t)[4], const uint8_t* __restrict__ r0,
                                             const uint8_t* __restrict__ m0, int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;
      continue;
    }
    const bool on = !MASK || m0[t[j].mx0 & 0xffff];
#pragma unroll
    for (int c = 0; c < 3; ++c) v[j][c] = on ? (int)r0[t[j].off0 + c] : 0;
  }
}

template <int FMT, bool MASK>
__global__ void __launch_bounds__(kThreads) k_letterbox(const __grid_constant__ PreParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t full[kMaxStages];
  __shared__ TapY s_ty[kMaxRowsPerCta];

  TIMELINE_BEGIN(p.dbg, 42);
  const int frame = blockIdx.y;
  const PreFrame& f = p.f[frame];
  if (p.skip && p.skip[f.out_idx]) return;  // gated off on the device (pipeline.py:156-170): nobody reads this frame's tensor
  const TapX* __restrict__ xt = reinterpret_cast<const TapX*>(p.tabs + f.xtab);
  const TapY* __restrict__ yt = reinterpret_cast<const TapY*>(p.tabs + f.ytab);
  const int S = p.stages;
  const int row_begin = blockIdx.x * p.rows_per_cta;
  const int nrows = min(p.rows_per_cta, p.dst_h - row_begin);
  const bool bulk = f.bulk_ok != 0;
  const uint32_t stage_bytes = (uint32_t)p.rows_per_stage * (uint32_t)p.row_stride;
  const uint32_t mstage_bytes = (uint32_t)p.rows_per_stage * (uint32_t)p.mask_stride;
  uint8_t* const rows_base = smem;
  uint8_t* const mask_base = smem + (size_t)S * stage_bytes;
  const uint32_t row_bytes = 3u * (uint32_t)f.src_w;

  if (threadIdx.x < nrows) s_ty[threadIdx.x] = yt[row_begin + threadIdx.x];
  if (bulk && threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  // tick schedule 5: this grid was launched while the decode kernel still runs; its CTAs are resident and set up, and
  // their first bulk copy goes out the moment that grid has drained (no launch latency between the two HBM kernels)
  if (p.pdl_wait) griddep_wait();

  // one elected thread feeds the TMA engine: whole source rows, one bulk copy each
  auto issue = [&](int i, int s) {
    const TapY ty = s_ty[i];
    if (ty.y0 < 0) return;
    const uint32_t per_row = row_bytes + (MASK ? (uint32_t)f.src_w : 0u);
    mbar_expect_tx(&full[s], (ty.b0 ? per_row : 0u) + (ty.b1 ? per_row : 0u));
    uint8_t* r0 = rows_base + (size_t)s * stage_bytes;
    uint8_t* m0 = mask_base + (size_t)s * mstage_bytes;
    if (ty.b0) {
      bulk_g2s(r0, f.src + (long long)ty.y0 * f.pitch, row_bytes, &full[s]);
      if (MASK) bulk_g2s(m0, f.mask + (size_t)ty.y0 * f.src_w, f.src_w, &full[s]);
    }
    if (ty.b1) {
      bulk_g2s(r0 + p.row_stride, f.src + (long long)ty.y1 * f.pitch, row_bytes, &full[s]);
      if (MASK) bulk_g2s(m0 + p.mask_stride, f.mask + (size_t)ty.y1 * f.src_w, f.src_w, &full[s]);
    }
  };

  int s_issue = 0;  // stage the next issued row goes to (thread 0 only)
  if (bulk && threadIdx.x == 0) {
    for (int i = 0; i < S - 1 && i < nrows; ++i) {
      issue(i, s_issue);
      s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
    }
  }

  const int ngroups = (p.dst_w + 3) >> 2;
  const int nthreads = blockDim.x;
  // tap entries of this thread's first pixel group stay in registers across all rows
  TapX tx[4];
  bool ident = true, box = !MASK;  // (an ROI mask zeroes single taps: the general path)
  {
    const int g = threadIdx.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int x = 4 * g + j;
      if (g < ngroups && x < p.dst_w) {
        int4 e = __ldg(reinterpret_cast<const int4*>(xt) + x);
        tx[j] = *reinterpret_cast<TapX*>(&e);
      } else {
        tx[j].off0 = -1;
        tx[j].off1 = -1;
        tx[j].a0 = tx[j].a1 = 0;
        tx[j].mx0 = 0;
      }
      ident = ident && (tx[j].off0 < 0 || (tx[j].a0 == 2048 && tx[j].a1 == 0));
      box = box && (tx[j].off0 < 0 || (tx[j].a0 == 1024 && tx[j].a1 == 1024 && tx[j].off1 == tx[j].off0 + 3));
    }
  }
  const size_t plane = (size_t)p.dst_h * p.dst_w;
  const size_t esize = FMT == B200VA_OUT_F32_RGB_NCHW ? 4 : (FMT == B200VA_OUT_F16_RGB_NCHW ? 2 : 1);
  const bool nhwc = FMT == B200VA_OUT_U8_BGR_NHWC;
  // element (frame, plane 0, row_begin, 4*tid) / pixel (frame, row_begin, 4*tid)
  uint8_t* optr = (f.out ? (uint8_t*)f.out : (uint8_t*)p.out + ((size_t)f.out_idx * 3 * plane) * esize) +
                  (nhwc ? ((size_t)row_begin * p.dst_w + 4 * threadIdx.x) * 3
                        : ((size_t)row_begin * p.dst_w + 4 * threadIdx.x) * esize);
  const size_t row_step = nhwc ? (size_t)p.dst_w * 3 : (size_t)p.dst_w * esize;
  const bool vec_ok = p.vec_ok != 0;
  const int nvalid0 = min(4, p.dst_w - 4 * (int)threadIdx.x);

  uint32_t phase_bits = 0;
  int s = 0;
  for (int i = 0; i < nrows; ++i, optr += row_step) {
    const TapY ty = s_ty[i];
    const bool pad_row = ty.y0 < 0;
    const int sc = bulk ? s : 0;
    const uint8_t* r0 = rows_base + (size_t)sc * stage_bytes;
    const uint8_t* r1 = r0 + p.row_stride;
    const uint8_t* m0 = mask_base + (size_t)sc * mstage_bytes;
    const uint8_t* m1 = m0 + p.mask_stride;

    if (bulk) {
      if (threadIdx.x == 0 && i + S - 1 < nrows) {
        issue(i + S - 1, s_issue);
        s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
      }
      if (!pad_row) {
        mbar_wait(&full[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
      }
    } else if (!pad_row) {
      if (ty.b0) {
        coop_copy(const_cast<uint8_t*>(r0), f.src + (long long)ty.y0 * f.pitch, row_bytes);
        if (MASK) coop_copy(const_cast<uint8_t*>(m0), f.mask + (size_t)ty.y0 * f.src_w, f.src_w);
      }
      if (ty.b1) {
        coop_copy(const_cast<uint8_t*>(r1), f.src + (long long)ty.y1 * f.pitch, row_bytes);
        if (MASK) coop_copy(const_cast<uint8_t*>(m1), f.mask + (size_t)ty.y1 * f.src_w, f.src_w);
      }
      __syncthreads();
    }

    const bool skip_row = pad_row && p.keep_pad_rows;  // written by an earlier call into the same buffer
    if ((int)threadIdx.x < ngroups && !skip_row) {
      int v[4][3];
      if (pad_row) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j][0] = v[j][1] = v[j][2] = 114;
      } else if (ident && ty.b0 == 2048 && ty.b1 == 0) {
        px4_identity<MASK>(tx, r0, m0, v);
      } else if (box && ty.b0 == 1024 && ty.b1 == 1024) {
        px4_box(tx, r0, r1, v);
      } else {
        px4_general<MASK>(tx, r0, r1, m0, m1, ty.b0, ty.b1, v);
      }
      store_px4<FMT>(optr, plane, vec_ok, nvalid0, v);
    }
    // destination rows wider than 4 * blockDim pixels: remaining groups read their taps from global
    for (int g = threadIdx.x + nthreads; g < ngroups && !skip_row; g += nthreads) {
      TapX t[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = 4 * g + j;
        if (x < p.dst_w) {
          int4 e = __ldg(reinterpret_cast<const int4*>(xt) + x);
          t[j] = *reinterpret_cast<TapX*>(&e);
        } else {
          t[j].off0 = -1;
        }
      }
      int v[4][3];
      if (pad_row) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j][0] = v[j][1] = v[j][2] = 114;
      } else {
        px4_general<MASK>(t, r0, r1, m0, m1, ty.b0, ty.b1, v);
      }
      store_px4<FMT>(optr + (size_t)(g - (int)threadIdx.x) * 4 * (nhwc ? 3 : esize), plane, vec_ok,
                     min(4, p.dst_w - 4 * g), v);
    }
    // the stage read in this iteration is refilled by the next iteration's issue()
    if (!pad_row) __syncthreads();
    s = s + 1 == S ? 0 : s + 1;
  }
  TIMELINE_END(p.dbg, 42);
}

// ---- NV12 sources ---------------------------------------------------------------------------
// The same letterbox / resize with cv2.cvtColor(frame, COLOR_YUV2BGR_NV12) folded into the taps: each tapped luma row
// and the CbCr row it uses (row y >> 1 of the interleaved chroma plane; the two luma taps of an output row often share
// it, and then it is fetched once) are staged by one bulk copy each, and every tap pixel is converted to B, G, R with
// OpenCV's BT.601 limited-range fixed point and nearest chroma before the unchanged integer interpolation.  Two planes
// per frame do not fit 64 frames in a 4 KB parameter block: an NV12 launch takes 32.
struct Nv12Frame {
  const uint8_t* y;
  const uint8_t* uv;    // src_h / 2 rows of src_w bytes: Cb, Cr of each 2 x 2 block
  const uint8_t* mask;  // optional ROI mask [src_h, src_w], 0 = outside
  void* out;            // b200va_resize_linear_u8_nv12: this frame's own destination buffer
  long long y_pitch, uv_pitch;
  int src_h, src_w;
  int xtab, ytab;
  int bulk_ok;
  int out_idx;
};

constexpr int kNv12LaunchFrames = 32;
struct PreParamsNv12 {
  Nv12Frame f[kNv12LaunchFrames];
  const int4* tabs;
  void* out;
  int dst_h, dst_w, fmt, rows_per_cta;
  int row_stride, mask_stride, stages, vec_ok;
  int rows_per_stage;
  int keep_pad_rows;
  long long* dbg;
  const uint8_t* skip;
  int pdl_wait;
};
static_assert(sizeof(PreParamsNv12) <= 4000, "kernel parameter block too large");

// pixel x of a staged luma row and its chroma row (chroma rows start 128-byte aligned: the pair load is aligned)
__device__ __forceinline__ uint32_t nv12_tap(const uint8_t* __restrict__ yr, const uint8_t* __restrict__ cr, int x) {
  return nv12_bgr(yr[x], *reinterpret_cast<const uint16_t*>(cr + (x & ~1)));
}

// byte c of p and byte c of q in bytes 0 / 1, zeros above (byte 3 of a packed pixel is zero)
__device__ __forceinline__ uint32_t pair_c(uint32_t p, uint32_t q, int c) {
  return __byte_perm(p, q, (uint32_t)c | ((uint32_t)(4 + c) << 4) | 0x3300u);
}

// one tapped row: per channel a0 * p + a1 * q with one IDP.2A, as in taps_row
__device__ __forceinline__ void nv12_taps_row(const uint8_t* __restrict__ yr, const uint8_t* __restrict__ cr, int i0, int i1,
                                              uint32_t coef, int (&s)[3]) {
  const uint32_t p = nv12_tap(yr, cr, i0), q = nv12_tap(yr, cr, i1);
#pragma unroll
  for (int c = 0; c < 3; ++c) s[c] = (int)__dp2a_lo(coef, pair_c(p, q, c), 0u);
}

template <bool MASK>
__device__ __forceinline__ void nv12_px4_general(const TapX (&t)[4], const uint8_t* __restrict__ y0, const uint8_t* __restrict__ c0r,
                                                 const uint8_t* __restrict__ y1, const uint8_t* __restrict__ c1r,
                                                 const uint8_t* __restrict__ m0, const uint8_t* __restrict__ m1, int b0, int b1,
                                                 int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;  // copyMakeBorder value, detector.py:233-241
      continue;
    }
    const int i0 = t[j].mx0 & 0xffff, i1 = (int)((unsigned)t[j].mx0 >> 16);
    int s0[3] = {0, 0, 0}, s1[3] = {0, 0, 0};
    if (b0) {
      int a0 = t[j].a0, a1 = t[j].a1;
      if (MASK) {  // apply_roi zeroes masked source pixels before the resize (pipeline.py:149-154)
        a0 = m0[i0] ? a0 : 0;
        a1 = m0[i1] ? a1 : 0;
      }
      nv12_taps_row(y0, c0r, i0, i1, (uint32_t)a0 | ((uint32_t)a1 << 16), s0);
    }
    if (b1) {
      int a0 = t[j].a0, a1 = t[j].a1;
      if (MASK) {
        a0 = m1[i0] ? a0 : 0;
        a1 = m1[i1] ? a1 : 0;
      }
      nv12_taps_row(y1, c1r, i0, i1, (uint32_t)a0 | ((uint32_t)a1 << 16), s1);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) v[j][c] = (((b0 * (s0[c] >> 4)) >> 16) + ((b1 * (s1[c] >> 4)) >> 16) + 2) >> 2;
  }
}

// 2 x 2 box (all four weights 1024): the rounded mean of the four converted pixels, as in px4_box
__device__ __forceinline__ void nv12_px4_box(const TapX (&t)[4], const uint8_t* __restrict__ y0, const uint8_t* __restrict__ c0r,
                                             const uint8_t* __restrict__ y1, const uint8_t* __restrict__ c1r, int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;
      continue;
    }
    const int x = t[j].mx0 & 0xffff;
    const uint32_t p00 = nv12_tap(y0, c0r, x), p01 = nv12_tap(y0, c0r, x + 1);
    const uint32_t p10 = nv12_tap(y1, c1r, x), p11 = nv12_tap(y1, c1r, x + 1);
#pragma unroll
    for (int c = 0; c < 3; ++c)
      v[j][c] = (int)(__dp4a(pair_c(p00, p01, c), 0x0101u, __dp4a(pair_c(p10, p11, c), 0x0101u, 2u)) >> 2);
  }
}

// every tap (2048, 0) on both axes: the converted source pixel itself
template <bool MASK>
__device__ __forceinline__ void nv12_px4_identity(const TapX (&t)[4], const uint8_t* __restrict__ y0, const uint8_t* __restrict__ c0r,
                                                  const uint8_t* __restrict__ m0, int (&v)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (t[j].off0 < 0) {
      v[j][0] = v[j][1] = v[j][2] = 114;
      continue;
    }
    const int x = t[j].mx0 & 0xffff;
    const uint32_t p = (!MASK || m0[x]) ? nv12_tap(y0, c0r, x) : 0u;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[j][c] = (int)((p >> (8 * c)) & 0xffu);
  }
}

// k_letterbox for NV12 frames.  A stage holds rows_per_stage luma rows, then as many chroma rows (row_stride bytes
// apart); the ROI mask rows follow all stages, as in k_letterbox.
template <int FMT, bool MASK>
__global__ void __launch_bounds__(kThreads, 4) k_letterbox_nv12(const __grid_constant__ PreParamsNv12 p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t full[kMaxStages];
  __shared__ TapY s_ty[kMaxRowsPerCta];

  TIMELINE_BEGIN(p.dbg, 42);  // the tick's letterbox slot, whichever source format
  const int frame = blockIdx.y;
  const Nv12Frame& f = p.f[frame];
  if (p.skip && p.skip[f.out_idx]) return;  // gated off on the device: nobody reads this frame's tensor
  const TapX* __restrict__ xt = reinterpret_cast<const TapX*>(p.tabs + f.xtab);
  const TapY* __restrict__ yt = reinterpret_cast<const TapY*>(p.tabs + f.ytab);
  const int S = p.stages;
  const int row_begin = blockIdx.x * p.rows_per_cta;
  const int nrows = min(p.rows_per_cta, p.dst_h - row_begin);
  const bool bulk = f.bulk_ok != 0;
  const uint32_t chroma_off = (uint32_t)p.rows_per_stage * (uint32_t)p.row_stride;
  const uint32_t stage_bytes = 2u * chroma_off;
  const uint32_t mstage_bytes = (uint32_t)p.rows_per_stage * (uint32_t)p.mask_stride;
  uint8_t* const rows_base = smem;
  uint8_t* const mask_base = smem + (size_t)S * stage_bytes;
  const uint32_t w = (uint32_t)f.src_w;  // bytes per luma row and per chroma row

  if (threadIdx.x < nrows) s_ty[threadIdx.x] = yt[row_begin + threadIdx.x];
  if (bulk && threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  if (p.pdl_wait) griddep_wait();

  auto shared_chroma = [](const TapY& ty) { return ty.b0 != 0 && ty.b1 != 0 && (ty.y0 >> 1) == (ty.y1 >> 1); };
  auto issue = [&](int i, int s) {
    const TapY ty = s_ty[i];
    if (ty.y0 < 0) return;
    const bool cs = shared_chroma(ty);
    const uint32_t mb = MASK ? w : 0u;
    mbar_expect_tx(&full[s], (ty.b0 ? 2u * w + mb : 0u) + (ty.b1 ? (cs ? w : 2u * w) + mb : 0u));
    uint8_t* r0 = rows_base + (size_t)s * stage_bytes;
    uint8_t* m0 = mask_base + (size_t)s * mstage_bytes;
    if (ty.b0) {
      bulk_g2s(r0, f.y + (long long)ty.y0 * f.y_pitch, w, &full[s]);
      bulk_g2s(r0 + chroma_off, f.uv + (long long)(ty.y0 >> 1) * f.uv_pitch, w, &full[s]);
      if (MASK) bulk_g2s(m0, f.mask + (size_t)ty.y0 * f.src_w, w, &full[s]);
    }
    if (ty.b1) {
      bulk_g2s(r0 + p.row_stride, f.y + (long long)ty.y1 * f.y_pitch, w, &full[s]);
      if (!cs) bulk_g2s(r0 + chroma_off + p.row_stride, f.uv + (long long)(ty.y1 >> 1) * f.uv_pitch, w, &full[s]);
      if (MASK) bulk_g2s(m0 + p.mask_stride, f.mask + (size_t)ty.y1 * f.src_w, w, &full[s]);
    }
  };

  int s_issue = 0;
  if (bulk && threadIdx.x == 0) {
    for (int i = 0; i < S - 1 && i < nrows; ++i) {
      issue(i, s_issue);
      s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
    }
  }

  const int ngroups = (p.dst_w + 3) >> 2;
  const int nthreads = blockDim.x;
  TapX tx[4];
  bool ident = true, box = !MASK;
  {
    const int g = threadIdx.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int x = 4 * g + j;
      if (g < ngroups && x < p.dst_w) {
        int4 e = __ldg(reinterpret_cast<const int4*>(xt) + x);
        tx[j] = *reinterpret_cast<TapX*>(&e);
      } else {
        tx[j].off0 = -1;
        tx[j].off1 = -1;
        tx[j].a0 = tx[j].a1 = 0;
        tx[j].mx0 = 0;
      }
      ident = ident && (tx[j].off0 < 0 || (tx[j].a0 == 2048 && tx[j].a1 == 0));
      box = box && (tx[j].off0 < 0 || (tx[j].a0 == 1024 && tx[j].a1 == 1024 && tx[j].off1 == tx[j].off0 + 3));
    }
  }
  const size_t plane = (size_t)p.dst_h * p.dst_w;
  const size_t esize = FMT == B200VA_OUT_F32_RGB_NCHW ? 4 : (FMT == B200VA_OUT_F16_RGB_NCHW ? 2 : 1);
  const bool nhwc = FMT == B200VA_OUT_U8_BGR_NHWC;
  uint8_t* optr = (f.out ? (uint8_t*)f.out : (uint8_t*)p.out + ((size_t)f.out_idx * 3 * plane) * esize) +
                  (nhwc ? ((size_t)row_begin * p.dst_w + 4 * threadIdx.x) * 3
                        : ((size_t)row_begin * p.dst_w + 4 * threadIdx.x) * esize);
  const size_t row_step = nhwc ? (size_t)p.dst_w * 3 : (size_t)p.dst_w * esize;
  const bool vec_ok = p.vec_ok != 0;
  const int nvalid0 = min(4, p.dst_w - 4 * (int)threadIdx.x);

  uint32_t phase_bits = 0;
  int s = 0;
  for (int i = 0; i < nrows; ++i, optr += row_step) {
    const TapY ty = s_ty[i];
    const bool pad_row = ty.y0 < 0;
    const int sc = bulk ? s : 0;
    const uint8_t* y0 = rows_base + (size_t)sc * stage_bytes;
    const uint8_t* y1 = y0 + p.row_stride;
    const uint8_t* c0 = y0 + chroma_off;
    const uint8_t* c1 = shared_chroma(ty) ? c0 : c0 + p.row_stride;
    const uint8_t* m0 = mask_base + (size_t)sc * mstage_bytes;
    const uint8_t* m1 = m0 + p.mask_stride;

    if (bulk) {
      if (threadIdx.x == 0 && i + S - 1 < nrows) {
        issue(i + S - 1, s_issue);
        s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
      }
      if (!pad_row) {
        mbar_wait(&full[s], (phase_bits >> s) & 1u);
        phase_bits ^= 1u << s;
      }
    } else if (!pad_row) {
      if (ty.b0) {
        coop_copy(const_cast<uint8_t*>(y0), f.y + (long long)ty.y0 * f.y_pitch, w);
        coop_copy(const_cast<uint8_t*>(c0), f.uv + (long long)(ty.y0 >> 1) * f.uv_pitch, w);
        if (MASK) coop_copy(const_cast<uint8_t*>(m0), f.mask + (size_t)ty.y0 * f.src_w, w);
      }
      if (ty.b1) {
        coop_copy(const_cast<uint8_t*>(y1), f.y + (long long)ty.y1 * f.y_pitch, w);
        if (c1 != c0) coop_copy(const_cast<uint8_t*>(c1), f.uv + (long long)(ty.y1 >> 1) * f.uv_pitch, w);
        if (MASK) coop_copy(const_cast<uint8_t*>(m1), f.mask + (size_t)ty.y1 * f.src_w, w);
      }
      __syncthreads();
    }

    const bool skip_row = pad_row && p.keep_pad_rows;
    if ((int)threadIdx.x < ngroups && !skip_row) {
      int v[4][3];
      if (pad_row) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j][0] = v[j][1] = v[j][2] = 114;
      } else if (ident && ty.b0 == 2048 && ty.b1 == 0) {
        nv12_px4_identity<MASK>(tx, y0, c0, m0, v);
      } else if (box && ty.b0 == 1024 && ty.b1 == 1024) {
        nv12_px4_box(tx, y0, c0, y1, c1, v);
      } else {
        nv12_px4_general<MASK>(tx, y0, c0, y1, c1, m0, m1, ty.b0, ty.b1, v);
      }
      store_px4<FMT>(optr, plane, vec_ok, nvalid0, v);
    }
    for (int g = threadIdx.x + nthreads; g < ngroups && !skip_row; g += nthreads) {
      TapX t[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = 4 * g + j;
        if (x < p.dst_w) {
          int4 e = __ldg(reinterpret_cast<const int4*>(xt) + x);
          t[j] = *reinterpret_cast<TapX*>(&e);
        } else {
          t[j].off0 = -1;
        }
      }
      int v[4][3];
      if (pad_row) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j][0] = v[j][1] = v[j][2] = 114;
      } else {
        nv12_px4_general<MASK>(t, y0, c0, y1, c1, m0, m1, ty.b0, ty.b1, v);
      }
      store_px4<FMT>(optr + (size_t)(g - (int)threadIdx.x) * 4 * (nhwc ? 3 : esize), plane, vec_ok,
                     min(4, p.dst_w - 4 * g), v);
    }
    if (!pad_row) __syncthreads();
    s = s + 1 == S ? 0 : s + 1;
  }
  TIMELINE_END(p.dbg, 42);
}

// ---- host side ---------------------------------------------------------------------------

struct TapKey {
  int axis, src, dst_new, pad, dst_full;
  bool operator<(const TapKey& o) const {
    return std::tie(axis, src, dst_new, pad, dst_full) < std::tie(o.axis, o.src, o.dst_new, o.pad, o.dst_full);
  }
};

}  // namespace

struct TapCache {
  int4* arena = nullptr;  // device
  size_t capacity = 0;    // entries
  size_t used = 0;
  struct Entry {
    int off;
    bool single;  // y tables: no row ever needs the second source row (all b1 == 0)
  };
  std::map<TapKey, Entry> index;
};

static const size_t kTapArenaEntries = (size_t)1 << 19;  // 8 MiB of 16-byte entries

int tap_cache_create(b200va_ctx* h) {
  h->taps = new TapCache();
  h->taps->capacity = kTapArenaEntries;
  CUDA_TRY(h, cudaMalloc(&h->taps->arena, kTapArenaEntries * sizeof(int4)));
  return B200VA_OK;
}

void tap_cache_destroy(b200va_ctx* h) {
  if (!h->taps) return;
  if (h->taps->arena) cudaFree(h->taps->arena);
  delete h->taps;
  h->taps = nullptr;
}

// One axis of cv::resize's 8-bit linear tap table (OpenCV resize.cpp, restated; see
// oracle/cv_restate.py linear_taps).  clamp_frac = x axis.
static void linear_tap(int src, int dst, int d, bool clamp_frac, int* i0, int* i1, short* c0, short* c1) {
  const double inv = (double)dst / (double)src;
  const double scale = 1.0 / inv;
  float fx = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(fx);
  fx -= (float)s;
  if (clamp_frac) {
    if (s < 0) {
      fx = 0.f;
      s = 0;
    }
    if (s >= src - 1) {
      fx = 0.f;
      s = src - 1;
    }
  }
  const float one_minus = 1.f - fx;
  *c0 = (short)lrintf(one_minus * 2048.f);  // cvRound: round-half-even
  *c1 = (short)lrintf(fx * 2048.f);
  int a = s < 0 ? 0 : (s > src - 1 ? src - 1 : s);
  int b = s + 1 < 0 ? 0 : (s + 1 > src - 1 ? src - 1 : s + 1);
  *i0 = a;
  *i1 = b;
}

// Returns the arena offset of the table, building and uploading it on first use.
static int get_table(b200va_ctx* h, int axis, int src, int dst_new, int pad, int dst_full, int* off_out,
                     bool* single_out) {
  TapCache* tc = h->taps;
  TapKey key{axis, src, dst_new, pad, dst_full};
  auto it = tc->index.find(key);
  if (it != tc->index.end()) {
    *off_out = it->second.off;
    if (single_out) *single_out = it->second.single;
    return B200VA_OK;
  }
  if (tc->used + (size_t)dst_full > tc->capacity) {
    // arena full: drop every cached table (synchronise first, launches may still read them)
    CUDA_TRY(h, cudaDeviceSynchronize());
    tc->index.clear();
    tc->used = 0;
    if ((size_t)dst_full > tc->capacity) return set_error(h, B200VA_ERR_CAPACITY, "tap table of %d entries does not fit", dst_full);
  }
  std::vector<int4> host((size_t)dst_full);
  bool single = true;
  for (int d = 0; d < dst_full; ++d) {
    const int k = d - pad;
    if (axis == 0) {
      TapX t;
      if (k < 0 || k >= dst_new) {
        t.off0 = t.off1 = -1;
        t.a0 = t.a1 = 0;
        t.mx0 = 0;
      } else {
        int i0, i1;
        linear_tap(src, dst_new, k, true, &i0, &i1, &t.a0, &t.a1);
        t.off0 = 3 * i0;
        t.off1 = 3 * i1;
        t.mx0 = i0 | (i1 << 16);
      }
      memcpy(&host[d], &t, sizeof(int4));
    } else {
      TapY t;
      t.pad_ = 0;
      if (k < 0 || k >= dst_new) {
        t.y0 = t.y1 = -1;
        t.b0 = t.b1 = 0;
      } else {
        linear_tap(src, dst_new, k, false, &t.y0, &t.y1, &t.b0, &t.b1);
        if (t.b1 != 0) single = false;
      }
      memcpy(&host[d], &t, sizeof(int4));
    }
  }
  const int off = (int)tc->used;
  // synchronous copy: the table is visible to every stream once this returns
  CUDA_TRY(h, cudaMemcpy(tc->arena + off, host.data(), host.size() * sizeof(int4), cudaMemcpyHostToDevice));
  tc->used += (size_t)dst_full;
  tc->index[key] = TapCache::Entry{off, single};
  *off_out = off;
  if (single_out) *single_out = single;
  return B200VA_OK;
}

// Auxiliary int tables for the fused pass, cached in the same arena under axis ids 2 (rowmap) and 3 (colstart).
static int get_aux_table(b200va_ctx* h, int axis, int src, int dst_new, int pad, int dst_full, int* off_out, bool* ok_out) {
  TapCache* tc = h->taps;
  TapKey key{axis, src, dst_new, pad, dst_full};
  auto it = tc->index.find(key);
  if (it != tc->index.end()) {
    *off_out = it->second.off;
    *ok_out = it->second.single;
    return B200VA_OK;
  }
  std::vector<int> vals;
  bool ok = true;
  if (axis == 2) {  // rowmap
    vals.assign((size_t)src, -1);
    int prev_y0 = -1;
    for (int k = 0; k < dst_new; ++k) {
      int y0, y1;
      short b0, b1;
      linear_tap(src, dst_new, k, false, &y0, &y1, &b0, &b1);
      if (!(y0 > prev_y0) || !(b1 == 0 || y1 == y0 + 1) || y0 < 0 || y0 >= src) ok = false;
      else vals[(size_t)y0] = k + pad;
      prev_y0 = y0;
    }
  } else {  // colstart
    const int strips = (src + 255) / 256;
    vals.assign((size_t)strips + 1, pad + dst_new);
    int prev_x0 = -1, s_next = 0;
    for (int k = 0; k < dst_new; ++k) {
      int x0, x1;
      short a0, a1;
      linear_tap(src, dst_new, k, true, &x0, &x1, &a0, &a1);
      if (x0 < prev_x0 || !(a1 == 0 || x1 == x0 + 1 || x1 == x0)) ok = false;
      prev_x0 = x0;
      while (s_next <= strips && s_next * 256 <= x0) vals[(size_t)s_next++] = k + pad;
    }
  }
  const size_t entries = (vals.size() + 3) / 4;
  vals.resize(entries * 4, -1);
  if (tc->used + entries > tc->capacity) {
    CUDA_TRY(h, cudaDeviceSynchronize());
    tc->index.clear();
    tc->used = 0;
    if (entries > tc->capacity) return set_error(h, B200VA_ERR_CAPACITY, "table of %zu entries does not fit", entries);
  }
  const int off = (int)tc->used;
  CUDA_TRY(h, cudaMemcpy(tc->arena + off, vals.data(), entries * sizeof(int4), cudaMemcpyHostToDevice));
  tc->used += entries;
  tc->index[key] = TapCache::Entry{off, ok};
  *off_out = off;
  *ok_out = ok;
  return B200VA_OK;
}

int letterbox_fuse_plan(b200va_ctx* h, int src_h, int src_w, int new_h, int new_w, int pad_top, int pad_left, int dst_h,
                        int dst_w, FusePlan* out) {
  bool ok_r = false, ok_c = false;
  // the aux tables first: they may reset the arena, the tap tables fetched after them stay valid
  int rc = get_aux_table(h, 2, src_h, new_h, pad_top, dst_h, &out->rowmap, &ok_r);
  if (rc) return rc;
  rc = get_aux_table(h, 3, src_w, new_w, pad_left, dst_w, &out->colstart, &ok_c);
  if (rc) return rc;
  rc = get_table(h, 0, src_w, new_w, pad_left, dst_w, &out->xtab, nullptr);
  if (rc) return rc;
  rc = get_table(h, 1, src_h, new_h, pad_top, dst_h, &out->ytab, nullptr);
  if (rc) return rc;
  // a reset in between would have dropped the earlier offsets: make sure all four are still cached
  TapCache* tc = h->taps;
  const bool all_cached = tc->index.count(TapKey{2, src_h, new_h, pad_top, dst_h}) && tc->index.count(TapKey{3, src_w, new_w, pad_left, dst_w}) &&
                          tc->index.count(TapKey{0, src_w, new_w, pad_left, dst_w}) && tc->index.count(TapKey{1, src_h, new_h, pad_top, dst_h});
  out->eligible = ok_r && ok_c && all_cached;
  return B200VA_OK;
}

const int4* tap_arena(b200va_ctx* h) { return h->taps->arena; }

extern "C" int b200va_letterbox_meta(int src_h, int src_w, int dst_h, int dst_w, b200va_letterbox* out) {
  if (!out || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0) return B200VA_ERR_INVALID;
  const double sw = (double)dst_w / (double)src_w, sh = (double)dst_h / (double)src_h;
  const double scale = sw < sh ? sw : sh;        // min(target_w / w, target_h / h), detector.py:211
  out->src_h = src_h;
  out->src_w = src_w;
  out->new_w = (int)((double)src_w * scale);     // int() truncation, detector.py:214-215
  out->new_h = (int)((double)src_h * scale);
  out->pad_left = (dst_w - out->new_w) / 2;      // pad // 2, detector.py:228-230 (pads are >= 0)
  out->pad_top = (dst_h - out->new_h) / 2;
  out->scale = scale;
  return B200VA_OK;
}

// pdl: launch as a programmatic dependent of the kernel before it in the stream WITHOUT ever waiting for it
// (b200va_tick schedule 3: the letterbox shares no data with the decode kernel it follows, it only wants to start
// filling the SMs that kernel leaves free)
template <int FMT, bool MASK>
static cudaError_t launch_one(const PreParams& p, dim3 grid, size_t smem, cudaStream_t st, bool pdl) {
  return launch_pdl(k_letterbox<FMT, MASK>, grid, dim3(kThreads), smem, st, pdl, p);
}

template <int FMT, bool MASK>
static cudaError_t launch_one(const PreParamsNv12& p, dim3 grid, size_t smem, cudaStream_t st, bool pdl) {
  return launch_pdl(k_letterbox_nv12<FMT, MASK>, grid, dim3(kThreads), smem, st, pdl, p);
}

template <int FMT, typename P>
static cudaError_t launch_letterbox(const P& p, bool mask, dim3 grid, size_t smem, cudaStream_t st, bool pdl) {
  return mask ? launch_one<FMT, true>(p, grid, smem, st, pdl) : launch_one<FMT, false>(p, grid, smem, st, pdl);
}

static const int kLetterboxSmemMax = 200 * 1024;

template <typename K>
static cudaError_t configure_kernel(K kernel, bool uniform_carveout) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLetterboxSmemMax + 128);
  if (e != cudaSuccess || !uniform_carveout) return e;
  return prefer_max_shared(kernel);
}

template <int FMT>
static cudaError_t configure_fmt(bool uniform_carveout) {
  cudaError_t e = configure_kernel(k_letterbox<FMT, false>, uniform_carveout);
  if (e == cudaSuccess) e = configure_kernel(k_letterbox<FMT, true>, uniform_carveout);
  if (e == cudaSuccess) e = configure_kernel(k_letterbox_nv12<FMT, false>, uniform_carveout);
  if (e == cudaSuccess) e = configure_kernel(k_letterbox_nv12<FMT, true>, uniform_carveout);
  return e;
}

int preprocess_configure(b200va_ctx* h) {
  CUDA_TRY(h, configure_fmt<B200VA_OUT_F32_RGB_NCHW>(h->tune.uniform_carveout != 0));
  CUDA_TRY(h, configure_fmt<B200VA_OUT_F16_RGB_NCHW>(h->tune.uniform_carveout != 0));
  CUDA_TRY(h, configure_fmt<B200VA_OUT_U8_BGR_NCHW>(h->tune.uniform_carveout != 0));
  CUDA_TRY(h, configure_fmt<B200VA_OUT_U8_BGR_NHWC>(h->tune.uniform_carveout != 0));
  return B200VA_OK;
}

// The source frames of one resample call: packed BGR (frames + pitches) or NV12 planes.
struct SrcFrames {
  const uint8_t* const* bgr = nullptr;
  const int64_t* pitch = nullptr;         // BGR row pitches (NULL = 3 * w)
  const b200va_nv12_frame* nv12 = nullptr;
};

// Fills the source fields of one frame descriptor; returns the bytes of one staged source row (-1: refused).
static int set_source(b200va_ctx* h, const SrcFrames& src, int b, int src_h, int src_w, PreFrame& f) {
  REQUIRE(h, src.bgr[b] != nullptr, "frame %d is NULL", b);
  const int64_t pitch = src.pitch ? src.pitch[b] : (int64_t)3 * src_w;
  REQUIRE(h, pitch >= (int64_t)3 * src_w, "frame %d: pitch %lld < 3*width", b, (long long)pitch);
  f.src = src.bgr[b];
  f.pitch = pitch;
  const int rb = 3 * src_w;
  f.bulk_ok = ((uintptr_t)f.src % 16 == 0) && (pitch % 16 == 0) && (rb % 16 == 0);
  return B200VA_OK;
}

static int set_source(b200va_ctx* h, const SrcFrames& src, int b, int src_h, int src_w, Nv12Frame& f) {
  const b200va_nv12_frame& n = src.nv12[b];
  REQUIRE(h, n.y != nullptr && n.uv != nullptr, "frame %d: NULL plane", b);
  REQUIRE(h, src_h % 2 == 0 && src_w % 2 == 0, "frame %d: NV12 needs an even size, got %dx%d", b, src_w, src_h);
  REQUIRE(h, n.y_pitch >= src_w && n.uv_pitch >= src_w, "frame %d: plane pitch %lld / %lld < width %d", b,
          (long long)n.y_pitch, (long long)n.uv_pitch, src_w);
  f.y = n.y;
  f.uv = n.uv;
  f.y_pitch = n.y_pitch;
  f.uv_pitch = n.uv_pitch;
  f.bulk_ok = ((uintptr_t)n.y % 16 == 0) && ((uintptr_t)n.uv % 16 == 0) && (n.y_pitch % 16 == 0) && (n.uv_pitch % 16 == 0) &&
              (src_w % 16 == 0);
  return B200VA_OK;
}

// Shared by b200va_preprocess* (letterbox geometry) and b200va_resize_linear_u8* (no padding).
// Frames with and without an ROI mask go to separate launches (the mask is a template switch).
// P = PreParams (BGR frames, k_letterbox) or PreParamsNv12 (NV12 frames, k_letterbox_nv12).
template <typename P>
static int run_resample(b200va_ctx* h, const SrcFrames& src, const int* src_h, const int* src_w, int batch,
                        const uint8_t* const* roi_masks, void* out, const int* new_h, const int* new_w, const int* pad_top,
                        const int* pad_left, int dst_h, int dst_w, int fmt_and_flags, cudaStream_t st,
                        uint8_t* const* outs = nullptr) {
  constexpr bool kNv12 = std::is_same<P, PreParamsNv12>::value;
  constexpr int kGroup = kNv12 ? kNv12LaunchFrames : B200VA_LAUNCH_FRAMES;
  const int fmt = fmt_and_flags & 0xff;
  REQUIRE(h, fmt >= 0 && fmt <= 3 && (fmt_and_flags & ~(0xff | B200VA_OUT_FLAG_PADS_VALID)) == 0, "unknown output format %d",
          fmt_and_flags);
  PhaseScope phase(h, outs ? B200VA_PHASE_RESIZE : B200VA_PHASE_PREPROCESS, st);
  std::vector<int> order[2];
  for (int b = 0; b < batch; ++b) order[(roi_masks && roi_masks[b]) ? 1 : 0].push_back(b);
  for (int with_mask = 0; with_mask < 2; ++with_mask) {
    const std::vector<int>& idx = order[with_mask];
    for (size_t base = 0; base < idx.size(); base += kGroup) {
      const int n = (int)std::min<size_t>(kGroup, idx.size() - base);
      P p;
      memset(&p, 0, sizeof(p));
      int max_row = 0, max_w = 0;
      bool all_single = true;
      for (int i = 0; i < n; ++i) {
        const int b = idx[base + i];
        auto& f = p.f[i];
        REQUIRE(h, src_h[b] > 0 && src_w[b] > 0 && src_w[b] < 65536, "frame %d has unsupported size %dx%d", b, src_w[b], src_h[b]);
        int rc = set_source(h, src, b, src_h[b], src_w[b], f);
        if (rc) return rc;
        REQUIRE(h, new_h[b] > 0 && new_w[b] > 0, "frame %d: resized size %dx%d is empty (cv2.resize would raise)", b, new_w[b], new_h[b]);
        f.mask = with_mask ? roi_masks[b] : nullptr;
        f.src_h = src_h[b];
        f.src_w = src_w[b];
        f.out_idx = b;
        f.out = outs ? outs[b] : nullptr;
        bool single = true;
        rc = get_table(h, 0, src_w[b], new_w[b], pad_left[b], dst_w, &f.xtab, nullptr);
        if (rc) return rc;
        rc = get_table(h, 1, src_h[b], new_h[b], pad_top[b], dst_h, &f.ytab, &single);
        if (rc) return rc;
        all_single = all_single && single;
        const int rb = (kNv12 ? 1 : 3) * src_w[b];  // one staged source row (NV12: a luma row, and a chroma row as long)
        f.bulk_ok = f.bulk_ok && (!f.mask || (((uintptr_t)f.mask % 16 == 0) && (src_w[b] % 16 == 0)));
        if (rb > max_row) max_row = rb;
        if (src_w[b] > max_w) max_w = src_w[b];
      }
      p.tabs = h->taps->arena;
      p.dbg = h->dbg;
      p.skip = outs ? nullptr : h->skip_dev;  // the downsample runs before the gates (pipeline.py:152-154)
      p.pdl_wait = (h->pdl_preprocess && h->pdl_preprocess_wait) ? 1 : 0;
      p.out = out;
      p.dst_h = dst_h;
      p.dst_w = dst_w;
      p.fmt = fmt;
      p.keep_pad_rows = (fmt_and_flags & B200VA_OUT_FLAG_PADS_VALID) ? 1 : 0;
      p.row_stride = (max_row + 127) & ~127;
      p.mask_stride = with_mask ? ((max_w + 127) & ~127) : 0;
      p.rows_per_stage = all_single ? 1 : 2;
      // an NV12 stage holds each luma row and its chroma row: 2 * src_w bytes per tapped row against 3 * src_w
      const size_t per_stage = (size_t)p.rows_per_stage * ((kNv12 ? 2 : 1) * (size_t)p.row_stride + p.mask_stride);
      // ring depth: up to kMaxStages, but shallow enough that several CTAs share an SM -- with whole 4K rows a
      // 4-deep ring is 90-120 KB and leaves ONE 160-thread CTA per SM (7.6 % warps active, 0.59 of HBM peak)
      // (measured, 32 x 4K + ROI: 133 us with the deepest ring, 84 us = 0.94 of peak with a 32-56 KB budget)
      const size_t budget = (size_t)48 * 1024;
      int stages = (int)(budget / per_stage);
      if (stages < 2) stages = 2;
      if ((size_t)stages * per_stage > (size_t)kLetterboxSmemMax) stages = (int)((size_t)kLetterboxSmemMax / per_stage);
      if (stages > kMaxStages) stages = kMaxStages;
      REQUIRE(h, stages >= 1, "source rows of %d bytes do not fit in shared memory", max_row);
      p.stages = stages;
      // enough CTAs for several waves over the SMs, few enough that the tap registers amortise
      const long long total_rows = (long long)n * dst_h;
      int rpc = (int)(total_rows / ((long long)h->num_sms * 16));
      if (rpc < 2) rpc = 2;
      if (rpc > kMaxRowsPerCta) rpc = kMaxRowsPerCta;
      p.rows_per_cta = rpc;
      const uintptr_t ob = (uintptr_t)out;
      const size_t frame_elems = (size_t)3 * dst_h * dst_w;
      switch (fmt) {
        case B200VA_OUT_F32_RGB_NCHW: p.vec_ok = (dst_w % 4 == 0) && (ob % 16 == 0); break;
        case B200VA_OUT_F16_RGB_NCHW: p.vec_ok = (dst_w % 4 == 0) && (ob % 8 == 0); break;
        default: p.vec_ok = (dst_w % 4 == 0) && (ob % 4 == 0) && (frame_elems % 4 == 0); break;
      }
      if (outs)  // per-frame destinations: every one of them has to allow the vector stores
        for (int i = 0; i < n; ++i)
          if ((uintptr_t)outs[idx[base + i]] % 16 != 0) p.vec_ok = 0;
      dim3 grid((dst_h + rpc - 1) / rpc, n);
      // (taps_row reads up to 8 bytes past the end of a row.)  The floor keeps at most six CTAs on an SM: with the 48
      // registers the kernel needs since the word-load taps, eight would fit, and the 32 x 1080p launch is 5 % slower
      // that way (43.2 against 41.4 us: more rows in flight than the memory system wants; the same was measured in
      // round 1 by forcing 7 / 8 CTAs per SM with __launch_bounds__).
      const size_t smem = std::max((size_t)stages * per_stage + 16, (size_t)std::max(h->tune.lb_smem_floor, 0));
      cudaError_t e;
      const bool pdl = h->pdl_preprocess && h->tune.pdl != 0;
      h->pdl_preprocess = false;  // only the first launch of the call directly follows the decode kernel
      switch (fmt) {
        case B200VA_OUT_F32_RGB_NCHW: e = launch_letterbox<B200VA_OUT_F32_RGB_NCHW>(p, with_mask, grid, smem, st, pdl); break;
        case B200VA_OUT_F16_RGB_NCHW: e = launch_letterbox<B200VA_OUT_F16_RGB_NCHW>(p, with_mask, grid, smem, st, pdl); break;
        case B200VA_OUT_U8_BGR_NCHW: e = launch_letterbox<B200VA_OUT_U8_BGR_NCHW>(p, with_mask, grid, smem, st, pdl); break;
        default: e = launch_letterbox<B200VA_OUT_U8_BGR_NHWC>(p, with_mask, grid, smem, st, pdl); break;
      }
      h->launches.fetch_add(1, std::memory_order_relaxed);
      if (e != cudaSuccess) return set_error(h, B200VA_ERR_CUDA, "letterbox launch failed: %s", cudaGetErrorString(e));
    }
  }
  return B200VA_OK;
}

static int run_resample(b200va_ctx* h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                        const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks, void* out,
                        const int* new_h, const int* new_w, const int* pad_top, const int* pad_left, int dst_h,
                        int dst_w, int fmt_and_flags, cudaStream_t st, uint8_t* const* outs = nullptr) {
  SrcFrames src;
  src.bgr = frames;
  src.pitch = src_pitch;
  return run_resample<PreParams>(h, src, src_h, src_w, batch, roi_masks, out, new_h, new_w, pad_top, pad_left, dst_h, dst_w,
                                 fmt_and_flags, st, outs);
}

extern "C" int b200va_preprocess(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                 const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks, void* out,
                                 int dst_h, int dst_w, int out_format, b200va_letterbox* meta_out, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && out, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  REQUIRE(h, dst_h > 0 && dst_w > 0 && dst_w < 65536, "bad destination size %dx%d", dst_w, dst_h);
  if (batch == 0) return B200VA_OK;
  std::vector<int> nh(batch), nw(batch), pt(batch), pl(batch);
  for (int b = 0; b < batch; ++b) {
    b200va_letterbox m;
    REQUIRE(h, b200va_letterbox_meta(src_h[b], src_w[b], dst_h, dst_w, &m) == B200VA_OK, "frame %d: bad size %dx%d", b, src_w[b], src_h[b]);
    nh[b] = m.new_h;
    nw[b] = m.new_w;
    pt[b] = m.pad_top;
    pl[b] = m.pad_left;
    if (meta_out) meta_out[b] = m;
  }
  return run_resample(h, frames, src_h, src_w, src_pitch, batch, roi_masks, out, nh.data(), nw.data(), pt.data(),
                      pl.data(), dst_h, dst_w, out_format, (cudaStream_t)stream);
}

// ultralytics LetterBox.__call__ (data/augment.py; scaleup = True, center = True): sizes are ROUNDED
// (Python round = round-half-even = nearbyint), the padding is split with round(d / 2 -+ 0.1), and with
// auto = True only the remainder modulo `stride` is padded (the "rect" shape predict() uses for a single image).
extern "C" int b200va_letterbox_meta_ultralytics(int src_h, int src_w, int dst_h, int dst_w, int auto_pad, int stride,
                                                 b200va_letterbox* out, int* out_h, int* out_w) {
  if (!out || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0 || (auto_pad && stride <= 0)) return B200VA_ERR_INVALID;
  const double r0 = (double)dst_h / (double)src_h, r1 = (double)dst_w / (double)src_w;
  const double r = r0 < r1 ? r0 : r1;
  const int new_w = (int)nearbyint((double)src_w * r), new_h = (int)nearbyint((double)src_h * r);
  if (new_w <= 0 || new_h <= 0) return B200VA_ERR_INVALID;
  int dwi = dst_w - new_w, dhi = dst_h - new_h;
  if (auto_pad) {
    dwi %= stride;  // np.mod of non-negative integers
    dhi %= stride;
  }
  const double dw = dwi / 2.0, dh = dhi / 2.0;
  const int top = (int)nearbyint(dh - 0.1), bottom = (int)nearbyint(dh + 0.1);
  const int left = (int)nearbyint(dw - 0.1), right = (int)nearbyint(dw + 0.1);
  out->src_h = src_h;
  out->src_w = src_w;
  out->new_h = new_h;
  out->new_w = new_w;
  out->pad_left = left;
  out->pad_top = top;
  out->scale = r;
  if (out_h) *out_h = new_h + top + bottom;
  if (out_w) *out_w = new_w + left + right;
  return B200VA_OK;
}

// b200va_preprocess_geom*: the caller's geometry must describe each frame and fit the dst_h x dst_w canvas.
template <typename P>
static int preprocess_geom_impl(b200va_handle h, const SrcFrames& src, const int* src_h, const int* src_w, int batch,
                                const uint8_t* const* roi_masks, const b200va_letterbox* geom, void* out, int dst_h,
                                int dst_w, int out_format, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, (src.bgr || src.nv12) && src_h && src_w && out && geom, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  REQUIRE(h, dst_h > 0 && dst_w > 0 && dst_w < 65536, "bad destination size %dx%d", dst_w, dst_h);
  if (batch == 0) return B200VA_OK;
  std::vector<int> nh(batch), nw(batch), pt(batch), pl(batch);
  for (int b = 0; b < batch; ++b) {
    const b200va_letterbox& m = geom[b];
    REQUIRE(h, m.src_h == src_h[b] && m.src_w == src_w[b], "frame %d: geometry is for %dx%d, frame is %dx%d", b, m.src_w,
            m.src_h, src_w[b], src_h[b]);
    REQUIRE(h, m.new_h > 0 && m.new_w > 0 && m.pad_top >= 0 && m.pad_left >= 0 && m.pad_top + m.new_h <= dst_h &&
                   m.pad_left + m.new_w <= dst_w,
            "frame %d: resized %dx%d at (%d, %d) does not fit %dx%d", b, m.new_w, m.new_h, m.pad_left, m.pad_top, dst_w, dst_h);
    nh[b] = m.new_h;
    nw[b] = m.new_w;
    pt[b] = m.pad_top;
    pl[b] = m.pad_left;
  }
  return run_resample<P>(h, src, src_h, src_w, batch, roi_masks, out, nh.data(), nw.data(), pt.data(), pl.data(), dst_h,
                         dst_w, out_format, (cudaStream_t)stream);
}

extern "C" int b200va_preprocess_geom(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                      const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks,
                                      const b200va_letterbox* geom, void* out, int dst_h, int dst_w, int out_format,
                                      void* stream) {
  SrcFrames src;
  src.bgr = frames;
  src.pitch = src_pitch;
  return preprocess_geom_impl<PreParams>(h, src, src_h, src_w, batch, roi_masks, geom, out, dst_h, dst_w, out_format, stream);
}

extern "C" int b200va_preprocess_geom_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                           const int* src_w, int batch, const uint8_t* const* roi_masks,
                                           const b200va_letterbox* geom, void* out, int dst_h, int dst_w, int out_format,
                                           void* stream) {
  SrcFrames src;
  src.nv12 = frames;
  return preprocess_geom_impl<PreParamsNv12>(h, src, src_h, src_w, batch, roi_masks, geom, out, dst_h, dst_w, out_format,
                                             stream);
}

extern "C" int b200va_resize_linear_u8(b200va_handle h, const uint8_t* const* frames, const int* src_h,
                                       const int* src_w, const int64_t* src_pitch, int batch,
                                       const uint8_t* const* roi_masks, uint8_t* const* dst, const int* dst_h,
                                       const int* dst_w, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && dst && dst_h && dst_w, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  // frames that share a destination size go out in ONE launch (per-frame destination pointers); a batch of
  // streams with the same downsample ratio is one launch, not one per stream
  std::map<std::pair<int, int>, std::vector<int>> groups;
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, dst[b] != nullptr, "dst %d is NULL", b);
    REQUIRE(h, dst_h[b] > 0 && dst_w[b] > 0 && dst_w[b] < 65536, "frame %d: bad destination size %dx%d", b, dst_w[b], dst_h[b]);
    groups[{dst_h[b], dst_w[b]}].push_back(b);
  }
  for (const auto& kv : groups) {
    const std::vector<int>& idx = kv.second;
    const int n = (int)idx.size();
    std::vector<const uint8_t*> g_frames(n), g_masks(n);
    std::vector<uint8_t*> g_out(n);
    std::vector<int> g_h(n), g_w(n), g_nh(n, kv.first.first), g_nw(n, kv.first.second), g_zero(n, 0);
    std::vector<int64_t> g_pitch(n);
    bool any_mask = false;
    for (int i = 0; i < n; ++i) {
      const int b = idx[i];
      g_frames[i] = frames[b];
      g_masks[i] = roi_masks ? roi_masks[b] : nullptr;
      any_mask = any_mask || g_masks[i] != nullptr;
      g_out[i] = dst[b];
      g_h[i] = src_h[b];
      g_w[i] = src_w[b];
      g_pitch[i] = src_pitch ? src_pitch[b] : (int64_t)3 * src_w[b];
    }
    int rc = run_resample(h, g_frames.data(), g_h.data(), g_w.data(), g_pitch.data(), n, any_mask ? g_masks.data() : nullptr,
                          g_out[0], g_nh.data(), g_nw.data(), g_zero.data(), g_zero.data(), kv.first.first, kv.first.second,
                          B200VA_OUT_U8_BGR_NHWC, (cudaStream_t)stream, g_out.data());
    if (rc) return rc;
  }
  return B200VA_OK;
}

extern "C" int b200va_preprocess_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h, const int* src_w,
                                      int batch, const uint8_t* const* roi_masks, void* out, int dst_h, int dst_w,
                                      int out_format, b200va_letterbox* meta_out, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && out, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  REQUIRE(h, dst_h > 0 && dst_w > 0 && dst_w < 65536, "bad destination size %dx%d", dst_w, dst_h);
  if (batch == 0) return B200VA_OK;
  std::vector<int> nh(batch), nw(batch), pt(batch), pl(batch);
  for (int b = 0; b < batch; ++b) {
    b200va_letterbox m;
    REQUIRE(h, b200va_letterbox_meta(src_h[b], src_w[b], dst_h, dst_w, &m) == B200VA_OK, "frame %d: bad size %dx%d", b, src_w[b], src_h[b]);
    nh[b] = m.new_h;
    nw[b] = m.new_w;
    pt[b] = m.pad_top;
    pl[b] = m.pad_left;
    if (meta_out) meta_out[b] = m;
  }
  SrcFrames src;
  src.nv12 = frames;
  return run_resample<PreParamsNv12>(h, src, src_h, src_w, batch, roi_masks, out, nh.data(), nw.data(), pt.data(), pl.data(),
                                     dst_h, dst_w, out_format, (cudaStream_t)stream);
}

extern "C" int b200va_resize_linear_u8_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                            const int* src_w, int batch, const uint8_t* const* roi_masks,
                                            uint8_t* const* dst, const int* dst_h, const int* dst_w, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && dst && dst_h && dst_w, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  // frames that share a destination size go out in one launch, as in b200va_resize_linear_u8
  std::map<std::pair<int, int>, std::vector<int>> groups;
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, dst[b] != nullptr, "dst %d is NULL", b);
    REQUIRE(h, dst_h[b] > 0 && dst_w[b] > 0 && dst_w[b] < 65536, "frame %d: bad destination size %dx%d", b, dst_w[b], dst_h[b]);
    groups[{dst_h[b], dst_w[b]}].push_back(b);
  }
  for (const auto& kv : groups) {
    const std::vector<int>& idx = kv.second;
    const int n = (int)idx.size();
    std::vector<b200va_nv12_frame> g_frames(n);
    std::vector<const uint8_t*> g_masks(n);
    std::vector<uint8_t*> g_out(n);
    std::vector<int> g_h(n), g_w(n), g_nh(n, kv.first.first), g_nw(n, kv.first.second), g_zero(n, 0);
    bool any_mask = false;
    for (int i = 0; i < n; ++i) {
      const int b = idx[i];
      g_frames[i] = frames[b];
      g_masks[i] = roi_masks ? roi_masks[b] : nullptr;
      any_mask = any_mask || g_masks[i] != nullptr;
      g_out[i] = dst[b];
      g_h[i] = src_h[b];
      g_w[i] = src_w[b];
    }
    SrcFrames src;
    src.nv12 = g_frames.data();
    int rc = run_resample<PreParamsNv12>(h, src, g_h.data(), g_w.data(), n, any_mask ? g_masks.data() : nullptr, g_out[0],
                                         g_nh.data(), g_nw.data(), g_zero.data(), g_zero.data(), kv.first.first,
                                         kv.first.second, B200VA_OUT_U8_BGR_NHWC, (cudaStream_t)stream, g_out.data());
    if (rc) return rc;
  }
  return B200VA_OK;
}

// ---- host -> device staging of decoded frames ---------------------------------------------------
// The letterbox reads only the source rows that carry a non-zero vertical weight (every third row
// for 1080p -> 640x360, two rows in six for 4K).  With rows_mode = 1 only those rows cross PCIe, into
// their original positions of the device frame, as one strided 2-D DMA per frame; the kernels then
// run unchanged.  Frames that feed the motion gate or a downsample need every row (rows_mode = 0).
namespace {
struct RowPattern {
  bool regular = false;  // needed rows = runs of `run` rows every `period` rows starting at `first`
  int first = 0, run = 0, period = 0, count = 0;
};
std::map<std::pair<int, int>, RowPattern> g_row_patterns;
std::mutex g_row_mu;

// The source rows a letterbox that resizes src_h rows to new_h reads: those with a non-zero vertical tap weight.
std::vector<char> tapped_rows(int src_h, int new_h) {
  std::vector<char> need((size_t)src_h, 0);
  for (int d = 0; d < new_h; ++d) {
    int y0, y1;
    short b0, b1;
    linear_tap(src_h, new_h, d, false, &y0, &y1, &b0, &b1);
    if (b0) need[y0] = 1;
    if (b1) need[y1] = 1;
  }
  return need;
}

RowPattern needed_rows(int src_h, int new_h) {
  std::lock_guard<std::mutex> lock(g_row_mu);
  auto key = std::make_pair(src_h, new_h);
  auto it = g_row_patterns.find(key);
  if (it != g_row_patterns.end()) return it->second;
  const std::vector<char> need = tapped_rows(src_h, new_h);
  std::vector<std::pair<int, int>> runs;  // (start, length)
  for (int y = 0; y < src_h;) {
    if (!need[y]) {
      ++y;
      continue;
    }
    int e = y;
    while (e < src_h && need[e]) ++e;
    runs.push_back({y, e - y});
    y = e;
  }
  RowPattern rp;
  if (!runs.empty()) {
    rp.regular = true;
    rp.first = runs[0].first;
    rp.run = runs[0].second;
    rp.count = (int)runs.size();
    rp.period = runs.size() > 1 ? runs[1].first - runs[0].first : rp.run;
    for (size_t i = 0; i < runs.size(); ++i)
      if (runs[i].second != rp.run || runs[i].first != rp.first + (int)i * rp.period) rp.regular = false;
    // nothing to gain when (nearly) every row is needed
    if ((long long)rp.run * rp.count * 10 > (long long)src_h * 8) rp.regular = false;
  }
  g_row_patterns[key] = rp;
  return rp;
}

// The resized height of each frame whose tapped rows alone are to be uploaded: from the reference geometry to
// dst_h x dst_w (geom == NULL) or from the caller's per-frame geometry.  Empty when rows_mode asks for every row.
int upload_heights(b200va_ctx* h, const int* src_h, const int* src_w, int batch, int dst_h, int dst_w, int rows_mode,
                   const b200va_letterbox* geom, std::vector<int>* new_h) {
  new_h->clear();
  if (rows_mode != 1) return B200VA_OK;
  REQUIRE(h, src_h && src_w, "NULL argument");
  REQUIRE(h, batch >= 0, "negative batch");
  new_h->resize(batch);
  for (int b = 0; b < batch; ++b) {
    if (geom) {
      const b200va_letterbox& m = geom[b];
      REQUIRE(h, m.src_h == src_h[b] && m.src_w == src_w[b] && m.new_h > 0, "frame %d: geometry is for %dx%d (new_h %d), frame is %dx%d",
              b, m.src_w, m.src_h, m.new_h, src_w[b], src_h[b]);
      (*new_h)[b] = m.new_h;
    } else {
      b200va_letterbox m;
      REQUIRE(h, b200va_letterbox_meta(src_h[b], src_w[b], dst_h, dst_w, &m) == B200VA_OK && m.new_h > 0, "frame %d: bad letterbox geometry", b);
      (*new_h)[b] = m.new_h;
    }
  }
  return B200VA_OK;
}
}  // namespace

namespace {
// One plane's needed rows as at most `max_runs` strided copies (start, step, count): from the first row not yet
// covered, the longest arithmetic progression through one of the next four such rows.  1080p -> 640 x 640 needs luma
// rows 1, 4, 7, ... (one progression) and chroma rows 0, 2, 3, 5, 6, ... = {0, 3, 6, ...} + {2, 5, 8, ...}.
// Returns false when the rows need more copies than that.
struct RowRun {
  int start, step, count;
};
bool row_progressions(const std::vector<char>& need, size_t max_runs, std::vector<RowRun>* out) {
  const int n = (int)need.size();
  std::vector<char> left(need);
  out->clear();
  for (int r = 0; r < n; ++r) {
    if (!left[r]) continue;
    if (out->size() == max_runs) return false;
    RowRun best{r, 1, 1};
    int tried = 0;
    for (int q = r + 1; q < n && tried < 4; ++q) {
      if (!left[q]) continue;
      ++tried;
      int count = 1;
      for (int y = q; y < n && left[y]; y += q - r) ++count;
      if (count > best.count) best = RowRun{r, q - r, count};
    }
    for (int k = 0; k < best.count; ++k) left[r + k * best.step] = 0;
    out->push_back(best);
  }
  return true;
}

// Copies the needed rows of one plane (every row when `need` is empty or the rows are too scattered to gain).
int copy_plane_rows(b200va_ctx* h, uint8_t* dst, int64_t dp, const uint8_t* src, int64_t hp, int64_t row_bytes, int rows,
                    const std::vector<char>& need, cudaStream_t st, int64_t* moved) {
  if (!need.empty()) {
    std::vector<RowRun> runs;
    int64_t n = 0;
    for (char c : need) n += c ? 1 : 0;
    // nothing to gain when (nearly) every row is needed
    if (n * 10 <= (int64_t)rows * 8 && row_progressions(need, 8, &runs)) {
      for (const RowRun& r : runs)
        CUDA_TRY(h, cudaMemcpy2DAsync(dst + (size_t)r.start * dp, (size_t)r.step * dp, src + (size_t)r.start * hp,
                                      (size_t)r.step * hp, (size_t)row_bytes, r.count, cudaMemcpyHostToDevice, st));
      *moved += n * row_bytes;
      return B200VA_OK;
    }
  }
  if (hp == row_bytes && dp == row_bytes)
    CUDA_TRY(h, cudaMemcpyAsync(dst, src, (size_t)row_bytes * rows, cudaMemcpyHostToDevice, st));
  else
    CUDA_TRY(h, cudaMemcpy2DAsync(dst, dp, src, hp, (size_t)row_bytes, rows, cudaMemcpyHostToDevice, st));
  *moved += row_bytes * rows;
  return B200VA_OK;
}
}  // namespace

// new_h empty: every row of every frame; else the rows the letterbox to new_h[b] rows reads.
static int upload_bgr(b200va_handle h, const uint8_t* const* host_frames, uint8_t* const* dev_frames, const int* src_h,
                      const int* src_w, const int64_t* host_pitch, const int64_t* dev_pitch, int batch,
                      const std::vector<int>& new_h, int64_t* bytes_copied, cudaStream_t st) {
  REQUIRE(h, host_frames && dev_frames && src_h && src_w, "NULL argument");
  REQUIRE(h, batch >= 0, "negative batch");
  PhaseScope phase(h, B200VA_PHASE_UPLOAD, st);
  int64_t total = 0;
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, host_frames[b] && dev_frames[b] && src_h[b] > 0 && src_w[b] > 0, "frame %d: bad arguments", b);
    const size_t rb = (size_t)3 * src_w[b];
    const size_t hp = host_pitch ? (size_t)host_pitch[b] : rb, dp = dev_pitch ? (size_t)dev_pitch[b] : rb;
    REQUIRE(h, hp >= rb && dp >= rb, "frame %d: pitch smaller than 3*width", b);
    RowPattern rp;
    if (!new_h.empty()) rp = needed_rows(src_h[b], new_h[b]);
    if (rp.regular) {
      if (hp == rb && dp == rb) {
        // a run of consecutive rows is one contiguous span
        CUDA_TRY(h, cudaMemcpy2DAsync(dev_frames[b] + (size_t)rp.first * dp, (size_t)rp.period * dp,
                                      host_frames[b] + (size_t)rp.first * hp, (size_t)rp.period * hp,
                                      (size_t)rp.run * rb, rp.count, cudaMemcpyHostToDevice, st));
      } else {
        for (int r = 0; r < rp.run; ++r)
          CUDA_TRY(h, cudaMemcpy2DAsync(dev_frames[b] + (size_t)(rp.first + r) * dp, (size_t)rp.period * dp,
                                        host_frames[b] + (size_t)(rp.first + r) * hp, (size_t)rp.period * hp, rb,
                                        rp.count, cudaMemcpyHostToDevice, st));
      }
      total += (int64_t)rp.run * rp.count * (int64_t)rb;
    } else {
      // irregular rows go as a few strided copies, like an NV12 plane (every row when they are too scattered)
      const int rc = copy_plane_rows(h, dev_frames[b], dp, host_frames[b], hp, rb, src_h[b],
                                     new_h.empty() ? std::vector<char>() : tapped_rows(src_h[b], new_h[b]), st, &total);
      if (rc) return rc;
    }
  }
  if (bytes_copied) *bytes_copied = total;
  return B200VA_OK;
}

extern "C" int b200va_upload_frames(b200va_handle h, const uint8_t* const* host_frames, uint8_t* const* dev_frames,
                                    const int* src_h, const int* src_w, const int64_t* host_pitch,
                                    const int64_t* dev_pitch, int batch, int dst_h, int dst_w, int rows_mode,
                                    int64_t* bytes_copied, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  std::vector<int> new_h;
  const int rc = upload_heights(h, src_h, src_w, batch, dst_h, dst_w, rows_mode, nullptr, &new_h);
  if (rc) return rc;
  return upload_bgr(h, host_frames, dev_frames, src_h, src_w, host_pitch, dev_pitch, batch, new_h, bytes_copied,
                    (cudaStream_t)stream);
}

extern "C" int b200va_upload_frames_geom(b200va_handle h, const uint8_t* const* host_frames, uint8_t* const* dev_frames,
                                         const int* src_h, const int* src_w, const int64_t* host_pitch,
                                         const int64_t* dev_pitch, int batch, const b200va_letterbox* geom,
                                         int64_t* bytes_copied, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, geom || batch == 0, "NULL geometry");
  std::vector<int> new_h;
  const int rc = upload_heights(h, src_h, src_w, batch, 0, 0, 1, geom, &new_h);
  if (rc) return rc;
  return upload_bgr(h, host_frames, dev_frames, src_h, src_w, host_pitch, dev_pitch, batch, new_h, bytes_copied,
                    (cudaStream_t)stream);
}

// new_h as in upload_bgr; a needed luma row brings the chroma row it uses.
static int upload_nv12(b200va_handle h, const b200va_nv12_frame* host, const b200va_nv12_frame* dev, const int* src_h,
                       const int* src_w, int batch, const std::vector<int>& new_h, int64_t* bytes_copied, cudaStream_t st) {
  REQUIRE(h, host && dev && src_h && src_w, "NULL argument");
  REQUIRE(h, batch >= 0, "negative batch");
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, host[b].y && host[b].uv && dev[b].y && dev[b].uv, "frame %d: NULL plane", b);
    REQUIRE(h, src_h[b] > 0 && src_w[b] > 0 && src_h[b] % 2 == 0 && src_w[b] % 2 == 0, "frame %d: NV12 needs an even size, got %dx%d",
            b, src_w[b], src_h[b]);
    REQUIRE(h, host[b].y_pitch >= src_w[b] && host[b].uv_pitch >= src_w[b] && dev[b].y_pitch >= src_w[b] &&
                   dev[b].uv_pitch >= src_w[b],
            "frame %d: plane pitch smaller than the width", b);
  }
  PhaseScope phase(h, B200VA_PHASE_UPLOAD, st);
  int64_t total = 0;
  for (int b = 0; b < batch; ++b) {
    const int H = src_h[b], W = src_w[b];
    std::vector<char> need_y, need_uv;
    if (!new_h.empty()) {
      need_y = tapped_rows(H, new_h[b]);
      need_uv.assign((size_t)H / 2, 0);
      for (int y = 0; y < H; ++y)
        if (need_y[y]) need_uv[y >> 1] = 1;
    }
    int rc = copy_plane_rows(h, const_cast<uint8_t*>(dev[b].y), dev[b].y_pitch, host[b].y, host[b].y_pitch, W, H, need_y, st, &total);
    if (rc) return rc;
    rc = copy_plane_rows(h, const_cast<uint8_t*>(dev[b].uv), dev[b].uv_pitch, host[b].uv, host[b].uv_pitch, W, H / 2, need_uv, st,
                         &total);
    if (rc) return rc;
  }
  if (bytes_copied) *bytes_copied = total;
  return B200VA_OK;
}

extern "C" int b200va_upload_frames_nv12(b200va_handle h, const b200va_nv12_frame* host, const b200va_nv12_frame* dev,
                                         const int* src_h, const int* src_w, int batch, int dst_h, int dst_w, int rows_mode,
                                         int64_t* bytes_copied, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, rows_mode == 0 || rows_mode == 1, "unknown rows_mode %d", rows_mode);
  std::vector<int> new_h;
  const int rc = upload_heights(h, src_h, src_w, batch, dst_h, dst_w, rows_mode, nullptr, &new_h);
  if (rc) return rc;
  return upload_nv12(h, host, dev, src_h, src_w, batch, new_h, bytes_copied, (cudaStream_t)stream);
}

extern "C" int b200va_upload_frames_nv12_geom(b200va_handle h, const b200va_nv12_frame* host, const b200va_nv12_frame* dev,
                                              const int* src_h, const int* src_w, int batch, const b200va_letterbox* geom,
                                              int64_t* bytes_copied, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, geom || batch == 0, "NULL geometry");
  std::vector<int> new_h;
  const int rc = upload_heights(h, src_h, src_w, batch, 0, 0, 1, geom, &new_h);
  if (rc) return rc;
  return upload_nv12(h, host, dev, src_h, src_w, batch, new_h, bytes_copied, (cudaStream_t)stream);
}
