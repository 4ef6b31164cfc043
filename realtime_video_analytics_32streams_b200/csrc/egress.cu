// 8f-3: the egress side of the hot path -- what KafkaSink.send_tracks / _render_frame
// (sinks/kafka_sink.py:93-149, 200-310 of the reference) do to a frame and its tracks before the encoder:
//
//   b200va_resize_area_u8   cv2.resize(image, (new_w, new_h), interpolation=cv2.INTER_AREA)        kafka_sink.py:227-232
//   b200va_resize_area_u8_nv12  the same on cv2.cvtColor(frame, COLOR_YUV2BGR_NV12), converted in the taps
//   b200va_draw_rects       cv2.rectangle(.., color, 2) and cv2.rectangle(.., color, -1) in order   kafka_sink.py:240, 249-255
//   b200va_tracks_json      json.dumps(payload) of the track event (host code, no device work)      kafka_sink.py:88, 105-134
//
// OpenCV semantics restated (resize.cpp: ResizeAreaFastVec_SIMD_8u / ResizeAreaFast_ / ResizeArea_ with
// computeResizeAreaTab; drawing.cpp: rectangle -> PolyLine -> ThickLine + round caps, FillConvexPoly): oracle/egress.py
// states them in NumPy and is pinned against the installed cv2 and against the reference's own KafkaSink.
#include <charconv>
#include <cmath>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"

namespace {

// ---- INTER_AREA --------------------------------------------------------------------------------
struct AreaEntry {
  int32_t src;   // source column (x table) or row (y table)
  float alpha;   // weight (float32, computed in double and narrowed like OpenCV's DecimateAlpha)
};
// what a launch's frames share: one (source, destination) size
struct AreaGeom {
  int dst_h, dst_w;
  int iscale_x, iscale_y;          // integer block (fast path) -- 0 when the general tables are used
  const int32_t* xofs;             // [dst_w + 1] CSR offsets into xtab
  const AreaEntry* xtab;
  const int32_t* yofs;             // [dst_h + 1]
  const AreaEntry* ytab;
};
struct AreaFrame {
  const uint8_t* src;
  uint8_t* dst;
  long long pitch;
  int src_h, src_w;
};
struct AreaParams {
  AreaFrame f[B200VA_LAUNCH_FRAMES];
  AreaGeom g;
};
// b200va_resize_area_u8_nv12: the two planes of each frame, each with its own base and pitch
struct AreaFrameNv12 {
  const uint8_t* y;
  const uint8_t* uv;   // src_h / 2 rows of src_w bytes: Cb, Cr of each 2 x 2 block
  uint8_t* dst;
  long long y_pitch, uv_pitch;
  int src_h, src_w;
};
struct AreaParamsNv12 {
  AreaFrameNv12 f[B200VA_LAUNCH_FRAMES];
  AreaGeom g;
};
static_assert(sizeof(AreaParamsNv12) <= 4000, "kernel parameter block too large");

// Source pixel loaders of the INTER_AREA bodies: src.row(y) is source row y, src.block(dx, sx, dy, sy) the same source
// seen from block (dx, dy) of sx x sy pixels on, and row.px(x, b, g, r) reads pixel x of a row.  Packed BGR: three
// bytes.  NV12: luma byte x of the row and the Cb, Cr pair at (x & ~1) of its chroma row, converted and saturated per
// pixel (cv2 converts first and resizes the BGR image), so every sum below adds converted pixels.
struct BgrRow {
  const uint8_t* p;
  __device__ __forceinline__ void px(int x, int& b, int& g, int& r) const {
    b = p[3 * x];
    g = p[3 * x + 1];
    r = p[3 * x + 2];
  }
};
struct BgrSrc {
  const uint8_t* src;
  long long pitch;
  __device__ __forceinline__ BgrSrc(const AreaFrame& f) : src(f.src), pitch(f.pitch) {}
  __device__ __forceinline__ BgrRow row(int y) const { return BgrRow{src + (long long)y * pitch}; }
  __device__ __forceinline__ BgrSrc block(int dx, int sx, int dy, int sy) const {
    return BgrSrc(src + (long long)dy * sy * pitch + (size_t)dx * sx * 3, pitch);
  }
  __device__ __forceinline__ BgrSrc(const uint8_t* s, long long p) : src(s), pitch(p) {}
};
struct Nv12Row {
  const uint8_t* y;
  const uint8_t* uv;
  int x0;
  __device__ __forceinline__ void px(int x, int& b, int& g, int& r) const {
    x += x0;
    const uint8_t* c = uv + (x & ~1);  // two byte loads: a chroma row may start at any address
    const uint32_t v = nv12_bgr(y[x], (uint32_t)c[0] | ((uint32_t)c[1] << 8));
    b = (int)(v & 0xffu);
    g = (int)((v >> 8) & 0xffu);
    r = (int)(v >> 16);
  }
};
struct Nv12Src {
  const uint8_t* y;
  const uint8_t* uv;
  long long y_pitch, uv_pitch;
  int x0 = 0, y0 = 0;  // the chroma pair of a pixel depends on its absolute position
  __device__ __forceinline__ Nv12Src(const AreaFrameNv12& f) : y(f.y), uv(f.uv), y_pitch(f.y_pitch), uv_pitch(f.uv_pitch) {}
  __device__ __forceinline__ Nv12Row row(int r) const {
    r += y0;
    return Nv12Row{y + (long long)r * y_pitch, uv + (long long)(r >> 1) * uv_pitch, x0};
  }
  __device__ __forceinline__ Nv12Src block(int dx, int sx, int dy, int sy) const {
    Nv12Src s = *this;
    s.x0 = dx * sx;
    s.y0 = dy * sy;
    return s;
  }
};

// whole iscale_x x iscale_y source blocks per destination pixel (ResizeAreaFast_).  2 x 2: the vector kernel's
// (a + b + c + d + 2) >> 2; any other block: saturate_cast<uchar>(sum * (1.f / area)), float multiply, ties to even.
template <class Src, class F>
__device__ __forceinline__ void area_fast_body(const AreaGeom& g, const F& f) {
  const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;
  if (dx >= g.dst_w) return;
  const Src src = Src(f).block(dx, g.iscale_x, dy, g.iscale_y);
  int sb = 0, sg = 0, sr = 0;
  for (int y = 0; y < g.iscale_y; ++y) {
    const auto row = src.row(y);
    for (int x = 0; x < g.iscale_x; ++x) {
      int b, gg, r;
      row.px(x, b, gg, r);
      sb += b;
      sg += gg;
      sr += r;
    }
  }
  uint8_t* d = f.dst + ((size_t)dy * g.dst_w + dx) * 3;
  if (g.iscale_x == 2 && g.iscale_y == 2) {
    d[0] = (uint8_t)((sb + 2) >> 2);
    d[1] = (uint8_t)((sg + 2) >> 2);
    d[2] = (uint8_t)((sr + 2) >> 2);
  } else {
    const float scale = 1.f / (float)(g.iscale_x * g.iscale_y);
    d[0] = (uint8_t)min(255, max(0, __float2int_rn(__fmul_rn((float)sb, scale))));
    d[1] = (uint8_t)min(255, max(0, __float2int_rn(__fmul_rn((float)sg, scale))));
    d[2] = (uint8_t)min(255, max(0, __float2int_rn(__fmul_rn((float)sr, scale))));
  }
}

__global__ void __launch_bounds__(256) k_area_fast(const __grid_constant__ AreaParams p) {
  area_fast_body<BgrSrc>(p.g, p.f[blockIdx.z]);
}

// NV12 blocks of any size: 1 x 1 is cv2.cvtColor itself; an odd block may see the chroma pair change inside it
__global__ void __launch_bounds__(256) k_area_nv12_fast(const __grid_constant__ AreaParamsNv12 p) {
  area_fast_body<Nv12Src>(p.g, p.f[blockIdx.z]);
}

// The 2 x 2 case on aligned frames (what a 4K camera sends): a thread owns four destination pixels -- two source rows
// of 24 bytes each as three 8-byte loads, twelve result bytes as three 4-byte stores, both fully coalesced.
__device__ __forceinline__ uint32_t byte_of(const uint32_t (&w)[6], int i) { return (w[i >> 2] >> ((i & 3) * 8)) & 0xffu; }

__global__ void __launch_bounds__(256) k_area_2x2_vec(const __grid_constant__ AreaParams p) {
  const AreaFrame& f = p.f[blockIdx.z];
  const int q = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;  // q: group of four destination pixels
  if (q * 4 >= p.g.dst_w) return;
  const uint8_t* s0 = f.src + (long long)(2 * dy) * f.pitch + (size_t)q * 24;
  const uint8_t* s1 = s0 + f.pitch;
  uint32_t a[6], b[6];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint2 va = __ldcs(reinterpret_cast<const uint2*>(s0) + k), vb = __ldcs(reinterpret_cast<const uint2*>(s1) + k);
    a[2 * k] = va.x;
    a[2 * k + 1] = va.y;
    b[2 * k] = vb.x;
    b[2 * k + 1] = vb.y;
  }
  uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const uint32_t v = (byte_of(a, 6 * j + c) + byte_of(a, 6 * j + 3 + c) + byte_of(b, 6 * j + c) + byte_of(b, 6 * j + 3 + c) + 2u) >> 2;
      const int ob = 3 * j + c;
      o[ob >> 2] |= v << ((ob & 3) * 8);
    }
  }
  uint32_t* d = reinterpret_cast<uint32_t*>(f.dst + ((size_t)dy * p.g.dst_w + (size_t)q * 4) * 3);
  __stcs(d, o[0]);
  __stcs(d + 1, o[1]);
  __stcs(d + 2, o[2]);
}

// The 2 x 2 case on aligned NV12 frames (4K -> 1080p): a thread owns four destination pixels and loads 8 bytes each of
// luma rows 2 dy and 2 dy + 1 and of chroma row dy -- the eight luma columns of its four blocks and their four Cb, Cr
// pairs.  A block starts at an even x and y, so its four pixels share one pair: the chroma terms are computed once per
// destination pixel, each of the four pixels is saturated on its own, then (a + b + c + d + 2) >> 2 per channel.
__global__ void __launch_bounds__(256) k_area_nv12_2x2_vec(const __grid_constant__ AreaParamsNv12 p) {
  const AreaFrameNv12& f = p.f[blockIdx.z];
  const int q = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;
  if (q * 4 >= p.g.dst_w) return;
  const uint8_t* y0 = f.y + (long long)(2 * dy) * f.y_pitch + (size_t)q * 8;
  const uint2 l0 = __ldcs(reinterpret_cast<const uint2*>(y0));
  const uint2 l1 = __ldcs(reinterpret_cast<const uint2*>(y0 + f.y_pitch));
  const uint2 cc = __ldcs(reinterpret_cast<const uint2*>(f.uv + (long long)dy * f.uv_pitch + (size_t)q * 8));
  uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t w0 = j < 2 ? l0.x : l0.y, w1 = j < 2 ? l1.x : l1.y, wc = j < 2 ? cc.x : cc.y;
    const int sh = (j & 1) * 16;  // block j: luma bytes 2j, 2j + 1 of both rows, chroma pair j
    const int3 t = nv12_chroma((wc >> sh) & 0xffffu);
    const int ya = nv12_luma((w0 >> sh) & 0xff), yb = nv12_luma((w0 >> (sh + 8)) & 0xff);
    const int yc = nv12_luma((w1 >> sh) & 0xff), yd = nv12_luma((w1 >> (sh + 8)) & 0xff);
    const int term[3] = {t.x, t.y, t.z};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const uint32_t v = (nv12_sat(ya, term[c]) + nv12_sat(yb, term[c]) + nv12_sat(yc, term[c]) + nv12_sat(yd, term[c]) + 2u) >> 2;
      const int ob = 3 * j + c;
      o[ob >> 2] |= v << ((ob & 3) * 8);
    }
  }
  uint32_t* d = reinterpret_cast<uint32_t*>(f.dst + ((size_t)dy * p.g.dst_w + (size_t)q * 4) * 3);
  __stcs(d, o[0]);
  __stcs(d + 1, o[1]);
  __stcs(d + 2, o[2]);
}

// ResizeArea_<uchar, float>: for every source row of the destination row (y table order) a horizontal float sum in
// x table order starting from 0, then sum = beta * buf for the first row and sum += beta * buf for the others; no
// contraction (the file is compiled with -fmad=false and the operations are spelled out).
template <class Src, class F>
__device__ __forceinline__ void area_general_body(const AreaGeom& g, const F& f) {
  const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;
  if (dx >= g.dst_w) return;
  const Src src(f);
  const int x0 = g.xofs[dx], x1 = g.xofs[dx + 1];
  const int y0 = g.yofs[dy], y1 = g.yofs[dy + 1];
  float ab = 0.f, ag = 0.f, ar = 0.f;
  for (int j = y0; j < y1; ++j) {
    const AreaEntry ye = g.ytab[j];
    const auto row = src.row(ye.src);
    float bb = 0.f, bg = 0.f, br = 0.f;
    for (int k = x0; k < x1; ++k) {
      const AreaEntry xe = g.xtab[k];
      int b, gg, r;
      row.px(xe.src, b, gg, r);
      bb = __fadd_rn(bb, __fmul_rn((float)b, xe.alpha));
      bg = __fadd_rn(bg, __fmul_rn((float)gg, xe.alpha));
      br = __fadd_rn(br, __fmul_rn((float)r, xe.alpha));
    }
    if (j == y0) {
      ab = __fmul_rn(ye.alpha, bb);
      ag = __fmul_rn(ye.alpha, bg);
      ar = __fmul_rn(ye.alpha, br);
    } else {
      ab = __fadd_rn(ab, __fmul_rn(ye.alpha, bb));
      ag = __fadd_rn(ag, __fmul_rn(ye.alpha, bg));
      ar = __fadd_rn(ar, __fmul_rn(ye.alpha, br));
    }
  }
  uint8_t* d = f.dst + ((size_t)dy * g.dst_w + dx) * 3;
  d[0] = (uint8_t)min(255, max(0, __float2int_rn(ab)));
  d[1] = (uint8_t)min(255, max(0, __float2int_rn(ag)));
  d[2] = (uint8_t)min(255, max(0, __float2int_rn(ar)));
}

__global__ void __launch_bounds__(256) k_area_general(const __grid_constant__ AreaParams p) {
  area_general_body<BgrSrc>(p.g, p.f[blockIdx.z]);
}

__global__ void __launch_bounds__(256) k_area_nv12_general(const __grid_constant__ AreaParamsNv12 p) {
  area_general_body<Nv12Src>(p.g, p.f[blockIdx.z]);
}

// computeResizeAreaTab (resize.cpp), double arithmetic, float weights; CSR per destination index
void area_tab(int ssize, int dsize, double scale, std::vector<int32_t>& ofs, std::vector<AreaEntry>& tab) {
  ofs.assign(dsize + 1, 0);
  tab.clear();
  for (int dx = 0; dx < dsize; ++dx) {
    ofs[dx] = (int32_t)tab.size();
    const double fsx1 = dx * scale, fsx2 = fsx1 + scale;
    const double cell = std::min(scale, ssize - fsx1);
    int sx1 = (int)std::ceil(fsx1), sx2 = (int)std::floor(fsx2);
    sx2 = std::min(sx2, ssize - 1);
    sx1 = std::min(sx1, sx2);
    if (sx1 - fsx1 > 1e-3) tab.push_back({sx1 - 1, (float)((sx1 - fsx1) / cell)});
    for (int sx = sx1; sx < sx2; ++sx) tab.push_back({sx, (float)(1.0 / cell)});
    if (fsx2 - sx2 > 1e-3) tab.push_back({sx2, (float)(std::min(std::min(fsx2 - sx2, 1.), cell) / cell)});
  }
  ofs[dsize] = (int32_t)tab.size();
}

struct AreaTables {
  int32_t* xofs = nullptr;
  AreaEntry* xtab = nullptr;
  int32_t* yofs = nullptr;
  AreaEntry* ytab = nullptr;
  void* base = nullptr;
};

// ---- rectangles ----------------------------------------------------------------------------------
struct RectImage {
  uint8_t* img;
  long long pitch;
  int h, w;
  int op0, op1;  // this image's operations: ops[op0 .. op1)
};
struct RectParams {
  RectImage im[B200VA_LAUNCH_FRAMES];
  const b200va_rect_op* ops;
};

__device__ __forceinline__ bool in_box(int x, int y, int x1, int y1, int x2, int y2) {
  return x >= x1 && x <= x2 && y >= y1 && y <= y2;
}

// The reference draws its rectangles one after another, so a pixel ends up with the colour of the LAST operation that
// covers it.  A CTA owns a 64 x 4 pixel tile: its threads first collect the operations whose bounding box (grown by the
// outline's stroke) touches the tile -- most tiles of a frame collect none and leave -- then every thread takes the
// highest-numbered collected operation that covers its pixel.
//   kind 1  cv2.rectangle(.., -1): the inclusive box
//   kind 0  cv2.rectangle(.., 2):  four 3-pixel bands between the corner points (ThickLine's polygon at half-thickness
//           1) whose round caps (Circle radius 1: a plus shape) add nothing the neighbouring band does not cover
constexpr int kTileW = 64, kTileH = 4, kTileOps = 256;

__device__ __forceinline__ bool op_hits(const b200va_rect_op& o, int x, int y) {
  const int x1 = min(o.x1, o.x2), x2 = max(o.x1, o.x2), y1 = min(o.y1, o.y2), y2 = max(o.y1, o.y2);
  if (o.kind) return in_box(x, y, x1, y1, x2, y2);
  return in_box(x, y, x1, y1 - 1, x2, y1 + 1) || in_box(x, y, x1, y2 - 1, x2, y2 + 1) || in_box(x, y, x1 - 1, y1, x1 + 1, y2) ||
         in_box(x, y, x2 - 1, y1, x2 + 1, y2);
}

__global__ void __launch_bounds__(kTileW * kTileH) k_draw_rects(const __grid_constant__ RectParams p) {
  const RectImage& im = p.im[blockIdx.z];
  const int tx0 = blockIdx.x * kTileW, ty0 = blockIdx.y * kTileH;
  if (tx0 >= im.w || ty0 >= im.h) return;
  __shared__ int s_n;
  __shared__ int s_ops[kTileOps];
  const int tid = threadIdx.y * kTileW + threadIdx.x;
  if (tid == 0) s_n = 0;
  __syncthreads();
  const int tx1 = tx0 + kTileW - 1, ty1 = ty0 + kTileH - 1;
  for (int k = im.op0 + tid; k < im.op1; k += kTileW * kTileH) {
    const b200va_rect_op o = p.ops[k];
    const int x1 = min(o.x1, o.x2) - 1, x2 = max(o.x1, o.x2) + 1, y1 = min(o.y1, o.y2) - 1, y2 = max(o.y1, o.y2) + 1;
    if (x1 <= tx1 && x2 >= tx0 && y1 <= ty1 && y2 >= ty0) {
      const int slot = atomicAdd(&s_n, 1);
      if (slot < kTileOps) s_ops[slot] = k;
    }
  }
  __syncthreads();
  const int n = s_n;
  if (n == 0) return;
  const int x = tx0 + threadIdx.x, y = ty0 + threadIdx.y;
  if (x >= im.w || y >= im.h) return;
  int best = -1;
  if (n <= kTileOps) {
    for (int i = 0; i < n; ++i) {
      const int k = s_ops[i];
      if (k > best && op_hits(p.ops[k], x, y)) best = k;
    }
  } else {  // a tile under more operations than the list holds: walk the whole list backwards
    for (int k = im.op1 - 1; k >= im.op0; --k)
      if (op_hits(p.ops[k], x, y)) {
        best = k;
        break;
      }
  }
  if (best >= 0) {
    const b200va_rect_op o = p.ops[best];
    uint8_t* d = im.img + (long long)y * im.pitch + (size_t)x * 3;
    d[0] = o.b;
    d[1] = o.g;
    d[2] = o.r;
  }
}

}  // namespace

struct EgressState {
  std::map<std::pair<std::pair<int, int>, std::pair<int, int>>, AreaTables> tables;  // ((src_h, src_w), (dst_h, dst_w))
  b200va_rect_op* ops = nullptr;
  size_t ops_cap = 0;
};

static EgressState* egress(b200va_ctx* h) {
  if (!h->egress) h->egress = new EgressState();
  return (EgressState*)h->egress;
}

void egress_destroy(b200va_ctx* h) {
  EgressState* e = (EgressState*)h->egress;
  if (!e) return;
  for (auto& kv : e->tables)
    if (kv.second.base) cudaFree(kv.second.base);
  if (e->ops) cudaFree(e->ops);
  delete e;
  h->egress = nullptr;
}

// The geometry of one (source, destination) size group: cv::resize's integer-block test and, for fractional ratios,
// the cached x / y tables (they depend on the sizes only, so BGR and NV12 frames share them).  Sets *fast.
static int area_geom(b200va_ctx* h, int sh, int sw, int dh, int dw, AreaGeom& g, bool* fast) {
  // cv::resize: inv_scale = dsize / ssize, scale = 1 / inv_scale (double)
  const double scale_x = 1.0 / ((double)dw / sw), scale_y = 1.0 / ((double)dh / sh);
  const int iscale_x = (int)std::nearbyint(scale_x), iscale_y = (int)std::nearbyint(scale_y);
  *fast = std::fabs(scale_x - iscale_x) < 2.220446049250313e-16 && std::fabs(scale_y - iscale_y) < 2.220446049250313e-16;
  memset(&g, 0, sizeof(g));
  g.dst_h = dh;
  g.dst_w = dw;
  if (*fast) {
    g.iscale_x = iscale_x;
    g.iscale_y = iscale_y;
    return B200VA_OK;
  }
  EgressState* e = egress(h);
  AreaTables& t = e->tables[{{sh, sw}, {dh, dw}}];
  if (!t.base) {
    std::vector<int32_t> xo, yo;
    std::vector<AreaEntry> xt, yt;
    area_tab(sw, dw, scale_x, xo, xt);
    area_tab(sh, dh, scale_y, yo, yt);
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o1 = al(xo.size() * 4), o2 = o1 + al(xt.size() * sizeof(AreaEntry)), o3 = o2 + al(yo.size() * 4),
                 total = o3 + al(yt.size() * sizeof(AreaEntry));
    CUDA_TRY(h, cudaMalloc(&t.base, total));
    uint8_t* b = (uint8_t*)t.base;
    t.xofs = (int32_t*)b;
    t.xtab = (AreaEntry*)(b + o1);
    t.yofs = (int32_t*)(b + o2);
    t.ytab = (AreaEntry*)(b + o3);
    // (synchronous copies: the tables of a geometry are built once)
    CUDA_TRY(h, cudaMemcpy(t.xofs, xo.data(), xo.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(t.xtab, xt.data(), xt.size() * sizeof(AreaEntry), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(t.yofs, yo.data(), yo.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(t.ytab, yt.data(), yt.size() * sizeof(AreaEntry), cudaMemcpyHostToDevice));
  }
  g.xofs = t.xofs;
  g.xtab = t.xtab;
  g.yofs = t.yofs;
  g.ytab = t.ytab;
  return B200VA_OK;
}

using AreaGroups = std::map<std::pair<std::pair<int, int>, std::pair<int, int>>, std::vector<int>>;

extern "C" int b200va_resize_area_u8(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                     const int64_t* src_pitch, int batch, uint8_t* const* dst, const int* dst_h,
                                     const int* dst_w, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && dst && dst_h && dst_w, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  cudaStream_t st = (cudaStream_t)stream;
  PhaseScope phase(h, B200VA_PHASE_EGRESS, st);
  // frames that share source and destination size go out in one launch
  AreaGroups groups;
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, frames[b] && dst[b], "frame %d: NULL pointer", b);
    REQUIRE(h, src_h[b] > 0 && src_w[b] > 0 && dst_h[b] > 0 && dst_w[b] > 0, "frame %d: bad size", b);
    REQUIRE(h, dst_h[b] <= src_h[b] && dst_w[b] <= src_w[b], "frame %d: INTER_AREA is implemented for shrinking only (%dx%d -> %dx%d)", b,
            src_w[b], src_h[b], dst_w[b], dst_h[b]);
    REQUIRE(h, dst_h[b] < 65536, "frame %d: destination too tall", b);
    groups[{{src_h[b], src_w[b]}, {dst_h[b], dst_w[b]}}].push_back(b);
  }
  for (const auto& kv : groups) {
    const int sh = kv.first.first.first, sw = kv.first.first.second, dh = kv.first.second.first, dw = kv.first.second.second;
    AreaParams p;
    memset(&p, 0, sizeof(p));
    bool fast = false;
    const int rc = area_geom(h, sh, sw, dh, dw, p.g, &fast);
    if (rc) return rc;
    const std::vector<int>& idx = kv.second;
    for (size_t base = 0; base < idx.size(); base += B200VA_LAUNCH_FRAMES) {
      const int n = (int)std::min<size_t>(B200VA_LAUNCH_FRAMES, idx.size() - base);
      for (int i = 0; i < n; ++i) {
        const int b = idx[base + i];
        p.f[i] = AreaFrame{frames[b], dst[b], src_pitch ? (long long)src_pitch[b] : 3ll * sw, sh, sw};
      }
      const dim3 grid((dw + 255) / 256, dh, n);
      bool vec = fast && p.g.iscale_x == 2 && p.g.iscale_y == 2 && dw % 4 == 0;
      for (int i = 0; i < n && vec; ++i)
        vec = ((uintptr_t)p.f[i].src % 8 == 0) && (p.f[i].pitch % 8 == 0) && ((uintptr_t)p.f[i].dst % 4 == 0);
      if (vec) k_area_2x2_vec<<<dim3((dw / 4 + 255) / 256, dh, n), 256, 0, st>>>(p);
      else if (fast) k_area_fast<<<grid, 256, 0, st>>>(p);
      else k_area_general<<<grid, 256, 0, st>>>(p);
      LAUNCH_CHECK(h);
    }
  }
  return B200VA_OK;
}

extern "C" int b200va_resize_area_u8_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                          const int* src_w, int batch, uint8_t* const* dst, const int* dst_h,
                                          const int* dst_w, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, frames && src_h && src_w && dst && dst_h && dst_w, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  cudaStream_t st = (cudaStream_t)stream;
  PhaseScope phase(h, B200VA_PHASE_EGRESS, st);
  AreaGroups groups;
  for (int b = 0; b < batch; ++b) {
    const b200va_nv12_frame& n = frames[b];
    REQUIRE(h, n.y && n.uv, "frame %d: NULL plane", b);
    REQUIRE(h, dst[b], "dst %d is NULL", b);
    REQUIRE(h, src_h[b] > 0 && src_w[b] > 0 && dst_h[b] > 0 && dst_w[b] > 0, "frame %d: bad size", b);
    REQUIRE(h, src_h[b] % 2 == 0 && src_w[b] % 2 == 0, "frame %d: NV12 needs an even size, got %dx%d", b, src_w[b], src_h[b]);
    REQUIRE(h, n.y_pitch >= src_w[b] && n.uv_pitch >= src_w[b], "frame %d: plane pitch %lld / %lld < width %d", b,
            (long long)n.y_pitch, (long long)n.uv_pitch, src_w[b]);
    REQUIRE(h, dst_h[b] <= src_h[b] && dst_w[b] <= src_w[b], "frame %d: INTER_AREA is implemented for shrinking only (%dx%d -> %dx%d)", b,
            src_w[b], src_h[b], dst_w[b], dst_h[b]);
    REQUIRE(h, dst_h[b] < 65536, "frame %d: destination too tall", b);
    groups[{{src_h[b], src_w[b]}, {dst_h[b], dst_w[b]}}].push_back(b);
  }
  for (const auto& kv : groups) {
    const int sh = kv.first.first.first, sw = kv.first.first.second, dh = kv.first.second.first, dw = kv.first.second.second;
    AreaParamsNv12 p;
    memset(&p, 0, sizeof(p));
    bool fast = false;
    const int rc = area_geom(h, sh, sw, dh, dw, p.g, &fast);
    if (rc) return rc;
    const std::vector<int>& idx = kv.second;
    for (size_t base = 0; base < idx.size(); base += B200VA_LAUNCH_FRAMES) {
      const int n = (int)std::min<size_t>(B200VA_LAUNCH_FRAMES, idx.size() - base);
      bool vec = fast && p.g.iscale_x == 2 && p.g.iscale_y == 2 && dw % 4 == 0;
      for (int i = 0; i < n; ++i) {
        const int b = idx[base + i];
        const b200va_nv12_frame& s = frames[b];
        p.f[i] = AreaFrameNv12{s.y, s.uv, dst[b], (long long)s.y_pitch, (long long)s.uv_pitch, sh, sw};
        vec = vec && (uintptr_t)s.y % 8 == 0 && (uintptr_t)s.uv % 8 == 0 && s.y_pitch % 8 == 0 && s.uv_pitch % 8 == 0 &&
              (uintptr_t)dst[b] % 4 == 0;
      }
      const dim3 grid((dw + 255) / 256, dh, n);
      if (vec) k_area_nv12_2x2_vec<<<dim3((dw / 4 + 255) / 256, dh, n), 256, 0, st>>>(p);
      else if (fast) k_area_nv12_fast<<<grid, 256, 0, st>>>(p);
      else k_area_nv12_general<<<grid, 256, 0, st>>>(p);
      LAUNCH_CHECK(h);
    }
  }
  return B200VA_OK;
}

extern "C" int b200va_draw_rects(b200va_handle h, uint8_t* const* images, const int* img_h, const int* img_w,
                                 const int64_t* pitch, int batch, const b200va_rect_op* ops, const int* op_offsets,
                                 void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, images && img_h && img_w && op_offsets, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  if (batch == 0) return B200VA_OK;
  const int n_ops = op_offsets[batch];
  REQUIRE(h, op_offsets[0] == 0 && n_ops >= 0, "op_offsets must start at 0 and be non-decreasing");
  for (int b = 0; b < batch; ++b) {
    REQUIRE(h, op_offsets[b + 1] >= op_offsets[b], "op_offsets must be non-decreasing");
    REQUIRE(h, images[b] && img_h[b] > 0 && img_w[b] > 0 && img_h[b] < 65536, "image %d: bad pointer or size", b);
  }
  if (n_ops == 0) return B200VA_OK;
  REQUIRE(h, ops != nullptr, "NULL ops");
  cudaStream_t st = (cudaStream_t)stream;
  PhaseScope phase(h, B200VA_PHASE_EGRESS, st);
  EgressState* e = egress(h);
  if ((size_t)n_ops > e->ops_cap) {
    if (e->ops) {
      CUDA_TRY(h, cudaStreamSynchronize(st));  // an earlier launch may still read the old list
      CUDA_TRY(h, cudaFree(e->ops));
      e->ops = nullptr;
    }
    e->ops_cap = std::max<size_t>(1024, (size_t)n_ops * 2);
    CUDA_TRY(h, cudaMalloc(&e->ops, e->ops_cap * sizeof(b200va_rect_op)));
  }
  // (pageable source: the call returns once the list is staged, the caller may reuse `ops` at once)
  CUDA_TRY(h, cudaMemcpyAsync(e->ops, ops, (size_t)n_ops * sizeof(b200va_rect_op), cudaMemcpyHostToDevice, st));
  for (int base = 0; base < batch; base += B200VA_LAUNCH_FRAMES) {
    const int n = std::min(B200VA_LAUNCH_FRAMES, batch - base);
    RectParams p;
    memset(&p, 0, sizeof(p));
    p.ops = e->ops;
    int mh = 0, mw = 0;
    for (int i = 0; i < n; ++i) {
      const int b = base + i;
      p.im[i] = RectImage{images[b], pitch ? (long long)pitch[b] : 3ll * img_w[b], img_h[b], img_w[b], op_offsets[b], op_offsets[b + 1]};
      mh = std::max(mh, img_h[b]);
      mw = std::max(mw, img_w[b]);
    }
    k_draw_rects<<<dim3((mw + kTileW - 1) / kTileW, (mh + kTileH - 1) / kTileH, n), dim3(kTileW, kTileH), 0, st>>>(p);
    LAUNCH_CHECK(h);
  }
  return B200VA_OK;
}

// ---- json.dumps(payload) ---------------------------------------------------------------------
namespace {

struct Out {
  char* buf;
  int64_t cap, n = 0;
  void put(char c) {
    if (n < cap) buf[n] = c;
    ++n;
  }
  void put(const char* s) {
    while (*s) put(*s++);
  }
  void put_int(long long v) {
    char tmp[24];
    auto r = std::to_chars(tmp, tmp + sizeof(tmp), v);
    for (char* c = tmp; c != r.ptr; ++c) put(*c);
  }
  // float.__repr__ (CPython: PyOS_double_to_string(x, 'r', 0, Py_DTSF_ADD_DOT_0)): the shortest digit string that
  // round-trips, fixed notation while -4 < decpt <= 16, exponent notation (at least two exponent digits) otherwise;
  // json.dumps spells the non-finite values NaN / Infinity / -Infinity
  void put_double(double v) {
    if (std::isnan(v)) return put("NaN");
    if (std::isinf(v)) return put(v > 0 ? "Infinity" : "-Infinity");
    char tmp[40];
    auto r = std::to_chars(tmp, tmp + sizeof(tmp), v, std::chars_format::scientific);  // [-]d[.ddd]e[+-]xx, shortest
    const char* s = tmp;
    if (*s == '-') {
      put('-');
      ++s;
    }
    char digits[24];
    int nd = 0;
    const char* q = s;
    for (; q != r.ptr && *q != 'e'; ++q)
      if (*q != '.') digits[nd++] = *q;
    int exp10 = 0;
    std::from_chars(q + 1 + (q[1] == '+' ? 1 : 0), r.ptr, exp10);
    const int decpt = exp10 + 1;  // value = 0.d1d2.. x 10^decpt
    if (decpt > -4 && decpt <= 16) {
      if (decpt <= 0) {
        put("0.");
        for (int i = 0; i < -decpt; ++i) put('0');
        for (int i = 0; i < nd; ++i) put(digits[i]);
      } else if (decpt >= nd) {
        for (int i = 0; i < nd; ++i) put(digits[i]);
        for (int i = nd; i < decpt; ++i) put('0');
        put(".0");
      } else {
        for (int i = 0; i < decpt; ++i) put(digits[i]);
        put('.');
        for (int i = decpt; i < nd; ++i) put(digits[i]);
      }
    } else {
      put(digits[0]);
      if (nd > 1) {
        put('.');
        for (int i = 1; i < nd; ++i) put(digits[i]);
      }
      put('e');
      const int e = decpt - 1;
      put(e < 0 ? '-' : '+');
      const int a = e < 0 ? -e : e;
      if (a < 10) put('0');
      put_int(a);
    }
  }
  // json.dumps string with ensure_ascii=True: \" \\ \n \r \t \b \f, other control characters and everything beyond
  // ASCII as \uXXXX (UTF-16 surrogate pairs above the BMP)
  void put_string(const char* s) {
    static const char* hex = "0123456789abcdef";
    auto u4 = [&](unsigned c) {
      put("\\u");
      put(hex[(c >> 12) & 15]);
      put(hex[(c >> 8) & 15]);
      put(hex[(c >> 4) & 15]);
      put(hex[c & 15]);
    };
    put('"');
    const unsigned char* p = (const unsigned char*)s;
    while (*p) {
      unsigned c = *p;
      int extra = 0;
      if (c >= 0xF0) { c &= 0x07; extra = 3; }
      else if (c >= 0xE0) { c &= 0x0F; extra = 2; }
      else if (c >= 0xC0) { c &= 0x1F; extra = 1; }
      ++p;
      for (; extra > 0 && (*p & 0xC0) == 0x80; --extra) c = (c << 6) | (*p++ & 0x3F);
      if (c == '"') put("\\\"");
      else if (c == '\\') put("\\\\");
      else if (c == '\n') put("\\n");
      else if (c == '\r') put("\\r");
      else if (c == '\t') put("\\t");
      else if (c == '\b') put("\\b");
      else if (c == '\f') put("\\f");
      else if (c < 0x20 || (c >= 0x7F && c < 0x10000)) {  // json's ESCAPE_ASCII: everything outside ' ' .. '~'
        u4(c);
      } else if (c >= 0x10000) {
        const unsigned v = c - 0x10000;
        u4(0xD800 | (v >> 10));
        u4(0xDC00 | (v & 0x3FF));
      } else {
        put((char)c);
      }
    }
    put('"');
  }
};

}  // namespace

extern "C" int64_t b200va_tracks_json(const char* stream_name, int64_t frame_id, const int64_t* track_id, const int32_t* cls,
                                      const double* conf, const double* bbox_xyxy, int n, const char* frame_data_url,
                                      char* out, int64_t cap) {
  if (!stream_name || n < 0 || (n > 0 && (!track_id || !cls || !conf || !bbox_xyxy)) || cap < 0 || (cap > 0 && !out)) return -1;
  Out o{out, cap};
  o.put("{\"stream\": ");
  o.put_string(stream_name);
  o.put(", \"frame_id\": ");
  o.put_int(frame_id);
  o.put(", \"tracks\": [");
  for (int i = 0; i < n; ++i) {
    if (i) o.put(", ");
    o.put("{\"track_id\": ");
    o.put_int(track_id[i]);
    o.put(", \"class_id\": ");
    o.put_int(cls[i]);
    o.put(", \"confidence\": ");
    o.put_double(conf[i]);
    o.put(", \"bbox_xyxy\": [");
    for (int k = 0; k < 4; ++k) {
      if (k) o.put(", ");
      o.put_double(bbox_xyxy[4 * i + k]);
    }
    o.put("]}");
  }
  o.put("], \"is_temporal\": false");
  if (frame_data_url) {
    o.put(", \"frame_jpeg\": ");
    o.put_string(frame_data_url);
  }
  o.put('}');
  return o.n;
}
