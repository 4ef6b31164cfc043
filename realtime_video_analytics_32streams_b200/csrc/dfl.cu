// a14: DFL box decode of a raw YOLOv8 Detect head (named by the north star).
//
// NOT in the reference tree: the tensors the reference's _postprocess consumes are already decoded; the
// decode lives in the third-party Ultralytics `Detect` head (ultralytics==8.3.209, pylock.toml:1432-1433,
// reached only through YOLO(...).predict, detector.py:129,147-155).  Its published algorithm, restated:
//   raw [B, 4*reg_max + nc, A];  per box side: softmax over reg_max bins, expectation with weights 0..reg_max-1;
//   anchor points = cell centres (x + 0.5, y + 0.5) of the 80x80 / 40x40 / 20x20 grids (A = 8400 at 640x640);
//   x1y1 = anchor - (l, t), x2y2 = anchor + (r, b);  (cx, cy) = (x1y1 + x2y2) / 2, (w, h) = x2y2 - x1y1;
//   all four times the level's stride;  class scores = sigmoid(logits).
// Output [B, 4 + nc, A] is exactly what b200va_postprocess reads (channel major).  Floating point with
// exp: compared with the float64 decode (oracle/dfl.py) under an error bound derived from the float32
// operation order below (tests/dfl_bound.py), "parity unpinned" by the reference.
// HBM bound: (4*reg_max + nc) * A * 4 bytes read + (4 + nc) * A * 4 written per frame (7.7 MB at nc = 80).
#include <climits>

#include "common.cuh"

namespace {

constexpr int kMaxLevels = 8;

struct DflParams {
  const float* raw;
  float* out;
  int nc, reg_max, A, n_levels;
  int off[kMaxLevels + 1];  // first anchor of each level
  int w[kMaxLevels];        // grid width of each level
  float stride[kMaxLevels];
};

// VEC consecutive anchors of one channel row: one 16-byte access when VEC = 4
template <int VEC>
struct Lanes {
  float v[VEC];
};
template <int VEC>
__device__ __forceinline__ Lanes<VEC> load_row(const float* __restrict__ p) {
  Lanes<VEC> r;
  if (VEC == 4) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    r.v[0] = q.x;
    r.v[1 % VEC] = q.y;
    r.v[2 % VEC] = q.z;
    r.v[3 % VEC] = q.w;
  } else {
    r.v[0] = __ldg(p);
  }
  return r;
}
template <int VEC>
__device__ __forceinline__ void store_row(float* __restrict__ p, const Lanes<VEC>& r) {
  if (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1 % VEC], r.v[2 % VEC], r.v[3 % VEC]);
  else *p = r.v[0];
}

// softmax expectation over the bins of one box side (bins RM at compile time, or reg_max at run time), VEC anchors
template <int RM, int VEC>
__device__ __forceinline__ Lanes<VEC> side_expectation(const float* __restrict__ base, size_t A, int a, int reg_max) {
  Lanes<VEC> res;
  if (RM > 0) {
    Lanes<VEC> x[RM > 0 ? RM : 1];
#pragma unroll
    for (int k = 0; k < RM; ++k) x[k] = load_row<VEC>(base + (size_t)k * A + a);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      float m = -INFINITY;
#pragma unroll
      for (int k = 0; k < RM; ++k) m = fmaxf(m, x[k].v[j]);
      float s = 0.f, e = 0.f;
#pragma unroll
      for (int k = 0; k < RM; ++k) {
        const float ek = expf(x[k].v[j] - m);
        s += ek;
        e += (float)k * ek;
      }
      res.v[j] = e / s;
    }
    return res;
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    float m = -INFINITY;
    for (int k = 0; k < reg_max; ++k) m = fmaxf(m, __ldg(base + (size_t)k * A + a + j));
    float s = 0.f, e = 0.f;
    for (int k = 0; k < reg_max; ++k) {
      const float ek = expf(__ldg(base + (size_t)k * A + a + j) - m);
      s += ek;
      e += (float)k * ek;
    }
    res.v[j] = e / s;
  }
  return res;
}

// Work is split along the channels as well as the anchors: blockIdx.z = 0 decodes the box of 128 * VEC anchors
// (4 * reg_max rows in, 4 rows out), blockIdx.z = j >= 1 the class rows [kClsRows (j - 1), kClsRows j).  One block per
// 128 anchors doing all 144 rows was 2100 blocks of ~14 dependent load rounds each on 1480 block slots: 1.42 waves,
// the second one 42 % full -- the kernel sat at 0.68 of peak whatever its arithmetic cost (fast exp: -2 us).  Shorter
// blocks (the heavy box blocks are scheduled first) leave no such tail: 0.80; that version issued 38.6 M warp
// instructions with the issue slots 84 % busy, so a thread now owns four consecutive anchors (16-byte accesses, a
// quarter of the address arithmetic) and the sigmoid's division is a correctly rounded reciprocal (same result).
constexpr int kClsRows = 8;

template <int RM, int VEC>
__global__ void __launch_bounds__(128) k_dfl_decode(const __grid_constant__ DflParams p) {
  const int a = (blockIdx.x * blockDim.x + threadIdx.x) * VEC;  // (VEC = 4: A is a multiple of 4)
  if (a >= p.A) return;
  const size_t A = (size_t)p.A;
  const int cin = 4 * p.reg_max + p.nc, cout = 4 + p.nc;
  const float* __restrict__ in = p.raw + (size_t)blockIdx.y * cin * A;
  float* __restrict__ out = p.out + (size_t)blockIdx.y * cout * A;
  if (blockIdx.z == 0) {
    Lanes<VEC> d[4];
#pragma unroll
    for (int sd = 0; sd < 4; ++sd) d[sd] = side_expectation<RM, VEC>(in + (size_t)sd * p.reg_max * A, A, a, p.reg_max);
    Lanes<VEC> cx, cy, bw, bh;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      int l = 0;
      while (l + 1 < p.n_levels && a + j >= p.off[l + 1]) ++l;
      const int idx = a + j - p.off[l];
      const float ax = (float)(idx % p.w[l]) + 0.5f, ay = (float)(idx / p.w[l]) + 0.5f;
      const float st = p.stride[l];
      const float x1 = ax - d[0].v[j], y1 = ay - d[1].v[j], x2 = ax + d[2].v[j], y2 = ay + d[3].v[j];
      cx.v[j] = (x1 + x2) * 0.5f * st;
      cy.v[j] = (y1 + y2) * 0.5f * st;
      bw.v[j] = (x2 - x1) * st;
      bh.v[j] = (y2 - y1) * st;
    }
    store_row<VEC>(out + a, cx);
    store_row<VEC>(out + A + a, cy);
    store_row<VEC>(out + 2 * A + a, bw);
    store_row<VEC>(out + 3 * A + a, bh);
    return;
  }
  const float* __restrict__ cl = in + (size_t)4 * p.reg_max * A;
  const int c0 = ((int)blockIdx.z - 1) * kClsRows, c1 = min(p.nc, c0 + kClsRows);
  if (c1 - c0 == kClsRows) {
    Lanes<VEC> v[kClsRows];
#pragma unroll
    for (int u = 0; u < kClsRows; ++u) v[u] = load_row<VEC>(cl + (size_t)(c0 + u) * A + a);
#pragma unroll
    for (int u = 0; u < kClsRows; ++u) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) v[u].v[j] = __frcp_rn(1.f + expf(-v[u].v[j]));  // = 1 / x, correctly rounded
      store_row<VEC>(out + (size_t)(4 + c0 + u) * A + a, v[u]);
    }
  } else {
    for (int c = c0; c < c1; ++c) {
      Lanes<VEC> v = load_row<VEC>(cl + (size_t)c * A + a);
#pragma unroll
      for (int j = 0; j < VEC; ++j) v.v[j] = __frcp_rn(1.f + expf(-v.v[j]));
      store_row<VEC>(out + (size_t)(4 + c) * A + a, v);
    }
  }
}

}  // namespace

extern "C" int b200va_dfl_decode(b200va_handle h, const float* raw, int batch, int num_classes, int reg_max,
                                 const int* level_hw, const float* level_stride, int n_levels, float* out,
                                 void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, raw && out && level_hw && level_stride, "NULL argument");
  REQUIRE(h, batch >= 0 && num_classes >= 0 && reg_max >= 1 && reg_max <= 64, "bad head geometry");
  REQUIRE(h, n_levels >= 1 && n_levels <= kMaxLevels, "n_levels must be in [1, %d]", kMaxLevels);
  if (batch == 0) return B200VA_OK;
  DflParams p;
  memset(&p, 0, sizeof(p));
  // the kernel's anchor indices are int: count in 64 bits and refuse what would wrap
  int64_t total = 0;
  for (int l = 0; l < n_levels; ++l) {
    REQUIRE(h, level_hw[2 * l] > 0 && level_hw[2 * l + 1] > 0, "level %d has an empty grid", l);
    p.off[l] = (int)total;
    p.w[l] = level_hw[2 * l + 1];
    p.stride[l] = level_stride[l];
    total += (int64_t)level_hw[2 * l] * level_hw[2 * l + 1];
    REQUIRE(h, total <= INT_MAX, "more than %d anchors", INT_MAX);
  }
  p.off[n_levels] = (int)total;
  p.raw = raw;
  p.out = out;
  p.nc = num_classes;
  p.reg_max = reg_max;
  p.A = (int)total;
  p.n_levels = n_levels;
  PhaseScope phase(h, B200VA_PHASE_DFL, (cudaStream_t)stream);
  // four anchors per thread when every channel row starts 16-byte aligned
  const bool vec = total % 4 == 0 && (uintptr_t)raw % 16 == 0 && (uintptr_t)out % 16 == 0;
  const int per_block = 128 * (vec ? 4 : 1);
  dim3 grid((unsigned)((total + per_block - 1) / per_block), batch, 1 + (num_classes + kClsRows - 1) / kClsRows);
  cudaStream_t st = (cudaStream_t)stream;
  if (reg_max == 16) {
    if (vec) k_dfl_decode<16, 4><<<grid, 128, 0, st>>>(p);
    else k_dfl_decode<16, 1><<<grid, 128, 0, st>>>(p);
  } else {
    if (vec) k_dfl_decode<0, 4><<<grid, 128, 0, st>>>(p);
    else k_dfl_decode<0, 1><<<grid, 128, 0, st>>>(p);
  }
  LAUNCH_CHECK(h);
  return B200VA_OK;
}
