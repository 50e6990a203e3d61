// orb.cu — shot threading (pyannote/video/structure/thread.py): RGB resize then gray, cv2.ORB_create() features
// (8-level 1.2 pyramid, FAST-9/16 + non-max suppression, Harris re-ranking, intensity-centroid angle, rBRIEF) and
// the exact Hamming 2-NN ratio count of shot pairs.  Every stage is bit-exact against cv2 4.13 through the numpy
// restatements of oracle/thread.py; float arithmetic uses explicit _rn intrinsics (and fmaf where OpenCV's
// vectorised filter fuses) so the order of operations is the one pinned there.
#include "../../include/pv_b200.h"
#include "pv_common.cuh"
#include "orb_pattern.cuh"
#include <atomic>

extern std::atomic<long long> g_pv_launches;

namespace {

constexpr int kThreads = 1024;
constexpr int kEdge = 31;
constexpr int kHalfPatch = 15;
constexpr int kFastT = 20;

// row half-widths of the radius-15 circular patch (OpenCV's symmetric umax construction for patch size 31; pinned
// against oracle/thread.py:umax by tests/test_thread_cpu.py).  Like the pattern, a static initialiser: __constant__
// memory is per device, and an initialised symbol is loaded on every device the module is loaded on.
__constant__ int c_umax[kHalfPatch + 1] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};

// --------------------------------------------------------------------------------------------------- resize + gray
// per channel: OpenCV's 11-bit INTER_LINEAR (the taps of shot.gray_table), then RGB2GRAY (15-bit weights)
__global__ void __launch_bounds__(256) orb_resize_gray_kernel(const uint8_t* __restrict__ rgb, int H, int W,
                                                              const int* __restrict__ tab, int h, int w,
                                                              uint8_t* __restrict__ out) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h * w) return;
  const int oy = i / w, ox = i - oy * w;
  const int* tx = tab;
  const int* ty = tab + 4 * w;
  const int x0 = tx[ox], x1 = tx[w + ox], cx0 = tx[2 * w + ox], cx1 = tx[3 * w + ox];
  const int y0 = ty[oy], y1 = ty[h + oy], cy0 = ty[2 * h + oy], cy1 = ty[3 * h + oy];
  const uint8_t* img = rgb + (size_t)b * H * W * 3;
  const uint8_t* r0 = img + (size_t)y0 * W * 3;
  const uint8_t* r1 = img + (size_t)y1 * W * 3;
  int c[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const int s0 = (int)r0[3 * x0 + ch] * cx0 + (int)r0[3 * x1 + ch] * cx1;
    const int s1 = (int)r1[3 * x0 + ch] * cx0 + (int)r1[3 * x1 + ch] * cx1;
    c[ch] = min(max(((((s0 >> 4) * cy0) >> 16) + (((s1 >> 4) * cy1) >> 16) + 2) >> 2, 0), 255);
  }
  out[(size_t)b * h * w + i] = (uint8_t)((c[0] * 9798 + c[1] * 19235 + c[2] * 3735 + (1 << 14)) >> 15);
}

// --------------------------------------------------------------------------------------------------- per-frame ORB
struct Work {
  uint8_t* pyr;     // level images (plane bytes)
  uint8_t* blr;     // blurred level images
  uint8_t* score;   // FAST scores (0: not a corner)
  float* tmp;       // horizontal blur pass
  int4* cand;       // (x, y, level, FAST score) of border-filtered NMS survivors
  int* keep1;       // candidates kept by FAST score
  float* resp;      // their Harris responses
  int* keep2;       // indices into keep1 kept by Harris response
};

__host__ __device__ __forceinline__ size_t al16(size_t v) { return (v + 15) & ~(size_t)15; }

// layout: three byte planes | float plane | int4 candidates | keep1, resp, keep2 (each 16-byte aligned section)
__host__ __device__ inline size_t work_bytes(const PvOrbGeo& g) {
  const size_t p = (size_t)g.plane;
  return al16(3 * p) + al16(4 * p) + 16 * (size_t)g.cand_cap + 12 * (size_t)g.cand_cap;
}

__device__ Work carve(uint8_t* base, const PvOrbGeo& g) {
  Work w;
  const size_t p = (size_t)g.plane;
  w.pyr = base;
  w.blr = base + p;
  w.score = base + 2 * p;
  size_t o = al16(3 * p);
  w.tmp = reinterpret_cast<float*>(base + o);
  o += al16(4 * p);
  w.cand = reinterpret_cast<int4*>(base + o);
  o += 16 * (size_t)g.cand_cap;
  w.keep1 = reinterpret_cast<int*>(base + o);
  w.resp = reinterpret_cast<float*>(base + o + 4 * (size_t)g.cand_cap);
  w.keep2 = reinterpret_cast<int*>(base + o + 8 * (size_t)g.cand_cap);
  return w;
}

__device__ __forceinline__ int refl(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
  return i;
}

// FAST-9/16 circle (x, y) in OpenCV's order
__constant__ int c_ring_x[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
__constant__ int c_ring_y[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};

// FAST-9/16 score (largest threshold keeping the pixel a corner, minus 1: OpenCV's cornerScore<16>) or 0 if the
// pixel is not a corner at kFastT
__device__ int fast_score(const uint8_t* img, int cols, int x, int y) {
  const int v = img[y * cols + x];
  int d[25];
  for (int k = 0; k < 16; ++k) d[k] = v - (int)img[(y + c_ring_y[k]) * cols + x + c_ring_x[k]];
  for (int k = 16; k < 25; ++k) d[k] = d[k - 16];
  int a0 = kFastT;
  for (int k = 0; k < 16; k += 2) {
    int a = min(min(d[k + 1], d[k + 2]), min(d[k + 3], d[k + 4]));
    a = min(min(a, d[k + 5]), min(min(d[k + 6], d[k + 7]), d[k + 8]));
    a0 = max(a0, max(min(a, d[k]), min(a, d[k + 9])));
  }
  int b0 = -a0;
  for (int k = 0; k < 16; k += 2) {
    int b = max(max(d[k + 1], d[k + 2]), max(d[k + 3], d[k + 4]));
    b = max(max(b, d[k + 5]), max(max(d[k + 6], d[k + 7]), d[k + 8]));
    b0 = min(b0, min(max(b, d[k]), max(b, d[k + 9])));
  }
  const int score = -b0 - 1;
  return score >= kFastT ? score : 0;
}

__device__ float harris(const uint8_t* img, int cols, int x, int y) {
  int a = 0, b = 0, c = 0;
  for (int i = -3; i <= 3; ++i)
    for (int j = -3; j <= 3; ++j) {
      const uint8_t* p = img + (y + i) * cols + x + j;
      const int Ix = (p[1] - p[-1]) * 2 + (p[-cols + 1] - p[-cols - 1]) + (p[cols + 1] - p[cols - 1]);
      const int Iy = (p[cols] - p[-cols]) * 2 + (p[cols - 1] - p[-cols - 1]) + (p[cols + 1] - p[-cols + 1]);
      a += Ix * Ix;
      b += Iy * Iy;
      c += Ix * Iy;
    }
  const float scale = __fdiv_rn(1.f, 4.f * 7.f * 255.f);
  const float s4 = __fmul_rn(__fmul_rn(__fmul_rn(scale, scale), scale), scale);
  const float fa = (float)a, fb = (float)b, fc = (float)c;
  const float ab = __fadd_rn(fa, fb);
  float v = __fsub_rn(__fmul_rn(fa, fb), __fmul_rn(fc, fc));
  v = __fsub_rn(v, __fmul_rn(__fmul_rn(0.04f, ab), ab));
  return __fmul_rn(v, s4);
}

__device__ float fast_atan2(float y, float x) {
  const float k = (float)(180.0 / 3.14159265358979323846);
  const float p1 = 0.9997878412794807f * k, p3 = -0.3258083974640975f * k;
  const float p5 = 0.1555786518463281f * k, p7 = -0.04432655554792128f * k;
  const float eps = (float)2.220446049250313e-16;
  const float ax = fabsf(x), ay = fabsf(y);
  const bool flat = ax >= ay;
  const float c = flat ? __fdiv_rn(ay, __fadd_rn(ax, eps)) : __fdiv_rn(ax, __fadd_rn(ay, eps));
  const float c2 = __fmul_rn(c, c);
  float a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
  if (!flat) a = __fsub_rn(90.f, a);
  if (x < 0) a = __fsub_rn(180.f, a);
  if (y < 0) a = __fsub_rn(360.f, a);
  return a;
}

__global__ void __launch_bounds__(kThreads) orb_detect_kernel(const uint8_t* __restrict__ gray, PvOrbGeo g,
                                                              const int* __restrict__ tab, uint8_t* work,
                                                              size_t work_stride, float* kp,
                                                              uint8_t* desc, int* count) {
  const int f = blockIdx.x;
  const Work w = carve(work + (size_t)f * work_stride, g);
  __shared__ int hist[PV_ORB_LEVELS][256];
  __shared__ int cnt[PV_ORB_LEVELS], cut[PV_ORB_LEVELS];
  __shared__ int n_cand, n1, n2, overflow;
  for (int i = threadIdx.x; i < PV_ORB_LEVELS * 256; i += blockDim.x) (&hist[0][0])[i] = 0;
  if (threadIdx.x < PV_ORB_LEVELS) cnt[threadIdx.x] = 0;
  if (threadIdx.x == 0) n_cand = n1 = n2 = overflow = 0;
  const int n0 = g.rows[0] * g.cols[0];
  const uint8_t* src = gray + (size_t)f * n0;
  for (int i = threadIdx.x; i < n0; i += blockDim.x) w.pyr[i] = src[i];
  __syncthreads();
  // pyramid: level k from level k - 1, INTER_LINEAR_EXACT (8-bit taps, round from 16 fractional bits)
  for (int lv = 1; lv < g.n_levels; ++lv) {
    const int R = g.rows[lv], C = g.cols[lv], pc = g.cols[lv - 1];
    const int* xo = tab + g.tab_off[lv];
    const int* xc = xo + C;
    const int* yo = xc + C;
    const int* yc = yo + R;
    const uint8_t* s = w.pyr + g.off[lv - 1];
    uint8_t* d = w.pyr + g.off[lv];
    for (int i = threadIdx.x; i < R * C; i += blockDim.x) {
      const int y = i / C, x = i - y * C;
      const int a = xo[x], ca = xc[x], r = yo[y], cr = yc[y];
      const uint8_t* s0 = s + r * pc + a;
      const uint8_t* s1 = s0 + pc;
      const int h0 = (256 - ca) * s0[0] + ca * s0[1];
      const int h1 = (256 - ca) * s1[0] + ca * s1[1];
      d[i] = (uint8_t)min((h0 * (256 - cr) + h1 * cr + (1 << 15)) >> 16, 255);
    }
    __syncthreads();
  }
  // blur, horizontal pass (fmaf in tap order), FAST scores
  for (int lv = 0; lv < g.n_levels; ++lv) {
    const int R = g.rows[lv], C = g.cols[lv];
    const uint8_t* img = w.pyr + g.off[lv];
    float* t = w.tmp + g.off[lv];
    uint8_t* sc = w.score + g.off[lv];
    for (int i = threadIdx.x; i < R * C; i += blockDim.x) {
      const int y = i / C, x = i - y * C;
      float acc = __fmul_rn((float)img[y * C + refl(x - 3, C)], g.gauss[0]);
      for (int j = 1; j < 7; ++j) acc = __fmaf_rn((float)img[y * C + refl(x - 3 + j, C)], g.gauss[j], acc);
      t[i] = acc;
      sc[i] = (x >= 3 && x < C - 3 && y >= 3 && y < R - 3) ? (uint8_t)fast_score(img, C, x, y) : 0;
    }
  }
  __syncthreads();
  // blur, vertical pass (symmetric, centre first); non-max suppression + border filter into the candidate list
  for (int lv = 0; lv < g.n_levels; ++lv) {
    const int R = g.rows[lv], C = g.cols[lv];
    const float* t = w.tmp + g.off[lv];
    const uint8_t* sc = w.score + g.off[lv];
    uint8_t* bl = w.blr + g.off[lv];
    const bool any = R > 2 * kEdge && C > 2 * kEdge;
    for (int i = threadIdx.x; i < R * C; i += blockDim.x) {
      const int y = i / C, x = i - y * C;
      float acc = __fmul_rn(t[i], g.gauss[3]);
      for (int j = 1; j <= 3; ++j)
        acc = __fmaf_rn(__fadd_rn(t[refl(y - j, R) * C + x], t[refl(y + j, R) * C + x]), g.gauss[3 - j], acc);
      bl[i] = (uint8_t)min(max(__float2int_rn(acc), 0), 255);
      const int s = sc[i];
      if (!any || s == 0 || x < kEdge || x >= C - kEdge || y < kEdge || y >= R - kEdge) continue;
      bool peak = true;
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx)
          if ((dx || dy) && sc[(y + dy) * C + x + dx] >= s) peak = false;
      if (!peak) continue;
      const int k = atomicAdd(&n_cand, 1);
      if (k >= g.cand_cap) {
        overflow = 1;
        continue;
      }
      w.cand[k] = make_int4(x, y, lv, s);
      atomicAdd(&cnt[lv], 1);
      atomicAdd(&hist[lv][s], 1);
    }
  }
  __syncthreads();
  // retain-best by FAST score: keep every candidate whose score reaches the (2 * quota)-th best
  if (threadIdx.x < g.n_levels) {
    const int lv = threadIdx.x, q = 2 * g.quota[lv];
    int c = 0;
    if (cnt[lv] > q) {
      int acc = 0;
      for (c = 255; c > 0; --c) {
        acc += hist[lv][c];
        if (acc >= q) break;
      }
      if (q == 0) c = 256;
    }
    cut[lv] = c;
  }
  __syncthreads();
  const int nc = min(n_cand, g.cand_cap);
  for (int i = threadIdx.x; i < nc; i += blockDim.x) {
    const int4 c = w.cand[i];
    if (c.w < cut[c.z]) continue;
    const int k = atomicAdd(&n1, 1);
    w.keep1[k] = i;
    w.resp[k] = harris(w.pyr + g.off[c.z], g.cols[c.z], c.x, c.y);
  }
  __syncthreads();
  // retain-best by Harris response: kept iff fewer than `quota` responses of its level are strictly greater
  for (int i = threadIdx.x; i < n1; i += blockDim.x) {
    const int lv = w.cand[w.keep1[i]].z;
    const float r = w.resp[i];
    int greater = 0;
    for (int j = 0; j < n1; ++j) greater += (w.resp[j] > r && w.cand[w.keep1[j]].z == lv);
    if (greater < g.quota[lv]) w.keep2[atomicAdd(&n2, 1)] = i;
  }
  __syncthreads();
  // angle + descriptor; output slot = rank of (level, y, x) among the kept points (deterministic order)
  const int nk = n2;
  for (int i = threadIdx.x; i < nk; i += blockDim.x) {
    const int4 c = w.cand[w.keep1[w.keep2[i]]];
    const long long key = ((long long)c.z << 40) | ((long long)c.y << 20) | c.x;
    int slot = 0;
    for (int j = 0; j < nk; ++j) {
      const int4 o = w.cand[w.keep1[w.keep2[j]]];
      slot += (((long long)o.z << 40) | ((long long)o.y << 20) | o.x) < key;
    }
    const int C = g.cols[c.z];
    const uint8_t* img = w.pyr + g.off[c.z] + c.y * C + c.x;
    int m01 = 0, m10 = 0;
    for (int u = -kHalfPatch; u <= kHalfPatch; ++u) m10 += u * img[u];
    for (int v = 1; v <= kHalfPatch; ++v) {
      const int d = c_umax[v];
      int vs = 0;
      for (int u = -d; u <= d; ++u) {
        const int p = img[u + v * C], m = img[u - v * C];
        vs += p - m;
        m10 += u * (p + m);
      }
      m01 += v * vs;
    }
    const float angle = fast_atan2((float)m01, (float)m10);
    const float sc = g.scale[c.z];
    const float px = __fmul_rn((float)c.x, sc), py = __fmul_rn((float)c.y, sc);
    float* o = kp + ((size_t)f * g.cand_cap + slot) * 5;
    o[0] = px;
    o[1] = py;
    o[2] = (float)c.z;
    o[3] = w.resp[w.keep2[i]];
    o[4] = angle;
    // rBRIEF on the blurred level: centre from the scaled point, pattern rotated in float32, cvRound
    const float inv = __fdiv_rn(1.f, sc);
    const int cx = __float2int_rn(__fmul_rn(px, inv)), cy = __float2int_rn(__fmul_rn(py, inv));
    const float rad = __fmul_rn(angle, (float)(3.14159265358979323846 / 180.0));
    const float ca = (float)cos((double)rad), sa = (float)sin((double)rad);
    const uint8_t* center = w.blr + g.off[c.z] + cy * C + cx;
    uint8_t* dd = desc + ((size_t)f * g.cand_cap + slot) * 32;
    for (int byte = 0; byte < 32; ++byte) {
      int val = 0;
      for (int bit = 0; bit < 8; ++bit) {
        const int* p = c_orb_pattern + 4 * (8 * byte + bit);
        int t[2];
        for (int e = 0; e < 2; ++e) {
          const float fx = (float)p[2 * e], fy = (float)p[2 * e + 1];
          const float x = __fsub_rn(__fmul_rn(fx, ca), __fmul_rn(fy, sa));
          const float y = __fadd_rn(__fmul_rn(fx, sa), __fmul_rn(fy, ca));
          t[e] = center[__float2int_rn(y) * C + __float2int_rn(x)];
        }
        val |= (t[0] < t[1]) << bit;
      }
      dd[byte] = (uint8_t)val;
    }
  }
  if (threadIdx.x == 0) count[f] = overflow ? -1 : nk;
}

// --------------------------------------------------------------------------------------------------- matching
// one CTA per pair: every query descriptor of frame pairs[p].x against every train descriptor of pairs[p].y, train
// tiles staged in shared memory; the two smallest Hamming distances decide the float64 ratio test
constexpr int kMatchThreads = 256;

__global__ void __launch_bounds__(kMatchThreads) thread_match_kernel(const uint4* __restrict__ desc,
                                                                     const int* __restrict__ offsets,
                                                                     const int2* __restrict__ pairs,
                                                                     int* __restrict__ counts) {
  __shared__ uint4 tile[kMatchThreads * 2];
  __shared__ int red[kMatchThreads / 32];
  const int2 pr = pairs[blockIdx.x];
  const int q0 = offsets[pr.x], nq = offsets[pr.x + 1] - q0;
  const int t0 = offsets[pr.y], nt = offsets[pr.y + 1] - t0;
  int good = 0;
  if (nq >= 2 && nt >= 2) {
    for (int qb = 0; qb < nq; qb += kMatchThreads) {
      const int qi = qb + threadIdx.x;
      uint4 a = make_uint4(0, 0, 0, 0), b = a;
      if (qi < nq) {
        a = desc[2 * (size_t)(q0 + qi)];
        b = desc[2 * (size_t)(q0 + qi) + 1];
      }
      int best = 1 << 20, second = 1 << 20;
      for (int tb = 0; tb < nt; tb += kMatchThreads) {
        const int n = min(kMatchThreads, nt - tb);
        __syncthreads();
        if (threadIdx.x < n) {
          tile[2 * threadIdx.x] = desc[2 * (size_t)(t0 + tb + threadIdx.x)];
          tile[2 * threadIdx.x + 1] = desc[2 * (size_t)(t0 + tb + threadIdx.x) + 1];
        }
        __syncthreads();
        if (qi < nq)
          for (int j = 0; j < n; ++j) {
            const uint4 c = tile[2 * j], d = tile[2 * j + 1];
            const int dist = __popc(a.x ^ c.x) + __popc(a.y ^ c.y) + __popc(a.z ^ c.z) + __popc(a.w ^ c.w) +
                             __popc(b.x ^ d.x) + __popc(b.y ^ d.y) + __popc(b.z ^ d.z) + __popc(b.w ^ d.w);
            if (dist < best) {
              second = best;
              best = dist;
            } else if (dist < second) {
              second = dist;
            }
          }
      }
      if (qi < nq && (double)best < __dmul_rn(0.7, (double)second)) ++good;
    }
  }
  for (int o = 16; o > 0; o >>= 1) good += __shfl_xor_sync(0xffffffffu, good, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = good;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int k = 0; k < kMatchThreads / 32; ++k) s += red[k];
    counts[blockIdx.x] = s;
  }
}

bool geo_ok(const PvOrbGeo* g) {
  if (!g || g->n_levels < 1 || g->n_levels > PV_ORB_LEVELS || g->cand_cap < 1) return false;
  long long plane = 0;
  for (int k = 0; k < g->n_levels; ++k) {
    if (g->rows[k] < 1 || g->cols[k] < 1 || g->off[k] != plane || g->quota[k] < 0) return false;
    plane += (long long)g->rows[k] * g->cols[k];
  }
  return plane == g->plane && g->rows[0] < (1 << 20) && g->cols[0] < (1 << 20);
}

}  // namespace

// --------------------------------------------------------------------------------------------------- C ABI
extern "C" int pv_orb_resize_gray(const void* rgb, int B, int H, int W, const int* tab, int h, int w, void* gray,
                                  void* stream) {
  PV_REQUIRE(rgb && tab && gray, "pv_orb_resize_gray: null argument");
  PV_REQUIRE(B > 0 && H > 0 && W > 0 && h > 0 && w > 0 && B <= 65535, "pv_orb_resize_gray: B=%d %dx%d -> %dx%d", B, H,
             W, h, w);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  orb_resize_gray_kernel<<<dim3((unsigned)((h * w + 255) / 256), (unsigned)B), 256, 0, st>>>(
      static_cast<const uint8_t*>(rgb), H, W, tab, h, w, static_cast<uint8_t*>(gray));
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}

extern "C" int64_t pv_orb_work_bytes(const PvOrbGeo* geo) {
  if (!geo_ok(geo)) return -1;
  return (int64_t)((work_bytes(*geo) + 255) & ~(size_t)255);
}

extern "C" int pv_orb_detect(const void* gray, int B, const PvOrbGeo* geo, const int* tab, void* work, float* kp,
                             void* desc, int* count, void* stream) {
  PV_REQUIRE(gray && geo && tab && work && kp && desc && count, "pv_orb_detect: null argument");
  PV_REQUIRE(geo_ok(geo) && B > 0, "pv_orb_detect: bad geometry or B=%d", B);
  const size_t stride = (work_bytes(*geo) + 255) & ~(size_t)255;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  orb_detect_kernel<<<(unsigned)B, kThreads, 0, st>>>(static_cast<const uint8_t*>(gray), *geo, tab,
                                                      static_cast<uint8_t*>(work), stride, kp,
                                                      static_cast<uint8_t*>(desc), count);
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}

extern "C" int pv_thread_match(const void* desc, const int* offsets, const int* pairs, int P, int* counts,
                               void* stream) {
  PV_REQUIRE(desc && offsets && pairs && counts, "pv_thread_match: null argument");
  PV_REQUIRE(P > 0, "pv_thread_match: P=%d", P);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  thread_match_kernel<<<(unsigned)P, kMatchThreads, 0, st>>>(static_cast<const uint4*>(desc), offsets,
                                                             reinterpret_cast<const int2*>(pairs), counts);
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}
