// shot.cu — shot boundary detection by displaced frame difference (pyannote/video/structure/shot.py):
// RGB -> gray -> resize (OpenCV's fixed-point INTER_LINEAR, bit-exact), Farneback polynomial expansion once per
// frame (every pyramid level), then per consecutive pair the Farneback flow (update matrices, 15x15 box filter,
// 2x2 solve; 3 iterations per level) and the DFD as an exact integer sum.  Every launch covers a whole batch of
// frames or pairs; nothing is launched per frame.  Float arithmetic uses explicit _rn intrinsics so ptxas cannot
// contract mul+add pairs: the order of operations is the one of oracle/shot.py.
#include "../../include/pv_b200.h"
#include "pv_common.cuh"
#include <atomic>

extern std::atomic<long long> g_pv_launches;

namespace {

constexpr int kThreads = 512;
constexpr int kSmemMax = 227 * 1024 - 1024;   // leaves room for the static reduction array

__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double dm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double da(double a, double b) { return __dadd_rn(a, b); }

// --------------------------------------------------------------------------------------------------- gray + resize
// tab: x0[w] x1[w] cx0[w] cx1[w] y0[h] y1[h] cy0[h] cy1[h] (11-bit weights)
__device__ __forceinline__ int gray_px(const uint8_t* p) {
  return ((int)p[0] * 9798 + (int)p[1] * 19235 + (int)p[2] * 3735 + (1 << 14)) >> 15;
}

__global__ void __launch_bounds__(256) shot_gray_resize_kernel(const uint8_t* __restrict__ rgb, int H, int W,
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
  const int s0 = gray_px(r0 + 3 * x0) * cx0 + gray_px(r0 + 3 * x1) * cx1;
  const int s1 = gray_px(r1 + 3 * x0) * cx0 + gray_px(r1 + 3 * x1) * cx1;
  // the vertical pass in the 16-bit multiply-high form: (S >> 4) * beta >> 16, two terms, +2 >> 2
  const int v = ((((s0 >> 4) * cy0) >> 16) + (((s1 >> 4) * cy1) >> 16) + 2) >> 2;
  out[(size_t)b * h * w + i] = (uint8_t)min(max(v, 0), 255);
}

// --------------------------------------------------------------------------------------------------- helpers
// linear resize table at `off` for a (rows x cols) destination: x0 x1 ax0 ax1 [cols] then y0 y1 ay0 ay1 [rows]
struct LinTab {
  const float* p;
  int rows, cols;
  __device__ int x0(int x) const { return (int)p[x]; }
  __device__ int x1(int x) const { return (int)p[cols + x]; }
  __device__ float ax0(int x) const { return p[2 * cols + x]; }
  __device__ float ax1(int x) const { return p[3 * cols + x]; }
  __device__ int y0(int y) const { return (int)p[4 * cols + y]; }
  __device__ int y1(int y) const { return (int)p[4 * cols + rows + y]; }
  __device__ float ay0(int y) const { return p[4 * cols + 2 * rows + y]; }
  __device__ float ay1(int y) const { return p[4 * cols + 3 * rows + y]; }
};

// dst[rows x cols] = linear resize of src[sh x sw] (float32, products and sums rounded in order)
__device__ void resize_linear(const float* src, int sw, float* dst, const LinTab& t) {
  for (int i = threadIdx.x; i < t.rows * t.cols; i += blockDim.x) {
    const int y = i / t.cols, x = i - y * t.cols;
    const float* s0 = src + t.y0(y) * sw;
    const float* s1 = src + t.y1(y) * sw;
    const int a = t.x0(x), b = t.x1(x);
    const float wa = t.ax0(x), wb = t.ax1(x);
    const float h0 = fa(fm(s0[a], wa), fm(s0[b], wb));
    const float h1 = fa(fm(s1[a], wa), fm(s1[b], wb));
    dst[i] = fa(fm(h0, t.ay0(y)), fm(h1, t.ay1(y)));
  }
}

__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
  return i;
}

// --------------------------------------------------------------------------------------------------- polynomial expansion
// one CTA per (frame, level): level image (pre-blur, resize) then the separable expansion into R [5, rows, cols]
__global__ void __launch_bounds__(kThreads) shot_polyexp_kernel(const uint8_t* __restrict__ gray, PvShotGeo g,
                                                                const float* __restrict__ tab, float* __restrict__ gwork,
                                                                int64_t work_floats, int use_smem, float* __restrict__ R) {
  extern __shared__ float smem[];
  const int f = blockIdx.x, lv = blockIdx.y;
  const PvShotLevel& L = g.lv[lv];
  __shared__ float taps[PV_SHOT_MAX_TAPS];
  if (threadIdx.x < PV_SHOT_MAX_TAPS) taps[threadIdx.x] = L.taps[threadIdx.x];
  float* ws = use_smem ? smem : gwork + ((int64_t)f * gridDim.y + lv) * work_floats;
  const int h = g.h, w = g.w, N0 = h * w;
  const int rows = L.rows, cols = L.cols, N = rows * cols;
  float* A = ws;
  float* B = ws + N0;
  float* I = B + N0;
  float* row3 = I + N;
  const uint8_t* src = gray + (int64_t)f * N0;
  for (int i = threadIdx.x; i < N0; i += blockDim.x) A[i] = (float)src[i];
  __syncthreads();
  // pre-blur: taps along rows, then along columns (reflect-101), sums in tap order
  const int r = L.radius;
  for (int i = threadIdx.x; i < N0; i += blockDim.x) {
    const int y = i / w, x = i - y * w;
    float acc = 0.f;
    for (int j = -r; j <= r; ++j) acc = fa(acc, fm(taps[j + r], A[y * w + reflect101(x + j, w)]));
    B[i] = acc;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < N0; i += blockDim.x) {
    const int y = i / w, x = i - y * w;
    float acc = 0.f;
    for (int j = -r; j <= r; ++j) acc = fa(acc, fm(taps[j + r], B[reflect101(y + j, h) * w + x]));
    A[i] = acc;
  }
  __syncthreads();
  if (rows == h && cols == w) {
    I = A;
  } else if (L.area2x) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const int y = i / cols, x = i - y * cols;
      const float* s = A + (2 * y) * w + 2 * x;
      I[i] = fm(fa(fa(fa(s[0], s[1]), s[w]), s[w + 1]), 0.25f);
    }
  } else {
    resize_linear(A, w, I, LinTab{tab + L.dn_off, rows, cols});
  }
  __syncthreads();
  // columns: float32, rows clamped
  const int n = PV_SHOT_POLY_N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int y = i / cols, x = i - y * cols;
    float t0 = fm(I[i], g.pg[n]), t1 = 0.f, t2 = 0.f;
    for (int k = 1; k <= n; ++k) {
      const float up = I[max(y - k, 0) * cols + x];
      const float dn = I[min(y + k, rows - 1) * cols + x];
      const float p = fa(up, dn);
      t0 = fa(t0, fm(g.pg[n + k], p));
      t1 = fa(t1, fm(g.pxg[n + k], fs(dn, up)));
      t2 = fa(t2, fm(g.pxxg[n + k], p));
    }
    row3[i] = t0;
    row3[N + i] = t1;
    row3[2 * N + i] = t2;
  }
  __syncthreads();
  // rows: float64, columns replicated
  float* Rf = R + (int64_t)f * g.r_stride + L.r_off;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int y = i / cols, x = i - y * cols;
    const float* c0 = row3 + y * cols;
    const float* c1 = c0 + N;
    const float* c2 = c1 + N;
    const double g0 = g.pg[n];
    double b1 = dm(c0[x], g0), b3 = dm(c1[x], g0), b5 = dm(c2[x], g0), b2 = 0, b4 = 0, b6 = 0;
    for (int k = 1; k <= n; ++k) {
      const int xl = max(x - k, 0), xr = min(x + k, cols - 1);
      const double tg = da(c0[xr], c0[xl]);
      b1 = da(b1, dm(tg, (double)g.pg[n + k]));
      b4 = da(b4, dm(tg, (double)g.pxxg[n + k]));
      b2 = da(b2, dm(__dsub_rn(c0[xr], c0[xl]), (double)g.pxg[n + k]));
      b3 = da(b3, dm(da(c1[xr], c1[xl]), (double)g.pg[n + k]));
      b6 = da(b6, dm(__dsub_rn(c1[xr], c1[xl]), (double)g.pxg[n + k]));
      b5 = da(b5, dm(da(c2[xr], c2[xl]), (double)g.pg[n + k]));
    }
    Rf[i] = (float)dm(b3, g.ig11);
    Rf[N + i] = (float)dm(b2, g.ig11);
    Rf[2 * N + i] = (float)da(dm(b1, g.ig03), dm(b5, g.ig33));
    Rf[3 * N + i] = (float)da(dm(b1, g.ig03), dm(b4, g.ig33));
    Rf[4 * N + i] = (float)dm(b6, g.ig55);
  }
}

// --------------------------------------------------------------------------------------------------- flow + DFD
__constant__ float c_border[5] = {0.14f, 0.14f, 0.4472f, 0.8f, 1.0f};

// M [5, rows, cols] from R0, R1 (planes of N) and the flow [rows, cols, 2]
__device__ void update_matrices(const float* __restrict__ R0, const float* __restrict__ R1, const float* flow,
                                float* M, int rows, int cols) {
  const int N = rows * cols;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int y = i / cols, x = i - y * cols;
    const float dx = flow[2 * i], dy = flow[2 * i + 1];
    float fx = fa((float)x, dx), fy = fa((float)y, dy);
    const int x1 = (int)floorf(fx), y1 = (int)floorf(fy);
    fx = fs(fx, (float)x1);
    fy = fs(fy, (float)y1);
    float r2, r3, r4, r5, r6;
    if (x1 >= 0 && x1 < cols && y1 >= 0 && y1 < rows) {
      const int xb = min(x1 + 1, cols - 1), yb = min(y1 + 1, rows - 1);
      const float a00 = fm(fs(1.f, fx), fs(1.f, fy)), a01 = fm(fx, fs(1.f, fy));
      const float a10 = fm(fs(1.f, fx), fy), a11 = fm(fx, fy);
      const int p00 = y1 * cols + x1, p01 = y1 * cols + xb, p10 = yb * cols + x1, p11 = yb * cols + xb;
      float s[5];
#pragma unroll
      for (int c = 0; c < 5; ++c) {
        const float* P = R1 + c * N;
        float v = fm(a00, P[p00]);
        v = fa(v, fm(a01, P[p01]));
        v = fa(v, fm(a10, P[p10]));
        s[c] = fa(v, fm(a11, P[p11]));
      }
      r2 = s[0];
      r3 = s[1];
      r4 = fm(fa(R0[2 * N + i], s[2]), 0.5f);
      r5 = fm(fa(R0[3 * N + i], s[3]), 0.5f);
      r6 = fm(fa(R0[4 * N + i], s[4]), 0.25f);
    } else {
      r2 = r3 = 0.f;
      r4 = R0[2 * N + i];
      r5 = R0[3 * N + i];
      r6 = fm(R0[4 * N + i], 0.5f);
    }
    r2 = fm(fs(R0[i], r2), 0.5f);
    r3 = fm(fs(R0[N + i], r3), 0.5f);
    r2 = fa(r2, fa(fm(r4, dy), fm(r6, dx)));
    r3 = fa(r3, fa(fm(r6, dy), fm(r5, dx)));
    if (x < 5 || x >= cols - 5 || y < 5 || y >= rows - 5) {
      const float sxl = x < 5 ? c_border[x] : 1.f;
      const float sxr = x >= cols - 5 ? c_border[cols - 1 - x] : 1.f;
      const float syt = y < 5 ? c_border[y] : 1.f;
      const float syb = y >= rows - 5 ? c_border[rows - 1 - y] : 1.f;
      const float sc = fm(fm(fm(sxl, sxr), syt), syb);
      r2 = fm(r2, sc);
      r3 = fm(r3, sc);
      r4 = fm(r4, sc);
      r5 = fm(r5, sc);
      r6 = fm(r6, sc);
    }
    M[i] = fa(fm(r4, r4), fm(r6, r6));
    M[N + i] = fm(fa(r4, r5), r6);
    M[2 * N + i] = fa(fm(r5, r5), fm(r6, r6));
    M[3 * N + i] = fa(fm(r4, r2), fm(r6, r3));
    M[4 * N + i] = fa(fm(r6, r2), fm(r5, r3));
  }
}

// flow = solve(box(M)): column sums of 15 rows (float32, rows clamped) into V, then row sums of 15 (float64,
// columns clamped), the 2x2 system with OpenCV's 1e-3 regulariser
__device__ void box_solve(const float* M, float* V, float* flow, int rows, int cols) {
  const int N = rows * cols, m = PV_SHOT_WINSIZE / 2;
  for (int i = threadIdx.x; i < 5 * N; i += blockDim.x) {
    const int c = i / N, p = i - c * N;
    const int y = p / cols, x = p - y * cols;
    const float* P = M + c * N + x;
    float acc = 0.f;
    for (int j = -m; j <= m; ++j) acc = fa(acc, P[min(max(y + j, 0), rows - 1) * cols]);
    V[i] = acc;
  }
  __syncthreads();
  const double scale = 1.0 / (PV_SHOT_WINSIZE * PV_SHOT_WINSIZE);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int y = i / cols, x = i - y * cols;
    double s[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      const float* P = V + c * N + y * cols;
      double acc = 0.0;
      for (int j = -m; j <= m; ++j) acc = da(acc, (double)P[min(max(x + j, 0), cols - 1)]);
      s[c] = dm(acc, scale);
    }
    const double g11 = s[0], g12 = s[1], g22 = s[2], h1 = s[3], h2 = s[4];
    const double idet = 1.0 / da(__dsub_rn(dm(g11, g22), dm(g12, g12)), 1e-3);
    flow[2 * i] = (float)dm(__dsub_rn(dm(g11, h2), dm(g12, h1)), idet);
    flow[2 * i + 1] = (float)dm(__dsub_rn(dm(g22, h1), dm(g12, h2)), idet);
  }
}

// one CTA per pair (frames p, p + 1): every pyramid level, coarsest first, then the DFD at level 0
__global__ void __launch_bounds__(kThreads) shot_flow_dfd_kernel(const uint8_t* __restrict__ gray, const float* __restrict__ R,
                                                                 PvShotGeo g, const float* __restrict__ tab,
                                                                 float* __restrict__ gwork, int64_t work_floats, int use_smem,
                                                                 double* __restrict__ dfd, float* __restrict__ flow_out) {
  extern __shared__ float smem[];
  const int p = blockIdx.x;
  const int N0 = g.h * g.w;
  float* ws = use_smem ? smem : gwork + (int64_t)p * work_floats;
  float* M = ws;
  float* V = ws + 5 * N0;
  float* flow = V + 5 * N0;
  const float* Ra = R + (int64_t)p * g.r_stride;
  const float* Rb = Ra + g.r_stride;
  int prow = 0, pcol = 0;
  for (int lv = 0; lv < g.n_levels; ++lv) {
    const PvShotLevel L = g.lv[lv];
    const int rows = L.rows, cols = L.cols, N = rows * cols;
    if (lv == 0) {
      for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) flow[i] = 0.f;
    } else {
      // the coarser flow, resized per component and scaled by 1 / pyr_scale
      for (int i = threadIdx.x; i < 2 * prow * pcol; i += blockDim.x) {
        const int c = i & 1, q = i >> 1;
        V[c * prow * pcol + q] = flow[i];
      }
      __syncthreads();
      const LinTab t{tab + L.up_off, rows, cols};
      for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) {
        const int c = i & 1, q = i >> 1;
        const int y = q / cols, x = q - y * cols;
        const float* src = V + c * prow * pcol;
        const float* s0 = src + t.y0(y) * pcol;
        const float* s1 = src + t.y1(y) * pcol;
        const int a = t.x0(x), b = t.x1(x);
        const float h0 = fa(fm(s0[a], t.ax0(x)), fm(s0[b], t.ax1(x)));
        const float h1 = fa(fm(s1[a], t.ax0(x)), fm(s1[b], t.ax1(x)));
        flow[i] = fm(fa(fm(h0, t.ay0(y)), fm(h1, t.ay1(y))), 2.0f);
      }
    }
    __syncthreads();
    const float* R0 = Ra + L.r_off;
    const float* R1 = Rb + L.r_off;
    update_matrices(R0, R1, flow, M, rows, cols);
    __syncthreads();
    for (int it = 0; it < PV_SHOT_ITERATIONS; ++it) {
      box_solve(M, V, flow, rows, cols);
      __syncthreads();
      if (it < PV_SHOT_ITERATIONS - 1) {
        update_matrices(R0, R1, flow, M, rows, cols);
        __syncthreads();
      }
    }
    prow = rows;
    pcol = cols;
  }
  // DFD: reconstruct[y,x] = cur[ry,rx], r = int(max(0, min(p + d, size - 1))) with p + d rounded to float32 (a
  // Python int plus a NumPy float32 scalar stays float32); exact integer sum.
  // The reference reads the flow vector as (dy, dx) while it is stored (dx, dy): the column index moves by the
  // y component and the row index by the x component.  Reproduced as is.
  const int h = g.h, w = g.w;
  const uint8_t* prev = gray + (int64_t)p * N0;
  const uint8_t* cur = prev + N0;
  unsigned int local = 0;
  for (int i = threadIdx.x; i < N0; i += blockDim.x) {
    const int y = i / w, x = i - y * w;
    float vx = fa((float)x, flow[2 * i + 1]), vy = fa((float)y, flow[2 * i]);
    vx = ((float)(w - 1) < vx) ? (float)(w - 1) : vx;       // Python min(v, w-1): NaN stays
    vy = ((float)(h - 1) < vy) ? (float)(h - 1) : vy;
    vx = (vx > 0.f) ? vx : 0.f;                             // Python max(0, v): NaN becomes 0
    vy = (vy > 0.f) ? vy : 0.f;
    const int rx = (int)vx, ry = (int)vy;
    local += (unsigned int)abs((int)prev[i] - (int)cur[ry * w + rx]);
    if (flow_out) {
      flow_out[(int64_t)p * 2 * N0 + 2 * i] = flow[2 * i];
      flow_out[(int64_t)p * 2 * N0 + 2 * i + 1] = flow[2 * i + 1];
    }
  }
  __shared__ unsigned long long red[kThreads / 32];
  unsigned long long v = local;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long s = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) s += red[k];
    dfd[p] = (double)s / (double)N0;
  }
}

bool geo_ok(const PvShotGeo* g) {
  if (!g || g->n_levels < 1 || g->n_levels > PV_SHOT_MAX_LEVELS || g->h < 1 || g->w < 1) return false;
  const PvShotLevel& f = g->lv[g->n_levels - 1];
  if (f.rows != g->h || f.cols != g->w || f.r_off + 5LL * g->h * g->w > g->r_stride) return false;
  for (int k = 0; k < g->n_levels; ++k)
    if (g->lv[k].radius < 0 || g->lv[k].radius > PV_SHOT_MAX_TAPS / 2 || g->lv[k].rows < 1 || g->lv[k].cols < 1) return false;
  return true;
}

}  // namespace

// --------------------------------------------------------------------------------------------------- C ABI
extern "C" int pv_shot_gray_resize(const void* rgb, int B, int H, int W, const int* tab, int h, int w, void* out,
                                   void* stream) {
  PV_REQUIRE(rgb && tab && out, "pv_shot_gray_resize: null argument");
  PV_REQUIRE(B > 0 && H > 0 && W > 0 && h > 0 && w > 0 && B <= 65535, "pv_shot_gray_resize: B=%d %dx%d -> %dx%d", B, H, W, h, w);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  shot_gray_resize_kernel<<<dim3((unsigned)((h * w + 255) / 256), (unsigned)B), 256, 0, st>>>(
      static_cast<const uint8_t*>(rgb), H, W, tab, h, w, static_cast<uint8_t*>(out));
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}

extern "C" int64_t pv_shot_polyexp_work_floats(const PvShotGeo* geo) {
  if (!geo_ok(geo)) return -1;
  return 6LL * geo->h * geo->w;
}

extern "C" int64_t pv_shot_flow_work_floats(const PvShotGeo* geo) {
  if (!geo_ok(geo)) return -1;
  return 12LL * geo->h * geo->w;
}

extern "C" int pv_shot_polyexp(const void* gray, int B, const PvShotGeo* geo, const float* tab, float* work, float* R,
                               void* stream) {
  PV_REQUIRE(gray && geo && tab && R, "pv_shot_polyexp: null argument");
  PV_REQUIRE(geo_ok(geo) && B > 0, "pv_shot_polyexp: bad geometry or B=%d", B);
  const int64_t wf = 6LL * geo->h * geo->w;
  const bool use_smem = wf * 4 <= kSmemMax;
  PV_REQUIRE(use_smem || work, "pv_shot_polyexp: %lld-float workspace needed", (long long)wf);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t smem = use_smem ? (size_t)wf * 4 : 0;
  static unsigned long long attr = 0;
  if (pv_attr_needed(&attr))
    PV_CUDA_CHECK(cudaFuncSetAttribute(shot_polyexp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
  shot_polyexp_kernel<<<dim3((unsigned)B, (unsigned)geo->n_levels), kThreads, smem, st>>>(
      static_cast<const uint8_t*>(gray), *geo, tab, work, wf, use_smem ? 1 : 0, R);
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}

extern "C" int pv_shot_flow_dfd(const void* gray, const float* R, int P, const PvShotGeo* geo, const float* tab,
                                float* work, double* dfd, float* flow_out, void* stream) {
  PV_REQUIRE(gray && R && geo && tab && dfd, "pv_shot_flow_dfd: null argument");
  PV_REQUIRE(geo_ok(geo) && P > 0, "pv_shot_flow_dfd: bad geometry or P=%d", P);
  const int64_t wf = 12LL * geo->h * geo->w;
  const bool use_smem = wf * 4 <= kSmemMax;
  PV_REQUIRE(use_smem || work, "pv_shot_flow_dfd: %lld-float workspace needed", (long long)wf);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t smem = use_smem ? (size_t)wf * 4 : 0;
  static unsigned long long attr = 0;
  if (pv_attr_needed(&attr))
    PV_CUDA_CHECK(cudaFuncSetAttribute(shot_flow_dfd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
  shot_flow_dfd_kernel<<<(unsigned)P, kThreads, smem, st>>>(static_cast<const uint8_t*>(gray), R, *geo, tab, work, wf,
                                                            use_smem ? 1 : 0, dfd, flow_out);
  g_pv_launches.fetch_add(1);
  PV_CUDA_CHECK(cudaGetLastError());
  return PV_OK;
}
