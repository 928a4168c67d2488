// SIFT extractor: OpenCV's cv::SIFT::detectAndCompute (sift.dispatch.cpp / sift.simd.hpp, firstOctave = -1) followed by
// the LightGlue wrapper's pixel de-duplication (filter_dog_point, nms_radius 0), top-k and RootSIFT, for a batch of
// same-size gray images.
//
// Per pass of SIFT_SUB images:
//   base      trunc(x * 255) -> x2 INTER_LINEAR up-sample -> Gaussian blur (row pass fused with the up-sample)
//   pyramid   L+3 Gaussian layers per octave, each blurred from the previous one (OpenCV's incremental order);
//             layer 0 of octave o is layer L of octave o-1 sub-sampled with INTER_NEAREST
//   detect    DoG formed on the fly from the Gaussian layers (one subtraction: bit-identical to a stored DoG), the
//             26-neighbour test, adjustLocalExtrema (Newton steps, contrast and edge tests); one record per surviving
//             extremum, appended with an integer atomic
//   sort      per image, one CTA: records in descending (response, position) order -- a total order on content, so the
//             atomic append order never reaches an output; equal positions are adjacent (removeDuplicatedSorted)
//   orient    one warp per record: calcOrientationHist, each lane owning a bin so every bin sums its samples in
//             OpenCV's order; one keypoint per histogram peak
//   select    per image, one CTA: retainBest (ties at the cut kept), the filter_dog_point pixel rule, top-k
//   describe  one warp per kept keypoint: calcSIFTDescriptor (lanes own the 16 spatial cells, samples accumulate in
//             OpenCV's order), clip / renormalise / uchar rounding, optional RootSIFT
// No floating-point atomics: the same image in two batch slots gives the same bits.
#include <float.h>
#include <limits.h>
#include <math.h>
#include <string.h>

#include "../../include/imw_b200.h"
#include "common.cuh"

namespace {

constexpr int SIFT_SUB = 16;          // images per pass (bounds the pyramid workspace)
constexpr int IMG_BORDER = 5;         // SIFT_IMG_BORDER
constexpr int MAX_INTERP_STEPS = 5;   // SIFT_MAX_INTERP_STEPS
constexpr int ORI_BINS = 36;          // SIFT_ORI_HIST_BINS
constexpr int MAX_PEAKS = ORI_BINS / 2; // orientation peaks per extremum: strict local maxima of a circular 36-bin
                                         // histogram are never adjacent, so there are at most 18 and none is dropped
constexpr int DESC_D = 4, DESC_N = 8; // SIFT_DESCR_WIDTH, SIFT_DESCR_HIST_BINS
constexpr int MAX_TAPS = IMW_SIFT_MAX_TAPS;
constexpr int MAX_OCT = 15;

struct Taps { float k[MAX_TAPS]; int n; };

// one extremum after adjustLocalExtrema, in pyramid-octave coordinates (o = 0 is the doubled image)
struct Cand {
  float ptx, pty;   // (c + xc) * 2^o, (r + xr) * 2^o
  float size;       // sigma * 2^((layer + xi) / L) * 2^o * 2
  float resp;       // |contr|
  int o, layer, r, c;
};

struct Octave { int h, w; long long off; };   // offset of layer 0 in floats from the image's pyramid base
struct Plan {
  int n_oct, L, H, W;
  Octave oct[MAX_OCT];
  long long pyr_floats;   // per image
};

// ---------------------------------------------------------------------------------------------------------------
// host: OpenCV's kernel arithmetic
// ---------------------------------------------------------------------------------------------------------------
// getGaussianKernel(n, sigma, CV_32F) as OpenCV 4 computes it (getGaussianKernelBitExact): the half kernel
// exp(x^2 * -0.125 / sigma^2) over x = 1 - n, 3 - n, ..., sum = 2 * half + 1 (centre), scaled by 1 / sum in double,
// then cast to float
void gaussian_taps(double sigma, Taps& t) {
  int n = (int)lrint(sigma * 8 + 1) | 1;   // GaussianBlur's ksize for float images: cvRound(sigma * 4 * 2 + 1) | 1
  if (n > MAX_TAPS) n = MAX_TAPS;
  const double scale2 = -0.125 / (sigma * sigma);
  const int h = (n - 1) / 2;
  double v[MAX_TAPS], sum = 0;
  for (int i = 0, x = 1 - n; i < h; i++, x += 2) {
    v[i] = exp((double)(x * x) * scale2);
    sum += v[i];
  }
  sum = sum * 2 + 1;
  const double mul = 1 / sum;
  for (int i = 0; i < h; i++) t.k[i] = t.k[n - 1 - i] = (float)(v[i] * mul);
  t.k[h] = (float)mul;
  t.n = n;
}

int plan_octaves(int H, int W, int L, Plan& p) {
  int hb = 2 * H, wb = 2 * W;
  // nOctaves = cvRound(log2(min(cols, rows)) - 2) - firstOctave
  int n = (int)lrint(log((double)(hb < wb ? hb : wb)) / log(2.) - 2) + 1;
  if (n > MAX_OCT) n = MAX_OCT;
  if (n < 1) n = 1;
  p.n_oct = n; p.L = L; p.H = H; p.W = W;
  long long off = 0;
  int h = hb, w = wb;
  for (int o = 0; o < n; o++) {
    p.oct[o] = {h, w, off};
    off += (long long)(L + 3) * h * w;
    h /= 2; w /= 2;
  }
  p.pyr_floats = off;
  return n;
}

void layer_sigmas(const imw_sift_conf* c, double* sig) {
  // buildGaussianPyramid: sig[i] = sqrt(sig_total^2 - sig_prev^2), sig_prev = k^(i-1) sigma
  int L = c->n_octave_layers;
  double k = pow(2., 1. / L);
  // createInitialImage (doubled image) works in float: sqrtf(max(sigma^2 - 0.5f^2 * 4, 0.01f)) with a float sigma
  const float sf = (float)c->sigma;
  sig[0] = (double)sqrtf(fmaxf(sf * sf - 0.5f * 0.5f * 4, 0.01f));
  for (int i = 1; i < L + 3; i++) {
    double prev = pow(k, (double)(i - 1)) * c->sigma, total = prev * k;
    sig[i] = sqrt(total * total - prev * prev);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int p, int len) {
  if (len == 1) return 0;
  while ((unsigned)p >= (unsigned)len) p = p < 0 ? -p : 2 * len - 2 - p;
  return p;
}

// cv::hal::fastAtan32f (degrees)
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
  const float p1 = 0.9997878412794807f * (float)(180 / M_PI), p3 = -0.3258083974640975f * (float)(180 / M_PI);
  const float p5 = 0.1555786518463281f * (float)(180 / M_PI), p7 = -0.04432655554792128f * (float)(180 / M_PI);
  float ax = fabsf(x), ay = fabsf(y);
  float c = fminf(ax, ay) / (fmaxf(ax, ay) + (float)DBL_EPSILON);
  float cc = __fmul_rn(c, c);
  float a = __fmul_rn(fmaf(fmaf(fmaf(cc, p7, p5), cc, p3), cc, p1), c);
  if (!(ax >= ay)) a = 90.f - a;
  if (x < 0) a = 180.f - a;
  if (y < 0) a = 360.f - a;
  return a;
}

// ---------------------------------------------------------------------------------------------------------------
// pyramid kernels
// ---------------------------------------------------------------------------------------------------------------
// row pass of the base blur over the x2 up-sampled uint8(trunc(x * 255)) image, computed on the fly
// (INTER_LINEAR x2: weights 0.75 / 0.25, exact in fp32 on integer inputs; clamped at the borders)
__device__ __forceinline__ float up_px(const float* img, int H, int W, int y2, int x2) {
  auto q = [&](int y, int x) {
    float v = img[(size_t)y * W + x] * 255.f;
    v = fminf(fmaxf(v, 0.f), 255.f);
    return truncf(v);
  };
  int y0 = (y2 - 1) >> 1, x0 = (x2 - 1) >> 1;   // floor((d - 1) / 2)
  float fy = (y2 & 1) ? 0.25f : 0.75f, fx = (x2 & 1) ? 0.25f : 0.75f;
  int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
  y0 = max(y0, 0); x0 = max(x0, 0);
  float r0 = q(y0, x0) * (1.f - fx) + q(y0, x1) * fx;
  float r1 = q(y1, x0) * (1.f - fx) + q(y1, x1) * fx;
  return r0 * (1.f - fy) + r1 * fy;
}

__global__ void sift_base_rows(const float* __restrict__ images, int H, int W, Taps t, float* __restrict__ tmp,
                               long long tmp_stride) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  int wb = 2 * W;
  if (x >= wb) return;
  const float* img = images + (size_t)b * H * W;
  int r = t.n / 2;
  float acc = 0.f;
  for (int k = 0; k < t.n; k++) acc = fmaf(up_px(img, H, W, y, reflect101(x + k - r, wb)), t.k[k], acc);
  tmp[b * tmp_stride + (size_t)y * wb + x] = acc;
}

__global__ void sift_blur_rows(const float* __restrict__ src, long long src_stride, int h, int w, Taps t,
                               float* __restrict__ tmp, long long tmp_stride) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= w) return;
  const float* s = src + b * src_stride + (size_t)y * w;
  int r = t.n / 2;
  float acc = 0.f;
  for (int k = 0; k < t.n; k++) acc = fmaf(s[reflect101(x + k - r, w)], t.k[k], acc);
  tmp[b * tmp_stride + (size_t)y * w + x] = acc;
}

// symmetric column pass (SymmColumnFilter: centre tap, then pairs added before the multiply)
__global__ void sift_blur_cols(const float* __restrict__ tmp, long long tmp_stride, int h, int w, Taps t,
                               float* __restrict__ dst, long long dst_stride) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= w) return;
  const float* s = tmp + b * tmp_stride + x;
  int r = t.n / 2;
  float acc = s[(size_t)y * w] * t.k[r];
  for (int k = 1; k <= r; k++)
    acc = fmaf(s[(size_t)reflect101(y - k, h) * w] + s[(size_t)reflect101(y + k, h) * w], t.k[r + k], acc);
  dst[b * dst_stride + (size_t)y * w + x] = acc;
}

// INTER_NEAREST down-sampling to (h, w) = (sh / 2, sw / 2): source index floor(d * (s / d))
__global__ void sift_downsample(const float* __restrict__ src, long long stride, int sh, int sw, int h, int w, double ify,
                                double ifx, float* __restrict__ dst) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= w) return;
  int sy = min((int)floor(y * ify), sh - 1), sx = min((int)floor(x * ifx), sw - 1);
  dst[b * stride + (size_t)y * w + x] = src[b * stride + (size_t)sy * sw + sx];
}

// ---------------------------------------------------------------------------------------------------------------
// extrema + adjustLocalExtrema
// ---------------------------------------------------------------------------------------------------------------
struct DetectArgs {
  const float* pyr;        // image 0's pyramid
  long long pyr_stride;    // floats per image
  long long oct_off;       // layer 0 of this octave
  int h, w, o, layer, L;
  float contrast, edge, sigma;
  int threshold;           // floor(0.5 * contrast / L * 255)
  int cap;
  Cand* cands;             // [B][cap]
  unsigned long long* keys;// [B][cap]
  int* n_cands;            // [B]
};

__device__ __forceinline__ unsigned long long cand_key(float resp, int o, int layer, int r, int c) {
  // response (positive: 31 significant bits) then the position: a total order on content
  unsigned long long id = ((unsigned long long)(o * 8 + layer) << 26) | ((unsigned long long)r << 13) | (unsigned long long)c;
  return ((unsigned long long)__float_as_uint(resp) << 33) | id;
}

__global__ void sift_detect(DetectArgs a) {
  int c = blockIdx.x * blockDim.x + threadIdx.x + IMG_BORDER, r = blockIdx.y + IMG_BORDER, b = blockIdx.z;
  const int h = a.h, w = a.w;
  if (c >= w - IMG_BORDER) return;
  const size_t plane = (size_t)h * w;
  const float* g = a.pyr + b * a.pyr_stride + a.oct_off;   // Gaussian layers 0..L+2 of this octave
  auto dog = [&](int l, int y, int x) {
    size_t i = (size_t)y * w + x;
    return g[(l + 1) * plane + i] - g[l * plane + i];
  };
  int layer = a.layer;
  float val = dog(layer, r, c);
  if (!(fabsf(val) > (float)a.threshold)) return;
  bool is_max = val > 0, ok = true;
  for (int l = layer - 1; l <= layer + 1 && ok; l++)
    for (int dy = -1; dy <= 1 && ok; dy++)
      for (int dx = -1; dx <= 1; dx++) {
        if (l == layer && dy == 0 && dx == 0) continue;
        float v = dog(l, r + dy, c + dx);
        if (is_max ? !(val >= v) : !(val <= v)) { ok = false; break; }
      }
  if (!ok) return;

  const float img_scale = 1.f / 255.f, deriv_scale = img_scale * 0.5f, second_scale = img_scale,
              cross_scale = img_scale * 0.25f;
  float xi = 0, xr = 0, xc = 0, dDx = 0, dDy = 0, dDs = 0;
  int i = 0;
  for (; i < MAX_INTERP_STEPS; i++) {
    float v2 = dog(layer, r, c) * 2;
    dDx = (dog(layer, r, c + 1) - dog(layer, r, c - 1)) * deriv_scale;
    dDy = (dog(layer, r + 1, c) - dog(layer, r - 1, c)) * deriv_scale;
    dDs = (dog(layer + 1, r, c) - dog(layer - 1, r, c)) * deriv_scale;
    float dxx = (dog(layer, r, c + 1) + dog(layer, r, c - 1) - v2) * second_scale;
    float dyy = (dog(layer, r + 1, c) + dog(layer, r - 1, c) - v2) * second_scale;
    float dss = (dog(layer + 1, r, c) + dog(layer - 1, r, c) - v2) * second_scale;
    float dxy = (dog(layer, r + 1, c + 1) - dog(layer, r + 1, c - 1) - dog(layer, r - 1, c + 1) + dog(layer, r - 1, c - 1)) * cross_scale;
    float dxs = (dog(layer + 1, r, c + 1) - dog(layer + 1, r, c - 1) - dog(layer - 1, r, c + 1) + dog(layer - 1, r, c - 1)) * cross_scale;
    float dys = (dog(layer + 1, r + 1, c) - dog(layer + 1, r - 1, c) - dog(layer - 1, r + 1, c) + dog(layer - 1, r - 1, c)) * cross_scale;
    // Matx33f::solve(DECOMP_LU) on a 3x3 system: Cramer's rule (Matx_FastSolveOp<float, 3, 1>); zeros when singular
    float a00 = dxx, a01 = dxy, a02 = dxs, a10 = dxy, a11 = dyy, a12 = dys, a20 = dxs, a21 = dys, a22 = dss;
    float det = a00 * (a11 * a22 - a21 * a12) - a01 * (a10 * a22 - a20 * a12) + a02 * (a10 * a21 - a20 * a11);
    float X0 = 0, X1 = 0, X2 = 0;
    if (det != 0) {
      float d = 1.f / det, b0 = dDx, b1 = dDy, b2 = dDs;
      X0 = d * (b0 * (a11 * a22 - a12 * a21) - a01 * (b1 * a22 - a12 * b2) + a02 * (b1 * a21 - a11 * b2));
      X1 = d * (a00 * (b1 * a22 - a12 * b2) - b0 * (a10 * a22 - a12 * a20) + a02 * (a10 * b2 - b1 * a20));
      X2 = d * (a00 * (a11 * b2 - b1 * a21) - a01 * (a10 * b2 - b1 * a20) + b0 * (a10 * a21 - a11 * a20));
    }
    xi = -X2; xr = -X1; xc = -X0;
    if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
    const float big = (float)(INT_MAX / 3);
    if (fabsf(xi) > big || fabsf(xr) > big || fabsf(xc) > big) return;
    c += __float2int_rn(xc); r += __float2int_rn(xr); layer += __float2int_rn(xi);
    if (layer < 1 || layer > a.L || c < IMG_BORDER || c >= w - IMG_BORDER || r < IMG_BORDER || r >= h - IMG_BORDER) return;
  }
  if (i >= MAX_INTERP_STEPS) return;
  float contr;
  {
    dDx = (dog(layer, r, c + 1) - dog(layer, r, c - 1)) * deriv_scale;
    dDy = (dog(layer, r + 1, c) - dog(layer, r - 1, c)) * deriv_scale;
    dDs = (dog(layer + 1, r, c) - dog(layer - 1, r, c)) * deriv_scale;
    float t = dDx * xc + dDy * xr + dDs * xi;
    contr = dog(layer, r, c) * img_scale + t * 0.5f;
    if (fabsf(contr) * a.L < a.contrast) return;
    float v2 = dog(layer, r, c) * 2.f;
    float dxx = (dog(layer, r, c + 1) + dog(layer, r, c - 1) - v2) * second_scale;
    float dyy = (dog(layer, r + 1, c) + dog(layer, r - 1, c) - v2) * second_scale;
    float dxy = (dog(layer, r + 1, c + 1) - dog(layer, r + 1, c - 1) - dog(layer, r - 1, c + 1) + dog(layer, r - 1, c - 1)) * cross_scale;
    float tr = dxx + dyy, det = dxx * dyy - dxy * dxy;
    if (det <= 0 || tr * tr * a.edge >= (a.edge + 1) * (a.edge + 1) * det) return;
  }
  Cand k;
  k.ptx = (c + xc) * (float)(1 << a.o);
  k.pty = (r + xr) * (float)(1 << a.o);
  k.size = a.sigma * powf(2.f, (layer + xi) / a.L) * (float)(1 << a.o) * 2;
  k.resp = fabsf(contr);
  k.o = a.o; k.layer = layer; k.r = r; k.c = c;
  int slot = atomicAdd(&a.n_cands[b], 1);
  if (slot < a.cap) {
    a.cands[(size_t)b * a.cap + slot] = k;
    a.keys[(size_t)b * a.cap + slot] = cand_key(k.resp, a.o, layer, r, c);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// per-image sort: descending 64-bit keys with an int payload, bitonic over the next power of two (one CTA)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) sift_sort(unsigned long long* keys, int* vals, const int* n_cands, int cap) {
  const int b = blockIdx.x;
  unsigned long long* K = keys + (size_t)b * cap;
  int* V = vals + (size_t)b * cap;
  const int n = min(n_cands[b], cap);
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    if (i >= n) K[i] = 0ull;   // below every real key (responses are > 0)
    V[i] = i;
  }
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        int ixj = i ^ j;
        if (ixj > i) {
          unsigned long long x = K[i], y = K[ixj];
          bool desc = (i & k) == 0;
          if (desc ? (x < y) : (x > y)) {
            K[i] = y; K[ixj] = x;
            int t = V[i]; V[i] = V[ixj]; V[ixj] = t;
          }
        }
      }
      __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// calcOrientationHist: one warp per sorted record
// ---------------------------------------------------------------------------------------------------------------
struct OrientArgs {
  const float* pyr; long long pyr_stride;
  Plan plan;
  const Cand* cands; const unsigned long long* keys; const int* order; const int* n_cands; int cap;
  float* angles;   // [B][cap][MAX_PEAKS] (sorted-slot order)
  int* n_peaks;    // [B][cap]
};

constexpr int ORIENT_WARPS = 8;

__global__ void __launch_bounds__(ORIENT_WARPS * 32) sift_orient(OrientArgs a) {
  __shared__ float s_val[ORIENT_WARPS][32];
  __shared__ int s_bin[ORIENT_WARPS][32];
  __shared__ float s_hist[ORIENT_WARPS][ORI_BINS + 4];
  __shared__ float s_smooth[ORIENT_WARPS][ORI_BINS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y, s = blockIdx.x * ORIENT_WARPS + wid;
  const int n = min(a.n_cands[b], a.cap);
  if (s >= n) return;
  const size_t base = (size_t)b * a.cap;
  int np = 0;
  if (!(s > 0 && a.keys[base + s] == a.keys[base + s - 1])) {   // removeDuplicatedSorted: same (o, layer, r, c)
    const Cand k = a.cands[base + a.order[base + s]];
    const Octave oc = a.plan.oct[k.o];
    const float* img = a.pyr + b * a.pyr_stride + oc.off + (size_t)k.layer * oc.h * oc.w;
    const float scl = k.size * 0.5f / (float)(1 << k.o);
    const int radius = __float2int_rn(4.5f * scl);
    const float sigma = 1.5f * scl, expf_scale = -1.f / (2.f * sigma * sigma);
    const int side = 2 * radius + 1, total = side * side;
    float acc0 = 0.f, acc1 = 0.f;   // bins lane and lane + 32
    for (int t0 = 0; t0 < total; t0 += 32) {
      int t = t0 + lane, bin = -1;
      float v = 0.f;
      if (t < total) {
        int i = t / side - radius, j = t % side - radius;
        int y = k.r + i, x = k.c + j;
        if (y > 0 && y < oc.h - 1 && x > 0 && x < oc.w - 1) {
          float dx = img[(size_t)y * oc.w + x + 1] - img[(size_t)y * oc.w + x - 1];
          float dy = img[(size_t)(y - 1) * oc.w + x] - img[(size_t)(y + 1) * oc.w + x];
          float wgt = expf((float)(i * i + j * j) * expf_scale);
          float ori = fast_atan2_deg(dy, dx);
          float mag = sqrtf(fmaf(dx, dx, __fmul_rn(dy, dy)));
          bin = __float2int_rn((ORI_BINS / 360.f) * ori);
          if (bin >= ORI_BINS) bin -= ORI_BINS;
          if (bin < 0) bin += ORI_BINS;
          v = __fmul_rn(wgt, mag);
        }
      }
      s_bin[wid][lane] = bin;
      s_val[wid][lane] = v;
      __syncwarp();
      const int m = min(32, total - t0);
      for (int q = 0; q < m; q++) {   // every bin adds its samples in sample order
        int bq = s_bin[wid][q];
        if (bq == lane) acc0 += s_val[wid][q];
        else if (bq == lane + 32) acc1 += s_val[wid][q];
      }
      __syncwarp();
    }
    float* th = s_hist[wid] + 2;
    th[lane] = acc0;
    if (lane < ORI_BINS - 32) th[lane + 32] = acc1;
    __syncwarp();
    if (lane == 0) {
      th[-1] = th[ORI_BINS - 1]; th[-2] = th[ORI_BINS - 2]; th[ORI_BINS] = th[0]; th[ORI_BINS + 1] = th[1];
      float* hist = s_smooth[wid];
      float omax;
      for (int q = 0; q < ORI_BINS; q++)
        hist[q] = (th[q - 2] + th[q + 2]) * (1.f / 16.f) + (th[q - 1] + th[q + 1]) * (4.f / 16.f) + th[q] * (6.f / 16.f);
      omax = hist[0];
      for (int q = 1; q < ORI_BINS; q++) omax = fmaxf(omax, hist[q]);
      const float thr = omax * 0.8f;
      for (int q = 0; q < ORI_BINS; q++) {
        int l = q > 0 ? q - 1 : ORI_BINS - 1, r2 = q < ORI_BINS - 1 ? q + 1 : 0;
        if (hist[q] > hist[l] && hist[q] > hist[r2] && hist[q] >= thr) {
          float bin = q + 0.5f * (hist[l] - hist[r2]) / (hist[l] - 2 * hist[q] + hist[r2]);
          bin = bin < 0 ? ORI_BINS + bin : bin >= ORI_BINS ? bin - ORI_BINS : bin;
          float angle = 360.f - (360.f / ORI_BINS) * bin;
          if (fabsf(angle - 360.f) < FLT_EPSILON) angle = 0.f;
          a.angles[(base + s) * MAX_PEAKS + np++] = angle;
        }
      }
    }
  }
  if (lane == 0) a.n_peaks[base + s] = np;
}

// ---------------------------------------------------------------------------------------------------------------
// per-image selection (one CTA): retainBest, filter_dog_point, top-k
// ---------------------------------------------------------------------------------------------------------------
constexpr int SEL_THREADS = 1024;

// exclusive scan of v over the CTA; returns the block total
__device__ int block_scan(int v, int* excl, int* s_warp) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int x = v;
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[wid] = x;
  __syncthreads();
  if (wid == 0) {
    int t = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += y;
    }
    s_warp[lane] = t;   // inclusive warp totals
  }
  __syncthreads();
  int total = s_warp[31];
  *excl = x - v + (wid > 0 ? s_warp[wid - 1] : 0);
  __syncthreads();
  return total;
}

struct SelectArgs {
  const Cand* cands; const unsigned long long* keys; const int* order; const int* n_cands; int cap;
  const float* angles; const int* n_peaks;
  int* kp_slot;            // [B][cap]: keypoint -> (sorted slot << 5) | peak, before the pixel rule
  int* sel;                // [B][cap]: selected keypoints (same encoding)
  unsigned long long* pix; // [B][H][W] pixel-rule map (zeroed)
  int H, W;
  int nfeatures, max_keypoints, pixel_rule, out_cap;
  int* counts_out;         // [2][B_total] at this pass's offset
  int B_total;
  int* n_sel;              // [B]
};

__global__ void __launch_bounds__(SEL_THREADS) sift_select(SelectArgs a) {
  __shared__ int s_warp[32];
  __shared__ int s_carry, s_cut;
  __shared__ float s_thr;
  const int b = blockIdx.x, tid = threadIdx.x;
  const size_t base = (size_t)b * a.cap;
  const int n_raw = a.n_cands[b], n = min(n_raw, a.cap);
  if (tid == 0) { s_carry = 0; s_cut = -1; }
  __syncthreads();
  // keypoint list in slot order (descending response; peaks of one extremum share its response)
  for (int s0 = 0; s0 < n; s0 += SEL_THREADS) {
    int s = s0 + tid, np = s < n ? a.n_peaks[base + s] : 0, ex;
    int tot = block_scan(np, &ex, s_warp);
    int off = s_carry + ex;
    for (int p = 0; p < np; p++)
      if (off + p < a.cap) a.kp_slot[base + off + p] = (s << 5) | p;
    __syncthreads();
    if (tid == 0) s_carry += tot;
    __syncthreads();
  }
  int total = s_carry;
  __syncthreads();   // every thread has read s_carry before thread 0 reuses it below
  bool overflow = n_raw > a.cap || total > a.cap;
  total = min(total, a.cap);
  int kept = total;
  if (a.nfeatures > 0 && total > a.nfeatures) {   // retainBest: every keypoint whose response ties the n-th is kept
    if (tid == 0) s_thr = a.cands[base + a.order[base + (a.kp_slot[base + a.nfeatures - 1] >> 5)]].resp;
    __syncthreads();
    const float thr = s_thr;
    for (int k = a.nfeatures - 1 + tid; k < total; k += SEL_THREADS) {
      bool in = a.cands[base + a.order[base + (a.kp_slot[base + k] >> 5)]].resp >= thr;
      bool next_in = k + 1 < total && a.cands[base + a.order[base + (a.kp_slot[base + k + 1] >> 5)]].resp >= thr;
      if (in && !next_in) s_cut = k + 1;
    }
    __syncthreads();
    kept = s_cut;
  }
  // filter_dog_point(nms_radius = 0): per pixel round(pt - 0.5), the highest score wins, then the lowest |ori|;
  // exact ties all stay.  One 64-bit integer max per pixel: (score bits, ~|ori| bits).
  unsigned long long* pix = a.pix + (size_t)b * a.H * a.W;
  auto kp_key = [&](int k, int* pidx) {
    int e = a.kp_slot[base + k], s = e >> 5, p = e & 31;
    const Cand c = a.cands[base + a.order[base + s]];
    float x = c.ptx * 0.5f, y = c.pty * 0.5f;
    int ix = min(max(__float2int_rn(x - 0.5f), 0), a.W - 1), iy = min(max(__float2int_rn(y - 0.5f), 0), a.H - 1);
    *pidx = iy * a.W + ix;
    float ori = fabsf(a.angles[(base + s) * MAX_PEAKS + p] * (float)(M_PI / 180));
    return ((unsigned long long)__float_as_uint(c.resp) << 32) | (unsigned long long)(~__float_as_uint(ori));
  };
  if (a.pixel_rule) {
    for (int k = tid; k < kept; k += SEL_THREADS) {
      int pi;
      unsigned long long key = kp_key(k, &pi);
      atomicMax(&pix[pi], key);
    }
    __syncthreads();
  }
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int k0 = 0; k0 < kept; k0 += SEL_THREADS) {
    int k = k0 + tid, keep = 0, ex;
    if (k < kept) {
      keep = 1;
      if (a.pixel_rule) {
        int pi;
        unsigned long long key = kp_key(k, &pi);
        keep = atomicOr(&pix[pi], 0ull) == key;
      }
    }
    int tot = block_scan(keep, &ex, s_warp);
    if (keep) a.sel[base + s_carry + ex] = a.kp_slot[base + k];
    __syncthreads();
    if (tid == 0) s_carry += tot;
    __syncthreads();
  }
  int n_final = s_carry;
  if (a.max_keypoints > 0 && n_final > a.max_keypoints) n_final = a.max_keypoints;   // top-k of a descending list
  if (tid == 0) {
    int written = min(n_final, a.out_cap);
    a.n_sel[b] = written;
    a.counts_out[b] = written;
    a.counts_out[a.B_total + b] = overflow ? -1 : n_final;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// calcSIFTDescriptor: one warp per selected keypoint; lanes 0..15 own the 16 interior cells of the (d+2)^2 grid
// (the border cells only ever receive samples that are discarded), so each bin sums in OpenCV's sample order
// ---------------------------------------------------------------------------------------------------------------
struct DescArgs {
  const float* pyr; long long pyr_stride;
  Plan plan;
  const Cand* cands; const int* order; const float* angles; const int* sel; const int* n_sel; int cap;
  int out_cap, rootsift;
  float* keypoints; float* scores; float* scales; float* oris; float* descriptors;   // this pass's slice
};

constexpr int DESC_WARPS = 8;

__global__ void __launch_bounds__(DESC_WARPS * 32) sift_describe(DescArgs a) {
  __shared__ float s_v[DESC_WARPS][8][33];
  __shared__ int s_idx[DESC_WARPS][32];   // (r0 + 1) * 6 + (c0 + 1) << 4 | o0, -1 = no sample
  __shared__ float s_hist[DESC_WARPS][16][DESC_N + 2];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y, j = blockIdx.x * DESC_WARPS + wid;
  if (j >= a.n_sel[b]) return;
  const size_t base = (size_t)b * a.cap;
  const int e = a.sel[base + j], s = e >> 5, p = e & 31;
  const Cand k = a.cands[base + a.order[base + s]];
  const float kangle = a.angles[(base + s) * MAX_PEAKS + p];
  const size_t o_ = (size_t)b * a.out_cap + j;
  if (lane == 0) {
    a.keypoints[o_ * 2] = k.ptx * 0.5f;
    a.keypoints[o_ * 2 + 1] = k.pty * 0.5f;
    a.scores[o_] = k.resp;
    a.scales[o_] = k.size * 0.5f;
    a.oris[o_] = kangle * (float)(M_PI / 180);
  }
  const Octave oc = a.plan.oct[k.o];
  const float* img = a.pyr + b * a.pyr_stride + oc.off + (size_t)k.layer * oc.h * oc.w;
  const int rows = oc.h, cols = oc.w;
  // calcDescriptors: the keypoint mapped back to its octave (powers of two: exact), angle 360 - kpt.angle
  const float ptx = k.ptx / (float)(1 << k.o), pty = k.pty / (float)(1 << k.o);
  const float scl = k.size / (float)(1 << k.o) * 0.5f;
  float ori = 360.f - kangle;
  if (fabsf(ori - 360.f) < FLT_EPSILON) ori = 0.f;
  const int px = __float2int_rn(ptx), py = __float2int_rn(pty);
  // cosf / sinf of the fp32 angle in radians, evaluated as double cospi / sinpi (no large-argument reduction path)
  // and rounded once to float, which is what a correctly rounded cosf / sinf returns
  const double ang = (double)(ori * (float)(M_PI / 180)) / M_PI;
  float cos_t = (float)cospi(ang), sin_t = (float)sinpi(ang);
  const float bins_per_rad = DESC_N / 360.f, exp_scale = -1.f / (DESC_D * DESC_D * 0.5f);
  const float hist_width = 3.f * scl;
  int radius = __float2int_rn(hist_width * 1.4142135623730951f * (DESC_D + 1) * 0.5f);
  radius = min(radius, (int)sqrt((double)cols * cols + (double)rows * rows));
  cos_t /= hist_width;
  sin_t /= hist_width;
  float* hist = s_hist[wid][lane & 15];
  for (int q = 0; q < DESC_N + 2; q++) if (lane < 16) hist[q] = 0.f;
  const int my_r = (lane & 15) / DESC_D + 1, my_c = (lane & 15) % DESC_D + 1;
  const int side = 2 * radius + 1, total = side * side;
  for (int t0 = 0; t0 < total; t0 += 32) {
    int t = t0 + lane, idx = -1;
    if (t < total) {
      int i = t / side - radius, jj = t % side - radius;
      float c_rot = __fmul_rn((float)jj, cos_t) - __fmul_rn((float)i, sin_t);
      float r_rot = __fmul_rn((float)jj, sin_t) + __fmul_rn((float)i, cos_t);
      float rbin = r_rot + DESC_D / 2 - 0.5f, cbin = c_rot + DESC_D / 2 - 0.5f;
      int r = py + i, c = px + jj;
      if (rbin > -1 && rbin < DESC_D && cbin > -1 && cbin < DESC_D && r > 0 && r < rows - 1 && c > 0 && c < cols - 1) {
        float dx = img[(size_t)r * cols + c + 1] - img[(size_t)r * cols + c - 1];
        float dy = img[(size_t)(r - 1) * cols + c] - img[(size_t)(r + 1) * cols + c];
        float wgt = expf(__fmul_rn(__fmul_rn(c_rot, c_rot) + __fmul_rn(r_rot, r_rot), exp_scale));
        float gori = fast_atan2_deg(dy, dx);
        float gmag = sqrtf(fmaf(dx, dx, __fmul_rn(dy, dy)));
        float obin = __fmul_rn(gori - ori, bins_per_rad);
        float mag = __fmul_rn(gmag, wgt);
        int r0 = (int)floorf(rbin), c0 = (int)floorf(cbin), o0 = (int)floorf(obin);
        rbin -= r0; cbin -= c0; obin -= o0;
        if (o0 < 0) o0 += DESC_N;
        if (o0 >= DESC_N) o0 -= DESC_N;
        float v_r1 = __fmul_rn(mag, rbin), v_r0 = mag - v_r1;
        float v_rc11 = __fmul_rn(v_r1, cbin), v_rc10 = v_r1 - v_rc11;
        float v_rc01 = __fmul_rn(v_r0, cbin), v_rc00 = v_r0 - v_rc01;
        float v111 = __fmul_rn(v_rc11, obin), v110 = v_rc11 - v111;
        float v101 = __fmul_rn(v_rc10, obin), v100 = v_rc10 - v101;
        float v011 = __fmul_rn(v_rc01, obin), v010 = v_rc01 - v011;
        float v001 = __fmul_rn(v_rc00, obin), v000 = v_rc00 - v001;
        // [dr][dc][do]
        s_v[wid][0][lane] = v000; s_v[wid][1][lane] = v001; s_v[wid][2][lane] = v010; s_v[wid][3][lane] = v011;
        s_v[wid][4][lane] = v100; s_v[wid][5][lane] = v101; s_v[wid][6][lane] = v110; s_v[wid][7][lane] = v111;
        idx = (((r0 + 1) * (DESC_D + 2) + (c0 + 1)) << 4) | o0;
      }
    }
    s_idx[wid][lane] = idx;
    __syncwarp();
    if (lane < 16) {
      const int m = min(32, total - t0);
      for (int q = 0; q < m; q++) {
        int e2 = s_idx[wid][q];
        if (e2 < 0) continue;
        int cell = e2 >> 4, o0 = e2 & 15;
        int dr = my_r - cell / (DESC_D + 2), dc = my_c - cell % (DESC_D + 2);
        if ((unsigned)dr <= 1u && (unsigned)dc <= 1u) {
          int v = (dr * 2 + dc) * 2;
          hist[o0] += s_v[wid][v][q];
          hist[o0 + 1] += s_v[wid][v + 1][q];
        }
      }
    }
    __syncwarp();
  }
  // circular orientation wrap, then clip at 0.2 |h|, renormalise, uchar rounding of h * 512 / |h|
  float d[DESC_N];
  float ss = 0.f;
  if (lane < 16) {
    hist[0] += hist[DESC_N];
    hist[1] += hist[DESC_N + 1];
#pragma unroll
    for (int q = 0; q < DESC_N; q++) { d[q] = hist[q]; ss += d[q] * d[q]; }
  } else {
#pragma unroll
    for (int q = 0; q < DESC_N; q++) d[q] = 0.f;
  }
  float nrm2 = warp_sum(ss);
  const float thr = sqrtf(nrm2) * 0.2f;
  ss = 0.f;
#pragma unroll
  for (int q = 0; q < DESC_N; q++) { d[q] = fminf(d[q], thr); ss += d[q] * d[q]; }
  nrm2 = 512.f / fmaxf(sqrtf(warp_sum(ss)), FLT_EPSILON);
#pragma unroll
  for (int q = 0; q < DESC_N; q++) d[q] = fminf(fmaxf(rintf(d[q] * nrm2), 0.f), 255.f);
  if (a.rootsift) {   // sift_to_rootsift: L1 normalise (eps 1e-6), clip(1e-6).sqrt, L2 normalise (eps 1e-6)
    float l1 = 0.f;
#pragma unroll
    for (int q = 0; q < DESC_N; q++) l1 += fabsf(d[q]);
    l1 = fmaxf(warp_sum(l1), 1e-6f);
    float l2 = 0.f;
#pragma unroll
    for (int q = 0; q < DESC_N; q++) { d[q] = sqrtf(fmaxf(d[q] / l1, 1e-6f)); if (lane < 16) l2 += d[q] * d[q]; }
    l2 = fmaxf(sqrtf(warp_sum(l2)), 1e-6f);
#pragma unroll
    for (int q = 0; q < DESC_N; q++) d[q] = d[q] / l2;
  }
  if (lane < 16) {
    float* out = a.descriptors + o_ * 128 + lane * DESC_N;
#pragma unroll
    for (int q = 0; q < DESC_N; q++) out[q] = d[q];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// workspace
// ---------------------------------------------------------------------------------------------------------------
int cand_cap(int H, int W) {
  long long n = (long long)H * W / 8;
  int c = 4096;
  while (c < n && c < (1 << 22)) c <<= 1;
  return c;
}

struct SiftBuffers {
  float *pyr, *tmp;
  Cand* cands;
  unsigned long long *keys, *pix;
  int *order, *n_cands, *n_peaks, *kp_slot, *sel, *n_sel;
  float* angles;
};

void sift_carve(Workspace& ws, SiftBuffers& s, const Plan& p, int sub) {
  const int cap = cand_cap(p.H, p.W);
  s.pyr = ws.take<float>((size_t)sub * p.pyr_floats);
  s.tmp = ws.take<float>((size_t)sub * 4 * p.H * p.W);
  s.cands = ws.take<Cand>((size_t)sub * cap);
  s.keys = ws.take<unsigned long long>((size_t)sub * cap);
  s.pix = ws.take<unsigned long long>((size_t)sub * p.H * p.W);
  s.order = ws.take<int>((size_t)sub * cap);
  s.n_cands = ws.take<int>(sub);
  s.n_peaks = ws.take<int>((size_t)sub * cap);
  s.kp_slot = ws.take<int>((size_t)sub * cap);
  s.sel = ws.take<int>((size_t)sub * cap);
  s.n_sel = ws.take<int>(sub);
  s.angles = ws.take<float>((size_t)sub * cap * MAX_PEAKS);
}

int check_conf(const imw_sift_conf* c, int H, int W) {
  IMW_REQUIRE(c != nullptr, "imw_sift: conf is NULL");
  IMW_REQUIRE(c->n_octave_layers >= 1 && c->n_octave_layers <= 7, "imw_sift: n_octave_layers %d not in [1, 7]", c->n_octave_layers);
  IMW_REQUIRE(c->sigma > 0, "imw_sift: sigma %g must be > 0", c->sigma);
  double sig[16];
  layer_sigmas(c, sig);
  for (int i = 0; i < c->n_octave_layers + 3; i++)
    IMW_REQUIRE(((int)lrint(sig[i] * 8 + 1) | 1) <= MAX_TAPS, "imw_sift: blur sigma %g needs more than %d taps", sig[i], MAX_TAPS);
  IMW_REQUIRE(c->nms_radius == -1 || c->nms_radius == 0, "imw_sift: nms_radius %d (only None = -1 and 0 are built)", c->nms_radius);
  IMW_REQUIRE(H >= 1 && W >= 1 && 2 * H <= 8192 && 2 * W <= 8192, "imw_sift: image %dx%d out of range (1..4096)", W, H);
  return 0;
}

}  // namespace

extern "C" int imw_sift_plan(const imw_sift_conf* conf, int height, int width, int* n_octaves, int* ksizes, float* taps) {
  int rc = check_conf(conf, height, width);
  if (rc) return rc;
  Plan p;
  plan_octaves(height, width, conf->n_octave_layers, p);
  if (n_octaves) *n_octaves = p.n_oct;
  double sig[16];
  layer_sigmas(conf, sig);
  for (int i = 0; i < conf->n_octave_layers + 3; i++) {
    Taps t;
    gaussian_taps(sig[i], t);
    if (ksizes) ksizes[i] = t.n;
    if (taps) for (int q = 0; q < MAX_TAPS; q++) taps[i * MAX_TAPS + q] = q < t.n ? t.k[q] : 0.f;
  }
  return 0;
}

extern "C" size_t imw_sift_workspace_bytes(const imw_sift_conf* conf, int batch, int height, int width) {
  if (check_conf(conf, height, width)) return 0;
  Plan p;
  plan_octaves(height, width, conf->n_octave_layers, p);
  SiftBuffers s;
  Workspace ws(nullptr, 0);
  sift_carve(ws, s, p, batch < SIFT_SUB ? batch : SIFT_SUB);
  return ws.off + 256;
}

extern "C" int imw_sift_forward(const imw_sift_conf* conf, int batch, int height, int width, const float* images, int cap,
                                float* keypoints, float* scores, float* scales, float* oris, float* descriptors, int* counts,
                                float* dbg_pyramid, void* workspace, size_t workspace_bytes, imw_stream_t stream) {
  int rc = check_conf(conf, height, width);
  if (rc) return rc;
  IMW_REQUIRE(batch >= 0 && cap >= 0, "imw_sift_forward: batch %d / cap %d", batch, cap);
  if (batch == 0) return 0;
  IMW_REQUIRE(images && counts && (cap == 0 || (keypoints && scores && scales && oris && descriptors)),
              "imw_sift_forward: NULL output");
  cudaStream_t st = (cudaStream_t)stream;
  const int L = conf->n_octave_layers, H = height, W = width;
  Plan p;
  plan_octaves(H, W, L, p);
  const int sub = batch < SIFT_SUB ? batch : SIFT_SUB;
  SiftBuffers s;
  Workspace ws(workspace, workspace_bytes);
  sift_carve(ws, s, p, sub);
  if (ws.overflow || !workspace) {
    imw_set_error("imw_sift_forward: workspace too small (%zu < %zu)", workspace_bytes, ws.off);
    return IMW_ERR_WORKSPACE;
  }
  const int ccap = cand_cap(H, W);
  double sig[16];
  layer_sigmas(conf, sig);
  Taps taps[10];
  for (int i = 0; i < L + 3; i++) gaussian_taps(sig[i], taps[i]);
  const long long ps = p.pyr_floats, ts = 4LL * H * W;
  const int threshold = (int)floor(0.5 * conf->contrast_threshold / L * 255);
  const int nf = conf->max_keypoints > 0 ? conf->max_keypoints : 0;

  for (int b0 = 0; b0 < batch; b0 += sub) {
    const int nb = batch - b0 < sub ? batch - b0 : sub;
    // --- Gaussian pyramid
    for (int o = 0; o < p.n_oct; o++) {
      const Octave oc = p.oct[o];
      dim3 blk(128), grd(ceil_div(oc.w, 128), oc.h, nb);
      float* L0 = s.pyr + oc.off;
      if (o == 0) {
        sift_base_rows<<<grd, blk, 0, st>>>(images + (size_t)b0 * H * W, H, W, taps[0], s.tmp, ts);
        IMW_CHECK_LAUNCH_T("sift_base_rows");
        sift_blur_cols<<<grd, blk, 0, st>>>(s.tmp, ts, oc.h, oc.w, taps[0], L0, ps);
        IMW_CHECK_LAUNCH_T("sift_blur_cols");
      } else {
        const Octave pc = p.oct[o - 1];
        sift_downsample<<<grd, blk, 0, st>>>(s.pyr + pc.off + (size_t)L * pc.h * pc.w, ps, pc.h, pc.w, oc.h, oc.w,
                                             1.0 / ((double)oc.h / pc.h), 1.0 / ((double)oc.w / pc.w), L0);
        // (same stride: the destination pointer is offset, the per-image stride is the pyramid's)
        IMW_CHECK_LAUNCH_T("sift_downsample");
      }
      for (int i = 1; i < L + 3; i++) {
        float* src = L0 + (size_t)(i - 1) * oc.h * oc.w;
        sift_blur_rows<<<grd, blk, 0, st>>>(src, ps, oc.h, oc.w, taps[i], s.tmp, ts);
        IMW_CHECK_LAUNCH_T("sift_blur_rows");
        sift_blur_cols<<<grd, blk, 0, st>>>(s.tmp, ts, oc.h, oc.w, taps[i], src + (size_t)oc.h * oc.w, ps);
        IMW_CHECK_LAUNCH_T("sift_blur_cols");
      }
    }
    if (dbg_pyramid)
      IMW_CHECK_CUDA(cudaMemcpyAsync(dbg_pyramid + (size_t)b0 * ps, s.pyr, (size_t)nb * ps * sizeof(float),
                                     cudaMemcpyDeviceToDevice, st));
    // --- extrema
    IMW_CHECK_CUDA(cudaMemsetAsync(s.n_cands, 0, sizeof(int) * nb, st));
    for (int o = 0; o < p.n_oct; o++) {
      const Octave oc = p.oct[o];
      if (oc.h <= 2 * IMG_BORDER || oc.w <= 2 * IMG_BORDER) continue;
      for (int i = 1; i <= L; i++) {
        DetectArgs da{s.pyr, ps, oc.off, oc.h, oc.w, o, i, L, conf->contrast_threshold, conf->edge_threshold, (float)conf->sigma,
                      threshold, ccap, s.cands, s.keys, s.n_cands};
        dim3 grd(ceil_div(oc.w - 2 * IMG_BORDER, 128), oc.h - 2 * IMG_BORDER, nb);
        sift_detect<<<grd, 128, 0, st>>>(da);
        IMW_CHECK_LAUNCH_T("sift_detect");
      }
    }
    sift_sort<<<nb, 1024, 0, st>>>(s.keys, s.order, s.n_cands, ccap);
    IMW_CHECK_LAUNCH_T("sift_sort");
    // --- orientations (one warp per record; the grid covers the capacity, warps past the count return at once)
    OrientArgs oa{s.pyr, ps, p, s.cands, s.keys, s.order, s.n_cands, ccap, s.angles, s.n_peaks};
    sift_orient<<<dim3(ceil_div(ccap, ORIENT_WARPS), nb), ORIENT_WARPS * 32, 0, st>>>(oa);
    IMW_CHECK_LAUNCH_T("sift_orient");
    // --- selection
    if (conf->nms_radius == 0) IMW_CHECK_CUDA(cudaMemsetAsync(s.pix, 0, sizeof(unsigned long long) * nb * H * W, st));
    SelectArgs sa{s.cands, s.keys, s.order, s.n_cands, ccap, s.angles, s.n_peaks, s.kp_slot, s.sel, s.pix, H, W,
                  nf, nf, conf->nms_radius == 0, cap, counts + b0, batch, s.n_sel};
    sift_select<<<nb, SEL_THREADS, 0, st>>>(sa);
    IMW_CHECK_LAUNCH_T("sift_select");
    // --- descriptors of the kept keypoints
    if (cap > 0) {
      DescArgs dsa{s.pyr, ps, p, s.cands, s.order, s.angles, s.sel, s.n_sel, ccap, cap, conf->rootsift,
                   keypoints + (size_t)b0 * cap * 2, scores + (size_t)b0 * cap, scales + (size_t)b0 * cap,
                   oris + (size_t)b0 * cap, descriptors + (size_t)b0 * cap * 128};
      sift_describe<<<dim3(ceil_div(cap, DESC_WARPS), nb), DESC_WARPS * 32, 0, st>>>(dsa);
      IMW_CHECK_LAUNCH_T("sift_describe");
    }
  }
  return 0;
}
