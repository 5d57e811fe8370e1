/*
 * oracle/gaussian_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-C restatement of the reference's CPU Gaussian blur (GaussianBlur over SeparableConvolutionCpu) that the GPU tests of
 * fn.gaussian_blur compare with bit for bit.  Compiled on demand by oracle/pygaussian.py into a temporary directory with the flags
 * of oracle/Makefile (-O2, -ffp-contract=off: the reference binary is built for baseline x86-64, so every a*b+c is two roundings).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* include/dali/core/convert.h:306-324 -- host ConvertSat<uint8_t>(float) = clamp(std::round(x)) */
static inline uint8_t sat_u8_half_away(float x) {
  float r = roundf(x);
  return (uint8_t)(r <= 0.0f ? 0 : r >= 255.0f ? 255 : (int)r);
}


/* ------------------------------------------------------------------ Gaussian blur (separable convolution, reflect-101) */
/* FillGaussian (dali/operators/image/convolution/gaussian_blur_params.h), restated in double: the left half is exp(-x^2 s) rounded to
 * float, summed in double (the float widened back), sum = 2 sum + 1, the centre tap is the scale, every other tap is rounded again
 * after the scaling and mirrored.  Restatement-pinned (DESIGN §2): not yet compared with the compiled reference. */
void oracle_gaussian_window(float sigma, int diameter, float *out) {
  int r = (diameter - 1) / 2;
  double s = 0.5 / ((double)sigma * (double)sigma);
  double sum = 0.0;
  for (int x = -r; x < 0; x++) {
    out[x + r] = (float)exp(-(double)(x * x) * s);
    sum += out[x + r];
  }
  sum = 2 * sum + 1;
  double scale = 1 / sum;
  out[r] = (float)scale;
  for (int x = 0; x < r; x++) {
    out[x] = (float)(out[x] * scale);
    out[2 * r - x] = out[x];
  }
}

/* include/dali/core/boundary.h idx_reflect_101, repeated while the index is outside (windows longer than the axis) */
static int64_t gb_reflect101(int64_t idx, int64_t size) {
  if (size < 2) return 0;
  for (;;) {
    if (idx < 0) idx = -idx;
    else if (idx >= size) idx = 2 * size - 2 - idx;
    else break;
  }
  return idx;
}

/* SeparableConvolutionCpu (dali/kernels/imgproc/convolution/separable_convolution_cpu.h, convolution_cpu.h): ndim = 2 (HWC) or
 * 3 (DHWC) spatial axes, shape[] outermost first; windows[] holds the per-axis windows back to back in the same order.  Passes run
 * innermost axis first (W, H, D) over fp32 intermediates; every element is acc = 0; acc = acc + w[k] * v[reflect101(i - r + k)],
 * k ascending, product and sum rounded to float separately (built with -ffp-contract=off).  u8 output: ConvertSat (half away). */
int oracle_sepconv(const void *in, int in_dtype, int ndim, const int *shape, int C, const int *diam, const float *windows,
                   void *out, int out_dtype) {
  if (ndim < 2 || ndim > 3 || C < 0) return -1;
  int64_t vol = C;
  for (int a = 0; a < ndim; a++) vol *= shape[a];
  if (vol == 0) return 0;
  const float *win[3];
  {
    size_t o = 0;
    for (int a = 0; a < ndim; a++) { win[a] = windows + o; o += (size_t)diam[a]; }
  }
  float *cur = (float *)malloc((size_t)vol * sizeof(float)), *nxt = (float *)malloc((size_t)vol * sizeof(float));
  for (int64_t e = 0; e < vol; e++) cur[e] = in_dtype == 0 ? (float)((const uint8_t *)in)[e] : ((const float *)in)[e];
  int64_t inner = C;
  for (int k = 0; k < ndim; k++) {
    int a = ndim - 1 - k;
    int64_t n = shape[a];
    int r = (diam[a] - 1) / 2;
    const float *w = win[a];
    for (int64_t e = 0; e < vol; e++) {
      int64_t i = (e / inner) % n;
      const float *base = cur + (e - i * inner);
      float acc = 0.0f;
      for (int t = 0; t < diam[a]; t++) {
        float p = w[t] * base[gb_reflect101(i - r + t, n) * inner];
        acc = acc + p;
      }
      nxt[e] = acc;
    }
    float *sw = cur; cur = nxt; nxt = sw;
    inner *= n;
  }
  for (int64_t e = 0; e < vol; e++) {
    if (out_dtype == 0) ((uint8_t *)out)[e] = sat_u8_half_away(cur[e]);
    else ((float *)out)[e] = cur[e];
  }
  free(cur); free(nxt);
  return 0;
}
