// dali_b200/csrc/sepconv.cu -- separable convolution with reflect-101 borders: fn.gaussian_blur on images, sequences and volumes.
//
// Replaces kernels::SeparableConvolutionGpu (dali/kernels/imgproc/convolution/separable_convolution_gpu.h) behind GaussianBlurOpGpu
// (dali/operators/image/convolution/gaussian_blur_gpu.cu); numerics follow SeparableConvolutionCpu (separable_convolution_cpu.h,
// convolution_cpu.h): passes innermost spatial axis first (W, H, D), fp32 intermediates holding every channel, each output element
// acc = 0; acc = acc + w[k] * v[reflect101(i - r + k)] for ascending k, product and sum rounded separately (DESIGN §2).
// The kernels know nothing about Gaussians: they take per-sample, per-axis windows from one coefficient table.
//
//   sepconv_stream_kernel   2-D frames (HW / HWC), u8 or f32, rows 16-byte aligned, vertical diameter <= kScMaxDiam.  Work item =
//                           a column strip of a frame.  A producer lane streams the strip's source rows ONCE, in order, into a
//                           shared-memory ring with TMA bulk copies (cp.async.bulk, as resample_stream_kernel); every row is filtered
//                           horizontally once into a ring of 2 r_y + 1 float rows; each output row is the vertical sum over that ring
//                           in ascending tap order.  A consumer thread owns the same two strip elements in every row, so the float
//                           ring is thread-private: no barrier between the passes.
//   sepconv_pass_kernel     everything else (volumes, larger windows, unaligned rows): one launch per axis over the whole batch, an
//                           output element per thread, float temporaries back to back in one grow-only device buffer of the plan.
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <map>

namespace dalib200 {

constexpr int kScMaxDiameter = 8191;      // per axis: a window of 8191 taps is sigma ~ 1365; beyond that Setup refuses
constexpr int kScConsumers = 256;
constexpr int kScThreads = kScConsumers + 32;
constexpr int kScStrip = 2 * kScConsumers; // strip elements (pixels x channels) per row: two per consumer thread
constexpr int kScStages = 8;               // raw source rows in flight
constexpr int kScSlotMax = 4096;           // bytes of one raw row slot: the strip plus its horizontal halo must fit
constexpr int kScMaxDiam = 63;             // vertical diameter of the streaming kernel: 63 float rows x 2 KB = 126 KB of the ring
constexpr int kScMaxChannels = 64;
constexpr int kPassThreads = 256;

// One streaming frame.  item0 = index of its first strip in the launch (prefix over the frames).
struct ScFrame {
  const void *in;
  void *out;
  int32_t H, W, C;
  int32_t ry, rx, wy, wx;                  // radii and offsets of the windows in the coefficient table
  int32_t tw;                              // strip width in pixels
  int32_t item0;
};
// One (sample, axis) pass of the generic kernel.  chunk0 = its first chunk of kPassThreads elements in the launch.
struct ScPass {
  const void *in;
  void *out;
  int32_t total, n, inner, r, woff, out_u8;
  int32_t chunk0;
};

// reflect-101 (include/dali/core/boundary.h idx_reflect_101), repeated for windows longer than the axis; an axis of 1 reads index 0
__host__ __device__ __forceinline__ int reflect101(int i, int n) {
  if (n < 2) return 0;
  const int p = 2 * n - 2;
  i %= p;
  if (i < 0) i += p;
  return i < n ? i : p - i;
}

// strip source span: columns [s0, s1) and the bytes of a row the ring slot holds (16-byte aligned start and size)
struct ScSpan { int s0, b0, bytes; };
template <typename In>
__host__ __device__ __forceinline__ ScSpan sc_span(int W, int C, int rx, int x0, int tw) {
  ScSpan s;
  s.s0 = std::max(0, x0 - rx);
  const int s1 = std::min(W, x0 + tw + rx);
  s.b0 = (int)((s.s0 * C * (int)sizeof(In)) & ~15);
  s.bytes = ((s1 * C * (int)sizeof(In) + 15) & ~15) - s.b0;
  return s;
}

#ifdef __CUDACC__
__device__ __forceinline__ float2 sc_add2(float2 a, float2 b) {
  float2 r;
  asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rc, ra, rb;\n\tmov.b64 {%0, %1}, rc;\n\t}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}
__device__ __forceinline__ float2 sc_fma2(float2 a, float2 b, float2 c) {
  float2 r;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return r;
}

template <typename Out> __device__ __forceinline__ Out sc_cvt(float v);
template <> __device__ __forceinline__ float sc_cvt<float>(float v) { return v; }
template <> __device__ __forceinline__ uint8_t sc_cvt<uint8_t>(float v) { return sat_u8_half_away(v); }

// Horizontal products of a pair of strip elements at tap k.  u8: RN(b * c) = fma(2^23 + b, c, -2^23 c) exactly, two at a time (FFMA2);
// f32: two scalar products (the packed add after them must not be fused with them).
template <typename In> struct ScTap;
template <> struct ScTap<uint8_t> {
  __device__ __forceinline__ static float2 prod(const uint8_t *row, int o0, int o1, float c) {
    const float2 m = make_float2(__uint_as_float(0x4B000000u | row[o0]), __uint_as_float(0x4B000000u | row[o1]));
    const float dd = mul_rn(c, -8388608.0f);
    return sc_fma2(m, make_float2(c, c), make_float2(dd, dd));
  }
};
template <> struct ScTap<float> {
  __device__ __forceinline__ static float2 prod(const uint8_t *row, int o0, int o1, float c) {
    return make_float2(mul_rn(c, *reinterpret_cast<const float *>(row + o0)), mul_rn(c, *reinterpret_cast<const float *>(row + o1)));
  }
};

template <typename In, typename Out>
__global__ void __launch_bounds__(kScThreads, 2) sepconv_stream_kernel(const ScFrame *__restrict__ frames, int nframes, const float *__restrict__ tab,
                                                                       int nitems, int slot_bytes, int ring_rows) {
  extern __shared__ __align__(128) uint8_t sc_smem[];
  uint8_t *raw = sc_smem;
  float *fring = reinterpret_cast<float *>(sc_smem + kScStages * slot_bytes);
  uint64_t *full = reinterpret_cast<uint64_t *>(fring + ring_rows * kScStrip);
  uint64_t *empty = full + kScStages;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int s = 0; s < kScStages; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kScConsumers / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int it0 = (int)((int64_t)nitems * blockIdx.x / gridDim.x), it1 = (int)((int64_t)nitems * (blockIdx.x + 1) / gridDim.x);
  int f = 0;
  {
    int hi = nframes - 1;
    while (f < hi) { const int mid = (f + hi + 1) >> 1; if (frames[mid].item0 <= it0) f = mid; else hi = mid - 1; }
  }
  constexpr int ES = (int)sizeof(In);
  if (tid >= kScConsumers) {
    // ------------------------------------------------------------------ producer: one lane issues the bulk copies, rows in order
    if (tid == kScConsumers) {
      uint32_t stage = 0, par = 1;
      for (int item = it0; item < it1; item++) {
        while (f + 1 < nframes && frames[f + 1].item0 <= item) f++;
        const ScFrame &d = frames[f];
        const int x0 = (item - d.item0) * d.tw;
        const ScSpan sp = sc_span<In>(d.W, d.C, d.rx, x0, d.tw);
        const uint8_t *src = static_cast<const uint8_t *>(d.in) + sp.b0;
        const int64_t pitch = (int64_t)d.W * d.C * ES;
        for (int y = 0; y < d.H; y++) {
          mbar_wait_backoff(&empty[stage], par);
          mbar_expect_tx(&full[stage], (uint32_t)sp.bytes);
          bulk_g2s(raw + stage * slot_bytes, src + y * pitch, (uint32_t)sp.bytes, &full[stage]);
          if (++stage == kScStages) { stage = 0; par ^= 1u; }
        }
      }
    }
    return;
  }
  // -------------------------------------------------------------------- consumers
  const int lane = tid & 31;
  uint32_t stage = 0, par = 0;
  for (int item = it0; item < it1; item++) {
    while (f + 1 < nframes && frames[f + 1].item0 <= item) f++;
    const ScFrame d = frames[f];
    const int C = d.C, H = d.H, W = d.W, rx = d.rx, ry = d.ry, D = 2 * ry + 1;
    const int x0 = (item - d.item0) * d.tw;
    const int tw = min(d.tw, W - x0), ne = tw * C;
    const ScSpan sp = sc_span<In>(W, C, rx, x0, d.tw);
    const float *wx = tab + d.wx, *wy = tab + d.wy;
    // the two elements of this thread (an idle one mirrors element 0: its loads stay inside the slot, its result is dropped)
    const int e0 = tid < ne ? tid : 0, e1 = tid + kScConsumers < ne ? tid + kScConsumers : e0;
    const int p0 = e0 / C, p1 = e1 / C;
    const int xa = x0 + p0, xb = x0 + p1, ca = e0 - p0 * C, cb = e1 - p1 * C;
    const bool interior = xa - rx >= 0 && xb - rx >= 0 && xa + rx < W && xb + rx < W;
    const int oa = ((xa - rx) * C + ca) * ES - sp.b0, ob = ((xb - rx) * C + cb) * ES - sp.b0;
    Out *out = static_cast<Out *>(d.out) + (int64_t)x0 * C;
    const int64_t opitch = (int64_t)W * C;
    float *ring0 = fring + tid, *ring1 = fring + tid + kScConsumers;

    auto emit = [&](int t) {
      float2 v = make_float2(0.f, 0.f);
      if (t - ry >= 0 && t + ry < H) {
        int s = (t - ry) % D;
        for (int k = 0; k < D; k++) {
          const float c = __ldg(wy + k);
          v = sc_add2(v, make_float2(mul_rn(c, ring0[s * kScStrip]), mul_rn(c, ring1[s * kScStrip])));
          if (++s == D) s = 0;
        }
      } else {
        for (int k = 0; k < D; k++) {
          const int s = reflect101(t - ry + k, H) % D;
          const float c = __ldg(wy + k);
          v = sc_add2(v, make_float2(mul_rn(c, ring0[s * kScStrip]), mul_rn(c, ring1[s * kScStrip])));
        }
      }
      Out *o = out + (int64_t)t * opitch;
      if (tid < ne) o[tid] = sc_cvt<Out>(v.x);
      if (tid + kScConsumers < ne) o[tid + kScConsumers] = sc_cvt<Out>(v.y);
    };

    for (int y = 0; y < H; y++) {
      mbar_wait(&full[stage], par);
      const uint8_t *row = raw + stage * slot_bytes;
      float2 acc = make_float2(0.f, 0.f);
      const int dx = 2 * rx + 1;
      if (interior) {
        for (int k = 0; k < dx; k++) acc = sc_add2(acc, ScTap<In>::prod(row, oa + k * C * ES, ob + k * C * ES, __ldg(wx + k)));
      } else {
        for (int k = 0; k < dx; k++) {
          const int ia = (reflect101(xa - rx + k, W) * C + ca) * ES - sp.b0, ib = (reflect101(xb - rx + k, W) * C + cb) * ES - sp.b0;
          acc = sc_add2(acc, ScTap<In>::prod(row, ia, ib, __ldg(wx + k)));
        }
      }
      // the slot goes back to the async proxy only once its values have been consumed (acc depends on every load)
      asm volatile("fence.proxy.async.shared::cta;" :: "f"(acc.x), "f"(acc.y) : "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
      if (++stage == kScStages) { stage = 0; par ^= 1u; }
      const int s = y % D;
      ring0[s * kScStrip] = acc.x;
      ring1[s * kScStrip] = acc.y;
      if (y >= ry) emit(y - ry);
    }
    for (int t = max(0, H - ry); t < H; t++) emit(t);
  }
}

// Generic pass along one axis: element e of a sample sits at i = (e / inner) % n on the axis; its taps are inner elements apart.
template <typename In>
__device__ __forceinline__ float sc_taps(const In *src, int e, int i, int n, int inner, int r, const float *w) {
  float acc = 0.f;
  const In *base = src + (e - i * inner);
  if (i - r >= 0 && i + r < n) {
    const In *p = base + (int64_t)(i - r) * inner;
    for (int k = 0; k <= 2 * r; k++, p += inner) acc = add_rn(acc, mul_rn(__ldg(w + k), (float)*p));
  } else {
    for (int k = 0; k <= 2 * r; k++) acc = add_rn(acc, mul_rn(__ldg(w + k), (float)base[(int64_t)reflect101(i - r + k, n) * inner]));
  }
  return acc;
}

template <typename In>
__global__ void __launch_bounds__(kPassThreads) sepconv_pass_kernel(const ScPass *__restrict__ passes, int npass, const float *__restrict__ tab,
                                                                    int nchunks) {
  const int c0 = (int)((int64_t)nchunks * blockIdx.x / gridDim.x), c1 = (int)((int64_t)nchunks * (blockIdx.x + 1) / gridDim.x);
  int s = 0;
  {
    int hi = npass - 1;
    while (s < hi) { const int mid = (s + hi + 1) >> 1; if (passes[mid].chunk0 <= c0) s = mid; else hi = mid - 1; }
  }
  for (int c = c0; c < c1; c++) {
    while (s + 1 < npass && passes[s + 1].chunk0 <= c) s++;
    const ScPass &p = passes[s];
    const int e = (c - p.chunk0) * kPassThreads + threadIdx.x;
    if (e >= p.total) continue;
    const int i = (e / p.inner) % p.n;
    const float v = sc_taps(static_cast<const In *>(p.in), e, i, p.n, p.inner, p.r, tab + p.woff);
    if (p.out_u8) static_cast<uint8_t *>(p.out)[e] = sat_u8_half_away(v);
    else static_cast<float *>(p.out)[e] = v;
  }
}
#endif  // __CUDACC__

}  // namespace dalib200

using namespace dalib200;

struct dalib200SepConvPlan {
  int max_batch = 0, n = 0;
  int in_dtype = DALIB200_UINT8, out_dtype = DALIB200_UINT8;
  std::vector<dalib200SepConvSample> samples;
  std::vector<int32_t> woff;       // per sample and axis (outermost first): offset of its window in `table`
  std::vector<float> table;        // the batch's distinct windows
  std::vector<int8_t> stream_ok;   // setup: the sample's shape and windows fit the streaming kernel
  std::vector<int8_t> path;        // 1 = streaming kernel, 0 = per-axis passes (last launch; the setup's choice before it)
  DescArena arena;                 // [table | ScFrame[] | ScPass[] stage 0 | stage 1 | stage 2]
  float *tmp = nullptr;
  size_t tmp_cap = 0;              // floats
  cudaEvent_t uploaded = nullptr;
  bool pending = false;
};

namespace {
int64_t SampleElems(const dalib200SepConvSample &s) {
  int64_t v = s.channels;
  for (int a = 0; a < s.ndim; a++) v *= s.shape[a];
  return v;
}
template <typename In> bool StreamFits(const dalib200SepConvSample &s) {
  const int H = s.shape[0], W = s.shape[1], C = s.channels;
  if (C > kScMaxChannels || s.diameter[0] > kScMaxDiam || ((int64_t)W * C * sizeof(In)) % 16 != 0) return false;
  const int tw = std::max(1, kScStrip / C), rx = (s.diameter[1] - 1) / 2;
  const int64_t span = ((int64_t)std::min(W, tw) + 2 * (int64_t)rx) * C * sizeof(In) + 32;
  return H > 0 && span <= kScSlotMax;
}
size_t AlignUp(size_t v, size_t a) { return (v + a - 1) / a * a; }
}  // namespace

extern "C" {

// Host helper: FillGaussian (dali/operators/image/convolution/gaussian_blur_params.h), in double, every tap rounded to float.
void dalib200GaussianWindow(float sigma, int diameter, float *out) {
  if (!out || diameter < 1) return;
  const int r = (diameter - 1) / 2;
  const double s = 0.5 / ((double)sigma * (double)sigma);
  double sum = 0.0;
  for (int x = -r; x < 0; x++) {
    out[x + r] = (float)std::exp(-(double)(x * x) * s);
    sum += out[x + r];
  }
  sum = 2 * sum + 1;
  const double scale = 1 / sum;
  out[r] = (float)scale;
  for (int x = 0; x < r; x++) {
    out[x] = (float)(out[x] * scale);
    out[2 * r - x] = out[x];
  }
}

int dalib200SepConvPlanCreate(dalib200SepConvPlan **plan, int max_batch) try {
  DB_CHECK_ARG(plan && max_batch > 0 && max_batch <= (1 << 24), "SepConvPlanCreate: bad arguments (1..2^24 samples)");
  auto *p = new dalib200SepConvPlan();
  p->max_batch = max_batch;
  if (cudaEventCreateWithFlags(&p->uploaded, cudaEventDisableTiming) != cudaSuccess) {
    SetLastError("SepConvPlanCreate: cudaEventCreate failed"); delete p; return DALIB200_ERROR_CUDA;
  }
  *plan = p;
  return DALIB200_SUCCESS;
} DB_API_CATCH

int dalib200SepConvPlanDestroy(dalib200SepConvPlan *p) try {
  if (!p) return DALIB200_SUCCESS;
  if (p->uploaded) { cudaEventSynchronize(p->uploaded); cudaEventDestroy(p->uploaded); }
  p->arena.Free();
  if (p->tmp) cudaFree(p->tmp);
  delete p;
  return DALIB200_SUCCESS;
} DB_API_CATCH

int dalib200SepConvPlanGetPath(const dalib200SepConvPlan *p, int sample) try {
  if (!p || sample < 0 || sample >= p->n) return -1;
  return p->path[sample];
} DB_API_CATCH

int dalib200SepConvPlanSetup(dalib200SepConvPlan *p, int n, const dalib200SepConvSample *samples, const float *windows,
                             int64_t num_window_floats, int in_dtype, int out_dtype) try {
  DB_CHECK_ARG(p && n >= 0 && (n == 0 || (samples && windows)), "SepConvPlanSetup: null argument");
  DB_CHECK_ARG(n <= p->max_batch, "SepConvPlanSetup: batch %d exceeds plan capacity %d", n, p->max_batch);
  DB_CHECK_ARG(num_window_floats >= 0, "SepConvPlanSetup: negative window array size");
  if (!((in_dtype == DALIB200_UINT8 && (out_dtype == DALIB200_UINT8 || out_dtype == DALIB200_FLOAT)) ||
        (in_dtype == DALIB200_FLOAT && out_dtype == DALIB200_FLOAT))) {
    SetLastError("SepConv: unsupported type combination in=%d out=%d (u8->u8, u8->f32, f32->f32)", in_dtype, out_dtype);
    return DALIB200_ERROR_UNSUPPORTED;
  }
  p->n = 0;
  p->samples.assign(samples, samples + n);
  p->woff.assign((size_t)n * 3, 0);
  p->stream_ok.assign(n, 0);
  std::vector<float> table;
  std::map<std::pair<int64_t, int>, int32_t> seen;     // (caller offset, diameter) -> offset in the table
  for (int i = 0; i < n; i++) {
    const dalib200SepConvSample &s = samples[i];
    DB_CHECK_ARG(s.ndim == 2 || s.ndim == 3, "SepConv: sample %d: spatial rank %d (2 or 3)", i, s.ndim);
    for (int a = 0; a < s.ndim; a++) DB_CHECK_ARG(s.shape[a] >= 0, "SepConv: sample %d: negative extent", i);
    DB_CHECK_ARG(s.channels >= 0, "SepConv: sample %d: negative channel count", i);
    const bool fits = s.ndim == 2 ? ElementsFit31(s.shape[0], s.shape[1], s.channels)
                                  : ElementsFit31(s.shape[0], s.shape[1], (int64_t)s.shape[2] * s.channels);
    DB_CHECK_ARG(fits, "SepConv: sample %d has 2^31 elements or more", i);
    for (int a = 0; a < s.ndim; a++) {
      const int d = s.diameter[a];
      DB_CHECK_ARG(d >= 1 && d % 2 == 1, "SepConv: sample %d axis %d: window diameter %d must be odd and positive", i, a, d);
      DB_CHECK_ARG(d <= kScMaxDiameter, "SepConv: sample %d axis %d: window diameter %d exceeds the limit of %d taps", i, a, d, kScMaxDiameter);
      const int64_t o = s.window_offset[a];
      DB_CHECK_ARG(o >= 0 && o + d <= num_window_floats, "SepConv: sample %d axis %d: window [%lld, %lld) outside the %lld window floats", i, a,
                   (long long)o, (long long)(o + d), (long long)num_window_floats);
      auto it = seen.find({o, d});
      if (it == seen.end()) {
        for (int k = 0; k < d; k++) DB_CHECK_ARG(std::isfinite(windows[o + k]), "SepConv: sample %d axis %d: window tap %d is not finite", i, a, k);
        it = seen.emplace(std::make_pair(o, d), (int32_t)table.size()).first;
        table.insert(table.end(), windows + o, windows + o + d);
      }
      p->woff[(size_t)i * 3 + a] = it->second;
    }
    if (s.ndim == 2 && SampleElems(s) > 0) p->stream_ok[i] = in_dtype == DALIB200_UINT8 ? StreamFits<uint8_t>(s) : StreamFits<float>(s);
  }
  p->path = p->stream_ok;
  p->table.swap(table);
  p->in_dtype = in_dtype; p->out_dtype = out_dtype;
  p->n = n;
  return DALIB200_SUCCESS;
} DB_API_CATCH

int dalib200SepConvLaunch(dalib200SepConvPlan *p, const void *const *in_ptrs, void *const *out_ptrs, dalib200Stream_t stream) try {
  DB_CHECK_ARG(p && (p->n == 0 || (in_ptrs && out_ptrs)), "SepConvLaunch: null argument");
  const int n = p->n;
  if (n == 0) return DALIB200_SUCCESS;
  if (p->pending) { DB_CUDA(cudaEventSynchronize(p->uploaded)); p->pending = false; }
  const bool u8in = p->in_dtype == DALIB200_UINT8, u8out = p->out_dtype == DALIB200_UINT8;
  const size_t es = u8in ? 1 : 4;
  std::vector<ScFrame> frames;
  std::vector<ScPass> passes[3];
  int64_t nitems = 0, nchunks[3] = { 0, 0, 0 };
  int max_d = 1;
  int64_t slot = 16;
  size_t need = 0;
  for (int i = 0; i < n; i++) {
    const dalib200SepConvSample &s = p->samples[i];
    const int64_t vol = SampleElems(s);
    if (vol == 0) continue;
    DB_CHECK_ARG(in_ptrs[i] && out_ptrs[i], "SepConvLaunch: sample %d: null pointer", i);
    p->path[i] = p->stream_ok[i] && (reinterpret_cast<uintptr_t>(in_ptrs[i]) & 15) == 0;      // bulk copies need 16-byte aligned rows
    if (p->path[i]) {
      ScFrame f;
      f.in = in_ptrs[i]; f.out = out_ptrs[i];
      f.H = s.shape[0]; f.W = s.shape[1]; f.C = s.channels;
      f.ry = (s.diameter[0] - 1) / 2; f.rx = (s.diameter[1] - 1) / 2;
      f.wy = p->woff[(size_t)i * 3]; f.wx = p->woff[(size_t)i * 3 + 1];
      f.tw = std::max(1, kScStrip / f.C);
      f.item0 = (int32_t)nitems;
      nitems += (f.W + f.tw - 1) / f.tw;
      max_d = std::max(max_d, s.diameter[0]);
      slot = std::max<int64_t>(slot, std::min<int64_t>(f.W, (int64_t)f.tw + 2 * f.rx) * f.C * es + 32);   // any strip's span
      frames.push_back(f);
      continue;
    }
    // per-axis passes, innermost first: W -> t0 -> H -> (t1 -> D ->) out
    const int nd = s.ndim;
    need += (size_t)vol * (nd - 1);
    int64_t inner = s.channels;
    for (int k = 0; k < nd; k++) {
      const int a = nd - 1 - k;
      ScPass q;
      q.total = (int32_t)vol; q.n = s.shape[a]; q.inner = (int32_t)inner; q.r = (s.diameter[a] - 1) / 2;
      q.woff = p->woff[(size_t)i * 3 + a];
      q.out_u8 = k == nd - 1 && u8out;
      q.in = nullptr; q.out = nullptr;                                  // temporaries are placed below, once the buffer is sized
      q.chunk0 = (int32_t)nchunks[k];
      nchunks[k] += (vol + kPassThreads - 1) / kPassThreads;
      passes[k].push_back(q);
      inner *= s.shape[a];
    }
  }
  DB_CHECK_ARG(nitems < (int64_t{1} << 31) && nchunks[0] < (int64_t{1} << 31), "SepConvLaunch: batch too large");
  if (need > p->tmp_cap) {
    if (p->tmp) { DB_CUDA(cudaFree(p->tmp)); p->tmp = nullptr; p->tmp_cap = 0; }     // cudaFree waits for the launches that still use it
    DB_CUDA(cudaMalloc(reinterpret_cast<void **>(&p->tmp), need * sizeof(float)));
    p->tmp_cap = need;
  }
  {
    // temporaries of sample j back to back: [t0 | t1]; pass k of a sample reads the input or t(k-1) and writes t(k) or the output
    size_t off = 0;
    std::vector<size_t> ks(3, 0);
    for (int i = 0; i < n; i++) {
      const dalib200SepConvSample &s = p->samples[i];
      const int64_t vol = SampleElems(s);
      if (vol == 0 || p->path[i]) continue;
      const int nd = s.ndim;
      float *t0 = p->tmp + off, *t1 = t0 + vol;
      off += (size_t)vol * (nd - 1);
      for (int k = 0; k < nd; k++) {
        ScPass &q = passes[k][ks[k]++];
        q.in = k == 0 ? in_ptrs[i] : static_cast<const void *>(k == 1 ? t0 : t1);
        q.out = k == nd - 1 ? out_ptrs[i] : static_cast<void *>(k == 0 ? t0 : t1);
      }
    }
  }
  const size_t tab_bytes = AlignUp(p->table.size() * sizeof(float), 64);
  const size_t fr_off = tab_bytes, ps_off = AlignUp(fr_off + frames.size() * sizeof(ScFrame), 64);
  size_t stage_off[3], total = ps_off;
  for (int k = 0; k < 3; k++) { stage_off[k] = total; total = AlignUp(total + passes[k].size() * sizeof(ScPass), 64); }
  int rc = p->arena.Reserve(std::max<size_t>(total, 64));
  if (rc) return rc;
  memcpy(p->arena.host, p->table.data(), p->table.size() * sizeof(float));
  if (!frames.empty()) memcpy(p->arena.host + fr_off, frames.data(), frames.size() * sizeof(ScFrame));
  for (int k = 0; k < 3; k++)
    if (!passes[k].empty()) memcpy(p->arena.host + stage_off[k], passes[k].data(), passes[k].size() * sizeof(ScPass));
  if (nitems == 0 && nchunks[0] == 0) return DALIB200_SUCCESS;          // nothing to do: no launch (an empty grid is a sticky error)
  if ((rc = p->arena.Upload(total, stream))) return rc;
  DB_CUDA(cudaEventRecord(p->uploaded, stream));
  p->pending = true;
  const float *dtab = reinterpret_cast<const float *>(p->arena.dev);
  if (nitems > 0) {
    slot = (int64_t)AlignUp((size_t)slot, 128);
    const int ring_rows = max_d;
    const size_t smem = (size_t)kScStages * slot + (size_t)ring_rows * kScStrip * sizeof(float) + 2 * kScStages * 8;
    const ScFrame *df = reinterpret_cast<const ScFrame *>(p->arena.dev + fr_off);
    const int nf = (int)frames.size();
    auto go = [&](auto kern) -> int {
      DB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int per_sm = 0;
      DB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kScThreads, smem));
      const int grid = (int)std::min<int64_t>(nitems, (int64_t)NumSMs() * std::max(per_sm, 1));
      ProfScope ps_("sepconv_stream", stream);
      kern<<<grid, kScThreads, smem, stream>>>(df, nf, dtab, (int)nitems, (int)slot, ring_rows);
      CountLaunch();
      DB_CUDA(cudaGetLastError());
      return DALIB200_SUCCESS;
    };
    rc = !u8in ? go(sepconv_stream_kernel<float, float>) : u8out ? go(sepconv_stream_kernel<uint8_t, uint8_t>) : go(sepconv_stream_kernel<uint8_t, float>);
    if (rc) return rc;
  }
  for (int k = 0; k < 3; k++) {
    if (nchunks[k] == 0) continue;
    const ScPass *dp = reinterpret_cast<const ScPass *>(p->arena.dev + stage_off[k]);
    const int grid = (int)std::min<int64_t>(nchunks[k], (int64_t)NumSMs() * 8);
    ProfScope ps_("sepconv_pass", stream);
    if (k == 0 && u8in) sepconv_pass_kernel<uint8_t><<<grid, kPassThreads, 0, stream>>>(dp, (int)passes[k].size(), dtab, (int)nchunks[k]);
    else sepconv_pass_kernel<float><<<grid, kPassThreads, 0, stream>>>(dp, (int)passes[k].size(), dtab, (int)nchunks[k]);
    CountLaunch();
    DB_CUDA(cudaGetLastError());
  }
  return DALIB200_SUCCESS;
} DB_API_CATCH

}  // extern "C"
