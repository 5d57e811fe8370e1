// dali_b200/host/operators.cc -- the hot-path operators behind the reference's operator boundary
// (Operator<GPUBackend>::SetupImpl / RunImpl + DALI_SCHEMA + DALI_REGISTER_OPERATOR), each a thin argument layer
// over the C-ABI of include/dali_b200.h:  SetupImpl -> ...PlanSetup (host, shapes + per-sample args),
// RunImpl -> ...Launch (enqueue on ws.stream(), no host sync).
//
// Argument handling restates the reference operators (schema names, defaults, meaning, error behaviour):
//   decoders__Image        dali/operators/imgcodec/decoder_schema.cc:21-168, mixed_decoder.cc:35-51
//   Resize                 dali/operators/image/resize/resize.cc:21-41, resize_attr.cc:23-259, resize_attr_base.{h,cc},
//                          resampling_attr.cc:22-133
//   CropMirrorNormalize    dali/operators/image/crop/crop_mirror_normalize.{h,cc}, crop_attr.cc:21-245
//   WarpAffine             dali/operators/image/remap/warp_affine.cc:19-57, warp_affine_params.h:50-83,
//                          warp_param_provider.h:234-314
//   Hsv                    dali/operators/image/color/color_twist.{h,cc}
//   ColorSpaceConversion   dali/operators/image/color/color_space_conversion.{h,cc}
//   Spectrogram            dali/operators/signal/fft/spectrogram.cc:30-311
//   MelFilterBank          dali/operators/audio/mel_scale/mel_filter_bank.cc:22-117
// There is no CPU implementation: the ops are registered for GPU / Mixed only.
#include <array>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include "dali.h"
#include "random_crop.h"
#include <ctime>
#include <cstdlib>
#include "../../include/dali_b200.h"

namespace dali {

static void CheckStatus(int rc, const char *what) {
  if (rc != DALIB200_SUCCESS) throw DALIException(make_string(what, ": ", dalib200GetLastError()));
}

// frames of a (F)HWC batch flattened into independent 2-D samples (SequenceOperator, sequence_operator.h:57-110)
struct FrameList {
  int first_spatial = 0;                       // index of H in the sample shape
  std::vector<int> sample_of_frame;            // frame -> sample
  std::vector<int64_t> frame_offset_elems;     // element offset of the frame inside its sample
  std::vector<int> h, w, c;
  int num_frames() const { return static_cast<int>(h.size()); }
};

static FrameList ExpandFrames(const TensorListShape &shape, const TensorLayout &layout, const char *op) {
  FrameList f;
  const int nd = shape.sample_dim();
  std::string l = layout.str();
  if (l.empty()) l = nd == 3 ? "HWC" : nd == 4 ? "FHWC" : "";
  DALI_ENFORCE(l == "HWC" || l == "FHWC", op, ": the GPU path supports HWC and FHWC inputs, got layout \"", l, "\" (", nd, "-D)");
  DALI_ENFORCE(static_cast<int>(l.size()) == nd, op, ": layout \"", l, "\" does not match a ", nd, "-D input");
  f.first_spatial = l == "HWC" ? 0 : 1;
  for (int i = 0; i < shape.num_samples(); i++) {
    const int64_t *s = shape.tensor_shape_span(i);
    const int64_t frames = f.first_spatial ? s[0] : 1;
    const int64_t H = s[f.first_spatial], W = s[f.first_spatial + 1], C = s[f.first_spatial + 2];
    for (int64_t k = 0; k < frames; k++) {
      f.sample_of_frame.push_back(i);
      f.frame_offset_elems.push_back(k * H * W * C);
      f.h.push_back(static_cast<int>(H)); f.w.push_back(static_cast<int>(W)); f.c.push_back(static_cast<int>(C));
    }
  }
  return f;
}

// Resize takes every layout of the reference's schema (resize.cc:28-29): the dimensions in front of the spatial ones collapse into
// frames -- which covers channel-first data: a CHW image is C one-channel frames --, those behind them into channels
// (resize_op_impl.h:56-101).  2-D layouts here; the volumetric ones go through SetupVolumes.
// ResizeAttr::ParseLayout (resize_attr.cc:102-123) over the layouts of the schema: number of spatial dimensions and index of the first
static void ParseResizeLayout(const std::string &l, int *spatial_ndim, int *first_spatial) {
  static const char *const kLayouts[] = { "HWC", "FHWC", "CHW", "FCHW", "CFHW", "DHWC", "FDHWC", "CDHW", "FCDHW", "CFDHW" };
  bool known = false;
  for (const char *k : kLayouts) known |= l == k;
  DALI_ENFORCE(known, "Resize: unsupported layout \"", l, "\"; expected one of HWC, FHWC, CHW, FCHW, CFHW, DHWC, FDHWC, CDHW, FCDHW, CFDHW");
  const size_t d = l.find('D');
  *spatial_ndim = d == std::string::npos ? 2 : 3;
  *first_spatial = static_cast<int>(d == std::string::npos ? l.find('H') : d);
}

static FrameList ExpandFramesAnyLayout(const TensorListShape &shape, const TensorLayout &layout, const char *op) {
  FrameList f;
  const int nd = shape.sample_dim();
  std::string l = layout.str();
  if (l.empty()) l = nd == 3 ? "HWC" : nd == 4 ? "FHWC" : "";
  int sd = 2, fs = 0;
  ParseResizeLayout(l, &sd, &fs);
  DALI_ENFORCE(sd == 2, op, ": a 2-D layout is expected here, got \"", l, "\"");
  DALI_ENFORCE(static_cast<int>(l.size()) == nd, op, ": layout \"", l, "\" does not match a ", nd, "-D input");
  f.first_spatial = fs;
  for (int i = 0; i < shape.num_samples(); i++) {
    const int64_t *s = shape.tensor_shape_span(i);
    int64_t frames = 1, C = 1;
    for (int d = 0; d < fs; d++) frames *= s[d];
    for (int d = fs + 2; d < nd; d++) C *= s[d];
    const int64_t H = s[fs], W = s[fs + 1];
    for (int64_t k = 0; k < frames; k++) {
      f.sample_of_frame.push_back(i);
      f.frame_offset_elems.push_back(k * H * W * C);
      f.h.push_back(static_cast<int>(H)); f.w.push_back(static_cast<int>(W)); f.c.push_back(static_cast<int>(C));
    }
  }
  return f;
}

template <typename TL>
static std::vector<const void *> FramePtrs(const TL &tl, const FrameList &f, size_t elem_size) {
  std::vector<const void *> p(f.num_frames());
  for (int k = 0; k < f.num_frames(); k++)
    p[k] = static_cast<const uint8_t *>(tl.raw_tensor(f.sample_of_frame[k])) + f.frame_offset_elems[k] * elem_size;
  return p;
}

// =============================================================================================== decoders.image
DALI_SCHEMA(decoders__Image)
    .DocStr("Decodes JPEG images on the GPU (Huffman + IDCT + upsampling + colour conversion in CUDA).")
    .NumInput(1).NumOutput(1)
    .AddOptionalArg("output_type", "Colour space of the output image.", DALI_RGB)
    .AddOptionalArg("dtype", "Output data type.", DALI_UINT8)
    .AddOptionalArg("adjust_orientation", "Use EXIF orientation metadata to rectify the images.", true)
    .AddOptionalArg("use_fast_idct", "ignored (the islow integer IDCT is always used)", false)
    // NOTE: the reference's mixed default is False (nvJPEG box upsampling); this build defaults to the CPU
    // backend's libjpeg-turbo "fancy" upsampling so that mixed == cpu bit-exactly (DESIGN.md, deviations).
    .AddOptionalArg("jpeg_fancy_upsampling", "Use libjpeg-turbo fancy (triangle) chroma upsampling.", true)
    .AddOptionalArg("hybrid_huffman_threshold", "ignored", 1000000)
    .AddOptionalArg("hw_decoder_load", "ignored (no hardware engine is used)", 0.9f)
    .AddOptionalArg("device_memory_padding", "ignored", 16777216)
    .AddOptionalArg("host_memory_padding", "ignored", 8388608)
    .AddOptionalArg("device_memory_padding_jpeg2k", "ignored", 0)
    .AddOptionalArg("host_memory_padding_jpeg2k", "ignored", 0)
    .AddOptionalArg("preallocate_width_hint", "ignored", 0)
    .AddOptionalArg("preallocate_height_hint", "ignored", 0)
    .AddOptionalArg("affine", "ignored", true)
    .AddOptionalArg("split_stages", "ignored", false)
    .AddOptionalArg("use_chunk_allocator", "ignored", false)
    .AddOptionalArg("memory_stats", "ignored", false)
    .AddOptionalArg("cache_size", "ignored (no decoder cache)", 0)
    .AddOptionalArg("cache_threshold", "ignored", 0)
    .AddOptionalArg("cache_debug", "ignored", false)
    .AddOptionalArg("cache_batch_copy", "ignored", true)
    .AddOptionalArg("cache_type", "ignored", std::string(""));

// Common part of decoders.image / image_crop / image_random_crop / image_slice: header parse, region of interest from the
// derived class (in OUTPUT = oriented coordinates, imgcodec.h:26-44), plan setup, launch, asynchronous status check.
class ImageDecoderBase : public Operator<MixedBackend>, public PlanarProducer {
 public:
  // ---- PlanarProducer: decode -> resize fusion (the launch is deferred to the consuming Resize)
  void EnableDeferredRun() override { deferred_ = true; }
  void SelectPlanar(const std::vector<uint8_t> &want, std::vector<uint8_t> &granted) override {
    granted.assign(want.size(), 0);
    CheckStatus(dalib200JpegPlanSetPlanesOnly(plan_, want.data(), granted.data()), name_);
  }
  void RunDeferred(cudaStream_t stream) override {
    CheckStatus(dalib200JpegUpload(plan_, stream), name_);
    CheckStatus(dalib200JpegLaunch(plan_, optr_.data(), stream), name_);
    CheckStatus(dalib200JpegStatusAsync(plan_, stream), name_);
    launched_ = static_cast<int>(optr_.size());
  }
  void GetPlanarSource(int sample, PlanarSource *out) override {
    dalib200PlanarImage pi;
    CheckStatus(dalib200JpegPlanGetPlanes(plan_, sample, &pi), name_);
    out->y = pi.y; out->cb = pi.cb; out->cr = pi.cr; out->pitch_y = pi.pitch_y; out->pitch_c = pi.pitch_c;
    out->width = pi.width; out->height = pi.height;
    out->crop_x = rois_[sample].use_roi ? rois_[sample].x0 : 0;
    out->crop_y = rois_[sample].use_roi ? rois_[sample].y0 : 0;
  }

  explicit ImageDecoderBase(const OpSpec &spec, const char *name) : Operator<MixedBackend>(spec), name_(name) {
    prm_.output_type = spec.GetArgument<DALIImageType>("output_type");
    const DALIDataType dt = spec.GetArgument<DALIDataType>("dtype");
    DALI_ENFORCE(dt == DALI_UINT8 || dt == DALI_FLOAT, name_, ": the GPU decoder supports dtype UINT8 and FLOAT");
    out_type_ = dt;
    prm_.dtype = dt == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT;
    prm_.fancy_upsampling = spec.GetArgument<bool>("jpeg_fancy_upsampling");
    prm_.adjust_orientation = spec.GetArgument<bool>("adjust_orientation");
    CheckStatus(dalib200JpegPlanCreate(&plan_, max_batch_size_), name_);
  }
  ~ImageDecoderBase() override { dalib200JpegPlanDestroy(plan_); }

 protected:
  // fills rois_[i] (use_roi = 0: whole image) for an image whose ORIENTED size is H x W
  virtual void SampleRoi(dalib200JpegRoi &roi, const Workspace &ws, int i, int H, int W) { roi.use_roi = 0; }
  virtual bool HasRoi() const { return false; }

  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<CPUBackend>(0);
    const int n = in.num_samples();
    DALI_ENFORCE(in.type() == DALI_UINT8, name_, " expects encoded streams as 1-D uint8 tensors");
    std::vector<const uint8_t *> ptrs(n);
    std::vector<size_t> lens(n);
    for (int i = 0; i < n; i++) { ptrs[i] = in.tensor<uint8_t>(i); lens[i] = static_cast<size_t>(in.shape().tensor_size(i)); }
    rois_.assign(n, dalib200JpegRoi{0, 0, 0, 0, 0});
    if (HasRoi()) {
      for (int i = 0; i < n; i++) {
        dalib200JpegInfo info;
        if (dalib200JpegGetInfo(ptrs[i], lens[i], &info) != DALIB200_SUCCESS)
          throw DALIException(make_string(name_, ": sample ", i, ": ", dalib200GetLastError()));
        int H = info.height, W = info.width;
        if (prm_.adjust_orientation && info.orientation >= 5) std::swap(H, W);      // image_decoder.h:678-681
        SampleRoi(rois_[i], ws, i, H, W);
      }
    }
    CheckStatus(dalib200JpegPlanSetSourceStable(plan_, in.stable() ? 1 : 0), name_);
    CheckStatus(dalib200JpegPlanSetupEx(plan_, n, ptrs.data(), lens.data(), &prm_, HasRoi() ? rois_.data() : nullptr), name_);
    out.resize(1);
    out[0].type = out_type_;
    out[0].shape.resize(n, 3);
    for (int i = 0; i < n; i++) {
      int32_t hwc[3];
      CheckStatus(dalib200JpegPlanGetOutputShape(plan_, i, hwc), name_);
      out[0].shape.set_tensor_shape(i, { hwc[0], hwc[1], hwc[2] });
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout("HWC");
    optr_.resize(out.num_samples());
    for (int i = 0; i < out.num_samples(); i++) optr_[i] = out.raw_mutable_tensor(i);
    if (deferred_) return;                  // the consuming Resize launches the decode (RunDeferred) once it has chosen the planar samples
    RunDeferred(ws.stream());
  }
  void CheckCompletion() override {
    if (launched_ <= 0) return;
    std::vector<int32_t> st(launched_);
    const int n = launched_;
    launched_ = 0;
    CheckStatus(dalib200JpegStatusFetch(plan_, st.data(), n), name_);
    for (int i = 0; i < n; i++)
      if (st[i] != 0)       // image_decoder.h:826-831: "Failed to decode sample #i"
        throw DALIException(make_string("Failed to decode sample #", i, ": the entropy-coded data ends early or is corrupt"));
  }
  int launched_ = 0;
  bool deferred_ = false;
  std::vector<void *> optr_;

  dalib200JpegPlan *plan_ = nullptr;
  dalib200JpegParams prm_{};
  DALIDataType out_type_ = DALI_UINT8;
  std::vector<dalib200JpegRoi> rois_;
  const char *name_;
};

class ImageDecoderMixed : public ImageDecoderBase {
 public:
  explicit ImageDecoderMixed(const OpSpec &spec) : ImageDecoderBase(spec, "decoders.image") {}
};
DALI_REGISTER_OPERATOR(decoders__Image, ImageDecoderMixed, Mixed);

#define DALIB200_DECODER_ARGS(schema)                                                                                         \
  schema.AddOptionalArg("output_type", "Colour space of the output image.", DALI_RGB)                                          \
      .AddOptionalArg("dtype", "Output data type.", DALI_UINT8)                                                                \
      .AddOptionalArg("adjust_orientation", "Use EXIF orientation metadata to rectify the images.", true)                      \
      .AddOptionalArg("use_fast_idct", "ignored (the islow integer IDCT is always used)", false)                               \
      .AddOptionalArg("jpeg_fancy_upsampling", "Use libjpeg-turbo fancy (triangle) chroma upsampling.", true)                  \
      .AddOptionalArg("hybrid_huffman_threshold", "ignored", 1000000)                                                          \
      .AddOptionalArg("hw_decoder_load", "ignored (no hardware engine is used)", 0.9f)                                         \
      .AddOptionalArg("device_memory_padding", "ignored", 16777216)                                                            \
      .AddOptionalArg("host_memory_padding", "ignored", 8388608)                                                               \
      .AddOptionalArg("affine", "ignored", true)                                                                               \
      .AddOptionalArg("split_stages", "ignored", false)                                                                        \
      .AddOptionalArg("use_chunk_allocator", "ignored", false)                                                                 \
      .AddOptionalArg("memory_stats", "ignored", false)

// ----------------------------------------------------------------------------------------------- decoders.image_crop
// imgcodec decoder_schema.cc:170-196 + CropAttr (crop_attr.cc:21-88,100-239): the window is anchored at
// round(crop_pos * (image - crop)) -- the same arithmetic as CropMirrorNormalize -- and only its MCUs are transformed.
struct CropWindowArgs {
  bool has_crop = false, has_hw = false, truncate = false;
  void Init(const OpSpec &spec, const char *name) {
    has_crop = spec.ArgumentDefined("crop");
    has_hw = spec.ArgumentDefined("crop_h") || spec.ArgumentDefined("crop_w");
    DALI_ENFORCE(!(has_crop && has_hw), "`crop` argument is not compatible with `crop_h`, `crop_w`, `crop_d`");
    DALI_ENFORCE(spec.ArgumentDefined("crop_h") == spec.ArgumentDefined("crop_w"), "`crop_h` and `crop_w` arguments must be provided together");
    const std::string r = spec.GetArgument<std::string>("rounding");
    DALI_ENFORCE(r == "round" || r == "truncate", "``rounding`` value ", r, " is not supported. Supported values are \"round\", or \"truncate\".");
    truncate = r == "truncate";
  }
  // window [y0, y0 + h) x [x0, x0 + w) for an H x W image
  void Get(const OpSpec &spec, const Workspace &ws, int i, int64_t H, int64_t W, int64_t &y0, int64_t &x0, int64_t &h, int64_t &w) const {
    h = H; w = W;
    float px = 0.5f, py = 0.5f;
    bool hh = false, hw = false;
    if (has_crop) {
      auto c = spec.GetFloatVecArgument("crop", &ws, i);
      DALI_ENFORCE(c.size() == 2, "`crop` argument should have 2 or 3 elements depending on the input data shape");
      h = static_cast<int>(c[0]); w = static_cast<int>(c[1]); hh = hw = true;
    } else if (has_hw) {
      h = static_cast<int>(spec.GetArgument<float>("crop_h", &ws, i)); w = static_cast<int>(spec.GetArgument<float>("crop_w", &ws, i));
      hh = hw = true;
    }
    if (!(hh && h > 0)) h = H; else py = spec.GetArgument<float>("crop_pos_y", &ws, i);
    if (!(hw && w > 0)) w = W; else px = spec.GetArgument<float>("crop_pos_x", &ws, i);
    DALI_ENFORCE(px >= 0.0f && px <= 1.0f && py >= 0.0f && py <= 1.0f, "Anchor for dimension is out of range [0.0, 1.0]");
    auto rnd = [&](double v) { return truncate ? static_cast<int64_t>(v) : static_cast<int64_t>(std::round(v)); };
    y0 = rnd(static_cast<double>(py) * (H - h)); x0 = rnd(static_cast<double>(px) * (W - w));
  }
};

#define DALIB200_CROP_ARGS(schema)                                                                                             \
  schema.AddOptionalArgNoDefault("crop", "Shape of the cropped image (H, W).", true)                                           \
      .AddOptionalArgNoDefault("crop_h", "Cropping window height.", true)                                                      \
      .AddOptionalArgNoDefault("crop_w", "Cropping window width.", true)                                                       \
      .AddOptionalArgNoDefault("crop_d", "not supported (2-D images only)", true)                                              \
      .AddOptionalArg("crop_pos_x", "Normalised horizontal position of the window.", 0.5f, true)                               \
      .AddOptionalArg("crop_pos_y", "Normalised vertical position of the window.", 0.5f, true)                                 \
      .AddOptionalArg("crop_pos_z", "unused", 0.5f, true)                                                                      \
      .AddOptionalArg("rounding", "round | truncate", std::string("round"))

DALI_SCHEMA(decoders__ImageCrop)
    .DocStr("Decodes JPEG images on the GPU and extracts a fixed crop window; only the blocks under the window are transformed.")
    .NumInput(1).NumOutput(1)
    DALIB200_DECODER_ARGS() DALIB200_CROP_ARGS();

class ImageDecoderCropMixed : public ImageDecoderBase {
 public:
  explicit ImageDecoderCropMixed(const OpSpec &spec) : ImageDecoderBase(spec, "decoders.image_crop") { crop_.Init(spec, name_); }
 protected:
  bool HasRoi() const override { return true; }
  void SampleRoi(dalib200JpegRoi &roi, const Workspace &ws, int i, int H, int W) override {
    int64_t y0, x0, h, w;
    crop_.Get(spec_, ws, i, H, W, y0, x0, h, w);
    DALI_ENFORCE(y0 >= 0 && x0 >= 0 && y0 + h <= H && x0 + w <= W, "decoders.image_crop: sample ", i, ": the crop window {", y0, ", ", x0,
                 "} + {", h, ", ", w, "} does not fit the image {", H, ", ", W, "}");
    roi = { 1, static_cast<int>(x0), static_cast<int>(y0), static_cast<int>(x0 + w), static_cast<int>(y0 + h) };
  }
  CropWindowArgs crop_;
};
DALI_REGISTER_OPERATOR(decoders__ImageCrop, ImageDecoderCropMixed, Mixed);

// ----------------------------------------------------------------------------------------------- decoders.image_random_crop
#define DALIB200_RANDOM_CROP_ARGS(schema)                                                                                      \
  schema.AddOptionalArg("random_aspect_ratio", "Range from which to choose random aspect ratio (width / height).", std::vector<float>{3.f / 4, 4.f / 3}) \
      .AddOptionalArg("random_area", "Range from which to choose random area fraction A.", std::vector<float>{0.08f, 1.0f})   \
      .AddOptionalArg("num_attempts", "Maximum number of attempts used to choose random area and aspect ratio.", 10)           \
      .AddOptionalArg("seed", "Random seed.", -1)

// The prefetch slots of a pipeline instantiate every operator once per slot, but a random operator is ONE stream of numbers in the
// reference (one instance serves all iterations).  Instances created from the same graph node (same `_state_key`, set by the
// pipeline) therefore share their generators; the slots run their Setup in iteration order on the pipeline's host thread.
using CropGenerators = std::shared_ptr<std::vector<RandomCropGenerator>>;
static std::vector<RandomCropGenerator> MakeCropGeneratorsImpl(const OpSpec &spec, int max_batch);
static CropGenerators MakeCropGenerators(const OpSpec &spec, int max_batch) {
  static std::map<std::string, std::weak_ptr<std::vector<RandomCropGenerator>>> shared;
  std::string key;
  if (spec.ArgumentDefined("_state_key")) key = spec.GetArgument<std::string>("_state_key");
  if (!key.empty()) {
    auto it = shared.find(key);
    if (it != shared.end()) if (auto sp = it->second.lock()) return sp;
  }
  auto sp = std::make_shared<std::vector<RandomCropGenerator>>(MakeCropGeneratorsImpl(spec, max_batch));
  if (!key.empty()) shared[key] = sp;
  return sp;
}
static std::vector<RandomCropGenerator> MakeCropGeneratorsImpl(const OpSpec &spec, int max_batch) {
  auto ar = spec.GetRepeatedArgument<float>("random_aspect_ratio");
  auto area = spec.GetRepeatedArgument<float>("random_area");
  if (ar.size() == 1) ar.push_back(ar[0]);
  if (area.size() == 1) area.push_back(area[0]);
  DALI_ENFORCE(ar.size() == 2 && area.size() == 2, "random_aspect_ratio / random_area expect a scalar or a [min, max] pair");
  DALI_ENFORCE(ar[0] <= ar[1], "Provided empty range");
  DALI_ENFORCE(area[0] <= area[1], "Provided empty range");
  int64_t seed = spec.GetArgument<int64_t>("seed");
  if (seed < 0) seed = static_cast<int64_t>(time(nullptr));         // random_crop_attr.h:50-52
  return MakeRandomCropGenerators(max_batch, seed, ar.data(), area.data(), spec.GetArgument<int>("num_attempts"));
}

DALI_SCHEMA(decoders__ImageRandomCrop)
    .DocStr("Decodes JPEG images on the GPU and extracts a randomly placed window of random area and aspect ratio.")
    .NumInput(1).NumOutput(1)
    DALIB200_DECODER_ARGS() DALIB200_RANDOM_CROP_ARGS();

class ImageDecoderRandomCropMixed : public ImageDecoderBase {
 public:
  explicit ImageDecoderRandomCropMixed(const OpSpec &spec)
      : ImageDecoderBase(spec, "decoders.image_random_crop"), gens_(MakeCropGenerators(spec, max_batch_size_)) {}
 protected:
  bool HasRoi() const override { return true; }
  void SampleRoi(dalib200JpegRoi &roi, const Workspace &, int i, int H, int W) override {
    const CropWindow2D c = (*gens_)[i].Generate(H, W);
    roi = { 1, c.anchor[1], c.anchor[0], c.anchor[1] + c.shape[1], c.anchor[0] + c.shape[0] };
  }
  CropGenerators gens_;
};
DALI_REGISTER_OPERATOR(decoders__ImageRandomCrop, ImageDecoderRandomCropMixed, Mixed);

// ----------------------------------------------------------------------------------------------- decoders.image_slice
// decoder_schema.cc:198-245 + SliceAttr (dali/operators/generic/slice/slice_attr.h): anchor / shape as positional CPU inputs
// (normalized by default) or as `start` / `rel_start` / `end` / `rel_end` / `shape` / `rel_shape` arguments, axes (1, 0) =
// (x, y) by default ("WH").
DALI_SCHEMA(decoders__ImageSlice)
    .DocStr("Decodes JPEG images on the GPU and extracts a region of interest given by anchor and shape.")
    .NumInput(1, 3).NumOutput(1)
    DALIB200_DECODER_ARGS()
    .AddOptionalArg("axes", "Order of the dimensions of anchor and shape.", std::vector<int>{1, 0})
    .AddOptionalArg("axis_names", "Order of the dimensions of anchor and shape, as layout characters.", std::string("WH"))
    .AddOptionalArg("normalized_anchor", "The anchor input is in normalised coordinates.", true)
    .AddOptionalArg("normalized_shape", "The shape input is in normalised coordinates.", true)
    .AddOptionalArgNoDefault("start", "Start of the slice (absolute).", true)
    .AddOptionalArgNoDefault("rel_start", "Start of the slice (relative).", true)
    .AddOptionalArgNoDefault("end", "End of the slice (absolute).", true)
    .AddOptionalArgNoDefault("rel_end", "End of the slice (relative).", true)
    .AddOptionalArgNoDefault("shape", "Shape of the slice (absolute).", true)
    .AddOptionalArgNoDefault("rel_shape", "Shape of the slice (relative).", true);

// slice_attr.h:36-345 (NamedSliceAttr / PositionalSliceAttr) for the H and W axes of an image
struct SliceArgs {
  std::vector<int> axes;
  bool norm_anchor = true, norm_shape = true, positional = false;
  void Init(const OpSpec &spec, const char *name) {
    const std::string names = spec.GetArgument<std::string>("axis_names");
    if (spec.ArgumentDefined("axes") || names.empty()) {
      axes = spec.GetRepeatedArgument<int>("axes");
    } else {
      for (char c : names) {
        DALI_ENFORCE(c == 'H' || c == 'W', name, ": axis_names may contain H and W only");
        axes.push_back(c == 'H' ? 0 : 1);
      }
    }
    for (int a : axes) DALI_ENFORCE(a == 0 || a == 1, name, ": only the H (0) and W (1) axes can be sliced");
    norm_anchor = spec.GetArgument<bool>("normalized_anchor"); norm_shape = spec.GetArgument<bool>("normalized_shape");
    positional = spec.NumInput() == 3;
    DALI_ENFORCE(spec.NumInput() == 1 || spec.NumInput() == 3, name, " expects 1 input (and slice arguments) or 3 inputs (data, anchor, shape)");
    const bool has_start = spec.ArgumentDefined("start") || spec.ArgumentDefined("rel_start");
    const bool has_end = spec.ArgumentDefined("end") || spec.ArgumentDefined("rel_end");
    const bool has_shape = spec.ArgumentDefined("shape") || spec.ArgumentDefined("rel_shape");
    DALI_ENFORCE(!(positional && (has_start || has_end || has_shape)), "Named slice arguments cannot be mixed with positional anchor / shape inputs");
    DALI_ENFORCE(!(has_end && has_shape), "`end`/`rel_end` and `shape`/`rel_shape` are mutually exclusive");
  }
  // [b, e) per axis (0 = H, 1 = W) for an H x W image; not clamped
  void Get(const OpSpec &spec_, const Workspace &ws, int i, int64_t H, int64_t W, int64_t b[2], int64_t e[2]) const {
    const int64_t dim[2] = { H, W };
    b[0] = b[1] = 0; e[0] = H; e[1] = W;
    const int na = static_cast<int>(axes.size());
    for (int k = 0; k < na; k++) {
      const int ax = axes[k];
      double anchor_val = 0, end_val = static_cast<double>(dim[ax]);
      if (positional) {
        // slice_attr.h:282-330 (PositionalSliceAttr)
        const auto &anc = ws.Input<CPUBackend>(1);
        const auto &shp = ws.Input<CPUBackend>(2);
        DALI_ENFORCE(anc.type() == DALI_FLOAT && shp.type() == DALI_FLOAT, "slice: anchor and shape inputs must be float");
        DALI_ENFORCE(anc.shape().tensor_size(i) == na && shp.shape().tensor_size(i) == na,
                     "Expected ", na, " elements for slice arguments (start/shape). Got ", anc.shape().tensor_size(i));
        anchor_val = anc.tensor<float>(i)[k];
        double shape_val = shp.tensor<float>(i)[k];
        if (norm_anchor && norm_shape) {          // multiply once, after the sum
          end_val = (anchor_val + shape_val) * dim[ax];
          anchor_val *= dim[ax];
        } else {
          if (norm_anchor) anchor_val *= dim[ax];
          if (norm_shape) shape_val *= dim[ax];
          end_val = anchor_val + shape_val;
        }
      } else {
        // slice_attr.h:111-181 (NamedSliceAttr); start / end / shape are integer arguments, rel_* are floats
        auto arg = [&](const char *name) { return static_cast<double>(spec_.GetFloatVecArgument(name, &ws, i, na)[k]); };
        const bool has_start = spec_.ArgumentDefined("start"), has_rel_start = spec_.ArgumentDefined("rel_start");
        if (has_start) anchor_val = static_cast<int>(arg("start"));
        else if (has_rel_start) anchor_val = static_cast<double>(static_cast<float>(arg("rel_start"))) * dim[ax];
        if (spec_.ArgumentDefined("end")) end_val = static_cast<int>(arg("end"));
        else if (spec_.ArgumentDefined("rel_end")) end_val = static_cast<double>(static_cast<float>(arg("rel_end"))) * dim[ax];
        else if (spec_.ArgumentDefined("shape")) end_val = anchor_val + static_cast<int>(arg("shape"));
        else if (has_rel_start && !has_start && spec_.ArgumentDefined("rel_shape"))
          end_val = (static_cast<double>(static_cast<float>(arg("rel_start"))) + static_cast<double>(static_cast<float>(arg("rel_shape")))) * dim[ax];
        else if (spec_.ArgumentDefined("rel_shape")) end_val = anchor_val + static_cast<double>(static_cast<float>(arg("rel_shape"))) * dim[ax];
      }
      DALI_ENFORCE(end_val >= anchor_val, "end coordinates can't be before start coordinates. Got: start=", anchor_val, " end=", end_val);
      b[ax] = std::llround(anchor_val);
      e[ax] = std::llround(end_val);
    }
  }
};

#define DALIB200_SLICE_ARGS(schema)                                                                                            \
  schema.AddOptionalArg("axes", "Order of the dimensions of anchor and shape.", std::vector<int>{1, 0})                        \
      .AddOptionalArg("axis_names", "Order of the dimensions of anchor and shape, as layout characters.", std::string("WH"))   \
      .AddOptionalArg("normalized_anchor", "The anchor input is in normalised coordinates.", true)                             \
      .AddOptionalArg("normalized_shape", "The shape input is in normalised coordinates.", true)                               \
      .AddOptionalArgNoDefault("start", "Start of the slice (absolute).", true)                                                \
      .AddOptionalArgNoDefault("rel_start", "Start of the slice (relative).", true)                                            \
      .AddOptionalArgNoDefault("end", "End of the slice (absolute).", true)                                                    \
      .AddOptionalArgNoDefault("rel_end", "End of the slice (relative).", true)                                                \
      .AddOptionalArgNoDefault("shape", "Shape of the slice (absolute).", true)                                                \
      .AddOptionalArgNoDefault("rel_shape", "Shape of the slice (relative).", true)

class ImageDecoderSliceMixed : public ImageDecoderBase {
 public:
  explicit ImageDecoderSliceMixed(const OpSpec &spec) : ImageDecoderBase(spec, "decoders.image_slice") { slice_.Init(spec, name_); }
 protected:
  bool HasRoi() const override { return true; }
  void SampleRoi(dalib200JpegRoi &roi, const Workspace &ws, int i, int H, int W) override {
    int64_t b[2], e[2];
    slice_.Get(spec_, ws, i, H, W, b, e);
    DALI_ENFORCE(b[0] >= 0 && b[1] >= 0 && e[0] <= H && e[1] <= W && b[0] < e[0] && b[1] < e[1],
                 "decoders.image_slice: sample ", i, ": slice [", b[0], ", ", e[0], ") x [", b[1], ", ", e[1], ") must be non-empty and inside the image {", H, ", ", W, "}");
    roi = { 1, static_cast<int>(b[1]), static_cast<int>(b[0]), static_cast<int>(e[1]), static_cast<int>(e[0]) };
  }
  SliceArgs slice_;
};
DALI_REGISTER_OPERATOR(decoders__ImageSlice, ImageDecoderSliceMixed, Mixed);

// =============================================================================================== Resize
DALI_SCHEMA(Resize)
    .DocStr("Resizes images (separable resampling, fused two-pass CUDA kernel).")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArgNoDefault("resize_x", "Length of the X dimension of the resized image (0 = keep aspect).", true)
    .AddOptionalArgNoDefault("resize_y", "Length of the Y dimension of the resized image (0 = keep aspect).", true)
    .AddOptionalArgNoDefault("resize_z", "Length of the Z dimension of the resized volume (DHWC / FDHWC inputs).", true)
    .AddOptionalArgNoDefault("size", "Desired output size (H, W) or (D, H, W).", true)
    .AddOptionalArgNoDefault("resize_shorter", "Length of the shorter dimension of the resized image.", true)
    .AddOptionalArgNoDefault("resize_longer", "Length of the longer dimension of the resized image.", true)
    .AddOptionalArgNoDefault("mode", "default | stretch | not_larger | not_smaller")
    .AddOptionalArgNoDefault("max_size", "Limit of the output size.")
    .AddOptionalArg("subpixel_scale", "Adjust the ROI so that fractional sizes keep the scale.", true)
    .AddOptionalArgNoDefault("roi_start", "Origin of the input region of interest.", true)
    .AddOptionalArgNoDefault("roi_end", "End of the input region of interest.", true)
    .AddOptionalArg("roi_relative", "ROI given in relative coordinates.", false)
    .AddOptionalArg("interp_type", "Type of interpolation.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("mag_filter", "Filter used when scaling up.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("min_filter", "Filter used when scaling down.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("antialias", "Apply an antialiasing filter when scaling down.", true)
    .AddOptionalArgNoDefault("dtype", "Output type: same as input or FLOAT.")
    .AddOptionalArg("minibatch_size", "ignored (the whole batch is one launch)", 32)
    .AddOptionalArg("temp_buffer_hint", "ignored (the intermediate lives in shared memory)", 0)
    .AddOptionalArg("save_attrs", "not supported", false);

namespace resize_detail {
enum class Mode { Default, Stretch, NotLarger, NotSmaller };

// resize_attr_base.cc:86-188
void AdjustOutputSize(float *out_size, const float *in_size, int ndim, Mode mode, const float *max_size) {
  double scale[3] = {1, 1, 1};
  bool mask[3] = {false, false, false};
  int provided = 0;
  for (int d = 0; d < ndim; d++) {
    mask[d] = (out_size[d] != 0 && in_size[d] != 0);
    scale[d] = in_size[d] ? out_size[d] / in_size[d] : 1;
    provided += mask[d];
  }
  if (provided == 0) {
    for (int d = 0; d < ndim; d++) out_size[d] = in_size[d];
    return;
  }
  if (mode == Mode::Default || mode == Mode::Stretch) {
    if (provided < ndim) {
      double avg = 1;
      if (mode == Mode::Default) {
        for (int d = 0; d < ndim; d++) if (mask[d]) avg *= std::abs(scale[d]);
        if (provided > 1) avg = std::pow(avg, 1.0 / provided);
      }
      for (int d = 0; d < ndim; d++) if (!mask[d]) { scale[d] = avg; out_size[d] = mode == Mode::Default ? in_size[d] * scale[d] : in_size[d]; }
    }
    if (max_size)
      for (int d = 0; d < ndim; d++)
        if (max_size[d] > 0 && std::abs(out_size[d]) > max_size[d]) { out_size[d] = std::copysignf(max_size[d], out_size[d]); scale[d] = out_size[d] / in_size[d]; }
  } else {
    double fs = 0; bool first = true;
    for (int d = 0; d < ndim; d++) if (mask[d]) {
      float s = std::abs(scale[d]);
      if (first || (mode == Mode::NotSmaller && s > fs) || (mode == Mode::NotLarger && s < fs)) fs = s;
      first = false;
    }
    if (max_size) for (int d = 0; d < ndim; d++) if (max_size[d] > 0) { double s = static_cast<double>(max_size[d]) / in_size[d]; if (s < fs) fs = s; }
    for (int d = 0; d < ndim; d++) if (!mask[d] || std::abs(scale[d]) != fs) { scale[d] = std::copysign(fs, scale[d]); out_size[d] = in_size[d] * scale[d]; }
  }
}

struct Params { int dst[3]; float lo[3], hi[3]; };

// resize_attr_base.h:51-119 (alignment = centre, size_round_fn = round_int); ndim = 2 (images) or 3 (volumes)
void CalculateSampleParams(Params &p, float *req, float *in_lo, float *in_hi, bool adjust_roi, bool empty_input, Mode mode,
                           const float *max_size, int ndim = 2) {
  float in_size[3];
  for (int d = 0; d < ndim; d++) {
    float sz = in_hi[d] - in_lo[d];
    if (sz < 0) { std::swap(in_hi[d], in_lo[d]); req[d] = -req[d]; sz = -sz; }
    in_size[d] = sz;
  }
  AdjustOutputSize(req, in_size, ndim, mode, max_size);
  for (int d = 0; d < ndim; d++) DALI_ENFORCE(in_lo[d] != in_hi[d] || req[d] == 0, "Cannot produce non-empty output from empty input");
  const int min_size = empty_input ? 0 : 1;
  for (int d = 0; d < ndim; d++) {
    p.lo[d] = in_lo[d]; p.hi[d] = in_hi[d];
    const float out_sz = req[d];
    const bool flip = out_sz < 0;
    p.dst[d] = std::max(min_size, static_cast<int>(std::roundf(std::fabs(out_sz))));
    if (flip) std::swap(p.lo[d], p.hi[d]);
    if (adjust_roi && p.dst[d] != std::fabs(out_sz)) {
      const double real_size = p.dst[d];
      double adjustment = real_size / std::fabs(out_sz);
      adjustment = std::min(std::max(adjustment, -10.0), 10.0);
      const double a = 0.5f;
      const double center = (1.0 - a) * p.lo[d] + a * p.hi[d];
      p.lo[d] = static_cast<float>(std::min(std::max(center + (p.lo[d] - center) * adjustment, -1e+9), 1e+9));
      p.hi[d] = static_cast<float>(std::min(std::max(center + (p.hi[d] - center) * adjustment, -1e+9), 1e+9));
    }
  }
}
}  // namespace resize_detail

static int Interp2Filter(int interp) {      // resampling_attr.cc:60-74
  switch (interp) {
    case DALI_INTERP_NN: return DALIB200_FILTER_NN;
    case DALI_INTERP_LINEAR: return DALIB200_FILTER_LINEAR;
    case DALI_INTERP_CUBIC: return DALIB200_FILTER_CUBIC;
    case DALI_INTERP_LANCZOS3: return DALIB200_FILTER_LANCZOS3;
    case DALI_INTERP_GAUSSIAN: return DALIB200_FILTER_GAUSSIAN;
    case DALI_INTERP_TRIANGULAR: return DALIB200_FILTER_TRIANGULAR;
    default: DALI_FAIL("Unknown interpolation type");
  }
}

class ResizeGPU : public Operator<GPUBackend>, public PlanarConsumer {
 public:
  void AttachProducer(PlanarProducer *p) override {
    producer_ = p;
    CheckStatus(dalib200ResamplePlanCreate(&plan_planar_, plan_cap_), "Resize");
    planar_cap_ = plan_cap_;
  }
  // hook of ResizeCropMirror: crop window and mirror applied to the per-sample parameters
  virtual void AdjustSampleParams(resize_detail::Params &, const Workspace &, int) {}
  explicit ResizeGPU(const OpSpec &spec, const char *name = "Resize") : Operator<GPUBackend>(spec) {
    using resize_detail::Mode;
    has_shorter_ = spec.ArgumentDefined("resize_shorter"); has_longer_ = spec.ArgumentDefined("resize_longer");
    has_x_ = spec.ArgumentDefined("resize_x"); has_y_ = spec.ArgumentDefined("resize_y");
    has_size_ = spec.ArgumentDefined("size"); has_max_ = spec.ArgumentDefined("max_size");
    const bool has_mode = spec.ArgumentDefined("mode");
    plain_resize_ = name == std::string("Resize");      // derived operators (ResizeCropMirror) stay 2-D
    DALI_ENFORCE(plain_resize_ || !spec.ArgumentDefined("resize_z"), name, ": `resize_z` (volumetric data) is not supported by the GPU path");
    has_z_ = plain_resize_ && spec.ArgumentDefined("resize_z");
    DALI_ENFORCE(!spec.GetArgument<bool>("save_attrs"), "Resize: `save_attrs` is not supported");
    DALI_ENFORCE((has_x_ || has_y_ || has_z_) + has_size_ + has_shorter_ + has_longer_ == 1,
                 "Exactly one method of specifying size must be used. The available methods:\n"
                 "    - separate resize_x, resize_y, resize_z arguments\n    - size argument\n    - resize_longer\n    - resize_shorter");
    DALI_ENFORCE(has_shorter_ + has_longer_ + has_mode <= 1, "`resize_shorter`, ``resize_longer`` and ``mode`` arguments are mutually exclusive");
    DALI_ENFORCE(spec.ArgumentDefined("roi_start") == spec.ArgumentDefined("roi_end"), "``roi_start`` and ``roi_end`` must be specified together");
    has_roi_ = spec.ArgumentDefined("roi_start");
    roi_relative_ = spec.GetArgument<bool>("roi_relative");
    subpixel_scale_ = spec.GetArgument<bool>("subpixel_scale");
    if (has_shorter_) mode_ = Mode::NotSmaller;
    else if (has_longer_) mode_ = Mode::NotLarger;
    else if (has_mode) {
      const std::string m = spec.GetArgument<std::string>("mode");
      if (m == "default") mode_ = Mode::Default; else if (m == "stretch") mode_ = Mode::Stretch;
      else if (m == "not_larger") mode_ = Mode::NotLarger; else if (m == "not_smaller") mode_ = Mode::NotSmaller;
      else DALI_FAIL(make_string("Invalid resize mode: \"", m, "\""));
    }
    antialias_ = spec.GetArgument<bool>("antialias");
    CheckStatus(dalib200ResamplePlanCreate(&plan_, max_batch_size_ * 64), "Resize");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~ResizeGPU() override {
    dalib200ResamplePlanDestroy(plan_);
    if (plan_planar_) dalib200ResamplePlanDestroy(plan_planar_);
    if (plan3_) dalib200Resample3DPlanDestroy(plan3_);
  }

 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    const int n = in.num_samples();
    DALI_ENFORCE(in.type() == DALI_UINT8 || in.type() == DALI_FLOAT, "Resize: the GPU path supports uint8 and float inputs");
    DALIDataType out_type = in.type();
    if (spec_.ArgumentDefined("dtype")) out_type = spec_.GetArgument<DALIDataType>("dtype");
    DALI_ENFORCE(out_type == in.type() || out_type == DALI_FLOAT, "Resize: output type must be the same as input or FLOAT");
    volumes_ = in.GetLayout().str().find('D') != std::string::npos;
    DALI_ENFORCE(!volumes_ || plain_resize_, "ResizeCropMirror: volumetric inputs are not supported by the GPU path");
    if (volumes_) return SetupVolumes(out, ws, out_type);
    frames_ = ExpandFramesAnyLayout(in.shape(), in.GetLayout(), "Resize");
    const int nf = frames_.num_frames();
    if (nf > plan_cap_) { dalib200ResamplePlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200ResamplePlanCreate(&plan_, nf), "Resize"); }
    std::vector<float> max_size(2, std::nextafter(static_cast<float>(std::numeric_limits<int>::max()), 0.0f));
    if (has_max_) max_size = spec_.GetFloatVecArgument("max_size", &ws, 0, 2);
    const bool has_interp = spec_.ArgumentDefined("interp_type"), has_min = spec_.ArgumentDefined("min_filter"),
               has_mag = spec_.ArgumentDefined("mag_filter");
    samples_.assign(nf, dalib200ResampleSample());
    out_hw_.assign(n, {0, 0});
    int fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      const float in_h = static_cast<float>(s[fs]), in_w = static_cast<float>(s[fs + 1]);
      float req[2] = {0, 0};     // (H, W) order
      if (has_x_ || has_y_ || has_z_) {          // `resize_z` alone on 2-D data: both extents unspecified (resize_attr.cc:214-245)
        if (has_y_) req[0] = spec_.GetArgument<float>("resize_y", &ws, i);
        if (has_x_) req[1] = spec_.GetArgument<float>("resize_x", &ws, i);
      } else if (has_shorter_ || has_longer_) {
        req[0] = req[1] = spec_.GetArgument<float>(has_shorter_ ? "resize_shorter" : "resize_longer", &ws, i);
      } else {
        auto v = spec_.GetFloatVecArgument("size", &ws, i, 2);
        req[0] = v[0]; req[1] = v[1];
      }
      float lo[2] = {0, 0}, hi[2] = {in_h, in_w};
      if (has_roi_) {          // resize_attr.cc:125-160
        auto rs = spec_.GetFloatVecArgument("roi_start", &ws, i, 2), re = spec_.GetFloatVecArgument("roi_end", &ws, i, 2);
        const float isz[2] = {in_h, in_w};
        for (int d = 0; d < 2; d++) if (isz[d] > 0) {
          double l = rs[d], h = re[d];
          if (roi_relative_) { l *= isz[d]; h *= isz[d]; }
          if (std::fabs(h - l) < 1e-3f) { float off = l <= h ? 0.5f * 1e-3f : -0.5f * 1e-3f; l -= off; h += off; }
          lo[d] = static_cast<float>(l); hi[d] = static_cast<float>(h);
        }
      }
      resize_detail::Params p;
      const bool empty_input = in.shape().tensor_size(i) == 0;
      resize_detail::CalculateSampleParams(p, req, lo, hi, subpixel_scale_, empty_input, mode_, has_max_ ? max_size.data() : nullptr);
      AdjustSampleParams(p, ws, i);
      // filters (resampling_attr.cc:76-133)
      int interp = spec_.GetArgument<int>("interp_type", &ws, i);
      int minf = DALIB200_FILTER_TRIANGULAR, magf = DALIB200_FILTER_LINEAR;
      auto conv = [](int t, bool aa) {
        if (aa && t == DALI_INTERP_LINEAR) t = DALI_INTERP_TRIANGULAR; else if (!aa && t == DALI_INTERP_TRIANGULAR) t = DALI_INTERP_LINEAR;
        return Interp2Filter(t);
      };
      if (has_min) minf = conv(spec_.GetArgument<int>("min_filter", &ws, i), antialias_); else if (has_interp) minf = conv(interp, antialias_);
      if (has_mag) magf = conv(spec_.GetArgument<int>("mag_filter", &ws, i), false); else if (has_interp) magf = conv(interp, false);
      out_hw_[i] = { p.dst[0], p.dst[1] };
      int64_t frames = 1, chans = 1;            // leading dimensions are frames, trailing ones channels (CHW: C frames of one channel)
      for (int d = 0; d < fs; d++) frames *= s[d];
      for (int d = fs + 2; d < in.shape().sample_dim(); d++) chans *= s[d];
      for (int64_t k = 0; k < frames; k++, fk++) {
        auto &r = samples_[fk];
        r.in_h = static_cast<int>(s[fs]); r.in_w = static_cast<int>(s[fs + 1]); r.channels = static_cast<int>(chans);
        r.out_h = p.dst[0]; r.out_w = p.dst[1];
        for (int d = 0; d < 2; d++) {
          r.use_roi[d] = p.lo[d] != p.hi[d];            // GetResamplingParams: roi only when non-degenerate
          r.roi_start[d] = p.lo[d]; r.roi_end[d] = p.hi[d];
          r.min_filter[d] = { minf, antialias_ ? 1 : 0, 0.0f };
          r.mag_filter[d] = { magf, 0, 0.0f };
        }
      }
    }
    // ---- fused with the decoder that produces the input: the samples the planar kernel can take never exist as RGB images
    planar_.assign(nf, 0);
    rest_.clear();
    if (producer_ && frames_.first_spatial == 0 && nf == n && in.type() == DALI_UINT8 && out_type == DALI_UINT8) {
      if (nf > planar_cap_) { dalib200ResamplePlanDestroy(plan_planar_); plan_planar_ = nullptr; planar_cap_ = nf; CheckStatus(dalib200ResamplePlanCreate(&plan_planar_, nf), "Resize"); }
      std::vector<uint8_t> ok(nf, 0), granted;
      CheckStatus(dalib200ResamplePlanSetupPlanar(plan_planar_, nf, samples_.data(), ok.data()), "Resize");
      producer_->SelectPlanar(ok, granted);
      if (ok != granted) {       // the resampler's item list must cover exactly the granted samples
        std::vector<dalib200ResampleSample> tmp(samples_);
        for (int i = 0; i < nf; i++) if (!granted[i]) tmp[i].channels = 1;      // 1-channel samples are never planar-eligible
        CheckStatus(dalib200ResamplePlanSetupPlanar(plan_planar_, nf, tmp.data(), ok.data()), "Resize");
      }
      planar_ = granted;
    } else if (producer_) {
      std::vector<uint8_t> none(n, 0), granted;
      producer_->SelectPlanar(none, granted);
    }
    for (int k = 0; k < nf; k++) if (!planar_[k]) rest_.push_back(k);
    if (static_cast<int>(rest_.size()) == nf) {
      CheckStatus(dalib200ResamplePlanSetup(plan_, nf, samples_.data(), in.type() == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT,
                                            out_type == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "Resize");
    } else if (!rest_.empty()) {
      std::vector<dalib200ResampleSample> sub(rest_.size());
      for (size_t q = 0; q < rest_.size(); q++) sub[q] = samples_[rest_[q]];
      CheckStatus(dalib200ResamplePlanSetup(plan_, static_cast<int>(sub.size()), sub.data(), DALIB200_UINT8, DALIB200_UINT8), "Resize");
    }
    out.resize(1);
    out[0].type = out_type;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      sh[frames_.first_spatial] = out_hw_[i].first; sh[frames_.first_spatial + 1] = out_hw_[i].second;
      out[0].shape.set_tensor_shape(i, sh);
    }
    out_type_ = out_type;
    return true;
  }

  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    if (volumes_) { RunVolumes(ws); return; }
    out.SetLayout(in.GetLayout().empty() ? TensorLayout(frames_.first_spatial ? "FHWC" : "HWC") : in.GetLayout());
    auto ip = FramePtrs(in, frames_, TypeSize(in.type()));
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      const int64_t fr = static_cast<int64_t>(out_hw_[s].first) * out_hw_[s].second * frames_.c[k] * TypeSize(out_type_);
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += fr;
    }
    if (producer_) {
      producer_->RunDeferred(ws.stream());
      if (rest_.size() != op.size()) {
        std::vector<dalib200PlanarImage> srcs(op.size());
        for (size_t k = 0; k < op.size(); k++) {
          memset(&srcs[k], 0, sizeof(srcs[k]));
          if (!planar_[k]) continue;
          PlanarSource ps;
          producer_->GetPlanarSource(static_cast<int>(k), &ps);
          srcs[k].y = ps.y; srcs[k].cb = ps.cb; srcs[k].cr = ps.cr; srcs[k].pitch_y = ps.pitch_y; srcs[k].pitch_c = ps.pitch_c;
          srcs[k].width = ps.width; srcs[k].height = ps.height; srcs[k].crop_x = ps.crop_x; srcs[k].crop_y = ps.crop_y;
        }
        CheckStatus(dalib200ResampleLaunchPlanar(plan_planar_, srcs.data(), op.data(), ws.stream()), "Resize");
      }
    }
    if (rest_.size() == op.size()) {
      CheckStatus(dalib200ResampleLaunch(plan_, ip.data(), op.data(), ws.stream()), "Resize");
    } else if (!rest_.empty()) {
      std::vector<const void *> ip2(rest_.size());
      std::vector<void *> op2(rest_.size());
      for (size_t q = 0; q < rest_.size(); q++) { ip2[q] = ip[rest_[q]]; op2[q] = op[rest_[q]]; }
      CheckStatus(dalib200ResampleLaunch(plan_, ip2.data(), op2.data(), ws.stream()), "Resize");
    }
  }

  // ---- volumes (DHWC, FDHWC): ResizeAttr with spatial_ndim = 3 (resize_attr.cc:102-255) over dalib200Resample3D*; the frames of an
  // FDHWC sample are independent volumes with the sample's parameters (SequenceOperator, sequence_operator.h:57-110)
  bool SetupVolumes(std::vector<OutputDesc> &out, const Workspace &ws, DALIDataType out_type) {
    const auto &in = ws.Input<GPUBackend>(0);
    const int n = in.num_samples();
    const std::string lay = in.GetLayout().str();
    const int nd = in.shape().sample_dim();
    int sd = 3, fs = 0;
    ParseResizeLayout(lay, &sd, &fs);
    DALI_ENFORCE(nd == static_cast<int>(lay.size()), "Resize: layout \"", lay, "\" does not match a ", nd, "-D input");
    if (producer_) { std::vector<uint8_t> none(n, 0), granted; producer_->SelectPlanar(none, granted); }
    std::vector<float> max_size(3, std::nextafter(static_cast<float>(std::numeric_limits<int>::max()), 0.0f));
    if (has_max_) max_size = spec_.GetFloatVecArgument("max_size", &ws, 0, 3);
    const bool has_interp = spec_.ArgumentDefined("interp_type"), has_min = spec_.ArgumentDefined("min_filter"),
               has_mag = spec_.ArgumentDefined("mag_filter");
    vsamples_.clear();
    vol_sample_.clear(); vol_offset_.clear();
    out_dhw_.assign(n, {0, 0, 0});
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const float isz[3] = { static_cast<float>(s[fs]), static_cast<float>(s[fs + 1]), static_cast<float>(s[fs + 2]) };
      float req[3] = {0, 0, 0};     // (D, H, W): the shape order of `size`
      if (has_x_ || has_y_ || has_z_) {
        if (has_z_) req[0] = spec_.GetArgument<float>("resize_z", &ws, i);
        if (has_y_) req[1] = spec_.GetArgument<float>("resize_y", &ws, i);
        if (has_x_) req[2] = spec_.GetArgument<float>("resize_x", &ws, i);
      } else if (has_shorter_ || has_longer_) {
        req[0] = req[1] = req[2] = spec_.GetArgument<float>(has_shorter_ ? "resize_shorter" : "resize_longer", &ws, i);
      } else {
        auto v = spec_.GetFloatVecArgument("size", &ws, i, 3);
        req[0] = v[0]; req[1] = v[1]; req[2] = v[2];
      }
      float lo[3] = {0, 0, 0}, hi[3] = { isz[0], isz[1], isz[2] };
      if (has_roi_) {          // resize_attr.cc:125-160
        auto rs = spec_.GetFloatVecArgument("roi_start", &ws, i, 3), re = spec_.GetFloatVecArgument("roi_end", &ws, i, 3);
        for (int d = 0; d < 3; d++) if (isz[d] > 0) {
          double l = rs[d], h = re[d];
          if (roi_relative_) { l *= isz[d]; h *= isz[d]; }
          if (std::fabs(h - l) < 1e-3f) { float off = l <= h ? 0.5f * 1e-3f : -0.5f * 1e-3f; l -= off; h += off; }
          lo[d] = static_cast<float>(l); hi[d] = static_cast<float>(h);
        }
      }
      resize_detail::Params p;
      const bool empty_input = in.shape().tensor_size(i) == 0;
      resize_detail::CalculateSampleParams(p, req, lo, hi, subpixel_scale_, empty_input, mode_, has_max_ ? max_size.data() : nullptr, 3);
      int interp = spec_.GetArgument<int>("interp_type", &ws, i);
      int minf = DALIB200_FILTER_TRIANGULAR, magf = DALIB200_FILTER_LINEAR;
      auto conv = [](int t, bool aa) {      // resampling_attr.cc:76-133
        if (aa && t == DALI_INTERP_LINEAR) t = DALI_INTERP_TRIANGULAR; else if (!aa && t == DALI_INTERP_TRIANGULAR) t = DALI_INTERP_LINEAR;
        return Interp2Filter(t);
      };
      if (has_min) minf = conv(spec_.GetArgument<int>("min_filter", &ws, i), antialias_); else if (has_interp) minf = conv(interp, antialias_);
      if (has_mag) magf = conv(spec_.GetArgument<int>("mag_filter", &ws, i), false); else if (has_interp) magf = conv(interp, false);
      out_dhw_[i] = { p.dst[0], p.dst[1], p.dst[2] };
      int64_t frames = 1, chans = 1;            // leading dimensions are frames, trailing ones channels (CDHW: C volumes of one channel)
      for (int d = 0; d < fs; d++) frames *= s[d];
      for (int d = fs + 3; d < nd; d++) chans *= s[d];
      const int64_t in_vol = s[fs] * s[fs + 1] * s[fs + 2] * chans;
      for (int64_t k = 0; k < frames; k++) {
        dalib200Resample3DSample r;
        memset(&r, 0, sizeof(r));
        r.channels = static_cast<int>(chans);
        for (int d = 0; d < 3; d++) {
          r.in_shape[d] = static_cast<int>(s[fs + d]); r.out_shape[d] = p.dst[d];
          r.use_roi[d] = p.lo[d] != p.hi[d];
          r.roi_start[d] = p.lo[d]; r.roi_end[d] = p.hi[d];
          r.min_filter[d] = { minf, antialias_ ? 1 : 0, 0.0f };
          r.mag_filter[d] = { magf, 0, 0.0f };
        }
        vsamples_.push_back(r);
        vol_sample_.push_back(i);
        vol_offset_.push_back(k * in_vol);
      }
    }
    const int nv = static_cast<int>(vsamples_.size());
    if (nv > plan3_cap_ || !plan3_) {
      if (plan3_) dalib200Resample3DPlanDestroy(plan3_);
      plan3_ = nullptr; plan3_cap_ = std::max(nv, max_batch_size_);
      CheckStatus(dalib200Resample3DPlanCreate(&plan3_, plan3_cap_), "Resize");
    }
    CheckStatus(dalib200Resample3DPlanSetup(plan3_, nv, vsamples_.data(), in.type() == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT,
                                            out_type == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "Resize");
    out.resize(1);
    out[0].type = out_type;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      for (int d = 0; d < 3; d++) sh[fs + d] = out_dhw_[i][d];
      out[0].shape.set_tensor_shape(i, sh);
    }
    out_type_ = out_type;
    return true;
  }

  void RunVolumes(Workspace &ws) {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout());
    if (producer_) producer_->RunDeferred(ws.stream());
    const size_t nv = vsamples_.size();
    std::vector<const void *> ip(nv);
    std::vector<void *> op(nv);
    std::vector<int64_t> next(out.num_samples(), 0);
    for (size_t k = 0; k < nv; k++) {
      const int s = vol_sample_[k];
      ip[k] = static_cast<const uint8_t *>(in.raw_tensor(s)) + vol_offset_[k] * TypeSize(in.type());
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(out_dhw_[s][0]) * out_dhw_[s][1] * out_dhw_[s][2] * vsamples_[k].channels * TypeSize(out_type_);
    }
    CheckStatus(dalib200Resample3DLaunch(plan3_, ip.data(), op.data(), ws.stream()), "Resize");
  }

 private:
  dalib200Resample3DPlan *plan3_ = nullptr;
  int plan3_cap_ = 0;
  bool volumes_ = false, has_z_ = false, plain_resize_ = true;
  std::vector<dalib200Resample3DSample> vsamples_;
  std::vector<int> vol_sample_;
  std::vector<int64_t> vol_offset_;
  std::vector<std::array<int, 3>> out_dhw_;
  dalib200ResamplePlan *plan_ = nullptr, *plan_planar_ = nullptr;
  int plan_cap_ = 0, planar_cap_ = 0;
  PlanarProducer *producer_ = nullptr;
  std::vector<uint8_t> planar_;
  std::vector<int> rest_;
  bool has_shorter_ = false, has_longer_ = false, has_x_ = false, has_y_ = false, has_size_ = false, has_max_ = false, has_roi_ = false;
  bool roi_relative_ = false, subpixel_scale_ = true, antialias_ = true;
  resize_detail::Mode mode_ = resize_detail::Mode::Default;
  FrameList frames_;
  std::vector<dalib200ResampleSample> samples_;
  std::vector<std::pair<int, int>> out_hw_;
  DALIDataType out_type_ = DALI_UINT8;
};
DALI_REGISTER_OPERATOR(Resize, ResizeGPU, GPU);

class ResizeCropMirrorGPU : public ResizeGPU {
 public:
  explicit ResizeCropMirrorGPU(const OpSpec &spec) : ResizeGPU(spec, "ResizeCropMirror") { crop_.Init(spec, "ResizeCropMirror"); }
  void AdjustSampleParams(resize_detail::Params &p, const Workspace &ws, int i) override {
    // resize_crop_mirror.cc:84-108; the crop window is computed on the RESIZED shape
    int64_t y0, x0, h, w;
    crop_.Get(spec_, ws, i, p.dst[0], p.dst[1], y0, x0, h, w);
    const int64_t anchor[2] = { y0, x0 }, shape[2] = { h, w };
    const int mirror = spec_.GetArgument<int>("mirror", &ws, i);
    for (int d = 0; d < 2; d++) {
      const double src_extent = p.hi[d] - p.lo[d];
      const double resize_ratio = src_extent / p.dst[d];
      const double resize_offset = p.lo[d];
      const double crop_lo = static_cast<double>(anchor[d]), crop_hi = static_cast<double>(anchor[d] + shape[d]);
      p.lo[d] = static_cast<float>(crop_lo * resize_ratio + resize_offset);
      p.hi[d] = static_cast<float>(crop_hi * resize_ratio + resize_offset);
      if (mirror & (1 << (2 - 1 - d))) std::swap(p.lo[d], p.hi[d]);
      p.dst[d] = static_cast<int>(shape[d]);
    }
  }
 private:
  CropWindowArgs crop_;
};
DALI_REGISTER_OPERATOR(ResizeCropMirror, ResizeCropMirrorGPU, GPU);

// =============================================================================================== ResizeCropMirror
// dali/operators/image/resize/resize_crop_mirror.{h,cc}: resize, then crop, then flip -- executed as ONE resampling whose ROI is the
// crop window projected back into the input (resize_crop_mirror.cc:73-110).
class ResizeCropMirrorGPU;
DALI_SCHEMA(ResizeCropMirror)
    .DocStr("Performs a fused resize, crop, mirror operation.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArgNoDefault("resize_x", "Length of the X dimension of the resized image (0 = keep aspect).", true)
    .AddOptionalArgNoDefault("resize_y", "Length of the Y dimension of the resized image (0 = keep aspect).", true)
    .AddOptionalArgNoDefault("resize_z", "not supported by the GPU path (2-D images only)", true)
    .AddOptionalArgNoDefault("size", "Desired output size (H, W).", true)
    .AddOptionalArgNoDefault("resize_shorter", "Length of the shorter dimension of the resized image.", true)
    .AddOptionalArgNoDefault("resize_longer", "Length of the longer dimension of the resized image.", true)
    .AddOptionalArgNoDefault("mode", "default | stretch | not_larger | not_smaller")
    .AddOptionalArgNoDefault("max_size", "Limit of the output size.")
    .AddOptionalArg("subpixel_scale", "Adjust the ROI so that fractional sizes keep the scale.", true)
    .AddOptionalArgNoDefault("roi_start", "Origin of the input region of interest.", true)
    .AddOptionalArgNoDefault("roi_end", "End of the input region of interest.", true)
    .AddOptionalArg("roi_relative", "ROI given in relative coordinates.", false)
    .AddOptionalArg("interp_type", "Type of interpolation.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("mag_filter", "Filter used when scaling up.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("min_filter", "Filter used when scaling down.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("antialias", "Apply an antialiasing filter when scaling down.", true)
    .AddOptionalArgNoDefault("dtype", "Output type: same as input or FLOAT.")
    .AddOptionalArg("minibatch_size", "ignored (the whole batch is one launch)", 32)
    .AddOptionalArg("temp_buffer_hint", "ignored (the intermediate lives in shared memory)", 0)
    .AddOptionalArg("save_attrs", "not supported", false)
    .AddOptionalArg("mirror", "Mask for flipping: 1 = horizontal, 2 = vertical.", 0, true)
    DALIB200_CROP_ARGS();

// =============================================================================================== RandomResizedCrop
// dali/operators/image/resize/random_resized_crop.{h,cc}: a random window (RandomCropAttr) resized to `size`; the window is
// the ROI of the resampling (the filter support may reach outside it, unlike crop-then-resize).
DALI_SCHEMA(RandomResizedCrop)
    .DocStr("Performs a crop with a randomly selected area and aspect ratio and resizes it to the specified size.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddArg("size", "Size of the resized image (H, W).")
    DALIB200_RANDOM_CROP_ARGS()
    .AddOptionalArg("interp_type", "Type of interpolation.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("mag_filter", "Filter used when scaling up.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("min_filter", "Filter used when scaling down.", DALI_INTERP_LINEAR, true)
    .AddOptionalArg("antialias", "Apply an antialiasing filter when scaling down.", true)
    .AddOptionalArgNoDefault("dtype", "Output type: same as input or FLOAT.")
    .AddOptionalArg("minibatch_size", "ignored (the whole batch is one launch)", 32)
    .AddOptionalArg("temp_buffer_hint", "ignored (the intermediate lives in shared memory)", 0);

class RandomResizedCropGPU : public Operator<GPUBackend> {
 public:
  explicit RandomResizedCropGPU(const OpSpec &spec) : Operator<GPUBackend>(spec), gens_(MakeCropGenerators(spec, max_batch_size_)) {
    size_ = spec.GetRepeatedArgument<int>("size");
    if (size_.size() == 1) size_.push_back(size_[0]);
    DALI_ENFORCE(size_.size() == 2 && size_[0] > 0 && size_[1] > 0, "RandomResizedCrop: `size` must be one or two positive integers");
    antialias_ = spec.GetArgument<bool>("antialias");
    CheckStatus(dalib200ResamplePlanCreate(&plan_, max_batch_size_ * 64), "RandomResizedCrop");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~RandomResizedCropGPU() override { dalib200ResamplePlanDestroy(plan_); }

 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    const int n = in.num_samples();
    DALI_ENFORCE(in.type() == DALI_UINT8 || in.type() == DALI_FLOAT, "RandomResizedCrop: the GPU path supports uint8 and float inputs");
    out_type_ = in.type();
    if (spec_.ArgumentDefined("dtype")) out_type_ = spec_.GetArgument<DALIDataType>("dtype");
    DALI_ENFORCE(out_type_ == in.type() || out_type_ == DALI_FLOAT, "RandomResizedCrop: output type must be the same as input or FLOAT");
    frames_ = ExpandFrames(in.shape(), in.GetLayout(), "RandomResizedCrop");
    const int nf = frames_.num_frames();
    if (nf > plan_cap_) { dalib200ResamplePlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200ResamplePlanCreate(&plan_, nf), "RandomResizedCrop"); }
    const bool has_interp = spec_.ArgumentDefined("interp_type"), has_min = spec_.ArgumentDefined("min_filter"),
               has_mag = spec_.ArgumentDefined("mag_filter");
    samples_.assign(nf, dalib200ResampleSample());
    crops_.resize(n);
    int fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      const int H = static_cast<int>(s[fs]), W = static_cast<int>(s[fs + 1]);
      crops_[i] = (*gens_)[i].Generate(H, W);
      int interp = spec_.GetArgument<int>("interp_type", &ws, i);
      int minf = DALIB200_FILTER_TRIANGULAR, magf = DALIB200_FILTER_LINEAR;
      auto conv = [](int t, bool aa) {
        if (aa && t == DALI_INTERP_LINEAR) t = DALI_INTERP_TRIANGULAR; else if (!aa && t == DALI_INTERP_TRIANGULAR) t = DALI_INTERP_LINEAR;
        return Interp2Filter(t);
      };
      if (has_min) minf = conv(spec_.GetArgument<int>("min_filter", &ws, i), antialias_); else if (has_interp) minf = conv(interp, antialias_);
      if (has_mag) magf = conv(spec_.GetArgument<int>("mag_filter", &ws, i), false); else if (has_interp) magf = conv(interp, false);
      const int64_t frames = fs ? s[0] : 1;
      for (int64_t k = 0; k < frames; k++, fk++) {
        auto &r = samples_[fk];
        r.in_h = H; r.in_w = W; r.channels = static_cast<int>(s[fs + 2]);
        r.out_h = size_[0]; r.out_w = size_[1];
        for (int d = 0; d < 2; d++) {
          r.use_roi[d] = 1;
          r.roi_start[d] = static_cast<float>(crops_[i].anchor[d]);
          r.roi_end[d] = static_cast<float>(crops_[i].anchor[d] + crops_[i].shape[d]);
          r.min_filter[d] = { minf, antialias_ ? 1 : 0, 0.0f };
          r.mag_filter[d] = { magf, 0, 0.0f };
        }
      }
    }
    CheckStatus(dalib200ResamplePlanSetup(plan_, nf, samples_.data(), in.type() == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT,
                                          out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "RandomResizedCrop");
    out.resize(1);
    out[0].type = out_type_;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      sh[frames_.first_spatial] = size_[0]; sh[frames_.first_spatial + 1] = size_[1];
      out[0].shape.set_tensor_shape(i, sh);
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout().empty() ? TensorLayout(frames_.first_spatial ? "FHWC" : "HWC") : in.GetLayout());
    auto ip = FramePtrs(in, frames_, TypeSize(in.type()));
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(size_[0]) * size_[1] * frames_.c[k] * TypeSize(out_type_);
    }
    CheckStatus(dalib200ResampleLaunch(plan_, ip.data(), op.data(), ws.stream()), "RandomResizedCrop");
  }
 private:
  dalib200ResamplePlan *plan_ = nullptr;
  int plan_cap_ = 0;
  bool antialias_ = true;
  std::vector<int> size_;
  CropGenerators gens_;
  std::vector<CropWindow2D> crops_;
  FrameList frames_;
  std::vector<dalib200ResampleSample> samples_;
  DALIDataType out_type_ = DALI_UINT8;
};
DALI_REGISTER_OPERATOR(RandomResizedCrop, RandomResizedCropGPU, GPU);

// =============================================================================================== CropMirrorNormalize
DALI_SCHEMA(CropMirrorNormalize)
    .DocStr("Fused cropping, horizontal mirroring, normalisation, layout permutation and type conversion.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("dtype", "Output data type (FLOAT or FLOAT16).", DALI_FLOAT)
    .AddOptionalArg("output_layout", "Tensor data layout for the output.", std::string("CHW"))
    .AddOptionalArg("pad_output", "Pad the channel dimension to the next power of two.", false)
    .AddOptionalArg("mirror", "Flip horizontally.", 0, true)
    .AddOptionalArg("mean", "Mean pixel values.", std::vector<float>{0.0f}, true)
    .AddOptionalArg("std", "Standard deviation values.", std::vector<float>{1.0f}, true)
    .AddOptionalArg("scale", "Value by which the result is multiplied.", 1.0f)
    .AddOptionalArg("shift", "Value added to the (scaled) result.", 0.0f)
    .AddOptionalArgNoDefault("crop", "Shape of the cropped image (H, W).", true)
    .AddOptionalArgNoDefault("crop_h", "Cropping window height.", true)
    .AddOptionalArgNoDefault("crop_w", "Cropping window width.", true)
    .AddOptionalArgNoDefault("crop_d", "not supported (2-D images only)", true)
    .AddOptionalArg("crop_pos_x", "Normalised horizontal position of the window.", 0.5f, true)
    .AddOptionalArg("crop_pos_y", "Normalised vertical position of the window.", 0.5f, true)
    .AddOptionalArg("crop_pos_z", "unused", 0.5f, true)
    .AddOptionalArg("rounding", "round | truncate", std::string("round"))
    .AddOptionalArg("out_of_bounds_policy", "error | pad | trim_to_shape", std::string("error"))
    .AddOptionalArg("fill_values", "Fill values for padding.", std::vector<float>{0.0f});

class CropMirrorNormalizeGPU : public Operator<GPUBackend> {
 public:
  explicit CropMirrorNormalizeGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    out_type_ = spec.GetArgument<DALIDataType>("dtype");
    DALI_ENFORCE(out_type_ == DALI_FLOAT || out_type_ == DALI_FLOAT16, "CropMirrorNormalize: the GPU path supports dtype FLOAT and FLOAT16");
    out_layout_ = spec.GetArgument<std::string>("output_layout");
    pad_output_ = spec.GetArgument<bool>("pad_output");
    scale_ = spec.GetArgument<float>("scale"); shift_ = spec.GetArgument<float>("shift");
    const std::string r = spec.GetArgument<std::string>("rounding");
    DALI_ENFORCE(r == "round" || r == "truncate", "``rounding`` value ", r, " is not supported. Supported values are \"round\", or \"truncate\".");
    truncate_ = r == "truncate";
    oob_ = spec.GetArgument<std::string>("out_of_bounds_policy");
    DALI_ENFORCE(oob_ == "error" || oob_ == "pad" || oob_ == "trim_to_shape", "Unsupported out_of_bounds_policy: ", oob_);
    fill_values_ = spec.GetRepeatedArgument<float>("fill_values");
    DALI_ENFORCE(!spec.ArgumentDefined("crop_d"), "CropMirrorNormalize: `crop_d` is not supported by the GPU path");
    const bool has_crop = spec.ArgumentDefined("crop");
    DALI_ENFORCE(!(has_crop && (spec.ArgumentDefined("crop_h") || spec.ArgumentDefined("crop_w"))),
                 "`crop` argument is not compatible with `crop_h`, `crop_w`, `crop_d`");
    DALI_ENFORCE(spec.ArgumentDefined("crop_h") == spec.ArgumentDefined("crop_w"), "`crop_h` and `crop_w` arguments must be provided together");
    CheckStatus(dalib200CmnPlanCreate(&plan_, max_batch_size_ * 64), "CropMirrorNormalize");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~CropMirrorNormalizeGPU() override { dalib200CmnPlanDestroy(plan_); }

 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "CropMirrorNormalize: the GPU path expects uint8 input");
    const int n = in.num_samples();
    frames_ = ExpandFrames(in.shape(), in.GetLayout(), "CropMirrorNormalize");
    const bool seq = frames_.first_spatial == 1;
    std::string ol = out_layout_.empty() ? (seq ? "FHWC" : "HWC") : out_layout_;
    if (seq && (ol == "CHW" || ol == "HWC")) ol = "F" + ol;       // fn.crop_mirror_normalize(output_layout="CHW") on FHWC -> FCHW
    DALI_ENFORCE(ol == (seq ? "FCHW" : "CHW") || ol == (seq ? "FHWC" : "HWC"),
                 "The requested output layout is not supported by the GPU path (", ol, ")");
    chw_ = ol.find("CHW") != std::string::npos;
    resolved_layout_ = ol;
    const int nf = frames_.num_frames();
    if (nf > plan_cap_) { dalib200CmnPlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200CmnPlanCreate(&plan_, nf), "CropMirrorNormalize"); }
    samples_.assign(nf, dalib200CmnSample());
    crop_hw_.assign(n, {0, 0});
    int out_c = 0, fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      const int64_t H = s[fs], W = s[fs + 1], C = s[fs + 2];
      DALI_ENFORCE(C >= 1 && C <= 4, "CropMirrorNormalize: 1..4 channels supported, got ", C);
      // ---- crop window (crop_attr.cc:100-239)
      int64_t ch = H, cw = W;
      float px = 0.5f, py = 0.5f;
      bool has_h = false, has_w = false;
      if (spec_.ArgumentDefined("crop")) {
        auto c = spec_.GetFloatVecArgument("crop", &ws, i);
        DALI_ENFORCE(c.size() == 2, "`crop` argument should have 2 or 3 elements depending on the input data shape");
        ch = static_cast<int>(c[0]); cw = static_cast<int>(c[1]); has_h = has_w = true;
      } else if (spec_.ArgumentDefined("crop_h")) {
        ch = static_cast<int>(spec_.GetArgument<float>("crop_h", &ws, i)); cw = static_cast<int>(spec_.GetArgument<float>("crop_w", &ws, i));
        has_h = has_w = true;
      }
      if (!(has_h && ch > 0)) { ch = H; } else { py = spec_.GetArgument<float>("crop_pos_y", &ws, i); }
      if (!(has_w && cw > 0)) { cw = W; } else { px = spec_.GetArgument<float>("crop_pos_x", &ws, i); }
      DALI_ENFORCE(px >= 0.0f && px <= 1.0f && py >= 0.0f && py <= 1.0f, "Anchor for dimension is out of range [0.0, 1.0]");
      auto rnd = [&](double v) { return truncate_ ? static_cast<int64_t>(v) : static_cast<int64_t>(std::round(v)); };
      int64_t ay = rnd(static_cast<double>(py) * (H - ch)), ax = rnd(static_cast<double>(px) * (W - cw));
      // ---- out of bounds policy (generic/slice/out_of_bounds_policy.h)
      const bool oob = ay < 0 || ax < 0 || ay + ch > H || ax + cw > W;
      if (oob) {
        if (oob_ == "error") {
          DALI_FAIL(make_string("Slice can't be placed out of bounds with current policy. Got: input_shape={", H, ", ", W, ", ", C,
                                "}, slice_anchor={", ay, ", ", ax, ", 0}, slice_shape={", ch, ", ", cw, ", ", C, "}"));
        } else if (oob_ == "trim_to_shape") {
          const int64_t y0 = std::min(std::max<int64_t>(ay, 0), H), x0 = std::min(std::max<int64_t>(ax, 0), W);
          const int64_t y1 = std::min(std::max<int64_t>(ay + ch, 0), H), x1 = std::min(std::max<int64_t>(ax + cw, 0), W);
          ay = y0; ax = x0; ch = y1 - y0; cw = x1 - x0;
        }
      }
      // ---- normalisation args (crop_mirror_normalize.h:120-149)
      auto mean_arg = spec_.GetFloatVecArgument("mean", &ws, i), std_arg = spec_.GetFloatVecArgument("std", &ws, i);
      DALI_ENFORCE(mean_arg.size() == std_arg.size() || mean_arg.size() == 1 || std_arg.size() == 1,
                   "``mean`` and ``std`` must either be of the same size, be scalars, or one of them can be a vector and the other a scalar.");
      const int nargs = static_cast<int>(std::max(mean_arg.size(), std_arg.size()));
      DALI_ENFORCE(nargs == 1 || nargs == C, "The number of per-channel arguments should match the number of channels");
      int oc = static_cast<int>(C);
      if (pad_output_) { oc = 1; while (oc < C) oc *= 2; }          // next power of two (crop_mirror_normalize.h:69-77)
      out_c = oc;
      const bool mirror = spec_.GetArgument<int>("mirror", &ws, i) != 0;
      const int64_t frames = fs ? s[0] : 1;
      for (int64_t k = 0; k < frames; k++, fk++) {
        auto &c = samples_[fk];
        c.in_h = static_cast<int>(H); c.in_w = static_cast<int>(W); c.channels = static_cast<int>(C);
        c.anchor_y = static_cast<int>(ay); c.anchor_x = static_cast<int>(ax); c.crop_h = static_cast<int>(ch); c.crop_w = static_cast<int>(cw);
        c.mirror = mirror;
        for (int d = 0; d < 4; d++) {
          if (d < C) {
            const double mean_val = mean_arg[d % mean_arg.size()], std_val = std_arg[d % std_arg.size()];
            c.mean[d] = static_cast<float>(std::fma(-static_cast<double>(shift_), std_val / scale_, mean_val));
            c.inv_std[d] = static_cast<float>(scale_ / std_val);
          } else { c.mean[d] = 0.0f; c.inv_std[d] = 1.0f; }
          c.fill[d] = fill_values_.empty() ? 0.0f : fill_values_.size() == 1 ? fill_values_[0] : (d < static_cast<int>(fill_values_.size()) ? fill_values_[d] : 0.0f);
        }
      }
      crop_hw_[i] = { static_cast<int>(ch), static_cast<int>(cw) };
    }
    if (n > 0) {
      for (int i = 0; i < n; i++) {
        int oc = static_cast<int>(in.shape().tensor_shape_span(i)[frames_.first_spatial + 2]);
        if (pad_output_) { int p2 = 1; while (p2 < oc) p2 *= 2; oc = p2; }
        DALI_ENFORCE(oc == out_c, "CropMirrorNormalize: all samples of a batch must have the same number of channels");
      }
    }
    out_c_ = out_c;
    CheckStatus(dalib200CmnPlanSetup(plan_, nf, samples_.data(), out_type_ == DALI_FLOAT ? DALIB200_FLOAT : DALIB200_FLOAT16,
                                     chw_ ? DALIB200_LAYOUT_CHW : DALIB200_LAYOUT_HWC, std::max(out_c, 1)), "CropMirrorNormalize");
    out.resize(1);
    out[0].type = out_type_;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh;
      if (seq) sh.push_back(in.shape().tensor_shape_span(i)[0]);
      if (chw_) { sh.push_back(out_c); sh.push_back(crop_hw_[i].first); sh.push_back(crop_hw_[i].second); }
      else { sh.push_back(crop_hw_[i].first); sh.push_back(crop_hw_[i].second); sh.push_back(out_c); }
      out[0].shape.set_tensor_shape(i, sh);
    }
    return true;
  }

  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(resolved_layout_);
    auto ip = FramePtrs(in, frames_, 1);
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(crop_hw_[s].first) * crop_hw_[s].second * out_c_ * TypeSize(out_type_);
    }
    CheckStatus(dalib200CmnLaunch(plan_, ip.data(), op.data(), ws.stream()), "CropMirrorNormalize");
  }

 private:
  dalib200CmnPlan *plan_ = nullptr;
  int plan_cap_ = 0, out_c_ = 3;
  DALIDataType out_type_ = DALI_FLOAT;
  std::string out_layout_, oob_, resolved_layout_;
  bool pad_output_ = false, truncate_ = false, chw_ = true;
  float scale_ = 1, shift_ = 0;
  std::vector<float> fill_values_;
  FrameList frames_;
  std::vector<dalib200CmnSample> samples_;
  std::vector<std::pair<int, int>> crop_hw_;
};
DALI_REGISTER_OPERATOR(CropMirrorNormalize, CropMirrorNormalizeGPU, GPU);

// =============================================================================================== WarpAffine
DALI_SCHEMA(WarpAffine)
    .DocStr("Applies an affine transformation to images.")
    .NumInput(1, 2).NumOutput(1).AllowSequences()
    .AddOptionalArgNoDefault("matrix", "2x3 transform matrix (row-major).", true)
    .AddOptionalArg("inverse_map", "True: the matrix maps destination to source coordinates.", true)
    .AddOptionalArgNoDefault("size", "Output size (H, W); default: input size.", true)
    .AddOptionalArgNoDefault("fill_value", "Value used outside the source image; absent = clamp to border.")
    .AddOptionalArgNoDefault("dtype", "Output type (same as input or FLOAT).")
    .AddOptionalArg("interp_type", "NN or LINEAR.", DALI_INTERP_LINEAR);

class WarpAffineGPU : public Operator<GPUBackend> {
 public:
  explicit WarpAffineGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    DALI_ENFORCE(spec.NumInput() == 1, "WarpAffine: passing the matrices as a second regular input is not supported; use the `matrix` argument");
    const int it = spec.GetArgument<int>("interp_type");
    DALI_ENFORCE(it == DALI_INTERP_NN || it == DALI_INTERP_LINEAR, "Unsupported interpolation type");   // warp_cpu.h:84-87
    interp_ = it == DALI_INTERP_LINEAR;
    invert_ = !spec.GetArgument<bool>("inverse_map");
    use_fill_ = spec.ArgumentDefined("fill_value");
    if (use_fill_) fill_ = spec.GetArgument<float>("fill_value");
    CheckStatus(dalib200WarpPlanCreate(&plan_, max_batch_size_ * 64), "WarpAffine");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~WarpAffineGPU() override { dalib200WarpPlanDestroy(plan_); }

 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "WarpAffine: the GPU path expects uint8 input");
    out_type_ = spec_.ArgumentDefined("dtype") ? spec_.GetArgument<DALIDataType>("dtype") : DALI_UINT8;
    DALI_ENFORCE(out_type_ == DALI_UINT8 || out_type_ == DALI_FLOAT, "WarpAffine: output type must be UINT8 or FLOAT");
    DALI_ENFORCE(spec_.ArgumentDefined("matrix"), "`matrix` argument must be provided when transforms are not passed as a regular input.");
    const int n = in.num_samples();
    frames_ = ExpandFrames(in.shape(), in.GetLayout(), "WarpAffine");
    const int nf = frames_.num_frames();
    if (nf > plan_cap_) { dalib200WarpPlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200WarpPlanCreate(&plan_, nf), "WarpAffine"); }
    samples_.assign(nf, dalib200WarpSample());
    out_hw_.assign(n, {0, 0});
    int fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      auto m = spec_.GetFloatVecArgument("matrix", &ws, i);
      DALI_ENFORCE(m.size() == 6, "`matrix` parameter must have 6 elements");
      float M[6];
      if (invert_) dalib200AffineInverse(m.data(), M); else std::copy(m.begin(), m.end(), M);
      int oh = static_cast<int>(s[fs]), ow = static_cast<int>(s[fs + 1]);
      if (spec_.ArgumentDefined("size")) {
        auto sz = spec_.GetFloatVecArgument("size", &ws, i);
        DALI_ENFORCE(sz.size() == 2, "output_size must specify same number of dimensions as the input (excluding channels)");
        DALI_ENFORCE(sz[0] > 0 && sz[1] > 0, "Output size must be positive");
        oh = std::max<int>(static_cast<int>(std::roundf(sz[0])), 1); ow = std::max<int>(static_cast<int>(std::roundf(sz[1])), 1);
      }
      out_hw_[i] = { oh, ow };
      const int64_t frames = fs ? s[0] : 1;
      for (int64_t k = 0; k < frames; k++, fk++) {
        auto &w = samples_[fk];
        w.in_h = static_cast<int>(s[fs]); w.in_w = static_cast<int>(s[fs + 1]); w.channels = static_cast<int>(s[fs + 2]);
        w.out_h = oh; w.out_w = ow;
        std::copy(M, M + 6, w.matrix);
      }
    }
    CheckStatus(dalib200WarpPlanSetup(plan_, nf, samples_.data(), interp_, use_fill_, fill_, out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT),
                "WarpAffine");
    out.resize(1);
    out[0].type = out_type_;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      sh[frames_.first_spatial] = out_hw_[i].first; sh[frames_.first_spatial + 1] = out_hw_[i].second;
      out[0].shape.set_tensor_shape(i, sh);
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout().empty() ? TensorLayout(frames_.first_spatial ? "FHWC" : "HWC") : in.GetLayout());
    auto ip = FramePtrs(in, frames_, 1);
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(out_hw_[s].first) * out_hw_[s].second * frames_.c[k] * TypeSize(out_type_);
    }
    CheckStatus(dalib200WarpLaunch(plan_, ip.data(), op.data(), ws.stream()), "WarpAffine");
  }
 private:
  dalib200WarpPlan *plan_ = nullptr;
  int plan_cap_ = 0;
  bool interp_ = true, invert_ = false, use_fill_ = false;
  float fill_ = 0;
  DALIDataType out_type_ = DALI_UINT8;
  FrameList frames_;
  std::vector<dalib200WarpSample> samples_;
  std::vector<std::pair<int, int>> out_hw_;
};
DALI_REGISTER_OPERATOR(WarpAffine, WarpAffineGPU, GPU);

// =============================================================================================== Hsv
DALI_SCHEMA(Hsv)
    .DocStr("Adjusts hue, saturation and value (brightness) of the images.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("hue", "Hue delta, in degrees.", 0.0f, true)
    .AddOptionalArg("saturation", "Saturation multiplier.", 1.0f, true)
    .AddOptionalArg("value", "Value multiplier.", 1.0f, true)
    .AddOptionalArg("dtype", "Output data type.", DALI_UINT8);

class PointwiseBase : public Operator<GPUBackend> {
 public:
  explicit PointwiseBase(const OpSpec &spec, const char *name) : Operator<GPUBackend>(spec), name_(name) {
    CheckStatus(dalib200PointwisePlanCreate(&plan_, max_batch_size_), name_);
    plan_cap_ = max_batch_size_;
  }
  ~PointwiseBase() override { dalib200PointwisePlanDestroy(plan_); }
 protected:
  void EnsureCap(int n) {
    if (n > plan_cap_) { dalib200PointwisePlanDestroy(plan_); plan_ = nullptr; plan_cap_ = n; CheckStatus(dalib200PointwisePlanCreate(&plan_, n), name_); }
  }
  void Launch(Workspace &ws) {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout());
    std::vector<const void *> ip(in.num_samples());
    std::vector<void *> op(in.num_samples());
    for (int i = 0; i < in.num_samples(); i++) { ip[i] = in.raw_tensor(i); op[i] = out.raw_mutable_tensor(i); }
    CheckStatus(dalib200PointwiseLaunch(plan_, ip.data(), op.data(), ws.stream()), name_);
  }
  dalib200PointwisePlan *plan_ = nullptr;
  int plan_cap_ = 0;
  const char *name_;
};

class HsvGPU : public PointwiseBase {
 public:
  explicit HsvGPU(const OpSpec &spec) : PointwiseBase(spec, "Hsv") {
    out_type_ = spec.GetArgument<DALIDataType>("dtype");
    DALI_ENFORCE(out_type_ == DALI_UINT8 || out_type_ == DALI_FLOAT, "Hsv: the GPU path supports dtype UINT8 and FLOAT");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "Hsv: the GPU path expects uint8 input");
    const int n = in.num_samples();
    EnsureCap(n);
    std::vector<dalib200ColorSample> cs(n);
    for (int i = 0; i < n; i++) {
      const int nd = in.shape().sample_dim();
      DALI_ENFORCE(in.shape().tensor_shape_span(i)[nd - 1] == 3, "Hsv expects 3-channel (channel-last) images");
      cs[i].num_pixels = in.shape().tensor_size(i) / 3;
      // half_range = 128 for integer inputs (color_twist.h:141-146)
      dalib200ColorTwistMatrix(spec_.GetArgument<float>("hue", &ws, i), spec_.GetArgument<float>("saturation", &ws, i),
                               spec_.GetArgument<float>("value", &ws, i), 1.0f, 1.0f, 128.0f, cs[i].matrix, cs[i].offset);
    }
    CheckStatus(dalib200LinearTransformSetup(plan_, n, cs.data(), out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "Hsv");
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = out_type_;
    return true;
  }
  void RunImpl(Workspace &ws) override { Launch(ws); }
 private:
  DALIDataType out_type_ = DALI_UINT8;
};
DALI_REGISTER_OPERATOR(Hsv, HsvGPU, GPU);

// =============================================================================================== ColorSpaceConversion
DALI_SCHEMA(ColorSpaceConversion)
    .DocStr("Converts between various image color models.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddArg("image_type", "The color space of the input image.")
    .AddArg("output_type", "The color space of the output image.");

class ColorSpaceConversionGPU : public PointwiseBase {
 public:
  explicit ColorSpaceConversionGPU(const OpSpec &spec) : PointwiseBase(spec, "ColorSpaceConversion") {
    in_t_ = spec.GetArgument<int>("image_type"); out_t_ = spec.GetArgument<int>("output_type");
    DALI_ENFORCE(in_t_ >= 0 && in_t_ <= 3 && out_t_ >= 0 && out_t_ <= 3, "ColorSpaceConversion: unsupported image type");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "Color space conversion accept only uint8 tensors");    // color_space_conversion.h:49
    const int n = in.num_samples(), nd = in.shape().sample_dim();
    EnsureCap(n);
    const int ic = in_t_ == DALI_GRAY ? 1 : 3, oc = out_t_ == DALI_GRAY ? 1 : 3;
    std::vector<int64_t> npx(n);
    out.resize(1);
    out[0].type = DALI_UINT8;
    out[0].shape.resize(n, nd);
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      DALI_ENFORCE(sh[nd - 1] == ic, "Incorrect number of channels: expected ", ic, ", got ", sh[nd - 1]);
      npx[i] = in.shape().tensor_size(i) / ic;
      sh[nd - 1] = oc;
      out[0].shape.set_tensor_shape(i, sh);
    }
    CheckStatus(dalib200ColorSpaceSetup(plan_, n, npx.data(), in_t_, out_t_), "ColorSpaceConversion");
    return true;
  }
  void RunImpl(Workspace &ws) override { Launch(ws); }
 private:
  int in_t_ = 0, out_t_ = 0;
};
DALI_REGISTER_OPERATOR(ColorSpaceConversion, ColorSpaceConversionGPU, GPU);

// =============================================================================================== Spectrogram
DALI_SCHEMA(Spectrogram)
    .DocStr("Produces a spectrogram from a 1D signal.")
    .NumInput(1).NumOutput(1)
    .AddOptionalArgNoDefault("nfft", "Size of the FFT (default: window_length).")
    .AddOptionalArg("window_length", "Window size in number of samples.", 512)
    .AddOptionalArg("window_step", "Step between the STFT windows in number of samples.", 256)
    .AddOptionalArgNoDefault("window_fn", "Samples of the window function (default: Hann).")
    .AddOptionalArg("power", "Exponent of the magnitude of the spectrum (1 or 2).", 2)
    .AddOptionalArg("center_windows", "Pad the signal so that windows are centred.", true)
    .AddOptionalArg("reflect_padding", "Reflect (True) or zero (False) padding.", true)
    .AddOptionalArg("layout", "Output layout: \"ft\" or \"tf\".", std::string("ft"));

class SpectrogramGPU : public Operator<GPUBackend>, public SpectrumProducer {
 public:
  // ---- SpectrumProducer
  void EnableDeferredRun() override { fuse_ = true; }
  bool Deferred() const override { return deferred_now_; }
  void *SpectrogramPlan() override { return plan_; }
  const std::vector<const void *> &DeferredInputs() const override { return deferred_in_; }

  explicit SpectrogramGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    args_.window_length = spec.GetArgument<int>("window_length");
    args_.window_step = spec.GetArgument<int>("window_step");
    args_.power = spec.GetArgument<int>("power");
    DALI_ENFORCE(args_.window_length > 0, "Invalid window length: ", args_.window_length);
    DALI_ENFORCE(args_.window_step > 0, "Invalid window step: ", args_.window_step);
    DALI_ENFORCE(args_.power == 1 || args_.power == 2, "Power argument should be either `2` for energy or `1` for complex magnitude.");
    args_.nfft = spec.ArgumentDefined("nfft") ? spec.GetArgument<int>("nfft") : args_.window_length;
    args_.center = spec.GetArgument<bool>("center_windows"); args_.reflect = spec.GetArgument<bool>("reflect_padding");
    layout_ = spec.GetArgument<std::string>("layout");
    DALI_ENFORCE(layout_ == "ft" || layout_ == "tf", "Unexpected layout: ", layout_);
    args_.layout_ft = layout_ == "ft";
    if (spec.ArgumentDefined("window_fn")) {
      window_ = spec.GetRepeatedArgument<float>("window_fn");
      DALI_ENFORCE(static_cast<int>(window_.size()) == args_.window_length, "Window function should match the specified `window_length`");
    }
    CheckStatus(dalib200SpectrogramPlanCreate(&plan_, max_batch_size_), "Spectrogram");
  }
  ~SpectrogramGPU() override { dalib200SpectrogramPlanDestroy(plan_); }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "Spectrogram: the GPU path expects float input");
    const int n = in.num_samples();
    std::vector<int64_t> lens(n);
    for (int i = 0; i < n; i++) {
      const int64_t vol = in.shape().tensor_size(i);
      const int64_t *s = in.shape().tensor_shape_span(i);
      for (int d = 0; d < in.shape().sample_dim(); d++)
        DALI_ENFORCE(s[d] == 1 || s[d] == vol, "Input data must be 1D or all but one dimensions must be degenerate (extent 1).");
      lens[i] = vol;
    }
    CheckStatus(dalib200SpectrogramPlanSetup(plan_, &args_, window_.empty() ? nullptr : window_.data(), n, lens.data()), "Spectrogram");
    out.resize(1);
    out[0].type = DALI_FLOAT;
    out[0].shape.resize(n, 2);
    const int nbin = args_.nfft / 2 + 1;
    for (int i = 0; i < n; i++) {
      const int64_t nw = dalib200SpectrogramNumWindows(plan_, i);
      out[0].shape.set_tensor_shape(i, args_.layout_ft ? TensorShape{nbin, nw} : TensorShape{nw, nbin});
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(layout_);
    std::vector<const void *> ip(in.num_samples());
    std::vector<void *> op(in.num_samples());
    for (int i = 0; i < in.num_samples(); i++) { ip[i] = in.raw_tensor(i); op[i] = out.raw_mutable_tensor(i); }
    // fused with the MelFilterBank that consumes this output: it launches STFT -> mel as one kernel and the spectrogram is never
    // written (the fused kernel exists for nfft = 1024, (f, t) layout)
    deferred_now_ = fuse_ && args_.nfft == 1024 && args_.layout_ft;
    if (deferred_now_) { deferred_in_ = ip; return; }
    CheckStatus(dalib200SpectrogramLaunch(plan_, ip.data(), op.data(), ws.stream()), "Spectrogram");
  }
 private:
  bool fuse_ = false, deferred_now_ = false;
  std::vector<const void *> deferred_in_;
  dalib200SpectrogramPlan *plan_ = nullptr;
  dalib200SpectrogramArgs args_{};
  std::vector<float> window_;
  std::string layout_;
};
DALI_REGISTER_OPERATOR(Spectrogram, SpectrogramGPU, GPU);

// =============================================================================================== MelFilterBank
DALI_SCHEMA(MelFilterBank)
    .DocStr("Converts a spectrogram to a mel spectrogram by applying a bank of triangular filters.")
    .NumInput(1).NumOutput(1)
    .AddOptionalArg("nfilter", "Number of mel filters.", 128)
    .AddOptionalArg("sample_rate", "Sampling rate of the audio signal.", 44100.0f)
    .AddOptionalArg("freq_low", "The minimum frequency.", 0.0f)
    .AddOptionalArg("freq_high", "The maximum frequency (0 = sample_rate / 2).", 0.0f)
    .AddOptionalArg("normalize", "Normalise the triangular filter weights by the width of their bands.", true)
    .AddOptionalArg("mel_formula", "slaney | htk", std::string("slaney"));

class MelFilterBankGPU : public Operator<GPUBackend>, public SpectrumConsumer {
 public:
  void AttachProducer(SpectrumProducer *p) override { producer_ = p; }
  explicit MelFilterBankGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    args_.nfilter = spec.GetArgument<int>("nfilter");
    args_.sample_rate = spec.GetArgument<float>("sample_rate");
    args_.freq_low = spec.GetArgument<float>("freq_low"); args_.freq_high = spec.GetArgument<float>("freq_high");
    args_.normalize = spec.GetArgument<bool>("normalize");
    const std::string f = spec.GetArgument<std::string>("mel_formula");
    DALI_ENFORCE(f == "slaney" || f == "htk", "Unsupported mel_formula value \"", f, "\". Supported values are: \"slaney\", \"htk\"");
    args_.htk = f == "htk";
    CheckStatus(dalib200MelPlanCreate(&plan_, max_batch_size_), "MelFilterBank");
    // opt-in: the dense-GEMM tensor-core path (tolerance ~1e-6 instead of bit-exact banded sums)
    if (const char *e = getenv("DALIB200_MEL_TENSOR_CORES")) CheckStatus(dalib200MelPlanSetTensorCores(plan_, atoi(e)), "MelFilterBank");
  }
  ~MelFilterBankGPU() override { dalib200MelPlanDestroy(plan_); }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "MelFilterBank: the GPU path expects float input");
    DALI_ENFORCE(in.shape().sample_dim() == 2, "MelFilterBank: the GPU path expects 2-D (frequency, time) spectrograms");
    const std::string l = in.GetLayout().str();
    DALI_ENFORCE(l.empty() || l == "ft", "MelFilterBank: the GPU path expects the \"ft\" layout, got \"", l, "\"");
    const int n = in.num_samples();
    std::vector<int64_t> nwin(n);
    int nbin = n ? static_cast<int>(in.shape().tensor_shape_span(0)[0]) : 2;
    for (int i = 0; i < n; i++) {
      DALI_ENFORCE(in.shape().tensor_shape_span(i)[0] == nbin, "MelFilterBank: all spectrograms of a batch must have the same number of bins");
      nwin[i] = in.shape().tensor_shape_span(i)[1];
    }
    CheckStatus(dalib200MelPlanSetup(plan_, &args_, nbin, n, nwin.data()), "MelFilterBank");
    out.resize(1);
    out[0].type = DALI_FLOAT;
    out[0].shape.resize(n, 2);
    for (int i = 0; i < n; i++) out[0].shape.set_tensor_shape(i, { args_.nfilter, nwin[i] });
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout("ft");
    std::vector<const void *> ip(in.num_samples());
    std::vector<void *> op(in.num_samples());
    for (int i = 0; i < in.num_samples(); i++) { ip[i] = in.raw_tensor(i); op[i] = out.raw_mutable_tensor(i); }
    if (producer_ && producer_->Deferred()) {
      auto *sp = static_cast<dalib200SpectrogramPlan *>(producer_->SpectrogramPlan());
      const auto &sin = producer_->DeferredInputs();
      if (dalib200SpectrogramMelSupported(sp, plan_)) {
        CheckStatus(dalib200SpectrogramMelLaunch(sp, plan_, sin.data(), nullptr, op.data(), ws.stream()), "MelFilterBank");
        return;
      }
      // not fusable after all (e.g. the tensor-core mel path was requested): materialise the spectrogram, then filter it
      std::vector<void *> sp_out(in.num_samples());
      for (int i = 0; i < in.num_samples(); i++) sp_out[i] = const_cast<void *>(in.raw_tensor(i));
      CheckStatus(dalib200SpectrogramLaunch(sp, sin.data(), sp_out.data(), ws.stream()), "Spectrogram");
    }
    CheckStatus(dalib200MelLaunch(plan_, ip.data(), op.data(), ws.stream()), "MelFilterBank");
  }
 private:
  SpectrumProducer *producer_ = nullptr;
  dalib200MelPlan *plan_ = nullptr;
  dalib200MelArgs args_{};
};
DALI_REGISTER_OPERATOR(MelFilterBank, MelFilterBankGPU, GPU);

// =============================================================================================== BrightnessContrast / ColorTwist
DALI_SCHEMA(BrightnessContrast)
    .DocStr("Adjusts the brightness and contrast of the images: out = brightness_shift * range + brightness * (center + contrast * (in - center)).")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("brightness", "Brightness multiplier.", 1.0f, true)
    .AddOptionalArg("brightness_shift", "The brightness shift (in units of the full range of the output type).", 0.0f, true)
    .AddOptionalArg("contrast", "The contrast multiplier.", 1.0f, true)
    .AddOptionalArgNoDefault("contrast_center", "The intensity level that is unaffected by contrast (default: half the input range).", true)
    .AddOptionalArgNoDefault("dtype", "Output data type (default: the input type).");

class GenericOpBase : public Operator<GPUBackend> {
 public:
  explicit GenericOpBase(const OpSpec &spec, const char *name) : Operator<GPUBackend>(spec), name_(name) {
    CheckStatus(dalib200GenericPlanCreate(&plan_, max_batch_size_ * 64), name_);
    plan_cap_ = max_batch_size_ * 64;
  }
  ~GenericOpBase() override { dalib200GenericPlanDestroy(plan_); }
 protected:
  void EnsureCap(int n) {
    if (n > plan_cap_) { dalib200GenericPlanDestroy(plan_); plan_ = nullptr; plan_cap_ = n; CheckStatus(dalib200GenericPlanCreate(&plan_, n), name_); }
  }
  dalib200GenericPlan *plan_ = nullptr;
  int plan_cap_ = 0;
  const char *name_;
};

class BrightnessContrastGPU : public GenericOpBase {
 public:
  explicit BrightnessContrastGPU(const OpSpec &spec) : GenericOpBase(spec, "BrightnessContrast") {}
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "BrightnessContrast: the GPU path expects uint8 input");
    out_type_ = spec_.ArgumentDefined("dtype") ? spec_.GetArgument<DALIDataType>("dtype") : DALI_UINT8;
    DALI_ENFORCE(out_type_ == DALI_UINT8 || out_type_ == DALI_FLOAT, "BrightnessContrast: the GPU path supports dtype UINT8 and FLOAT");
    const int n = in.num_samples();
    EnsureCap(n);
    std::vector<int64_t> vol(n);
    std::vector<float> mul(n), add(n);
    // brightness_contrast.h:84-103: FullRange<Out> = 255 (u8) or 1 (float); HalfRange<uint8_t> = 128
    const float range = out_type_ == DALI_UINT8 ? 255.0f : 1.0f;
    for (int i = 0; i < n; i++) {
      vol[i] = in.shape().tensor_size(i);
      const float brightness = spec_.GetArgument<float>("brightness", &ws, i), shift = spec_.GetArgument<float>("brightness_shift", &ws, i);
      const float contrast = spec_.GetArgument<float>("contrast", &ws, i);
      const float center = spec_.ArgumentDefined("contrast_center") ? spec_.GetArgument<float>("contrast_center", &ws, i) : 128.0f;
      volatile float t0 = contrast * center;            // every product / sum rounded to float, in the reference's order
      volatile float t1 = center - t0;
      volatile float t2 = brightness * t1;
      volatile float t3 = shift * range;
      add[i] = t3 + t2;
      mul[i] = brightness * contrast;
    }
    CheckStatus(dalib200MultiplyAddSetup(plan_, n, vol.data(), mul.data(), add.data(), out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), name_);
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = out_type_;
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout());
    std::vector<const void *> ip(in.num_samples());
    std::vector<void *> op(in.num_samples());
    for (int i = 0; i < in.num_samples(); i++) { ip[i] = in.raw_tensor(i); op[i] = out.raw_mutable_tensor(i); }
    CheckStatus(dalib200GenericLaunch(plan_, ip.data(), op.data(), ws.stream()), name_);
  }
  DALIDataType out_type_ = DALI_UINT8;
};
DALI_REGISTER_OPERATOR(BrightnessContrast, BrightnessContrastGPU, GPU);

DALI_SCHEMA(ColorTwist)
    .DocStr("Adjusts hue, saturation, brightness and contrast of the image.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("hue", "Hue change, in degrees.", 0.0f, true)
    .AddOptionalArg("saturation", "Saturation change factor.", 1.0f, true)
    .AddOptionalArg("contrast", "Contrast change factor.", 1.0f, true)
    .AddOptionalArg("brightness", "Brightness change factor.", 1.0f, true)
    .AddOptionalArg("image_type", "The color space of the input and the output image.", DALI_RGB)
    .AddOptionalArgNoDefault("dtype", "Output data type (default: the input type).");

class ColorTwistGPU : public PointwiseBase {
 public:
  explicit ColorTwistGPU(const OpSpec &spec) : PointwiseBase(spec, "ColorTwist") {
    out_type_ = spec.ArgumentDefined("dtype") ? spec.GetArgument<DALIDataType>("dtype") : DALI_UINT8;
    DALI_ENFORCE(out_type_ == DALI_UINT8 || out_type_ == DALI_FLOAT, "ColorTwist: the GPU path supports dtype UINT8 and FLOAT");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "ColorTwist: the GPU path expects uint8 input");
    const int n = in.num_samples();
    EnsureCap(n);
    std::vector<dalib200ColorSample> cs(n);
    for (int i = 0; i < n; i++) {
      const int nd = in.shape().sample_dim();
      DALI_ENFORCE(in.shape().tensor_shape_span(i)[nd - 1] == 3, "ColorTwist expects 3-channel (channel-last) images");
      cs[i].num_pixels = in.shape().tensor_size(i) / 3;
      // color_twist.h:156-170: value = 1; half_range = 128 for integer inputs
      dalib200ColorTwistMatrix(spec_.GetArgument<float>("hue", &ws, i), spec_.GetArgument<float>("saturation", &ws, i), 1.0f,
                               spec_.GetArgument<float>("brightness", &ws, i), spec_.GetArgument<float>("contrast", &ws, i), 128.0f,
                               cs[i].matrix, cs[i].offset);
    }
    CheckStatus(dalib200LinearTransformSetup(plan_, n, cs.data(), out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "ColorTwist");
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = out_type_;
    return true;
  }
  void RunImpl(Workspace &ws) override { Launch(ws); }
 private:
  DALIDataType out_type_ = DALI_UINT8;
};
DALI_REGISTER_OPERATOR(ColorTwist, ColorTwistGPU, GPU);

// =============================================================================================== Flip / Crop / Slice
// Window copies of interleaved u8 images (dali/operators/generic/flip.{h,cc}, image/crop/crop.{h,cc}, generic/slice/slice.{h,cc}).
class WindowOpBase : public GenericOpBase {
 public:
  explicit WindowOpBase(const OpSpec &spec, const char *name) : GenericOpBase(spec, name) {}
 protected:
  // fills w (anchor / out size / flips / fill) for frame-independent sample i of size H x W x C
  virtual void SampleWindow(dalib200WindowSample &w, const Workspace &ws, int i, int H, int W, int C) = 0;
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, name_, ": the GPU path expects uint8 input");
    const int n = in.num_samples();
    frames_ = ExpandFrames(in.shape(), in.GetLayout(), name_);
    const int nf = frames_.num_frames();
    EnsureCap(nf);
    samples_.assign(nf, dalib200WindowSample());
    out_hw_.assign(n, {0, 0});
    int fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      dalib200WindowSample w{};
      w.in_h = static_cast<int>(s[fs]); w.in_w = static_cast<int>(s[fs + 1]); w.channels = static_cast<int>(s[fs + 2]);
      DALI_ENFORCE(w.channels >= 1, name_, ": empty channel dimension");
      SampleWindow(w, ws, i, w.in_h, w.in_w, w.channels);
      out_hw_[i] = { w.out_h, w.out_w };
      const int64_t frames = fs ? s[0] : 1;
      for (int64_t k = 0; k < frames; k++) samples_[fk++] = w;
    }
    CheckStatus(dalib200WindowCopySetup(plan_, nf, samples_.data()), name_);
    out.resize(1);
    out[0].type = DALI_UINT8;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      sh[frames_.first_spatial] = out_hw_[i].first; sh[frames_.first_spatial + 1] = out_hw_[i].second;
      out[0].shape.set_tensor_shape(i, sh);
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout().empty() ? TensorLayout(frames_.first_spatial ? "FHWC" : "HWC") : in.GetLayout());
    auto ip = FramePtrs(in, frames_, 1);
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(out_hw_[s].first) * out_hw_[s].second * frames_.c[k];
    }
    CheckStatus(dalib200GenericLaunch(plan_, ip.data(), op.data(), ws.stream()), name_);
  }
  // out_of_bounds_policy handling shared by crop and slice (generic/slice/out_of_bounds_policy.h)
  void ApplyOob(dalib200WindowSample &w, const std::string &policy, const std::vector<float> &fill, int64_t ay, int64_t ax, int64_t h, int64_t wd) {
    const int64_t H = w.in_h, W = w.in_w;
    const bool oob = ay < 0 || ax < 0 || ay + h > H || ax + wd > W;
    if (oob) {
      if (policy == "error") {
        DALI_FAIL(make_string("Slice can't be placed out of bounds with current policy. Got: input_shape={", H, ", ", W, ", ", w.channels,
                              "}, slice_anchor={", ay, ", ", ax, ", 0}, slice_shape={", h, ", ", wd, ", ", w.channels, "}"));
      } else if (policy == "trim_to_shape") {
        const int64_t y0 = std::min(std::max<int64_t>(ay, 0), H), x0 = std::min(std::max<int64_t>(ax, 0), W);
        const int64_t y1 = std::min(std::max<int64_t>(ay + h, 0), H), x1 = std::min(std::max<int64_t>(ax + wd, 0), W);
        ay = y0; ax = x0; h = y1 - y0; wd = x1 - x0;
      }
    }
    w.anchor_y = static_cast<int>(ay); w.anchor_x = static_cast<int>(ax); w.out_h = static_cast<int>(h); w.out_w = static_cast<int>(wd);
    for (int k = 0; k < 4; k++) {
      const float f = fill.empty() ? 0.0f : fill.size() == 1 ? fill[0] : (k < static_cast<int>(fill.size()) ? fill[k] : 0.0f);
      w.fill[k] = static_cast<uint8_t>(std::min(255.0f, std::max(0.0f, std::round(f))));      // ConvertSat<uint8_t>
    }
  }
  FrameList frames_;
  std::vector<dalib200WindowSample> samples_;
  std::vector<std::pair<int, int>> out_hw_;
};

DALI_SCHEMA(Flip)
    .DocStr("Flips the images in selected dimensions (horizontal, vertical).")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("horizontal", "Flip the horizontal dimension.", 1, true)
    .AddOptionalArg("vertical", "Flip the vertical dimension.", 0, true)
    .AddOptionalArg("depthwise", "not supported (2-D images only)", 0, true);

class FlipGPU : public WindowOpBase {
 public:
  explicit FlipGPU(const OpSpec &spec) : WindowOpBase(spec, "Flip") {}
 protected:
  void SampleWindow(dalib200WindowSample &w, const Workspace &ws, int i, int H, int W, int) override {
    DALI_ENFORCE(spec_.GetArgument<int>("depthwise", &ws, i) == 0, "Flip: depthwise flips need volumetric data, which the GPU path does not support");
    w.anchor_y = w.anchor_x = 0; w.out_h = H; w.out_w = W;
    w.flip_x = spec_.GetArgument<int>("horizontal", &ws, i) != 0;
    w.flip_y = spec_.GetArgument<int>("vertical", &ws, i) != 0;
  }
};
DALI_REGISTER_OPERATOR(Flip, FlipGPU, GPU);

DALI_SCHEMA(Crop)
    .DocStr("Crops the images with the specified window dimensions and window position (upper left corner).")
    .NumInput(1).NumOutput(1).AllowSequences()
    DALIB200_CROP_ARGS()
    .AddOptionalArg("out_of_bounds_policy", "error | pad | trim_to_shape", std::string("error"))
    .AddOptionalArg("fill_values", "Fill values for padding.", std::vector<float>{0.0f})
    .AddOptionalArgNoDefault("dtype", "Output data type (UINT8 only on the GPU path).");

class CropGPU : public WindowOpBase {
 public:
  explicit CropGPU(const OpSpec &spec) : WindowOpBase(spec, "Crop") {
    crop_.Init(spec, name_);
    oob_ = spec.GetArgument<std::string>("out_of_bounds_policy");
    DALI_ENFORCE(oob_ == "error" || oob_ == "pad" || oob_ == "trim_to_shape", "Unsupported out_of_bounds_policy: ", oob_);
    fill_ = spec.GetRepeatedArgument<float>("fill_values");
    if (spec.ArgumentDefined("dtype")) DALI_ENFORCE(spec.GetArgument<DALIDataType>("dtype") == DALI_UINT8, "Crop: the GPU path keeps the uint8 input type");
  }
 protected:
  void SampleWindow(dalib200WindowSample &w, const Workspace &ws, int i, int H, int W, int) override {
    int64_t y0, x0, h, wd;
    crop_.Get(spec_, ws, i, H, W, y0, x0, h, wd);
    ApplyOob(w, oob_, fill_, y0, x0, h, wd);
  }
  CropWindowArgs crop_;
  std::string oob_;
  std::vector<float> fill_;
};
DALI_REGISTER_OPERATOR(Crop, CropGPU, GPU);

DALI_SCHEMA(Slice)
    .DocStr("Extracts a subtensor, or slice (H / W axes of interleaved images on the GPU path).")
    .NumInput(1, 3).NumOutput(1).AllowSequences()
    DALIB200_SLICE_ARGS()
    .AddOptionalArg("out_of_bounds_policy", "error | pad | trim_to_shape", std::string("error"))
    .AddOptionalArg("fill_values", "Fill values for padding.", std::vector<float>{0.0f})
    .AddOptionalArgNoDefault("dtype", "Output data type (UINT8 only on the GPU path).");

class SliceGPU : public WindowOpBase {
 public:
  explicit SliceGPU(const OpSpec &spec) : WindowOpBase(spec, "Slice") {
    slice_.Init(spec, name_);
    oob_ = spec.GetArgument<std::string>("out_of_bounds_policy");
    DALI_ENFORCE(oob_ == "error" || oob_ == "pad" || oob_ == "trim_to_shape", "Unsupported out_of_bounds_policy: ", oob_);
    fill_ = spec.GetRepeatedArgument<float>("fill_values");
  }
 protected:
  void SampleWindow(dalib200WindowSample &w, const Workspace &ws, int i, int H, int W, int) override {
    int64_t b[2], e[2];
    slice_.Get(spec_, ws, i, H, W, b, e);
    ApplyOob(w, oob_, fill_, b[0], b[1], e[0] - b[0], e[1] - b[1]);
  }
  SliceArgs slice_;
  std::string oob_;
  std::vector<float> fill_;
};
DALI_REGISTER_OPERATOR(Slice, SliceGPU, GPU);

// =============================================================================================== Rotate
// dali/operators/image/remap/rotate.cc + rotate_params.h: a WarpAffine whose matrix is
// translation(in / 2) * rotation2D(-a) * translation(-out / 2) with a = deg2rad(-angle) (counter-clockwise for a top-left origin)
// and whose canvas is the bounding box of the rotated image (parity kept, rotate_params.h:36-55,279-297) unless `size` / `keep_size`.
DALI_SCHEMA(Rotate)
    .DocStr("Rotates the images by the specified angle.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddArg("angle", "Angle, in degrees, by which the image is rotated (counter-clockwise).", true)
    .AddOptionalArg("keep_size", "If True, original canvas size is kept.", false)
    .AddOptionalArgNoDefault("axis", "3-D rotation axis: not supported (2-D images only).", true)
    .AddOptionalArgNoDefault("size", "Output size (H, W).", true)
    .AddOptionalArgNoDefault("fill_value", "Value used outside the source image; absent = clamp to border.")
    .AddOptionalArgNoDefault("dtype", "Output type (same as input or FLOAT).")
    .AddOptionalArg("interp_type", "NN or LINEAR.", DALI_INTERP_LINEAR);

namespace rotate_detail {
// geom/mat.h operator* for 3x3 floats: every element is a left-to-right sum of three separately rounded products
inline void Mul3(const float a[9], const float b[9], float r[9]) {
  float t[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      volatile float s = a[i * 3] * b[j];
      volatile float p = a[i * 3 + 1] * b[3 + j];
      s = s + p;
      p = a[i * 3 + 2] * b[6 + j];
      s = s + p;
      t[i * 3 + j] = s;
    }
  std::copy(t, t + 9, r);
}
inline void CanvasSize(int h, int w, double angle, int &h_out, int &w_out, int &par_w, int &par_h) {     // rotate_params.h:36-55
  const double eps = 1e-2;
  const double abs_cos = std::abs(std::cos(angle)), abs_sin = std::abs(std::sin(angle));
  w_out = static_cast<int>(std::ceil(abs_cos * w + abs_sin * h - eps));
  h_out = static_cast<int>(std::ceil(abs_cos * h + abs_sin * w - eps));
  if (abs_sin <= abs_cos) { par_w = w % 2; par_h = h % 2; } else { par_w = h % 2; par_h = w % 2; }
}
inline void Params(float angle_deg, int in_h, int in_w, bool keep_size, const float *size_hw, int &out_h, int &out_w, float M[6]) {
  const float d2r = M_PI / 180;
  const float neg = -angle_deg;                         // SetParams(): 2-D angles are negated
  volatile float a = neg * d2r;                         // deg2rad(float)
  if (size_hw) {                                        // warp_param_provider.h:234-314: explicit size, rounded
    out_h = std::max<int>(static_cast<int>(std::roundf(size_hw[0])), 1); out_w = std::max<int>(static_cast<int>(std::roundf(size_hw[1])), 1);
  } else if (keep_size) {
    out_h = in_h; out_w = in_w;
  } else {
    int pw, ph;
    CanvasSize(in_h, in_w, static_cast<double>(a), out_h, out_w, pw, ph);
    out_w += (out_w % 2) ^ (2 * pw > 1);                 // one frame: the majority vote is the frame's own parity
    out_h += (out_h % 2) ^ (2 * ph > 1);
  }
  const float ra = -a;
  const float c = std::cos(ra), sn = std::sin(ra);
  const float T1[9] = { 1, 0, in_w * 0.5f, 0, 1, in_h * 0.5f, 0, 0, 1 };
  const float R[9] = { c, -sn, 0, sn, c, 0, 0, 0, 1 };
  const float T2[9] = { 1, 0, -(out_w * 0.5f), 0, 1, -(out_h * 0.5f), 0, 0, 1 };
  float A[9], B[9];
  Mul3(T1, R, A);
  Mul3(A, T2, B);
  std::copy(B, B + 6, M);
}
}  // namespace rotate_detail

class RotateGPU : public Operator<GPUBackend> {
 public:
  explicit RotateGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    const int it = spec.GetArgument<int>("interp_type");
    DALI_ENFORCE(it == DALI_INTERP_NN || it == DALI_INTERP_LINEAR, "Unsupported interpolation type");
    interp_ = it == DALI_INTERP_LINEAR;
    keep_size_ = spec.GetArgument<bool>("keep_size");
    DALI_ENFORCE(!spec.ArgumentDefined("axis"), "Rotate: `axis` (3-D rotation) is not supported by the GPU path");
    use_fill_ = spec.ArgumentDefined("fill_value");
    if (use_fill_) fill_ = spec.GetArgument<float>("fill_value");
    CheckStatus(dalib200WarpPlanCreate(&plan_, max_batch_size_ * 64), "Rotate");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~RotateGPU() override { dalib200WarpPlanDestroy(plan_); }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8, "Rotate: the GPU path expects uint8 input");
    out_type_ = spec_.ArgumentDefined("dtype") ? spec_.GetArgument<DALIDataType>("dtype") : DALI_UINT8;
    DALI_ENFORCE(out_type_ == DALI_UINT8 || out_type_ == DALI_FLOAT, "Rotate: output type must be UINT8 or FLOAT");
    const int n = in.num_samples();
    frames_ = ExpandFrames(in.shape(), in.GetLayout(), "Rotate");
    const int nf = frames_.num_frames();
    if (nf > plan_cap_) { dalib200WarpPlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200WarpPlanCreate(&plan_, nf), "Rotate"); }
    samples_.assign(nf, dalib200WarpSample());
    out_hw_.assign(n, {0, 0});
    int fk = 0;
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const int fs = frames_.first_spatial;
      const int H = static_cast<int>(s[fs]), W = static_cast<int>(s[fs + 1]);
      const float angle = spec_.GetArgument<float>("angle", &ws, i);
      std::vector<float> sz;
      if (spec_.ArgumentDefined("size")) {
        sz = spec_.GetFloatVecArgument("size", &ws, i);
        DALI_ENFORCE(sz.size() == 2, "output_size must specify same number of dimensions as the input (excluding channels)");
        DALI_ENFORCE(sz[0] > 0 && sz[1] > 0, "Output size must be positive");
      }
      int oh, ow; float M[6];
      rotate_detail::Params(angle, H, W, keep_size_, sz.empty() ? nullptr : sz.data(), oh, ow, M);
      out_hw_[i] = { oh, ow };
      const int64_t frames = fs ? s[0] : 1;
      for (int64_t k = 0; k < frames; k++, fk++) {
        auto &w = samples_[fk];
        w.in_h = H; w.in_w = W; w.channels = static_cast<int>(s[fs + 2]);
        w.out_h = oh; w.out_w = ow;
        std::copy(M, M + 6, w.matrix);
      }
    }
    CheckStatus(dalib200WarpPlanSetup(plan_, nf, samples_.data(), interp_, use_fill_, fill_, out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "Rotate");
    out.resize(1);
    out[0].type = out_type_;
    out[0].shape.resize(n, in.shape().sample_dim());
    for (int i = 0; i < n; i++) {
      TensorShape sh = in.shape().tensor_shape(i);
      sh[frames_.first_spatial] = out_hw_[i].first; sh[frames_.first_spatial + 1] = out_hw_[i].second;
      out[0].shape.set_tensor_shape(i, sh);
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout().empty() ? TensorLayout(frames_.first_spatial ? "FHWC" : "HWC") : in.GetLayout());
    auto ip = FramePtrs(in, frames_, 1);
    std::vector<void *> op(frames_.num_frames());
    std::vector<int64_t> next(out.num_samples(), 0);
    for (int k = 0; k < frames_.num_frames(); k++) {
      const int s = frames_.sample_of_frame[k];
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(s)) + next[s];
      next[s] += static_cast<int64_t>(out_hw_[s].first) * out_hw_[s].second * frames_.c[k] * TypeSize(out_type_);
    }
    CheckStatus(dalib200WarpLaunch(plan_, ip.data(), op.data(), ws.stream()), "Rotate");
  }
 private:
  dalib200WarpPlan *plan_ = nullptr;
  int plan_cap_ = 0;
  bool interp_ = true, keep_size_ = false, use_fill_ = false;
  float fill_ = 0;
  DALIDataType out_type_ = DALI_UINT8;
  FrameList frames_;
  std::vector<dalib200WarpSample> samples_;
  std::vector<std::pair<int, int>> out_hw_;
};
DALI_REGISTER_OPERATOR(Rotate, RotateGPU, GPU);

// =============================================================================================== ToDecibels / MFCC / Normalize
class SignalOpBase : public Operator<GPUBackend> {
 public:
  explicit SignalOpBase(const OpSpec &spec, const char *name) : Operator<GPUBackend>(spec), name_(name) {
    CheckStatus(dalib200SignalPlanCreate(&plan_, max_batch_size_), name_);
  }
  ~SignalOpBase() override { dalib200SignalPlanDestroy(plan_); }
 protected:
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(in.GetLayout());
    std::vector<const void *> ip(in.num_samples());
    std::vector<void *> op(in.num_samples());
    for (int i = 0; i < in.num_samples(); i++) { ip[i] = in.raw_tensor(i); op[i] = out.raw_mutable_tensor(i); }
    CheckStatus(dalib200SignalLaunch(plan_, ip.data(), op.data(), ws.stream()), name_);
  }
  dalib200SignalPlan *plan_ = nullptr;
  const char *name_;
};

// dali/operators/audio/resample.{h,cc}: windowed-sinc resampling of [time] or [time, channels] float signals
DALI_SCHEMA(AudioResample)
    .DocStr("Resamples an audio signal (windowed sinc).")
    .NumInput(1).NumOutput(1)
    .AddOptionalArgNoDefault("in_rate", "Input sampling rate.", true)
    .AddOptionalArgNoDefault("out_rate", "Output sampling rate.", true)
    .AddOptionalArgNoDefault("scale", "The scaling factor (out_rate / in_rate).", true)
    .AddOptionalArgNoDefault("out_length", "The requested output length, in samples.", true)
    .AddOptionalArg("quality", "Resampling quality, 0 (lowest) .. 100 (highest); 50 = 16 lobes of the sinc.", 50.0f)
    .AddOptionalArgNoDefault("dtype", "Output type; the GPU path supports FLOAT.");

class AudioResampleGPU : public SignalOpBase {
 public:
  explicit AudioResampleGPU(const OpSpec &spec) : SignalOpBase(spec, "AudioResample") {
    has_rates_ = spec.ArgumentDefined("in_rate");
    DALI_ENFORCE(has_rates_ == spec.ArgumentDefined("out_rate"), "The parameters ``in_rate`` and ``out_rate`` must be specified together.");
    has_scale_ = spec.ArgumentDefined("scale"); has_len_ = spec.ArgumentDefined("out_length");
    DALI_ENFORCE(static_cast<int>(has_rates_) + has_scale_ + has_len_ <= 1, "The sampling rates, ``scale`` and ``out_length`` cannot be used together.");
    DALI_ENFORCE(has_rates_ || has_scale_ || has_len_, "No resampling factor specified! Please supply either the scale, the output length or "
                 "the input and output sampling rates.");
    quality_ = spec.GetArgument<float>("quality");
    DALI_ENFORCE(quality_ >= 0 && quality_ <= 100, "``quality`` out of range: ", quality_, "\nValid range is [0..100].");
    if (spec.ArgumentDefined("dtype"))
      DALI_ENFORCE(spec.GetArgument<int>("dtype") == DALI_FLOAT, "AudioResample: the GPU path produces FLOAT output only");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "AudioResample: the GPU path supports float input; got type ", static_cast<int>(in.type()));
    const int nd = in.shape().sample_dim();
    DALI_ENFORCE(nd == 1 || nd == 2, "Audio resampling supports only time series data, with an optional innermost channel dimension.");
    const int n = in.num_samples();
    std::vector<dalib200AudioResampleSample> s(n);
    out.resize(1);
    out[0].type = DALI_FLOAT;
    out[0].shape.resize(n, nd);
    for (int i = 0; i < n; i++) {
      const int64_t *sh = in.shape().tensor_shape_span(i);
      const int64_t in_len = sh[0];
      s[i].channels = nd == 2 ? static_cast<int>(sh[1]) : 1;
      s[i].in_length = in_len;
      if (has_rates_) {                                   // resample.h:73-101
        const double ir = spec_.GetArgument<float>("in_rate", &ws, i), orate = spec_.GetArgument<float>("out_rate", &ws, i);
        DALI_ENFORCE(ir > 0, "Input sampling rates must be positive. Got in_rate == ", ir);
        DALI_ENFORCE(orate > 0, "Output sampling rates must be positive on the GPU path. Got out_rate == ", orate);
        s[i].in_rate = ir; s[i].out_rate = orate;
        s[i].out_length = static_cast<int64_t>(std::ceil(in_len * orate / ir));
      } else if (has_scale_) {
        const double sc = spec_.GetArgument<float>("scale", &ws, i);
        DALI_ENFORCE(sc > 0, "The scaling factor must be positive on the GPU path. Got scale == ", sc);
        s[i].in_rate = 1.0; s[i].out_rate = sc;
        s[i].out_length = static_cast<int64_t>(std::ceil(in_len * sc / 1));
      } else {
        const int64_t ol = spec_.GetArgument<int64_t>("out_length", &ws, i);
        DALI_ENFORCE(!(in_len == 0 && ol != 0), "Cannot produce a non-empty signal from an empty input.\nError at sample ", i);
        s[i].in_rate = in_len ? static_cast<double>(in_len) : 1.0;
        s[i].out_rate = ol ? static_cast<double>(ol) : 1.0;
        s[i].out_length = ol;
      }
      if (nd == 2) out[0].shape.set_tensor_shape(i, { s[i].out_length, sh[1] });
      else out[0].shape.set_tensor_shape(i, { s[i].out_length });
    }
    CheckStatus(dalib200AudioResampleSetup(plan_, n, s.data(), quality_), name_);
    return true;
  }
  bool has_rates_ = false, has_scale_ = false, has_len_ = false;
  float quality_ = 50;
};
DALI_REGISTER_OPERATOR(AudioResample, AudioResampleGPU, GPU);

// dali/operators/audio/nonsilence_op.{h,cc}: leading / trailing silence detection; outputs (begin, length) as int32 scalars
DALI_SCHEMA(NonsilentRegion)
    .DocStr("Performs leading and trailing silence detection in an audio buffer.")
    .NumInput(1).NumOutput(2)
    .AddOptionalArg("cutoff_db", "The threshold, in dB, below which the signal is considered silent.", -60.0f, true)
    .AddOptionalArg("window_length", "Size of the sliding window used to calculate the short-term power of the signal.", 2048)
    .AddOptionalArgNoDefault("reference_power", "The reference power; when absent the maximum power of the signal is used.", true)
    .AddOptionalArg("reset_interval", "Number of samples after which the moving mean average is recalculated (-1: never).", 8192);

class NonsilentRegionGPU : public SignalOpBase {
 public:
  explicit NonsilentRegionGPU(const OpSpec &spec) : SignalOpBase(spec, "NonsilentRegion") {
    window_ = spec.GetArgument<int>("window_length");
    reset_ = spec.GetArgument<int>("reset_interval");
    has_ref_ = spec.ArgumentDefined("reference_power");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "NonsilentRegion: the GPU path supports float input; got type ", static_cast<int>(in.type()));
    const int n = in.num_samples();
    std::vector<int64_t> len(n);
    std::vector<dalib200NonsilentSample> args(n);
    for (int i = 0; i < n; i++) {
      len[i] = in.shape().tensor_size(i);
      args[i].cutoff_db = spec_.GetArgument<float>("cutoff_db", &ws, i);
      args[i].use_reference_power = has_ref_ ? 1 : 0;
      args[i].reference_power = has_ref_ ? spec_.GetArgument<float>("reference_power", &ws, i) : 0.0f;
      DALI_ENFORCE(!has_ref_ || args[i].reference_power > 0, "`reference_power` has to be positive. Got: ", args[i].reference_power);
    }
    CheckStatus(dalib200NonsilentSetup(plan_, n, len.data(), args.data(), window_, reset_), name_);
    out.resize(2);
    for (int o = 0; o < 2; o++) {
      out[o].type = DALI_INT32;
      out[o].shape.resize(n, 0);
    }
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &begin = ws.Output<GPUBackend>(0);
    auto &length = ws.Output<GPUBackend>(1);
    const int n = in.num_samples();
    std::vector<const void *> ip(n);
    std::vector<void *> bp(n), lp(n);
    for (int i = 0; i < n; i++) { ip[i] = in.raw_tensor(i); bp[i] = begin.raw_mutable_tensor(i); lp[i] = length.raw_mutable_tensor(i); }
    CheckStatus(dalib200NonsilentLaunch(plan_, ip.data(), bp.data(), lp.data(), ws.stream()), name_);
  }
  int window_ = 2048, reset_ = 8192;
  bool has_ref_ = false;
};
DALI_REGISTER_OPERATOR(NonsilentRegion, NonsilentRegionGPU, GPU);

DALI_SCHEMA(ToDecibels)
    .DocStr("Converts a magnitude (real, positive) to the decibel scale.")
    .NumInput(1).NumOutput(1)
    .AddOptionalArg("multiplier", "Factor by which the logarithm is multiplied (10 or 20).", 10.0f)
    .AddOptionalArgNoDefault("reference", "Reference magnitude; when absent the per-sample maximum is used.")
    .AddOptionalArg("cutoff_db", "Minimum or cut-off ratio in dB.", -200.0f);

class ToDecibelsGPU : public SignalOpBase {
 public:
  explicit ToDecibelsGPU(const OpSpec &spec) : SignalOpBase(spec, "ToDecibels") {
    args_.multiplier = spec.GetArgument<float>("multiplier");
    args_.ref_max = !spec.ArgumentDefined("reference");
    args_.reference = args_.ref_max ? 1.0f : spec.GetArgument<float>("reference");
    DALI_ENFORCE(args_.ref_max || args_.reference != 0, "`reference` argument can't be zero");
    args_.cutoff_db = spec.GetArgument<float>("cutoff_db");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "Unsupported data type: ", static_cast<int>(in.type()));
    const int n = in.num_samples();
    std::vector<int64_t> vol(n);
    for (int i = 0; i < n; i++) vol[i] = in.shape().tensor_size(i);
    CheckStatus(dalib200ToDecibelsSetup(plan_, &args_, n, vol.data()), name_);
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = DALI_FLOAT;
    return true;
  }
  dalib200ToDecibelsArgs args_{};
};
DALI_REGISTER_OPERATOR(ToDecibels, ToDecibelsGPU, GPU);

DALI_SCHEMA(MFCC)
    .DocStr("Computes Mel Frequency Cepstral Coefficients (MFCC) from a mel spectrogram.")
    .NumInput(1).NumOutput(1)
    .AddOptionalArg("n_mfcc", "Number of MFCC coefficients.", 20)
    .AddOptionalArg("dct_type", "Discrete Cosine Transform type (1, 2, 3, 4).", 2)
    .AddOptionalArg("normalize", "If set to True, the DCT uses an ortho-normal basis.", false)
    .AddOptionalArg("axis", "Axis over which the transform is applied.", 0)
    .AddOptionalArg("lifter", "Cepstral filtering (liftering) coefficient; 0 = none.", 0.0f);

class MfccGPU : public SignalOpBase {
 public:
  explicit MfccGPU(const OpSpec &spec) : SignalOpBase(spec, "MFCC") {
    args_.n_mfcc = spec.GetArgument<int>("n_mfcc");
    DALI_ENFORCE(args_.n_mfcc > 0, "number of MFCCs should be > 0");
    args_.dct_type = spec.GetArgument<int>("dct_type");
    DALI_ENFORCE(args_.dct_type >= 1 && args_.dct_type <= 4, "Unsupported DCT type: ", args_.dct_type, ". Supported types are: 1, 2, 3, 4.");
    args_.normalize = spec.GetArgument<bool>("normalize");
    DALI_ENFORCE(!(args_.normalize && args_.dct_type == 1), "Ortho-normalization is not supported for DCT type I.");
    axis_ = spec.GetArgument<int>("axis");
    DALI_ENFORCE(axis_ >= 0, "Provided axis cannot be negative.");
    args_.lifter = spec.GetArgument<float>("lifter");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "MFCC: unsupported data type");
    const int nd = in.shape().sample_dim();
    DALI_ENFORCE(axis_ < nd, "Axis ", axis_, " is out of bounds [0,", nd, ")");
    DALI_ENFORCE(nd == 2 && axis_ == 0, "MFCC: the GPU path transforms axis 0 of 2-D (frequency, time) inputs");
    const int n = in.num_samples();
    std::vector<int64_t> shp(2 * n);
    for (int i = 0; i < n; i++) { shp[2 * i] = in.shape().tensor_shape_span(i)[0]; shp[2 * i + 1] = in.shape().tensor_shape_span(i)[1]; }
    CheckStatus(dalib200MfccSetup(plan_, &args_, n, shp.data()), name_);
    out.resize(1);
    out[0].type = DALI_FLOAT;
    out[0].shape.resize(n, 2);
    for (int i = 0; i < n; i++) out[0].shape.set_tensor_shape(i, { dalib200SignalOutputRows(plan_), shp[2 * i + 1] });
    return true;
  }
  dalib200MfccArgs args_{};
  int axis_ = 0;
};
DALI_REGISTER_OPERATOR(MFCC, MfccGPU, GPU);

DALI_SCHEMA(Normalize)
    .DocStr("Normalizes the input by removing the mean and dividing by the standard deviation (per sample, 2-D float inputs).")
    .NumInput(1).NumOutput(1)
    .AddOptionalArg("batch", "not supported by the GPU path (per-sample statistics only)", false)
    .AddOptionalArgNoDefault("axes", "Indices of dimensions along which the input is normalized (default: all).")
    .AddOptionalArgNoDefault("axis_names", "Names of the reduced axes in the input layout.")
    .AddOptionalArg("shift", "The value to which the mean will map in the output.", 0.0f)
    .AddOptionalArg("scale", "The scaling factor applied to the output.", 1.0f)
    .AddOptionalArg("epsilon", "A value that is added to the variance.", 0.0f)
    .AddOptionalArg("ddof", "Delta Degrees of Freedom for Bessel's correction.", 0)
    .AddOptionalArg("dtype", "Output data type (FLOAT).", DALI_FLOAT);

class NormalizeGPU : public SignalOpBase {
 public:
  explicit NormalizeGPU(const OpSpec &spec) : SignalOpBase(spec, "Normalize") {
    DALI_ENFORCE(!spec.GetArgument<bool>("batch"), "Normalize: batch=True is not supported by the GPU path");
    DALI_ENFORCE(spec.GetArgument<DALIDataType>("dtype") == DALI_FLOAT, "Normalize: the GPU path produces FLOAT output");
    DALI_ENFORCE(!(spec.ArgumentDefined("axes") && spec.ArgumentDefined("axis_names")), "Arguments `axes` and `axis_names` are mutually exclusive");
    args_.scale = spec.GetArgument<float>("scale"); args_.shift = spec.GetArgument<float>("shift");
    args_.epsilon = spec.GetArgument<float>("epsilon"); args_.ddof = spec.GetArgument<int>("ddof");
  }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_FLOAT, "Normalize: the GPU path expects float input");
    const int nd = in.shape().sample_dim();
    DALI_ENFORCE(nd == 1 || nd == 2, "Normalize: the GPU path supports 1-D and 2-D inputs");
    bool red[2] = { true, true };
    if (spec_.ArgumentDefined("axes")) {
      red[0] = red[1] = false;
      for (int a : spec_.GetRepeatedArgument<int>("axes")) { DALI_ENFORCE(a >= 0 && a < nd, "Axis index out of range: ", a); red[nd == 1 ? 1 : a] = true; }
    } else if (spec_.ArgumentDefined("axis_names")) {
      red[0] = red[1] = false;
      const std::string names = spec_.GetArgument<std::string>("axis_names"), lay = in.GetLayout().str();
      for (char c : names) { const auto p = lay.find(c); DALI_ENFORCE(p != std::string::npos, "Axis '", std::string(1, c), "' not found in the input layout"); red[nd == 1 ? 1 : p] = true; }
    }
    if (nd == 1) red[0] = true;
    DALI_ENFORCE(red[0] || red[1], "Normalize: at least one axis must be reduced");
    args_.mode = red[0] && red[1] ? 0 : red[1] ? 1 : 2;
    const int n = in.num_samples();
    std::vector<int64_t> shp(2 * n);
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      shp[2 * i] = nd == 1 ? 1 : s[0]; shp[2 * i + 1] = nd == 1 ? s[0] : s[1];
    }
    CheckStatus(dalib200NormalizeSetup(plan_, &args_, n, shp.data()), name_);
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = DALI_FLOAT;
    return true;
  }
  dalib200NormalizeArgs args_{};
};
DALI_REGISTER_OPERATOR(Normalize, NormalizeGPU, GPU);

// =============================================================================================== GaussianBlur
// dali/operators/image/convolution/gaussian_blur.cc (schema), gaussian_blur_params.h (per-axis sigma / window resolution),
// gaussian_blur_gpu.cu; the convolution itself is dalib200SepConv* (separable, reflect-101, innermost axis first).
DALI_SCHEMA(GaussianBlur)
    .DocStr("Applies a Gaussian Blur to the input.\n\nGaussian blur is calculated by applying a convolution with a Gaussian kernel, "
            "which can be parametrized with `windows_size` and `sigma`. If only the sigma is specified, the radius of the kernel "
            "is 3 * sigma (rounded up), so the kernel window size is 2 * ceil(3 * sigma) + 1. If only the window size is provided, "
            "the sigma is calculated by using the following formula: radius = (window_size - 1) / 2; "
            "sigma = (radius - 1) * 0.3 + 0.8. The sigma and kernel window size can be specified as one value for all data "
            "axes or a value per data axis. When specifying the sigma or window size per axis, the axes are provided same as "
            "layouts, from outermost to innermost. The channel C dimension and the frame F dimension are not blurred.")
    .NumInput(1).NumOutput(1).AllowSequences()
    .AddOptionalArg("window_size", "The diameter of the kernel.", std::vector<int>{0}, true)
    .AddOptionalArg("sigma", "Sigma value for the Gaussian Kernel.", std::vector<float>{0.0f}, true)
    .AddOptionalArgNoDefault("dtype", "Output data type.\n\nSupported type: `FLOAT`. If not set, the input type is used.");

namespace gaussian_detail {
// channel-last layouts with an optional leading F; returns false for anything else
inline bool ParseLayout(const std::string &l, bool *frames, int *spatial) {
  static const char *const kLayouts[] = { "HW", "HWC", "FHW", "FHWC", "DHW", "DHWC", "FDHW", "FDHWC" };
  bool known = false;
  for (const char *k : kLayouts) known |= l == k;
  if (!known) return false;
  *frames = l[0] == 'F';
  *spatial = l.find('D') == std::string::npos ? 2 : 3;
  return true;
}
// GaussianBlurParams (gaussian_blur_params.h): window_size = 2 * ceil(3 sigma) + 1 when only sigma is given,
// sigma = (radius - 1) * 0.3 + 0.8 when only the window is given
inline void ResolveAxis(float sigma, float window, int sample, int axis, float *sigma_out, int *diameter_out) {
  DALI_ENFORCE(window == std::floor(window) && window >= 0 && window <= 1e9f, "GaussianBlur: sample ", sample, " axis ", axis,
               ": `window_size` must be a non-negative integer, got ", window);
  const int ws = static_cast<int>(window);
  DALI_ENFORCE(ws == 0 || ws % 2 == 1, "GaussianBlur: sample ", sample, " axis ", axis, ": kernel window should have odd length, got: ", ws);
  DALI_ENFORCE(sigma >= 0, "GaussianBlur: sample ", sample, " axis ", axis, ": sigma must be non-negative, got: ", sigma);
  DALI_ENFORCE(!(sigma == 0 && ws == 0), "GaussianBlur: sample ", sample, " axis ", axis,
               ": `sigma` and `window_size` shouldn't be 0 at the same time");
  int d = ws;
  if (d == 0) {
    const float r = std::ceil(sigma * 3);
    DALI_ENFORCE(r <= 1e6f, "GaussianBlur: sample ", sample, " axis ", axis, ": sigma ", sigma, " is too large");
    d = 2 * static_cast<int>(r) + 1;
  }
  float s = sigma;
  if (s == 0) s = static_cast<float>(((d - 1) / 2 - 1) * 0.3 + 0.8);
  *sigma_out = s;
  *diameter_out = d;
}
}  // namespace gaussian_detail

class GaussianBlurGPU : public Operator<GPUBackend> {
 public:
  explicit GaussianBlurGPU(const OpSpec &spec) : Operator<GPUBackend>(spec) {
    CheckStatus(dalib200SepConvPlanCreate(&plan_, max_batch_size_ * 64), "GaussianBlur");
    plan_cap_ = max_batch_size_ * 64;
  }
  ~GaussianBlurGPU() override { dalib200SepConvPlanDestroy(plan_); }
 protected:
  bool SetupImpl(std::vector<OutputDesc> &out, const Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    DALI_ENFORCE(in.type() == DALI_UINT8 || in.type() == DALI_FLOAT,
                 "GaussianBlur: the GPU path supports uint8 and float inputs, got type ", static_cast<int>(in.type()));
    out_type_ = spec_.ArgumentDefined("dtype") ? spec_.GetArgument<DALIDataType>("dtype") : in.type();
    DALI_ENFORCE(out_type_ == in.type() || out_type_ == DALI_FLOAT, "GaussianBlur: output type must be the input type or FLOAT");
    const int nd = in.shape().sample_dim();
    layout_ = in.GetLayout().str();
    if (layout_.empty()) layout_ = nd == 3 ? "HWC" : nd == 4 ? "FHWC" : "";
    bool frames = false;
    int spatial = 2;
    DALI_ENFORCE(gaussian_detail::ParseLayout(layout_, &frames, &spatial), "GaussianBlur: unsupported layout \"", layout_,
                 "\" (", nd, "-D input); expected one of HW, HWC, FHW, FHWC, DHW, DHWC, FDHW, FDHWC");
    DALI_ENFORCE(static_cast<int>(layout_.size()) == nd, "GaussianBlur: layout \"", layout_, "\" does not match a ", nd, "-D input");
    const bool has_c = layout_.back() == 'C';
    const int fs = frames ? 1 : 0;
    const int n = in.num_samples();
    samples_.clear();
    frame_sample_.clear();
    frame_off_.clear();
    std::vector<float> windows;
    std::map<std::pair<uint32_t, int>, int32_t> seen;      // (sigma bits, diameter) -> offset: one window per distinct pair
    for (int i = 0; i < n; i++) {
      const int64_t *s = in.shape().tensor_shape_span(i);
      const auto sig = spec_.GetFloatVecArgument("sigma", &ws, i, spatial);
      const auto win = spec_.GetFloatVecArgument("window_size", &ws, i, spatial);
      dalib200SepConvSample cs{};
      cs.ndim = spatial;
      cs.channels = has_c ? static_cast<int32_t>(s[nd - 1]) : 1;
      for (int a = 0; a < spatial; a++) {
        DALI_ENFORCE(s[fs + a] < (int64_t{1} << 31), "GaussianBlur: extent too large");
        cs.shape[a] = static_cast<int32_t>(s[fs + a]);
        float sigma;
        int d;
        gaussian_detail::ResolveAxis(sig[a], win[a], i, a, &sigma, &d);
        DALI_ENFORCE(d <= 8191, "GaussianBlur: sample ", i, " axis ", a, ": window of ", d, " taps exceeds the limit of 8191");
        uint32_t bits;
        std::memcpy(&bits, &sigma, 4);
        auto it = seen.find({bits, d});
        if (it == seen.end()) {
          it = seen.emplace(std::make_pair(bits, d), static_cast<int32_t>(windows.size())).first;
          windows.resize(windows.size() + d);
          dalib200GaussianWindow(sigma, d, windows.data() + it->second);
        }
        cs.diameter[a] = d;
        cs.window_offset[a] = it->second;
      }
      const int64_t nframes = frames ? s[0] : 1;
      int64_t fe = cs.channels;
      for (int a = 0; a < spatial; a++) fe *= cs.shape[a];
      for (int64_t k = 0; k < nframes; k++) { samples_.push_back(cs); frame_sample_.push_back(i); frame_off_.push_back(k * fe); }
    }
    const int nf = static_cast<int>(samples_.size());
    if (nf > plan_cap_) { dalib200SepConvPlanDestroy(plan_); plan_ = nullptr; plan_cap_ = nf; CheckStatus(dalib200SepConvPlanCreate(&plan_, nf), "GaussianBlur"); }
    CheckStatus(dalib200SepConvPlanSetup(plan_, nf, samples_.data(), windows.data(), static_cast<int64_t>(windows.size()),
                                         in.type() == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT,
                                         out_type_ == DALI_UINT8 ? DALIB200_UINT8 : DALIB200_FLOAT), "GaussianBlur");
    out.resize(1);
    out[0].shape = in.shape(); out[0].type = out_type_;
    return true;
  }
  void RunImpl(Workspace &ws) override {
    const auto &in = ws.Input<GPUBackend>(0);
    auto &out = ws.Output<GPUBackend>(0);
    out.SetLayout(TensorLayout(layout_));
    const int nf = static_cast<int>(samples_.size());
    std::vector<const void *> ip(nf);
    std::vector<void *> op(nf);
    const size_t ies = TypeSize(in.type()), oes = TypeSize(out_type_);
    for (int k = 0; k < nf; k++) {
      ip[k] = static_cast<const uint8_t *>(in.raw_tensor(frame_sample_[k])) + frame_off_[k] * ies;
      op[k] = static_cast<uint8_t *>(out.raw_mutable_tensor(frame_sample_[k])) + frame_off_[k] * oes;
    }
    CheckStatus(dalib200SepConvLaunch(plan_, ip.data(), op.data(), ws.stream()), "GaussianBlur");
  }
 private:
  dalib200SepConvPlan *plan_ = nullptr;
  int plan_cap_ = 0;
  DALIDataType out_type_ = DALI_UINT8;
  std::string layout_;
  std::vector<dalib200SepConvSample> samples_;
  std::vector<int> frame_sample_;        // frame -> sample
  std::vector<int64_t> frame_off_;       // element offset of the frame inside its sample
};
DALI_REGISTER_OPERATOR(GaussianBlur, GaussianBlurGPU, GPU);

}  // namespace dali

// ---------------------------------------------------------------------------------------------------------------
// Test hook (CPU): the Resize size / ROI arithmetic without a pipeline, so that the reference's known-answer vectors
// (dali/operators/image/resize/resize_attr_test.cc) can be checked where no GPU exists.
extern "C" int dalihTestResizeParams(int mode, const float *requested_hw, const float *in_lo_hw, const float *in_hi_hw,
                                     int subpixel_scale, const float *max_size_hw_or_null, int *dst_hw, float *lo_hw, float *hi_hw) {
  try {
    float req[2] = { requested_hw[0], requested_hw[1] }, lo[2] = { in_lo_hw[0], in_lo_hw[1] }, hi[2] = { in_hi_hw[0], in_hi_hw[1] };
    dali::resize_detail::Params p;
    dali::resize_detail::CalculateSampleParams(p, req, lo, hi, subpixel_scale != 0, false, static_cast<dali::resize_detail::Mode>(mode),
                                               max_size_hw_or_null);
    for (int d = 0; d < 2; d++) { dst_hw[d] = p.dst[d]; lo_hw[d] = p.lo[d]; hi_hw[d] = p.hi[d]; }
    return 0;
  } catch (...) { return 1; }
}

// Layout parsing of Resize (resize_attr_test.cc:22-51): returns 0 and (spatial_ndim, first_spatial_dim), or 1 for a layout it rejects.
extern "C" int dalihTestResizeLayout(const char *layout, int *spatial_ndim, int *first_spatial) {
  try { dali::ParseResizeLayout(layout, spatial_ndim, first_spatial); return 0; } catch (...) { return 1; }
}

// The same for volumes (spatial_ndim = 3; arrays in shape order depth, height, width): resize_attr_test.cc Resize3D* vectors.
extern "C" int dalihTestResizeParams3D(int mode, const float *requested_dhw, const float *in_lo_dhw, const float *in_hi_dhw,
                                       int subpixel_scale, const float *max_size_dhw_or_null, int *dst_dhw, float *lo_dhw, float *hi_dhw) {
  try {
    float req[3], lo[3], hi[3];
    for (int d = 0; d < 3; d++) { req[d] = requested_dhw[d]; lo[d] = in_lo_dhw[d]; hi[d] = in_hi_dhw[d]; }
    dali::resize_detail::Params p;
    dali::resize_detail::CalculateSampleParams(p, req, lo, hi, subpixel_scale != 0, false, static_cast<dali::resize_detail::Mode>(mode),
                                               max_size_dhw_or_null, 3);
    for (int d = 0; d < 3; d++) { dst_dhw[d] = p.dst[d]; lo_dhw[d] = p.lo[d]; hi_dhw[d] = p.hi[d]; }
    return 0;
  } catch (...) { return 1; }
}

// Test hook (CPU): the random crop windows of decoders.image_random_crop / random_resized_crop without a pipeline, so that they can be
// compared with the reference's own generator (oracle/_ref: random_crop_generator_util.cc + philox.cc) where no GPU exists.
extern "C" int dalihTestRandomCrop(int64_t seed, int sample_idx, int H, int W, float ar_lo, float ar_hi, float area_lo, float area_hi,
                                   int num_attempts, int ncalls, int *windows) {
  const uint64_t key = static_cast<uint64_t>(seed) ^ dali::kRandomCropSeedModifier;
  dali::RandomCropGenerator gen(ar_lo, ar_hi, area_lo, area_hi, key, static_cast<uint64_t>(dali::kSkipaheadPerSample) * sample_idx, num_attempts);
  for (int k = 0; k < ncalls; k++) {
    const dali::CropWindow2D w = gen.Generate(H, W);
    windows[4 * k] = w.anchor[0]; windows[4 * k + 1] = w.anchor[1]; windows[4 * k + 2] = w.shape[0]; windows[4 * k + 3] = w.shape[1];
  }
  return 0;
}

// Test hooks (CPU): Rotate's canvas size / matrix and BrightnessContrast's kernel arguments, for comparison with the reference's own
// code (oracle/_ref: rotate_params.h + geom/transform.h, brightness_contrast.h) where no GPU exists.
extern "C" int dalihTestRotateParams(float angle_deg, int in_h, int in_w, int keep_size, const float *size_hw_or_null, int *out_hw, float *m2x3) {
  dali::rotate_detail::Params(angle_deg, in_h, in_w, keep_size != 0, size_hw_or_null, out_hw[0], out_hw[1], m2x3);
  return 0;
}

// Test hooks (CPU): the crop-window and slice-window arithmetic of decoders.image_crop / crop / slice without a pipeline (no device
// calls), for known answers of the reference's rules: CropAttr::CalculateAnchor (crop_attr.cc:224-239: anchor = round(pos * (in - crop)),
// half away from zero, or truncation with rounding="truncate") and the slice attributes (slice_attr.h: std::llround of start / end).
extern "C" int dalihTestCropWindow(float crop_h, float crop_w, float pos_y, float pos_x, int truncate, int H, int W, int64_t *yxhw) {
  try {
    dali::OpSpec spec("Crop");
    spec.AddArg("crop_h", dali::MakeArg(crop_h)).AddArg("crop_w", dali::MakeArg(crop_w));
    spec.AddArg("crop_pos_y", dali::MakeArg(pos_y)).AddArg("crop_pos_x", dali::MakeArg(pos_x));
    spec.AddArg("rounding", dali::MakeArg(std::string(truncate ? "truncate" : "round")));
    dali::CropWindowArgs c;
    c.Init(spec, "Crop");
    dali::Workspace ws;
    c.Get(spec, ws, 0, H, W, yxhw[0], yxhw[1], yxhw[2], yxhw[3]);
    return 0;
  } catch (...) { return 1; }
}

// anchor / shape given per axis in (W, H) order like the operator's default `axis_names="WH"`; mode 0: absolute start + shape,
// 1: relative start + relative shape, 2: absolute start + end, 3: relative start + relative end.  out = {y0, y1, x0, x1}.
extern "C" int dalihTestSliceWindow(int mode, const float *a_wh, const float *b_wh, int H, int W, int64_t *out) {
  try {
    dali::OpSpec spec("Slice");
    spec.AddArg("axis_names", dali::MakeArg(std::string("WH")));
    spec.AddArg("normalized_anchor", dali::MakeArg(true)).AddArg("normalized_shape", dali::MakeArg(true));
    const std::vector<float> a(a_wh, a_wh + 2), b(b_wh, b_wh + 2);
    const char *an = (mode == 0 || mode == 2) ? "start" : "rel_start";
    const char *bn = mode == 0 ? "shape" : mode == 1 ? "rel_shape" : mode == 2 ? "end" : "rel_end";
    if (mode == 0 || mode == 2) {
      spec.AddArg(an, dali::MakeArg(std::vector<int>{ static_cast<int>(a[0]), static_cast<int>(a[1]) }));
      spec.AddArg(bn, dali::MakeArg(std::vector<int>{ static_cast<int>(b[0]), static_cast<int>(b[1]) }));
    } else {
      spec.AddArg(an, dali::MakeArg(a)).AddArg(bn, dali::MakeArg(b));
    }
    // one data input only: named arguments
    spec.AddInput("data", "gpu");
    dali::SliceArgs sl;
    sl.Init(spec, "Slice");
    dali::Workspace ws;
    int64_t bgn[2], end[2];
    sl.Get(spec, ws, 0, H, W, bgn, end);
    out[0] = bgn[0]; out[1] = end[0]; out[2] = bgn[1]; out[3] = end[1];
    return 0;
  } catch (...) { return 1; }
}
