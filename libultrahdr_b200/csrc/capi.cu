// The reference's public C API (ultrahdr_api.h:301-905, implemented in lib/src/ultrahdr_api.cpp)
// on top of the B200 codec.  Same handle state machine: setters are rejected once the handle has
// "sailed"; uhdr_encode / uhdr_decode are single shot and return their cached status when called
// again; reset restores the defaults of ultrahdr_api.cpp:1452-1484 / 2045-2083.  Inputs are
// uploaded to the device at set time (the reference deep-copies at the same point,
// ultrahdr_api.cpp:1033-1042), outputs stay owned by the handle.
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>

#include "codec.h"

using namespace uhdr_b200;

struct uhdr_codec_private {
  virtual ~uhdr_codec_private() {}
  JpegRCodec codec;
  bool sailed = false;
  bool ready = false;
  int init_rc = 0;
  int device = -1;  // the CUDA device that was current when the handle was created
  std::string init_err;
  // uhdr_add_effect_* in call order; cleared by reset, keeping its capacity.  Planned into one gather per image
  // (effects.h) when the handle sails.
  std::vector<Effect> effects;
  uhdr_codec_private() {
    if (cudaGetDevice(&device) != cudaSuccess) device = -1;
  }
  // CUDA's current device is per host thread: a handle may be driven from any thread, so every
  // entry point that touches the device re-selects the handle's own GPU first.
  void bind() {
    if (device >= 0) cudaSetDevice(device);
  }
  void ensure() {
    bind();
    if (ready) return;
    init_rc = codec.init();
    if (init_rc) init_err = last_error();
    ready = true;
  }
};

namespace {

uhdr_error_info_t ok() {
  uhdr_error_info_t s;
  memset(&s, 0, sizeof s);
  s.error_code = UHDR_CODEC_OK;
  return s;
}
uhdr_error_info_t err(uhdr_codec_err_t code, const char* fmt, ...) {
  uhdr_error_info_t s;
  memset(&s, 0, sizeof s);
  s.error_code = code;
  s.has_detail = 1;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(s.detail, sizeof s.detail, fmt, ap);
  va_end(ap);
  return s;
}
uhdr_error_info_t from_rc(int rc) {
  if (rc == E_OK) return ok();
  return err((uhdr_codec_err_t)rc, "%s", last_error());
}

struct Encoder : uhdr_codec_private {
  // keyed by uhdr_img_label_t (0..3); fixed slots: configuring / resetting a handle does not touch the heap
  SlotMap<DevImage, 4> raw;            // UHDR_HDR_IMG / UHDR_SDR_IMG, device resident
  SlotMap<int, 4> quality;
  struct Compressed { std::vector<uint8_t> bytes; int cg = 0, ct = 0, range = 0; };
  SlotMap<Compressed, 4> compressed;   // UHDR_SDR_IMG / UHDR_BASE_IMG / UHDR_GAIN_MAP_IMG (encode API-2/3/4)
  uhdr_gainmap_metadata_t metadata{};
  std::vector<uint8_t> exif;
  int scale = 1, multichannel = 1, preset = UHDR_USAGE_BEST_QUALITY, output_format = UHDR_CODEC_JPG;
  float gamma = 1.0f, min_boost = FLT_MIN, max_boost = FLT_MAX, target_nits = -1.0f;
  bool has_compressed = false;
  std::unique_ptr<uint8_t[]> out;  // kept across resets; never zero-filled
  size_t out_cap = 0;
  uhdr_compressed_image_t out_desc{};
  uhdr_error_info_t status = ok();
  void defaults() {
    raw.clear();
    compressed.clear([](Compressed& c) { c.bytes.clear(); });   // keeps the capacity
    memset(&metadata, 0, sizeof metadata);
    quality.clear();
    quality[UHDR_BASE_IMG] = 95;
    quality[UHDR_GAIN_MAP_IMG] = 95;
    exif.clear();
    scale = 1; multichannel = 1; preset = UHDR_USAGE_BEST_QUALITY; output_format = UHDR_CODEC_JPG;
    gamma = 1.0f; min_boost = FLT_MIN; max_boost = FLT_MAX; target_nits = -1.0f;
    has_compressed = false;
    effects.clear();
    sailed = false;
    memset(&out_desc, 0, sizeof out_desc);
    status = ok();
    if (ready && !init_rc) { bind(); codec.ws().clear_floor(); }
  }
  Encoder() { defaults(); }
};

struct Decoder : uhdr_codec_private {
  std::vector<uint8_t> stream;
  int out_fmt = UHDR_IMG_FMT_64bppRGBAHalfFloat, out_ct = UHDR_CT_LINEAR;
  float max_boost = FLT_MAX;
  bool probed = false;
  DecodedInfo info;
  uhdr_mem_block_t exif_blk{}, icc_blk{}, base_blk{}, gm_blk{};
  std::vector<uint8_t> decoded, gainmap;
  uhdr_raw_image_t decoded_desc{}, gainmap_desc{};
  uhdr_error_info_t probe_status = ok(), status = ok();
  void defaults() {
    stream.clear();
    effects.clear();
    out_fmt = UHDR_IMG_FMT_64bppRGBAHalfFloat;
    out_ct = UHDR_CT_LINEAR;
    max_boost = FLT_MAX;
    probed = sailed = false;
    info = DecodedInfo();
    decoded.clear();
    gainmap.clear();
    probe_status = status = ok();
  }
};

template <class T>
T* as(uhdr_codec_private_t* p) { return dynamic_cast<T*>(p); }

}  // namespace

extern "C" {

// ---- encoder -------------------------------------------------------------------------------------
UHDR_API uhdr_codec_private_t* uhdr_create_encoder(void) { return new (std::nothrow) Encoder(); }
UHDR_API void uhdr_release_encoder(uhdr_codec_private_t* enc) { if (as<Encoder>(enc)) delete enc; }

UHDR_API uhdr_error_info_t uhdr_enc_set_raw_image(uhdr_codec_private_t* enc, uhdr_raw_image_t* img,
                                                  uhdr_img_label_t intent) {
  Encoder* h = as<Encoder>(enc);
  if (!h) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
  if (!img) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for raw image handle");
  if (intent != UHDR_HDR_IMG && intent != UHDR_SDR_IMG)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid intent %d, expects one of {UHDR_HDR_IMG, UHDR_SDR_IMG}", intent);
  // validation ladder of ultrahdr_api.cpp:842-1025
  if (intent == UHDR_HDR_IMG && img->fmt != UHDR_IMG_FMT_24bppYCbCrP010 && img->fmt != UHDR_IMG_FMT_32bppRGBA1010102 &&
      img->fmt != UHDR_IMG_FMT_64bppRGBAHalfFloat)
    return err(UHDR_CODEC_INVALID_PARAM, "unsupported input pixel format for hdr intent %d, expects one of "
               "{UHDR_IMG_FMT_24bppYCbCrP010, UHDR_IMG_FMT_32bppRGBA1010102, UHDR_IMG_FMT_64bppRGBAHalfFloat}", img->fmt);
  if (intent == UHDR_SDR_IMG && img->fmt != UHDR_IMG_FMT_12bppYCbCr420 && img->fmt != UHDR_IMG_FMT_32bppRGBA8888)
    return err(UHDR_CODEC_INVALID_PARAM, "unsupported input pixel format for sdr intent %d, expects one of "
               "{UHDR_IMG_FMT_12bppYCbCr420, UHDR_IMG_FMT_32bppRGBA8888}", img->fmt);
  if (img->cg != UHDR_CG_BT_2100 && img->cg != UHDR_CG_DISPLAY_P3 && img->cg != UHDR_CG_BT_709)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid input color gamut %d, expects one of {UHDR_CG_BT_2100, "
               "UHDR_CG_DISPLAY_P3, UHDR_CG_BT_709}", img->cg);
  if (intent == UHDR_SDR_IMG && img->ct != UHDR_CT_SRGB)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid input color transfer for sdr intent image %d, expects UHDR_CT_SRGB", img->ct);
  if (intent == UHDR_HDR_IMG && img->fmt == UHDR_IMG_FMT_64bppRGBAHalfFloat && img->ct != UHDR_CT_LINEAR)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid input color transfer for hdr intent image %d with format "
               "UHDR_IMG_FMT_64bppRGBAHalfFloat, expects one of {UHDR_CT_LINEAR}", img->ct);
  if (intent == UHDR_HDR_IMG && img->fmt != UHDR_IMG_FMT_64bppRGBAHalfFloat && img->ct != UHDR_CT_HLG && img->ct != UHDR_CT_PQ)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid input color transfer for hdr intent image %d with format %d, "
               "expects one of {UHDR_CT_HLG, UHDR_CT_PQ}", img->fmt, img->ct);
  if ((img->w % 2 != 0 || img->h % 2 != 0) && (img->fmt == UHDR_IMG_FMT_12bppYCbCr420 || img->fmt == UHDR_IMG_FMT_24bppYCbCrP010))
    return err(UHDR_CODEC_INVALID_PARAM, "image dimensions cannot be odd for formats {UHDR_IMG_FMT_12bppYCbCr420, "
               "UHDR_IMG_FMT_24bppYCbCrP010}, received image dimensions %dx%d", img->w, img->h);
  if ((int)img->w < 8 || (int)img->h < 8)
    return err(UHDR_CODEC_INVALID_PARAM, "image dimensions cannot be less than %dx%d, received image dimensions %dx%d", 8, 8, img->w, img->h);
  if ((int)img->w > 8192 || (int)img->h > 8192)
    return err(UHDR_CODEC_INVALID_PARAM, "image dimensions cannot be larger than %dx%d, received image dimensions %dx%d", 8192, 8192, img->w, img->h);
  if (img->fmt == UHDR_IMG_FMT_24bppYCbCrP010) {
    if (!img->planes[UHDR_PLANE_Y] || !img->planes[UHDR_PLANE_UV])
      return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for data field(s), luma ptr %p, chroma_uv ptr %p",
                 img->planes[UHDR_PLANE_Y], img->planes[UHDR_PLANE_UV]);
    if (img->stride[UHDR_PLANE_Y] < img->w)
      return err(UHDR_CODEC_INVALID_PARAM, "luma stride must not be smaller than width, stride=%d, width=%d", img->stride[UHDR_PLANE_Y], img->w);
    if (img->stride[UHDR_PLANE_UV] < img->w)
      return err(UHDR_CODEC_INVALID_PARAM, "chroma_uv stride must not be smaller than width, stride=%d, width=%d", img->stride[UHDR_PLANE_UV], img->w);
    if (img->range != UHDR_CR_FULL_RANGE && img->range != UHDR_CR_LIMITED_RANGE)
      return err(UHDR_CODEC_INVALID_PARAM, "invalid range, expects one of {UHDR_CR_FULL_RANGE, UHDR_CR_LIMITED_RANGE}");
  } else if (img->fmt == UHDR_IMG_FMT_12bppYCbCr420) {
    if (!img->planes[UHDR_PLANE_Y] || !img->planes[UHDR_PLANE_U] || !img->planes[UHDR_PLANE_V])
      return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for data field(s) luma ptr %p, chroma_u ptr %p, chroma_v ptr %p",
                 img->planes[UHDR_PLANE_Y], img->planes[UHDR_PLANE_U], img->planes[UHDR_PLANE_V]);
    if (img->stride[UHDR_PLANE_Y] < img->w)
      return err(UHDR_CODEC_INVALID_PARAM, "luma stride must not be smaller than width, stride=%d, width=%d", img->stride[UHDR_PLANE_Y], img->w);
    if (img->stride[UHDR_PLANE_U] < img->w / 2)
      return err(UHDR_CODEC_INVALID_PARAM, "chroma_u stride must not be smaller than width / 2, stride=%d, width=%d", img->stride[UHDR_PLANE_U], img->w);
    if (img->stride[UHDR_PLANE_V] < img->w / 2)
      return err(UHDR_CODEC_INVALID_PARAM, "chroma_v stride must not be smaller than width / 2, stride=%d, width=%d", img->stride[UHDR_PLANE_V], img->w);
    if (img->range != UHDR_CR_FULL_RANGE) return err(UHDR_CODEC_INVALID_PARAM, "invalid range, expects one of {UHDR_CR_FULL_RANGE}");
  } else {
    if (!img->planes[UHDR_PLANE_PACKED])
      return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for data field(s) rgb plane packed ptr %p", img->planes[UHDR_PLANE_PACKED]);
    if (img->stride[UHDR_PLANE_PACKED] < img->w)
      return err(UHDR_CODEC_INVALID_PARAM, "rgb planar stride must not be smaller than width, stride=%d, width=%d", img->stride[UHDR_PLANE_PACKED], img->w);
    if (img->range != UHDR_CR_FULL_RANGE) return err(UHDR_CODEC_INVALID_PARAM, "invalid range, expects one of {UHDR_CR_FULL_RANGE}");
  }
  const int other = intent == UHDR_HDR_IMG ? UHDR_SDR_IMG : UHDR_HDR_IMG;
  auto it = h->raw.find(other);
  if (it != h->raw.end() && ((unsigned)it->second.v.w != img->w || (unsigned)it->second.v.h != img->h))
    return err(UHDR_CODEC_INVALID_PARAM, "image resolutions mismatch: hdr intent: %dx%d, sdr intent: %dx%d",
               intent == UHDR_HDR_IMG ? img->w : it->second.v.w, intent == UHDR_HDR_IMG ? img->h : it->second.v.h,
               intent == UHDR_SDR_IMG ? img->w : it->second.v.w, intent == UHDR_SDR_IMG ? img->h : it->second.v.h);
  if (h->sailed)
    return err(UHDR_CODEC_INVALID_OPERATION, "An earlier call to uhdr_encode() has switched the context from configurable "
               "state to end state. The context is no longer configurable. To reuse, call reset()");
  h->ensure();
  if (h->init_rc) return err((uhdr_codec_err_t)h->init_rc, "%s", h->init_err.c_str());
  // the reference deep-copies here; we upload: after this returns the caller may reuse its buffer
  DevImage d;
  int rc = upload_image(h->codec.ws(), *img, &d);
  if (rc) return from_rc(rc);
  if (h->codec.ws().sync() != E_OK) return err(UHDR_CODEC_ERROR, "upload failed");
  h->raw[intent] = d;
  h->codec.ws().set_floor();  // inputs stay resident; per-encode scratch is recycled above them
  return ok();
}

// uhdr_enc_validate_and_set_compressed_img, ultrahdr_api.cpp:512-617
static uhdr_error_info_t set_compressed(uhdr_codec_private_t* enc, uhdr_compressed_image_t* img, int intent) {
  Encoder* h = as<Encoder>(enc);
  if (!h) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
  if (!img) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for compressed image handle");
  if (!img->data) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for compressed img->data field");
  if (img->capacity < img->data_sz) return err(UHDR_CODEC_INVALID_PARAM, "img->capacity %zd is less than img->data_sz %zd", img->capacity, img->data_sz);
  if (h->sailed)
    return err(UHDR_CODEC_INVALID_OPERATION, "An earlier call to uhdr_encode() has switched the context from configurable "
               "state to end state. The context is no longer configurable. To reuse, call reset()");
  size_t off = 0, len = 0;
  const int n = count_jpeg_images((const uint8_t*)img->data, img->data_sz, &off, &len);
  if (n < 0) return err(UHDR_CODEC_INVALID_PARAM, "received bad/corrupted jpeg image as part of input configuration");
  if (n == 0) return err(UHDR_CODEC_INVALID_PARAM, "compressed image received as part of input config contains no valid jpeg images");
  // several images: the first one is taken, the rest ignored (:572-584)
  Encoder::Compressed& c = h->compressed[intent];   // the slot's buffer is reused across resets
  c.bytes.assign((const uint8_t*)img->data + off, (const uint8_t*)img->data + off + len);
  c.cg = img->cg; c.ct = img->ct; c.range = img->range;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_compressed_image(uhdr_codec_private_t* enc, uhdr_compressed_image_t* img, uhdr_img_label_t intent) {
  if (intent != UHDR_HDR_IMG && intent != UHDR_SDR_IMG && intent != UHDR_BASE_IMG)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid intent %d, expects one of {UHDR_HDR_IMG, UHDR_SDR_IMG, UHDR_BASE_IMG}", intent);
  return set_compressed(enc, img, intent);
}
UHDR_API uhdr_error_info_t uhdr_enc_set_gainmap_image(uhdr_codec_private_t* enc, uhdr_compressed_image_t* img, uhdr_gainmap_metadata_t* metadata) {
  if (!metadata) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for gainmap metadata descriptor");
  int rc = validate_metadata(*metadata);
  if (rc) return from_rc(rc);
  uhdr_error_info_t st = set_compressed(enc, img, UHDR_GAIN_MAP_IMG);
  if (st.error_code != UHDR_CODEC_OK) return st;
  as<Encoder>(enc)->metadata = *metadata;
  return st;
}

#define ENC_SETTER_PROLOGUE                                                                                   \
  Encoder* h = as<Encoder>(enc);                                                                              \
  if (!h) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
#define ENC_SAILED_CHECK                                                                                      \
  if (h->sailed)                                                                                              \
    return err(UHDR_CODEC_INVALID_OPERATION, "An earlier call to uhdr_encode() has switched the context from " \
               "configurable state to end state. The context is no longer configurable. To reuse, call reset()");

UHDR_API uhdr_error_info_t uhdr_enc_set_quality(uhdr_codec_private_t* enc, int quality, uhdr_img_label_t intent) {
  ENC_SETTER_PROLOGUE
  if (quality < 0 || quality > 100) return err(UHDR_CODEC_INVALID_PARAM, "invalid quality factor %d, expects in range [0-100]", quality);
  if (intent != UHDR_HDR_IMG && intent != UHDR_SDR_IMG && intent != UHDR_BASE_IMG && intent != UHDR_GAIN_MAP_IMG)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid intent %d, expects one of {UHDR_HDR_IMG, UHDR_SDR_IMG, UHDR_BASE_IMG, UHDR_GAIN_MAP_IMG}", intent);
  ENC_SAILED_CHECK
  h->quality[intent] = quality;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_exif_data(uhdr_codec_private_t* enc, uhdr_mem_block_t* exif) {
  ENC_SETTER_PROLOGUE
  if (!exif) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for exif image handle");
  if (!exif->data) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for exif->data field");
  if (exif->capacity < exif->data_sz) return err(UHDR_CODEC_INVALID_PARAM, "exif->capacity %zd is less than exif->data_sz %zd", exif->capacity, exif->data_sz);
  ENC_SAILED_CHECK
  h->exif.assign((uint8_t*)exif->data, (uint8_t*)exif->data + exif->data_sz);
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_using_multi_channel_gainmap(uhdr_codec_private_t* enc, int use) {
  ENC_SETTER_PROLOGUE
  ENC_SAILED_CHECK
  h->multichannel = use;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_gainmap_scale_factor(uhdr_codec_private_t* enc, int s) {
  ENC_SETTER_PROLOGUE
  if (s <= 0 || s > 128) return err(UHDR_CODEC_INVALID_PARAM, "gainmap scale factor is expected to be in range (0, 128], received %d", s);
  ENC_SAILED_CHECK
  h->scale = s;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_gainmap_gamma(uhdr_codec_private_t* enc, float gamma) {
  ENC_SETTER_PROLOGUE
  if (!std::isfinite(gamma) || gamma <= 0.0f) return err(UHDR_CODEC_INVALID_PARAM, "unsupported gainmap gamma %f, expects to be > 0", gamma);
  ENC_SAILED_CHECK
  h->gamma = gamma;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_min_max_content_boost(uhdr_codec_private_t* enc, float mn, float mx) {
  ENC_SETTER_PROLOGUE
  if (!std::isfinite(mn) || !std::isfinite(mx)) return err(UHDR_CODEC_INVALID_PARAM, "received an argument with value either NaN or infinite. Configured min boost %f, max boost %f", mx, mn);
  if (mx < mn) return err(UHDR_CODEC_INVALID_PARAM, "Invalid min boost / max boost configuration. configured max boost %f is less than min boost %f", mx, mn);
  if (mn <= 0.0f) return err(UHDR_CODEC_INVALID_PARAM, "Invalid min boost configuration %f, expects > 0.0f", mn);
  ENC_SAILED_CHECK
  h->min_boost = mn;
  h->max_boost = mx;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_target_display_peak_brightness(uhdr_codec_private_t* enc, float nits) {
  ENC_SETTER_PROLOGUE
  if (!std::isfinite(nits) || nits < 203.0f || nits > 10000.0f)
    return err(UHDR_CODEC_INVALID_PARAM, "unexpected target display peak brightness nits %f, expects to be with in range [%f, %f]", nits, 203.0f, 10000.0f);
  ENC_SAILED_CHECK
  h->target_nits = nits;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_preset(uhdr_codec_private_t* enc, uhdr_enc_preset_t preset) {
  ENC_SETTER_PROLOGUE
  if (preset != UHDR_USAGE_REALTIME && preset != UHDR_USAGE_BEST_QUALITY)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid preset %d, expects one of {UHDR_USAGE_REALTIME, UHDR_USAGE_BEST_QUALITY}", preset);
  ENC_SAILED_CHECK
  h->preset = preset;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_enc_set_output_format(uhdr_codec_private_t* enc, uhdr_codec_t media_type) {
  ENC_SETTER_PROLOGUE
  if (media_type != UHDR_CODEC_JPG && media_type != UHDR_CODEC_AVIF && media_type != UHDR_CODEC_HEIF)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid output format %d, expects one of {UHDR_CODEC_JPG, UHDR_CODEC_HEIF, UHDR_CODEC_AVIF}", media_type);
  if (media_type != UHDR_CODEC_JPG)
    return err(UHDR_CODEC_UNSUPPORTED_FEATURE, "invalid output format %d, expects {UHDR_CODEC_JPG}", media_type);
  ENC_SAILED_CHECK
  h->output_format = media_type;
  return ok();
}

UHDR_API uhdr_error_info_t uhdr_encode(uhdr_codec_private_t* enc) {
  Encoder* h = as<Encoder>(enc);
  if (!h) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
  if (h->sailed) return h->status;
  h->sailed = true;
  h->bind();
  auto hdr = h->raw.find(UHDR_HDR_IMG);
  auto sdr = h->raw.find(UHDR_SDR_IMG);
  auto cbase = h->compressed.find(UHDR_BASE_IMG), cgm = h->compressed.find(UHDR_GAIN_MAP_IMG), csdr = h->compressed.find(UHDR_SDR_IMG);
  const bool api4 = cbase != h->compressed.end() && cgm != h->compressed.end();
  if (!api4 && hdr == h->raw.end()) {
    h->status = err(UHDR_CODEC_INVALID_OPERATION, "resources required for uhdr_encode() operation are not present");
    return h->status;
  }
  // image effects (:1219-1262): raw intents only, planned and validated before the device is touched
  const bool fx = !h->effects.empty();
  ImageMap fx_hdr{}, fx_sdr{};
  if (fx) {
    if (api4 || csdr != h->compressed.end()) {
      h->status = err(UHDR_CODEC_INVALID_OPERATION, "image effects are not enabled for inputs with compressed intent");
      return h->status;
    }
    const int rc = plan_encoder_effects(h->effects.data(), (int)h->effects.size(), hdr->second.v.fmt,
                                        sdr == h->raw.end() ? -1 : sdr->second.v.fmt, hdr->second.v.w, hdr->second.v.h,
                                        &fx_hdr, &fx_sdr);
    if (rc) { h->status = from_rc(rc); return h->status; }
  }
  const size_t cap = api4 ? std::max<size_t>(64 * 1024, 2 * (cbase->second.bytes.size() + cgm->second.bytes.size()))
                   : fx   ? std::max<size_t>(64 * 1024, (size_t)fx_hdr.w * fx_hdr.h * 3 * 2)
                          : std::max<size_t>(64 * 1024, (size_t)hdr->second.v.w * hdr->second.v.h * 3 * 2);  // :1281,:1294
  if (h->out_cap < cap) {
    h->out.reset(new (std::nothrow) uint8_t[cap]);
    h->out_cap = h->out ? cap : 0;
  }
  if (!h->out) { h->status = err(UHDR_CODEC_MEM_ERROR, "unable to allocate %zu bytes for the encoded stream", cap); return h->status; }
  uhdr_b200_gm_config_t cfg;
  cfg.scale_factor = h->scale;
  cfg.quality = h->quality[UHDR_GAIN_MAP_IMG];
  cfg.multichannel = h->multichannel;
  cfg.gamma = h->gamma;
  cfg.preset = h->preset;
  cfg.min_content_boost = h->min_boost;
  cfg.max_content_boost = h->max_boost;
  cfg.target_disp_peak_nits = h->target_nits;
  cfg.sdr_is_601 = 0;
  cfg.use_luminance = 1;
  size_t n = 0;
  int rc;
  if (api4) {  // pre-compressed base + gain map: container work on the host
    rc = JpegRCodec::encode_from_compressed(cbase->second.bytes.data(), cbase->second.bytes.size(), cbase->second.cg,
                                            cgm->second.bytes.data(), cgm->second.bytes.size(), h->metadata, h->out.get(), cap, &n);
  } else {
    h->ensure();
    if (h->init_rc) { h->status = err((uhdr_codec_err_t)h->init_rc, "%s", h->init_err.c_str()); return h->status; }
    h->codec.ws().rewind();
    if (csdr != h->compressed.end())  // API-2 (raw sdr intent given too) / API-3
      rc = h->codec.encode_with_compressed_sdr(hdr->second, sdr == h->raw.end() ? nullptr : &sdr->second, csdr->second.bytes.data(),
                                               csdr->second.bytes.size(), csdr->second.cg, cfg, h->out.get(), cap, &n);
    else {
      // the effects gather the resident intents into per-encode scratch above the arena floor: the inputs are
      // never written, so a re-armed handle encodes the same bytes again
      DevImage hdr_img = hdr->second, sdr_img;
      if (sdr != h->raw.end()) sdr_img = sdr->second;
      rc = E_OK;
      if (fx) rc = apply_effects_dev(h->codec.ws(), hdr->second, fx_hdr, &hdr_img);
      if (fx && rc == E_OK && sdr != h->raw.end()) rc = apply_effects_dev(h->codec.ws(), sdr->second, fx_sdr, &sdr_img);
      if (rc == E_OK)
        rc = h->codec.encode(hdr_img, sdr == h->raw.end() ? nullptr : &sdr_img, cfg, h->quality[UHDR_BASE_IMG],
                             h->exif.empty() ? nullptr : h->exif.data(), h->exif.size(), h->out.get(), cap, &n);
    }
  }
  h->status = from_rc(rc);
  if (rc == E_OK) {
    h->out_desc.data = h->out.get();
    h->out_desc.data_sz = n;
    h->out_desc.capacity = cap;
    h->out_desc.cg = UHDR_CG_UNSPECIFIED;
    h->out_desc.ct = UHDR_CT_UNSPECIFIED;
    h->out_desc.range = UHDR_CR_UNSPECIFIED;
  }
  return h->status;
}

UHDR_API uhdr_compressed_image_t* uhdr_get_encoded_stream(uhdr_codec_private_t* enc) {
  Encoder* h = as<Encoder>(enc);
  if (!h || !h->sailed || h->status.error_code != UHDR_CODEC_OK) return nullptr;
  return &h->out_desc;
}
UHDR_API void uhdr_reset_encoder(uhdr_codec_private_t* enc) {
  Encoder* h = as<Encoder>(enc);
  if (h) h->defaults();
}

// ---- decoder -------------------------------------------------------------------------------------
UHDR_API int is_uhdr_image(void* data, int size) {
  if (!data || size <= 0) return 0;
  JpegRCodec c;  // probing is host-only work
  DecodedInfo info;
  return c.probe((const uint8_t*)data, (size_t)size, &info) == E_OK ? 1 : 0;
}
UHDR_API uhdr_codec_private_t* uhdr_create_decoder(void) { return new (std::nothrow) Decoder(); }
UHDR_API void uhdr_release_decoder(uhdr_codec_private_t* dec) { if (as<Decoder>(dec)) delete dec; }

#define DEC_PROLOGUE                                                                          \
  Decoder* h = as<Decoder>(dec);                                                              \
  if (!h) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
#define DEC_PROBED_CHECK                                                                                       \
  if (h->probed)                                                                                               \
    return err(UHDR_CODEC_INVALID_OPERATION, "An earlier call to uhdr_decode() has switched the context from " \
               "configurable state to end state. The context is no longer configurable. To reuse, call reset()");

UHDR_API uhdr_error_info_t uhdr_dec_set_image(uhdr_codec_private_t* dec, uhdr_compressed_image_t* img) {
  DEC_PROLOGUE
  if (!img) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for compressed image handle");
  if (!img->data) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for compressed img->data field");
  if (img->capacity < img->data_sz) return err(UHDR_CODEC_INVALID_PARAM, "img->capacity %zd is less than img->data_sz %zd", img->capacity, img->data_sz);
  DEC_PROBED_CHECK
  h->stream.assign((uint8_t*)img->data, (uint8_t*)img->data + img->data_sz);
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_dec_set_out_img_format(uhdr_codec_private_t* dec, uhdr_img_fmt_t fmt) {
  DEC_PROLOGUE
  if (fmt != UHDR_IMG_FMT_32bppRGBA8888 && fmt != UHDR_IMG_FMT_64bppRGBAHalfFloat && fmt != UHDR_IMG_FMT_32bppRGBA1010102)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid output format %d, expects one of {UHDR_IMG_FMT_32bppRGBA8888,  "
               "UHDR_IMG_FMT_64bppRGBAHalfFloat, UHDR_IMG_FMT_32bppRGBA1010102}", fmt);
  DEC_PROBED_CHECK
  h->out_fmt = fmt;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_dec_set_out_color_transfer(uhdr_codec_private_t* dec, uhdr_color_transfer_t ct) {
  DEC_PROLOGUE
  if (ct != UHDR_CT_HLG && ct != UHDR_CT_PQ && ct != UHDR_CT_LINEAR && ct != UHDR_CT_SRGB)
    return err(UHDR_CODEC_INVALID_PARAM, "invalid output color transfer %d, expects one of {UHDR_CT_HLG, UHDR_CT_PQ, UHDR_CT_LINEAR, UHDR_CT_SRGB}", ct);
  DEC_PROBED_CHECK
  h->out_ct = ct;
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_dec_set_out_max_display_boost(uhdr_codec_private_t* dec, float boost) {
  DEC_PROLOGUE
  if (!std::isfinite(boost) || boost < 1.0f) return err(UHDR_CODEC_INVALID_PARAM, "invalid display boost %f, expects to be >= 1.0f}", boost);
  DEC_PROBED_CHECK
  h->max_boost = boost;
  return ok();
}

UHDR_API uhdr_error_info_t uhdr_dec_probe(uhdr_codec_private_t* dec) {
  DEC_PROLOGUE
  if (h->stream.empty()) return err(UHDR_CODEC_INVALID_OPERATION, "did not receive any image for decoding");
  if (h->probed) return h->probe_status;
  h->probed = true;
  int rc = h->codec.probe(h->stream.data(), h->stream.size(), &h->info);
  h->probe_status = from_rc(rc);
  if (rc == E_OK) {
    auto blk = [](const ByteView& v, uhdr_mem_block_t* b) { b->data = const_cast<uint8_t*>(v.data); b->data_sz = b->capacity = v.size; };
    blk(h->info.exif, &h->exif_blk);
    blk(h->info.icc, &h->icc_blk);
    // the compressed base / gain-map images are views into the handle's copy of the stream
    h->base_blk.data = h->stream.data() + h->info.base_off;
    h->base_blk.data_sz = h->base_blk.capacity = h->info.base_len;
    h->gm_blk.data = h->stream.data() + h->info.gainmap_off;
    h->gm_blk.data_sz = h->gm_blk.capacity = h->info.gainmap_len;
  }
  return h->probe_status;
}
#define DEC_GETTER(cond, val, bad)                              \
  Decoder* h = as<Decoder>(dec);                                \
  if (!h || !h->probed || h->probe_status.error_code != UHDR_CODEC_OK || !(cond)) return bad; \
  return val;
UHDR_API int uhdr_dec_get_image_width(uhdr_codec_private_t* dec) { DEC_GETTER(true, h->info.width, -1) }
UHDR_API int uhdr_dec_get_image_height(uhdr_codec_private_t* dec) { DEC_GETTER(true, h->info.height, -1) }
UHDR_API int uhdr_dec_get_gainmap_width(uhdr_codec_private_t* dec) { DEC_GETTER(true, h->info.gm_width, -1) }
UHDR_API int uhdr_dec_get_gainmap_height(uhdr_codec_private_t* dec) { DEC_GETTER(true, h->info.gm_height, -1) }
UHDR_API uhdr_mem_block_t* uhdr_dec_get_exif(uhdr_codec_private_t* dec) { DEC_GETTER(true, &h->exif_blk, nullptr) }
UHDR_API uhdr_mem_block_t* uhdr_dec_get_icc(uhdr_codec_private_t* dec) { DEC_GETTER(true, &h->icc_blk, nullptr) }
UHDR_API uhdr_mem_block_t* uhdr_dec_get_base_image(uhdr_codec_private_t* dec) { DEC_GETTER(true, &h->base_blk, nullptr) }
UHDR_API uhdr_mem_block_t* uhdr_dec_get_gainmap_image(uhdr_codec_private_t* dec) { DEC_GETTER(true, &h->gm_blk, nullptr) }
UHDR_API uhdr_gainmap_metadata_t* uhdr_dec_get_gainmap_metadata(uhdr_codec_private_t* dec) { DEC_GETTER(h->info.has_metadata, &h->info.metadata, nullptr) }

UHDR_API uhdr_error_info_t uhdr_decode(uhdr_codec_private_t* dec) {
  DEC_PROLOGUE
  if (h->sailed) return h->status;
  h->status = uhdr_dec_probe(dec);
  if (h->status.error_code != UHDR_CODEC_OK) return h->status;
  h->sailed = true;
  if ((h->out_fmt == UHDR_IMG_FMT_32bppRGBA1010102 && h->out_ct != UHDR_CT_HLG && h->out_ct != UHDR_CT_PQ) ||
      (h->out_fmt == UHDR_IMG_FMT_64bppRGBAHalfFloat && h->out_ct != UHDR_CT_LINEAR) ||
      (h->out_fmt == UHDR_IMG_FMT_32bppRGBA8888 && h->out_ct != UHDR_CT_SRGB)) {
    h->status = err(UHDR_CODEC_INVALID_PARAM, "unsupported output pixel format and output color transfer pair");
    return h->status;
  }
  // image effects (:1996-1998, :289-429): planned from the probed sizes, so every error comes before device work
  const bool fx = !h->effects.empty();
  ImageMap fx_img{}, fx_map{};
  if (fx) {
    const int rc = plan_decoder_effects(h->effects.data(), (int)h->effects.size(), h->info.width, h->info.height,
                                        h->info.gm_width, h->info.gm_height, &fx_img, &fx_map);
    if (rc) { h->status = from_rc(rc); return h->status; }
  }
  h->ensure();
  if (h->init_rc) { h->status = err((uhdr_codec_err_t)h->init_rc, "%s", h->init_err.c_str()); return h->status; }
  const int w = h->info.width, ht = h->info.height;
  const size_t bpp = h->out_fmt == UHDR_IMG_FMT_64bppRGBAHalfFloat ? 8 : 4;
  // the pixel buffers come from the codec's pinned arena (allocated inside decode()): a zero-filled
  // pageable vector of w*h*8 bytes would cost more than the whole decode
  (void)bpp;
  memset(&h->decoded_desc, 0, sizeof h->decoded_desc);
  h->decoded_desc.fmt = (uhdr_img_fmt_t)h->out_fmt;
  h->decoded_desc.cg = UHDR_CG_UNSPECIFIED;
  h->decoded_desc.ct = (uhdr_color_transfer_t)h->out_ct;
  h->decoded_desc.range = UHDR_CR_UNSPECIFIED;
  h->decoded_desc.w = w;
  h->decoded_desc.h = ht;
  h->decoded_desc.planes[0] = nullptr;
  h->decoded_desc.stride[0] = w;
  memset(&h->gainmap_desc, 0, sizeof h->gainmap_desc);
  h->gainmap_desc.planes[0] = nullptr;
  h->gainmap_desc.stride[0] = h->info.gm_width;
  h->codec.set_lazy_gainmap(true);  // the map leaves HBM only if uhdr_get_decoded_gainmap_image() is called
  int rc = h->codec.decode(h->stream.data(), h->stream.size(), h->out_ct, h->out_fmt, h->max_boost, &h->decoded_desc,
                           &h->gainmap_desc, nullptr, &h->info,   // uhdr_dec_probe above already located the two images
                           fx ? &fx_img : nullptr, fx ? &fx_map : nullptr);
  h->status = from_rc(rc);
  return h->status;
}
UHDR_API uhdr_raw_image_t* uhdr_get_decoded_image(uhdr_codec_private_t* dec) {
  Decoder* h = as<Decoder>(dec);
  if (!h || !h->sailed || h->status.error_code != UHDR_CODEC_OK) return nullptr;
  return &h->decoded_desc;
}
UHDR_API uhdr_raw_image_t* uhdr_get_decoded_gainmap_image(uhdr_codec_private_t* dec) {
  Decoder* h = as<Decoder>(dec);
  if (!h || !h->sailed || h->status.error_code != UHDR_CODEC_OK) return nullptr;
  if (!h->gainmap_desc.planes[0]) {
    h->bind();
    if (h->codec.fetch_gainmap(&h->gainmap_desc) != E_OK) return nullptr;
  }
  return &h->gainmap_desc;
}
UHDR_API void uhdr_reset_decoder(uhdr_codec_private_t* dec) {
  Decoder* h = as<Decoder>(dec);
  if (h) h->defaults();
}

// ---- common --------------------------------------------------------------------------------------
UHDR_API uhdr_error_info_t uhdr_enable_gpu_acceleration(uhdr_codec_private_t* codec, int) {
  if (!codec) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
  return ok();  // the CUDA path is the only path
}
// uhdr_add_effect_*, ultrahdr_api.cpp:2113-2229: arguments are checked here, sizes when the handle sails
#define EFFECT_NULL_CHECK \
  if (!codec) return err(UHDR_CODEC_INVALID_PARAM, "received nullptr for uhdr codec instance");
static uhdr_error_info_t add_effect(uhdr_codec_private_t* codec, const Effect& e) {
  if (codec->sailed)
    return err(UHDR_CODEC_INVALID_OPERATION, "An earlier call to uhdr_encode()/uhdr_decode() has switched the context "
               "from configurable state to end state. The context is no longer configurable. To reuse, call reset()");
  codec->effects.push_back(e);
  return ok();
}
UHDR_API uhdr_error_info_t uhdr_add_effect_mirror(uhdr_codec_private_t* codec, uhdr_mirror_direction_t direction) {
  EFFECT_NULL_CHECK
  if (direction != UHDR_MIRROR_HORIZONTAL && direction != UHDR_MIRROR_VERTICAL)
    return err(UHDR_CODEC_INVALID_PARAM, "unsupported direction, expects one of {UHDR_MIRROR_HORIZONTAL, UHDR_MIRROR_VERTICAL}");
  return add_effect(codec, Effect{FX_MIRROR, (int)direction, 0, 0, 0});
}
UHDR_API uhdr_error_info_t uhdr_add_effect_rotate(uhdr_codec_private_t* codec, int degrees) {
  EFFECT_NULL_CHECK
  if (degrees != 90 && degrees != 180 && degrees != 270)
    return err(UHDR_CODEC_INVALID_PARAM, "unsupported degrees, expects one of {90, 180, 270}");
  return add_effect(codec, Effect{FX_ROTATE, degrees, 0, 0, 0});
}
UHDR_API uhdr_error_info_t uhdr_add_effect_crop(uhdr_codec_private_t* codec, int left, int right, int top, int bottom) {
  EFFECT_NULL_CHECK
  return add_effect(codec, Effect{FX_CROP, left, right, top, bottom});
}
UHDR_API uhdr_error_info_t uhdr_add_effect_resize(uhdr_codec_private_t* codec, int width, int height) {
  EFFECT_NULL_CHECK
  return add_effect(codec, Effect{FX_RESIZE, width, height, 0, 0});
}

// ---- measurement hooks (include/uhdr_b200.h) -------------------------------------------------------
UHDR_API void uhdr_b200_set_kernel_timing(int on) { set_kernel_timing(on != 0); }
UHDR_API void uhdr_b200_entropy_decoder_stats(unsigned long long out[3]) { jpeg_entropy_decoder_stats(out); }
UHDR_API int uhdr_b200_set_entropy_decoder(int mode) {
  const int prev = jpeg_get_entropy_decoder();
  jpeg_set_entropy_decoder(mode);
  return prev;
}
UHDR_API int uhdr_b200_kernel_timing_report(char* buf, size_t cap, int reset) {
  const std::string r = kernel_timing_report(reset != 0);
  if (r.size() + 1 > cap) return -(int)r.size();
  memcpy(buf, r.c_str(), r.size() + 1);
  return (int)r.size();
}
UHDR_API size_t uhdr_b200_trim_cache(void) { return trim_parked_blocks(); }
UHDR_API int uhdr_b200_enc_rearm(uhdr_codec_private_t* enc) {
  Encoder* h = as<Encoder>(enc);
  if (!h) return fail(E_INVALID_PARAM, "received nullptr for uhdr codec instance");
  h->sailed = false;
  h->status = ok();
  return E_OK;
}

// ---- stage-level JPEG entry points (include/uhdr_b200.h) ---------------------------------------------
static JpegRCodec* tls_codec() {
  static thread_local JpegRCodec* c = nullptr;
  if (!c) {
    c = new JpegRCodec();
    if (c->init() != E_OK) { delete c; c = nullptr; }
  }
  if (c) c->ws().rewind();
  return c;
}

UHDR_API int uhdr_b200_jpeg_forward(const uhdr_raw_image_t* img, int quality, int16_t* coefs[3]) {
  JpegRCodec* c = tls_codec();
  if (!c) return E_ERROR;
  DevImage d;
  int rc = upload_image(c->ws(), *img, &d);
  if (rc) return rc;
  JpegEncodeJob job;
  rc = jpeg_forward_dev(c->ws(), d, quality, &job);
  if (rc) return rc;
  for (int k = 0; k < job.frame.ncomp; k++)
    CUDA_TRY(cudaMemcpyAsync(coefs[k], job.d_coefs[k], job.frame.blocks(k) * 128, cudaMemcpyDeviceToHost, c->ws().stream()));
  return c->ws().sync();
}

UHDR_API int uhdr_b200_jpeg_encode(const uhdr_raw_image_t* img, int quality, const void* icc, size_t icc_size, void* out,
                                   size_t cap, size_t* out_size) {
  JpegRCodec* c = tls_codec();
  if (!c) return E_ERROR;
  DevImage d;
  int rc = upload_image(c->ws(), *img, &d);
  if (rc) return rc;
  JpegEncodeJob job;
  rc = jpeg_forward_dev(c->ws(), d, quality, &job, /*zigzag=*/true);
  if (rc) return rc;
  rc = jpeg_entropy_dev(c->ws(), &job);
  if (rc) return rc;
  rc = c->ws().sync();
  if (rc) return rc;
  rc = jpeg_entropy_fetch(c->ws(), &job);
  if (rc) return rc;
  rc = c->ws().sync();
  if (rc) return rc;
  std::vector<uint8_t> s;
  const bool gm = img->fmt == UHDR_IMG_FMT_24bppRGB888 || img->fmt == UHDR_IMG_FMT_8bppYCbCr400;
  rc = jpeg_finish_stream(job, icc, icc_size, gm ? jpeg_gainmap_comment() : nullptr, &s);
  if (rc) return rc;
  if (s.size() > cap) return fail(E_MEM, "output buffer too small: need %zu bytes", s.size());
  memcpy(out, s.data(), s.size());
  *out_size = s.size();
  return E_OK;
}

UHDR_API int uhdr_b200_jpeg_decode(const void* data, size_t size, int mode, uhdr_raw_image_t* out, size_t cap) {
  JpegRCodec* c = tls_codec();
  if (!c) return E_ERROR;
  DevImage d;
  JpegHeader h;
  int rc = c->decode_jpeg_dev((const uint8_t*)data, size, mode, &d, &h);
  if (rc) return rc;
  // host layout of JpegDecoderHelper::getDecompressedImage (:536-552)
  const JpegFrame& f = h.frame;
  uint8_t* base = (uint8_t*)out->planes[0];
  out->fmt = (uhdr_img_fmt_t)d.v.fmt;
  out->w = d.v.w;
  out->h = d.v.h;
  out->cg = UHDR_CG_UNSPECIFIED;
  out->ct = UHDR_CT_UNSPECIFIED;
  out->range = UHDR_CR_FULL_RANGE;
  size_t need = 0;
  if (d.v.fmt == F_RGBA8888) {
    need = (size_t)d.v.w * d.v.h * 4;
    if (need > cap) return fail(E_MEM, "output buffer too small: need %zu bytes", need);
    out->stride[0] = d.v.w;
    out->planes[1] = out->planes[2] = nullptr;
    out->stride[1] = out->stride[2] = 0;
    rc = download_image(c->ws(), d, out);
  } else {
    unsigned hs[3] = {0, 0, 0}, vs[3] = {0, 0, 0};
    for (int k = 0; k < f.ncomp; k++) {
      hs[k] = (f.comp[k].width + f.max_h - 1) / f.max_h * f.max_h;
      vs[k] = (f.comp[k].height + f.max_v - 1) / f.max_v * f.max_v;
      need += (size_t)hs[k] * vs[k];
    }
    if (need > cap) return fail(E_MEM, "output buffer too small: need %zu bytes", need);
    memset(base, 0, need);
    uint8_t* p = base;
    for (int k = 0; k < 3; k++) {
      out->planes[k] = p;
      out->stride[k] = hs[k];
      if (k < f.ncomp) {
        const size_t wbytes = (hs[k] % 8 == 0) ? hs[k] : (size_t)f.comp[k].width;
        const size_t rows = std::min<size_t>(vs[k], (size_t)f.comp[k].hblocks * 8);
        CUDA_TRY(cudaMemcpy2DAsync(p, hs[k], d.v.p[k], d.v.stride[k], wbytes, rows, cudaMemcpyDeviceToHost, c->ws().stream()));
      }
      p += (size_t)hs[k] * vs[k];
    }
  }
  if (rc) return rc;
  return c->ws().sync();
}

UHDR_API int uhdr_b200_encode_batch(int n, const uhdr_raw_image_t* hdr, const uhdr_raw_image_t* sdr,
                                    const uhdr_b200_gm_config_t* cfg, int base_quality, uhdr_compressed_image_t* out,
                                    int streams) {
  if (n <= 0 || !hdr || !cfg || !out) return fail(E_INVALID_PARAM, "bad batch arguments");
  if (streams < 1) streams = 1;
  if (streams > n) streams = n;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  // one worker (host thread + codec + stream) per pipeline slot; frames are dealt round robin.
  // While one worker assembles a stream on the CPU the others keep the copy engines and SMs busy.
  static thread_local std::vector<std::unique_ptr<JpegRCodec>> pool;
  while ((int)pool.size() < streams) {
    pool.emplace_back(new JpegRCodec());
    int rc = pool.back()->init();
    if (rc) { pool.pop_back(); return rc; }
  }
  std::vector<int> rcs(streams, 0);
  std::vector<std::string> errs(streams);
  std::vector<std::thread> th;
  // `pool` is thread_local: a worker naming it would see its own (empty) instance, so the workers get
  // the caller's codecs through a plain pointer
  std::unique_ptr<JpegRCodec>* codecs = pool.data();
  for (int s = 0; s < streams; s++)
    th.emplace_back([&, s, codecs]() {
      if (cudaSetDevice(dev) != cudaSuccess) { rcs[s] = E_ERROR; errs[s] = "cudaSetDevice failed in a batch worker"; return; }
      for (int i = s; i < n; i += streams) {
        size_t sz = 0;
        int rc = codecs[s]->encode_host(hdr[i], sdr ? &sdr[i] : nullptr, *cfg, base_quality, nullptr, 0,
                                      (uint8_t*)out[i].data, out[i].capacity, &sz);
        out[i].data_sz = sz;
        if (rc) { rcs[s] = rc; errs[s] = last_error(); return; }
      }
    });
  for (auto& t : th) t.join();
  for (int s = 0; s < streams; s++)
    if (rcs[s]) { set_last_error(errs[s]); return rcs[s]; }
  return E_OK;
}

}  // extern "C"
