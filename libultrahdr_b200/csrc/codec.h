// Codec orchestration: the B200 counterpart of ultrahdr::JpegR (lib/include/ultrahdr/jpegr.h:52-222).
// encodeJPEGR API-0 / API-1 and decodeJPEGR run their pixel and block stages on the device;
// the marker/container layer is host code.
#pragma once
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "container.h"
#include "effects.h"
#include "engine.h"
#include "jpeg.h"

namespace uhdr_b200 {

struct DecodedInfo {
  int width = 0, height = 0, gm_width = 0, gm_height = 0;
  ByteView exif, icc;   // views into the probed stream (the caller keeps it alive: the C API handle owns a copy)
  size_t base_off = 0, base_len = 0, gainmap_off = 0, gainmap_len = 0;  // the two JPEGs inside the probed stream
  uhdr_gainmap_metadata_t metadata{};
  bool has_metadata = false;
};

// One parked host thread per codec (spawned on first use, kept until the codec dies): runs the gain-map JPEG of a
// decode next to the primary one without creating a thread per call.
class ParkedThread {
 public:
  ~ParkedThread();
  void start(void (*fn)(void*), void* arg);   // fn(arg) on the parked thread
  void wait();                                // until that call has returned
 private:
  void loop();
  std::thread th_;
  std::mutex mu_;
  std::condition_variable cv_;
  void (*fn_)(void*) = nullptr;
  void* arg_ = nullptr;
  bool busy_ = false, quit_ = false;
};

class JpegRCodec {
 public:
  int init() { return ws_.init(); }
  Workspace& ws() { return ws_; }

  // JpegR::encodeJPEGR API-1 (jpegr.cpp:247-291) when sdr_dev != nullptr, API-0 (:179-244)
  // otherwise.  Inputs are device images previously uploaded on ws().stream().
  int encode(const DevImage& hdr, const DevImage* sdr, const uhdr_b200_gm_config_t& cfg, int base_quality,
             const uint8_t* exif, size_t exif_size, uint8_t* out, size_t cap, size_t* out_size);
  // JpegR::encodeJPEGR API-2 (jpegr.cpp:294-324, sdr != nullptr) / API-3 (:326-386, the compressed SDR is
  // decoded on the device and the map is computed with BT.601 luma): gain map from the intents, its JPEG,
  // appended to the caller's compressed SDR image.  `sdr_jpg_cg`: gamut of the compressed image when it
  // carries no ICC profile.
  int encode_with_compressed_sdr(const DevImage& hdr, const DevImage* sdr, const uint8_t* sdr_jpg, size_t sdr_jpg_size,
                                 int sdr_jpg_cg, const uhdr_b200_gm_config_t& cfg, uint8_t* out, size_t cap, size_t* out_size);
  // API-4 (:388-434): container work only, no device
  static int encode_from_compressed(const uint8_t* base, size_t base_size, int base_cg, const uint8_t* gainmap, size_t gainmap_size,
                                    const uhdr_gainmap_metadata_t& md, uint8_t* out, size_t cap, size_t* out_size);
  // convenience: host descriptors
  int encode_host(const uhdr_raw_image_t& hdr, const uhdr_raw_image_t* sdr, const uhdr_b200_gm_config_t& cfg,
                  int base_quality, const uint8_t* exif, size_t exif_size, uint8_t* out, size_t cap,
                  size_t* out_size);

  // JpegR::getJPEGRInfo (jpegr.cpp:1417-1430): sizes, exif/icc, metadata; no pixel work
  int probe(const uint8_t* data, size_t size, DecodedInfo* info);
  // JpegR::decodeJPEGR (jpegr.cpp:1469-1531).  dest: host descriptor with planes allocated by the
  // caller (fmt/stride set); gainmap_out optional host descriptor (planes allocated, Y400/RGBA8888).
  // `probed`: the result of probe() on the same stream (saves the second scan of the container), or null.
  // `fx_img` / `fx_map`: image effects planned for the decoded image and the gain map (plan_decoder_effects),
  // or null.  With effects the descriptors report the transformed size at stride ALIGNM(w, 64).
  int decode(const uint8_t* data, size_t size, int out_ct, int out_fmt, float max_display_boost,
             uhdr_raw_image_t* dest, uhdr_raw_image_t* gainmap_out, uhdr_gainmap_metadata_t* md_out,
             const DecodedInfo* probed = nullptr, const ImageMap* fx_img = nullptr, const ImageMap* fx_map = nullptr);

  // With gainmap_out->planes[0] == nullptr and lazy_gainmap set, decode() only fills the descriptor's
  // geometry and keeps the map in HBM; fetch_gainmap() copies it out when somebody asks for it
  // (uhdr_get_decoded_gainmap_image).  Valid until the next decode() on this codec.
  void set_lazy_gainmap(bool on) { lazy_gainmap_ = on; }
  int fetch_gainmap(uhdr_raw_image_t* gainmap_out);

  // JpegDecoderHelper::decompressImage equivalent producing a device image
  int decode_jpeg_dev(const uint8_t* data, size_t size, int mode, DevImage* out, JpegHeader* hdr) {
    return decode_jpeg_dev(ws_, data, size, mode, out, hdr);
  }
  ~JpegRCodec();

 private:
  int decode_jpeg_dev(Workspace& ws, const uint8_t* data, size_t size, int mode, DevImage* out, JpegHeader* hdr);
  Workspace ws_;
  // second stream + arenas: the gain-map JPEG of a decode is processed by a helper thread while the
  // calling thread handles the primary image (both entropy decoders alternate host and device phases)
  std::unique_ptr<Workspace> ws2_;
  ParkedThread helper_;
  cudaEvent_t map_ready_ = nullptr;
  bool lazy_gainmap_ = false, map_pending_ = false;
  DevImage last_map_{};
};


}  // namespace uhdr_b200
