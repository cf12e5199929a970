#include "codec.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include <cmath>
#include <cstring>
#include <thread>

namespace uhdr_b200 {

static ByteView find_marker(const uint8_t* d, const JpegHeader& h, uint8_t id, const char* sig, size_t sig_len);

// ------------------------------------------------------------------------------------------------
// encode
// ------------------------------------------------------------------------------------------------
// forward block stage + entropy coding, both on the device for every geometry (MCUs that reach past
// the block grid included: huffman.cu codes libjpeg's dummy blocks)
static int block_stage(Workspace& ws, const DevImage& img, int quality, JpegEncodeJob* job) {
  int rc = jpeg_forward_dev(ws, img, quality, job, /*zigzag=*/true);
  if (rc) return rc;
  return jpeg_entropy_dev(ws, job);
}

int JpegRCodec::encode(const DevImage& hdr, const DevImage* sdr_in, const uhdr_b200_gm_config_t& cfg_in,
                       int base_quality, const uint8_t* exif, size_t exif_size, uint8_t* out, size_t cap,
                       size_t* out_size) {
  uhdr_b200_gm_config_t cfg = cfg_in;
  DevImage sdr;
  int rc;
  if (sdr_in) {
    sdr = *sdr_in;
  } else {
    // API-0: tone map first (jpegr.cpp:181-213); preset forced to REALTIME, max-RGB gain
    int sdr_fmt;
    if (hdr.v.fmt == F_P010) sdr_fmt = F_YUV420;
    else if (hdr.v.fmt == F_YUV444_10) sdr_fmt = F_YUV444;
    else if (hdr.v.fmt == F_RGBA1010102 || hdr.v.fmt == F_RGBAF16) sdr_fmt = F_RGBA8888;
    else return fail(E_INVALID_PARAM, "unsupported hdr intent color format %d", hdr.v.fmt);
    rc = alloc_dev_image(ws_, sdr_fmt, hdr.v.w, hdr.v.h, 64, &sdr);
    if (rc) return rc;
    rc = tonemap_dev(ws_, hdr, &sdr);
    if (rc) return rc;
    cfg.preset = UHDR_USAGE_REALTIME;
    cfg.sdr_is_601 = 0;
    cfg.use_luminance = 0;
  }
  GainmapJob gm;
  rc = generate_gainmap_dev(ws_, sdr, hdr, cfg, 64, &gm);
  if (rc) return rc;
  JpegEncodeJob gm_jpeg, base_jpeg;
  rc = block_stage(ws_, gm.map, cfg.quality, &gm_jpeg);
  if (rc) return rc;
  // base image: icc of the sdr intent's gamut is chosen before the yuv re-encoding (:260)
  const int sdr_cg = sdr.cg;
  if (fmt_is_rgb_host(sdr.v.fmt)) {  // convert_raw_input_to_ycbcr (:221-228, :263-271)
    DevImage ycc;
    rc = rgb_to_ycbcr_dev(ws_, sdr, &ycc);
    if (rc) return rc;
    sdr = ycc;
  }
  if (sdr_in) {
    // :277.  `sdr` may be the caller's resident input (uhdr_enc_set_raw_image uploads once, the handle
    // can be encoded again): never convert it in place
    rc = convert_yuv_dev(ws_, &sdr, sdr.cg, UHDR_CG_DISPLAY_P3, /*in_place=*/false);
    if (rc) return rc;
  }
  rc = block_stage(ws_, sdr, base_quality, &base_jpeg);
  if (rc) return rc;
  rc = ws_.sync();
  if (rc) return rc;
  if (gm_jpeg.h_scan_bytes || base_jpeg.h_scan_bytes) {  // sizes are known now: fetch the segments
    if (gm_jpeg.h_scan_bytes && (rc = jpeg_entropy_fetch(ws_, &gm_jpeg))) return rc;
    if (base_jpeg.h_scan_bytes && (rc = jpeg_entropy_fetch(ws_, &base_jpeg))) return rc;
    rc = ws_.sync();
    if (rc) return rc;
  }
  uhdr_gainmap_metadata_t md;
  finish_gainmap_metadata(gm, &md);
  size_t icc_gm_n = 0, icc_base_n = 0;
  const uint8_t* icc_gm = icc_profile(gm.map.ct, gm.map.cg, &icc_gm_n);  // compressGainMap :520-528
  const uint8_t* icc_base = icc_profile(UHDR_CT_SRGB, sdr_cg, &icc_base_n);
  // the two JPEG heads are written into the workspace's host arena: no heap on this path
  JpegPieces pg, pb;
  const size_t gm_cap = jpeg_head_capacity(icc_gm_n, jpeg_gainmap_comment()), base_cap = jpeg_head_capacity(icc_base_n, nullptr);
  uint8_t* gm_head = (uint8_t*)ws_.halloc(gm_cap);
  uint8_t* base_head = (uint8_t*)ws_.halloc(base_cap);
  if (!gm_head || !base_head) return E_MEM;
  rc = jpeg_stream_pieces(gm_jpeg, icc_gm, icc_gm_n, jpeg_gainmap_comment(), gm_head, gm_cap, &pg.head_len, &pg.scan, &pg.scan_len);
  if (rc) return rc;
  rc = jpeg_stream_pieces(base_jpeg, icc_base, icc_base_n, nullptr, base_head, base_cap, &pb.head_len, &pb.scan, &pb.scan_len);
  if (rc) return rc;
  pg.head = gm_head;
  pb.head = base_head;
  return assemble_jpegr(pb, pg, exif, exif_size, md, out, cap, out_size);
}

int JpegRCodec::encode_from_compressed(const uint8_t* base, size_t base_size, int base_cg, const uint8_t* gainmap, size_t gainmap_size,
                                       const uhdr_gainmap_metadata_t& md, uint8_t* out, size_t cap, size_t* out_size) {
  JpegHeader bh;
  int rc = jpeg_read_header(base, base_size, &bh);  // parseImage :392
  if (rc) return rc;
  ByteView blob;
  if (!md.use_base_cg) {
    JpegHeader gh;
    rc = jpeg_read_header(gainmap, gainmap_size, &gh);
    if (rc) return rc;
    blob = find_marker(gainmap, gh, 0xE2, "ICC_PROFILE", 12);
    if (blob.empty())
      return fail(E_UNSUPPORTED, "For gainmap application space to be alternate image space, gainmap image is expected to "
                  "contain alternate image color space in the form of ICC. The ICC marker in gainmap jpeg is missing.");
  }
  blob = find_marker(base, bh, 0xE2, "ICC_PROFILE", 12);
  const uint8_t* icc = nullptr;
  size_t icc_n = 0;
  if (blob.empty()) {  // add ICC if not already present
    if (base_cg <= UHDR_CG_UNSPECIFIED || base_cg > UHDR_CG_BT_2100) return fail(E_INVALID_PARAM, "Unrecognized 420 color gamut %d", base_cg);
    icc = icc_profile(UHDR_CT_SRGB, base_cg, &icc_n);
  }
  JpegPieces pb, pg;
  pb.head = base; pb.head_len = base_size; pb.scan = nullptr; pb.scan_len = 0; pb.whole = true;
  pg.head = gainmap; pg.head_len = gainmap_size; pg.scan = nullptr; pg.scan_len = 0; pg.whole = true;
  return assemble_jpegr(pb, pg, nullptr, 0, md, out, cap, out_size, icc, icc_n);
}

int JpegRCodec::encode_with_compressed_sdr(const DevImage& hdr, const DevImage* sdr_in, const uint8_t* sdr_jpg, size_t sdr_jpg_size,
                                           int sdr_jpg_cg, const uhdr_b200_gm_config_t& cfg_in, uint8_t* out, size_t cap,
                                           size_t* out_size) {
  uhdr_b200_gm_config_t cfg = cfg_in;
  DevImage sdr;
  int rc;
  if (sdr_in) {  // API-2: only the size of the compressed image is looked at (PARSE_STREAM :297-311)
    JpegHeader h;
    rc = jpeg_read_header(sdr_jpg, sdr_jpg_size, &h);
    if (rc) return rc;
    if (hdr.v.w != h.frame.width || hdr.v.h != h.frame.height)
      return fail(E_INVALID_PARAM, "sdr intent resolution %dx%d and compressed image sdr intent resolution %dx%d do not match",
                  sdr_in->v.w, sdr_in->v.h, h.frame.width, h.frame.height);
    sdr = *sdr_in;
    cfg.sdr_is_601 = 0;
  } else {       // API-3: decode the input JPEG; its YCbCr encoding is BT.601
    JpegHeader h;
    rc = decode_jpeg_dev(ws_, sdr_jpg, sdr_jpg_size, 0, &sdr, &h);
    if (rc) return rc;
    const ByteView blob = find_marker(sdr_jpg, h, 0xE2, "ICC_PROFILE", 12);
    if (!blob.empty()) {
      const int cg = icc_read_gamut(blob.data, blob.size);
      if (cg == UHDR_CG_UNSPECIFIED || (sdr_jpg_cg != UHDR_CG_UNSPECIFIED && sdr_jpg_cg != cg))
        return fail(E_INVALID_PARAM, "configured color gamut %d does not match with color gamut specified in icc box %d", sdr_jpg_cg, cg);
      sdr.cg = cg;
    } else {
      if (sdr_jpg_cg <= UHDR_CG_UNSPECIFIED || sdr_jpg_cg > UHDR_CG_BT_2100) return fail(E_INVALID_PARAM, "Unrecognized 420 color gamut %d", sdr_jpg_cg);
      sdr.cg = sdr_jpg_cg;
    }
    if (hdr.v.w != sdr.v.w || hdr.v.h != sdr.v.h)
      return fail(E_INVALID_PARAM, "sdr intent resolution %dx%d and hdr intent resolution %dx%d do not match", sdr.v.w, sdr.v.h,
                  hdr.v.w, hdr.v.h);
    cfg.sdr_is_601 = 1;
  }
  cfg.use_luminance = 1;
  GainmapJob gm;
  rc = generate_gainmap_dev(ws_, sdr, hdr, cfg, 64, &gm);
  if (rc) return rc;
  JpegEncodeJob gm_jpeg;
  rc = block_stage(ws_, gm.map, cfg.quality, &gm_jpeg);
  if (rc) return rc;
  rc = ws_.sync();
  if (rc) return rc;
  if ((rc = jpeg_entropy_fetch(ws_, &gm_jpeg))) return rc;
  rc = ws_.sync();
  if (rc) return rc;
  uhdr_gainmap_metadata_t md;
  finish_gainmap_metadata(gm, &md);
  size_t icc_gm_n = 0;
  const uint8_t* icc_gm = icc_profile(gm.map.ct, gm.map.cg, &icc_gm_n);
  const size_t gm_cap = jpeg_head_capacity(icc_gm_n, jpeg_gainmap_comment()) + gm_jpeg.h_scan_bytes[3] + 2;
  uint8_t* gm_file = (uint8_t*)ws_.halloc(gm_cap);
  if (!gm_file) return E_MEM;
  size_t gm_file_n = 0;
  rc = jpeg_finish_stream_into(gm_jpeg, icc_gm, icc_gm_n, jpeg_gainmap_comment(), gm_file, gm_cap, &gm_file_n);
  if (rc) return rc;
  return encode_from_compressed(sdr_jpg, sdr_jpg_size, sdr_jpg_cg, gm_file, gm_file_n, md, out, cap, out_size);
}

int JpegRCodec::encode_host(const uhdr_raw_image_t& hdr, const uhdr_raw_image_t* sdr,
                            const uhdr_b200_gm_config_t& cfg, int base_quality, const uint8_t* exif,
                            size_t exif_size, uint8_t* out, size_t cap, size_t* out_size) {
  ws_.rewind();
  DevImage dh, ds;
  int rc = upload_image(ws_, hdr, &dh);
  if (rc) return rc;
  if (sdr) {
    rc = upload_image(ws_, *sdr, &ds);
    if (rc) return rc;
  }
  return encode(dh, sdr ? &ds : nullptr, cfg, base_quality, exif, exif_size, out, cap, out_size);
}

// ------------------------------------------------------------------------------------------------
// decode
// ------------------------------------------------------------------------------------------------
static int sampling_format(const JpegFrame& f) {  // jpegdecoderhelper.cpp:141-166
  if (f.ncomp == 1) return F_Y400;
  float r[6];
  for (int i = 0; i < 3; i++) {
    r[i * 2] = ((float)f.comp[i].h_samp) / f.max_h;
    r[i * 2 + 1] = ((float)f.comp[i].v_samp) / f.max_v;
  }
  if (r[0] == 1 && r[1] == 1 && r[2] == r[4] && r[3] == r[5]) {
    if (r[2] == 1 && r[3] == 1) return F_YUV444;
    if (r[2] == 1 && r[3] == 0.5) return 8;   // 440
    if (r[2] == 0.5 && r[3] == 1) return F_YUV422;
    if (r[2] == 0.5 && r[3] == 0.5) return F_YUV420;
    if (r[2] == 0.25 && r[3] == 1) return 9;  // 411
    if (r[2] == 0.25 && r[3] == 0.5) return 10;
  }
  return -1;
}

static int validate_header(const JpegHeader& h) {  // jpegdecoderhelper.cpp:244-342
  const JpegFrame& f = h.frame;
  if (f.width < 1 || f.height < 1)
    return fail(E_ERROR, "received bad image width or height, wd = %d, ht = %d. wd and height shall be >= 1", f.width, f.height);
  if (f.width > 8192 || f.height > 8192)
    return fail(E_ERROR, "max width, max supported by library are %d, %d respectively. Current image width and height are %d, %d. "
                "Recompile library with updated max supported dimensions to proceed", 8192, 8192, f.width, f.height);
  if (f.ncomp != 1 && f.ncomp != 3)
    return fail(E_ERROR, "ultrahdr primary image and supplimentary images are images encoded with 1 component (grayscale) "
                "or 3 components (YCbCr / RGB). Unrecognized number of components %d", f.ncomp);
  for (int i = 0, product = 0; i < f.ncomp; i++) {
    if (f.comp[i].h_samp < 1 || f.comp[i].h_samp > 4 || f.comp[i].v_samp < 1 || f.comp[i].v_samp > 4)
      return fail(E_ERROR, "received bad sampling factor for component index %d", i);
    product += f.comp[i].h_samp * f.comp[i].v_samp;
    if (product > 10) return fail(E_ERROR, "received bad sampling factors for components, sum of product of h_samp_factor, "
                                  "v_samp_factor across all components exceeds 10");
  }
  if (f.ncomp == 3) {
    if (f.comp[1].width > f.comp[0].width || f.comp[2].height > f.comp[0].height)
      return fail(E_ERROR, "cb, cr planes are upsampled wrt luma plane");
    if (f.comp[1].width != f.comp[2].width || f.comp[1].height != f.comp[2].height)
      return fail(E_ERROR, "cb, cr planes are not sampled identically");
  }
  return E_OK;
}

// first marker `id` whose payload starts with `sig`, as a view into the stream (jpegdecoderhelper.cpp:119-139 copies it)
static ByteView find_marker(const uint8_t* d, const JpegHeader& h, uint8_t id, const char* sig, size_t sig_len) {
  ByteView v;
  for (const JpegMarker& m : h.markers)
    if (m.id == id && m.length > sig_len && !memcmp(d + m.offset, sig, sig_len)) {
      v.data = d + m.offset;
      v.size = m.length;
      break;
    }
  return v;
}

ParkedThread::~ParkedThread() {
  if (!th_.joinable()) return;
  {
    std::lock_guard<std::mutex> lk(mu_);
    quit_ = true;
  }
  cv_.notify_all();
  th_.join();
}
void ParkedThread::loop() {
  std::unique_lock<std::mutex> lk(mu_);
  for (;;) {
    cv_.wait(lk, [&] { return quit_ || (busy_ && fn_); });
    if (quit_) return;
    void (*fn)(void*) = fn_;
    void* arg = arg_;
    fn_ = nullptr;
    lk.unlock();
    fn(arg);
    lk.lock();
    busy_ = false;
    cv_.notify_all();
  }
}
void ParkedThread::start(void (*fn)(void*), void* arg) {
  std::unique_lock<std::mutex> lk(mu_);
  if (!th_.joinable()) th_ = std::thread([this] { loop(); });
  fn_ = fn;
  arg_ = arg;
  busy_ = true;
  cv_.notify_all();
}
void ParkedThread::wait() {
  std::unique_lock<std::mutex> lk(mu_);
  cv_.wait(lk, [&] { return !busy_; });
}

JpegRCodec::~JpegRCodec() {
  if (map_ready_) cudaEventDestroy(map_ready_);
}

int JpegRCodec::decode_jpeg_dev(Workspace& ws, const uint8_t* data, size_t size, int mode, DevImage* out, JpegHeader* h) {
  if (!data) return fail(E_INVALID_PARAM, "received nullptr for compressed image data");
  if (size == 0) return fail(E_INVALID_PARAM, "received bad compressed image size %zd", size);
  int rc = jpeg_read_header(data, size, h);
  if (rc) return rc;
  rc = validate_header(*h);
  if (rc) return rc;
  const JpegFrame& f = h->frame;
  if (mode == 2) mode = f.ncomp == 1 ? 0 : 1;  // DECODE_STREAM :344-346
  if (h->adobe_transform == 0 && f.ncomp == 3)
    return fail(E_UNSUPPORTED, "RGB (Adobe transform 0) JPEG input is not supported by the B200 decoder");
  if (mode == 1 && f.ncomp == 1) return fail(E_ERROR, "expected input color space to be JCS_YCbCr or JCS_RGB but got %d", 1);
  memset(out, 0, sizeof *out);
  out->cg = out->ct = -1;
  out->range = UHDR_CR_FULL_RANGE;
  out->v.full_range = 1;
  out->v.w = f.width;
  out->v.h = f.height;
  uint8_t* planes[3] = {nullptr, nullptr, nullptr};
  int strides[3] = {0, 0, 0};
  for (int c = 0; c < f.ncomp; c++) {
    strides[c] = f.comp[c].wblocks * 8;
    planes[c] = (uint8_t*)ws.dalloc((size_t)strides[c] * f.comp[c].hblocks * 8);
    if (!planes[c]) return E_MEM;
  }
  // entropy decoding: on the device (huffdec.cu).  The host decoder is not a size-based alternative: it runs only
  // for streams the parallel decoder declines (restart markers, no fixed point, inconsistent data -- it also
  // produces the reference's error texts for those) or when a test / triage session selects it (mode 1).
  const int dec_mode = jpeg_get_entropy_decoder();
  bool on_device = dec_mode != 1;
  if (on_device) {
    int16_t* d_coefs[3] = {nullptr, nullptr, nullptr};
    rc = jpeg_entropy_decode_dev(ws, data, size, *h, d_coefs);
    if (rc == kHuffDecFallback) on_device = false;
    else if (rc) return rc;
    else rc = jpeg_idct_dev(ws, *h, d_coefs, planes, strides);
    if (on_device && rc) return rc;
  }
  if (!on_device) {
    int16_t* h_coefs[3] = {nullptr, nullptr, nullptr};
    for (int c = 0; c < f.ncomp; c++) {
      h_coefs[c] = (int16_t*)ws.halloc(f.blocks(c) * 128);
      if (!h_coefs[c]) return E_MEM;
    }
    rc = jpeg_host_decode_coefs(data, size, *h, h_coefs);
    if (rc) return rc;
    rc = jpeg_inverse_dev(ws, *h, h_coefs, planes, strides);
    if (rc) return rc;
  }
  if (mode == 1) {
    const bool s444 = f.max_h == 1 && f.max_v == 1, s422 = f.max_h == 2 && f.max_v == 1, s420 = f.max_h == 2 && f.max_v == 2;
    if (!(s444 || s422 || s420) || f.comp[0].h_samp != f.max_h || f.comp[0].v_samp != f.max_v || f.comp[1].h_samp != 1 ||
        f.comp[1].v_samp != 1 || f.comp[2].h_samp != 1 || f.comp[2].v_samp != 1)
      return fail(E_UNSUPPORTED, "RGB output is implemented for 4:4:4, 4:2:2 and 4:2:0 JPEG input");
    DevImage rgba;
    rc = alloc_dev_image(ws, F_RGBA8888, f.width, f.height, 1, &rgba);
    if (rc) return rc;
    YccToRgbaParams p;
    p.y = planes[0]; p.cb = planes[1]; p.cr = planes[2];
    p.src_stride = strides[0];
    p.w = f.width;
    p.h = f.height;
    p.hs = f.max_h;
    p.vs = f.max_v;
    p.c_stride = strides[1];
    p.cw = (f.width + f.max_h - 1) / f.max_h;
    p.ch = (f.height + f.max_v - 1) / f.max_v;
    p.dst = (uint8_t*)rgba.v.p[0];
    p.dst_stride = rgba.v.stride[0];
    TIMED(ws, "ycc_to_rgba", launch_ycc_to_rgba(p, ws.stream()));
    rgba.range = UHDR_CR_FULL_RANGE;
    *out = rgba;
    out->cg = out->ct = -1;
    return E_OK;
  }
  const int fmt = sampling_format(f);
  if (fmt < 0) return fail(E_ERROR, "unrecognized subsampling format for output color space JCS_YCbCr");
  out->v.fmt = fmt;
  for (int c = 0; c < f.ncomp; c++) {
    out->v.p[c] = planes[c];
    out->v.stride[c] = strides[c];
  }
  return E_OK;
}

int JpegRCodec::probe(const uint8_t* data, size_t size, DecodedInfo* info) {
  size_t po, pl, go, gl;
  int rc = split_jpegr(data, size, &po, &pl, &go, &gl);
  if (rc) return rc;
  JpegHeader ph, gh;
  rc = jpeg_read_header(data + po, pl, &ph);
  if (rc) return rc;
  rc = validate_header(ph);
  if (rc) return rc;
  rc = jpeg_read_header(data + go, gl, &gh);
  if (rc) return rc;
  rc = validate_header(gh);
  if (rc) return rc;
  info->width = ph.frame.width;
  info->height = ph.frame.height;
  info->gm_width = gh.frame.width;
  info->gm_height = gh.frame.height;
  info->base_off = po; info->base_len = pl;
  info->gainmap_off = go; info->gainmap_len = gl;
  info->exif = find_marker(data + po, ph, 0xE1, "Exif\0\0", 6);   // views into the caller's stream
  info->icc = find_marker(data + po, ph, 0xE2, "ICC_PROFILE", 12);
  const ByteView iso = find_marker(data + go, gh, 0xE2, "urn:iso:std:iso:ts:21496:-1", 28);
  const ByteView xmp = find_marker(data + go, gh, 0xE1, "http://ns.adobe.com/xap/1.0/", 29);
  rc = parse_gainmap_metadata(iso.data, iso.size, xmp.data, xmp.size, info->exif.data, info->exif.size, &info->metadata);
  if (rc) return rc;
  info->has_metadata = true;
  return E_OK;
}

int JpegRCodec::decode(const uint8_t* data, size_t size, int out_ct, int out_fmt, float max_display_boost,
                       uhdr_raw_image_t* dest, uhdr_raw_image_t* gainmap_out, uhdr_gainmap_metadata_t* md_out,
                       const DecodedInfo* probed, const ImageMap* fx_img, const ImageMap* fx_map) {
  (void)out_fmt;
  PhaseTrace tr;
  ws_.rewind();
  size_t po, pl, go, gl;
  int rc = E_OK;
  if (probed && probed->base_len && probed->gainmap_len && probed->gainmap_off + probed->gainmap_len <= size) {
    po = probed->base_off; pl = probed->base_len; go = probed->gainmap_off; gl = probed->gainmap_len;
  } else {
    rc = split_jpegr(data, size, &po, &pl, &go, &gl);
  }
  if (rc) return rc;
  tr.mark("container split");
  const bool sdr_only = out_ct == UHDR_CT_SRGB;  // :1479-1481, :1520-1523: the base image as RGBA8888, no gain map applied
  DevImage sdr, map;
  JpegHeader ph, gh;
  const bool want_map = gainmap_out || !sdr_only;  // :1484-1495
  // both images sizeable: the gain-map JPEG goes to a helper thread with its own stream
  const bool overlap = want_map && pl >= (256u << 10) && gl >= (256u << 10);
  struct MapJob {   // lives on this frame until helper_.wait() below
    JpegRCodec* self;
    const uint8_t* data;
    size_t len;
    DevImage* map;
    JpegHeader* gh;
    int dev, rc;
    char err[256];
  } mj{this, data + go, gl, &map, &gh, 0, E_OK, {0}};
  if (overlap) {
    if (!ws2_) {
      ws2_.reset(new Workspace());
      rc = ws2_->init();
      if (rc) { ws2_.reset(); return rc; }
      CUDA_TRY(cudaEventCreateWithFlags(&map_ready_, cudaEventDisableTiming));
    }
    ws2_->rewind();
    CUDA_TRY(cudaGetDevice(&mj.dev));
    helper_.start([](void* a) {
      MapJob& j = *static_cast<MapJob*>(a);
      auto fail_with = [&](int rc, const char* what) { j.rc = rc; snprintf(j.err, sizeof j.err, "%s", what); };
      if (cudaSetDevice(j.dev) != cudaSuccess) return fail_with(E_ERROR, "cudaSetDevice failed in the gain-map decode thread");
      j.rc = j.self->decode_jpeg_dev(*j.self->ws2_, j.data, j.len, 2, j.map, j.gh);  // DECODE_STREAM :1486
      if (j.rc) snprintf(j.err, sizeof j.err, "%s", last_error());
      else if (cudaEventRecord(j.self->map_ready_, j.self->ws2_->stream()) != cudaSuccess) fail_with(E_ERROR, "cudaEventRecord failed");
    }, &mj);
  }
  rc = decode_jpeg_dev(ws_, data + po, pl, sdr_only ? 1 : 0, &sdr, &ph);  // DECODE_TO_RGB_CS / DECODE_TO_YCBCR_CS
  if (overlap) helper_.wait();
  if (rc) return rc;
  tr.mark("primary jpeg enqueued");
  ByteView blob = find_marker(data + po, ph, 0xE2, "ICC_PROFILE", 12);
  sdr.cg = icc_read_gamut(blob.data, blob.size);
  map_pending_ = false;
  uhdr_gainmap_metadata_t md{};
  if (want_map) {
    if (overlap) {
      if (mj.rc) { set_last_error(mj.err); return mj.rc; }
      CUDA_TRY(cudaStreamWaitEvent(ws_.stream(), map_ready_, 0));
      if (kernel_timing_enabled()) ws2_->sync();
    } else {
      rc = decode_jpeg_dev(ws_, data + go, gl, 2, &map, &gh);  // DECODE_STREAM :1486
      if (rc) return rc;
    }
    blob = find_marker(data + go, gh, 0xE2, "ICC_PROFILE", 12);
    map.cg = icc_read_gamut(blob.data, blob.size);
    tr.mark("gainmap jpeg enqueued");
  }
  if (md_out || !sdr_only) {  // :1497-1518
    // the reference reads the gain-map image's markers only when it decodes that image (:1484-1495):
    // metadata alone with SDR output finds no buffer to parse
    if (!want_map) return fail(E_INVALID_PARAM, "received no valid buffer to parse gainmap metadata");
    blob = find_marker(data + go, gh, 0xE2, "urn:iso:std:iso:ts:21496:-1", 28);
    const ByteView xmp = find_marker(data + go, gh, 0xE1, "http://ns.adobe.com/xap/1.0/", 29);
    const ByteView exif = find_marker(data + po, ph, 0xE1, "Exif\0\0", 6);
    rc = parse_gainmap_metadata(blob.data, blob.size, xmp.data, xmp.size, exif.data, exif.size, &md);
    if (rc) return rc;
    if (md_out) *md_out = md;
  }
  if (gainmap_out) {
    DevImage gm = map;  // `map` itself stays as decoded: the gain map is applied untransformed
    if (fx_map) {
      rc = apply_effects_dev(ws_, map, *fx_map, &gm);
      if (rc) return rc;
    }
    const int gm_stride = fx_map ? gm.v.stride[0] : gm.v.w;
    gainmap_out->fmt = (uhdr_img_fmt_t)gm.v.fmt;
    gainmap_out->w = gm.v.w;
    gainmap_out->h = gm.v.h;
    gainmap_out->cg = UHDR_CG_UNSPECIFIED;
    gainmap_out->ct = UHDR_CT_UNSPECIFIED;
    gainmap_out->range = UHDR_CR_FULL_RANGE;
    if (!gainmap_out->planes[0] && lazy_gainmap_) {
      gainmap_out->stride[0] = gm_stride;
      last_map_ = gm;
      map_pending_ = true;
    } else {
      if (!gainmap_out->planes[0]) {  // handle-owned result: pinned memory of this codec, valid until its next decode
        gainmap_out->stride[0] = gm_stride;
        gainmap_out->planes[0] = ws_.halloc((size_t)gm_stride * gm.v.h * (gm.v.fmt == F_Y400 ? 1 : 4));
        if (!gainmap_out->planes[0]) return E_MEM;
      }
      rc = download_image(ws_, gm, gainmap_out);
      if (rc) return rc;
    }
  }
  DevImage dst;
  if (sdr_only) {  // copy_raw_image(&sdr_intent, dest) :1520-1523
    if (dest->fmt != UHDR_IMG_FMT_32bppRGBA8888)
      return fail(E_INVALID_PARAM, "unsupported output pixel format and output color transfer pair");
    dst = sdr;
    dest->cg = (uhdr_color_gamut_t)sdr.cg;
    dest->ct = UHDR_CT_UNSPECIFIED;
  } else {
    rc = alloc_dev_image(ws_, dest->fmt, sdr.v.w, sdr.v.h, 64, &dst);
    if (rc) return rc;
    rc = apply_gainmap_dev(ws_, sdr, map, md, out_ct, max_display_boost, &dst);
    if (rc) return rc;
    dest->cg = (uhdr_color_gamut_t)dst.cg;
    dest->ct = (uhdr_color_transfer_t)out_ct;
  }
  dest->range = UHDR_CR_FULL_RANGE;
  const size_t bpp = dest->fmt == UHDR_IMG_FMT_64bppRGBAHalfFloat ? 8 : 4;
  if (fx_img) {
    // the effects run on the device image, and only their result crosses to the host; the gather wrote
    // whole rows up to the stride (zeros past the width), so they go as one linear copy
    DevImage fx;
    rc = apply_effects_dev(ws_, dst, *fx_img, &fx);
    if (rc) return rc;
    const size_t bytes = (size_t)fx.v.stride[0] * fx.v.h * bpp;
    dest->w = fx.v.w;
    dest->h = fx.v.h;
    if (!dest->planes[0]) {
      dest->stride[0] = fx.v.stride[0];
      dest->planes[0] = ws_.halloc(bytes);
      if (!dest->planes[0]) return E_MEM;
    }
    tr.mark("apply + effects enqueued");
    if ((int)dest->stride[0] == fx.v.stride[0])
      CUDA_TRY(cudaMemcpyAsync(dest->planes[0], fx.v.p[0], bytes, cudaMemcpyDeviceToHost, ws_.stream()));
    else if ((rc = download_image(ws_, fx, dest)))
      return rc;
  } else {
    if (!dest->planes[0]) {  // handle-owned result (see above)
      dest->stride[0] = sdr.v.w;
      dest->planes[0] = ws_.halloc((size_t)sdr.v.w * sdr.v.h * bpp);
      if (!dest->planes[0]) return E_MEM;
    }
    tr.mark("apply enqueued");
    rc = download_image(ws_, dst, dest);
    if (rc) return rc;
  }
  rc = ws_.sync();
  tr.mark("pixels on the host");
  return rc;
}

int JpegRCodec::fetch_gainmap(uhdr_raw_image_t* gainmap_out) {
  if (!map_pending_) return E_OK;
  gainmap_out->planes[0] = ws_.halloc((size_t)gainmap_out->stride[0] * last_map_.v.h * (last_map_.v.fmt == F_Y400 ? 1 : 4));
  if (!gainmap_out->planes[0]) return E_MEM;
  int rc = download_image(ws_, last_map_, gainmap_out);
  if (rc) return rc;
  map_pending_ = false;
  return ws_.sync();
}

}  // namespace uhdr_b200
