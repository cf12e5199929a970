// Host planner of the image effects (effects.h).  Each effect maps an output coordinate of its plane to a
// coordinate of its input with an integer affine map, optionally transposed; composing the maps of a chain
// is exact integer arithmetic, so the composed gather reads the very element the reference's chain of
// buffer copies would have carried there.
#include "effects.h"

#include <algorithm>
#include <cstdlib>

namespace uhdr_b200 {

namespace {

constexpr int kMaxDim = 8192;  // ultrahdr::kMaxWidth / kMaxHeight

// (int)v for every v the checks below can accept; saturates where the plain cast would be undefined
int to_int(float v) { return v >= 2147483520.0f ? 2147483647 : v <= -2147483648.0f ? (-2147483647 - 1) : (int)v; }

struct Chain {  // one plane's composed map while a chain is walked
  long long w0, h0;  // source plane size
  long long w, h;    // current size
  long long ax = 1, bx = 0, ay = 1, by = 0;
  int swap = 0;
  Chain(long long w_, long long h_) : w0(w_), h0(h_), w(w_), h(h_) {}

  // append one effect whose output (x, y) reads input (cx*s + dx, cy*t + dy), (s, t) = sk ? (y, x) : (x, y)
  void then(int sk, long long cx, long long dx, long long cy, long long dy, long long nw, long long nh) {
    long long ax2, bx2, ay2, by2;
    if (!swap) { ax2 = ax * cx; bx2 = ax * dx + bx; ay2 = ay * cy; by2 = ay * dy + by; }
    else       { ax2 = ax * cy; bx2 = ax * dy + bx; ay2 = ay * cx; by2 = ay * dx + by; }
    ax = ax2; bx = bx2; ay = ay2; by = by2;
    swap ^= sk;
    w = nw; h = nh;
  }
  // editorhelper.cpp:20-86
  void rotate(int deg) {
    if (deg == 90) then(1, 1, 0, -1, h - 1, h, w);            // dst[i][j] = src[h-1-j][i]
    else if (deg == 180) then(0, -1, w - 1, -1, h - 1, w, h);  // dst[i][j] = src[h-1-i][w-1-j]
    else then(1, -1, w - 1, 1, 0, h, w);                       // dst[i][j] = src[j][w-1-i]
  }
  void mirror(int dir) {
    if (dir == UHDR_MIRROR_VERTICAL) then(0, 1, 0, -1, h - 1, w, h);
    else then(0, -1, w - 1, 1, 0, w, h);
  }
  void crop(long long left, long long top, long long wd, long long ht) { then(0, 1, left, 1, top, wd, ht); }
  // resize_buffer: integer ratios, so an upscale reads element (0, 0) everywhere
  void resize(long long dw, long long dh) { then(0, w / dw, 0, h / dh, 0, dw, dh); }

  // the composed map is affine in each output coordinate: its extremes are at the corners
  int finish(PlaneMap* p) const {
    const long long smax = (swap ? h : w) - 1, tmax = (swap ? w : h) - 1;
    const long long x0 = bx, x1 = ax * smax + bx, y0 = by, y1 = ay * tmax + by;
    if (w <= 0 || h <= 0 || std::min(x0, x1) < 0 || std::max(x0, x1) >= w0 || std::min(y0, y1) < 0 ||
        std::max(y0, y1) >= h0 || std::max({std::llabs(ax), std::llabs(ay)}) > kMaxDim * 2LL)
      return fail(E_ERROR, "image effects: composed map leaves the %lldx%lld source plane", w0, h0);
    p->w = (int)w; p->h = (int)h;
    p->ax = (int)ax; p->bx = (int)bx; p->ay = (int)ay; p->by = (int)by;
    return E_OK;
  }
};

// the planes of a format the effects are applied to: false = full size, true = half size (4:2:0 chroma, P010 UV)
int layout(int fmt, int* nplanes, bool half[3]) {
  half[0] = half[1] = half[2] = false;
  switch (fmt) {
    case F_P010: *nplanes = 2; half[1] = true; return E_OK;
    case F_YUV420: *nplanes = 3; half[1] = half[2] = true; return E_OK;
    case F_Y400: case F_RGBA8888: case F_RGBA1010102: case F_RGBAF16: *nplanes = 1; return E_OK;
  }
  return fail(E_UNSUPPORTED, "image effects: unsupported image format %d", fmt);
}

int emit(const Chain& full, const Chain* half_chain, int fmt, ImageMap* m) {
  bool half[3];
  int rc = layout(fmt, &m->nplanes, half);
  if (rc) return rc;
  m->src_w = (int)full.w0; m->src_h = (int)full.h0;
  m->w = (int)full.w; m->h = (int)full.h;
  m->transposed = full.swap;
  for (int i = 0; i < m->nplanes; i++) {
    rc = (half[i] ? *half_chain : full).finish(&m->plane[i]);
    if (rc) return rc;
  }
  return E_OK;
}

}  // namespace

int plan_encoder_effects(const Effect* fx, int n, int hdr_fmt, int sdr_fmt, int w, int h, ImageMap* hdr, ImageMap* sdr) {
  const bool p010 = hdr_fmt == F_P010, yuv420 = sdr_fmt == F_YUV420;
  Chain full(w, h), half(w / 2, h / 2);  // half: only walked when a plane uses it (then every size is even)
  const bool want_half = p010 || yuv420;
  for (int k = 0; k < n; k++) {
    const Effect& e = fx[k];
    if (e.kind == FX_ROTATE) {
      full.rotate(e.a);
      if (want_half) half.rotate(e.a);
    } else if (e.kind == FX_MIRROR) {
      full.mirror(e.a);
      if (want_half) half.mirror(e.a);
    } else if (e.kind == FX_CROP) {  // ultrahdr_api.cpp:150-224: clamped to the current hdr intent
      const long long left = std::max(0, e.a), right = std::min<long long>(full.w, e.b);
      const long long cw = right - left;
      if (cw <= 0)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop width is expected to be > 0, crop width is %d", (int)cw);
      if (cw % 2 != 0 && p010)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop width is expected to even for format "
                    "{UHDR_IMG_FMT_24bppYCbCrP010}, crop width is %d", (int)cw);
      const long long top = std::max(0, e.c), bottom = std::min<long long>(full.h, e.d);
      const long long ch = bottom - top;
      if (ch <= 0)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop height is expected to be > 0, crop height is %d", (int)ch);
      if (ch % 2 != 0 && p010)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop height is expected to even for format "
                    "{UHDR_IMG_FMT_24bppYCbCrP010}. crop height is %d", (int)ch);
      if (cw % 2 != 0 && yuv420)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop width is expected to even for format "
                    "{UHDR_IMG_FMT_12bppYCbCr420}, crop width is %d", (int)cw);
      if (ch % 2 != 0 && yuv420)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop height is expected to even for format "
                    "{UHDR_IMG_FMT_12bppYCbCr420}. crop height is %d", (int)ch);
      full.crop(left, top, cw, ch);
      if (want_half) half.crop(left / 2, top / 2, cw / 2, ch / 2);  // an odd left / top rounds down on the chroma plane
    } else if (e.kind == FX_RESIZE) {  // :225-264
      const int dw = e.a, dh = e.b;
      if (dw <= 0 || dh <= 0 || dw > kMaxDim || dh > kMaxDim)
        return fail(E_INVALID_PARAM, "destination dimensions must be in range (0, %d] x (0, %d]. dest image width "
                    "is %d, dest image height is %d", kMaxDim, kMaxDim, dw, dh);
      if ((dw % 2 != 0 || dh % 2 != 0) && p010)
        return fail(E_INVALID_PARAM, "destination dimensions cannot be odd for format {UHDR_IMG_FMT_24bppYCbCrP010}. "
                    "dest image width is %d, dest image height is %d", dw, dh);
      if ((dw % 2 != 0 || dh % 2 != 0) && yuv420)
        return fail(E_INVALID_PARAM, "destination dimensions cannot be odd for format {UHDR_IMG_FMT_12bppYCbCr420}. "
                    "dest image width is %d, dest image height is %d", dw, dh);
      full.resize(dw, dh);
      if (want_half) half.resize(dw / 2, dh / 2);
    } else {
      return fail(E_INVALID_PARAM, "unknown image effect %d", e.kind);
    }
  }
  int rc = emit(full, &half, hdr_fmt, hdr);
  if (rc == E_OK && sdr_fmt >= 0) rc = emit(full, &half, sdr_fmt, sdr);
  return rc;
}

int plan_decoder_effects(const Effect* fx, int n, int w, int h, int map_w, int map_h, ImageMap* img, ImageMap* map) {
  Chain im(w, h), gm(map_w, map_h);
  for (int k = 0; k < n; k++) {
    const Effect& e = fx[k];
    if (e.kind == FX_ROTATE) {
      im.rotate(e.a);
      gm.rotate(e.a);
    } else if (e.kind == FX_MIRROR) {
      im.mirror(e.a);
      gm.mirror(e.a);
    } else if (e.kind == FX_CROP) {  // ultrahdr_api.cpp:326-387
      const int left = std::max(0, e.a), right = std::min((int)im.w, e.b);
      if (right <= left)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop right is <= crop left, after crop image width is %d",
                    right - left);
      const int top = std::max(0, e.c), bottom = std::min((int)im.h, e.d);
      if (bottom <= top)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop bottom is <= crop top, after crop image height is %d",
                    bottom - top);
      // the map's rectangle, in float as the reference computes it
      const float wd_ratio = ((float)im.w) / gm.w, ht_ratio = ((float)im.h) / gm.h;
      const int gm_left = (int)(left / wd_ratio), gm_right = (int)(right / wd_ratio);
      if (gm_right <= gm_left)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop right is <= crop left for gainmap image, after "
                    "crop gainmap image width is %d", gm_right - gm_left);
      const int gm_top = (int)(top / ht_ratio), gm_bottom = (int)(bottom / ht_ratio);
      if (gm_bottom <= gm_top)
        return fail(E_INVALID_PARAM, "unexpected crop dimensions. crop bottom is <= crop top for gainmap image, after "
                    "crop gainmap image height is %d", gm_bottom - gm_top);
      im.crop(left, top, right - left, bottom - top);
      gm.crop(gm_left, gm_top, gm_right - gm_left, gm_bottom - gm_top);
    } else if (e.kind == FX_RESIZE) {  // :388-415
      const int dw = e.a, dh = e.b;
      const float wd_ratio = ((float)im.w) / gm.w, ht_ratio = ((float)im.h) / gm.h;
      const int dgw = to_int(dw / wd_ratio), dgh = to_int(dh / ht_ratio);
      if (dw <= 0 || dh <= 0 || dgw <= 0 || dgh <= 0 || dw > kMaxDim || dh > kMaxDim || dgw > kMaxDim || dgh > kMaxDim)
        return fail(E_INVALID_PARAM, "destination dimension must be in range (0, %d] x (0, %d]. dest image width is "
                    "%d, dest image height is %d, dest gainmap width is %d, dest gainmap height is %d",
                    kMaxDim, kMaxDim, dw, dh, dgw, dgh);
      im.resize(dw, dh);
      gm.resize(dgw, dgh);
    } else {
      return fail(E_INVALID_PARAM, "unknown image effect %d", e.kind);
    }
  }
  // both are packed single-plane images (RGBA output, Y400 / RGBA8888 map)
  int rc = emit(im, nullptr, F_RGBA8888, img);
  if (rc == E_OK) rc = emit(gm, nullptr, F_Y400, map);
  return rc;
}

}  // namespace uhdr_b200
