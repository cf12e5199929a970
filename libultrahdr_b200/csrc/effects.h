// Image effects of the C API (uhdr_add_effect_*): rotate, mirror, crop and resize, as the reference's
// editorhelper.cpp:20-86 buffer loops.  Every effect is an integer index map from output pixel to source
// pixel, so a whole chain composes into one map per plane and runs as one gather per image.
//
// The host planner walks the chain over the current sizes, applies the reference's validation ladders
// (encoder ultrahdr_api.cpp:131-283, decoder :289-429) and composes the maps; it does no device work,
// so every error is found before the device is touched.
#pragma once
#include "engine.h"

namespace uhdr_b200 {

enum : int { FX_MIRROR = 0, FX_ROTATE = 1, FX_CROP = 2, FX_RESIZE = 3 };
struct Effect {  // one uhdr_add_effect_* call, arguments as given
  int kind;
  int a, b, c, d;  // mirror: direction | rotate: degrees | crop: left, right, top, bottom | resize: width, height
};

// Output element (x, y) of a plane reads source element (ax*s + bx, ay*t + by), where (s, t) is (y, x)
// when the image's map is transposed (an odd number of 90/270 rotations) and (x, y) otherwise.
struct PlaneMap {
  int w, h;        // output size in elements
  int ax, bx, ay, by;
};
struct ImageMap {  // one image: every plane of it, all with the same orientation
  int src_w, src_h, w, h;  // input and output size (the format is unchanged by effects)
  int transposed;
  int nplanes;
  PlaneMap plane[3];
};

// Encoder chain on the raw intents (API-0: sdr_fmt < 0).  E_INVALID_PARAM with the reference's text when
// a crop or resize is rejected.
int plan_encoder_effects(const Effect* fx, int n, int hdr_fmt, int sdr_fmt, int w, int h, ImageMap* hdr, ImageMap* sdr);
// Decoder chain on the decoded image and its gain map; the map follows the image through the reference's
// float ratios of the two sizes.
int plan_decoder_effects(const Effect* fx, int n, int w, int h, int map_w, int map_h, ImageMap* img, ImageMap* map);

// Enqueues the gather of `src` through `m` into a new image from alloc_dev_image(..., 64).  Columns between
// a plane's width and its stride are written as zeros.  `src` is only read.
int apply_effects_dev(Workspace& ws, const DevImage& src, const ImageMap& m, DevImage* out);

}  // namespace uhdr_b200
