// The gather behind the image effects (effects.h): one launch per image covers all of its planes.  Pure data
// movement, so the design goal is coalesced traffic on both sides:
//   * untransposed maps (mirror, crop, resize, rotate 180): each thread writes 16 B of one output row; its
//     source elements lie on one source row (reversed for a mirror, strided or repeated for a resize);
//   * transposed maps (a rotate 90 / 270 in the chain): 32x32-element tiles through padded shared memory, so
//     that the source is read along its rows and the destination written along its rows.
#include <cstdint>

#include "effects.h"

namespace uhdr_b200 {

namespace {

constexpr int kThreads = 256;
constexpr int kTile = 32;

struct FxPlane {
  const uint8_t* src;
  uint8_t* dst;
  int src_stride, dst_stride;  // in elements
  int w, h;                    // output size; columns [w, dst_stride) receive zeros
  int ax, bx, ay, by;          // PlaneMap
  int esz;                     // element size in bytes: 1, 2, 4 or 8
  int block_end;               // cumulative block count up to and including this plane
};
struct FxParams {
  FxPlane p[3];
  int nplanes, transposed;
};

template <class T>
__device__ __forceinline__ void gather_rows(const FxPlane& P, int blk) {
  constexpr int N = 16 / sizeof(T);
  const int chunks = P.dst_stride / N;  // 16-byte chunks per output row
  const long long g = (long long)blk * kThreads + threadIdx.x;
  if (g >= (long long)chunks * P.h) return;
  const int y = (int)(g / chunks);
  const int x0 = (int)(g - (long long)y * chunks) * N;
  const T* srow = reinterpret_cast<const T*>(P.src) + (size_t)(P.ay * y + P.by) * P.src_stride;
  uint32_t word[4] = {0, 0, 0, 0};
#pragma unroll
  for (int k = 0; k < N; k++) {
    const int x = x0 + k;
    const unsigned long long e = x < P.w ? (unsigned long long)__ldg(srow + P.ax * x + P.bx) : 0ull;
    constexpr int bits = 8 * sizeof(T);
    if (bits == 64) {
      word[2 * k] = (uint32_t)e;
      word[2 * k + 1] = (uint32_t)(e >> 32);
    } else {
      word[k * bits / 32] |= (uint32_t)e << (k * bits % 32);
    }
  }
  *reinterpret_cast<uint4*>(reinterpret_cast<T*>(P.dst) + (size_t)y * P.dst_stride + x0) =
      make_uint4(word[0], word[1], word[2], word[3]);
}

// output (x, y) = source (ax*y + bx, ay*x + by): an output row is a source column
template <class T>
__device__ __forceinline__ void gather_tiles(const FxPlane& P, int blk, T* tile) {
  const int tiles_x = (P.dst_stride + kTile - 1) / kTile;
  const int x0 = (blk % tiles_x) * kTile, y0 = (blk / tiles_x) * kTile;
  const int tx = threadIdx.x % kTile, ty = threadIdx.x / kTile;
  const T* src = reinterpret_cast<const T*>(P.src);
  T* dst = reinterpret_cast<T*>(P.dst);
  // tile[i][j] = output (x0 + i, y0 + j); consecutive tx read consecutive source columns
  for (int i = ty; i < kTile; i += kThreads / kTile) {
    const int x = x0 + i, y = y0 + tx;
    if (x < P.w && y < P.h) tile[i * (kTile + 1) + tx] = __ldg(src + (size_t)(P.ay * x + P.by) * P.src_stride + P.ax * y + P.bx);
  }
  __syncthreads();
  for (int j = ty; j < kTile; j += kThreads / kTile) {
    const int x = x0 + tx, y = y0 + j;
    if (y < P.h && x < P.dst_stride) dst[(size_t)y * P.dst_stride + x] = x < P.w ? tile[tx * (kTile + 1) + j] : T(0);
  }
}

template <class T>
__device__ __forceinline__ void gather(const FxPlane& P, int blk, bool transposed, uint64_t* smem) {
  if (transposed) gather_tiles<T>(P, blk, reinterpret_cast<T*>(smem));
  else gather_rows<T>(P, blk);
}

__global__ void __launch_bounds__(kThreads, 4) k_effects_gather(const __grid_constant__ FxParams p) {
  __shared__ uint64_t smem[kTile * (kTile + 1)];
  // the block's plane, selected without a dynamic index into the parameter block (that would go through the stack)
  const int b = blockIdx.x;
  const int i = b < p.p[0].block_end || p.nplanes == 1 ? 0 : (b < p.p[1].block_end || p.nplanes == 2 ? 1 : 2);
  const FxPlane P = i == 0 ? p.p[0] : i == 1 ? p.p[1] : p.p[2];
  const int blk = b - (i == 0 ? 0 : i == 1 ? p.p[0].block_end : p.p[1].block_end);
  switch (P.esz) {  // uniform per block
    case 1: gather<uint8_t>(P, blk, p.transposed, smem); break;
    case 2: gather<uint16_t>(P, blk, p.transposed, smem); break;
    case 4: gather<uint32_t>(P, blk, p.transposed, smem); break;
    default: gather<uint64_t>(P, blk, p.transposed, smem); break;
  }
}

// element size of plane i as the reference's buffer loops move it: the P010 UV plane as 32-bit (U, V) pairs
int element_size(int fmt, int i) {
  switch (fmt) {
    case F_P010: return i == 0 ? 2 : 4;
    case F_YUV420: case F_Y400: return 1;
    case F_RGBA8888: case F_RGBA1010102: return 4;
    case F_RGBAF16: return 8;
  }
  return 0;
}

}  // namespace

int apply_effects_dev(Workspace& ws, const DevImage& src, const ImageMap& m, DevImage* out) {
  const int fmt = src.v.fmt;
  if (src.v.w != m.src_w || src.v.h != m.src_h || fmt_planes(fmt) != m.nplanes || element_size(fmt, 0) == 0)
    return fail(E_ERROR, "image effects: planned for a %dx%d image with %d planes, got %dx%d format %d", m.src_w, m.src_h,
                m.nplanes, src.v.w, src.v.h, fmt);
  int rc = alloc_dev_image(ws, fmt, m.w, m.h, 64, out);
  if (rc) return rc;
  out->cg = src.cg;
  out->ct = src.ct;
  out->range = src.range;
  out->v.full_range = src.v.full_range;
  FxParams p{};
  p.nplanes = m.nplanes;
  p.transposed = m.transposed;
  int blocks = 0;
  for (int i = 0; i < m.nplanes; i++) {
    FxPlane& q = p.p[i];
    const PlaneMap& pm = m.plane[i];
    q.esz = element_size(fmt, i);
    const int per = fmt == F_P010 && i == 1 ? 2 : 1;  // ImgView strides of the P010 UV plane count 16-bit samples
    q.src = static_cast<const uint8_t*>(src.v.p[i]);
    q.dst = static_cast<uint8_t*>(const_cast<void*>(out->v.p[i]));
    q.src_stride = src.v.stride[i] / per;
    q.dst_stride = out->v.stride[i] / per;
    q.w = pm.w; q.h = pm.h;
    q.ax = pm.ax; q.bx = pm.bx; q.ay = pm.ay; q.by = pm.by;
    // 16-byte row stores: alloc_dev_image's strides (64 or 32 elements) and arena alignment guarantee it
    if ((size_t)q.dst_stride * q.esz % 16 != 0 || reinterpret_cast<uintptr_t>(q.dst) % 16 != 0)
      return fail(E_ERROR, "image effects: destination plane %d is not 16-byte aligned", i);
    if (m.transposed)
      blocks += ((q.dst_stride + kTile - 1) / kTile) * ((q.h + kTile - 1) / kTile);
    else
      blocks += (int)(((long long)(q.dst_stride * q.esz / 16) * q.h + kThreads - 1) / kThreads);
    q.block_end = blocks;
  }
  count_launches(1);
  TIMED(ws, "effects_gather", (k_effects_gather<<<blocks, kThreads, 0, ws.stream()>>>(p), cudaGetLastError()));
  return E_OK;
}

}  // namespace uhdr_b200
