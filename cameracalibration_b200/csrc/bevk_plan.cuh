// bevk_plan.cuh -- the tile-plan compiler of the fused BEV kernel: pure host code (no CUDA calls), so that
// bevk_bev_finalize (bevk_api.cu) and the CPU tests (tests/host/kernel_math.cu) share one implementation.
//
// Input: per camera the BEV LUT planes  bev_map1 (int16 x,y) / bev_map2 (uint16 fraction)  that
// Camera.get_bev_maps builds (SurroundBirdEyeView/surroundBEV.py:105-108) and the camera's mask
// (Mask / BlendMask, :119-280).  Output: canvas tiles of 32x32 px, per tile the cameras that touch it
// (reference camera order), per (tile, camera) a block of 1024 thread-ordered 16-byte entries
//   .x = byte offset of tap (sy,sx) in the frame            (border entries: sx | sy<<16)
//   .y = w00 | w01 << 16, .z = w10 | w11 << 16              (bilinear weights as DP2A pairs)
//   .w = blend multiplier (257*mask+1) | frac << 17 | flags << 28
// and per (camera, source row) the span of columns any in-frame tap touches.
#pragma once
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <vector>

#include "bevk_bev.cuh"

namespace bevk {

struct BevPlan {
  std::vector<int4> tiles;      // x0, y0, first item, item count
  std::vector<BevItem> items;
  std::vector<uint4> lut;       // [item][4][256]
  std::vector<int2> spans;      // [camera][source row] -> [first, last+1) sampled column, (0,0) when none
};

inline void build_bev_plan(int NC, int FW, int FH, int BW, int BH, bool nearest, const short* const* m1,
                           const unsigned short* const* m2, const uint8_t* const* masks, BevPlan& out) {
  const unsigned pitch = (unsigned)FW * 3u;
  const long long frame_bytes = (long long)pitch * FH;
  const int tx = (BW + TILE - 1) / TILE, ty = (BH + TILE - 1) / TILE;
  std::vector<int4>& tiles = out.tiles;
  std::vector<BevItem>& items = out.items;
  std::vector<uint4>& lut = out.lut;
  tiles.clear(); items.clear(); lut.clear();
  tiles.reserve((size_t)tx * ty);
  // per camera and source row: [first, last+1) column any in-frame tap touches (for k_lum_spans)
  std::vector<int2>& spans = out.spans;
  spans.assign((size_t)NC * FH, make_int2(INT_MAX, -1));
  auto touch = [&](int k, int x, int y) {
    if (x < 0 || y < 0 || x >= FW || y >= FH) return;
    int2& sp = spans[(size_t)k * FH + y];
    sp.x = std::min(sp.x, x); sp.y = std::max(sp.y, x + 1);
  };
  for (int tj = 0; tj < ty; ++tj)
    for (int ti = 0; ti < tx; ++ti) {
      const int x0 = ti * TILE, y0 = tj * TILE;
      int4 t = make_int4(x0, y0, (int)items.size(), 0);
      for (int k = 0; k < NC; ++k) {
        const uint8_t* mk = masks[k];
        bool any = false;
        long long cx = 0, cy = 0;   // source-row changes along canvas x vs canvas y
        auto in_frame = [&](int sx, int sy) {
          const long long off = (long long)sy * pitch + (long long)sx * 3;
          return sx >= 0 && sy >= 0 && sx + 1 < FW && sy + 1 < FH && !(pitch & 3u) && off + pitch + 12 <= frame_bytes;
        };
        for (int y = y0; y < std::min(y0 + TILE, BH); ++y)
          for (int x = x0; x < std::min(x0 + TILE, BW); ++x) {
            const size_t p = (size_t)y * BW + x;
            if (!mk[p]) continue;
            any = true;
            int sx = m1[k][2 * p], sy = m1[k][2 * p + 1];
            if (nearest) {   // same shift as in the entry builder below
              sx += ((m2[k][p] & 31u) < 16u); sy += (((m2[k][p] >> 5) & 31u) < 16u);
            }
            touch(k, sx, sy); touch(k, sx + 1, sy); touch(k, sx, sy + 1); touch(k, sx + 1, sy + 1);
            if (x + 1 < BW && mk[p + 1]) cx += std::abs(m1[k][2 * (p + 1) + 1] - sy);
            if (y + 1 < BH && mk[p + BW]) cy += std::abs(m1[k][2 * (p + BW) + 1] - sy);
          }
        if (!any) continue;
        BevItem item{};
        item.cam = k;
        item.orient = cy < cx ? 1 : 0;
        const size_t base = lut.size();
        lut.resize(base + TILE * TILE, make_uint4(0u, 0u, 0u, 0u));
        for (int kk = 0; kk < 4; ++kk)
          for (int th = 0; th < 256; ++th) {
            const int lane = th & 31, major = (th >> 5) * 4 + kk;
            const int x = x0 + (item.orient ? major : lane), y = y0 + (item.orient ? lane : major);
            if (x >= BW || y >= BH) continue;
            const size_t p = (size_t)y * BW + x;
            const unsigned w = mk[p];
            if (!w) continue;
            int sx = m1[k][2 * p], sy = m1[k][2 * p + 1];
            unsigned frac = m2[k][p] & 1023u;
            if (nearest) {
              // cv2.remap INTER_NEAREST with fixed-point maps: OpenCV's inverted NNDeltaTab picks the +1
              // neighbour when the fraction is < 16; a zero fraction then makes the bilinear formula
              // return exactly that texel ((1024 p + 512) >> 10 == p), so the kernel needs no NN variant
              sx += ((frac & 31u) < 16u); sy += ((frac >> 5) < 16u);
              frac = 0;
            }
            const unsigned fx = frac & 31u, fy = frac >> 5;
            const unsigned w11 = fx * fy, w01 = (fx << 5) - w11, w10 = (fy << 5) - w11, w00 = 1024u - (fx << 5) - (fy << 5) + w11;
            uint4 e;
            e.y = w00 | (w01 << 16);                       // DP2A weight pairs, top / bottom source row
            e.z = w10 | (w11 << 16);
            e.w = (w * 257u + 1u) | (frac << 17) | LUT_ACTIVE;   // blend multiplier (w > 0 here), fraction, flags
            if (!in_frame(sx, sy)) {
              // out-of-frame taps, a pitch that is not a multiple of 4, or the very end of the frame:
              // per-tap checked path
              e.w |= LUT_BORDER;
              e.x = (unsigned)(unsigned short)sx | ((unsigned)(unsigned short)sy << 16);
            } else {
              e.x = (unsigned)((long long)sy * pitch + (long long)sx * 3);
            }
            lut[base + kk * 256 + th] = e;
          }
        items.push_back(item);
        t.w++;
      }
      tiles.push_back(t);
    }
  for (auto& sp : out.spans) if (sp.y < 0) sp = make_int2(0, 0);
}

// Sampled region of one camera as DMA_BANDS horizontal bands, each with its own byte range [bx2, bx3) over rows
// [bx0, bx1): what the host path uploads of a pageable frame.  The footprint of a fisheye camera under a BEV mask is
// fan-shaped: two bands already cut the plain bounding box from 34 % to 23 % of the frame.
constexpr int DMA_BANDS = 2;
inline void plan_bands(const int2* spans /* [FH] of one camera */, int FW, int FH, int (*box)[4]) {
  int y0 = FH, y1 = 0;
  for (int y = 0; y < FH; ++y)
    if (spans[y].y > spans[y].x) { y0 = std::min(y0, y); y1 = std::max(y1, y + 1); }
  for (int bnd = 0; bnd < DMA_BANDS; ++bnd) {
    int* bx = box[bnd];
    bx[0] = bx[1] = bx[2] = bx[3] = 0;
    if (y1 <= y0) continue;
    const int ya = y0 + (int)((long long)(y1 - y0) * bnd / DMA_BANDS), yb = y0 + (int)((long long)(y1 - y0) * (bnd + 1) / DMA_BANDS);
    int x0 = FW, x1 = 0;
    for (int y = ya; y < yb; ++y) {
      const int2 sp = spans[y];
      if (sp.y > sp.x) { x0 = std::min(x0, sp.x); x1 = std::max(x1, sp.y); }
    }
    if (x1 <= x0 || yb <= ya) continue;
    // the fast path reads whole aligned words around the taps: widen by 4 px each side (touched, never sampled)
    x0 = std::max(0, x0 - 4); x1 = std::min(FW, x1 + 4);
    bx[0] = ya; bx[1] = yb; bx[2] = x0 * 3; bx[3] = x1 * 3;
  }
}

}  // namespace bevk
