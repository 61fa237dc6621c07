// bevk_plan_tma.cuh -- plan compiler of the TMA-staged fused BEV kernel (bevk_bev_tma.cuh): pure host code, shared by
// bevk_bev_finalize (bevk_api.cu) and the CPU tests (tests/host/kernel_math.cu).
//
// Input: per camera the BEV LUT planes Camera.get_bev_maps builds (SurroundBirdEyeView/surroundBEV.py:105-108) and the
// camera's mask (Mask / BlendMask, :119-280).  Output, per canvas tile of 32x32 px and per camera whose mask touches it:
//   * one LUT block of 1024 thread-ordered entries (layout in bevk_bev_tma.cuh);
//   * one or more ITEMS covering the block's four groups of eight canvas lines.  An item whose taps fit a source box
//     of at most FS = `stage_bytes` is a TMA item (box origin, tensor-map shape index, bytes) whose four frame-sets
//     share a ring slot of 4 FS; the range is halved until that holds; an 8-line strip that still does not fit gets
//     2 FS (two frame-sets per pass) or 4 FS (one per pass), and only what exceeds 4 FS is a GATHER item (global loads).
//   * the box pitch is chosen among the next few 16-byte multiples to minimise the shared-memory bank conflicts of the
//     item's own warp loads (simulated here: the lanes of a warp follow a curved path through the box).
// Box shapes are quantised to a small menu so that a few dozen tensor maps serve the whole plan.  Tiles are ordered by
// decreasing estimated cost, so that the persistent CTAs' last rounds are the cheap ones.
#pragma once
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <vector>

#include "bevk_bev_tma.cuh"

namespace bevk {

struct TmaPlan {
  std::vector<int4> tiles;          // x0, y0, first item, item count
  std::vector<TmaItem> items;
  std::vector<uint4> lut;           // [block][4][256]
  std::vector<int2> shapes;         // box shapes: (width in 32-bit words, rows)
  long long box_bytes = 0;          // sum of tx_bytes over the TMA items (one frame-set)
  long long gather_entries = 0, tma_entries = 0;   // active entries by item kind
};

inline int floor_div(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// menu: widths in 16-byte units, heights in rows; fine steps for small boxes, coarse for large ones
inline int menu_w16(int w16) {
  if (w16 <= 16) return w16;                       // <= 256 B: 16-byte steps
  if (w16 <= 32) return (w16 + 1) & ~1;            // <= 512 B: 32-byte steps
  return (w16 + 3) & ~3;                           // 64-byte steps
}
inline int menu_h(int h) {
  if (h <= 16) return (h + 1) & ~1;
  if (h <= 32) return (h + 3) & ~3;
  if (h <= 64) return (h + 7) & ~7;
  return (h + 15) & ~15;
}

// bank-conflict degree of one warp-wide 32-bit shared load: the largest number of distinct words that share a bank
inline int lds_wavefronts(const unsigned* word, int n) {
  unsigned seen[32][4];
  int cnt[32] = {0};
  int deg = 0;
  for (int i = 0; i < n; ++i) {
    const unsigned b = word[i] & 31u;
    bool dup = false;
    for (int j = 0; j < cnt[b] && j < 4; ++j) dup |= seen[b][j] == word[i];
    if (dup) continue;
    if (cnt[b] < 4) seen[b][cnt[b]] = word[i];
    cnt[b]++;
    if (cnt[b] > deg) deg = cnt[b];
  }
  return deg;
}

// Largest multi-pass box, in stages: what exceeds 4 FS becomes a GATHER item.  Measured on 1x B200 at the bench workload
// (power limit not recorded; profiles/r02_k_bev_tma_ab_runs.txt §3): multi-pass boxes win at every stage size, at FS 7936
// 0.1087 ms with boxes of up to 4 FS against 0.1125 ms with 2 FS.
constexpr int TMA_MAX_MULT = 4;

// stage_bytes / max_groups: TMA_FS / TMA_EG in the library; the CPU tests also compile plans for other values to force
// strip splits, multi-pass and GATHER items
inline void build_tma_plan(int NC, int FW, int FH, int BW, int BH, bool nearest, const short* const* m1,
                           const unsigned short* const* m2, const uint8_t* const* masks, int stage_bytes, bool allow_tma,
                           TmaPlan& out, int max_groups = TMA_EG) {
  const unsigned pitch = (unsigned)FW * 3u;
  const long long frame_bytes = (long long)pitch * FH;
  const int tx = (BW + TILE - 1) / TILE, ty = (BH + TILE - 1) / TILE;
  out.tiles.clear(); out.items.clear(); out.lut.clear(); out.shapes.clear();
  out.box_bytes = 0; out.gather_entries = out.tma_entries = 0;
  out.tiles.reserve((size_t)tx * ty);
  // TMA needs 16-byte row strides; 4-byte pixel-row alignment is what the word loads need anyway
  const bool tma_ok = allow_tma && (pitch % 16u) == 0;
  struct Ent { int sx, sy; unsigned frac, w; bool active; };
  std::vector<Ent> ent(TILE * TILE);
  std::vector<long long> tile_cost;
  for (int tj = 0; tj < ty; ++tj)
    for (int ti = 0; ti < tx; ++ti) {
      const int x0 = ti * TILE, y0 = tj * TILE;
      int4 t = make_int4(x0, y0, (int)out.items.size(), 0);
      long long item_cost = 64;   // write-out
      // can cv2.add saturate anywhere on this tile?  (blend weights of the reference sum to <= 255: never)
      bool nosat = true;
      for (int y = y0; y < std::min(y0 + TILE, BH) && nosat; ++y)
        for (int x = x0; x < std::min(x0 + TILE, BW); ++x) {
          unsigned s = 0;
          for (int k = 0; k < NC; ++k) s += masks[k][(size_t)y * BW + x];
          if (s > 255u) { nosat = false; break; }
        }
      for (int k = 0; k < NC; ++k) {
        const uint8_t* mk = masks[k];
        bool any = false, full = true;
        long long cx = 0, cy = 0;   // source-row changes along canvas x vs canvas y
        for (int y = y0; y < std::min(y0 + TILE, BH); ++y)
          for (int x = x0; x < std::min(x0 + TILE, BW); ++x) {
            const size_t p = (size_t)y * BW + x;
            if (!mk[p]) continue;
            any = true;
            if (mk[p] != 255) full = false;
            const int sy = m1[k][2 * p + 1];
            if (x + 1 < BW && mk[p + 1]) cx += std::abs(m1[k][2 * (p + 1) + 1] - sy);
            if (y + 1 < BH && mk[p + BW]) cy += std::abs(m1[k][2 * (p + BW) + 1] - sy);
          }
        if (!any) continue;
        const int orient = cy < cx ? 1 : 0;
        const int block = (int)(out.lut.size() / (TILE * TILE));
        const size_t base = out.lut.size();
        out.lut.resize(base + TILE * TILE, make_uint4(0u, 0u, 0u, 0u));
        // decode the block's entries in thread order: group kk, thread th -> canvas line kk*8 + warp, position lane
        for (int kk = 0; kk < 4; ++kk)
          for (int th = 0; th < 256; ++th) {
            Ent& e = ent[kk * 256 + th];
            e.active = false;
            const int lane = th & 31, line = kk * 8 + (th >> 5);
            const int x = x0 + (orient ? line : lane), y = y0 + (orient ? lane : line);
            if (x >= BW || y >= BH) continue;
            const size_t p = (size_t)y * BW + x;
            if (!mk[p]) continue;
            e.active = true; e.w = mk[p];
            e.sx = m1[k][2 * p]; e.sy = m1[k][2 * p + 1];
            e.frac = m2[k][p] & 1023u;
            if (nearest) {   // cv2.remap INTER_NEAREST, fixed-point maps: OpenCV's inverted NNDeltaTab (bevk_plan.cuh)
              e.sx += ((e.frac & 31u) < 16u); e.sy += ((e.frac >> 5) < 16u);
              e.frac = 0;
            }
          }
        // recursive partition of the groups [g0,g1)
        struct Range { int g0, g1; };
        std::vector<Range> todo;   // a ring slot holds the entries of at most max_groups groups
        {
          const int mg = std::max(1, std::min(4, max_groups));
          for (int g = ((4 - 1) / mg) * mg; g >= 0; g -= mg) todo.push_back({g, std::min(4, g + mg)});   // popped in group order
        }
        std::vector<TmaItem> made;
        while (!todo.empty()) {
          const Range r = todo.back();
          todo.pop_back();
          // bounding box of every word the taps of the active entries read: bytes [al, al + 8 (+4 if the pair starts at byte 3))
          int wx0 = INT_MAX, wx1 = INT_MIN, ry0 = INT_MAX, ry1 = INT_MIN, n_act = 0;
          for (int i = r.g0 * 256; i < r.g1 * 256; ++i) {
            const Ent& e = ent[i];
            if (!e.active) continue;
            ++n_act;
            const int b = 3 * e.sx, w0 = floor_div(b, 4), sh = b - 4 * w0;
            wx0 = std::min(wx0, w0); wx1 = std::max(wx1, w0 + (sh == 3 ? 3 : 2));
            ry0 = std::min(ry0, e.sy); ry1 = std::max(ry1, e.sy + 2);
          }
          TmaItem it{};
          it.lut_block = block; it.cam = (short)k; it.orient = (unsigned char)orient;
          it.k0 = (unsigned char)r.g0; it.k1 = (unsigned char)r.g1;
          it.flags = (unsigned char)((nosat ? ITEM_NOSAT : 0) | (full ? ITEM_FULL : 0));
          bool fits = false;
          int bx0 = 0, w16 = 0, hh = 0, fs_bytes = stage_bytes;
          if (n_act && tma_ok) {
            bx0 = floor_div(wx0, 4) * 4;                       // 16-byte aligned box origin (in words)
            w16 = menu_w16((wx1 - bx0 + 3) / 4);
            hh = menu_h(ry1 - ry0);
            // box dims are limited to 256 elements (words) x 256 rows; offsets must fit 16 bits
            const bool shape_ok = w16 * 4 <= 256 && hh <= 256 && wx0 > -(1 << 24) && ry0 > -(1 << 24);
            const long long bytes = (long long)w16 * 16 * hh;
            fits = shape_ok && bytes <= stage_bytes;
            if (!fits && shape_ok && r.g1 - r.g0 == 1) {       // a single strip: give it 2 or 4 frame-set slots of the stage
              for (int m = 2; m <= TMA_MAX_MULT && !fits; m *= 2)
                if (bytes <= (long long)m * stage_bytes && (long long)m * stage_bytes <= 65536) { fits = true; fs_bytes = m * stage_bytes; }
            }
          }
          if (n_act && !fits && r.g1 - r.g0 > 1) {
            const int mid = (r.g0 + r.g1) / 2;
            todo.push_back({mid, r.g1});
            todo.push_back({r.g0, mid});   // processed first: items stay in group order
            continue;
          }
          if (n_act && fits) {
            // pitch: among w16 .. w16+7 (while the box still fits) the one with the fewest bank wavefronts for this item's loads
            int best_w = w16;
            long long best_cost = -1;
            for (int cand = w16; cand < w16 + 8; ++cand) {
              if (cand != w16 && ((long long)cand * 16 * hh > fs_bytes || cand * 4 > 256 || menu_w16(cand) != cand)) continue;
              long long cost = 0;
              unsigned word[32];
              for (int g = r.g0; g < r.g1; ++g)
                for (int wv = 0; wv < 8; ++wv)
                  for (int row = 0; row < 2; ++row)
                    for (int wi = 0; wi < 3; ++wi) {
                      int n = 0;
                      for (int lane = 0; lane < 32; ++lane) {
                        const Ent& e = ent[g * 256 + wv * 32 + lane];
                        if (!e.active) continue;
                        const int b = 3 * e.sx, w0 = floor_div(b, 4), sh = b - 4 * w0;
                        if (wi == 2 && sh != 3) continue;
                        word[n++] = (unsigned)((e.sy - ry0 + row) * (cand * 4) + (w0 - bx0) + wi);
                      }
                      cost += lds_wavefronts(word, n);
                    }
              if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_w = cand; }
            }
            w16 = best_w;
            int shape = -1;
            for (size_t s = 0; s < out.shapes.size(); ++s)
              if (out.shapes[s].x == w16 * 4 && out.shapes[s].y == hh) { shape = (int)s; break; }
            if (shape < 0) { shape = (int)out.shapes.size(); out.shapes.push_back(make_int2(w16 * 4, hh)); }
            it.shape = (unsigned short)shape; it.xw = bx0; it.y = ry0; it.tx_bytes = (unsigned)(w16 * 16 * hh);
            it.fs_bytes = fs_bytes; it.pitch = w16 * 16;
            out.box_bytes += it.tx_bytes;
            item_cost += (long long)n_act * (4 * stage_bytes / fs_bytes == 4 ? 10 : (fs_bytes == 2 * stage_bytes ? 13 : 18));
          } else {
            it.flags |= ITEM_GATHER;
            it.fs_bytes = stage_bytes;
            item_cost += (long long)n_act * 80;
          }
          // entries of this range
          for (int i = r.g0 * 256; i < r.g1 * 256; ++i) {
            const Ent& e = ent[i];
            if (!e.active) continue;
            uint4 u;
            scaled_weights(e.frac, u.y, u.z);
            const int b = 3 * e.sx, w0 = floor_div(b, 4), sh = b - 4 * w0;
            if (it.flags & ITEM_GATHER) {
              u.w = (e.w * 257u + 1u) | ((unsigned)sh << 17) | (e.frac << 19) | T_ACTIVE;
              const long long off = (long long)e.sy * pitch + (long long)e.sx * 3;
              const bool in_frame = e.sx >= 0 && e.sy >= 0 && e.sx + 1 < FW && e.sy + 1 < FH && !(pitch & 3u) &&
                                    off + pitch + 12 <= frame_bytes;
              if (in_frame) u.x = (unsigned)off;
              else { u.w |= T_SLOW; u.x = (unsigned)(unsigned short)e.sx | ((unsigned)(unsigned short)e.sy << 16); }
              ++out.gather_entries;
            } else {
              u.x = (unsigned)((e.sy - ry0) * (w16 * 16) + (w0 - bx0) * 4);   // row sy + 1: one box pitch further
              u.w = tma_entry_w(e.w, (unsigned)sh);
              ++out.tma_entries;
            }
            out.lut[base + i] = u;
          }
          made.push_back(it);
        }
        // the work list pops ranges in group order, so `made` is sorted by k0
        for (const TmaItem& it : made) { out.items.push_back(it); t.w++; }
      }
      out.tiles.push_back(t);
      tile_cost.push_back(item_cost);
    }
  // heavy tiles first: CTA c takes units c, c + G, c + 2G, ... of each frame-set group, so every CTA gets one tile of
  // each cost stratum and the last round consists of the cheapest tiles
  std::vector<int> order(out.tiles.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return tile_cost[a] > tile_cost[b]; });
  std::vector<int4> sorted(out.tiles.size());
  for (size_t i = 0; i < order.size(); ++i) sorted[i] = out.tiles[order[i]];
  out.tiles.swap(sorted);
}

// What one cp.async.bulk.tensor.3d of `shape` at (xw, y) of a frame delivers: the box, zero where it leaves the frame.
// (host model of the copy for the CPU interpreter in tests/host/kernel_math.cu)
inline void model_tma_box(const uint8_t* frame, int FW, int FH, int2 shape, int xw, int y, uint8_t* dst) {
  const int pitch_w = FW * 3 / 4;
  for (int r = 0; r < shape.y; ++r)
    for (int c = 0; c < shape.x; ++c) {
      const int gx = xw + c, gy = y + r;
      unsigned v = 0;
      if (gx >= 0 && gx < pitch_w && gy >= 0 && gy < FH) memcpy(&v, frame + ((size_t)gy * pitch_w + gx) * 4, 4);
      memcpy(dst + ((size_t)r * shape.x + c) * 4, &v, 4);
    }
}

}  // namespace bevk
