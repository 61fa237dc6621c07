// bevk_bev.cuh -- the fused per-frame surround-BEV kernel (sm_100a).
//
// Reference path fused here (SurroundBirdEyeView/surroundBEV.py:312-325): for every
// camera  raw2bev = cv2.remap(img, bev_map1, bev_map2, INTER_LINEAR)  (:116-117), then
// Mask / BlendMask.__call__ (:161-162 / :279-280), then the saturating cv2.add chain
// (:318-320), the optional car overlay (:323-324), and -- in the BALANCE variant -- the channel
// sums color_balance needs (:44-47); luminance_balance (:57-79) has then already been applied
// to the frames' sampled row spans by k_lum_spans.  No warped intermediate is written to HBM.
//
// Work decomposition
//   * canvas tiles of 32x32 px; per tile a list of "items" = cameras whose mask touches it;
//   * per item a thread-ordered LUT block of 1024 x 16 B, fully decoded at plan time
//     (bevk_bev_finalize):
//       .x = byte offset of tap (sy,sx) in the frame            (border entries: sx | sy<<16)
//       .y = w00 | w01 << 16, .z = w10 | w11 << 16              (bilinear weights as DP2A pairs)
//       .w = blend multiplier (257*mask+1) | frac << 17 | flags << 28
//     Lanes run along the canvas direction that walks source ROWS (orientation flag), so a
//     warp's taps fall into 1-2 cache lines per row;
//   * persistent CTAs (grid = resident CTAs) loop over (tile, group of NB frame-sets).  The LUT
//     entry is fetched and decoded ONCE and applied to NB frame-sets, which amortises the
//     table traffic and all the per-entry integer work over the batch;
//   * taps: two aligned 32-bit loads per source row (+1 predicated when the 6 bytes straddle a
//     third word), funnel-shifted into place; PRMT gathers the four taps of one channel into
//     one register and two DP2A (16-bit weights x 8-bit pixels) produce  sum w*p + 512 ;
//   * the blend weight is an exact integer form of the reference's float expression:
//       uint8(float32(px) * float32(mask/255.0)) == (px * (257*mask + 1)) >> 16   for all px, mask
//     in 0..255 (mask 0 -> 0; mask 255 -> identity), checked exhaustively in tests/;
//   * results go to a shared accumulator tile of packed BGRX words (saturating add for the
//     2nd..nth camera, camera order = reference order) and leave with 32-bit stores, 12 B per
//     thread.
#pragma once
#include "bevk_device.cuh"

namespace bevk {

constexpr int TILE = 32;
constexpr int ACC_WPITCH = TILE + 1;               // 33 words per row: rows and columns are both conflict-free
constexpr int ACC_WORDS = TILE * ACC_WPITCH;       // 1056 words = 4224 B per frame-set
constexpr unsigned LUT_ACTIVE = 1u << 28, LUT_BORDER = 2u << 28;

struct BevItem {
  int cam, orient;         // orient 0: lanes along canvas x, 1: lanes along canvas y
};

struct BevParams {
  const uint8_t* const* srcs;   // device array [batch * n_cam] of dense BGR frames
  int n_cam, FW, FH;
  unsigned pitch;               // source row pitch in bytes (= 3*FW)
  const int4* tiles;            // x0, y0, first item, item count
  const BevItem* items;
  const uint4* lut;             // [item][4][256]
  int n_tiles, batch;
  uint8_t* out; int BW, BH; long long canvas_bytes;
  const uint8_t* car;
  unsigned long long* csum;     // [batch * 3] channel sums of the composed canvas (BALANCE)
  int cam_lo, cam_hi;
  // output window (see TmaParams): canvas pixels [ox,ox1) x [oy,oy1) -> out + (y-oy)*out_pitch + (x-ox)*3
  int out_pitch, ox, oy, ox1, oy1;
};

// read-only global loads; the host forms serve tests/host/kernel_math.cu
__host__ __device__ __forceinline__ unsigned ldg32(const uint8_t* p) {
#ifdef __CUDA_ARCH__
  return __ldg(reinterpret_cast<const unsigned*>(p));
#else
  return *reinterpret_cast<const unsigned*>(p);
#endif
}
__host__ __device__ __forceinline__ int ldg8(const uint8_t* p) {
#ifdef __CUDA_ARCH__
  return __ldg(p);
#else
  return *p;
#endif
}
// Fast path, phase 2: the six words of one entry -> weighted pixel packed B | G<<8 | R<<16.
__host__ __device__ __forceinline__ unsigned interp_fast(unsigned sh, unsigned wpx, unsigned wpy, unsigned wm, unsigned a0,
                                                         unsigned a1, unsigned a2, unsigned b0, unsigned b1, unsigned b2) {
  const unsigned A = lane_funnel_r(a0, a1, sh), A2 = lane_funnel_r(a1, a2, sh);   // B0 G0 R0 B1 | G1 R1 . .
  const unsigned B = lane_funnel_r(b0, b1, sh), B2 = lane_funnel_r(b1, b2, sh);
  // four taps of one channel per register: [p00 p01 p10 p11]
  const unsigned pb = lane_perm(A, B, 0x7430);
  const unsigned pg = lane_perm(lane_perm(A, A2, 0x0041), lane_perm(B, B2, 0x0041), 0x5410);
  const unsigned pr = lane_perm(lane_perm(A, A2, 0x0052), lane_perm(B, B2, 0x0052), 0x5410);
  const unsigned ob = lane_dp2a_hi(wpy, pb, lane_dp2a_lo(wpx, pb, 512u)) >> 10;
  const unsigned og = lane_dp2a_hi(wpy, pg, lane_dp2a_lo(wpx, pg, 512u)) >> 10;
  const unsigned orr = lane_dp2a_hi(wpy, pr, lane_dp2a_lo(wpx, pr, 512u)) >> 10;
  // BlendMask.__call__ / Mask.__call__ in exact integer form (see header)
  // (v * wm) < 2^24 and the weighted value is its byte 2: pack the three byte-2s with two PRMTs
  return lane_perm(lane_perm(ob * wm, og * wm, 0x0062), orr * wm, 0x7610);
}

// Word w (0..23) of a packed-BGR tile row from its 32 BGRX accumulator words: bytes 4w..4w+3 of the row
// start in pixel w + w/3 at byte phase w % 3.
__host__ __device__ __forceinline__ void tile_word_src(int w, int& p, unsigned& sel) {   // pixel pair p, p+1 and the PRMT selector
  p = w + w / 3;
  const int ph = w - (w / 3) * 3;
  sel = ph == 0 ? 0x4210u : (ph == 1 ? 0x5421u : 0x6542u);
}
__host__ __device__ __forceinline__ unsigned tile_row_word(const unsigned* acc_row, int w) {
  int p; unsigned sel;
  tile_word_src(w, p, sel);
  return lane_perm(acc_row[p], acc_row[p + 1], sel);
}
// Interior write-out of k_bev_tma, who stores what: warp `wrp` owns tile rows wrp, wrp+8, wrp+16, wrp+24 (the rows it
// accumulates with lanes along canvas x); lane l < 24 stores word l of each of them.
__host__ __device__ __forceinline__ int tile_out_row32(int wrp, int i) { return wrp + 8 * i; }                 // i = 0..3

// Slow path (kept out of line so the hot loop stays inside the instruction cache): entries with
// out-of-frame taps (BORDER_CONSTANT 0 per tap; also every entry when the pitch is not a multiple
// of 4).
struct SlowGeo { unsigned pitch; int FW, FH; };
__host__ __device__ __forceinline__ unsigned sample_slow_core(const SlowGeo P, const uint8_t* __restrict__ src, unsigned ex,
                                                             unsigned ew) {
  int p[4][3];
  const unsigned wm = ew & 0x1ffffu;
  const int sx = (short)(ex & 0xffffu), sy = (short)(ex >> 16);
#pragma unroll 1
  for (int t = 0; t < 4; ++t) {
    const int tx = sx + (t & 1), ty = sy + (t >> 1);
    const bool in = ((unsigned)tx < (unsigned)P.FW) && ((unsigned)ty < (unsigned)P.FH);
    int c0 = 0, c1 = 0, c2 = 0;
    if (in) {
      const uint8_t* q = src + (size_t)ty * P.pitch + 3 * tx;
      c0 = ldg8(q); c1 = ldg8(q + 1); c2 = ldg8(q + 2);
    }
    p[t][0] = c0; p[t][1] = c1; p[t][2] = c2;
  }
  const int fx = (ew >> 17) & 31, fy = (ew >> 22) & 31;
  unsigned ob = (unsigned)bilerp_q10(p[0][0], p[1][0], p[2][0], p[3][0], fx, fy);
  unsigned og = (unsigned)bilerp_q10(p[0][1], p[1][1], p[2][1], p[3][1], fx, fy);
  unsigned orr = (unsigned)bilerp_q10(p[0][2], p[1][2], p[2][2], p[3][2], fx, fy);
  ob = (ob * wm) >> 16; og = (og * wm) >> 16; orr = (orr * wm) >> 16;
  return ob | (og << 8) | (orr << 16);
}
__device__ __noinline__ unsigned sample_slow(const SlowGeo P, const uint8_t* __restrict__ src, unsigned ex, unsigned ew) {
  return sample_slow_core(P, src, ex, ew);
}

// cv2.add of two packed BGR pixels: per-byte saturating add (bytes 0..2; byte 3 stays 0)
__host__ __device__ __forceinline__ unsigned sat_add_bgr(unsigned a, unsigned b) {
  const unsigned lo = (a & 0x00ff00ffu) + (b & 0x00ff00ffu);          // bytes 0 and 2 -> 9-bit sums in 16-bit lanes
  const unsigned hi = ((a >> 8) & 0xffu) + ((b >> 8) & 0xffu);        // byte 1
  const unsigned lo_s = (lo | (((lo >> 8) & 0x00010001u) * 0xffu)) & 0x00ff00ffu;
  const unsigned hi_s = hi < 255u ? hi : 255u;
  return lo_s | (hi_s << 8);
}

// NB = frame-sets per work unit (1 for single-frame latency, 4 for batches).
template <bool BAL, int NB>
#ifndef BEVK_MIN_CTAS
#define BEVK_MIN_CTAS 4
#endif
__global__ void __launch_bounds__(256, BEVK_MIN_CTAS) k_bev(BevParams P) {
  extern __shared__ __align__(16) unsigned smem_w[];
  unsigned* acc = smem_w;                                   // [NB][ACC_WORDS] packed BGRX
  __shared__ unsigned long long s_sum[BAL ? 3 * NB : 1];
  const int t = threadIdx.x, lane = t & 31, wrp = t >> 5;
  if (BAL && t < 3 * NB) s_sum[t] = 0ull;
  const int groups = (P.batch + NB - 1) / NB;
  const long long n_units = (long long)P.n_tiles * groups;
  // accumulator word of this thread's first pixel / step to the next one, per orientation
  const int posx = (wrp * 4) * ACC_WPITCH + lane, stepx = ACC_WPITCH;   // lanes along x, k walks rows
  const int posy = lane * ACC_WPITCH + wrp * 4, stepy = 1;              // lanes along y, k walks columns

  for (long long unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
    const int tile_id = (int)(unit % P.n_tiles);
    const int b0 = (int)(unit / P.n_tiles) * NB;
    const int nb = min(NB, P.batch - b0);
    const int4 tile = P.tiles[tile_id];
    __syncthreads();   // previous unit's write-out (and the table fill on the first pass) is done
    bool first = true;   // no camera has written this tile yet: the first one stores (zeros where masked out)
    for (int it = tile.z; it < tile.z + tile.w; ++it) {
      const BevItem item = P.items[it];
      if (item.cam < P.cam_lo || item.cam >= P.cam_hi) continue;
      const uint4* __restrict__ L = P.lut + (size_t)it * (TILE * TILE) + t;
      const uint8_t* src[NB];
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        const int b = b0 + (j < nb ? j : 0);   // j >= nb aliases frame-set b0: computed, never written out
        src[j] = P.srcs[b * P.n_cam + item.cam];
      }
      const int pos = item.orient ? posy : posx, step = item.orient ? stepy : stepx;
      uint4 nxt = __ldg(L);
#pragma unroll 1
      for (int k = 0; k < 4; ++k) {
        const uint4 e = nxt;
        if (k < 3) nxt = __ldg(L + (k + 1) * 256);   // prefetch the next entry under this one's work
        unsigned* a = acc + pos + k * step;
        if (!(e.w & LUT_ACTIVE)) {
          if (first) {
#pragma unroll
            for (int j = 0; j < NB; ++j) a[j * ACC_WORDS] = 0u;
          }
          continue;
        }
        if (e.w & LUT_BORDER) {
          const SlowGeo geo = {P.pitch, P.FW, P.FH};
#pragma unroll
          for (int j = 0; j < NB; ++j) {
            unsigned v = sample_slow(geo, src[j], e.x, e.w);
            if (!first) v = sat_add_bgr(v, a[j * ACC_WORDS]);
            a[j * ACC_WORDS] = v;
          }
        } else {
          // phase 1: every tap load of the NB frame-sets in flight before any is consumed;
          // phase 2: interpolate, weight, accumulate (cv2.add order: front, back, left, right)
          const unsigned off_al = e.x & ~3u, sh = (e.x & 3u) * 8u, wm = e.w & 0x1ffffu;
          const bool third = (sh == 24u);
          unsigned a0[NB], a1[NB], a2[NB], b0w[NB], b1w[NB], b2w[NB];
#pragma unroll
          for (int j = 0; j < NB; ++j) {
            const uint8_t* q0 = src[j] + off_al;
            const uint8_t* q1 = q0 + P.pitch;
            a0[j] = ldg32(q0); a1[j] = ldg32(q0 + 4); a2[j] = third ? ldg32(q0 + 8) : 0u;
            b0w[j] = ldg32(q1); b1w[j] = ldg32(q1 + 4); b2w[j] = third ? ldg32(q1 + 8) : 0u;
          }
          if (first) {
#pragma unroll
            for (int j = 0; j < NB; ++j)
              a[j * ACC_WORDS] = interp_fast(sh, e.y, e.z, wm, a0[j], a1[j], a2[j], b0w[j], b1w[j], b2w[j]);
          } else {
#pragma unroll
            for (int j = 0; j < NB; ++j)
              a[j * ACC_WORDS] =
                  sat_add_bgr(interp_fast(sh, e.y, e.z, wm, a0[j], a1[j], a2[j], b0w[j], b1w[j], b2w[j]), a[j * ACC_WORDS]);
          }
        }
      }
      first = false;
      __syncthreads();
    }
    if (tile.x >= P.ox1 || tile.x + TILE <= P.ox || tile.y >= P.oy1 || tile.y + TILE <= P.oy) continue;   // outside the output window
    // ---- write the tile(s): thread t -> row t/8, 4 pixels (12 bytes) at pixel 4*(t%8) ----
    const int row = t >> 3, chunk = t & 7;
    const int gy = tile.y + row, gx = tile.x + chunk * 4;
    const bool inb = (gy < P.oy1) && (gx < P.ox1);
    const size_t pix_off = (size_t)(gy - P.oy) * P.out_pitch + (size_t)(gx - P.ox) * 3;
    const bool full = inb && (gx + 4 <= P.ox1) && (P.out_pitch % 4 == 0) && (P.canvas_bytes % 4 == 0) && (P.ox % 4 == 0);
    const int npx = inb ? min(4, P.ox1 - gx) : 0;
    unsigned c0 = 0, c1 = 0, c2 = 0;
    if (!BAL && P.car && full) {
      const unsigned* c = reinterpret_cast<const unsigned*>(P.car + pix_off);
      c0 = __ldg(c); c1 = __ldg(c + 1); c2 = __ldg(c + 2);
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      if (j >= nb) break;
      const unsigned* a = acc + j * ACC_WORDS + row * ACC_WPITCH + chunk * 4;
      unsigned x0 = a[0], x1 = a[1], x2 = a[2], x3 = a[3];                 // BGRX BGRX BGRX BGRX
      if (first) x0 = x1 = x2 = x3 = 0u;                                   // tile without a camera (car hole)
      unsigned w0 = lane_perm(x0, x1, 0x4210);                             // B0 G0 R0 B1
      unsigned w1 = lane_perm(x1, x2, 0x5421);                             // G1 R1 B2 G2
      unsigned w2 = lane_perm(x2, x3, 0x6542);                             // R2 B3 G3 R3
      if (BAL) {   // channel sums of the composed canvas, before gains and car (surroundBEV.py:44-47)
        const unsigned px[4] = {x0, x1, x2, x3};
        unsigned sb = 0, sg = 0, sr = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < npx) { sb += px[q] & 255u; sg += (px[q] >> 8) & 255u; sr += (px[q] >> 16) & 255u; }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {   // every lane takes part (out-of-canvas lanes add 0)
          sb += __shfl_xor_sync(0xffffffffu, sb, s);
          sg += __shfl_xor_sync(0xffffffffu, sg, s);
          sr += __shfl_xor_sync(0xffffffffu, sr, s);
        }
        if (lane == 0) {
          atomicAdd(&s_sum[3 * j + 0], (unsigned long long)sb);
          atomicAdd(&s_sum[3 * j + 1], (unsigned long long)sg);
          atomicAdd(&s_sum[3 * j + 2], (unsigned long long)sr);
        }
      }
      if (!inb) continue;
      uint8_t* o = P.out + (size_t)(b0 + j) * P.canvas_bytes + pix_off;
      if (full) {
        if (!BAL && P.car) { w0 = lane_addus4(w0, c0); w1 = lane_addus4(w1, c1); w2 = lane_addus4(w2, c2); }
        unsigned* g = reinterpret_cast<unsigned*>(o);
        g[0] = w0; g[1] = w1; g[2] = w2;
      } else {
        const unsigned wv[3] = {w0, w1, w2};
#pragma unroll 1
        for (int i = 0; i < npx * 3; ++i) {
          int v = (wv[i >> 2] >> (8 * (i & 3))) & 255u;
          if (!BAL && P.car) v = min(255, v + P.car[pix_off + i]);
          o[i] = (uint8_t)v;
        }
      }
    }
    if (BAL) {
      __syncthreads();
      if (t < 3 * nb) { atomicAdd(P.csum + (size_t)(b0 + t / 3) * 3 + (t % 3), s_sum[t]); s_sum[t] = 0ull; }
    }
  }
}

constexpr size_t bev_smem_bytes(bool /*bal*/, int nb) { return (size_t)nb * ACC_WORDS * 4; }

}  // namespace bevk
