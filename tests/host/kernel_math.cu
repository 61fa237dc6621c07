// Host-side unit test of the kernels' packed integer arithmetic (no GPU, no CUDA runtime calls):
// the __host__ __device__ helpers of bevk_device.cuh / bevk_bev.cuh against their scalar definitions.
//   interp_fast      == per channel ((sum w*p + 512) >> 10) * (257*mask+1) >> 16   (cv2.remap INTER_LINEAR, surroundBEV.py:116-117,
//                                                                                   then BlendMask.__call__ :279-280)
//   sat_add_bgr      == per-byte min(a+b, 255)                                       (cv2.add, :318-320)
//   tile_row_word    == byte packing of a BGRX accumulator row into dense BGR words  (canvas layout)
//   lane_addus4      == per-byte saturating add                                      (car overlay, :323-324)
// Built and run by tests/test_host_math.py with nvcc (host code only is executed).
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../cameracalibration_b200/csrc/bevk_bev.cuh"
#include "../../cameracalibration_b200/csrc/bevk_kernels.cuh"
#include "../../cameracalibration_b200/csrc/bevk_plan.cuh"
#include "../../cameracalibration_b200/csrc/bevk_plan_tma.cuh"
#include "../../cameracalibration_b200/csrc/bevk_gather4.cuh"

using namespace bevk;

static uint64_t rng_state = 0x9e3779b97f4a7c15ull;
static uint32_t rnd() {
  rng_state ^= rng_state << 7; rng_state ^= rng_state >> 9; rng_state *= 0x2545f4914f6cdd1dull;
  return (uint32_t)(rng_state >> 24);
}

static int fails = 0;
#define CHECK(cond, ...)                                   \
  do {                                                     \
    if (!(cond)) {                                         \
      if (fails < 10) { printf("FAIL %s:%d: ", __FILE__, __LINE__); printf(__VA_ARGS__); printf("\n"); } \
      ++fails;                                             \
    }                                                      \
  } while (0)

// ---- coordinate modes: run the kernels' FP64 code (undistort_point / quantise_uv / warp_point, host forms) over a
// whole map and dump it, so tests/test_host_math.py can compare with live cv2.
//   kernel_math maps <model> <w> <h> <out.bin>   stdin: K[9] D[5] P[9] as C99 hex floats
//   kernel_math warp <w> <h> <unit> <out.bin>    stdin: H[9]
static bool read_doubles(double* v, int n) {
  for (int i = 0; i < n; ++i) {
    char tok[64];
    if (scanf("%63s", tok) != 1) return false;
    v[i] = strtod(tok, nullptr);
  }
  return true;
}

static int mode_maps(int model, int w, int h, const char* path) {
  double K[9], D[5], P[9];
  if (!read_doubles(K, 9) || !read_doubles(D, 5) || !read_doubles(P, 9)) return 2;
  CamModel cm;
  memset(&cm, 0, sizeof cm);
  if (!inv3(P, cm.iR)) return 3;
  for (int i = 0; i < (model == 0 ? 4 : 5); ++i) cm.k[i] = D[i];
  cm.fx = K[0]; cm.fy = K[4]; cm.cx = K[2]; cm.cy = K[5];
  cm.model = model; cm.w = w; cm.h = h;
  FILE* f = fopen(path, "wb");
  if (!f) return 4;
  short* m1 = (short*)malloc((size_t)w * h * 4);
  unsigned short* m2 = (unsigned short*)malloc((size_t)w * h * 2);
  for (int i = 0; i < h; ++i)
    for (int j = 0; j < w; ++j) {
      double u, v;
      undistort_point(cm, j, i, u, v);
      const size_t q = (size_t)i * w + j;
      quantise_uv(u, v, m1[2 * q], m1[2 * q + 1], m2[q], pack_saturates(model, j, w));
    }
  fwrite(m1, 4, (size_t)w * h, f);
  fwrite(m2, 2, (size_t)w * h, f);
  fclose(f);
  return 0;
}

static int mode_warp(int w, int h, double unit, const char* path) {
  double H[9];
  if (!read_doubles(H, 9)) return 2;
  Homog hm;
  if (!inv3(H, hm.M)) memset(hm.M, 0, sizeof hm.M);
  FILE* f = fopen(path, "wb");
  if (!f) return 4;
  int* xy = (int*)malloc((size_t)w * h * 8);
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) warp_point(hm, x, y, unit, xy[2 * ((size_t)y * w + x)], xy[2 * ((size_t)y * w + x) + 1]);
  fwrite(xy, 8, (size_t)w * h, f);
  fclose(f);
  return 0;
}

//   kernel_math hsv <delta> <tail 0|1> <out.bin>   all 2^24 BGR colours through hsv_roundtrip (luminance_balance's
//                                                  8-bit HSV round trip), colour index = b | g<<8 | r<<16
static int mode_hsv(int delta, int tail, const char* path) {
  static int sdiv[256], hdiv[256];   // as bevk_bev_finalize fills them (OpenCV's sdiv_table / hdiv_table180)
  sdiv[0] = hdiv[0] = 0;
  for (int i = 1; i < 256; ++i) {
    sdiv[i] = (int)nearbyint((255 << 12) / (1. * i));
    hdiv[i] = (int)nearbyint((180 << 12) / (6. * i));
  }
  FILE* f = fopen(path, "wb");
  if (!f) return 4;
  uint8_t* out = (uint8_t*)malloc((size_t)3 << 24);
  for (int c = 0; c < (1 << 24); ++c) {
    int b = c & 255, g = (c >> 8) & 255, r = c >> 16;
    hsv_roundtrip(b, g, r, delta, tail != 0, sdiv, hdiv);
    out[3 * (size_t)c] = (uint8_t)b; out[3 * (size_t)c + 1] = (uint8_t)g; out[3 * (size_t)c + 2] = (uint8_t)r;
  }
  fwrite(out, 3, (size_t)1 << 24, f);
  fclose(f);
  return 0;
}

//   kernel_math bevmaps <und_w> <und_h> <bw> <bh> <out.bin>   stdin: K[9] D[4] P[9] H[9]
//       Camera.get_bev_maps (surroundBEV.py:105-108) the way bevk_bev_set_camera builds it: k_warp_maps<1>, i.e. the
//       undistort map evaluated at the four taps of every canvas pixel, never materialised
//   kernel_math warpmaps <sw> <sh> <dw> <dh> <in.bin> <out.bin> stdin: H[9]   (k_warp_maps<0>: planes given)
static int write_planes(const char* path, const short* m1, const unsigned short* m2, size_t n) {
  FILE* f = fopen(path, "wb");
  if (!f) return 4;
  fwrite(m1, 4, n, f);
  fwrite(m2, 2, n, f);
  fclose(f);
  return 0;
}

static int mode_bevmaps(int uw, int uh, int bw, int bh, const char* path) {
  double K[9], D[4], P[9], H[9];
  if (!read_doubles(K, 9) || !read_doubles(D, 4) || !read_doubles(P, 9) || !read_doubles(H, 9)) return 2;
  WarpMapsArgs a;
  memset(&a, 0, sizeof a);
  if (!inv3(P, a.cm.iR)) return 3;
  for (int i = 0; i < 4; ++i) a.cm.k[i] = D[i];
  a.cm.fx = K[0]; a.cm.fy = K[4]; a.cm.cx = K[2]; a.cm.cy = K[5];
  a.cm.model = 0; a.cm.w = uw; a.cm.h = uh;
  if (!inv3(H, a.hm.M)) memset(a.hm.M, 0, sizeof a.hm.M);
  a.sw = uw; a.sh = uh; a.dw = bw; a.dh = bh;
  const size_t n = (size_t)bw * bh;
  short* m1 = (short*)malloc(n * 4);
  unsigned short* m2 = (unsigned short*)malloc(n * 2);
  for (int y = 0; y < bh; ++y)
    for (int x = 0; x < bw; ++x) {
      const size_t q = (size_t)y * bw + x;
      warp_maps_pixel<1>(a, x, y, m1[2 * q], m1[2 * q + 1], m2[q]);
    }
  return write_planes(path, m1, m2, n);
}

static int mode_warpmaps(int sw, int sh, int dw, int dh, const char* in_path, const char* out_path) {
  double H[9];
  if (!read_doubles(H, 9)) return 2;
  const size_t ns = (size_t)sw * sh, nd = (size_t)dw * dh;
  short2* i1 = (short2*)malloc(ns * 4);
  unsigned short* i2 = (unsigned short*)malloc(ns * 2);
  FILE* f = fopen(in_path, "rb");
  if (!f || fread(i1, 4, ns, f) != ns || fread(i2, 2, ns, f) != ns) return 5;
  fclose(f);
  WarpMapsArgs a;
  memset(&a, 0, sizeof a);
  if (!inv3(H, a.hm.M)) memset(a.hm.M, 0, sizeof a.hm.M);
  a.in1 = i1; a.in2 = i2; a.sw = sw; a.sh = sh; a.dw = dw; a.dh = dh;
  short* m1 = (short*)malloc(nd * 4);
  unsigned short* m2 = (unsigned short*)malloc(nd * 2);
  for (int y = 0; y < dh; ++y)
    for (int x = 0; x < dw; ++x) {
      const size_t q = (size_t)y * dw + x;
      warp_maps_pixel<0>(a, x, y, m1[2 * q], m1[2 * q + 1], m2[q]);
    }
  return write_planes(out_path, m1, m2, nd);
}

//   kernel_math blend <w> <h> <polys.bin> <out.bin>   stdin: lines[8][4]   (BlendMask.get_blend_mask, :270-277, k_blend_masks code)
static int mode_blend(int w, int h, const char* in_path, const char* out_path) {
  double L[32];
  if (!read_doubles(L, 32)) return 2;
  const size_t n = (size_t)w * h * 4;
  uint8_t* polys = (uint8_t*)malloc(n);
  uint8_t* out = (uint8_t*)malloc(n);
  FILE* f = fopen(in_path, "rb");
  if (!f || fread(polys, 1, n, f) != n) return 5;
  fclose(f);
  BlendArgs a;
  a.polys = polys; a.out = out; a.w = w; a.h = h;
  for (int i = 0; i < 8; ++i) for (int j = 0; j < 4; ++j) a.lines[i][j] = (int)L[i * 4 + j];
  for (int y = 0; y < h; ++y) for (int x = 0; x < w; ++x) blend_pixel(a, x, y);
  f = fopen(out_path, "wb");
  if (!f) return 4;
  fwrite(out, 1, n, f);
  fclose(f);
  return 0;
}

//   kernel_math balance   stdin: npix_frames npix_canvas  vsum[4]  csum[3]  -> prints 4 luminance offsets and the 3 x 256 gain table
static int mode_balance() {
  double v[9];
  if (!read_doubles(v, 9)) return 2;
  unsigned long long vsum[4], csum[3];
  for (int i = 0; i < 4; ++i) vsum[i] = (unsigned long long)v[2 + i];
  for (int i = 0; i < 3; ++i) csum[i] = (unsigned long long)v[6 + i];
  int delta[4];
  lum_deltas(vsum, 4, v[0], delta);
  printf("%d %d %d %d\n", delta[0], delta[1], delta[2], delta[3]);
  double gain[3];
  gray_world_gains(csum, v[1], gain);
  for (int c = 0; c < 3; ++c) {
    for (int i = 0; i < 256; ++i) printf("%d ", (int)gain_entry(gain[c], i));
    printf("\n");
  }
  return 0;
}

//   kernel_math bev <in.bin> <out.bin>
//   kernel_math bevtma <in.bin> <out.bin> shipped | <stage bytes> [<entry groups per slot>]
//       the same through the TMA plan (bevk_plan_tma.cuh) at the library's TMA_FS / TMA_EG or at other settings
// One frame-set through the product's plan compiler (bevk_plan.cuh, the code bevk_bev_finalize runs) and a plain-loop
// interpreter of that plan that uses the kernels' own per-entry arithmetic (interp_fast, sample_slow_core, sat_add_bgr,
// hsv_roundtrip, lum_deltas, gray_world_gains / gain_entry).  It mirrors k_bev's work decomposition -- tile, item,
// entry index -> accumulator position by orientation, first-camera store vs saturating add -- and run_device's
// BALANCE sequence (V sums, offsets, balanced row spans, gather, channel sums, gains, car), without threads.
// in.bin : int32 NC FW FH BW BH nearest balance has_car; per camera map1 int16[BH*BW*2], map2 uint16[BH*BW],
//          mask u8[BH*BW]; NC frames u8[FH*FW*3]; car u8[BH*BW*3] if has_car.   out.bin: canvas u8[BH*BW*3]
static int mode_bev(const char* in_path, const char* out_path, int tma_stage_bytes /* 0: round-1 gather plan */, int max_groups = TMA_EG) {
  FILE* f = fopen(in_path, "rb");
  if (!f) return 5;
  int hd[8];
  if (fread(hd, 4, 8, f) != 8) return 5;
  const int NC = hd[0], FW = hd[1], FH = hd[2], BW = hd[3], BH = hd[4], nearest = hd[5], balance = hd[6], has_car = hd[7];
  const size_t npx = (size_t)BW * BH, fbytes = (size_t)FW * FH * 3;
  std::vector<std::vector<short>> m1(NC, std::vector<short>(npx * 2));
  std::vector<std::vector<unsigned short>> m2(NC, std::vector<unsigned short>(npx));
  std::vector<std::vector<uint8_t>> mk(NC, std::vector<uint8_t>(npx)), frames(NC, std::vector<uint8_t>(fbytes));
  for (int k = 0; k < NC; ++k)
    if (fread(m1[k].data(), 4, npx, f) != npx || fread(m2[k].data(), 2, npx, f) != npx || fread(mk[k].data(), 1, npx, f) != npx) return 5;
  for (int k = 0; k < NC; ++k) if (fread(frames[k].data(), 1, fbytes, f) != fbytes) return 5;
  std::vector<uint8_t> car(has_car ? npx * 3 : 0);
  if (has_car && fread(car.data(), 1, npx * 3, f) != npx * 3) return 5;
  fclose(f);

  BevPlan plan;
  {
    std::vector<const short*> p1(NC);
    std::vector<const unsigned short*> p2(NC);
    std::vector<const uint8_t*> pm(NC);
    for (int k = 0; k < NC; ++k) { p1[k] = m1[k].data(); p2[k] = m2[k].data(); pm[k] = mk[k].data(); }
    build_bev_plan(NC, FW, FH, BW, BH, nearest != 0, p1.data(), p2.data(), pm.data(), plan);
  }
  // ---- BALANCE, part 1 (k_vsum, k_delta, k_lum_spans): balanced copies hold ONLY the sampled row spans
  std::vector<std::vector<uint8_t>> bal;
  if (balance) {
    int sdiv[256] = {0}, hdiv[256] = {0};
    for (int i = 1; i < 256; ++i) {
      sdiv[i] = (int)nearbyint((255 << 12) / (1. * i));
      hdiv[i] = (int)nearbyint((180 << 12) / (6. * i));
    }
    std::vector<unsigned long long> vsum(NC, 0ull);
    for (int k = 0; k < NC; ++k)
      for (size_t i = 0; i < (size_t)FW * FH; ++i) {
        const uint8_t* q = frames[k].data() + 3 * i;
        vsum[k] += (unsigned)(q[0] > q[1] ? (q[0] > q[2] ? q[0] : q[2]) : (q[1] > q[2] ? q[1] : q[2]));
      }
    std::vector<int> delta(NC);
    lum_deltas(vsum.data(), NC, (double)FW * (double)FH, delta.data());
    bal.assign(NC, std::vector<uint8_t>(fbytes, 0xA5));          // poison: anything outside the spans must never be sampled
    const int tail = FW - (FW % 32);
    for (int k = 0; k < NC; ++k)
      for (int y = 0; y < FH; ++y) {
        const int2 sp = plan.spans[(size_t)k * FH + y];
        for (int x = sp.x; x < sp.y; ++x) {
          const uint8_t* q = frames[k].data() + ((size_t)y * FW + x) * 3;
          int b = q[0], g = q[1], r = q[2];
          hsv_roundtrip(b, g, r, delta[k], x >= tail, sdiv, hdiv);
          uint8_t* o = bal[k].data() + ((size_t)y * FW + x) * 3;
          o[0] = (uint8_t)b; o[1] = (uint8_t)g; o[2] = (uint8_t)r;
        }
      }
  }
  std::vector<uint8_t> canvas(npx * 3, 0);
  const SlowGeo geo = {(unsigned)FW * 3u, FW, FH};
  if (tma_stage_bytes > 0) {
    // ---- k_bev_tma: the TMA plan, boxes modelled as the copy delivers them (zero outside the frame)
    TmaPlan tp;
    {
      std::vector<const short*> p1(NC);
      std::vector<const unsigned short*> p2(NC);
      std::vector<const uint8_t*> pm(NC);
      for (int k = 0; k < NC; ++k) { p1[k] = m1[k].data(); p2[k] = m2[k].data(); pm[k] = mk[k].data(); }
      build_tma_plan(NC, FW, FH, BW, BH, nearest != 0, p1.data(), p2.data(), pm.data(), tma_stage_bytes, true, tp, max_groups);
    }
    std::vector<uint8_t> stage((size_t)4 * tma_stage_bytes + 16, 0xEE);   // one ring slot = 4 FS
    long long two_pass = 0, four_pass = 0, gather_items = 0;   // items by slot kind
    for (const int4& tile : tp.tiles) {
      unsigned acc[ACC_WORDS];
      for (auto& a : acc) a = 0xdeadbeefu;                 // every word must be written before the write-out reads it
      int first_cam = -1;
      for (int it = tile.z; it < tile.z + tile.w; ++it) {
        const TmaItem item = tp.items[it];
        if (first_cam < 0) first_cam = item.cam;
        const bool first = item.cam == first_cam, nosat = (item.flags & ITEM_NOSAT) != 0, gather = (item.flags & ITEM_GATHER) != 0;
        const uint8_t* src = (balance ? bal : frames)[item.cam].data();
        if (gather) ++gather_items;
        else {
          two_pass += item.fs_bytes == 2 * tma_stage_bytes;
          four_pass += item.fs_bytes == 4 * tma_stage_bytes;
          memset(stage.data(), 0xEE, stage.size());
          const int2 shape = tp.shapes[item.shape];
          CHECK((unsigned)(shape.x * 4 * shape.y) == item.tx_bytes && (int)item.tx_bytes <= item.fs_bytes, "box bytes");
          CHECK(item.pitch == shape.x * 4, "box pitch");
          CHECK(item.fs_bytes == tma_stage_bytes || ((item.fs_bytes == 2 * tma_stage_bytes || item.fs_bytes == 4 * tma_stage_bytes) &&
                                                     item.k1 - item.k0 == 1), "frame-set slot size");
          CHECK((item.xw & 3) == 0 && (shape.x & 3) == 0, "box alignment");
          CHECK(item.k1 - item.k0 <= max_groups, "item exceeds the slot's entry groups");
          model_tma_box(src, FW, FH, shape, item.xw, item.y, stage.data());
        }
        for (int k = item.k0; k < item.k1; ++k)
          for (int t = 0; t < 256; ++t) {
            const int lane = t & 31, wrp = t >> 5;
            const int pos = item.orient ? lane * ACC_WPITCH + wrp : wrp * ACC_WPITCH + lane;
            const int step = item.orient ? 8 : 8 * ACC_WPITCH;
            const uint4 e = tp.lut[(size_t)item.lut_block * (TILE * TILE) + k * 256 + t];
            unsigned* a = acc + pos + k * step;
            if (!(e.w & T_ACTIVE)) { if (first) *a = 0u; continue; }
            unsigned v;
            if (gather && (e.w & T_SLOW)) {
              v = sample_slow_core(geo, src, e.x, (e.w & 0x1ffffu) | (((e.w >> 19) & 1023u) << 17));
            } else if (gather) {   // round-1 entry layout, taps from the frame
              const unsigned sh8 = (e.w >> 14) & 24u, wm = e.w & 0x1ffffu;
              const bool third = sh8 == 24u;
              const uint8_t *q0 = src + (e.x & ~3u), *q1 = q0 + geo.pitch;
              unsigned sb, sg, sr;
              interp_sums(sh8, e.y, e.z, ldg32(q0), ldg32(q0 + 4), third ? ldg32(q0 + 8) : 0u, ldg32(q1), ldg32(q1 + 4),
                          third ? ldg32(q1 + 8) : 0u, sb, sg, sr);
              v = weight_pack<false>(sb, sg, sr, wm);
            } else {               // TMA entry: fields as tma_item decodes them, taps from the staged box
              const unsigned sh = tma_entry_shift(e.w), c = tma_entry_round(e.w);
              const bool third = (e.w & T_THIRD) != 0;
              CHECK(third == ((sh & 31u) == 24u) && (sh & 7u) == 0, "entry shift / third-word flag");
              CHECK(e.x % 4 == 0 && e.x + (unsigned)item.pitch + (third ? 12u : 8u) <= item.tx_bytes, "entry reads past its box");
              const uint8_t *q0 = stage.data() + e.x, *q1 = q0 + item.pitch;
              // a word the kernel does not load (predicated third word) is poison here: the result must not depend on it
              unsigned sb, sg, sr;
              interp_sums(sh, e.y, e.z, ldg32(q0), ldg32(q0 + 4), third ? ldg32(q0 + 8) : 0xA5A5A5A5u, ldg32(q1), ldg32(q1 + 4),
                          third ? ldg32(q1 + 8) : 0x5A5A5A5Au, sb, sg, sr);
              CHECK((sb >> 24) == 0 && (sg >> 24) == 0 && (sr >> 24) == 0, "interpolation sum reaches byte 3");
              v = (item.flags & ITEM_FULL) ? weight_pack16<true>(sb, sg, sr, e.w, c) : weight_pack16<false>(sb, sg, sr, e.w, c);
            }
            *a = first ? v : (nosat ? v + *a : sat_add_bgr(v, *a));
          }
      }
      for (int row = 0; row < TILE; ++row)
        for (int col = 0; col < TILE; ++col) {
          const int gx = tile.x + col, gy = tile.y + row;
          if (gx >= BW || gy >= BH) continue;
          const unsigned px = first_cam < 0 ? 0u : acc[row * ACC_WPITCH + col];
          CHECK(first_cam < 0 || (px >> 24) == 0, "accumulator word not written or carried into byte 3");
          uint8_t* o = canvas.data() + ((size_t)gy * BW + gx) * 3;
          o[0] = px & 255u; o[1] = (px >> 8) & 255u; o[2] = (px >> 16) & 255u;
        }
    }
    printf("tma plan: tiles=%zu items=%zu shapes=%zu box_bytes=%lld tma_entries=%lld gather_entries=%lld two_pass=%lld four_pass=%lld "
           "gather_items=%lld\n", tp.tiles.size(), tp.items.size(), tp.shapes.size(), tp.box_bytes, tp.tma_entries, tp.gather_entries,
           two_pass, four_pass, gather_items);
  } else {
  // ---- the gather (k_bev)
  for (const int4& tile : plan.tiles) {
    unsigned acc[ACC_WORDS];
    bool first = true;
    for (int it = tile.z; it < tile.z + tile.w; ++it) {
      const BevItem item = plan.items[it];
      const uint8_t* src = (balance ? bal : frames)[item.cam].data();
      for (int t = 0; t < 256; ++t) {
        const int lane = t & 31, wrp = t >> 5;
        const int pos = item.orient ? lane * ACC_WPITCH + wrp * 4 : (wrp * 4) * ACC_WPITCH + lane;
        const int step = item.orient ? 1 : ACC_WPITCH;
        for (int k = 0; k < 4; ++k) {
          const uint4 e = plan.lut[(size_t)it * (TILE * TILE) + k * 256 + t];
          unsigned* a = acc + pos + k * step;
          if (!(e.w & LUT_ACTIVE)) { if (first) *a = 0u; continue; }
          unsigned v;
          if (e.w & LUT_BORDER) v = sample_slow_core(geo, src, e.x, e.w);
          else {
            const unsigned off_al = e.x & ~3u, sh = (e.x & 3u) * 8u, wm = e.w & 0x1ffffu;
            const bool third = (sh == 24u);
            const uint8_t* q0 = src + off_al;
            const uint8_t* q1 = q0 + geo.pitch;
            v = interp_fast(sh, e.y, e.z, wm, ldg32(q0), ldg32(q0 + 4), third ? ldg32(q0 + 8) : 0u, ldg32(q1), ldg32(q1 + 4),
                            third ? ldg32(q1 + 8) : 0u);
          }
          *a = first ? v : sat_add_bgr(v, *a);
        }
      }
      first = false;
    }
    for (int row = 0; row < TILE; ++row)
      for (int col = 0; col < TILE; ++col) {
        const int gx = tile.x + col, gy = tile.y + row;
        if (gx >= BW || gy >= BH) continue;
        const unsigned px = first ? 0u : acc[row * ACC_WPITCH + col];
        uint8_t* o = canvas.data() + ((size_t)gy * BW + gx) * 3;
        o[0] = px & 255u; o[1] = (px >> 8) & 255u; o[2] = (px >> 16) & 255u;
      }
  }
  }
  // ---- BALANCE, part 2 (channel sums in k_bev<true>, k_gain) and the car overlay
  if (balance) {
    unsigned long long csum[3] = {0, 0, 0};
    for (size_t i = 0; i < npx; ++i) for (int c = 0; c < 3; ++c) csum[c] += canvas[3 * i + c];
    double gain[3];
    gray_world_gains(csum, (double)BW * (double)BH, gain);
    uint8_t tab[3][256];
    for (int c = 0; c < 3; ++c) for (int v = 0; v < 256; ++v) tab[c][v] = gain_entry(gain[c], v);
    for (size_t i = 0; i < npx; ++i) for (int c = 0; c < 3; ++c) canvas[3 * i + c] = tab[c][canvas[3 * i + c]];
  }
  if (has_car)
    for (size_t i = 0; i < npx * 3; i += 4) {
      unsigned a = 0, b = 0;
      const size_t n = npx * 3 - i < 4 ? npx * 3 - i : 4;
      memcpy(&a, canvas.data() + i, n); memcpy(&b, car.data() + i, n);
      const unsigned r = lane_addus4(a, b);
      memcpy(canvas.data() + i, &r, n);
    }
  f = fopen(out_path, "wb");
  if (!f) return 4;
  fwrite(canvas.data(), 1, npx * 3, f);
  fclose(f);
  printf("tiles=%zu items=%zu lut_bytes=%zu\n", plan.tiles.size(), plan.items.size(), plan.lut.size() * sizeof(uint4));
  return 0;
}

//   kernel_math gather <mode> <sw> <sh> <dw> <dh> <src.bin> <out.bin>   3-channel INTER_LINEAR through gather_px
//       mode 1: stdin K[9] D[5] P[9] + model  -> fused undistort (k_gather4<1>: camera model evaluated per pixel)
//       mode 2: stdin H[9]                    -> cv2.warpPerspective (k_gather4<2>)
static int mode_gather(int mode, int sw, int sh, int dw, int dh, const char* in_path, const char* out_path) {
  CamModel cm;
  Homog hm;
  memset(&cm, 0, sizeof cm);
  if (mode == 1) {
    double K[9], D[5], P[9], model;
    if (!read_doubles(K, 9) || !read_doubles(D, 5) || !read_doubles(P, 9) || !read_doubles(&model, 1)) return 2;
    if (!inv3(P, cm.iR)) return 3;
    for (int i = 0; i < 5; ++i) cm.k[i] = D[i];
    cm.fx = K[0]; cm.fy = K[4]; cm.cx = K[2]; cm.cy = K[5];
    cm.model = (int)model; cm.w = dw; cm.h = dh;
  } else {
    double H[9];
    if (!read_doubles(H, 9)) return 2;
    if (!inv3(H, hm.M)) memset(hm.M, 0, sizeof hm.M);
  }
  const size_t sbytes = (size_t)sw * sh * 3;
  std::vector<uint8_t> src(sbytes + 16, 0), dst((size_t)dw * dh * 3);   // slack: the library's buffers have it too
  FILE* f = fopen(in_path, "rb");
  if (!f || fread(src.data(), 1, sbytes, f) != sbytes) return 5;
  fclose(f);
  for (int y = 0; y < dh; ++y)
    for (int x = 0; x < dw; ++x) {
      int sx, sy;
      unsigned fx, fy;
      if (mode == 2) {
        int X, Y;
        warp_point(hm, x, y, (double)TAB, X, Y);
        sx = sat_i16(X >> INTER_BITS); sy = sat_i16(Y >> INTER_BITS);
        fx = X & (TAB - 1); fy = Y & (TAB - 1);
      } else {
        double u, v;
        short mx, my;
        unsigned short fr;
        undistort_point(cm, x, y, u, v);
        quantise_uv(u, v, mx, my, fr, pack_saturates(cm.model, x, cm.w));
        sx = mx; sy = my; fx = fr & (TAB - 1); fy = (fr >> INTER_BITS) & (TAB - 1);
      }
      const unsigned px = gather_px(src.data(), (unsigned)sw * 3u, sw, sh, sx, sy, fx, fy);
      uint8_t* o = dst.data() + ((size_t)y * dw + x) * 3;
      o[0] = px & 255u; o[1] = (px >> 8) & 255u; o[2] = (px >> 16) & 255u;
    }
  f = fopen(out_path, "wb");
  if (!f) return 4;
  fwrite(dst.data(), 1, dst.size(), f);
  fclose(f);
  return 0;
}

int main(int argc, char** argv) {
  if (argc == 9 && !strcmp(argv[1], "gather"))
    return mode_gather(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), argv[7], argv[8]);
  if (argc == 4 && !strcmp(argv[1], "bev")) return mode_bev(argv[2], argv[3], 0);
  if ((argc == 5 || argc == 6) && !strcmp(argv[1], "bevtma")) {
    const bool shipped = !strcmp(argv[4], "shipped");
    const int r = mode_bev(argv[2], argv[3], shipped ? TMA_FS : atoi(argv[4]), argc == 6 ? atoi(argv[5]) : TMA_EG);
    return r ? r : (fails ? 1 : 0);
  }
  if (argc == 2 && !strcmp(argv[1], "balance")) return mode_balance();
  if (argc == 6 && !strcmp(argv[1], "blend")) return mode_blend(atoi(argv[2]), atoi(argv[3]), argv[4], argv[5]);
  if (argc == 7 && !strcmp(argv[1], "bevmaps")) return mode_bevmaps(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), argv[6]);
  if (argc == 8 && !strcmp(argv[1], "warpmaps"))
    return mode_warpmaps(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), argv[6], argv[7]);
  if (argc == 5 && !strcmp(argv[1], "hsv")) return mode_hsv(atoi(argv[2]), atoi(argv[3]), argv[4]);
  if (argc == 6 && !strcmp(argv[1], "maps")) return mode_maps(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), argv[5]);
  if (argc == 6 && !strcmp(argv[1], "warp")) return mode_warp(atoi(argv[2]), atoi(argv[3]), atof(argv[4]), argv[5]);
  // ---- interp_fast: every byte alignment, every fraction, random pixels and masks
  long long n_interp = 0;
  for (int align = 0; align < 4; ++align)
    for (int fx = 0; fx < 32; ++fx)
      for (int fy = 0; fy < 32; ++fy)
        for (int rep = 0; rep < 24; ++rep) {
          uint8_t rows[2][16];
          for (auto& r : rows) for (auto& b : r) b = (uint8_t)rnd();
          if (rep == 0) memset(rows, 255, sizeof rows);              // saturation / rounding stress
          if (rep == 1) memset(rows, 0, sizeof rows);
          const unsigned mask = rep < 4 ? (rep & 1 ? 255u : 0u) : (rnd() & 255u);
          const unsigned wm = mask ? 257u * mask + 1u : 0u;           // plan compiler: mask 0 -> 0
          unsigned w[2][3];
          for (int r = 0; r < 2; ++r)
            for (int k = 0; k < 3; ++k) memcpy(&w[r][k], rows[r] + 4 * k, 4);
          const bool third = align == 3;
          const unsigned w11 = fx * fy, w01 = (fx << 5) - w11, w10 = (fy << 5) - w11, w00 = 1024 - (fx << 5) - (fy << 5) + w11;
          const unsigned got = interp_fast(align * 8, w00 | (w01 << 16), w10 | (w11 << 16), wm, w[0][0], w[0][1],
                                           third ? w[0][2] : 0u, w[1][0], w[1][1], third ? w[1][2] : 0u);
          unsigned want = 0;
          for (int c = 0; c < 3; ++c) {
            const int p00 = rows[0][align + c], p01 = rows[0][align + 3 + c], p10 = rows[1][align + c], p11 = rows[1][align + 3 + c];
            const unsigned v = (unsigned)bilerp_q10(p00, p01, p10, p11, fx, fy);
            const float fm = (float)((double)mask / 255.0);          // BlendMask weight as the reference forms it
            const unsigned ref_blend = (unsigned)(uint8_t)((float)v * fm);
            const unsigned mine = (v * wm) >> 16;
            CHECK(mine == ref_blend, "blend identity v=%u mask=%u: %u vs %u", v, mask, mine, ref_blend);
            want |= mine << (8 * c);
          }
          CHECK(got == want, "interp_fast align=%d fx=%d fy=%d mask=%u: %08x vs %08x", align, fx, fy, mask, got, want);
          ++n_interp;
        }
  // ---- the blend identity exhaustively (256 x 256)
  for (unsigned v = 0; v < 256; ++v)
    for (unsigned m = 0; m < 256; ++m) {
      const float fm = (float)((double)m / 255.0);
      const unsigned wm = m ? 257u * m + 1u : 0u;
      CHECK(((v * wm) >> 16) == (unsigned)(uint8_t)((float)v * fm), "identity v=%u m=%u", v, m);
    }
  // ---- the same weight as k_bev_tma applies it: ONE DP2A per channel on the interpolation sum (byte 2 = value, byte 3 = 0,
  //      bytes 0..1 = whatever the sum left there), 16-bit multiplier + rounding byte from the entry (tma_entry_w), for every
  //      (value, mask > 0), every funnel shift, two settings of the sum's low bytes
  for (unsigned v = 0; v < 256; ++v)
    for (unsigned m = 1; m < 256; ++m)
      for (unsigned sh = 0; sh < 4; ++sh)
        for (unsigned low = 0; low < 2; ++low) {
          const unsigned ew = tma_entry_w(m, sh), c = tma_entry_round(ew), sum = (v << 16) | (low ? 0xffffu : 0x0000u);
          const unsigned want = (unsigned)(uint8_t)((float)v * (float)((double)m / 255.0));
          const unsigned packed = weight_pack16<false>(sum, sum, sum, ew, c);
          CHECK(packed == want * 0x010101u, "dp2a blend v=%u m=%u: %06x vs %02x", v, m, packed, want);
          CHECK((tma_entry_shift(ew) & 31u) == 8u * sh && ((ew & T_THIRD) != 0) == (sh == 3u) && (ew & T_ACTIVE), "entry fields");
          CHECK(weight_pack16<true>(sum, sum, sum, ew, 0u) == v * 0x010101u, "full-weight pack");
        }
  // ---- sat_add_bgr / lane_addus4
  for (int i = 0; i < 2000000; ++i) {
    unsigned a = rnd() & 0x00ffffffu, b = rnd() & 0x00ffffffu;
    if (i < 256) { a = 0x00ffffffu; b = (unsigned)i * 0x010101u; }
    unsigned want = 0, want4 = 0;
    const unsigned a4 = a | (rnd() << 24), b4 = b | (rnd() << 24);
    for (int c = 0; c < 4; ++c) {
      const unsigned s3 = ((a >> (8 * c)) & 255u) + ((b >> (8 * c)) & 255u);
      const unsigned s4 = ((a4 >> (8 * c)) & 255u) + ((b4 >> (8 * c)) & 255u);
      if (c < 3) want |= (s3 > 255u ? 255u : s3) << (8 * c);
      want4 |= (s4 > 255u ? 255u : s4) << (8 * c);
    }
    CHECK(sat_add_bgr(a, b) == want, "sat_add_bgr %08x + %08x: %08x vs %08x", a, b, sat_add_bgr(a, b), want);
    CHECK(lane_addus4(a4, b4) == want4, "lane_addus4 %08x + %08x", a4, b4);
  }
  // ---- tile_row_word and the 4-pixel write-out selectors: BGRX accumulator row -> dense BGR bytes
  for (int rep = 0; rep < 2000; ++rep) {
    unsigned acc[TILE + 1];
    uint8_t dense[TILE * 3];
    for (int p = 0; p < TILE; ++p) {
      acc[p] = rnd() & 0x00ffffffu;
      dense[3 * p] = acc[p] & 255u; dense[3 * p + 1] = (acc[p] >> 8) & 255u; dense[3 * p + 2] = (acc[p] >> 16) & 255u;
    }
    acc[TILE] = 0xdeadbeefu;   // the pad word of the 33-word pitch is never selected
    for (int w = 0; w < 24; ++w) {
      unsigned want;
      memcpy(&want, dense + 4 * w, 4);
      CHECK(tile_row_word(acc, w) == want, "tile_row_word w=%d", w);
    }
    for (int chunk = 0; chunk < 8; ++chunk) {   // the shipped write-out: thread = 4 pixels -> 3 words
      const unsigned* a = acc + chunk * 4;
      unsigned want[3];
      memcpy(want, dense + 12 * chunk, 12);
      CHECK(lane_perm(a[0], a[1], 0x4210) == want[0] && lane_perm(a[1], a[2], 0x5421) == want[1] &&
            lane_perm(a[2], a[3], 0x6542) == want[2], "4-pixel write-out chunk=%d", chunk);
    }
  }
  // ---- interior write-out of k_bev_tma (bevk_bev_tma.cuh): who stores what.  The lane map -- warp w, lane l < 24 -> word l
  //      of rows w + 8i -- must cover the 32 rows x 24 words of a tile exactly once, stay inside the warp's own rows (the
  //      rows it accumulates with lanes along canvas x: barrier-free units rely on it) and deliver the dense BGR bytes
  for (int rep = 0; rep < 50; ++rep) {
    unsigned acc[TILE][TILE + 1];
    uint8_t dense[TILE][TILE * 3];
    for (int r = 0; r < TILE; ++r) {
      for (int p = 0; p < TILE; ++p) {
        acc[r][p] = rnd() & 0x00ffffffu;
        dense[r][3 * p] = acc[r][p] & 255u; dense[r][3 * p + 1] = (acc[r][p] >> 8) & 255u; dense[r][3 * p + 2] = (acc[r][p] >> 16) & 255u;
      }
      acc[r][TILE] = 0xdeadbeefu;
    }
    for (int form = 0; form < 1; ++form) {
      int seen[TILE][24] = {};
      uint8_t out[TILE][TILE * 3];
      memset(out, 0xEE, sizeof out);
      for (int wrp = 0; wrp < 8; ++wrp)
        for (int lane = 0; lane < 24; ++lane)
          for (int i = 0; i < (form ? 2 : 4); ++i) {
            const int row = tile_out_row32(wrp, i);
            CHECK(row >= 0 && row < TILE && (row & 7) == wrp, "write-out row %d is not warp %d's", row, wrp);
            for (int q = 0; q < (form ? 2 : 1); ++q) {
              const int w = form ? 2 * (lane % 12) + q : lane;
              int p; unsigned sel;
              tile_word_src(w, p, sel);
              CHECK(p + 1 <= TILE, "pixel pair of word %d", w);
              const unsigned v = lane_perm(acc[row][p], acc[row][p + 1], sel);
              memcpy(out[row] + 4 * w, &v, 4);
              seen[row][w]++;
            }
          }
      for (int r = 0; r < TILE; ++r)
        for (int w = 0; w < 24; ++w) CHECK(seen[r][w] == 1, "form %d: word (%d,%d) written %d times", form, r, w, seen[r][w]);
      CHECK(memcmp(out, dense, sizeof out) == 0, "form %d: write-out bytes", form);
    }
  }
  printf("kernel_math: %lld interp cases, fails=%d\n", n_interp, fails);
  return fails ? 1 : 0;
}
