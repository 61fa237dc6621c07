// bevk_bev_tma.cuh -- the fused surround-BEV kernel with TMA-staged source boxes (sm_100a).
//
// Same reference path as bevk_bev.cuh (SurroundBirdEyeView/surroundBEV.py:312-325: cv2.remap per camera :116-117,
// Mask / BlendMask.__call__ :161-162 / :279-280, the saturating cv2.add chain :318-320, car overlay :323-324), same
// arithmetic, different memory movement:
//
//   * the frames of a batch are one 3-D tensor  uint32[frame][row][pitch/4]  (frames at a uniform stride); for every
//     work item -- (canvas tile, camera, range of 8-line strips) -- the plan compiler (bevk_plan_tma.cuh) knows the
//     bounding box of the source words its taps read, and a producer warp fetches that box for each of the NB
//     frame-sets of the unit with ONE cp.async.bulk.tensor.3d (SASS UTMALDG) into a ring of shared-memory stages,
//     completion on an mbarrier.  Taps outside the frame need no special path: TMA zero-fills out-of-bounds words,
//     which is exactly cv2.remap's BORDER_CONSTANT 0.
//   * the producer also copies the item's LUT entries (cp.async.bulk, SASS UBLKCP) and writes a 32-byte descriptor of
//     the work (what to do with the slot, where the tile is, whether a write-out follows) into the same ring slot, so the
//     eight consumer warps never touch global memory on their way: they wait for a slot, read the descriptor, the
//     entries (LDS.128) and their taps (LDS with immediate offsets for frame-set and word; ~1.4 bank wavefronts per
//     load instead of 4.4 L1 tag look-ups per global load, profiles/) from shared memory, and release the slot through
//     a second mbarrier.  Every latency of the global side is the producer's, which runs TMA_STAGES slots ahead;
//   * a stage holds 4 FS bytes: the boxes of four frame-sets of FS bytes each, or -- for the heavily minified near
//     field, where 256 samples need 12-24 KB of source -- two boxes of 2 FS or one of 4 FS; such items take 2 or 4
//     PASSES over their entries, one ring slot per pass.  Only what does not even fit 4 FS (discontinuities of the
//     LUT, about 1 % of the entries) is a GATHER item: entries carry global byte offsets and take the 32-bit
//     global loads of the round-1 kernel.
//
// LUT entry (16 B, thread order t = warp*32 + lane, group k: canvas line k*8 + warp, position lane along it):
//   .y  w00' | w10' << 16,  .z  w01' | w11' << 16   with w' = min(64 w, 65535): the DP2A sums carry
//       64 (sum w p + 512), so byte 2 of each sum is the interpolated channel -- no shifts
//   TMA item (every field is where one instruction finds it):
//   .x  byte offset of the aligned word holding tap (sy,sx) inside the frame-set's staged box; row sy+1 lies one box
//       pitch (slot descriptor) further
//   .w  16-bit blend multiplier (bits 0..15, third DP2A operand as it is) | its rounding byte (16..23) |
//       8 * (3 sx mod 4) = funnel-shift amount (24..28) | T_ACTIVE | T_THIRD (the tap pair starts at byte 3 of its word)
//   GATHER item (boxes that fit no stage, ~1 % of the entries; the round-1 layout):
//   .x  byte offset of tap (sy,sx) in the frame (slow entries: sx | sy << 16)
//   .w  blend multiplier 257*mask+1 (17 bits) | (3 sx mod 4) << 17 | fraction << 19 | T_ACTIVE | T_SLOW
#pragma once
#include "bevk_bev.cuh"

namespace bevk {

constexpr unsigned T_ACTIVE = 1u << 29, T_SLOW = 1u << 30 /* GATHER entries */, T_THIRD = 1u << 30 /* TMA entries */;
constexpr int ITEM_GATHER = 1, ITEM_NOSAT = 2, ITEM_FULL = 4;
constexpr int TMA_CONSUMERS = 256, TMA_THREADS = TMA_CONSUMERS + 32;
constexpr int TMA_DESC_BYTES = 128;   // sizeof(CUtensorMap)

// The one configuration of k_bev_tma.  Every value won a measurement on 1x B200 at the bench workload (power limit not
// recorded; profiles/r02_k_bev_tma_ab_runs.txt §3, experiments/README.md):
//   TMA_FS        bytes of one frame-set's staged source box; a ring slot holds 4 FS of boxes.  With two CTAs per SM the
//                 largest slots that fit win (fewer, fuller slots: 0.121 ms at FS 4096 -> 0.109 ms at FS 7936).  7936:
//                 2 x (2 x 48256 + 16896 + 1056) + static/reserved = 233024 of the SM's 233472 bytes.
//   TMA_STAGES    ring slots: a third, smaller slot does not pay (three slots of FS 4096 / 5120: 0.121 / 0.120 ms).
//   TMA_MIN_CTAS  resident CTAs per SM the register budget (96) is set for: 3 CTAs/SM at 72 registers measured 0.18 vs
//                 0.14 ms (the spills land in the item loop).
//   TMA_EG        LUT-entry groups a slot holds, i.e. all four of a block (the plan's items never span more).
constexpr int TMA_FS = 7936, TMA_STAGES = 2, TMA_MIN_CTAS = 2, TMA_EG = 4;
// ring slot: boxes (4 FS) | LUT entries of up to EG groups (EG * 4 KB) | descriptor (128 B reserved); a multiple of 128:
// TMA destinations
constexpr int TMA_SLOT_BYTES = 4 * TMA_FS + TMA_EG * 4096 + 128;
constexpr size_t bev_tma_smem_bytes(int nb) {
  return (size_t)TMA_STAGES * TMA_SLOT_BYTES + (size_t)nb * ACC_WORDS * 4 + (size_t)TMA_STAGES * 16 + 1024;   // + alignment slack
}

struct __align__(16) TmaItem {   // 32 B, read as two 16-byte words
  int lut_block;                 // LUT block of this (tile, camera): entries [lut_block*1024, +1024)
  short cam; unsigned char orient, flags;
  unsigned char k0, k1; unsigned short shape;   // entry groups [k0,k1); index of the box shape's tensor map
  int xw;                        // box origin: word column (may be negative) ...
  int y;                         // ... and row; TMA zero-fills what lies outside the frame
  unsigned tx_bytes;             // bytes the box of ONE frame-set delivers
  int fs_bytes;                  // stage bytes reserved per frame-set: FS, 2 FS or 4 FS (a stage holds 4, 2 or 1 frame-sets)
  int pitch;                     // row pitch of the staged box in bytes
};
static_assert(sizeof(TmaItem) == 32, "TmaItem is read as two int4");

struct TmaParams {
  const uint8_t* maps;           // [n_shapes] CUtensorMap (128 B each) in global memory
  const uint8_t* base;           // frame 0 of the stack (GATHER items, slow entries)
  long long frame_stride;        // bytes between consecutive frames
  int n_cam, FW, FH;
  unsigned pitch;
  const int4* tiles;             // x0, y0, first item, item count
  const TmaItem* items;
  const uint4* lut;
  int n_tiles, batch;
  uint8_t* out; int BW, BH; long long canvas_bytes;   // canvas_bytes: stride between the frame-sets' outputs
  const uint8_t* car;
  unsigned long long* csum;
  int cam_lo, cam_hi;
  // output window (camera-sharded runs render only the tile-aligned bounding box of their cameras' masks, a "slab"):
  // canvas pixels [ox,ox1) x [oy,oy1) go to out + (y-oy)*out_pitch + (x-ox)*3; the full canvas is 0,0,BW,BH, pitch 3*BW
  int out_pitch, ox, oy, ox1, oy1;
  unsigned* unit_counter;        // zeroed before the launch: next unit to hand out
  // camera-sharded runs with peer stores (bevk_bev_run_scattered): the output of frame-set b goes straight into the memory
  // of the rank that owns b -- peer[b % world] + src_off + (b / world) * canvas_bytes -- over NVLink; world == 0: plain `out`
  uint8_t* peer[8];
  int world;
  long long src_off;
  unsigned long long* trace;     // -DBEVK_TRACE builds (tools/gpu/trace_slots.py): [cta < 8][slot < 512][16] clock64 stamps; else unused
};

// The six words of one entry -> three sums whose byte 2 is the interpolated channel.
__host__ __device__ __forceinline__ void interp_sums(unsigned sh8, unsigned wl, unsigned wr, unsigned a0, unsigned a1, unsigned a2,
                                                     unsigned b0, unsigned b1, unsigned b2, unsigned& sb, unsigned& sg, unsigned& sr) {
  const unsigned A = lane_funnel_r(a0, a1, sh8), A2 = lane_funnel_r(a1, a2, sh8);   // B0 G0 R0 B1 | G1 R1 . .
  const unsigned B = lane_funnel_r(b0, b1, sh8), B2 = lane_funnel_r(b1, b2, sh8);   // same, source row + 1
  const unsigned v0 = lane_perm(A, B, 0x5140);     // B0 B0' G0 G0'
  const unsigned v1 = lane_perm(A, B, 0x7362);     // R0 R0' B1 B1'
  const unsigned v2 = lane_perm(A2, B2, 0x5140);   // G1 G1' R1 R1'
  sb = lane_dp2a_hi(wr, v1, lane_dp2a_lo(wl, v0, 32768u));
  sg = lane_dp2a_lo(wr, v2, lane_dp2a_hi(wl, v0, 32768u));
  sr = lane_dp2a_hi(wr, v2, lane_dp2a_lo(wl, v1, 32768u));
}

// BlendMask.__call__ / Mask.__call__ in exact integer form (bevk_bev.cuh header), then pack B | G<<8 | R<<16.
// FULL: every weight of the item is 255 (multiplier 65536): the weighted value is the value.
template <bool FULL>
__host__ __device__ __forceinline__ unsigned weight_pack(unsigned sb, unsigned sg, unsigned sr, unsigned wm) {
  if (FULL) return lane_perm(lane_perm(sb, sg, 0x0062), sr, 0x7610);
  const unsigned ob = (sb >> 16) * wm, og = (sg >> 16) * wm, orr = (sr >> 16) * wm;   // < 2^24, byte 2 is the result
  return lane_perm(lane_perm(ob, og, 0x0062), orr, 0x7610);
}

__host__ __device__ __forceinline__ unsigned interp_v(unsigned sh8, unsigned wl, unsigned wr, unsigned wm, unsigned a0, unsigned a1,
                                                      unsigned a2, unsigned b0, unsigned b1, unsigned b2) {
  unsigned sb, sg, sr;
  interp_sums(sh8, wl, wr, a0, a1, a2, b0, b1, b2, sb, sg, sr);
  return weight_pack<false>(sb, sg, sr, wm);
}

// The same blend weight as ONE DP2A per channel (TMA entries).  The interpolated channel p is byte 2 of its sum and
// byte 3 is 0 (the sums stay below 2^24), so dp2a_hi(ew, s, c) = (ew & 0xffff) * p + c whatever bits 16..31 of ew hold:
//   mask < 255:  multiplier 257 mask + 1 (< 65536), c = 0    -> byte 2 = (p (257 mask + 1)) >> 16, the reference's value
//   mask = 255:  multiplier 65535, c = 255                    -> 65535 p + 255 = 65536 p + (255 - p): byte 2 = p
// (exhaustive check over all (p, mask): tests/host/kernel_math.cu).  .w of a TMA entry, fields as tma_item reads them:
__host__ __device__ __forceinline__ unsigned tma_entry_w(unsigned mask, unsigned sh /* 3 sx mod 4 */) {
  return (mask == 255u ? 65535u | (255u << 16) : mask * 257u + 1u) | (sh * 8u) << 24 | (sh == 3u ? T_THIRD : 0u) | T_ACTIVE;
}
template <bool FULL>
__host__ __device__ __forceinline__ unsigned weight_pack16(unsigned sb, unsigned sg, unsigned sr, unsigned ew, unsigned c) {
  if (FULL) return lane_perm(lane_perm(sb, sg, 0x0062), sr, 0x7610);
  const unsigned ob = lane_dp2a_hi(ew, sb, c), og = lane_dp2a_hi(ew, sg, c), orr = lane_dp2a_hi(ew, sr, c);   // < 2^24
  return lane_perm(lane_perm(ob, og, 0x0062), orr, 0x7610);
}
// fields of a TMA entry's .w: funnel-shift amount (the shifter uses bits 0..4 only), rounding byte
__host__ __device__ __forceinline__ unsigned tma_entry_shift(unsigned ew) { return ew >> 24; }
__host__ __device__ __forceinline__ unsigned tma_entry_round(unsigned ew) { return lane_perm(ew, 0u, 0x4442); }

// DP2A weight pairs of a 10-bit fraction (fy*32 + fx), scaled by 64 (see header)
__host__ __device__ __forceinline__ void scaled_weights(unsigned frac, unsigned& wl, unsigned& wr) {
  const unsigned fx = frac & 31u, fy = (frac >> 5) & 31u;
  const unsigned w11 = fx * fy, w01 = (fx << 5) - w11, w10 = (fy << 5) - w11, w00 = 1024u - (fx << 5) - (fy << 5) + w11;
  const unsigned s00 = w00 == 1024u ? 65535u : w00 << 6;   // (65535 p + 32768) >> 16 == p for p < 32768
  wl = s00 | (w10 << 22);
  wr = (w01 << 6) | (w11 << 22);
}

#ifdef __CUDACC__
// ---- mbarrier / TMA primitives (PTX ISA 8.x, sm_90+) ---------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  // the suspend-time hint lets the hardware park the warp instead of re-issuing the poll (profiles/r02_d: 9 polls per
  // wait and 5 % of all issue slots without it)
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra D_%=;\n\t"
      "bra W_%=;\n\t"
      "D_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(20000u) : "memory");
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const void* map, int x, int y, int z, unsigned bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(z), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_copy(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds128(unsigned addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(unsigned addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ unsigned lds32(unsigned addr) {
  unsigned v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// Predicated load: the destination keeps whatever it held when `pred` is 0.  Used for the third word of a tap pair,
// which only pairs starting at byte 3 of a word read (interp_sums never looks at it otherwise).
__device__ __forceinline__ unsigned lds32_if(unsigned addr, unsigned pred) {
  unsigned v;
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p ld.shared.u32 %0, [%1];\n\t}" : "=r"(v) : "r"(addr), "r"(pred));
  return v;
}
__device__ __forceinline__ void sts32(unsigned addr, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
// one lane of the (converged) warp
__device__ __forceinline__ bool elect_one() {
  unsigned p;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(TMA_CONSUMERS) : "memory"); }

// Slot descriptor: two 16-byte words written by the producer, everything pre-digested so that a consumer warp spends a
// handful of instructions per slot.
//   word 0  .x flags (below) | groups in the slot << 16 | pass kind << 20 (0: four boxes FS apart, 1: two boxes 2 FS
//              apart, 2: one box)
//           .y row pitch of the staged boxes in bytes
//           .z byte offset of the slot's first accumulator word relative to the thread's own (first group, first
//              frame-set of the pass)
//           .w accumulator bytes between consecutive groups
//   word 1  (read by GATHER slots and by the slot that ends a unit)
//           .x tile x | y << 16, .y first frame-set of the unit | frame-sets in it << 16, .z camera
constexpr unsigned D_END = 1u, D_GATHER = 2u, D_FIRST = 4u, D_FULL = 8u, D_NOSAT = 16u, D_ORIENT = 32u, D_SYNC = 64u, D_LAST = 128u,
                   D_NONE = 256u, D_ROWS = 512u;
// Barriers among the consumer warps.  Warp w accumulates canvas rows w, w+8, w+16, w+24 of the tile when the lanes run
// along canvas x (orientation 0) and columns w, w+8, ... when they run along y; the interior write-out gives warp w the
// rows w, w+8, w+16, w+24.  So a unit whose items all have orientation 0 never lets a warp touch another warp's words:
//   * D_SYNC (barrier before the slot is applied): the orientation changes inside a unit, or the unit's first item has
//     orientation 1 (other warps may still be writing out the rows it stores into), or the previous unit left through
//     the generic write-out (edge tiles, BALANCE), which reads across rows;
//   * D_ROWS on the slot that ends a unit: every item had orientation 0 and the tile takes the interior write-out --
//     no barrier before the write-out either.  Otherwise the warps meet once before they write.

// GATHER items (boxes that do not fit a stage): one entry applied to the NB frame-sets of the unit, taps from global
// memory as in the round-1 kernel.  `aa`: shared address of the entry's accumulator word of frame-set 0.
template <int NB>
__device__ __forceinline__ void gather_entry(const TmaParams& P, const uint4 e, unsigned aa, bool first, bool nosat,
                                             const uint8_t* frame0, long long set_stride, int nb) {
  if (!(e.w & T_ACTIVE)) {
    if (first) {
#pragma unroll
      for (int j = 0; j < NB; ++j) sts32(aa + j * ACC_WORDS * 4, 0u);
    }
    return;
  }
  if (e.w & T_SLOW) {   // out-of-frame taps: per-tap checked path
    const SlowGeo geo = {P.pitch, P.FW, P.FH};
    const unsigned ew = (e.w & 0x1ffffu) | (((e.w >> 19) & 1023u) << 17);   // sample_slow's layout: weight | fraction << 17
#pragma unroll 1
    for (int j = 0; j < NB; ++j) {
      unsigned v = sample_slow(geo, frame0 + (j < nb ? j : 0) * set_stride, e.x, ew);   // the batch tail aliases frame-set 0: never written out
      if (!first) v = sat_add_bgr(v, lds32(aa + j * ACC_WORDS * 4));
      sts32(aa + j * ACC_WORDS * 4, v);
    }
    return;
  }
  const unsigned sh8 = (e.w >> 14) & 24u, wm = e.w & 0x1ffffu, off_al = e.x & ~3u;
  const bool third = sh8 == 24u;
#pragma unroll 2
  for (int j = 0; j < NB; ++j) {
    const uint8_t* q0 = frame0 + (j < nb ? j : 0) * set_stride + off_al;
    const uint8_t* q1 = q0 + P.pitch;
    const unsigned a0 = ldg32(q0), a1 = ldg32(q0 + 4), a2 = third ? ldg32(q0 + 8) : 0u;
    const unsigned b0 = ldg32(q1), b1 = ldg32(q1 + 4), b2 = third ? ldg32(q1 + 8) : 0u;
    unsigned sb, sg, sr;
    interp_sums(sh8, e.y, e.z, a0, a1, a2, b0, b1, b2, sb, sg, sr);
    unsigned v = weight_pack<false>(sb, sg, sr, wm);
    if (!first) {
      const unsigned old = lds32(aa + j * ACC_WORDS * 4);
      v = nosat ? v + old : sat_add_bgr(v, old);                          // cv2.add chain, reference camera order
    }
    sts32(aa + j * ACC_WORDS * 4, v);
  }
}

// TMA slots: `nk` groups of LUT entries (in the slot, `ent` = this thread's first entry) applied to NBP staged boxes.
// RS: slot bytes between the boxes of consecutive frame-sets; `pitch`: bytes between the rows of a box.  FIRST: this
// camera stores (zeros where its mask is 0), later cameras add; FULL: every weight of the item is 255.
template <int NBP, int RS, bool FIRST, bool FULL, bool NOSAT>
__device__ __forceinline__ void tma_item(unsigned ent, int nk, unsigned sbase, unsigned pitch, unsigned aa, unsigned astep) {
  uint4 nxt = lds128(ent);
#pragma unroll 1
  for (int k = 0; k < nk; ++k, aa += astep) {
    const uint4 e = nxt;
    ent += 4096;
    if (k + 1 < nk) nxt = lds128(ent);
    if (!(e.w & T_ACTIVE)) {
      if (FIRST) {
#pragma unroll
        for (int j = 0; j < NBP; ++j) sts32(aa + j * ACC_WORDS * 4, 0u);
      }
      continue;
    }
    const unsigned o0 = sbase + e.x, o1 = o0 + pitch;
    const unsigned sh = tma_entry_shift(e.w), third = e.w & T_THIRD, c = FULL ? 0u : tma_entry_round(e.w);
    unsigned a0[NBP], a1[NBP], a2[NBP], b0[NBP], b1[NBP], b2[NBP];
#pragma unroll
    for (int j = 0; j < NBP; ++j) {
      const unsigned r0 = o0 + j * RS, r1 = o1 + j * RS;
      a0[j] = lds32(r0); a1[j] = lds32(r0 + 4); a2[j] = lds32_if(r0 + 8, third);
      b0[j] = lds32(r1); b1[j] = lds32(r1 + 4); b2[j] = lds32_if(r1 + 8, third);
    }
#pragma unroll
    for (int j = 0; j < NBP; ++j) {
      unsigned sb, sg, sr;
      interp_sums(sh, e.y, e.z, a0[j], a1[j], a2[j], b0[j], b1[j], b2[j], sb, sg, sr);
      unsigned v = weight_pack16<FULL>(sb, sg, sr, e.w, c);
      if (!FIRST) {
        const unsigned old = lds32(aa + j * ACC_WORDS * 4);
        v = NOSAT ? v + old : sat_add_bgr(v, old);                        // cv2.add chain, reference camera order
      }
      sts32(aa + j * ACC_WORDS * 4, v);
    }
  }
}

// one pass of a TMA item: NBP frame-sets whose boxes lie RS bytes apart in the slot
template <int NBP, int RS>
__device__ __forceinline__ void tma_pass(unsigned ent, int nk, unsigned sbase, unsigned pitch, unsigned aa, unsigned astep,
                                         unsigned flags) {
  if (!(flags & D_FIRST)) {   // NOSAT: the masks of the tile sum to <= 255 everywhere (always so for the reference's blend masks): plain add
    if (flags & D_NOSAT) tma_item<NBP, RS, false, false, true>(ent, nk, sbase, pitch, aa, astep);
    else tma_item<NBP, RS, false, false, false>(ent, nk, sbase, pitch, aa, astep);
  } else if (NBP == 4 && (flags & D_FULL)) tma_item<NBP, RS, true, true, true>(ent, nk, sbase, pitch, aa, astep);
  else tma_item<NBP, RS, true, false, true>(ent, nk, sbase, pitch, aa, astep);
}

// where frame-set b of the call is written: the caller's buffer, or (scattered mode) the owning rank's slab buffer
template <bool SCATTER>
__device__ __forceinline__ uint8_t* out_base(const TmaParams& P, int b) {
  if (!SCATTER) return P.out + (size_t)b * P.canvas_bytes;
  return P.peer[b % P.world] + P.src_off + (size_t)(b / P.world) * P.canvas_bytes;
}

// interior write-out of one lane: `rows` row pieces (one 32-bit word each, tile rows w, w+8, w+16, w+24 of warp w) of
// `nb` frame-sets, the first at byte offset `off` of frame-set b0's output; wacc/wsel: the lane's accumulator word pair
// and byte selector (k_bev_tma).  WHOLE: four rows, NB frame-sets, at least one camera -- the common case, without
// per-word checks.
template <int NB, bool SCATTER, bool CAR, bool WHOLE>
__device__ __forceinline__ void tile_rows_out(const TmaParams& P, unsigned wacc, unsigned wsel, size_t off, int rows, int b0, int nb, bool none) {
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    if (!WHOLE && j >= nb) break;
    uint8_t* o = out_base<SCATTER>(P, b0 + j) + off;   // SCATTER: straight into the owning rank over NVLink
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (!WHOLE && i >= rows) break;
      const unsigned ra = wacc + (unsigned)(i * 8 * ACC_WPITCH * 4 + j * ACC_WORDS * 4);
      unsigned v = (!WHOLE && none) ? 0u : lane_perm(lds32(ra), lds32(ra + 4), wsel);
      if (CAR) v = lane_addus4(v, __ldg(reinterpret_cast<const unsigned*>(P.car + off + (size_t)i * 8 * P.out_pitch)));
      *reinterpret_cast<unsigned*>(o + (size_t)i * 8 * P.out_pitch) = v;
    }
  }
}

template <bool BAL, int NB, bool SCATTER = false>
__global__ void __launch_bounds__(TMA_THREADS, TMA_MIN_CTAS) k_bev_tma(const TmaParams P) {
  constexpr int SB = 4 * TMA_FS;                  // box bytes of one ring slot
  constexpr int SLOT = TMA_SLOT_BYTES;            // boxes | entries | descriptor
  constexpr int ENT_OFF = SB, DESC_OFF = SB + TMA_EG * 4096;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // slots need 128-byte alignment for cp.async.bulk.tensor; align the base to 1024 (pointer arithmetic only, so the
  // compiler keeps the shared address space)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned* acc = reinterpret_cast<unsigned*>(smem + (size_t)TMA_STAGES * SLOT);   // [NB][ACC_WORDS] packed BGRX
  const unsigned bar_full = smem_u32(acc + NB * ACC_WORDS), bar_empty = bar_full + 8 * TMA_STAGES;
  const unsigned stage0 = smem_u32(smem), acc_u32 = smem_u32(acc);
  __shared__ unsigned long long s_sum[BAL ? 3 * NB : 1];
  const int t = threadIdx.x, lane = t & 31, wrp = t >> 5;
  if (BAL && t < 3 * NB) s_sum[t] = 0ull;
  if (t == 0) {
    for (int s = 0; s < TMA_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);                      // the producer's arrive(.expect_tx)
      mbar_init(bar_empty + 8 * s, TMA_CONSUMERS / 32);    // one arrival per consumer warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int groups = (P.batch + NB - 1) / NB;
  const long long n_units = (long long)P.n_tiles * groups;

  if (t >= TMA_CONSUMERS) {
    // ---------------- producer: one thread turns the plan into ring slots and stays TMA_STAGES slots ahead of the consumers
    if (t == TMA_CONSUMERS) {
      unsigned s = 0, ph = 0;   // ring position: slot, phase of its barriers
#ifdef BEVK_TRACE
      unsigned tn = 0;
#endif
      auto post = [&](uint4 d0, uint4 d1, unsigned tx, const void* ent_src, unsigned ent_bytes, const uint8_t* map, int np, int rs,
                      int bx, int by, int z0) {
        const unsigned slot = stage0 + s * SLOT, full = bar_full + 8 * s;
#ifdef BEVK_TRACE
        const bool tr = P.trace && blockIdx.x < 8 && tn < 512;
        unsigned long long* T = P.trace + ((size_t)blockIdx.x * 512 + tn) * 16;
        if (tr) T[0] = clock64();
#endif
        mbar_wait(bar_empty + 8 * s, ph ^ 1u);   // consumers have left this slot
#ifdef BEVK_TRACE
        if (tr) { T[1] = clock64(); T[6] = tx; T[7] = d0.x; }
#endif
        sts128(slot + DESC_OFF, d0);
        sts128(slot + DESC_OFF + 16, d1);
        if (tx) mbar_expect_tx(full, tx); else mbar_arrive(full);
        if (ent_bytes) bulk_copy(slot + ENT_OFF, ent_src, ent_bytes, full);
        for (int j = 0; j < np; ++j) tma_load_3d(slot + j * rs, map, bx, by, z0 + j * P.n_cam, full);
        if (++s == TMA_STAGES) { s = 0; ph ^= 1u; }
#ifdef BEVK_TRACE
        if (tr) T[2] = clock64();
        ++tn;
#endif
      };
      const bool filtered = P.cam_lo > 0 || P.cam_hi < 8;   // BEVK_MAX_CAMERAS
      const bool words_ok = !BAL && (P.out_pitch & 3) == 0 && (P.canvas_bytes & 3) == 0 && (P.ox & 3) == 0;   // as the consumers decide
      bool prev_generic = false;   // the previous unit left through the generic write-out (reads across the warps' rows)
      // Units are handed out dynamically (one atomic per unit, only this thread needs it: the consumers follow the ring):
      // unit u = tile u / groups of the cost-sorted tile list, frame-set group u % groups -- heavy tiles first, so the
      // CTAs finish together.  The next unit's id and tile record are fetched while the current unit is being posted.
      long long unit = (long long)atomicAdd(P.unit_counter, 1u);
      int4 tile = unit < n_units ? __ldg(P.tiles + (int)(unit / groups)) : make_int4(0, 0, 0, 0);
      while (unit < n_units) {
        const long long next_unit = (long long)atomicAdd(P.unit_counter, 1u);
        const int4 next_tile = next_unit < n_units ? __ldg(P.tiles + (int)(next_unit / groups)) : make_int4(0, 0, 0, 0);
        const int b0 = (int)(unit % groups) * NB;
        const int nb = min(NB, P.batch - b0);
        uint4 d1 = make_uint4((unsigned)tile.x | ((unsigned)tile.y << 16), (unsigned)b0 | ((unsigned)nb << 16), 0u, 0u);
        const bool interior = words_ok && tile.x + TILE <= P.ox1;   // row-wise write-out: warp w reads its own rows only
        // last item of this unit that belongs to a camera of the call
        int last_it = tile.z + tile.w - 1;
        if (filtered)
          for (; last_it >= tile.z; --last_it) {
            const int cam = (short)(__ldg(reinterpret_cast<const int*>(P.items + last_it) + 1) & 0xffff);
            if (cam >= P.cam_lo && cam < P.cam_hi) break;
          }
        if (last_it < tile.z) {   // no camera of the call touches the tile (car hole, or another rank's cameras): zeros --
          // unless the tile lies outside the output window altogether (camera-sharded slabs): then there is nothing to do
          if (!(tile.x >= P.ox1 || tile.x + TILE <= P.ox || tile.y >= P.oy1 || tile.y + TILE <= P.oy)) {
            post(make_uint4((interior ? D_ROWS : D_SYNC) | D_LAST | D_NONE, 0u, 0u, 0u), d1, 0u, nullptr, 0u, nullptr, 0, 0, 0, 0, 0);
            // an interior tile without a camera passes no barrier and reads no accumulator word: a generic write-out before it
            // is still unfenced (tests/test_barrier_rules.py found the sequence edge tile -> empty tile -> rows-first tile)
            if (!interior) prev_generic = true;
          }
        } else {
          int first_cam = -1, prev_orient = -1;
          bool columns = false;   // an item of the unit ran its lanes along canvas y
          int4 n0 = __ldg(reinterpret_cast<const int4*>(P.items + tile.z));
          int4 n1 = __ldg(reinterpret_cast<const int4*>(P.items + tile.z) + 1);
          for (int it = tile.z; it <= last_it; ++it) {
            const int4 i0 = n0, i1 = n1;
            if (it < last_it) {   // the next item's record travels while this one is posted
              n0 = __ldg(reinterpret_cast<const int4*>(P.items + it + 1));
              n1 = __ldg(reinterpret_cast<const int4*>(P.items + it + 1) + 1);
            }
            const int cam = (short)(i0.y & 0xffff), orient = (i0.y >> 16) & 0xff, iflags = (i0.y >> 24) & 0xff;
            if (cam < P.cam_lo || cam >= P.cam_hi) continue;
            const int k0 = i0.z & 0xff, nk = ((i0.z >> 8) & 0xff) - k0;
            unsigned f = 0;
            if (first_cam < 0) {   // other warps may still be writing out rows this item stores into (see D_SYNC above)
              first_cam = cam;
              if (orient || prev_generic) f |= D_SYNC;
            }
            columns |= orient != 0;
            if (cam == first_cam) f |= D_FIRST;                                // this camera stores, later ones add (cv2.add order)
            if (prev_orient >= 0 && prev_orient != orient) f |= D_SYNC;         // accumulator ownership changes with the orientation
            prev_orient = orient;
            if (orient) f |= D_ORIENT;
            if (iflags & ITEM_NOSAT) f |= D_NOSAT;
            if (iflags & ITEM_FULL) f |= D_FULL;
            f |= (unsigned)nk << 16;
            // accumulator walk of the item: lanes along canvas x -> a group is 8 rows; along y -> 8 columns
            const unsigned astep = 4u * (unsigned)(orient ? 8 : 8 * ACC_WPITCH);
            const uint4* ent_src = P.lut + (size_t)i0.x * (TILE * TILE) + k0 * 256;
            const unsigned ent_bytes = (unsigned)nk * 4096u;
            d1.z = (unsigned)cam;
            if (iflags & ITEM_GATHER) {
              post(make_uint4(f | D_GATHER | (it == last_it ? D_LAST | (!columns && interior ? D_ROWS : 0u) : 0u), 0u, (unsigned)k0 * astep, astep),
                   d1, ent_bytes, ent_src, ent_bytes, nullptr, 0, 0, 0, 0, 0);
              continue;
            }
            const uint8_t* map = P.maps + (size_t)((unsigned)i0.z >> 16) * TMA_DESC_BYTES;
            const int rs = i1.z, fpp = min(NB, SB / rs);                       // frame-sets per pass
            f |= (fpp >= 4 ? 0u : (fpp == 2 ? 1u : 2u)) << 20;
            for (int p = 0; p < nb; p += fpp) {
              const int np = min(fpp, nb - p);
              const unsigned fl = (p == 0 ? f : (f & ~D_SYNC)) | ((it == last_it && p + fpp >= nb) ? D_LAST | (!columns && interior ? D_ROWS : 0u) : 0u);
              post(make_uint4(fl, (unsigned)i1.w, (unsigned)k0 * astep + (unsigned)p * (ACC_WORDS * 4), astep), d1,
                   ent_bytes + (unsigned)np * (unsigned)i1.y,
                   ent_src, ent_bytes, map, np, rs, i0.w, i1.x, (b0 + p) * P.n_cam + cam);
            }
          }
          prev_generic = !interior;
        }
        unit = next_unit; tile = next_tile;
      }
      post(make_uint4(D_END, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u), 0u, nullptr, 0u, nullptr, 0, 0, 0, 0, 0);
    }
    return;
  }

  // ---------------- consumers: follow the ring; nothing below reads global memory except GATHER taps and the car overlay
  const unsigned posx = acc_u32 + 4u * (unsigned)(wrp * ACC_WPITCH + lane);   // lanes along canvas x: line k*8+wrp is a row
  const unsigned posy = acc_u32 + 4u * (unsigned)(lane * ACC_WPITCH + wrp);   // lanes along canvas y: line k*8+wrp is a column
  const unsigned ent0 = stage0 + ENT_OFF + (unsigned)t * 16u;
  const bool words_ok = !BAL && (P.out_pitch & 3) == 0 && (P.canvas_bytes & 3) == 0 && (P.ox & 3) == 0;
  unsigned s = 0, ph = 0;
#ifdef BEVK_TRACE
  unsigned tn = 0;
#endif
  for (;;) {
    const unsigned slot = stage0 + s * SLOT;
#ifdef BEVK_TRACE
    const bool tr = P.trace && blockIdx.x < 8 && tn < 512 && t == 0;
    unsigned long long* T = P.trace + ((size_t)blockIdx.x * 512 + tn) * 16;
    ++tn;
    if (tr) T[3] = clock64();
#endif
    mbar_wait(bar_full + 8 * s, ph);                     // descriptor, entries and boxes of this slot have landed
#ifdef BEVK_TRACE
    if (tr) T[4] = clock64();
#endif
    const uint4 d = lds128(slot + DESC_OFF);
    const unsigned flags = d.x;
    if (flags & D_END) break;
    if (flags & D_SYNC) consumer_sync();
    const int nk = (flags >> 16) & 15;
    if (nk) {
      const unsigned aa = ((flags & D_ORIENT) ? posy : posx) + d.z;
      const unsigned ent = ent0 + s * SLOT;
      if (flags & D_GATHER) {
        const uint4 d1 = lds128(slot + DESC_OFF + 16);
        const int b0 = (int)(d1.y & 0xffffu), nb = (int)(d1.y >> 16);
        const uint8_t* frame0 = P.base + (long long)(b0 * P.n_cam + (int)d1.z) * P.frame_stride;
        const long long set_stride = (long long)P.n_cam * P.frame_stride;
#pragma unroll 1
        for (int k = 0; k < nk; ++k)
          gather_entry<NB>(P, lds128(ent + k * 4096), aa + k * d.w, (flags & D_FIRST) != 0, (flags & D_NOSAT) != 0, frame0, set_stride, nb);
      } else {
        const unsigned kind = (flags >> 20) & 3u;
        if (NB == 4 && kind == 0u) tma_pass<(NB == 4 ? 4 : 1), TMA_FS>(ent, nk, slot, d.y, aa, d.w, flags);
        else if (NB == 4 && kind == 1u) tma_pass<(NB == 4 ? 2 : 1), 2 * TMA_FS>(ent, nk, slot, d.y, aa, d.w, flags);
        else tma_pass<1, 0>(ent, nk, slot, d.y, aa, d.w, flags);
      }
    }
    // word 1 (tile, frame-sets) is needed by the slot that ends a unit; it is read before this warp releases the slot
    uint4 d1 = make_uint4(0u, 0u, 0u, 0u);
    if (flags & D_LAST) d1 = lds128(slot + DESC_OFF + 16);
    __syncwarp();
#ifdef BEVK_TRACE
    if (tr) T[5] = clock64();
#endif
    if (elect_one()) mbar_arrive(bar_empty + 8 * s);     // this warp no longer reads the slot
    if (++s == TMA_STAGES) { s = 0; ph ^= 1u; }
#ifdef BEVK_TRACE
    if (tr) T[8] = clock64();
#endif
    if (!(flags & D_LAST)) continue;
    // ---- the unit is complete: write the tile(s)
    const bool none = (flags & D_NONE) != 0;              // tile without a camera (car hole): zeros
    if (!(flags & D_ROWS)) consumer_sync();               // other warps accumulated into the rows this warp writes
#ifdef BEVK_TRACE
    if (tr) T[9] = clock64();
#endif
    const int4 tile = make_int4((int)(d1.x & 0xffffu), (int)(d1.x >> 16), 0, 0);
    const int b0 = (int)(d1.y & 0xffffu), nb = (int)(d1.y >> 16);
    if (tile.x >= P.ox1 || tile.x + TILE <= P.ox || tile.y >= P.oy1 || tile.y + TILE <= P.oy) continue;   // outside the output window
    if (words_ok && tile.x + TILE <= P.ox1) {
      // interior tile: warp w stores rows w, w+8, w+16, w+24, lanes 0..23 one packed-BGR word each (bytes 4l..4l+3 of a
      // row start in BGRX word l + l/3 at byte phase l % 3): four 96-byte row pieces per frame-set and warp
      if (lane < 24) {
        int wp; unsigned wsel;
        tile_word_src(lane, wp, wsel);
        const int gy0 = tile.y + tile_out_row32(wrp, 0);
        const unsigned wacc = acc_u32 + 4u * (unsigned)(tile_out_row32(wrp, 0) * ACC_WPITCH + wp);
        const int rows = max(0, min(4, (P.oy1 - gy0 + 7) / 8));
        const size_t off = (size_t)(gy0 - P.oy) * P.out_pitch + (size_t)(tile.x - P.ox) * 3 + (size_t)lane * 4;
        if (P.car) tile_rows_out<NB, SCATTER, true, false>(P, wacc, wsel, off, rows, b0, nb, none);
        else if (rows == 4 && nb == NB && !none) tile_rows_out<NB, SCATTER, false, true>(P, wacc, wsel, off, rows, b0, nb, none);
        else tile_rows_out<NB, SCATTER, false, false>(P, wacc, wsel, off, rows, b0, nb, none);
      }
      // the next unit may start without a CTA barrier (D_SYNC rules): lanes 24..31, which store nothing here, must not run
      // ahead and overwrite accumulator words that lanes 0..23 of this warp are still reading
      __syncwarp();
#ifdef BEVK_TRACE
      if (tr) T[10] = clock64();
#endif
      continue;
    }
    // edge tiles and the BALANCE variant: thread t -> row t/8, 4 pixels (12 bytes) at pixel 4*(t%8)
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
      if (none) x0 = x1 = x2 = x3 = 0u;
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
        for (int d = 16; d > 0; d >>= 1) {   // every lane takes part (out-of-canvas lanes add 0)
          sb += __shfl_xor_sync(0xffffffffu, sb, d);
          sg += __shfl_xor_sync(0xffffffffu, sg, d);
          sr += __shfl_xor_sync(0xffffffffu, sr, d);
        }
        if (lane == 0) {
          atomicAdd(&s_sum[3 * j + 0], (unsigned long long)sb);
          atomicAdd(&s_sum[3 * j + 1], (unsigned long long)sg);
          atomicAdd(&s_sum[3 * j + 2], (unsigned long long)sr);
        }
      }
      if (!inb) continue;
      uint8_t* o = out_base<SCATTER>(P, b0 + j) + pix_off;
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
      consumer_sync();
      if (t < 3 * nb) { atomicAdd(P.csum + (size_t)(b0 + t / 3) * 3 + (t % 3), s_sum[t]); s_sum[t] = 0ull; }
    }
  }
}
#endif  // __CUDACC__

}  // namespace bevk
