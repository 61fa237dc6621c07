// bevk_api.cu -- C ABI of libbevk.so (see include/bevk.h) over the sm_100a kernels.
// Host side: argument checks, 3x3 inverses the way OpenCV computes them, device
// buffer management, the tile-plan compiler, stream ordering.  No CPU fallback.
// Environment: BEVK_TMA=0 (read at bevk_bev_finalize) builds no TMA plan, so every call takes the gather kernel k_bev --
// the reference the GPU tests compare k_bev_tma with; BEVK_TRACE_FILE (-DBEVK_TRACE builds only) receives a slot timeline.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "../../include/bevk.h"
#include "bevk_kernels.cuh"
#include "bevk_bev.cuh"
#include "bevk_gather4.cuh"
#include "bevk_plan.cuh"
#include "bevk_bev_tma.cuh"
#include "bevk_plan_tma.cuh"
#include "bevk_shard.cuh"

#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges cost nothing unless a profiler injects itself

using namespace bevk;

// ------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(e_ == cudaErrorMemoryAllocation ? BEVK_ERR_OOM : BEVK_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e_), __FILE__, __LINE__);                                     \
  } while (0)
#define RET(call)             \
  do {                        \
    int r_ = (call);          \
    if (r_ != BEVK_OK) return r_; \
  } while (0)

// NVTX range for the lifetime of a scope (visible in nsys / ncu timelines: ingest, render, read-back)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ------------------------------------------------------------------ small helpers
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return BEVK_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    n = (n + 255) & ~size_t(255);
    CU(cudaMalloc(&p, n + 256));   // 256 B of slack: the kernels' 32-bit tap loads may touch 3 bytes past a frame
    cap = n;
    return BEVK_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

static int make_model(int model, const double* K, const double* D, int n_dist, const double* P, int w, int h,
                      CamModel* cm) {
  if (!K || !P || (n_dist > 0 && !D)) return fail(BEVK_ERR_ARG, "null K/D/P");
  if (model != BEVK_MODEL_FISHEYE && model != BEVK_MODEL_PINHOLE) return fail(BEVK_ERR_ARG, "bad camera model %d", model);
  if (w <= 0 || h <= 0) return fail(BEVK_ERR_ARG, "bad map size %dx%d", w, h);
  memset(cm, 0, sizeof *cm);
  if (!inv3(P, cm->iR)) return fail(BEVK_ERR_ARG, "P is singular");
  const int want = model == BEVK_MODEL_FISHEYE ? 4 : 5;
  for (int i = 0; i < want && i < n_dist; ++i) cm->k[i] = D[i];
  cm->fx = K[0]; cm->fy = K[4]; cm->cx = K[2]; cm->cy = K[5];
  cm->model = model; cm->w = w; cm->h = h;
  return BEVK_OK;
}

static int make_homog(const double* H, Homog* hm) {
  if (!H) return fail(BEVK_ERR_ARG, "null H");
  if (!inv3(H, hm->M)) memset(hm->M, 0, sizeof hm->M);   // cv::invert leaves zeros for a singular matrix
  return BEVK_OK;
}

static dim3 grid2d(int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8); }

// ------------------------------------------------------------------ context
struct Undistorter {
  bool valid = false, fused = false;
  CamModel cm;
  DevBuf map1, map2;
};

struct BevCam {
  bool has_maps = false, has_mask = false;
  DevBuf map1, map2;              // device BEV maps
  std::vector<uint8_t> mask;      // host mask
};

struct bevk_ctx {
  int device = 0;
  cudaStream_t own = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_switch = nullptr;
  cudaStream_t copy_stream = nullptr;                      // H2D side of the host-pointer pipeline
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  const void* ptrs_for = nullptr; const void* ptrs_tab = nullptr; long long ptrs_n = 0; size_t ptrs_pad = 0;   // cached frame pointer table
  bool timed = false;
  long long launches = 0;
  DevBuf s_src, s_dst, s_m1, s_m2, s_o1, s_o2;   // scratch for the host-pointer entry points
  Undistorter und[8];
  // BEV engine
  int n_cam = 0, FW = 0, FH = 0, BW = 0, BH = 0;
  BevCam cam[BEVK_MAX_CAMERAS];
  bool planned = false;
  long long n_tiles = 0, n_items = 0, span_px = 0;
  int bev_interp = BEVK_INTER_LINEAR;   // cv2.remap interpolation the BEV LUT is compiled for
  DevBuf d_hptrs;                           // device copy of the mapped host frame pointers (per half)
  const uint8_t** h_hptrs = nullptr;        // pinned staging of those pointers
  cudaEvent_t ev_hp[2] = {nullptr, nullptr};
  long long span_fetch_bytes = 0;           // bytes k_fetch_spans moves per frame-set
  long long last_h2d_bytes = 0;             // host->device bytes of the last bevk_bev_run call
  int cam_box[BEVK_MAX_CAMERAS][DMA_BANDS][4] = {};   // per camera and band: sampled rows [y0,y1), bytes [bx0,bx1)
  DevBuf d_tiles, d_items, d_lut, d_hsv;
  int bev_grid[4] = {0, 0, 0, 0};         // resident CTAs of k_bev<BAL, NB>: index = 2*BAL + {NB=1:0, 4:1}
  DevBuf d_frames, d_ptrs, d_canvas, d_car, d_vsum, d_delta, d_csum;
  DevBuf d_spans, d_bal, d_bal_ptrs;        // BALANCE: sampled row spans per camera, balanced frame copies + their table
  const void* bal_ptrs_for = nullptr; long long bal_ptrs_n = 0; size_t bal_ptrs_pad = 0;
  DevBuf d_user_ptrs;                       // bevk_bev_run_frames: device copy of the caller's frame table
  std::vector<const void*> user_tab;        // ... and what it currently holds
  // TMA-staged kernel (bevk_bev_tma.cuh): its plan, and the tensor maps of the frame stacks seen recently
  bool tma_planned = false;
  long long tma_items = 0, tma_box_bytes = 0, tma_entries = 0, tma_gather_entries = 0;
  std::vector<int2> tma_shapes;
  DevBuf d_ttiles, d_titems, d_tlut, d_unit_counter;
  struct MapSet { const void* base = nullptr; long long stride = 0, frames = 0; DevBuf d; unsigned long long used = 0; };
  MapSet maps[4];
  unsigned long long map_clock = 0;
  int tma_grid[4] = {};                     // resident CTAs of k_bev_tma<BAL, NB>: index = 2*BAL + {NB=1:0, 4:1}
  DevBuf d_stack_ptrs;                      // pointer table of a frame stack (BALANCE pre-passes read frames through a table)
  const void* stack_ptrs_base = nullptr; long long stack_ptrs_stride = 0, stack_ptrs_n = 0;
  int last_path = 0;                        // 1: k_bev (pointer-table gather), 2: k_bev_tma
  // multi-GPU sharding (bevk_shard_*): partition, slab geometry, NCCL communicator
  struct Shard {
    bool configured = false, geometry = false;
    int policy = 0, rank = 0, world = 1;
    int cam_lo[SHARD_MAX_RANKS] = {}, cam_hi[SHARD_MAX_RANKS] = {};
    SlabRect rect[SHARD_MAX_RANKS] = {};
    long long slab_bytes = 0;
    void* comm = nullptr;                   // ncclComm_t
    DevBuf d_slabs;
    long long last_link_bytes = 0;
    // peer-store exchange (bevk_bev_run_scattered): this rank's receive buffer [2 halves][world][own_max][slab_bytes],
    // the same buffer of every peer mapped through CUDA IPC, and a 4-byte-per-rank scratch for the step barrier
    void* recv = nullptr; size_t recv_bytes = 0; int prepared_batch = 0, own_max = 0;
    void* peer_recv[SHARD_MAX_RANKS] = {}; bool attached = false;
    DevBuf d_flag;
    unsigned step = 0;
  } shard;
  // nvJPEG ingest (bevk_jpeg_decode): library handle + decoder state, created on first use
  void* jpeg_handle = nullptr; void* jpeg_state = nullptr;
  DevBuf d_jpeg_frames, d_jpeg_canvas;
  // CUDA graphs captured from the device-pointer entry points (bevk_graph_*)
  bool capturing = false;
  long long capture_launches0 = 0;
  struct Graph { cudaGraph_t g = nullptr; cudaGraphExec_t x = nullptr; long long kernels = 0; };
  std::vector<Graph> graphs;
};

static int use(bevk_ctx* c) {
  if (!c) return fail(BEVK_ERR_ARG, "null ctx");
  CU(cudaSetDevice(c->device));
  return BEVK_OK;
}
#define LAUNCHED(c)                 \
  do {                              \
    (c)->launches++;                \
    CU(cudaGetLastError());         \
  } while (0)

// All bevk_* functions get C linkage from their declarations in include/bevk.h.

int bevk_version(void) { return 100; }
const char* bevk_last_error(void) { return g_err.c_str(); }

int bevk_ctx_create(int device, bevk_ctx** out) {
  if (!out) return fail(BEVK_ERR_ARG, "null out");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(BEVK_ERR_CUDA, "no CUDA device (%s); libbevk has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(BEVK_ERR_ARG, "device %d out of range [0,%d)", device, n);
  CU(cudaSetDevice(device));
  bevk_ctx* c = new (std::nothrow) bevk_ctx;
  if (!c) return fail(BEVK_ERR_OOM, "host allocation failed");
  c->device = device;
  cudaError_t e1 = cudaStreamCreateWithFlags(&c->own, cudaStreamNonBlocking);
  cudaError_t e2 = e1 == cudaSuccess ? cudaEventCreate(&c->ev0) : e1;
  cudaError_t e3 = e2 == cudaSuccess ? cudaEventCreate(&c->ev1) : e2;
  if (e3 != cudaSuccess) {
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->own) cudaStreamDestroy(c->own);
    delete c;
    return fail(BEVK_ERR_CUDA, "context setup: %s", cudaGetErrorString(e3));
  }
  c->stream = c->own;
  *out = c;
  return BEVK_OK;
}

static void shard_release(bevk_ctx* c);
static void jpeg_release(bevk_ctx* c);

int bevk_ctx_destroy(bevk_ctx* c) {
  if (!c) return BEVK_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();   // not c->stream: a caller-owned stream handed to bevk_ctx_set_stream may be gone by now
  for (DevBuf* b : {&c->s_src, &c->s_dst, &c->s_m1, &c->s_m2, &c->s_o1, &c->s_o2, &c->d_tiles, &c->d_items, &c->d_lut,
                    &c->d_hsv, &c->d_frames, &c->d_ptrs, &c->d_canvas, &c->d_car, &c->d_vsum, &c->d_delta, &c->d_csum,
                    &c->d_spans, &c->d_bal, &c->d_bal_ptrs, &c->d_user_ptrs, &c->d_ttiles, &c->d_titems, &c->d_tlut,
                    &c->d_stack_ptrs, &c->d_jpeg_frames, &c->d_jpeg_canvas, &c->d_unit_counter})
    b->release();
  for (auto& m : c->maps) m.d.release();
  shard_release(c);
  jpeg_release(c);
  for (auto& g : c->graphs) { if (g.x) cudaGraphExecDestroy(g.x); if (g.g) cudaGraphDestroy(g.g); }
  for (auto& u : c->und) { u.map1.release(); u.map2.release(); }
  for (auto& k : c->cam) { k.map1.release(); k.map2.release(); }
  cudaEventDestroy(c->ev0);
  cudaEventDestroy(c->ev1);
  if (c->ev_switch) cudaEventDestroy(c->ev_switch);
  if (c->copy_stream) {
    cudaStreamSynchronize(c->copy_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_in[i]); cudaEventDestroy(c->ev_free[i]); cudaEventDestroy(c->ev_hp[i]); }
    if (c->h_hptrs) cudaFreeHost(c->h_hptrs);
    c->d_hptrs.release();
    cudaStreamDestroy(c->copy_stream);
  }
  cudaStreamDestroy(c->own);
  delete c;
  return BEVK_OK;
}

int bevk_ctx_set_stream(bevk_ctx* c, void* s) {
  RET(use(c));
  cudaStream_t next = s ? reinterpret_cast<cudaStream_t>(s) : c->own;
  if (next == c->stream) return BEVK_OK;
  if (c->capturing) return fail(BEVK_ERR_ARG, "cannot change the stream inside a graph capture");
  // Everything this ctx enqueued so far (kernels that read its cached tables, uploads that wrote them) is ordered before
  // whatever it enqueues on the new stream: no host synchronisation, no table is dropped.
  if (!c->ev_switch) CU(cudaEventCreateWithFlags(&c->ev_switch, cudaEventDisableTiming));
  if (cudaEventRecord(c->ev_switch, c->stream) == cudaSuccess) CU(cudaStreamWaitEvent(next, c->ev_switch, 0));
  else cudaGetLastError();   // the old (caller-owned) stream is gone: nothing of it can still be running
  c->stream = next;
  return BEVK_OK;
}

int bevk_ctx_sync(bevk_ctx* c) {
  RET(use(c));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_device_pci_bus_id(int device, char* out, int len) {
  if (!out || len < 16) return fail(BEVK_ERR_ARG, "bus id buffer too small");
  CU(cudaDeviceGetPCIBusId(out, len, device));
  return BEVK_OK;
}

int bevk_host_alloc(uint64_t bytes, void** out) {
  if (!out) return fail(BEVK_ERR_ARG, "null out");
  CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return BEVK_OK;
}
int bevk_host_free(void* p) {
  if (p) CU(cudaFreeHost(p));
  return BEVK_OK;
}

// ------------------------------------------------------------------ K1
int bevk_undistort_map(bevk_ctx* c, int model, const double K[9], const double* D, int n_dist, const double P[9], int w,
                       int h, int16_t* map1, uint16_t* map2) {
  RET(use(c));
  if (!map1 || !map2) return fail(BEVK_ERR_ARG, "null output map");
  CamModel cm;
  RET(make_model(model, K, D, n_dist, P, w, h, &cm));
  const size_t n = (size_t)w * h;
  RET(c->s_m1.ensure(n * 4));
  RET(c->s_m2.ensure(n * 2));
  k_undistort_map<<<grid2d(w, h), 256, 0, c->stream>>>(cm, c->s_m1.as<short2>(), c->s_m2.as<unsigned short>());
  LAUNCHED(c);
  CU(cudaMemcpyAsync(map1, c->s_m1.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(map2, c->s_m2.p, n * 2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

// ------------------------------------------------------------------ gather dispatch
template <int MODE>
static int launch_gather(bevk_ctx* c, const GatherArgs& a, int channels, int interp) {
  if (channels == 3 && interp == BEVK_INTER_LINEAR && (a.dw % 4) == 0 && a.dpitch == (long long)a.dw * 3 && (a.spitch % 4) == 0 &&
      a.spitch < (1ll << 31) / std::max(1, a.sh) && (MODE != 0 || a.map2 != nullptr)) {
    // 4 output pixels per thread, 32-bit tap loads and 12-byte stores
    k_gather4<MODE><<<dim3((a.dw / 4 + 31) / 32, (a.dh + 7) / 8), 256, 0, c->stream>>>(a);
    LAUNCHED(c);
    return BEVK_OK;
  }
  const dim3 g = grid2d(a.dw, a.dh);
#define GO(C, L) k_gather<MODE, C, L><<<g, 256, 0, c->stream>>>(a)
  if (interp == BEVK_INTER_LINEAR) {
    if (channels == 1) GO(1, 1); else if (channels == 3) GO(3, 1); else GO(4, 1);
  } else {
    if (channels == 1) GO(1, 0); else if (channels == 3) GO(3, 0); else GO(4, 0);
  }
#undef GO
  LAUNCHED(c);
  return BEVK_OK;
}

static int check_image(const void* p, int w, int h, int64_t stride, int channels, const char* what) {
  if (!p) return fail(BEVK_ERR_ARG, "null %s", what);
  if (w <= 0 || h <= 0) return fail(BEVK_ERR_ARG, "bad %s size %dx%d", what, w, h);
  if (channels != 1 && channels != 3 && channels != 4) return fail(BEVK_ERR_UNSUPPORTED, "channels must be 1, 3 or 4");
  if (stride < (int64_t)w * channels) return fail(BEVK_ERR_ARG, "%s stride %lld < row bytes", what, (long long)stride);
  return BEVK_OK;
}

static int upload_image(bevk_ctx* c, DevBuf& buf, const uint8_t* src, int w, int h, int64_t stride, int channels) {
  const size_t row = (size_t)w * channels;
  RET(buf.ensure(row * h));
  if ((size_t)stride == row) CU(cudaMemcpyAsync(buf.p, src, row * h, cudaMemcpyHostToDevice, c->stream));   // dense: one DMA
  else CU(cudaMemcpy2DAsync(buf.p, row, src, (size_t)stride, row, h, cudaMemcpyHostToDevice, c->stream));
  return BEVK_OK;
}
static int download_image(bevk_ctx* c, const DevBuf& buf, uint8_t* dst, int w, int h, int64_t stride, int channels) {
  const size_t row = (size_t)w * channels;
  if ((size_t)stride == row) CU(cudaMemcpyAsync(dst, buf.p, row * h, cudaMemcpyDeviceToHost, c->stream));
  else CU(cudaMemcpy2DAsync(dst, (size_t)stride, buf.p, row, row, h, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_remap(bevk_ctx* c, const uint8_t* src, int sw, int sh, int64_t sstride, int channels, const int16_t* map1,
               const uint16_t* map2, int dw, int dh, uint8_t* dst, int64_t dstride, int interp) {
  RET(use(c));
  RET(check_image(src, sw, sh, sstride, channels, "src"));
  RET(check_image(dst, dw, dh, dstride, channels, "dst"));
  if (!map1) return fail(BEVK_ERR_ARG, "null map1");
  if (interp == BEVK_INTER_LINEAR && !map2) return fail(BEVK_ERR_ARG, "INTER_LINEAR needs map2");
  if (interp != BEVK_INTER_LINEAR && interp != BEVK_INTER_NEAREST) return fail(BEVK_ERR_UNSUPPORTED, "interp %d", interp);
  const size_t n = (size_t)dw * dh;
  RET(upload_image(c, c->s_src, src, sw, sh, sstride, channels));
  RET(c->s_m1.ensure(n * 4));
  RET(c->s_m2.ensure(n * 2));
  RET(c->s_dst.ensure(n * channels));
  CU(cudaMemcpyAsync(c->s_m1.p, map1, n * 4, cudaMemcpyHostToDevice, c->stream));
  if (map2) CU(cudaMemcpyAsync(c->s_m2.p, map2, n * 2, cudaMemcpyHostToDevice, c->stream));
  GatherArgs a{};
  a.src = c->s_src.as<uint8_t>(); a.sw = sw; a.sh = sh; a.spitch = (long long)sw * channels;
  a.dst = c->s_dst.as<uint8_t>(); a.dw = dw; a.dh = dh; a.dpitch = (long long)dw * channels;
  a.map1 = c->s_m1.as<short2>(); a.map2 = map2 ? c->s_m2.as<unsigned short>() : nullptr;
  RET(launch_gather<0>(c, a, channels, interp));
  return download_image(c, c->s_dst, dst, dw, dh, dstride, channels);
}

// ------------------------------------------------------------------ cached-map undistortion
int bevk_undistorter_set(bevk_ctx* c, int slot, int model, const double K[9], const double* D, int n_dist,
                         const double P[9], int dw, int dh, int fused) {
  RET(use(c));
  if (slot < 0 || slot >= 8) return fail(BEVK_ERR_ARG, "slot %d out of range", slot);
  Undistorter& u = c->und[slot];
  u.valid = false;
  RET(make_model(model, K, D, n_dist, P, dw, dh, &u.cm));
  u.fused = fused != 0;
  if (!u.fused) {
    const size_t n = (size_t)dw * dh;
    RET(u.map1.ensure(n * 4));
    RET(u.map2.ensure(n * 2));
    k_undistort_map<<<grid2d(dw, dh), 256, 0, c->stream>>>(u.cm, u.map1.as<short2>(), u.map2.as<unsigned short>());
    LAUNCHED(c);
  }
  u.valid = true;
  return BEVK_OK;
}

int bevk_undistorter_maps(bevk_ctx* c, int slot, int16_t* map1, uint16_t* map2) {
  RET(use(c));
  if (slot < 0 || slot >= 8 || !c->und[slot].valid) return fail(BEVK_ERR_ARG, "undistorter slot %d not set", slot);
  if (!map1 || !map2) return fail(BEVK_ERR_ARG, "null output map");
  Undistorter& u = c->und[slot];
  const size_t n = (size_t)u.cm.w * u.cm.h;
  const short2* m1 = u.map1.as<short2>();
  const unsigned short* m2 = u.map2.as<unsigned short>();
  if (u.fused) {   // no resident map: evaluate into scratch
    RET(c->s_m1.ensure(n * 4));
    RET(c->s_m2.ensure(n * 2));
    k_undistort_map<<<grid2d(u.cm.w, u.cm.h), 256, 0, c->stream>>>(u.cm, c->s_m1.as<short2>(), c->s_m2.as<unsigned short>());
    LAUNCHED(c);
    m1 = c->s_m1.as<short2>(); m2 = c->s_m2.as<unsigned short>();
  }
  CU(cudaMemcpyAsync(map1, m1, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(map2, m2, n * 2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_undistort(bevk_ctx* c, int slot, const uint8_t* src, int sw, int sh, int64_t sstride, int channels,
                   uint8_t* dst, int dw, int dh, int64_t dstride, int interp) {
  RET(use(c));
  if (slot < 0 || slot >= 8 || !c->und[slot].valid) return fail(BEVK_ERR_ARG, "undistorter slot %d not set", slot);
  Undistorter& u = c->und[slot];
  if (dw != u.cm.w || dh != u.cm.h)   // the caller sized dst for another map: never write past it
    return fail(BEVK_ERR_ARG, "undistorter slot %d holds a %dx%d map, the caller expects %dx%d", slot, u.cm.w, u.cm.h, dw, dh);
  RET(check_image(src, sw, sh, sstride, channels, "src"));
  RET(check_image(dst, dw, dh, dstride, channels, "dst"));
  if (interp != BEVK_INTER_LINEAR && interp != BEVK_INTER_NEAREST) return fail(BEVK_ERR_UNSUPPORTED, "interp %d", interp);
  RET(upload_image(c, c->s_src, src, sw, sh, sstride, channels));
  RET(c->s_dst.ensure((size_t)dw * dh * channels));
  GatherArgs a{};
  a.src = c->s_src.as<uint8_t>(); a.sw = sw; a.sh = sh; a.spitch = (long long)sw * channels;
  a.dst = c->s_dst.as<uint8_t>(); a.dw = dw; a.dh = dh; a.dpitch = (long long)dw * channels;
  if (u.fused) {
    a.cm = u.cm;
    RET(launch_gather<1>(c, a, channels, interp));
  } else {
    a.map1 = u.map1.as<short2>(); a.map2 = u.map2.as<unsigned short>();
    RET(launch_gather<0>(c, a, channels, interp));
  }
  return download_image(c, c->s_dst, dst, dw, dh, dstride, channels);
}

// ------------------------------------------------------------------ K4 / K2
int bevk_warp_perspective(bevk_ctx* c, const uint8_t* src, int sw, int sh, int64_t sstride, int channels,
                          const double H[9], uint8_t* dst, int dw, int dh, int64_t dstride, int interp) {
  RET(use(c));
  RET(check_image(src, sw, sh, sstride, channels, "src"));
  RET(check_image(dst, dw, dh, dstride, channels, "dst"));
  if (interp != BEVK_INTER_LINEAR && interp != BEVK_INTER_NEAREST) return fail(BEVK_ERR_UNSUPPORTED, "interp %d", interp);
  GatherArgs a{};
  RET(make_homog(H, &a.hm));
  RET(upload_image(c, c->s_src, src, sw, sh, sstride, channels));
  RET(c->s_dst.ensure((size_t)dw * dh * channels));
  a.src = c->s_src.as<uint8_t>(); a.sw = sw; a.sh = sh; a.spitch = (long long)sw * channels;
  a.dst = c->s_dst.as<uint8_t>(); a.dw = dw; a.dh = dh; a.dpitch = (long long)dw * channels;
  RET(launch_gather<2>(c, a, channels, interp));
  return download_image(c, c->s_dst, dst, dw, dh, dstride, channels);
}

int bevk_warp_maps(bevk_ctx* c, const int16_t* map1, const uint16_t* map2, int sw, int sh, const double H[9], int dw,
                   int dh, int16_t* out1, uint16_t* out2) {
  RET(use(c));
  if (!map1 || !map2 || !out1 || !out2) return fail(BEVK_ERR_ARG, "null map pointer");
  if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0) return fail(BEVK_ERR_ARG, "bad size");
  WarpMapsArgs a{};
  RET(make_homog(H, &a.hm));
  const size_t ns = (size_t)sw * sh, nd = (size_t)dw * dh;
  RET(c->s_m1.ensure(ns * 4));
  RET(c->s_m2.ensure(ns * 2));
  RET(c->s_o1.ensure(nd * 4));
  RET(c->s_o2.ensure(nd * 2));
  CU(cudaMemcpyAsync(c->s_m1.p, map1, ns * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->s_m2.p, map2, ns * 2, cudaMemcpyHostToDevice, c->stream));
  a.in1 = c->s_m1.as<short2>(); a.in2 = c->s_m2.as<unsigned short>(); a.sw = sw; a.sh = sh;
  a.out1 = c->s_o1.as<short2>(); a.out2 = c->s_o2.as<unsigned short>(); a.dw = dw; a.dh = dh;
  k_warp_maps<0><<<grid2d(dw, dh), 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  CU(cudaMemcpyAsync(out1, c->s_o1.p, nd * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(out2, c->s_o2.p, nd * 2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

// ------------------------------------------------------------------ BEV engine: setup
int bevk_bev_configure(bevk_ctx* c, int n_cam, int fw, int fh, int bw, int bh) {
  RET(use(c));
  if (n_cam < 1 || n_cam > BEVK_MAX_CAMERAS) return fail(BEVK_ERR_ARG, "n_cam %d out of range", n_cam);
  if (fw <= 0 || fh <= 0 || bw <= 0 || bh <= 0) return fail(BEVK_ERR_ARG, "bad geometry");
  if (fw > 32767 || fh > 32767) return fail(BEVK_ERR_UNSUPPORTED, "frames larger than 32767 px");
  if ((long long)fw * fh * 3 + 16 > 0xffffffffLL) return fail(BEVK_ERR_UNSUPPORTED, "frame too large for 32-bit offsets");
  c->n_cam = n_cam; c->FW = fw; c->FH = fh; c->BW = bw; c->BH = bh;
  c->bev_interp = BEVK_INTER_LINEAR;
  c->planned = false;
  c->tma_planned = false;
  // cached pointer tables are keyed on buffer addresses: a new geometry changes the strides behind the same addresses
  c->ptrs_for = nullptr; c->bal_ptrs_for = nullptr; c->bal_ptrs_n = 0; c->stack_ptrs_base = nullptr;
  for (auto& k : c->cam) { k.has_maps = false; k.has_mask = false; k.mask.clear(); }
  return BEVK_OK;
}

static int need_cam(bevk_ctx* c, int cam) {
  if (c->n_cam == 0) return fail(BEVK_ERR_ARG, "bevk_bev_configure not called");
  if (cam < 0 || cam >= c->n_cam) return fail(BEVK_ERR_ARG, "camera %d out of range", cam);
  return BEVK_OK;
}

int bevk_bev_set_camera(bevk_ctx* c, int cam, const double K[9], const double D[4], const double P[9], int und_w,
                        int und_h, const double H[9]) {
  RET(use(c));
  RET(need_cam(c, cam));
  WarpMapsArgs a{};
  RET(make_model(BEVK_MODEL_FISHEYE, K, D, 4, P, und_w, und_h, &a.cm));
  RET(make_homog(H, &a.hm));
  BevCam& k = c->cam[cam];
  const size_t n = (size_t)c->BW * c->BH;
  RET(k.map1.ensure(n * 4));
  RET(k.map2.ensure(n * 2));
  a.sw = und_w; a.sh = und_h;
  a.out1 = k.map1.as<short2>(); a.out2 = k.map2.as<unsigned short>(); a.dw = c->BW; a.dh = c->BH;
  k_warp_maps<1><<<grid2d(c->BW, c->BH), 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  k.has_maps = true;
  c->planned = false;
  return BEVK_OK;
}

int bevk_bev_set_maps(bevk_ctx* c, int cam, const int16_t* map1, const uint16_t* map2) {
  RET(use(c));
  RET(need_cam(c, cam));
  if (!map1 || !map2) return fail(BEVK_ERR_ARG, "null map");
  BevCam& k = c->cam[cam];
  const size_t n = (size_t)c->BW * c->BH;
  RET(k.map1.ensure(n * 4));
  RET(k.map2.ensure(n * 2));
  CU(cudaMemcpyAsync(k.map1.p, map1, n * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(k.map2.p, map2, n * 2, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  k.has_maps = true;
  c->planned = false;
  return BEVK_OK;
}

int bevk_bev_get_maps(bevk_ctx* c, int cam, int16_t* map1, uint16_t* map2) {
  RET(use(c));
  RET(need_cam(c, cam));
  BevCam& k = c->cam[cam];
  if (!k.has_maps) return fail(BEVK_ERR_ARG, "camera %d has no maps", cam);
  if (!map1 || !map2) return fail(BEVK_ERR_ARG, "null map");
  const size_t n = (size_t)c->BW * c->BH;
  CU(cudaMemcpyAsync(map1, k.map1.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(map2, k.map2.p, n * 2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_bev_set_interpolation(bevk_ctx* c, int interp) {
  RET(use(c));
  if (c->n_cam == 0) return fail(BEVK_ERR_ARG, "bevk_bev_configure not called");
  if (interp != BEVK_INTER_LINEAR && interp != BEVK_INTER_NEAREST) return fail(BEVK_ERR_UNSUPPORTED, "interp %d", interp);
  c->bev_interp = interp;
  c->planned = false;
  return BEVK_OK;
}

int bevk_bev_set_mask(bevk_ctx* c, int cam, const uint8_t* mask) {
  RET(use(c));
  RET(need_cam(c, cam));
  if (!mask) return fail(BEVK_ERR_ARG, "null mask");
  BevCam& k = c->cam[cam];
  k.mask.assign(mask, mask + (size_t)c->BW * c->BH);
  k.has_mask = true;
  c->planned = false;
  return BEVK_OK;
}

int bevk_blend_masks(bevk_ctx* c, const uint8_t* polys, const int32_t* lines, int bw, int bh, uint8_t* out) {
  RET(use(c));
  if (!polys || !lines || !out) return fail(BEVK_ERR_ARG, "null argument");
  if (bw <= 0 || bh <= 0) return fail(BEVK_ERR_ARG, "bad size");
  const size_t n = (size_t)bw * bh * 4;
  RET(c->s_src.ensure(n));
  RET(c->s_dst.ensure(n));
  CU(cudaMemcpyAsync(c->s_src.p, polys, n, cudaMemcpyHostToDevice, c->stream));
  BlendArgs a{};
  a.polys = c->s_src.as<uint8_t>(); a.out = c->s_dst.as<uint8_t>(); a.w = bw; a.h = bh;
  for (int i = 0; i < 8; ++i) for (int j = 0; j < 4; ++j) a.lines[i][j] = lines[i * 4 + j];
  k_blend_masks<<<grid2d(bw, bh), 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  CU(cudaMemcpyAsync(out, c->s_dst.p, n, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

// the instantiations of k_bev_tma: {BAL=0,NB=1}, {0,4}, {1,1}, {1,4}, and the peer-store forms of the first two
static const void* const kTmaFns[6] = {(const void*)k_bev_tma<false, 1>, (const void*)k_bev_tma<false, 4>,
                                       (const void*)k_bev_tma<true, 1>, (const void*)k_bev_tma<true, 4>,
                                       (const void*)k_bev_tma<false, 1, true>, (const void*)k_bev_tma<false, 4, true>};

// Tile-plan compiler: LUT maps + masks -> per-tile item lists and thread-ordered LUT blocks.
int bevk_bev_finalize(bevk_ctx* c) {
  RET(use(c));
  if (c->n_cam == 0) return fail(BEVK_ERR_ARG, "bevk_bev_configure not called");
  const int BW = c->BW, BH = c->BH, FW = c->FW, FH = c->FH, NC = c->n_cam;
  const size_t npx = (size_t)BW * BH;
  std::vector<std::vector<short>> m1(NC);
  std::vector<std::vector<unsigned short>> m2(NC);
  for (int k = 0; k < NC; ++k) {
    if (!c->cam[k].has_maps) return fail(BEVK_ERR_ARG, "camera %d has no maps", k);
    if (!c->cam[k].has_mask) return fail(BEVK_ERR_ARG, "camera %d has no mask", k);
    m1[k].resize(npx * 2);
    m2[k].resize(npx);
    CU(cudaMemcpyAsync(m1[k].data(), c->cam[k].map1.p, npx * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(m2[k].data(), c->cam[k].map2.p, npx * 2, cudaMemcpyDeviceToHost, c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));
  BevPlan plan;
  {
    std::vector<const short*> p1(NC);
    std::vector<const unsigned short*> p2(NC);
    std::vector<const uint8_t*> pm(NC);
    for (int k = 0; k < NC; ++k) { p1[k] = m1[k].data(); p2[k] = m2[k].data(); pm[k] = c->cam[k].mask.data(); }
    build_bev_plan(NC, FW, FH, BW, BH, c->bev_interp == BEVK_INTER_NEAREST, p1.data(), p2.data(), pm.data(), plan);
  }
  std::vector<int4>& tiles = plan.tiles;
  std::vector<BevItem>& items = plan.items;
  std::vector<uint4>& lut = plan.lut;
  std::vector<int2>& spans = plan.spans;
  c->n_tiles = (long long)tiles.size();
  c->n_items = (long long)items.size();
  RET(c->d_tiles.ensure(tiles.size() * sizeof(int4)));
  RET(c->d_items.ensure(std::max<size_t>(1, items.size()) * sizeof(BevItem)));
  RET(c->d_lut.ensure(std::max<size_t>(1, lut.size()) * sizeof(uint4)));
  CU(cudaMemcpyAsync(c->d_tiles.p, tiles.data(), tiles.size() * sizeof(int4), cudaMemcpyHostToDevice, c->stream));
  if (!items.empty()) {
    CU(cudaMemcpyAsync(c->d_items.p, items.data(), items.size() * sizeof(BevItem), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_lut.p, lut.data(), lut.size() * sizeof(uint4), cudaMemcpyHostToDevice, c->stream));
  }
  RET(c->d_spans.ensure(spans.size() * sizeof(int2)));
  CU(cudaMemcpyAsync(c->d_spans.p, spans.data(), spans.size() * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
  c->span_px = 0;
  for (const auto& sp : spans) c->span_px += sp.y - sp.x;
  // Host-path ingest: page-locked frames are read span by span (k_fetch_spans), pageable ones as a few DMA
  // rectangles per frame (plan_bands); BALANCE needs whole frames (its V means cover them).
  c->span_fetch_bytes = 0;
  for (const auto& sp : spans)
    if (sp.y > sp.x) c->span_fetch_bytes += std::min<int>(FW * 3, (3 * sp.y + 12 + 15) & ~15) - (std::max(0, 3 * sp.x - 12) & ~15);
  for (int k = 0; k < NC; ++k) plan_bands(spans.data() + (size_t)k * FH, FW, FH, c->cam_box[k]);
  // OpenCV's 8-bit HSV division tables (color_hsv: sdiv_table / hdiv_table180, hsv_shift = 12)
  std::vector<int> tab(512, 0);
  for (int i = 1; i < 256; ++i) {
    tab[i] = (int)std::nearbyint((255 << 12) / (1. * i));
    tab[256 + i] = (int)std::nearbyint((180 << 12) / (6. * i));
  }
  RET(c->d_hsv.ensure(512 * sizeof(int)));
  CU(cudaMemcpyAsync(c->d_hsv.p, tab.data(), 512 * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  // ---- the TMA-staged kernel's plan (frames whose row pitch is a multiple of 16 bytes)
  c->tma_planned = false;
  {
    TmaPlan tp;
    std::vector<const short*> p1(NC);
    std::vector<const unsigned short*> p2(NC);
    std::vector<const uint8_t*> pm(NC);
    for (int k = 0; k < NC; ++k) { p1[k] = m1[k].data(); p2[k] = m2[k].data(); pm[k] = c->cam[k].mask.data(); }
    const char* env = getenv("BEVK_TMA");
    const bool want = !(env && atoi(env) == 0) && ((unsigned)FW * 3u) % 16u == 0;
    if (want) {
      build_tma_plan(NC, FW, FH, BW, BH, c->bev_interp == BEVK_INTER_NEAREST, p1.data(), p2.data(), pm.data(), TMA_FS, true, tp);
      RET(c->d_ttiles.ensure(tp.tiles.size() * sizeof(int4)));
      RET(c->d_titems.ensure(std::max<size_t>(1, tp.items.size()) * sizeof(TmaItem)));
      RET(c->d_tlut.ensure(std::max<size_t>(1, tp.lut.size()) * sizeof(uint4)));
      CU(cudaMemcpyAsync(c->d_ttiles.p, tp.tiles.data(), tp.tiles.size() * sizeof(int4), cudaMemcpyHostToDevice, c->stream));
      if (!tp.items.empty()) {
        CU(cudaMemcpyAsync(c->d_titems.p, tp.items.data(), tp.items.size() * sizeof(TmaItem), cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(c->d_tlut.p, tp.lut.data(), tp.lut.size() * sizeof(uint4), cudaMemcpyHostToDevice, c->stream));
      }
      CU(cudaStreamSynchronize(c->stream));
      c->tma_shapes = tp.shapes;
      c->tma_items = (long long)tp.items.size(); c->tma_box_bytes = tp.box_bytes;
      c->tma_entries = tp.tma_entries; c->tma_gather_entries = tp.gather_entries;
      for (auto& m : c->maps) m.base = nullptr;   // tensor maps are per shape table
      c->tma_planned = true;
    }
  }
  if (c->tma_planned && c->tma_grid[0] == 0) {
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, c->device));
    for (int i = 0; i < 6; ++i) {
      int per_sm = 0;
      const size_t smem = bev_tma_smem_bytes(i % 2 ? 4 : 1);
      CU(cudaFuncSetAttribute(kTmaFns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      // two CTAs fill the SM's shared memory to within 448 bytes: ask for the full carve-out
      CU(cudaFuncSetAttribute(kTmaFns[i], cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kTmaFns[i], TMA_THREADS, smem));
      if (i < 4) c->tma_grid[i] = std::max(1, per_sm) * prop.multiProcessorCount;
    }
  }
  if (c->bev_grid[0] == 0) {   // persistent grid = resident CTAs of each variant
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, c->device));
    const void* fn[4] = {(const void*)k_bev<false, 1>, (const void*)k_bev<false, 4>, (const void*)k_bev<true, 1>,
                         (const void*)k_bev<true, 4>};
    for (int i = 0; i < 4; ++i) {
      int per_sm = 0;
      const size_t smem = bev_smem_bytes(i >= 2, i % 2 ? 4 : 1);
      CU(cudaFuncSetAttribute(fn[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn[i], 256, smem));
      c->bev_grid[i] = std::max(1, per_sm) * prop.multiProcessorCount;
    }
  }
  c->planned = true;
  c->shard.geometry = false;   // slabs follow the masks
  return BEVK_OK;
}

int bevk_bev_plan_info(bevk_ctx* c, int64_t* n_tiles, int64_t* n_items, int64_t* lut_bytes) {
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if (n_tiles) *n_tiles = c->n_tiles;
  if (n_items) *n_items = c->n_items;
  if (lut_bytes) *lut_bytes = c->n_items * TILE * TILE * (int64_t)sizeof(uint4);
  return BEVK_OK;
}

int bevk_bev_tma_plan_info(bevk_ctx* c, int64_t* n_items, int64_t* n_shapes, int64_t* box_bytes, int64_t* tma_entries,
                           int64_t* gather_entries) {
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  const bool t = c->tma_planned;
  if (n_items) *n_items = t ? c->tma_items : 0;
  if (n_shapes) *n_shapes = t ? (int64_t)c->tma_shapes.size() : 0;
  if (box_bytes) *box_bytes = t ? c->tma_box_bytes : 0;
  if (tma_entries) *tma_entries = t ? c->tma_entries : 0;
  if (gather_entries) *gather_entries = t ? c->tma_gather_entries : 0;
  return BEVK_OK;
}

int64_t bevk_bev_last_h2d_bytes(bevk_ctx* c) { return c ? c->last_h2d_bytes : 0; }

int bevk_bev_host_copy_bytes(bevk_ctx* c, int flags, int64_t* h2d, int64_t* d2h) {
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  int64_t up = 0;
  for (int k = 0; k < c->n_cam; ++k) {
    if (flags & BEVK_FLAG_BALANCE) { up += (int64_t)c->FW * c->FH * 3; continue; }
    for (int bnd = 0; bnd < DMA_BANDS; ++bnd)
      up += (int64_t)(c->cam_box[k][bnd][1] - c->cam_box[k][bnd][0]) * (c->cam_box[k][bnd][3] - c->cam_box[k][bnd][2]);
  }
  if (h2d) *h2d = up;
  if (d2h) *d2h = (int64_t)c->BW * c->BH * 3;
  return BEVK_OK;
}

// ------------------------------------------------------------------ BEV engine: run
// Where the frames of a call live: a device table of frame pointers (any layout), or a frame STACK (frame i at
// base + i * stride), which is what the TMA-staged kernel's 3-D tensor maps describe.
struct FrameSrc {
  const void* table = nullptr;
  const uint8_t* base = nullptr;
  long long stride = 0;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  }
  return fn;
}

// Tensor maps (one per box shape of the plan) of the frame stack (base, stride, frames): uint32[frames][FH][pitch/4].
static int stack_maps(bevk_ctx* c, const uint8_t* base, long long stride, long long frames, const uint8_t** d_maps) {
  bevk_ctx::MapSet* slot = &c->maps[0];
  for (auto& m : c->maps) {
    if (m.base == base && m.stride == stride && m.frames >= frames) { m.used = ++c->map_clock; *d_maps = m.d.as<uint8_t>(); return BEVK_OK; }
    if (m.used < slot->used) slot = &m;
  }
  EncodeTiledFn enc = encode_tiled();
  if (!enc) return fail(BEVK_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available from this driver");
  static_assert(sizeof(CUtensorMap) == TMA_DESC_BYTES, "tensor map size");
  const size_t n = c->tma_shapes.size();
  std::vector<CUtensorMap> maps(std::max<size_t>(1, n));
  const cuuint64_t dims[3] = {(cuuint64_t)c->FW * 3u / 4u, (cuuint64_t)c->FH, (cuuint64_t)frames};
  const cuuint64_t strides[2] = {(cuuint64_t)c->FW * 3u, (cuuint64_t)stride};
  const cuuint32_t estr[3] = {1, 1, 1};
  for (size_t i = 0; i < n; ++i) {
    const cuuint32_t box[3] = {(cuuint32_t)c->tma_shapes[i].x, (cuuint32_t)c->tma_shapes[i].y, 1};
    const CUresult r = enc(&maps[i], CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
      return fail(BEVK_ERR_CUDA, "cuTensorMapEncodeTiled(box %u x %u words, stride %lld) failed: %d", box[0], box[1], stride, (int)r);
  }
  // the slot being replaced may still be read by launches in flight on this stream: stream order protects it
  RET(slot->d.ensure(maps.size() * sizeof(CUtensorMap)));
  CU(cudaMemcpyAsync(slot->d.p, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));   // maps is a stack-lifetime staging vector
  slot->base = base; slot->stride = stride; slot->frames = frames; slot->used = ++c->map_clock;
  *d_maps = slot->d.as<uint8_t>();
  return BEVK_OK;
}

__global__ void k_fill_ptrs(const uint8_t** table, const uint8_t* base, long long stride, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) table[i] = base + (long long)i * stride;
}

// pointer table of a frame stack (the BALANCE pre-passes and the round-1 gather kernel read frames through a table)
static int stack_table(bevk_ctx* c, const uint8_t* base, long long stride, int n, const void** table) {
  RET(c->d_stack_ptrs.ensure(sizeof(void*) * (size_t)n));
  if (c->stack_ptrs_base != base || c->stack_ptrs_stride != stride || c->stack_ptrs_n < n) {
    k_fill_ptrs<<<(n + 255) / 256, 256, 0, c->stream>>>(c->d_stack_ptrs.as<const uint8_t*>(), base, stride, n);
    LAUNCHED(c);
    c->stack_ptrs_base = base; c->stack_ptrs_stride = stride; c->stack_ptrs_n = n;
  }
  *table = c->d_stack_ptrs.p;
  return BEVK_OK;
}

static int launch_bev_tma(bevk_ctx* c, const TmaParams& P, int nbu, bool bal) {
  const long long units = c->n_tiles * ((P.batch + nbu - 1) / nbu);
  const int variant = (bal ? 2 : 0) + (nbu == 4 ? 1 : 0);
  const unsigned blocks = (unsigned)std::max<long long>(1, std::min<long long>(units, c->tma_grid[variant]));
  const size_t smem = bev_tma_smem_bytes(nbu);
  const bool scatter = P.world != 0;   // peer-store output: only without BALANCE (run_device checks)
#ifdef BEVK_TRACE
  // slot timeline (tools/gpu/trace_slots.py): the 12th launch of the process records clock64 stamps of the first 8 CTAs
  // into BEVK_TRACE_FILE; a -DBEVK_TRACE build is for this measurement only
  static unsigned long long* d_trace = nullptr;
  static int n_launch = 0;
  constexpr size_t kTraceWords = 8 * 512 * 16;
  TmaParams PT = P;
  const char* trace_file = getenv("BEVK_TRACE_FILE");
  if (trace_file) {
    if (!d_trace) CU(cudaMalloc(&d_trace, kTraceWords * 8));
    if (++n_launch == 12) { CU(cudaMemsetAsync(d_trace, 0, kTraceWords * 8, c->stream)); PT.trace = d_trace; }
  }
  void* args[] = {&PT};
#else
  void* args[] = {const_cast<TmaParams*>(&P)};
#endif
  CU(cudaLaunchKernel(kTmaFns[scatter ? 4 + (nbu == 4 ? 1 : 0) : variant], dim3(blocks), dim3(TMA_THREADS), args, smem, c->stream));
  LAUNCHED(c);
#ifdef BEVK_TRACE
  if (trace_file && n_launch == 12) {
    CU(cudaStreamSynchronize(c->stream));
    std::vector<unsigned long long> h(kTraceWords);
    CU(cudaMemcpy(h.data(), d_trace, kTraceWords * 8, cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(trace_file, "wb")) { fwrite(h.data(), 8, h.size(), f); fclose(f); }
  }
#endif
  return BEVK_OK;
}

// Output window of a render: the full canvas by default; camera-sharded runs render the tile-aligned bounding box of
// their cameras' masks ("slab") with its own pitch and frame-set stride.
struct OutWin {
  int pitch = 0, ox = 0, oy = 0, ox1 = 0, oy1 = 0; long long stride = 0;
  // scattered mode (peer stores): frame-set b -> peer[b % world] + src_off + (b / world) * stride
  uint8_t* peer[SHARD_MAX_RANKS] = {}; int world = 0; long long src_off = 0;
};

static int run_device(bevk_ctx* c, FrameSrc src, int batch, const void* d_car, int flags, void* d_out, int cam_lo, int cam_hi,
                      const OutWin* win = nullptr) {
  NvtxRange nvtx_render("bevk render (fused BEV kernels)");
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if ((!src.table && !src.base) || (!d_out && !(win && win->world))) return fail(BEVK_ERR_ARG, "null device pointer");
  if (batch < 1 || batch > 65535) return fail(BEVK_ERR_ARG, "batch %d out of range [1,65535]", batch);
  const bool bal = (flags & BEVK_FLAG_BALANCE) != 0;
  const int nf = batch * c->n_cam;
  if (bal && nf > 65535) return fail(BEVK_ERR_ARG, "batch %d x %d cameras exceeds the 65535 frames of a BALANCE call", batch, c->n_cam);
  BevParams P{};
  P.n_cam = c->n_cam; P.FW = c->FW; P.FH = c->FH; P.pitch = (unsigned)c->FW * 3u;
  P.tiles = c->d_tiles.as<int4>(); P.items = c->d_items.as<BevItem>(); P.lut = c->d_lut.as<uint4>();
  P.out = reinterpret_cast<uint8_t*>(d_out); P.BW = c->BW; P.BH = c->BH;
  P.canvas_bytes = (long long)c->BW * c->BH * 3;
  P.out_pitch = c->BW * 3; P.ox = 0; P.oy = 0; P.ox1 = c->BW; P.oy1 = c->BH;
  if (win) {
    if (bal || d_car) return fail(BEVK_ERR_ARG, "balance and the car overlay need the full canvas");
    P.canvas_bytes = win->stride; P.out_pitch = win->pitch; P.ox = win->ox; P.oy = win->oy; P.ox1 = win->ox1; P.oy1 = win->oy1;
  }
  P.car = reinterpret_cast<const uint8_t*>(d_car);
  P.cam_lo = cam_lo; P.cam_hi = cam_hi;
  P.n_tiles = (int)c->n_tiles; P.batch = batch;
  // frame-sets per work unit: 4 amortises the LUT decode over a batch; 1 for single frames
  const int nbu = batch >= 4 ? 4 : 1;
  if (c->timed && !c->capturing) CU(cudaEventRecord(c->ev0, c->stream));
  FrameSrc gsrc = src;                         // what the fused gather reads
  if (bal) {
    RET(c->d_vsum.ensure((size_t)nf * 8));
    RET(c->d_delta.ensure((size_t)nf * 4));
    RET(c->d_csum.ensure((size_t)batch * 24));
    CU(cudaMemsetAsync(c->d_vsum.p, 0, (size_t)nf * 8, c->stream));
    CU(cudaMemsetAsync(c->d_csum.p, 0, (size_t)batch * 24, c->stream));
    const void* table = src.table;
    if (!table) RET(stack_table(c, src.base, src.stride, nf, &table));
    const uint8_t* const* srcs = reinterpret_cast<const uint8_t* const*>(table);
    const long long frame_bytes = (long long)P.pitch * c->FH;
    const int blocks = (int)std::max<long long>(1, std::min<long long>(148 * 4 / std::max(1, std::min(nf, 64)) + 1, frame_bytes / (48 * 256) + 1));
    k_vsum<<<dim3(blocks, nf), 256, 0, c->stream>>>(srcs, frame_bytes, c->d_vsum.as<unsigned long long>());
    LAUNCHED(c);
    k_delta<<<(batch + 127) / 128, 128, 0, c->stream>>>(c->d_vsum.as<unsigned long long>(), c->n_cam, batch,
                                                         (double)c->FW * (double)c->FH, c->d_delta.as<int>());
    LAUNCHED(c);
    // luminance_balance once per sampled source pixel into balanced frame copies, then the ordinary
    // fused gather reads those copies
    const size_t fpad = ((size_t)frame_bytes + 255) & ~size_t(255);
    RET(c->d_bal.ensure(fpad * nf));
    RET(c->d_bal_ptrs.ensure(sizeof(void*) * nf));
    if (c->bal_ptrs_for != c->d_bal.p || c->bal_ptrs_n != nf || c->bal_ptrs_pad != fpad) {
      k_fill_ptrs<<<(nf + 255) / 256, 256, 0, c->stream>>>(c->d_bal_ptrs.as<const uint8_t*>(), c->d_bal.as<uint8_t>(), (long long)fpad, nf);
      LAUNCHED(c);
      c->bal_ptrs_for = c->d_bal.p; c->bal_ptrs_n = nf; c->bal_ptrs_pad = fpad;
    }
    k_lum_spans<<<dim3((c->FH + LUM_ROWS - 1) / LUM_ROWS, nf), 128, 0, c->stream>>>(srcs, c->d_bal_ptrs.as<uint8_t*>(), c->d_spans.as<int2>(), c->n_cam,
                                                       c->FW, c->FH, c->d_delta.as<int>(), c->d_hsv.as<int>());
    LAUNCHED(c);
    gsrc.table = c->d_bal_ptrs.p; gsrc.base = c->d_bal.as<uint8_t>(); gsrc.stride = (long long)fpad;
    P.csum = c->d_csum.as<unsigned long long>();
  }
  // TMA-staged kernel for frame stacks (16-byte aligned base and stride); pointer-table gather otherwise
  const bool use_tma = c->tma_planned && gsrc.base && (reinterpret_cast<uintptr_t>(gsrc.base) & 15) == 0 && (gsrc.stride & 15) == 0 &&
                       gsrc.stride >= (long long)P.pitch * c->FH;
  if (use_tma) {
    TmaParams T{};
    RET(stack_maps(c, gsrc.base, gsrc.stride, nf, &T.maps));
    T.base = gsrc.base; T.frame_stride = gsrc.stride;
    T.n_cam = P.n_cam; T.FW = P.FW; T.FH = P.FH; T.pitch = P.pitch;
    T.tiles = c->d_ttiles.as<int4>(); T.items = c->d_titems.as<TmaItem>(); T.lut = c->d_tlut.as<uint4>();
    T.n_tiles = P.n_tiles; T.batch = batch; T.out = P.out; T.BW = P.BW; T.BH = P.BH; T.canvas_bytes = P.canvas_bytes;
    T.car = P.car; T.csum = P.csum; T.cam_lo = cam_lo; T.cam_hi = cam_hi;
    T.out_pitch = P.out_pitch; T.ox = P.ox; T.oy = P.oy; T.ox1 = P.ox1; T.oy1 = P.oy1;
    if (win && win->world) { for (int r = 0; r < SHARD_MAX_RANKS; ++r) T.peer[r] = win->peer[r]; T.world = win->world; T.src_off = win->src_off; }
    RET(c->d_unit_counter.ensure(256));
    CU(cudaMemsetAsync(c->d_unit_counter.p, 0, 4, c->stream));
    T.unit_counter = c->d_unit_counter.as<unsigned>();
    RET(launch_bev_tma(c, T, nbu, bal));
    c->last_path = 2;
  } else {
    if (win && win->world) return fail(BEVK_ERR_UNSUPPORTED, "peer-store output needs the TMA-staged kernel (a 16-byte friendly frame stack)");
    if (!gsrc.table) RET(stack_table(c, gsrc.base, gsrc.stride, nf, &gsrc.table));
    P.srcs = reinterpret_cast<const uint8_t* const*>(gsrc.table);
    const long long units = c->n_tiles * ((batch + nbu - 1) / nbu);
    const int variant = (bal ? 2 : 0) + (nbu == 4 ? 1 : 0);
    const unsigned bev_blocks = (unsigned)std::max<long long>(1, std::min<long long>(units, c->bev_grid[variant]));
    const size_t bev_smem = bev_smem_bytes(bal, nbu);
    if (bal) {
      if (nbu == 4) k_bev<true, 4><<<bev_blocks, 256, bev_smem, c->stream>>>(P);
      else k_bev<true, 1><<<bev_blocks, 256, bev_smem, c->stream>>>(P);
    } else {
      if (nbu == 4) k_bev<false, 4><<<bev_blocks, 256, bev_smem, c->stream>>>(P);
      else k_bev<false, 1><<<bev_blocks, 256, bev_smem, c->stream>>>(P);
    }
    LAUNCHED(c);
    c->last_path = 1;
  }
  if (bal) {
    const int gblocks = (int)std::max<long long>(1, std::min<long long>(P.canvas_bytes / (12 * 256) + 1, 148 * 8 / std::max(1, std::min(batch, 64)) + 1));
    k_gain<<<dim3(gblocks, batch), 256, 0, c->stream>>>(P.out, P.canvas_bytes, (double)c->BW * (double)c->BH,
                                                        c->d_csum.as<unsigned long long>(), P.car);
    LAUNCHED(c);
  }
  if (c->timed && !c->capturing) CU(cudaEventRecord(c->ev1, c->stream));
  return BEVK_OK;
}

static FrameSrc table_src(const void* d_srcs) { FrameSrc s; s.table = d_srcs; return s; }
static FrameSrc stack_src(const void* base, long long stride) { FrameSrc s; s.base = reinterpret_cast<const uint8_t*>(base); s.stride = stride; return s; }

int bevk_bev_run_device(bevk_ctx* c, const void* d_srcs, int batch, const void* d_car, int flags, void* d_out) {
  RET(use(c));
  c->timed = true;
  return run_device(c, table_src(d_srcs), batch, d_car, flags, d_out, 0, BEVK_MAX_CAMERAS);
}

// frames[i] == frames[0] + i * stride with a 16-byte friendly stride?  (a frame stack: the TMA-staged kernel applies)
static bool affine_table(const void* const* frames, size_t n, long long* stride) {
  const uintptr_t b = reinterpret_cast<uintptr_t>(frames[0]);
  if (n == 1) { *stride = 1ll << 32; return (b & 15) == 0; }   // a single frame is a stack of one
  const long long st = (long long)(reinterpret_cast<uintptr_t>(frames[1]) - b);
  if (st <= 0 || (st & 15) || (b & 15)) return false;
  for (size_t i = 2; i < n; ++i)
    if (reinterpret_cast<uintptr_t>(frames[i]) != b + (uintptr_t)st * i) return false;
  *stride = st;
  return true;
}

int bevk_bev_run_frames(bevk_ctx* c, const void* const* frames, int batch, const void* d_car, int flags, void* d_out) {
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if (!frames || !d_out) return fail(BEVK_ERR_ARG, "null pointer");
  if (batch < 1) return fail(BEVK_ERR_ARG, "batch must be >= 1");
  const size_t n = (size_t)batch * c->n_cam;
  for (size_t i = 0; i < n; ++i)
    if (!frames[i] || (reinterpret_cast<uintptr_t>(frames[i]) & 3)) return fail(BEVK_ERR_ARG, "frame %zu null or not 4-byte aligned", i);
  long long stride = 0;
  if (c->tma_planned && affine_table(frames, n, &stride)) {   // no table upload at all
    c->timed = true;
    return run_device(c, stack_src(frames[0], stride), batch, d_car, flags, d_out, 0, BEVK_MAX_CAMERAS);
  }
  if (c->user_tab.size() != n || memcmp(c->user_tab.data(), frames, n * sizeof(void*)) != 0) {
    RET(c->d_user_ptrs.ensure(n * sizeof(void*)));
    c->user_tab.assign(frames, frames + n);
    // pageable source: the driver stages it before returning, and stream order protects launches still reading the old table
    const cudaError_t e = cudaMemcpyAsync(c->d_user_ptrs.p, c->user_tab.data(), n * sizeof(void*), cudaMemcpyHostToDevice, c->stream);
    if (e != cudaSuccess) {
      c->user_tab.clear();   // nothing cached: the next call uploads again
      return fail(BEVK_ERR_CUDA, "frame table upload: %s", cudaGetErrorString(e));
    }
  }
  c->timed = true;
  return run_device(c, table_src(c->d_user_ptrs.p), batch, d_car, flags, d_out, 0, BEVK_MAX_CAMERAS);
}

static int check_stack(bevk_ctx* c, const void* d_frames, int64_t frame_stride) {
  if (!d_frames) return fail(BEVK_ERR_ARG, "null frame stack");
  if (reinterpret_cast<uintptr_t>(d_frames) & 3) return fail(BEVK_ERR_ARG, "frame stack not 4-byte aligned");
  if (frame_stride < (int64_t)c->FW * c->FH * 3 || (frame_stride & 3)) return fail(BEVK_ERR_ARG, "frame_stride %lld smaller than a frame or not a multiple of 4", (long long)frame_stride);
  return BEVK_OK;
}

int bevk_bev_run_stack(bevk_ctx* c, const void* d_frames, int64_t frame_stride, int batch, const void* d_car, int flags, void* d_out) {
  RET(use(c));
  RET(check_stack(c, d_frames, frame_stride));
  c->timed = true;
  return run_device(c, stack_src(d_frames, frame_stride), batch, d_car, flags, d_out, 0, BEVK_MAX_CAMERAS);
}

int bevk_bev_run_stack_cams(bevk_ctx* c, const void* d_frames, int64_t frame_stride, int batch, int cam_lo, int cam_hi, void* d_out) {
  RET(use(c));
  RET(check_stack(c, d_frames, frame_stride));
  if (cam_lo < 0 || cam_hi > c->n_cam || cam_lo > cam_hi) return fail(BEVK_ERR_ARG, "bad camera range [%d,%d)", cam_lo, cam_hi);
  c->timed = true;
  return run_device(c, stack_src(d_frames, frame_stride), batch, nullptr, 0, d_out, cam_lo, cam_hi);
}

int bevk_bev_last_path(bevk_ctx* c) { return c ? c->last_path : 0; }

int bevk_bev_run_device_cams(bevk_ctx* c, const void* d_srcs, int batch, int cam_lo, int cam_hi, void* d_out) {
  RET(use(c));
  if (cam_lo < 0 || cam_hi > c->n_cam || cam_lo > cam_hi) return fail(BEVK_ERR_ARG, "bad camera range [%d,%d)", cam_lo, cam_hi);
  c->timed = true;
  return run_device(c, table_src(d_srcs), batch, nullptr, 0, d_out, cam_lo, cam_hi);
}

int bevk_sat_sum_device(bevk_ctx* c, const void* const* parts, int n, uint64_t bytes, const void* d_car, void* d_out) {
  RET(use(c));
  if (!parts || !d_out || n < 1 || n > BEVK_MAX_CAMERAS) return fail(BEVK_ERR_ARG, "bad partial list");
  SatSumArgs a{};
  for (int i = 0; i < n; ++i) {
    if (!parts[i] || (reinterpret_cast<uintptr_t>(parts[i]) & 15)) return fail(BEVK_ERR_ARG, "partial %d null or not 16-B aligned", i);
    a.parts[i] = reinterpret_cast<const uint8_t*>(parts[i]);
  }
  if ((reinterpret_cast<uintptr_t>(d_out) & 15) || (d_car && (reinterpret_cast<uintptr_t>(d_car) & 15)))
    return fail(BEVK_ERR_ARG, "out/car not 16-B aligned");
  a.n = n; a.bytes = bytes; a.car = reinterpret_cast<const uint8_t*>(d_car); a.out = reinterpret_cast<uint8_t*>(d_out);
  const int blocks = (int)std::max<uint64_t>(1, std::min<uint64_t>(148 * 8, bytes / (16 * 256) + 1));
  k_sat_sum<<<blocks, 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  return BEVK_OK;
}

// Frame-sets per chunk of the host pipeline: 4 = one kernel work unit; finer chunks shorten pipeline fill / drain.
// Measured end to end on 1x B200 at the bench workload (power limit not recorded; profiles/r01_e2e_probe.txt): chunk 4
// 4.295 ms, 2 4.313 ms, 8 4.598 ms per 32 frame-sets.
constexpr int kHostChunk = 4;

int bevk_bev_run(bevk_ctx* c, const uint8_t* const* srcs, int64_t src_stride, int batch, const uint8_t* car, int flags,
                 uint8_t* out) {
  NvtxRange nvtx_call("bevk_bev_run (host frames -> host canvases)");
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if (!srcs || !out) return fail(BEVK_ERR_ARG, "null host pointer");
  if (batch < 1) return fail(BEVK_ERR_ARG, "batch must be >= 1");
  const size_t row = (size_t)c->FW * 3, fbytes = row * c->FH, fpad = (fbytes + 255) & ~size_t(255);
  if (src_stride < (int64_t)row) return fail(BEVK_ERR_ARG, "src_stride %lld < row bytes", (long long)src_stride);
  const size_t cbytes = (size_t)c->BW * c->BH * 3;
  // Two-deep pipeline over chunks of frame-sets: the H2D copies of chunk i+1 run on the copy
  // stream while chunk i is rendered and its canvases go back on the main stream, so the two
  // PCIe directions overlap and the kernel hides under the copies.
  const int chunk = std::min(batch, kHostChunk);
  const size_t set_frames = (size_t)c->n_cam;
  RET(c->d_frames.ensure(fpad * set_frames * chunk * 2));
  RET(c->d_ptrs.ensure(sizeof(void*) * set_frames * chunk * 2));
  RET(c->d_canvas.ensure(cbytes * chunk * 2));
  if (!c->copy_stream) {
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CU(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&c->ev_free[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&c->ev_hp[i], cudaEventDisableTiming));
    }
  }
  if (car) {
    RET(c->d_car.ensure(cbytes));
    CU(cudaMemcpyAsync(c->d_car.p, car, cbytes, cudaMemcpyHostToDevice, c->stream));
  }
  if (c->ptrs_for != c->d_frames.p || c->ptrs_tab != c->d_ptrs.p || c->ptrs_n != (long long)(set_frames * chunk * 2) || c->ptrs_pad != fpad) {
    std::vector<const uint8_t*> ptrs(set_frames * chunk * 2);
    for (size_t i = 0; i < ptrs.size(); ++i) ptrs[i] = c->d_frames.as<uint8_t>() + i * fpad;
    CU(cudaMemcpyAsync(c->d_ptrs.p, ptrs.data(), ptrs.size() * sizeof(void*), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));   // ptrs is a stack-lifetime staging vector
    c->ptrs_for = c->d_frames.p; c->ptrs_tab = c->d_ptrs.p; c->ptrs_n = (long long)ptrs.size(); c->ptrs_pad = fpad;
  }
  // the copy stream must not start before work already queued on the main stream (e.g. the car upload,
  // or a previous call's D2H that still reads the canvases) has been ordered
  CU(cudaEventRecord(c->ev_free[0], c->stream));
  CU(cudaEventRecord(c->ev_free[1], c->stream));
  int half = 0;
  // Page-locked host frames whose rows are 16-byte friendly are ingested by k_fetch_spans (the SMs read
  // only the sampled row spans over PCIe); anything else goes through DMA copies (at the bench workload, 1x B200:
  // 4.295 ms per 32 frame-sets zero-copy vs 6.245 ms with DMA bands for every camera, profiles/r01_e2e_probe.txt).
  bool zero_copy = !(flags & BEVK_FLAG_BALANCE) && (row % 16 == 0) && (src_stride % 16 == 0);
  std::vector<const uint8_t*> dev_view((size_t)batch * c->n_cam, nullptr);
  if (zero_copy) {
    for (size_t i = 0; i < dev_view.size() && zero_copy; ++i) {
      cudaPointerAttributes at{};
      if (!srcs[i] || cudaPointerGetAttributes(&at, srcs[i]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer ||
          (reinterpret_cast<uintptr_t>(at.devicePointer) & 15)) {
        zero_copy = false;
        cudaGetLastError();   // a pageable pointer makes cudaPointerGetAttributes fail on old drivers: not an error here
      } else {
        dev_view[i] = static_cast<const uint8_t*>(at.devicePointer);
      }
    }
  }
  if (zero_copy) {
    RET(c->d_hptrs.ensure(sizeof(void*) * set_frames * chunk * 2));
    if (!c->h_hptrs) CU(cudaHostAlloc(reinterpret_cast<void**>(&c->h_hptrs), sizeof(void*) * BEVK_MAX_CAMERAS * kHostChunk * 2, cudaHostAllocDefault));
  }
  c->last_h2d_bytes = 0;
  for (int b0 = 0; b0 < batch; b0 += chunk, half ^= 1) {
    const int nb = std::min(chunk, batch - b0);
    uint8_t* dframes = c->d_frames.as<uint8_t>() + (size_t)half * chunk * set_frames * fpad;
    std::unique_ptr<NvtxRange> nvtx_ingest(new NvtxRange("bevk ingest (H2D / zero-copy spans)"));
    CU(cudaStreamWaitEvent(c->copy_stream, c->ev_free[half], 0));   // this half's previous chunk has been rendered
    if (zero_copy) {
      const uint8_t** hp = c->h_hptrs + (size_t)half * chunk * set_frames;
      // the pinned pointer staging area of this half was consumed by the copy two chunks ago (ordered by ev_free + stream order)
      CU(cudaEventSynchronize(c->ev_hp[half]));
      for (int i = 0; i < nb * c->n_cam; ++i) hp[i] = dev_view[(size_t)b0 * c->n_cam + i];
      const uint8_t** dhp = c->d_hptrs.as<const uint8_t*>() + (size_t)half * chunk * set_frames;
      CU(cudaMemcpyAsync(dhp, hp, sizeof(void*) * nb * c->n_cam, cudaMemcpyHostToDevice, c->copy_stream));
      CU(cudaEventRecord(c->ev_hp[half], c->copy_stream));
      k_fetch_spans<<<dim3(c->FH, nb * c->n_cam), 128, 0, c->copy_stream>>>(
          dhp, c->d_ptrs.as<uint8_t*>() + (size_t)half * chunk * set_frames, c->d_spans.as<int2>(), c->n_cam, c->FH,
          (long long)src_stride, (int)row);
      LAUNCHED(c);
      c->last_h2d_bytes += (long long)c->span_fetch_bytes * nb;
    }
    for (int i = 0; i < nb * c->n_cam && !zero_copy; ++i) {
      const uint8_t* s = srcs[(size_t)b0 * c->n_cam + i];
      if (!s) return fail(BEVK_ERR_ARG, "null frame pointer %d", b0 * c->n_cam + i);
      uint8_t* d = dframes + (size_t)i * fpad;
      if (flags & BEVK_FLAG_BALANCE) {   // luminance_balance averages V over the whole raw frame: everything goes up
        if ((size_t)src_stride == row) CU(cudaMemcpyAsync(d, s, fbytes, cudaMemcpyHostToDevice, c->copy_stream));
        else CU(cudaMemcpy2DAsync(d, row, s, (size_t)src_stride, row, c->FH, cudaMemcpyHostToDevice, c->copy_stream));
        c->last_h2d_bytes += (long long)fbytes;
      } else {                           // only the rectangle of the frame this camera's LUT can sample
        for (int bnd = 0; bnd < DMA_BANDS; ++bnd) {
          const int* bx = c->cam_box[i % c->n_cam][bnd];
          if (bx[1] > bx[0]) {
            CU(cudaMemcpy2DAsync(d + (size_t)bx[0] * row + bx[2], row, s + (size_t)bx[0] * src_stride + bx[2],
                                 (size_t)src_stride, (size_t)(bx[3] - bx[2]), (size_t)(bx[1] - bx[0]), cudaMemcpyHostToDevice,
                                 c->copy_stream));
            c->last_h2d_bytes += (long long)(bx[3] - bx[2]) * (bx[1] - bx[0]);
          }
        }
      }
    }
    CU(cudaEventRecord(c->ev_in[half], c->copy_stream));
    nvtx_ingest.reset();
    CU(cudaStreamWaitEvent(c->stream, c->ev_in[half], 0));
    c->timed = false;
    uint8_t* dcanvas = c->d_canvas.as<uint8_t>() + (size_t)half * chunk * cbytes;
    const void* dptrs = c->d_ptrs.as<const uint8_t*>() + (size_t)half * chunk * set_frames;
    FrameSrc fsrc = stack_src(dframes, (long long)fpad);   // the staging buffers are a frame stack: TMA-staged kernel
    fsrc.table = dptrs;
    RET(run_device(c, fsrc, nb, car ? c->d_car.p : nullptr, flags, dcanvas, 0, BEVK_MAX_CAMERAS));
    CU(cudaEventRecord(c->ev_free[half], c->stream));               // frames of this half are free again
    {
      NvtxRange nvtx_d2h("bevk read-back (D2H canvases)");
      CU(cudaMemcpyAsync(out + (size_t)b0 * cbytes, dcanvas, cbytes * nb, cudaMemcpyDeviceToHost, c->stream));
    }
  }
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

// ------------------------------------------------------------------ stand-alone helpers
static int ensure_hsv(bevk_ctx* c) {
  if (c->d_hsv.p) return BEVK_OK;
  std::vector<int> tab(512, 0);
  for (int i = 1; i < 256; ++i) {
    tab[i] = (int)std::nearbyint((255 << 12) / (1. * i));
    tab[256 + i] = (int)std::nearbyint((180 << 12) / (6. * i));
  }
  RET(c->d_hsv.ensure(512 * sizeof(int)));
  CU(cudaMemcpyAsync(c->d_hsv.p, tab.data(), 512 * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

static int stream_blocks(long long n_items) {
  return (int)std::max<long long>(1, std::min<long long>(148 * 8, (n_items + 255) / 256));
}

int bevk_apply_mask(bevk_ctx* c, const uint8_t* img, const uint8_t* mask, int w, int h, int blend, uint8_t* out) {
  RET(use(c));
  if (!img || !mask || !out || w <= 0 || h <= 0) return fail(BEVK_ERR_ARG, "bad argument");
  const size_t npx = (size_t)w * h;
  RET(c->s_src.ensure(npx * 3));
  RET(c->s_m1.ensure(npx));
  RET(c->s_dst.ensure(npx * 3));
  CU(cudaMemcpyAsync(c->s_src.p, img, npx * 3, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->s_m1.p, mask, npx, cudaMemcpyHostToDevice, c->stream));
  k_apply_mask<<<stream_blocks(npx), 256, 0, c->stream>>>(c->s_src.as<uint8_t>(), c->s_m1.as<uint8_t>(),
                                                          c->s_dst.as<uint8_t>(), (long long)npx, blend);
  LAUNCHED(c);
  CU(cudaMemcpyAsync(out, c->s_dst.p, npx * 3, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_color_balance(bevk_ctx* c, const uint8_t* img, int w, int h, uint8_t* out) {
  RET(use(c));
  if (!img || !out || w <= 0 || h <= 0) return fail(BEVK_ERR_ARG, "bad argument");
  const size_t npx = (size_t)w * h;
  RET(c->s_dst.ensure(npx * 3));
  RET(c->d_csum.ensure(24));
  CU(cudaMemcpyAsync(c->s_dst.p, img, npx * 3, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(c->d_csum.p, 0, 24, c->stream));
  k_chan_sum<<<stream_blocks(npx), 256, 0, c->stream>>>(c->s_dst.as<uint8_t>(), (long long)npx,
                                                        c->d_csum.as<unsigned long long>());
  LAUNCHED(c);
  k_gain<<<dim3(stream_blocks(npx / 4 + 1), 1), 256, 0, c->stream>>>(c->s_dst.as<uint8_t>(), (long long)npx * 3, (double)npx,
                                                                   c->d_csum.as<unsigned long long>(), nullptr);
  LAUNCHED(c);
  CU(cudaMemcpyAsync(out, c->s_dst.p, npx * 3, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

int bevk_luminance_balance(bevk_ctx* c, const uint8_t* const* imgs, int n, int w, int h, uint8_t* const* outs) {
  RET(use(c));
  if (!imgs || !outs || n < 1 || n > BEVK_MAX_CAMERAS || w <= 0 || h <= 0) return fail(BEVK_ERR_ARG, "bad argument");
  RET(ensure_hsv(c));
  const size_t fbytes = (size_t)w * h * 3, fpad = (fbytes + 255) & ~size_t(255);
  RET(c->s_src.ensure(fpad * n));
  RET(c->s_dst.ensure(fpad * n));
  RET(c->d_ptrs.ensure(sizeof(void*) * 2 * BEVK_MAX_CAMERAS));
  c->ptrs_for = nullptr;   // the BEV host path's cached pointer table is overwritten below
  RET(c->d_vsum.ensure(8 * n));
  RET(c->d_delta.ensure(4 * n));
  const uint8_t* ptrs[2 * BEVK_MAX_CAMERAS];
  for (int i = 0; i < n; ++i) {
    if (!imgs[i] || !outs[i]) return fail(BEVK_ERR_ARG, "null frame %d", i);
    ptrs[i] = c->s_src.as<uint8_t>() + i * fpad;
    ptrs[BEVK_MAX_CAMERAS + i] = c->s_dst.as<uint8_t>() + i * fpad;
    CU(cudaMemcpyAsync(const_cast<uint8_t*>(ptrs[i]), imgs[i], fbytes, cudaMemcpyHostToDevice, c->stream));
  }
  CU(cudaMemcpyAsync(c->d_ptrs.p, ptrs, sizeof ptrs, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(c->d_vsum.p, 0, 8 * n, c->stream));
  const uint8_t* const* d_in = c->d_ptrs.as<const uint8_t*>();
  uint8_t* const* d_out = reinterpret_cast<uint8_t* const*>(c->d_ptrs.as<uint8_t*>() + BEVK_MAX_CAMERAS);
  k_vsum<<<dim3(stream_blocks(fbytes / 48 + 1) / n + 1, n), 256, 0, c->stream>>>(d_in, (long long)fbytes,
                                                                                 c->d_vsum.as<unsigned long long>());
  LAUNCHED(c);
  k_delta<<<1, 32, 0, c->stream>>>(c->d_vsum.as<unsigned long long>(), n, 1, (double)w * (double)h, c->d_delta.as<int>());
  LAUNCHED(c);
  k_lum_apply<<<dim3(stream_blocks((long long)w * h) / n + 1, n), 256, 0, c->stream>>>(d_in, d_out, w, h, c->d_delta.as<int>(),
                                                                                       c->d_hsv.as<int>());
  LAUNCHED(c);
  for (int i = 0; i < n; ++i)
    CU(cudaMemcpyAsync(outs[i], ptrs[BEVK_MAX_CAMERAS + i], fbytes, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));   // also keeps the stack-resident ptrs[] alive long enough
  return BEVK_OK;
}

// ------------------------------------------------------------------ multi-GPU sharding (one process per GPU)
// NCCL is loaded at run time (dlopen): libbevk.so has no link-time dependency on it, and a process that already holds
// a libnccl.so.2 (torch's) shares it.
namespace {
struct NcclId { char b[128]; };   // ncclUniqueId (passed by value to ncclCommInitRank)
struct Nccl {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
Nccl& nccl() {
  static Nccl n;
  static bool tried = false;
  if (!tried) {
    tried = true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      n.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (n.lib) break;
    }
    if (n.lib) {
      n.GetUniqueId = reinterpret_cast<decltype(n.GetUniqueId)>(dlsym(n.lib, "ncclGetUniqueId"));
      n.CommInitRank = reinterpret_cast<decltype(n.CommInitRank)>(dlsym(n.lib, "ncclCommInitRank"));
      n.CommDestroy = reinterpret_cast<decltype(n.CommDestroy)>(dlsym(n.lib, "ncclCommDestroy"));
      n.AllGather = reinterpret_cast<decltype(n.AllGather)>(dlsym(n.lib, "ncclAllGather"));
      n.GetErrorString = reinterpret_cast<decltype(n.GetErrorString)>(dlsym(n.lib, "ncclGetErrorString"));
      n.ok = n.GetUniqueId && n.CommInitRank && n.CommDestroy && n.AllGather && n.GetErrorString;
    }
  }
  return n;
}
const int kNcclUint8 = 1;   // ncclUint8 (nccl.h: ncclInt8 = 0, ncclUint8 = 1)
}  // namespace

static void shard_peers_release(bevk_ctx* c) {
  bevk_ctx::Shard& s = c->shard;
  for (int r = 0; r < SHARD_MAX_RANKS; ++r) {
    if (s.peer_recv[r] && s.peer_recv[r] != s.recv) cudaIpcCloseMemHandle(s.peer_recv[r]);
    s.peer_recv[r] = nullptr;
  }
  s.attached = false;
}

static void shard_release(bevk_ctx* c) {
  shard_peers_release(c);
  if (c->shard.recv) cudaFree(c->shard.recv);
  c->shard.recv = nullptr; c->shard.recv_bytes = 0; c->shard.prepared_batch = 0;
  c->shard.d_flag.release();
  if (c->shard.comm && nccl().ok) nccl().CommDestroy(c->shard.comm);
  c->shard.comm = nullptr;
  c->shard.d_slabs.release();
}

int bevk_shard_configure(bevk_ctx* c, int policy, int rank, int world) {
  RET(use(c));
  if (policy != BEVK_SHARD_FRAMES && policy != BEVK_SHARD_CAMERAS) return fail(BEVK_ERR_ARG, "bad policy %d", policy);
  if (world < 1 || rank < 0 || rank >= world) return fail(BEVK_ERR_ARG, "rank %d outside world %d", rank, world);
  if (policy == BEVK_SHARD_CAMERAS && world > SHARD_MAX_RANKS)
    return fail(BEVK_ERR_UNSUPPORTED, "camera sharding supports up to %d ranks (there are at most %d cameras)", SHARD_MAX_RANKS, BEVK_MAX_CAMERAS);
  if (c->shard.comm && (c->shard.rank != rank || c->shard.world != world)) shard_release(c);
  c->shard.configured = true; c->shard.geometry = false;
  c->shard.policy = policy; c->shard.rank = rank; c->shard.world = world;
  return BEVK_OK;
}

static int shard_geometry(bevk_ctx* c) {
  bevk_ctx::Shard& s = c->shard;
  if (!s.configured) return fail(BEVK_ERR_ARG, "bevk_shard_configure not called");
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if (s.geometry) return BEVK_OK;
  std::vector<const uint8_t*> pm(c->n_cam);
  for (int k = 0; k < c->n_cam; ++k) pm[k] = c->cam[k].mask.data();
  s.slab_bytes = 0;
  for (int r = 0; r < s.world && r < SHARD_MAX_RANKS; ++r) {
    shard_block(c->n_cam, r, s.world, &s.cam_lo[r], &s.cam_hi[r]);
    s.rect[r] = slab_rect(pm.data(), s.cam_lo[r], s.cam_hi[r], c->BW, c->BH);
    const long long bytes = (long long)(s.rect[r].ox1 - s.rect[r].ox) * (s.rect[r].oy1 - s.rect[r].oy) * 3;
    s.slab_bytes = std::max(s.slab_bytes, bytes);
  }
  s.slab_bytes = (s.slab_bytes + 255) & ~255ll;   // equal counts for the all-gather, 256-byte aligned slabs
  s.geometry = true;
  return BEVK_OK;
}

int bevk_shard_unique_id(void* id, int len) {
  if (!id || len < 128) return fail(BEVK_ERR_ARG, "id buffer must hold 128 bytes");
  if (!nccl().ok) return fail(BEVK_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror() ? dlerror() : "missing symbols");
  NcclId u;
  const int r = nccl().GetUniqueId(&u);
  if (r != 0) return fail(BEVK_ERR_CUDA, "ncclGetUniqueId: %s", nccl().GetErrorString(r));
  memcpy(id, &u, 128);
  return BEVK_OK;
}

int bevk_shard_connect(bevk_ctx* c, const void* id, int len) {
  RET(use(c));
  if (!c->shard.configured) return fail(BEVK_ERR_ARG, "bevk_shard_configure not called");
  if (!id || len < 128) return fail(BEVK_ERR_ARG, "id must be the 128 bytes bevk_shard_unique_id produced on one rank");
  if (!nccl().ok) return fail(BEVK_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) could not be loaded");
  if (c->shard.comm) { nccl().CommDestroy(c->shard.comm); c->shard.comm = nullptr; }
  NcclId u;
  memcpy(&u, id, 128);
  const int r = nccl().CommInitRank(&c->shard.comm, c->shard.world, u, c->shard.rank);
  if (r != 0) { c->shard.comm = nullptr; return fail(BEVK_ERR_CUDA, "ncclCommInitRank(rank %d of %d): %s", c->shard.rank, c->shard.world, nccl().GetErrorString(r)); }
  return BEVK_OK;
}

int bevk_shard_info(bevk_ctx* c, int rank, int* cam_lo, int* cam_hi, int32_t rect[4], int64_t* slab_bytes) {
  RET(use(c));
  RET(shard_geometry(c));
  if (rank < 0 || rank >= c->shard.world || rank >= SHARD_MAX_RANKS) return fail(BEVK_ERR_ARG, "rank %d out of range", rank);
  if (cam_lo) *cam_lo = c->shard.cam_lo[rank];
  if (cam_hi) *cam_hi = c->shard.cam_hi[rank];
  if (rect) { rect[0] = c->shard.rect[rank].ox; rect[1] = c->shard.rect[rank].oy; rect[2] = c->shard.rect[rank].ox1; rect[3] = c->shard.rect[rank].oy1; }
  if (slab_bytes) *slab_bytes = c->shard.slab_bytes;
  return BEVK_OK;
}

// rank `as_rank`'s slabs of `batch` frame-sets into d_slabs[as_rank][batch][slab_bytes]
static int shard_render(bevk_ctx* c, FrameSrc src, int batch, int as_rank, void* d_slabs) {
  bevk_ctx::Shard& s = c->shard;
  const SlabRect q = s.rect[as_rank];
  uint8_t* dst = reinterpret_cast<uint8_t*>(d_slabs) + (size_t)as_rank * batch * s.slab_bytes;
  if (q.ox1 <= q.ox || s.cam_hi[as_rank] <= s.cam_lo[as_rank]) return BEVK_OK;   // a rank without cameras contributes nothing
  OutWin w;
  w.pitch = (q.ox1 - q.ox) * 3; w.ox = q.ox; w.oy = q.oy; w.ox1 = q.ox1; w.oy1 = q.oy1; w.stride = s.slab_bytes;
  return run_device(c, src, batch, nullptr, 0, dst, s.cam_lo[as_rank], s.cam_hi[as_rank], &w);
}

static int shard_compose(bevk_ctx* c, const void* d_slabs, int batch, const void* d_car, void* d_out, long long rank_stride = 0) {
  bevk_ctx::Shard& s = c->shard;
  ComposeArgs a{};
  a.slabs = reinterpret_cast<const uint8_t*>(d_slabs); a.slab_bytes = s.slab_bytes; a.world = std::min(s.world, SHARD_MAX_RANKS);
  a.rank_stride = rank_stride ? rank_stride : (long long)batch * s.slab_bytes;
  a.batch = batch; a.BW = c->BW; a.BH = c->BH;
  for (int r = 0; r < a.world; ++r) a.rect[r] = s.rect[r];
  a.car = reinterpret_cast<const uint8_t*>(d_car); a.out = reinterpret_cast<uint8_t*>(d_out);
  const bool wide = (c->BW % 8) == 0 && (reinterpret_cast<uintptr_t>(d_out) & 7) == 0 && (!d_car || (reinterpret_cast<uintptr_t>(d_car) & 7) == 0) &&
                    (reinterpret_cast<uintptr_t>(d_slabs) & 7) == 0 && (s.slab_bytes & 7) == 0 && (a.rank_stride & 7) == 0;
  if (batch > 65535 || c->BH > 65535 * COMPOSE_ROWS) return fail(BEVK_ERR_UNSUPPORTED, "compose grid too large");
  const int units = wide ? c->BW * 3 / 8 : c->BW * 3;
  const dim3 grid((units + 255) / 256, (c->BH + COMPOSE_ROWS - 1) / COMPOSE_ROWS, batch);
  if (wide) k_compose_slabs<8><<<grid, 256, 0, c->stream>>>(a);
  else k_compose_slabs<1><<<grid, 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  return BEVK_OK;
}

int bevk_shard_render(bevk_ctx* c, const void* d_frames, int64_t frame_stride, int batch, int as_rank, void* d_slabs) {
  RET(use(c));
  RET(shard_geometry(c));
  RET(check_stack(c, d_frames, frame_stride));
  if (as_rank < 0 || as_rank >= c->shard.world || as_rank >= SHARD_MAX_RANKS) return fail(BEVK_ERR_ARG, "rank %d out of range", as_rank);
  if (!d_slabs || (reinterpret_cast<uintptr_t>(d_slabs) & 15)) return fail(BEVK_ERR_ARG, "slab buffer null or not 16-byte aligned");
  c->timed = true;
  return shard_render(c, stack_src(d_frames, frame_stride), batch, as_rank, d_slabs);
}

int bevk_shard_compose(bevk_ctx* c, const void* d_slabs, int batch, const void* d_car, void* d_out) {
  RET(use(c));
  RET(shard_geometry(c));
  if (!d_slabs || !d_out || batch < 1) return fail(BEVK_ERR_ARG, "bad argument");
  return shard_compose(c, d_slabs, batch, d_car, d_out);
}

int bevk_bev_run_sharded(bevk_ctx* c, const void* d_frames, int64_t frame_stride, int batch, const void* d_car, int flags, void* d_out) {
  NvtxRange nvtx_call("bevk_bev_run_sharded (render slabs, all-gather, compose)");
  RET(use(c));
  if (!c->shard.configured) return fail(BEVK_ERR_ARG, "bevk_shard_configure not called");
  RET(check_stack(c, d_frames, frame_stride));
  bevk_ctx::Shard& s = c->shard;
  s.last_link_bytes = 0;
  if (s.policy == BEVK_SHARD_FRAMES || s.world == 1) {   // every rank renders its own frame-sets: no exchange
    c->timed = true;
    return run_device(c, stack_src(d_frames, frame_stride), batch, d_car, flags, d_out, 0, BEVK_MAX_CAMERAS);
  }
  if (flags & BEVK_FLAG_BALANCE) return fail(BEVK_ERR_UNSUPPORTED, "balance needs every camera's V mean before the warp: not available with camera sharding");
  if (!s.comm) return fail(BEVK_ERR_ARG, "bevk_shard_connect not called");
  RET(shard_geometry(c));
  const size_t per_rank = (size_t)batch * s.slab_bytes;
  RET(s.d_slabs.ensure(per_rank * s.world));
  c->timed = false;
  RET(shard_render(c, stack_src(d_frames, frame_stride), batch, s.rank, s.d_slabs.p));
  // ONE all-gather of the slabs (in place: this rank's block is already where it belongs)
  const int r = nccl().AllGather(s.d_slabs.as<uint8_t>() + per_rank * s.rank, s.d_slabs.p, per_rank, kNcclUint8, s.comm, c->stream);
  if (r != 0) return fail(BEVK_ERR_CUDA, "ncclAllGather: %s", nccl().GetErrorString(r));
  s.last_link_bytes = (long long)per_rank * (s.world - 1);
  return shard_compose(c, s.d_slabs.p, batch, d_car, d_out);
}

// ---- camera sharding with peer stores: compute and exchange in one kernel ----------------------------------------
// Frame-set b of the batch is OWNED by rank b % world, which ends up with its canvas.  Every rank renders its cameras'
// slabs of ALL frame-sets, and the fused kernel's write-out stores each slab straight into the owner's receive buffer
// over NVLink (CUDA IPC mapping) -- no send buffer, no separate collective; one 4-byte all-gather per step is the
// barrier that tells an owner its slabs have landed, then it composes its own canvases.  Each rank sends and receives
// (world-1)/world of ONE slab set instead of receiving world-1 whole ones as the all-gather form does.
static int own_count(int batch, int rank, int world) { return (batch - rank + world - 1) / world; }

int bevk_shard_prepare(bevk_ctx* c, int batch, void* handle64) {
  RET(use(c));
  RET(shard_geometry(c));
  bevk_ctx::Shard& s = c->shard;
  if (s.policy != BEVK_SHARD_CAMERAS) return fail(BEVK_ERR_ARG, "peer stores belong to the CAMERAS policy");
  if (batch < 1 || !handle64) return fail(BEVK_ERR_ARG, "bad argument");
  CU(cudaStreamSynchronize(c->stream));
  shard_peers_release(c);
  s.own_max = (batch + s.world - 1) / s.world;
  const size_t need = 2 * (size_t)s.world * s.own_max * s.slab_bytes;
  if (need > s.recv_bytes) {   // plain cudaMalloc: IPC handles cannot be taken from pool / async allocations
    if (s.recv) cudaFree(s.recv);
    s.recv = nullptr; s.recv_bytes = 0;
    CU(cudaMalloc(&s.recv, need));
    s.recv_bytes = need;
  }
  CU(cudaMemsetAsync(s.recv, 0, s.recv_bytes, c->stream));   // slabs of ranks without cameras are never written: keep them zero
  CU(cudaStreamSynchronize(c->stream));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, s.recv));
  static_assert(sizeof h == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  s.prepared_batch = batch;
  RET(s.d_flag.ensure(sizeof(int) * (SHARD_MAX_RANKS + 1)));
  return BEVK_OK;
}

int bevk_shard_attach(bevk_ctx* c, const void* handles) {
  RET(use(c));
  bevk_ctx::Shard& s = c->shard;
  if (!s.prepared_batch || !handles) return fail(BEVK_ERR_ARG, "bevk_shard_prepare not called");
  shard_peers_release(c);
  for (int r = 0; r < s.world && r < SHARD_MAX_RANKS; ++r) {
    if (r == s.rank) { s.peer_recv[r] = s.recv; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, reinterpret_cast<const uint8_t*>(handles) + 64 * r, 64);
    const cudaError_t e = cudaIpcOpenMemHandle(&s.peer_recv[r], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { s.peer_recv[r] = nullptr; shard_peers_release(c); return fail(BEVK_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e)); }
  }
  s.attached = true;
  return BEVK_OK;
}

int bevk_bev_run_scattered(bevk_ctx* c, const void* d_frames, int64_t frame_stride, int batch, const void* d_car, int flags,
                           void* d_out_own, int* n_own) {
  NvtxRange nvtx_call("bevk_bev_run_scattered (render with peer stores, barrier, compose own)");
  RET(use(c));
  bevk_ctx::Shard& s = c->shard;
  if (!s.configured || s.policy != BEVK_SHARD_CAMERAS) return fail(BEVK_ERR_ARG, "bevk_shard_configure(CAMERAS) not called");
  RET(check_stack(c, d_frames, frame_stride));
  if (flags & BEVK_FLAG_BALANCE) return fail(BEVK_ERR_UNSUPPORTED, "balance is not available with camera sharding");
  RET(shard_geometry(c));
  if (!s.comm && s.world > 1) return fail(BEVK_ERR_ARG, "bevk_shard_connect not called");
  if (!s.attached || batch > s.prepared_batch || (batch + s.world - 1) / s.world != s.own_max)
    return fail(BEVK_ERR_ARG, "bevk_shard_prepare / bevk_shard_attach not called for a batch of %d", batch);
  const int mine = own_count(batch, s.rank, s.world);
  if (n_own) *n_own = mine;
  if (mine > 0 && !d_out_own) return fail(BEVK_ERR_ARG, "null output");
  const size_t half = (size_t)s.world * s.own_max * s.slab_bytes, rank_stride = (size_t)s.own_max * s.slab_bytes;
  const unsigned par = s.step++ & 1u;     // double buffer: a peer may already store step n+1 while this rank composes step n
  const SlabRect q = s.rect[s.rank];
  s.last_link_bytes = 0;
  if (q.ox1 > q.ox && s.cam_hi[s.rank] > s.cam_lo[s.rank]) {
    OutWin w;
    w.pitch = (q.ox1 - q.ox) * 3; w.ox = q.ox; w.oy = q.oy; w.ox1 = q.ox1; w.oy1 = q.oy1; w.stride = s.slab_bytes;
    w.world = s.world; w.src_off = (long long)(par * half + (size_t)s.rank * rank_stride);
    for (int r = 0; r < s.world; ++r) w.peer[r] = reinterpret_cast<uint8_t*>(s.peer_recv[r]);
    c->timed = false;
    RET(run_device(c, stack_src(d_frames, frame_stride), batch, nullptr, 0, nullptr, s.cam_lo[s.rank], s.cam_hi[s.rank], &w));
    s.last_link_bytes = (long long)(batch - mine) * s.slab_bytes;   // what this rank stored into its peers
  }
  if (s.world > 1) {   // the step barrier: every rank's stores are complete (its kernel has finished) when this returns on the stream
    int* f = s.d_flag.as<int>();
    const int r = nccl().AllGather(f + SHARD_MAX_RANKS, f, 4, kNcclUint8, s.comm, c->stream);
    if (r != 0) return fail(BEVK_ERR_CUDA, "ncclAllGather (step barrier): %s", nccl().GetErrorString(r));
  }
  if (mine > 0) RET(shard_compose(c, reinterpret_cast<const uint8_t*>(s.recv) + par * half, mine, d_car, d_out_own, (long long)rank_stride));
  return BEVK_OK;
}

int64_t bevk_shard_last_link_bytes(bevk_ctx* c) { return c ? c->shard.last_link_bytes : 0; }

// ------------------------------------------------------------------ JPEG ingest on the device (nvJPEG, dlopen'ed)
// The reference reads its frames with cv2.imread (SurroundBirdEyeView/surroundBEV.py:328-332, Tools/undistort.py:65):
// decode on the host, then -- here -- 3 bytes per pixel over PCIe.  bevk_jpeg_decode ships the compressed stream
// instead and decodes it straight into the frame stack the BEV / undistort entry points read.
namespace {
struct NvjpegImage { unsigned char* channel[4]; size_t pitch[4]; };
struct Nvjpeg {
  void* lib = nullptr;
  int (*CreateSimple)(void**) = nullptr;
  int (*Destroy)(void*) = nullptr;
  int (*StateCreate)(void*, void**) = nullptr;
  int (*StateDestroy)(void*) = nullptr;
  int (*GetImageInfo)(void*, const unsigned char*, size_t, int*, int*, int*, int*) = nullptr;
  int (*Decode)(void*, void*, const unsigned char*, size_t, int, NvjpegImage*, cudaStream_t) = nullptr;
  bool ok = false;
};
Nvjpeg& nvjpeg() {
  static Nvjpeg n;
  static bool tried = false;
  if (!tried) {
    tried = true;
    for (const char* name : {"libnvjpeg.so.12", "libnvjpeg.so", "/usr/local/cuda/lib64/libnvjpeg.so.12"}) {
      n.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (n.lib) break;
    }
    if (n.lib) {
      n.CreateSimple = reinterpret_cast<decltype(n.CreateSimple)>(dlsym(n.lib, "nvjpegCreateSimple"));
      n.Destroy = reinterpret_cast<decltype(n.Destroy)>(dlsym(n.lib, "nvjpegDestroy"));
      n.StateCreate = reinterpret_cast<decltype(n.StateCreate)>(dlsym(n.lib, "nvjpegJpegStateCreate"));
      n.StateDestroy = reinterpret_cast<decltype(n.StateDestroy)>(dlsym(n.lib, "nvjpegJpegStateDestroy"));
      n.GetImageInfo = reinterpret_cast<decltype(n.GetImageInfo)>(dlsym(n.lib, "nvjpegGetImageInfo"));
      n.Decode = reinterpret_cast<decltype(n.Decode)>(dlsym(n.lib, "nvjpegDecode"));
      n.ok = n.CreateSimple && n.Destroy && n.StateCreate && n.StateDestroy && n.GetImageInfo && n.Decode;
    }
  }
  return n;
}
const int kNvjpegOutputBGRI = 6;   // NVJPEG_OUTPUT_BGRI: interleaved BGR in channel[0], what cv2.imread's layout is
}  // namespace

static void jpeg_release(bevk_ctx* c) {
  if (c->jpeg_state && nvjpeg().ok) nvjpeg().StateDestroy(c->jpeg_state);
  if (c->jpeg_handle && nvjpeg().ok) nvjpeg().Destroy(c->jpeg_handle);
  c->jpeg_state = c->jpeg_handle = nullptr;
}

int bevk_jpeg_decode(bevk_ctx* c, const uint8_t* const* jpegs, const uint64_t* sizes, int n, int width, int height, void* d_frames,
                     int64_t frame_stride) {
  NvtxRange nvtx_call("bevk_jpeg_decode (nvJPEG -> frame stack)");
  RET(use(c));
  if (!jpegs || !sizes || !d_frames || n < 1) return fail(BEVK_ERR_ARG, "bad argument");
  if (width <= 0 || height <= 0 || frame_stride < (int64_t)width * height * 3) return fail(BEVK_ERR_ARG, "bad frame geometry / stride");
  if (!nvjpeg().ok) return fail(BEVK_ERR_UNSUPPORTED, "nvJPEG (libnvjpeg.so.12) could not be loaded");
  if (!c->jpeg_handle) {
    int r = nvjpeg().CreateSimple(&c->jpeg_handle);
    if (r != 0) { c->jpeg_handle = nullptr; return fail(BEVK_ERR_CUDA, "nvjpegCreateSimple failed: %d", r); }
    r = nvjpeg().StateCreate(c->jpeg_handle, &c->jpeg_state);
    if (r != 0) { jpeg_release(c); return fail(BEVK_ERR_CUDA, "nvjpegJpegStateCreate failed: %d", r); }
  }
  for (int i = 0; i < n; ++i) {
    if (!jpegs[i] || !sizes[i]) return fail(BEVK_ERR_ARG, "JPEG stream %d is empty", i);
    int comps = 0, sub = 0, w[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0};
    int r = nvjpeg().GetImageInfo(c->jpeg_handle, jpegs[i], (size_t)sizes[i], &comps, &sub, w, h);
    if (r != 0) return fail(BEVK_ERR_ARG, "stream %d is not a JPEG nvJPEG can parse (status %d)", i, r);
    if (w[0] != width || h[0] != height) return fail(BEVK_ERR_ARG, "stream %d is %dx%d, the frame stack holds %dx%d", i, w[0], h[0], width, height);
    NvjpegImage dst{};
    dst.channel[0] = reinterpret_cast<unsigned char*>(d_frames) + (size_t)i * frame_stride;
    dst.pitch[0] = (size_t)width * 3;
    r = nvjpeg().Decode(c->jpeg_handle, c->jpeg_state, jpegs[i], (size_t)sizes[i], kNvjpegOutputBGRI, &dst, c->stream);
    if (r != 0) return fail(BEVK_ERR_CUDA, "nvjpegDecode(stream %d) failed: %d", i, r);
  }
  return BEVK_OK;
}

// BevGenerator.__call__ on JPEG streams: decode the batch into the library's frame stack, render, read the canvases back.
int bevk_bev_run_jpeg(bevk_ctx* c, const uint8_t* const* jpegs, const uint64_t* sizes, int batch, const uint8_t* car, int flags,
                      uint8_t* out) {
  NvtxRange nvtx_call("bevk_bev_run_jpeg (JPEG streams -> host canvases)");
  RET(use(c));
  if (!c->planned) return fail(BEVK_ERR_ARG, "bevk_bev_finalize not called");
  if (!jpegs || !sizes || !out || batch < 1) return fail(BEVK_ERR_ARG, "bad argument");
  const size_t fbytes = (size_t)c->FW * c->FH * 3, fpad = (fbytes + 255) & ~size_t(255), cbytes = (size_t)c->BW * c->BH * 3;
  const int nf = batch * c->n_cam;
  RET(c->d_jpeg_frames.ensure(fpad * nf));
  RET(c->d_jpeg_canvas.ensure(cbytes * batch));
  RET(bevk_jpeg_decode(c, jpegs, sizes, nf, c->FW, c->FH, c->d_jpeg_frames.p, (int64_t)fpad));
  if (car) {
    RET(c->d_car.ensure(cbytes));
    CU(cudaMemcpyAsync(c->d_car.p, car, cbytes, cudaMemcpyHostToDevice, c->stream));
  }
  c->timed = false;
  RET(run_device(c, stack_src(c->d_jpeg_frames.p, (long long)fpad), batch, car ? c->d_car.p : nullptr, flags, c->d_jpeg_canvas.p, 0,
                 BEVK_MAX_CAMERAS));
  CU(cudaMemcpyAsync(out, c->d_jpeg_canvas.p, cbytes * batch, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BEVK_OK;
}

// ------------------------------------------------------------------ CUDA graphs
// Stream capture of whatever the device-pointer entry points enqueue between begin and end; replayed with one call.
int bevk_graph_begin(bevk_ctx* c) {
  RET(use(c));
  if (c->capturing) return fail(BEVK_ERR_ARG, "a capture is already open on this context");
  CU(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
  c->capturing = true;
  c->capture_launches0 = c->launches;
  return BEVK_OK;
}

int bevk_graph_end(bevk_ctx* c, int* graph_id) {
  RET(use(c));
  if (!c->capturing) return fail(BEVK_ERR_ARG, "bevk_graph_begin was not called");
  c->capturing = false;
  bevk_ctx::Graph g;
  cudaError_t e = cudaStreamEndCapture(c->stream, &g.g);
  if (e != cudaSuccess || !g.g) {
    cudaGetLastError();
    return fail(BEVK_ERR_CUDA, "stream capture failed (%s): a call inside the capture allocated or synchronised -- run the same "
                               "calls once before capturing so that every buffer and table exists", cudaGetErrorString(e));
  }
  e = cudaGraphInstantiate(&g.x, g.g, 0);
  if (e != cudaSuccess) { cudaGraphDestroy(g.g); return fail(BEVK_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
  g.kernels = c->launches - c->capture_launches0;
  c->launches = c->capture_launches0;            // nothing ran yet: replays are counted by bevk_graph_launch
  size_t slot = 0;
  while (slot < c->graphs.size() && c->graphs[slot].x) ++slot;
  if (slot == c->graphs.size()) c->graphs.push_back(g); else c->graphs[slot] = g;
  if (graph_id) *graph_id = (int)slot;
  return BEVK_OK;
}

int bevk_graph_launch(bevk_ctx* c, int graph_id, int times) {
  RET(use(c));
  if (graph_id < 0 || (size_t)graph_id >= c->graphs.size() || !c->graphs[graph_id].x) return fail(BEVK_ERR_ARG, "no graph %d", graph_id);
  if (times < 1) return fail(BEVK_ERR_ARG, "times must be >= 1");
  if (c->capturing) return fail(BEVK_ERR_ARG, "cannot launch a graph inside a capture");
  for (int i = 0; i < times; ++i) CU(cudaGraphLaunch(c->graphs[graph_id].x, c->stream));
  c->launches += (long long)times * c->graphs[graph_id].kernels;
  return BEVK_OK;
}

int bevk_graph_destroy(bevk_ctx* c, int graph_id) {
  RET(use(c));
  if (graph_id < 0 || (size_t)graph_id >= c->graphs.size() || !c->graphs[graph_id].x) return fail(BEVK_ERR_ARG, "no graph %d", graph_id);
  CU(cudaStreamSynchronize(c->stream));
  cudaGraphExecDestroy(c->graphs[graph_id].x);
  cudaGraphDestroy(c->graphs[graph_id].g);
  c->graphs[graph_id] = bevk_ctx::Graph();
  return BEVK_OK;
}

int64_t bevk_launch_count(bevk_ctx* c) { return c ? c->launches : 0; }

int bevk_last_kernel_ms(bevk_ctx* c, float* ms) {
  RET(use(c));
  if (!ms) return fail(BEVK_ERR_ARG, "null ms");
  if (!c->timed) return fail(BEVK_ERR_ARG, "no timed bevk_bev_run_device call yet");
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaEventElapsedTime(ms, c->ev0, c->ev1));
  return BEVK_OK;
}

