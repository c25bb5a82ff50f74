// extract.cu -- B200 (sm_100a) ORB extractor: pyramid + border + Gaussian blur as a register-resident column walk
// (pyr_walk.cuh), FAST with one warp per run of tiles (fast_tile.cuh: tensor-map TMA windows, packed quick reject,
// 16x2-SIMD score, tile retry + non-max suppression), block-parallel quadtree, orientation + rBRIEF, and the C ABI of
// the extractor (include/swm_orb.h).  Batched over frames: every launch covers all frames of a batch, nothing
// returns to the host between stages.
//
// Reference behaviour restated (paths relative to /root/reference/code/):
//   ORBextractor::operator()            src/ORBextractor.cc:746-819
//   ORBextractor::ComputePyramid        src/ORBextractor.cc:821-855   (cv::resize INTER_LINEAR 8U semantics)
//   ComputeKeyPointsOctTree             src/ORBextractor.cc:691-744
//   tileCalcKeypoints_kernel            src/cuda/Fast_gpu.cu:284-341  (lock-step deterministic form, fast_tile.cuh)
//   DistributeOctTree                   src/ORBextractor.cc:465-689   (octree_core.cuh)
//   IC_Angle_kernel / addBorder_kernel  src/cuda/Fast_gpu.cu:403-471
//   Gaussian 7x7 sigma 2                src/ORBextractor.cc:835,719,742 (cv::GaussianBlur 8U semantics)
//   calcOrb_kernel                      src/cuda/Orb_gpu.cu:67-100
#include <cuda.h>  // CUtensorMap (types only: cuTensorMapEncodeTiled is fetched with cudaGetDriverEntryPoint, no libcuda link)

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "octree_core.cuh"
#include "orb_pattern.inc"
#include "swm_internal.cuh"

namespace swm {

// rBRIEF test points as floats, transposed so that lane t reads entry [k*32 + t] = (P0.x, P0.y, P1.x, P1.y)
// of its k-th comparison with one coalesced 16-byte load (constant memory would serialise: every lane
// indexes a different address).
__device__ float4 g_pattern[8 * 32];
__constant__ int c_umax[16];

// ---- mbarrier helpers (PTX ISA: mbarrier); the TMA tile copies are issued in pyr_walk.cuh / fast_tile.cuh
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  uint32_t done;
  int spins = 0;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    if (!done && ++spins > (1 << 22)) __trap();  // a lost transaction must abort, not hang the GPU
  } while (!done);
}

}  // namespace swm
#include "pyr_walk.cuh"
#include "fast_tile.cuh"
#include "stereo.cuh"
namespace swm {

// ------------------------------------------------------------------------------------------------
// Quadtree: one CTA per (level, frame).
// ------------------------------------------------------------------------------------------------
template <int kMaxLive>
__global__ void __launch_bounds__(256) octree_kernel(const FrameLayout* __restrict__ L, const uint32_t* __restrict__ cand,
                                                     const int* __restrict__ cand_count, int max_pts,
                                                     uint32_t* __restrict__ pts_scratch, uint16_t* __restrict__ pnode_scratch,
                                                     uint8_t* __restrict__ pchild_scratch, uint32_t* __restrict__ sel,
                                                     int* __restrict__ sel_count) {
  extern __shared__ __align__(16) uint8_t smem[];
  OtState<kMaxLive>& S = *reinterpret_cast<OtState<kMaxLive>*>(smem);
  const int lvl = blockIdx.x, f = blockIdx.y;
  const LevelGeom& g = L->lv[lvl];
  const int tid = threadIdx.x;
  const long long slot = ((long long)f * L->nlevels + lvl) * max_pts;
  uint16_t* pnode = pnode_scratch + slot;
  uint8_t* pchild = pchild_scratch + slot;
  int n_all = cand_count[f * L->nlevels + lvl];
  if (n_all > g.cand_cap) n_all = g.cand_cap;
  const uint32_t* src = cand + (long long)f * L->cand_total + g.cand_off;
  const uint32_t* pts = src;
  int n = n_all;
  if (n_all > max_pts) {
    // More survivors than the reference's buffer (Fast.hpp:30): keep the first max_pts in raster
    // order = the max_pts smallest packed words.  Bisect on the value, then gather them.
    int* cnt = &S.scalars[OT_TMP0];
    uint32_t lo = 0, hi = 0xFFFFFFFFu;
    for (int it = 0; it < 32; it++) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      if (tid == 0) *cnt = 0;
      __syncthreads();
      int local = 0;
      for (int i = tid; i < n_all; i += blockDim.x) local += src[i] <= mid;
      if (local) atomicAdd(cnt, local);
      __syncthreads();
      if (*cnt >= max_pts) hi = mid;
      else lo = mid + 1;
      __syncthreads();
    }
    if (tid == 0) *cnt = 0;
    __syncthreads();
    uint32_t* dst = pts_scratch + slot;
    for (int i = tid; i < n_all; i += blockDim.x) {
      const uint32_t v = src[i];
      if (v <= lo) {
        const int k = atomicAdd(cnt, 1);
        if (k < max_pts) dst[k] = v;
      }
    }
    pts = dst;
    n = max_pts;
  }
  __syncthreads();
  const int k = ot_distribute(S, pts, pnode, pchild, n, g.w - 2 * kBand, g.h - 2 * kBand, g.quota,
                              sel + (long long)f * L->sel_total + g.sel_off, g.sel_cap);
  if (tid == 0) sel_count[f * L->nlevels + lvl] = k;
}

// ------------------------------------------------------------------------------------------------
// Orientation (un-blurred plane) + rBRIEF (blurred plane) + keypoint record, one warp per keypoint.
// ------------------------------------------------------------------------------------------------
// 8 CTAs per SM (32 registers): the kernel waits on loads, more resident warps hide them (0.359 vs 0.366 ms at 40 registers)
__global__ void __launch_bounds__(256, 8) describe_kernel(const FrameLayout* __restrict__ L, const uint8_t* __restrict__ plain,
                                                       const uint8_t* __restrict__ blur, const uint32_t* __restrict__ sel,
                                                       const int* __restrict__ sel_count, swm_keypoint* __restrict__ kps,
                                                       uint8_t* __restrict__ desc, int cap, int32_t* __restrict__ n_out) {
  __shared__ __align__(16) uint32_t s_patch[8 * 37 * 11];
  const int f = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int gidx = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int nl = L->nlevels;
  int total = 0, lvl = -1, in_level = 0;
  for (int l = 0; l < nl; l++) {
    const int c = sel_count[f * nl + l];
    if (lvl < 0 && gidx < total + c) {
      lvl = l;
      in_level = gidx - total;
    }
    total += c;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) n_out[f] = total < cap ? total : cap;
  if (lvl < 0 || gidx >= cap) return;
  const LevelGeom& g = L->lv[lvl];
  const uint32_t p = sel[(long long)f * L->sel_total + g.sel_off + in_level];
  const int x = pt_x(p) + kBand, y = pt_y(p) + kBand;  // addBorder_kernel, Fast_gpu.cu:462-471
  const long long off = (long long)f * L->slab_bytes + g.plane_off + (long long)(y + kEdge) * g.pitch + kPadX + x;
  const int pitch = g.pitch;

  // The 37x37 neighbourhood of the BLURRED plane (rBRIEF's samples) is requested first, as 4-byte cp.async copies
  // straight into shared memory (LDGSTS: no registers held): it does not depend on the angle, so its latency overlaps
  // the orientation's own loads instead of following them.
  constexpr int kPR = 18, kPW = 11;  // patch radius (max rotated pattern offset is 18), words per patch row
  uint32_t* patch = s_patch + (threadIdx.x >> 5) * ((2 * kPR + 1) * kPW);
  const int ox = (x - kPR) & ~3;
  {
    const uint8_t* b0 = blur + (long long)f * L->slab_bytes + g.plane_off + (long long)(y - kPR + kEdge) * g.pitch + kPadX + ox;
    const uint32_t p0 = smem_u32(patch);
#pragma unroll
    for (int it = 0; it < 13; it++) {
      const int idx = lane + 32 * it;
      const int r = idx / kPW, wd = idx - r * kPW;
      if (idx < (2 * kPR + 1) * kPW)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(p0 + 4u * idx), "l"(b0 + (long long)r * g.pitch + 4 * wd) : "memory");
    }
  }
  // IC_Angle (Fast_gpu.cu:403-460): integer moments over the radius-15 disc, one lane per column
  // (row pointers advance by the pitch and the disc half-widths are compile-time offsets: the loop is 2 loads + 6
  // integer instructions per row pair, where index arithmetic per load used to be a third of this kernel)
  const uint8_t* rp = plain + off + lane;  // row y + v, my column of the 31-wide window shifted by umax below
  const uint8_t* rm = rp;                  // row y - v
  int m10 = 0, m01 = 0;
  if (lane <= 2 * kHalfPatch) m10 = (lane - kHalfPatch) * (int)rp[-kHalfPatch];
#pragma unroll
  for (int v = 1; v <= kHalfPatch; ++v) {
    constexpr int kUmax[kHalfPatch + 1] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};  // ORBextractor.cc:380-404
    const int d = kUmax[v];
    rp += pitch;
    rm -= pitch;
    if (lane <= 2 * d) {
      const int u = lane - d;
      const int vp = rp[-d], vm = rm[-d];
      m01 += v * (vp - vm);
      m10 += u * (vp + vm);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m10 += __shfl_xor_sync(0xffffffffu, m10, o);
    m01 += __shfl_xor_sync(0xffffffffu, m01, o);
  }
  const float kPiF = 3.14159265f;  // CV_PI_F
  float ang = atan2f((float)m01, (float)m10);
  if (ang < 0) ang = __fadd_rn(ang, 2.0f * kPiF);
  ang = __fmul_rn(ang, 180.0f / kPiF);

  // calcOrb_kernel (Orb_gpu.cu:67-100): lane t -> descriptor byte t.  The 37x37 neighbourhood of the
  // blurred plane is staged per warp with aligned word loads (2-3 sectors per row instead of one sector
  // per sample), then the 512 rotated samples are read from shared memory.
  const float factor_pi = (float)(3.1415926535897932384626433832795 / 180.f);
  const float rad = __fmul_rn(ang, factor_pi);
  const float ca = cosf(rad), sb = sinf(rad);
  // the patch requested before the orientation loop has landed
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncwarp();
  const uint8_t* b = reinterpret_cast<const uint8_t*>(patch) + kPR * (kPW * 4) + (x - ox);
  int val = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const float4 pp = __ldg(&g_pattern[k * 32 + lane]);
    const float x0 = pp.x, y0 = pp.y, x1 = pp.z, y1 = pp.w;
    const int t0 = b[__float2int_rn(__fadd_rn(__fmul_rn(x0, sb), __fmul_rn(y0, ca))) * (kPW * 4) +
                     __float2int_rn(__fsub_rn(__fmul_rn(x0, ca), __fmul_rn(y0, sb)))];
    const int t1 = b[__float2int_rn(__fadd_rn(__fmul_rn(x1, sb), __fmul_rn(y1, ca))) * (kPW * 4) +
                     __float2int_rn(__fsub_rn(__fmul_rn(x1, ca), __fmul_rn(y1, sb)))];
    val |= (t0 < t1) << k;
  }
  const long long o = (long long)f * cap + gidx;
  desc[o * 32 + lane] = (uint8_t)val;
  if (lane == 0) {
    swm_keypoint kp;
    kp.x = lvl ? __fmul_rn((float)x, g.scale) : (float)x;  // ORBextractor.cc:808-814
    kp.y = lvl ? __fmul_rn((float)y, g.scale) : (float)y;
    kp.size = (float)g.kp_size;
    kp.angle = ang;
    kp.response = (float)pt_score(p);
    kp.octave = lvl;
    kp.class_id = -1;
    kps[o] = kp;
  }
}

}  // namespace swm

// =================================================================================================
// Host side: handle, tables, C ABI
// =================================================================================================
using namespace swm;

namespace {

thread_local std::string g_create_error;
std::once_flag g_const_once[64];

#define SWM_CK(h, call)                                                     \
  do {                                                                      \
    cudaError_t e_ = (call);                                                \
    if (e_ != cudaSuccess) {                                                \
      (h)->err = cuda_err(#call, e_);                                       \
      return SWM_E_CUDA;                                                    \
    }                                                                       \
  } while (0)

inline int cv_round_f(float v) { return (int)lrintf(v); }
inline int cv_floor_f(float v) {
  int i = (int)v;
  return i - (i > v);
}
inline short sat_s16(int v) { return (short)(v < -32768 ? -32768 : (v > 32767 ? 32767 : v)); }
inline long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }

}  // namespace

int swm::check_device(int device, std::string* err) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    *err = "no CUDA device visible (" + std::string(cudaGetErrorString(e)) +
           "); libswm_orb has no CPU fallback";
    return SWM_E_NODEVICE;
  }
  if (device < 0 || device >= count) {
    *err = "device index out of range";
    return SWM_E_INVALID;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    *err = cuda_err("cudaGetDeviceProperties", e);
    return SWM_E_CUDA;
  }
  if (prop.major != 10) {
    *err = "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
           "; libswm_orb is built for sm_100a only";
    return SWM_E_NODEVICE;
  }
  return SWM_OK;
}

struct swm_orb {
  swm_orb_cfg cfg;
  int device = 0;
  std::string err;
  cudaStream_t stream = nullptr;
  // tables (ORBextractor.cc:346-378)
  float sf[SWM_MAX_LEVELS], inv_sf[SWM_MAX_LEVELS], sig2[SWM_MAX_LEVELS], inv_sig2[SWM_MAX_LEVELS];
  int quota[SWM_MAX_LEVELS];
  int max_kp = 0;
  int max_pts = 10000;
  // geometry for the current frame size
  FrameLayout lay;
  bool allocated = false;
  FrameLayout* d_lay = nullptr;
  ResizeTap *d_xtab = nullptr, *d_ytab = nullptr;
  CUtensorMap* d_maps = nullptr;  // per level: the un-blurred plane over all frames, for pyr_walk_kernel's TMA tiles
  CUtensorMap* d_fmaps = nullptr; // the same planes with fast_tile_kernel's box
  // stereo matching (left-view handle owns the scratch): per (frame, left keypoint) uRight, depth, SAD
  float *d_uright = nullptr, *d_depth = nullptr;
  int32_t* d_sad = nullptr;
  size_t stereo_cap = 0;
  cudaEvent_t stereo_ev = nullptr;
  uint8_t *d_plain = nullptr, *d_blur = nullptr, *d_score = nullptr;
  uint8_t* d_retry = nullptr;
  int4* d_fblk = nullptr;       // per FAST block: (level, bx, by, 0)
  int* d_retry_list = nullptr;  // [0] = count, then (frame * blocks + block) ids holding a retry tile
  int n_sm = 148;
  int fast_run = kFT;           // FAST tiles per warp: kFT for batch handles, 1 for a single-frame handle (shorter critical path)
  uint32_t *d_cand = nullptr, *d_sel = nullptr;
  uint32_t* d_pts = nullptr;     // quadtree scratch per (frame, level): capped point list, node labels, child ids
  uint16_t* d_pnode = nullptr;
  uint8_t* d_pchild = nullptr;
  int *d_counts = nullptr;  // [2][B][nlevels]: candidate counts, selection counts
  // staging for the host-buffer entry points
  uint8_t* d_img = nullptr;
  int img_pitch = 0;
  swm_keypoint* d_kps = nullptr;
  uint8_t* d_desc = nullptr;
  int32_t* d_n = nullptr;
  int last_batch = 0;
  int last_launches = 0;
  // single-frame latency path: the launches of one frame captured once per geometry and replayed as a CUDA graph
  cudaGraphExec_t graph = nullptr;
  int graph_runs = 0;  // host-chunk calls with nb == 1 since the buffers were (re)allocated
  bool debug_score = false;  // keep a FAST score map in HBM for parity tests (swm_orb_set_debug)
  // last input (for swm_orb_run_stage)
  const uint8_t* last_img = nullptr;
  int last_stride = 0;
  long long last_frame_stride = 0;
  swm_keypoint* last_kps = nullptr;
  cudaStream_t last_stream = nullptr;
  uint8_t* last_desc = nullptr;
  int32_t* last_n = nullptr;
  int last_cap = 0;
  // async host-buffer call in flight (swm_orb_extract_batch_async .. swm_orb_sync)
  int32_t* pending_n = nullptr;
  int pending_batch = 0;
  int pending_cap = 0;
  // single frame into pageable caller memory: results are staged through a pinned buffer and handed over in
  // swm_orb_sync (only the n valid entries are copied)
  uint8_t* h_stage = nullptr;
  size_t stage_cap = 0;
  swm_keypoint* stage_kps = nullptr;
  uint8_t* stage_desc = nullptr;
  int stage_ccap = 0;
  int graph_stride = 0;  // row stride the single-frame graph was captured with
};

namespace {

void free_frame_buffers(swm_orb* h) {
  if (h->h_stage) cudaFreeHost(h->h_stage);
  h->h_stage = nullptr;
  h->stage_cap = 0;
  if (h->graph) cudaGraphExecDestroy(h->graph);
  h->graph = nullptr;
  h->graph_runs = 0;
  cudaFree(h->d_lay); cudaFree(h->d_xtab); cudaFree(h->d_ytab); cudaFree(h->d_maps); cudaFree(h->d_fmaps); cudaFree(h->d_uright); cudaFree(h->d_depth); cudaFree(h->d_sad);
  cudaFree(h->d_plain); cudaFree(h->d_blur); cudaFree(h->d_score);
  cudaFree(h->d_retry); cudaFree(h->d_retry_list); cudaFree(h->d_fblk); cudaFree(h->d_pts); cudaFree(h->d_pnode); cudaFree(h->d_pchild); cudaFree(h->d_cand); cudaFree(h->d_sel); cudaFree(h->d_counts);
  cudaFree(h->d_img); cudaFree(h->d_kps); cudaFree(h->d_desc); cudaFree(h->d_n);
  h->d_lay = nullptr; h->d_xtab = h->d_ytab = nullptr; h->d_maps = nullptr; h->d_fmaps = nullptr; h->d_uright = h->d_depth = nullptr; h->d_sad = nullptr; h->stereo_cap = 0;
  h->d_plain = h->d_blur = h->d_score = nullptr;
  h->d_retry = nullptr; h->d_retry_list = nullptr; h->d_fblk = nullptr; h->d_pts = nullptr; h->d_pnode = nullptr; h->d_pchild = nullptr; h->d_cand = h->d_sel = nullptr; h->d_counts = nullptr;
  h->d_img = nullptr; h->d_kps = nullptr; h->d_desc = nullptr; h->d_n = nullptr;
  h->allocated = false;
}

// pyr_walk_kernel's strips: the bordered row [-20, w + 20) in lanes of 4 columns, at most kWalkLanes useful lanes per warp
void walk_strips(int w, int* nstrips, int* strip_lanes) {
  const int nl = (w + 2 * (-kWalkX0) + 3) / 4;
  *nstrips = (nl + kWalkLanes - 1) / kWalkLanes;
  *strip_lanes = (nl + *nstrips - 1) / *nstrips;
}

// cv::resize INTER_LINEAR coefficient tables (OpenCV imgproc resize.cpp, restated): for each
// destination coordinate the source offset and two 11-bit fixed-point weights.
void build_taps(int s, int d, std::vector<ResizeTap>& out, bool horizontal) {
  const double inv_scale = (double)d / s;
  const double scale = 1. / inv_scale;
  for (int i = 0; i < d; i++) {
    float f = (float)((i + 0.5) * scale - 0.5);
    int o = cv_floor_f(f);
    f -= o;
    if (horizontal) {
      if (o < 0) { f = 0; o = 0; }
      if (o >= s - 1) { f = 0; o = s - 1; }
    }
    ResizeTap t;
    t.ofs = (int16_t)o;
    t.a0 = sat_s16(cv_round_f((1.f - f) * 2048));
    t.a1 = sat_s16(cv_round_f(f * 2048));
    t.pad = 0;
    out.push_back(t);
  }
}

int setup_geometry(swm_orb* h, int w, int hh) {
  if (h->allocated && h->lay.w == w && h->lay.h == hh) return SWM_OK;
  free_frame_buffers(h);  // unconditional: a set-up that failed part-way leaves buffers behind with allocated == false
  const int nl = h->cfg.nlevels;
  FrameLayout& L = h->lay;
  memset(&L, 0, sizeof(L));
  L.nlevels = nl;
  L.w = w;
  L.h = hh;
  std::vector<ResizeTap> xt, yt;
  long long off = 0;
  int tile_off = 0, cand_off = 0, sel_off = 0, fblk_off = 0;
  for (int l = 0; l < nl; l++) {
    LevelGeom& g = L.lv[l];
    g.w = cv_round_f((float)w * h->inv_sf[l]);
    g.h = cv_round_f((float)hh * h->inv_sf[l]);
    if (g.w < 2 * kEdge + 1 || g.h < 2 * kEdge + 1 || g.w > 4000 || g.h > 4000) {
      h->err = "image size unsupported: every pyramid level must be between 39 and 4000 pixels per side";
      return SWM_E_INVALID;
    }
    const int n_ini = (int)lroundf((float)(g.w - 2 * kBand) / (float)(g.h - 2 * kBand));
    if (n_ini < 1 || n_ini > kOtMaxIni) {
      h->err = "unsupported aspect ratio (DistributeOctTree needs 1 <= round(W/H) <= 16)";
      return SWM_E_INVALID;
    }
    g.pitch = (int)align_up(kPadX + g.w + kEdge, 128);
    g.rows = g.h + 2 * kEdge;
    g.plane_off = off;
    off += align_up((long long)g.pitch * g.rows, 256);
    g.xtab_off = (int)xt.size();
    g.ytab_off = (int)yt.size();
    if (l > 0) {
      build_taps(L.lv[l - 1].w, g.w, xt, true);
      build_taps(L.lv[l - 1].h, g.h, yt, false);
    }
    if (l > 0) {  // pyr_walk_kernel: limits of its per-lane window and of its staged source rows
      const ResizeTap* xt0 = xt.data() + g.xtab_off;
      const ResizeTap* yt0 = yt.data() + g.ytab_off;
      const int sh = L.lv[l - 1].h;
      int nstrips, sl;
      walk_strips(g.w, &nstrips, &sl);
      bool ok = true;
      for (int st = 0; st < nstrips && ok; st++) {
        int xb = 1 << 30, xend = -1;
        for (int lane = 0; lane < 32; lane++) {
          const int X = kWalkX0 + 4 * (st * sl + lane - 1);
          int lo = 1 << 30, hi = -1;
          for (int k = 0; k < 4; k++) {
            const int o = xt0[reflect101(X + k, g.w)].ofs;
            lo = std::min(lo, o);
            hi = std::max(hi, o);
          }
          if (hi - lo > 6) ok = false;  // four adjacent columns' taps within 7 source bytes
          xb = std::min(xb, lo & ~3);
          xend = std::max(xend, (lo & ~3) + 12);
        }
        if (((xend - (xb & ~15) + 15) & ~15) > kWalkRowBytes) ok = false;
      }
      for (int v0 = -5; v0 <= g.h + 2 && ok; v0++) {
        int lo = 1 << 30, hi = -1;
        for (int i = 0; i < 4; i++) {
          const int v = v0 + i, ay = v < 0 ? -v : (v >= g.h ? 2 * g.h - 2 - v : v);
          lo = std::min(lo, (int)yt0[ay].ofs);
          hi = std::max(hi, std::min(yt0[ay].ofs + 1, sh - 1));
        }
        if (hi - lo + 1 > kWalkStageRows) ok = false;
      }
      if (!ok) { h->err = "scale factor too large for the pyramid kernel"; return SWM_E_INVALID; }
    }
    g.tiles_x = (g.w - 2 * kEdge + 31) / 32;
    g.tiles_y = (g.h - 2 * kEdge + 31) / 32;
    g.tile_off = tile_off;
    tile_off += g.tiles_x * g.tiles_y;
    g.fblk_x = (g.tiles_x + h->fast_run - 1) / h->fast_run;
    g.fblk_off = fblk_off;
    fblk_off += g.fblk_x * g.tiles_y;
    // strict 8-neighbour maxima cannot be adjacent: at most one per 2x2 block
    g.cand_cap = ((g.w - 2 * kEdge + 1) / 2 + 1) * ((g.h - 2 * kEdge + 1) / 2 + 1);
    g.cand_off = cand_off;
    cand_off += (g.cand_cap + 31) / 32 * 32;
    g.quota = h->quota[l];
    g.sel_cap = std::max(g.quota + 3, 4 * n_ini) + 1;  // also the bound on live quadtree nodes (<= quota + 64)
    g.sel_off = sel_off;
    sel_off += (g.sel_cap + 31) / 32 * 32;
    g.scale = h->sf[l];
    g.kp_size = (int)(kPatch * h->sf[l]);
  }
  if (xt.empty()) { xt.push_back(ResizeTap{0, 2048, 0, 0}); yt.push_back(ResizeTap{0, 2048, 0, 0}); }
  L.slab_bytes = off;
  L.tiles_total = tile_off;
  L.fblk_total = fblk_off;
  L.cand_total = cand_off;
  L.sel_total = sel_off;
  int maxkp = 0;
  for (int l = 0; l < nl; l++) maxkp += L.lv[l].sel_cap;
  h->max_kp = maxkp;

  const int B = h->cfg.max_batch;
  SWM_CK(h, cudaSetDevice(h->device));
  SWM_CK(h, cudaMalloc(&h->d_lay, sizeof(FrameLayout)));
  SWM_CK(h, cudaMalloc(&h->d_xtab, xt.size() * sizeof(ResizeTap)));
  SWM_CK(h, cudaMalloc(&h->d_ytab, yt.size() * sizeof(ResizeTap)));
  SWM_CK(h, cudaMalloc(&h->d_plain, (size_t)L.slab_bytes * B + 1024));  // + slack: bulk-copied rows may overhang the last plane
  SWM_CK(h, cudaMalloc(&h->d_blur, (size_t)L.slab_bytes * B));
  if (h->debug_score) SWM_CK(h, cudaMalloc(&h->d_score, (size_t)L.slab_bytes * B));
  SWM_CK(h, cudaMalloc(&h->d_retry, (size_t)L.tiles_total * B));
  SWM_CK(h, cudaMalloc(&h->d_retry_list, ((size_t)L.fblk_total * B + 1) * sizeof(int)));
  SWM_CK(h, cudaMalloc(&h->d_cand, (size_t)L.cand_total * B * sizeof(uint32_t)));
  SWM_CK(h, cudaMalloc(&h->d_sel, (size_t)L.sel_total * B * sizeof(uint32_t)));
  SWM_CK(h, cudaMalloc(&h->d_pts, (size_t)h->max_pts * nl * B * sizeof(uint32_t)));
  SWM_CK(h, cudaMalloc(&h->d_pnode, (size_t)h->max_pts * nl * B * sizeof(uint16_t)));
  SWM_CK(h, cudaMalloc(&h->d_pchild, (size_t)h->max_pts * nl * B));
  SWM_CK(h, cudaMalloc(&h->d_counts, (size_t)2 * B * nl * sizeof(int)));
  h->img_pitch = (int)align_up(w, 4);  // rows stay word-aligned; equals the usual host stride so uploads are 1-D
  SWM_CK(h, cudaMalloc(&h->d_img, (size_t)h->img_pitch * hh * B));
  SWM_CK(h, cudaMalloc(&h->d_kps, (size_t)h->max_kp * B * sizeof(swm_keypoint)));
  SWM_CK(h, cudaMalloc(&h->d_desc, (size_t)h->max_kp * B * 32));
  SWM_CK(h, cudaMalloc(&h->d_n, (size_t)B * sizeof(int32_t)));
  {
    std::vector<int4> desc(L.fblk_total);
    for (int l = 0; l < nl; l++)
      for (int by = 0; by < L.lv[l].tiles_y; by++)
        for (int bx = 0; bx < L.lv[l].fblk_x; bx++) desc[L.lv[l].fblk_off + by * L.lv[l].fblk_x + bx] = make_int4(l, bx, by, 0);
    SWM_CK(h, cudaMalloc(&h->d_fblk, desc.size() * sizeof(int4)));
    SWM_CK(h, cudaMemcpy(h->d_fblk, desc.data(), desc.size() * sizeof(int4), cudaMemcpyHostToDevice));
  }
  SWM_CK(h, cudaMemcpy(h->d_lay, &L, sizeof(L), cudaMemcpyHostToDevice));
  SWM_CK(h, cudaMemcpy(h->d_xtab, xt.data(), xt.size() * sizeof(ResizeTap), cudaMemcpyHostToDevice));
  SWM_CK(h, cudaMemcpy(h->d_ytab, yt.data(), yt.size() * sizeof(ResizeTap), cudaMemcpyHostToDevice));
  {
    // tensor maps of the un-blurred planes: u8 tensor (row byte, row, frame), box kWalkRowBytes x kWalkStageRows x 1
    typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    SWM_CK(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) { h->err = "cuTensorMapEncodeTiled is not available in this driver"; return SWM_E_CUDA; }
    std::vector<CUtensorMap> maps(2 * nl);
    memset(maps.data(), 0, sizeof(CUtensorMap) * 2 * nl);
    for (int l = 0; l < nl; l++) {
      const LevelGeom& g = L.lv[l];
      const cuuint64_t dims[3] = {(cuuint64_t)g.pitch, (cuuint64_t)g.rows, (cuuint64_t)B};
      const cuuint64_t strides[2] = {(cuuint64_t)g.pitch, (cuuint64_t)L.slab_bytes};
      const cuuint32_t estr[3] = {1u, 1u, 1u};
      for (int which = 0; which < 2; which++) {  // 0: pyramid walk (source rows of level l + 1), 1: FAST tile window
        const cuuint32_t box[3] = {(cuuint32_t)(which ? FT_PITCH : kWalkRowBytes), (cuuint32_t)(which ? FT_ROWS : kWalkStageRows), 1u};
        const CUresult r = ((EncodeTiled)fn)(&maps[which * nl + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, h->d_plain + g.plane_off, dims, strides,
                                             box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { h->err = "cuTensorMapEncodeTiled failed for a pyramid plane (code " + std::to_string((int)r) + ")"; return SWM_E_CUDA; }
      }
    }
    SWM_CK(h, cudaMalloc(&h->d_maps, sizeof(CUtensorMap) * nl));
    SWM_CK(h, cudaMalloc(&h->d_fmaps, sizeof(CUtensorMap) * nl));
    SWM_CK(h, cudaMemcpy(h->d_maps, maps.data(), sizeof(CUtensorMap) * nl, cudaMemcpyHostToDevice));
    SWM_CK(h, cudaMemcpy(h->d_fmaps, maps.data() + nl, sizeof(CUtensorMap) * nl, cudaMemcpyHostToDevice));
  }
  // planes start zeroed so padding bytes are deterministic
  SWM_CK(h, cudaMemset(h->d_plain, 0, (size_t)L.slab_bytes * B));
  SWM_CK(h, cudaMemset(h->d_blur, 0, (size_t)L.slab_bytes * B));
  if (h->debug_score) SWM_CK(h, cudaMemset(h->d_score, 0, (size_t)L.slab_bytes * B));
  h->allocated = true;
  return SWM_OK;
}

// quadtree instantiations by the largest per-level quota of the handle
int octree_variant(const swm_orb* h) {
  int q = 0;
  for (int l = 0; l < h->cfg.nlevels; l++) q = std::max(q, h->quota[l]);
  return q <= 512 ? 0 : (q <= 1024 ? 1 : 2);
}
size_t octree_smem(const swm_orb* h) {
  const int v = octree_variant(h);
  return v == 0 ? sizeof(OtState<ot_max_live(512)>) : (v == 1 ? sizeof(OtState<ot_max_live(1024)>) : sizeof(OtState<ot_max_live(2048)>));
}

// Enqueue the stages selected by `mask` for `batch` frames on `st`.
int enqueue(swm_orb* h, int mask, const uint8_t* d_imgs, int batch, int stride, long long frame_stride,
            swm_keypoint* d_kps, uint8_t* d_desc, int cap, int32_t* d_n, cudaStream_t st) {
  const FrameLayout& L = h->lay;
  const int nl = L.nlevels;
  int launches = 0;
  int* d_cand_count = h->d_counts;
  int* d_sel_count = h->d_counts + (size_t)h->cfg.max_batch * nl;
  if (mask & SWM_STAGE_PYRAMID) {
    for (int l = 0; l < nl; l++) {
      PyrArgs a;
      a.dst = L.lv[l];
      a.src = L.lv[l ? l - 1 : 0];
      a.img = d_imgs;
      a.img_stride = stride;
      a.img_frame_stride = frame_stride;
      a.plain = h->d_plain;
      a.blur = h->d_blur;
      a.slab_bytes = L.slab_bytes;
      a.xtab = h->d_xtab;
      a.ytab = h->d_ytab;
      a.src_map = h->d_maps + (l ? l - 1 : 0);
      // one warp per (strip of <= 120 columns of the bordered row, block of rows).  Row blocks are as long as the
      // batch allows while the level still fills the GPU about twice over (the 8-row blur warm-up is amortised over
      // 64 rows for large batches; a single frame gets 16-row blocks and several hundred warps per level).
      walk_strips(a.dst.w, &a.nstrips, &a.strip_lanes);
#ifndef SWM_WALK_WAVES
#define SWM_WALK_WAVES 2
#endif
      const int want_jobs = SWM_WALK_WAVES * h->n_sm * 24;
      const int nrb_want = std::max(1, (want_jobs + batch * a.nstrips - 1) / (batch * a.nstrips));
      int rows = (int)align_up((a.dst.h + nrb_want - 1) / nrb_want, 4);
#ifndef SWM_WALK_MAXROWS
#define SWM_WALK_MAXROWS 64
#endif
      rows = std::min(SWM_WALK_MAXROWS, std::max(batch >= 4 ? 16 : 8, rows));
      a.nrb = (a.dst.h + rows - 1) / rows;
      a.rows_per_job = (int)align_up((a.dst.h + a.nrb - 1) / a.nrb, 4);
      a.nrb = (a.dst.h + a.rows_per_job - 1) / a.rows_per_job;
      dim3 grid(a.nstrips, a.nrb, batch);
      if (l == 0) pyr_walk_kernel<true><<<grid, 32, 0, st>>>(a);
      else pyr_walk_kernel<false><<<grid, 32, 0, st>>>(a);
      launches++;
    }
  }
  if (mask & SWM_STAGE_NMS) {
    SWM_CK(h, cudaMemsetAsync(h->d_counts, 0, (size_t)2 * h->cfg.max_batch * nl * sizeof(int), st));
    SWM_CK(h, cudaMemsetAsync(h->d_retry_list, 0, sizeof(int), st));
    dim3 grid(L.fblk_total, batch);
    uint8_t* dbg = h->debug_score ? h->d_score : nullptr;
    FastArgs fa;
    fa.L = h->d_lay;
    fa.maps = h->d_fmaps;
    fa.fblk_desc = h->d_fblk;
    fa.ini_th = h->cfg.ini_th_fast;
    fa.min_th = h->cfg.min_th_fast;
    fa.retry = h->d_retry;
    fa.retry_list = h->d_retry_list;
    fa.cand = h->d_cand;
    fa.cand_count = d_cand_count;
    fa.dbg_score = dbg;
    fa.run_len = h->fast_run;
    if (dbg) fast_tile_kernel<1, true><<<grid, 32, 0, st>>>(fa);
    else fast_tile_kernel<1, false><<<grid, 32, 0, st>>>(fa);
    fa.dbg_score = nullptr;
    // pass 2 walks the retry list with a persistent grid; a single frame has few runs, so it gets few warps to start
    const int grid2 = std::min(h->n_sm * 24, std::max(h->n_sm, L.fblk_total * batch / 4));
    fast_tile_kernel<2, false><<<grid2, 32, 0, st>>>(fa);
    launches += 2;
  }
  if (mask & SWM_STAGE_OCTREE) {
    dim3 grid(nl, batch);
    const int v = octree_variant(h);
    if (v == 0)
      octree_kernel<ot_max_live(512)><<<grid, 256, octree_smem(h), st>>>(h->d_lay, h->d_cand, d_cand_count, h->max_pts, h->d_pts,
                                                                         h->d_pnode, h->d_pchild, h->d_sel, d_sel_count);
    else if (v == 1)
      octree_kernel<ot_max_live(1024)><<<grid, 256, octree_smem(h), st>>>(h->d_lay, h->d_cand, d_cand_count, h->max_pts, h->d_pts,
                                                                          h->d_pnode, h->d_pchild, h->d_sel, d_sel_count);
    else
      octree_kernel<ot_max_live(2048)><<<grid, 256, octree_smem(h), st>>>(h->d_lay, h->d_cand, d_cand_count, h->max_pts, h->d_pts,
                                                                          h->d_pnode, h->d_pchild, h->d_sel, d_sel_count);
    launches++;
  }
  if (mask & SWM_STAGE_DESCRIBE) {
    const int eff_cap = cap < h->max_kp ? cap : h->max_kp;
    dim3 grid((eff_cap + 7) / 8, batch);
    describe_kernel<<<grid, 256, 0, st>>>(h->d_lay, h->d_plain, h->d_blur, h->d_sel, d_sel_count, d_kps, d_desc, cap,
                                          d_n);
    launches++;
  }
  SWM_CK(h, cudaGetLastError());
  h->last_launches = launches;
  return SWM_OK;
}

}  // namespace

extern "C" {

const char* swm_version(void) { return "swm_orb 0.1 sm_100a " __DATE__; }

int swm_orb_create(const swm_orb_cfg* cfg, int device, swm_orb** out) {
  if (!cfg || !out) return SWM_E_INVALID;
  *out = nullptr;
  if (cfg->nfeatures <= 0 || cfg->nlevels < 1 || cfg->nlevels > SWM_MAX_LEVELS || !(cfg->scale_factor > 1.0f) ||
      cfg->scale_factor > 1.5f || cfg->min_th_fast < 1 || cfg->ini_th_fast > 126 ||
      cfg->ini_th_fast < cfg->min_th_fast || cfg->ini_th_fast > 254 || cfg->max_batch < 1) {
    g_create_error = "invalid swm_orb_cfg";
    return SWM_E_INVALID;
  }
  int rc = check_device(device, &g_create_error);
  if (rc != SWM_OK) return rc;
  swm_orb* h = new swm_orb;
  h->cfg = *cfg;
  h->device = device;
  h->max_pts = cfg->max_fast_per_level > 0 ? cfg->max_fast_per_level : 10000;
  h->fast_run = cfg->max_batch >= 8 ? kFT : 1;
  if (h->max_pts > 20000) h->max_pts = 20000;
  // scale tables: float chain with a double scale factor (ORBextractor.cc:346-362, ORBextractor.h:108)
  const double s = cfg->scale_factor;
  h->sf[0] = 1.0f;
  h->sig2[0] = 1.0f;
  for (int i = 1; i < cfg->nlevels; i++) {
    h->sf[i] = (float)(h->sf[i - 1] * s);
    h->sig2[i] = h->sf[i] * h->sf[i];
  }
  for (int i = 0; i < cfg->nlevels; i++) {
    h->inv_sf[i] = 1.0f / h->sf[i];
    h->inv_sig2[i] = 1.0f / h->sig2[i];
  }
  // per-level quotas (ORBextractor.cc:367-378)
  {
    const float factor = (float)(1.0f / s);
    float per = (float)(cfg->nfeatures * (1.0f - factor) / (1.0f - std::pow((double)factor, cfg->nlevels)));
    int sum = 0;
    for (int l = 0; l < cfg->nlevels - 1; l++) {
      h->quota[l] = cv_round_f(per);
      sum += h->quota[l];
      per *= factor;
    }
    h->quota[cfg->nlevels - 1] = std::max(cfg->nfeatures - sum, 0);
    for (int l = 0; l < cfg->nlevels; l++)
      if (h->quota[l] > kOtMaxQuota) {
        g_create_error = "nfeatures too large: per-level quota exceeds 2048";
        delete h;
        return SWM_E_INVALID;
      }
  }
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->n_sm, cudaDevAttrMultiProcessorCount, device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) {
    // constant tables are per device; identical for every handle (ORBextractor.cc:380-404)
    std::call_once(g_const_once[device & 63], [&]() {
      int umax[16];
      const int hp = kHalfPatch;
      int v, v0;
      const int vmax = cv_floor_f(hp * std::sqrt(2.f) / 2 + 1);
      const int vmin = (int)std::ceil(hp * std::sqrt(2.f) / 2);
      for (v = 0; v <= vmax; ++v) umax[v] = (int)lrint(std::sqrt((double)hp * hp - v * v));
      for (v = hp, v0 = 0; v >= vmin; --v) {
        while (umax[v0] == umax[v0 + 1]) ++v0;
        umax[v] = v0;
        ++v0;
      }
      static const int kUmaxExpected[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
      cudaError_t e2 = memcmp(umax, kUmaxExpected, sizeof(umax)) == 0 ? cudaSuccess : cudaErrorInvalidValue;  // describe_kernel's compile-time table
      if (e2 == cudaSuccess) e2 = cudaMemcpyToSymbol(c_umax, umax, sizeof(umax));
      if (e2 == cudaSuccess) {
        std::vector<float> pat(8 * 32 * 4);
        for (int t = 0; t < 32; t++)
          for (int k = 0; k < 8; k++)
            for (int c = 0; c < 4; c++) pat[(k * 32 + t) * 4 + c] = (float)kSwmOrbPattern[32 * t + 4 * k + c];
        e2 = cudaMemcpyToSymbol(g_pattern, pat.data(), pat.size() * sizeof(float));
      }
      if (e2 != cudaSuccess) e = e2;
    });
  }
  if (e == cudaSuccess) {
    const int v = octree_variant(h);
    const void* fn = v == 0 ? (const void*)octree_kernel<ot_max_live(512)>
                            : (v == 1 ? (const void*)octree_kernel<ot_max_live(1024)> : (const void*)octree_kernel<ot_max_live(2048)>);
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)octree_smem(h));
  }
  if (e != cudaSuccess) {
    g_create_error = cuda_err("swm_orb_create", e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return SWM_E_CUDA;
  }
  *out = h;
  return SWM_OK;
}

void swm_orb_destroy(swm_orb* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  free_frame_buffers(h);  // unconditional: a set-up that failed part-way leaves buffers behind with allocated == false
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* swm_last_error(const swm_orb* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int swm_orb_extract_batch_device(swm_orb* h, const uint8_t* d_imgs, int batch, int w, int h_px, int stride,
                                 size_t frame_stride, swm_keypoint* d_kps, uint8_t* d_desc, int cap, int32_t* d_n,
                                 void* stream) {
  if (!h) return SWM_E_INVALID;
  if (batch < 0 || !d_kps || !d_desc || !d_n || cap < 1) { h->err = "bad argument"; return SWM_E_INVALID; }
  if (batch == 0) return SWM_OK;
  if (!d_imgs || w <= 0 || h_px <= 0 || stride < w) { h->err = "bad image argument"; return SWM_E_INVALID; }
  if (batch > h->cfg.max_batch) { h->err = "batch exceeds cfg.max_batch"; return SWM_E_CAPACITY; }
  SWM_CK(h, cudaSetDevice(h->device));
  int rc = setup_geometry(h, w, h_px);
  if (rc != SWM_OK) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  h->last_img = d_imgs; h->last_stride = stride; h->last_frame_stride = (long long)frame_stride;
  h->last_kps = d_kps; h->last_desc = d_desc; h->last_n = d_n; h->last_cap = cap;
  h->last_batch = batch;
  h->last_stream = st;
  return enqueue(h, 15, d_imgs, batch, stride, (long long)frame_stride, d_kps, d_desc, cap, d_n, st);
}

static int enqueue_host_chunk(swm_orb* h, const uint8_t* src, int nb, int w, int h_px, int stride,
                              size_t frame_stride, swm_keypoint* kps, uint8_t* desc, int cap, int32_t* n) {
  const int kcap = h->max_kp;
  const int ccap = cap < kcap ? cap : kcap;
  // Device-side row stride of the uploaded frames.  Tightly packed host frames (stride == w, e.g. the 1241-pixel
  // KITTI rows) go up as ONE linear copy and keep their stride: a 2-D copy of odd-length rows runs at a fraction of the
  // link rate, while the level-0 kernel reads rows of any alignment (byte path) at the device-resident rate.
  int dstride = h->img_pitch;
  if (frame_stride == (size_t)stride * h_px && (stride == h->img_pitch || stride == w)) {
    dstride = stride;
    SWM_CK(h, cudaMemcpyAsync(h->d_img, src, (size_t)stride * h_px * nb, cudaMemcpyHostToDevice, h->stream));
  } else if (frame_stride == (size_t)stride * h_px) {
    SWM_CK(h, cudaMemcpy2DAsync(h->d_img, h->img_pitch, src, stride, w, (size_t)h_px * nb, cudaMemcpyHostToDevice,
                                h->stream));
  } else {
    for (int f = 0; f < nb; f++)
      SWM_CK(h, cudaMemcpy2DAsync(h->d_img + (size_t)f * h->img_pitch * h_px, h->img_pitch,
                                  src + (size_t)f * frame_stride, stride, w, h_px, cudaMemcpyHostToDevice, h->stream));
  }
  int rc = SWM_OK;
  // One frame = 13 launches + 2 memsets, all on handle-owned buffers: launch-latency bound.  The first single-frame
  // call after (re)allocation runs normally (lazy initialisation done), the second is captured into a CUDA graph,
  // later ones replay it.  SWM_NO_GRAPH=1 disables this (A/B measurement); the debug score map changes kernel
  // arguments and is never captured.
  static const bool no_graph = getenv("SWM_NO_GRAPH") != nullptr;
  const bool graphable = nb == 1 && !no_graph && !h->debug_score;
  if (graphable && h->graph && h->graph_stride == dstride) {
    h->last_img = h->d_img; h->last_stride = dstride; h->last_frame_stride = (long long)dstride * h_px;
    h->last_kps = h->d_kps; h->last_desc = h->d_desc; h->last_n = h->d_n; h->last_cap = kcap;
    h->last_batch = 1;
    h->last_stream = h->stream;
    SWM_CK(h, cudaGraphLaunch(h->graph, h->stream));
  } else if (graphable && h->graph_runs >= 1) {
    cudaGraph_t g = nullptr;
    if (h->graph) { cudaGraphExecDestroy(h->graph); h->graph = nullptr; }  // captured for another row stride
    h->graph_stride = dstride;
    SWM_CK(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    rc = swm_orb_extract_batch_device(h, h->d_img, 1, w, h_px, dstride, (size_t)dstride * h_px, h->d_kps,
                                      h->d_desc, kcap, h->d_n, h->stream);
    const cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
    if (rc != SWM_OK) { if (g) cudaGraphDestroy(g); return rc; }
    SWM_CK(h, ce);
    const cudaError_t ie = cudaGraphInstantiate(&h->graph, g, 0);
    cudaGraphDestroy(g);
    SWM_CK(h, ie);
    SWM_CK(h, cudaGraphLaunch(h->graph, h->stream));
  } else {
    rc = swm_orb_extract_batch_device(h, h->d_img, nb, w, h_px, dstride, (size_t)dstride * h_px, h->d_kps,
                                      h->d_desc, kcap, h->d_n, h->stream);
    if (rc != SWM_OK) return rc;
  }
  if (nb == 1) h->graph_runs++;
  // A cudaMemcpyAsync into pageable memory is a staged, blocking transfer per call; the one-frame operator() path
  // (std::vector / cv::Mat destinations) therefore goes through a pinned staging buffer: three back-to-back async
  // copies, one synchronisation, then plain memcpy of the n valid entries.
  bool staged = false;
  if (nb == 1) {
    cudaPointerAttributes pa;
    const bool pageable = cudaPointerGetAttributes(&pa, kps) != cudaSuccess || pa.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if (pageable) {
      const size_t off_k = 64, off_d = off_k + (((size_t)ccap * sizeof(swm_keypoint) + 63) & ~(size_t)63);
      const size_t need = off_d + (size_t)ccap * 32;
      if (need > h->stage_cap) {
        if (h->h_stage) cudaFreeHost(h->h_stage);
        h->h_stage = nullptr;
        h->stage_cap = 0;
        SWM_CK(h, cudaMallocHost(&h->h_stage, need + need / 2));
        h->stage_cap = need + need / 2;
      }
      SWM_CK(h, cudaMemcpyAsync(h->h_stage, h->d_n, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
      SWM_CK(h, cudaMemcpyAsync(h->h_stage + off_k, h->d_kps, (size_t)ccap * sizeof(swm_keypoint), cudaMemcpyDeviceToHost, h->stream));
      SWM_CK(h, cudaMemcpyAsync(h->h_stage + off_d, h->d_desc, (size_t)ccap * 32, cudaMemcpyDeviceToHost, h->stream));
      h->stage_kps = kps;
      h->stage_desc = desc;
      h->stage_ccap = ccap;
      staged = true;
    }
  }
  if (staged) {
    h->pending_n = n;
    h->pending_batch = 1;
    h->pending_cap = cap;
    return SWM_OK;
  }
  SWM_CK(h, cudaMemcpyAsync(n, h->d_n, nb * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  if (cap == kcap) {
    SWM_CK(h, cudaMemcpyAsync(kps, h->d_kps, (size_t)kcap * nb * sizeof(swm_keypoint), cudaMemcpyDeviceToHost, h->stream));
    SWM_CK(h, cudaMemcpyAsync(desc, h->d_desc, (size_t)kcap * nb * 32, cudaMemcpyDeviceToHost, h->stream));
  } else {
    SWM_CK(h, cudaMemcpy2DAsync(kps, (size_t)cap * sizeof(swm_keypoint), h->d_kps, (size_t)kcap * sizeof(swm_keypoint),
                                (size_t)ccap * sizeof(swm_keypoint), nb, cudaMemcpyDeviceToHost, h->stream));
    SWM_CK(h, cudaMemcpy2DAsync(desc, (size_t)cap * 32, h->d_desc, (size_t)kcap * 32, (size_t)ccap * 32, nb,
                                cudaMemcpyDeviceToHost, h->stream));
  }
  h->pending_n = n;
  h->pending_batch = nb;
  h->pending_cap = cap;
  return SWM_OK;
}

int swm_orb_sync(swm_orb* h) {
  if (!h) return SWM_E_INVALID;
  SWM_CK(h, cudaSetDevice(h->device));
  SWM_CK(h, cudaStreamSynchronize(h->stream));
  if (h->pending_n && h->stage_kps) {  // staged single-frame result -> caller's arrays
    int32_t cnt;
    memcpy(&cnt, h->h_stage, sizeof(cnt));
    h->pending_n[0] = cnt;
    const size_t take = (size_t)std::max(0, std::min(cnt, h->stage_ccap));
    const size_t off_k = 64, off_d = off_k + (((size_t)h->stage_ccap * sizeof(swm_keypoint) + 63) & ~(size_t)63);
    memcpy(h->stage_kps, h->h_stage + off_k, take * sizeof(swm_keypoint));
    memcpy(h->stage_desc, h->h_stage + off_d, take * 32);
    h->stage_kps = nullptr;
    h->stage_desc = nullptr;
  }
  if (h->pending_n) {
    for (int f = 0; f < h->pending_batch; f++)
      if (h->pending_n[f] > h->pending_cap) h->pending_n[f] = h->pending_cap;
    h->pending_n = nullptr;
  }
  return SWM_OK;
}

int swm_orb_extract_batch_async(swm_orb* h, const uint8_t* imgs, int batch, int w, int h_px, int stride,
                                size_t frame_stride, swm_keypoint* kps, uint8_t* desc, int cap, int32_t* n) {
  if (!h) return SWM_E_INVALID;
  if (batch < 1 || !imgs || !kps || !desc || !n || cap < 1 || w <= 0 || h_px <= 0 || stride < w) {
    h->err = "bad argument";
    return SWM_E_INVALID;
  }
  if (batch > h->cfg.max_batch) { h->err = "batch exceeds cfg.max_batch"; return SWM_E_CAPACITY; }
  if (h->pending_n) { h->err = "previous async batch not synchronised"; return SWM_E_STATE; }
  SWM_CK(h, cudaSetDevice(h->device));
  int rc = setup_geometry(h, w, h_px);
  if (rc != SWM_OK) return rc;
  return enqueue_host_chunk(h, imgs, batch, w, h_px, stride, frame_stride, kps, desc, cap, n);
}

int swm_orb_extract_batch(swm_orb* h, const uint8_t* imgs, int batch, int w, int h_px, int stride,
                          size_t frame_stride, swm_keypoint* kps, uint8_t* desc, int cap, int32_t* n) {
  if (!h) return SWM_E_INVALID;
  if (batch < 0 || !kps || !desc || !n || cap < 1) { h->err = "bad argument"; return SWM_E_INVALID; }
  if (batch == 0) return SWM_OK;
  if (!imgs || w <= 0 || h_px <= 0) {  // empty image: silent return (ORBextractor.cc:750-751)
    for (int f = 0; f < batch; f++) n[f] = 0;
    return SWM_OK;
  }
  if (stride < w) { h->err = "stride < width"; return SWM_E_INVALID; }
  if (h->pending_n) { h->err = "previous async batch not synchronised"; return SWM_E_STATE; }
  SWM_CK(h, cudaSetDevice(h->device));
  int rc = setup_geometry(h, w, h_px);
  if (rc != SWM_OK) return rc;
  const int B = h->cfg.max_batch;
  for (int f0 = 0; f0 < batch; f0 += B) {
    const int nb = batch - f0 < B ? batch - f0 : B;
    rc = enqueue_host_chunk(h, imgs + (size_t)f0 * frame_stride, nb, w, h_px, stride, frame_stride,
                            kps + (size_t)f0 * cap, desc + (size_t)f0 * cap * 32, cap, n + f0);
    if (rc != SWM_OK) return rc;
    rc = swm_orb_sync(h);
    if (rc != SWM_OK) return rc;
  }
  return SWM_OK;
}

int swm_orb_extract(swm_orb* h, const uint8_t* img, int w, int h_px, int stride, swm_keypoint* kps, uint8_t* desc,
                    int cap, int* n) {
  if (!h || !n) return SWM_E_INVALID;
  int32_t nn = 0;
  if (!img || w <= 0 || h_px <= 0) { *n = 0; return SWM_OK; }
  int rc = swm_orb_extract_batch(h, img, 1, w, h_px, stride, (size_t)stride * h_px, kps, desc, cap, &nn);
  *n = nn;
  return rc;
}

int swm_orb_stereo_match(swm_orb* left, swm_orb* right, float bf, float b, float* u_right, float* depth, int cap,
                         int batch) {
  if (!left || !right) return SWM_E_INVALID;
  swm_orb* h = left;
  if (!u_right || !depth || !(bf > 0) || !(b > 0) || batch < 1) { h->err = "bad argument"; return SWM_E_INVALID; }
  if (!left->last_kps || !right->last_kps || left->last_batch < 1) { h->err = "both extractors must hold an extracted batch"; return SWM_E_STATE; }
  if (left->device != right->device || left->last_batch != right->last_batch || left->lay.w != right->lay.w ||
      left->lay.h != right->lay.h || left->cfg.nlevels != right->cfg.nlevels || left->cfg.scale_factor != right->cfg.scale_factor) {
    h->err = "left and right extractor differ in device, batch, frame size or pyramid";
    return SWM_E_INVALID;
  }
  if (left->last_cap >= 65536 || right->last_cap >= 65536) { h->err = "more than 65535 keypoints per frame"; return SWM_E_CAPACITY; }
  const int B = left->last_batch, capl = left->last_cap;
  if (cap < capl) { h->err = "output capacity below the extractor's keypoint capacity"; return SWM_E_CAPACITY; }
  // The outputs hold `batch` rows and the results cover the resident batch: swm_orb_extract_batch splits a call into
  // chunks of cfg.max_batch frames and only the last chunk stays resident, so more rows than that cannot be filled.
  if (batch < B) {
    h->err = "output rows (" + std::to_string(batch) + ") below the extracted batch of " + std::to_string(B) + " frames";
    return SWM_E_CAPACITY;
  }
  if (batch > B) {
    h->err = "batch " + std::to_string(batch) + " exceeds the extracted batch of " + std::to_string(B) +
             " frames (only the last chunk of at most max_batch frames of an extract call stays resident)";
    return SWM_E_INVALID;
  }
  SWM_CK(h, cudaSetDevice(h->device));
  const size_t need = (size_t)B * capl;
  if (need > h->stereo_cap) {
    cudaFree(h->d_uright); cudaFree(h->d_depth); cudaFree(h->d_sad);
    h->d_uright = h->d_depth = nullptr; h->d_sad = nullptr; h->stereo_cap = 0;
    const size_t want = std::max(need, (size_t)h->cfg.max_batch * capl);
    SWM_CK(h, cudaMalloc(&h->d_uright, want * 4));
    SWM_CK(h, cudaMalloc(&h->d_depth, want * 4));
    SWM_CK(h, cudaMalloc(&h->d_sad, want * 4));
    h->stereo_cap = want;
  }
  if (!h->stereo_ev) SWM_CK(h, cudaEventCreateWithFlags(&h->stereo_ev, cudaEventDisableTiming));
  cudaStream_t st = left->last_stream;
  if (right->last_stream != st) {  // the right view's batch may still be in flight on its own stream
    SWM_CK(h, cudaEventRecord(h->stereo_ev, right->last_stream));
    SWM_CK(h, cudaStreamWaitEvent(st, h->stereo_ev, 0));
  }
  StereoArgs a;
  a.L = left->d_lay;
  a.kl = left->last_kps; a.dl = left->last_desc; a.nl = left->last_n;
  a.kr = right->last_kps; a.dr = right->last_desc; a.nr = right->last_n;
  a.cap_l = capl; a.cap_r = right->last_cap;
  a.plain_l = left->d_plain; a.plain_r = right->d_plain;
  a.blur_l = left->d_blur; a.blur_r = right->d_blur;
  for (int i = 0; i < SWM_MAX_LEVELS; i++) {
    a.sf[i] = i < left->cfg.nlevels ? left->sf[i] : 1.0f;
    a.inv_sf[i] = i < left->cfg.nlevels ? left->inv_sf[i] : 1.0f;
  }
  a.mbf = bf; a.mb = b;
  a.u_right = h->d_uright; a.depth = h->d_depth; a.sad = h->d_sad;
  stereo_match_kernel<<<dim3((capl + 7) / 8, B), 256, 0, st>>>(a);
  stereo_filter_kernel<<<B, 1024, 0, st>>>(left->last_n, capl, h->d_uright, h->d_depth, h->d_sad);
  SWM_CK(h, cudaGetLastError());
  SWM_CK(h, cudaMemcpy2DAsync(u_right, (size_t)cap * 4, h->d_uright, (size_t)capl * 4, (size_t)capl * 4, B, cudaMemcpyDeviceToHost, st));
  SWM_CK(h, cudaMemcpy2DAsync(depth, (size_t)cap * 4, h->d_depth, (size_t)capl * 4, (size_t)capl * 4, B, cudaMemcpyDeviceToHost, st));
  SWM_CK(h, cudaStreamSynchronize(st));
  return SWM_OK;
}

int swm_orb_run_stage(swm_orb* h, int stage_mask, int batch, void* stream) {
  if (!h) return SWM_E_INVALID;
  if (!h->allocated || !h->last_img) { h->err = "run_stage before extract"; return SWM_E_STATE; }
  if (batch < 1 || batch > h->last_batch) { h->err = "bad batch"; return SWM_E_INVALID; }
  SWM_CK(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  return enqueue(h, stage_mask, h->last_img, batch, h->last_stride, h->last_frame_stride, h->last_kps, h->last_desc,
                 h->last_cap, h->last_n, st);
}

int swm_orb_level_ptr(swm_orb* h, int frame, int level, int which, const uint8_t** dev, int* w, int* h_px, int* pitch) {
  if (!h || !dev) return SWM_E_INVALID;
  if (!h->allocated) { h->err = "level_ptr before the first extract"; return SWM_E_STATE; }
  if (frame < 0 || frame >= h->cfg.max_batch || level < 0 || level >= h->lay.nlevels || which < 0 || which > 1) {
    h->err = "bad frame/level/which";
    return SWM_E_INVALID;
  }
  const LevelGeom& g = h->lay.lv[level];
  const uint8_t* base = which == 0 ? h->d_plain : h->d_blur;
  *dev = base + (size_t)frame * h->lay.slab_bytes + g.plane_off + (size_t)kEdge * g.pitch + kPadX;
  if (w) *w = g.w;
  if (h_px) *h_px = g.h;
  if (pitch) *pitch = g.pitch;
  return SWM_OK;
}

int swm_orb_scale_tables(const swm_orb* h, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2) {
  if (!h) return SWM_E_INVALID;
  for (int i = 0; i < h->cfg.nlevels; i++) {
    if (scale) scale[i] = h->sf[i];
    if (inv_scale) inv_scale[i] = h->inv_sf[i];
    if (sigma2) sigma2[i] = h->sig2[i];
    if (inv_sigma2) inv_sigma2[i] = h->inv_sig2[i];
  }
  return SWM_OK;
}

int swm_orb_level_quotas(const swm_orb* h, int32_t* quotas) {
  if (!h || !quotas) return SWM_E_INVALID;
  for (int i = 0; i < h->cfg.nlevels; i++) quotas[i] = h->quota[i];
  return SWM_OK;
}

int swm_orb_max_keypoints(const swm_orb* h) {
  if (!h) return SWM_E_INVALID;
  if (h->allocated) return h->max_kp;
  int m = 0;  // before the first frame n_ini is unknown: assume the worst aspect ratio allowed
  for (int l = 0; l < h->cfg.nlevels; l++) m += std::max(h->quota[l] + 3, 4 * kOtMaxIni) + 1;
  return m;
}

int swm_orb_last_launches(const swm_orb* h) { return h ? h->last_launches : SWM_E_INVALID; }

int swm_orb_set_debug(swm_orb* h, int keep_score_map) {
  if (!h) return SWM_E_INVALID;
  if (h->allocated) { h->err = "set_debug must precede the first extract"; return SWM_E_STATE; }
  h->debug_score = keep_score_map != 0;
  return SWM_OK;
}

int swm_orb_debug_plane(swm_orb* h, int frame, int level, int which, uint8_t* out, int out_stride) {
  if (!h || !out) return SWM_E_INVALID;
  if (!h->allocated) { h->err = "debug_plane before extract"; return SWM_E_STATE; }
  if (frame < 0 || frame >= h->cfg.max_batch || level < 0 || level >= h->lay.nlevels) return SWM_E_INVALID;
  const LevelGeom& g = h->lay.lv[level];
  SWM_CK(h, cudaSetDevice(h->device));
  SWM_CK(h, cudaStreamSynchronize(h->stream));
  const size_t fo = (size_t)frame * h->lay.slab_bytes + g.plane_off;
  if (which == 0) {
    SWM_CK(h, cudaMemcpy2D(out, out_stride, h->d_plain + fo + (kPadX - kEdge), g.pitch, g.w + 2 * kEdge, g.rows,
                           cudaMemcpyDeviceToHost));
  } else if (which == 1 || which == 2) {
    if (which == 2 && !h->d_score) { h->err = "score map not kept: call swm_orb_set_debug(h, 1) before the first extract"; return SWM_E_STATE; }
    const uint8_t* base = which == 1 ? h->d_blur : h->d_score;
    SWM_CK(h, cudaMemcpy2D(out, out_stride, base + fo + (size_t)kEdge * g.pitch + kPadX, g.pitch, g.w, g.h,
                           cudaMemcpyDeviceToHost));
  } else {
    return SWM_E_INVALID;
  }
  return SWM_OK;
}

int swm_orb_debug_points(swm_orb* h, int frame, int level, int which, int32_t* xys, int cap) {
  if (!h || !xys) return SWM_E_INVALID;
  if (!h->allocated) { h->err = "debug_points before extract"; return SWM_E_STATE; }
  if (frame < 0 || frame >= h->cfg.max_batch || level < 0 || level >= h->lay.nlevels || which < 0 || which > 1)
    return SWM_E_INVALID;
  const LevelGeom& g = h->lay.lv[level];
  const int nl = h->lay.nlevels;
  SWM_CK(h, cudaSetDevice(h->device));
  SWM_CK(h, cudaStreamSynchronize(h->stream));
  int count = 0;
  const int* d_count = h->d_counts + (which ? (size_t)h->cfg.max_batch * nl : 0) + (size_t)frame * nl + level;
  SWM_CK(h, cudaMemcpy(&count, d_count, sizeof(int), cudaMemcpyDeviceToHost));
  const int lim = which ? g.sel_cap : g.cand_cap;
  if (count > lim) count = lim;
  std::vector<uint32_t> buf(count);
  const uint32_t* d_src = which ? h->d_sel + (size_t)frame * h->lay.sel_total + g.sel_off
                                : h->d_cand + (size_t)frame * h->lay.cand_total + g.cand_off;
  if (count) SWM_CK(h, cudaMemcpy(buf.data(), d_src, (size_t)count * 4, cudaMemcpyDeviceToHost));
  const int m = count < cap ? count : cap;
  for (int i = 0; i < m; i++) {
    xys[3 * i] = (int)((buf[i] >> 8) & 0xFFF);
    xys[3 * i + 1] = (int)(buf[i] >> 20);
    xys[3 * i + 2] = (int)(buf[i] & 0xFF);
  }
  return count;
}

}  // extern "C"

namespace swm {
int orb_device_view(swm_orb* h, OrbDeviceView* out) {
  if (!h || !out) return SWM_E_INVALID;
  if (!h->last_kps || h->last_batch < 1) { h->err = "no extracted batch is resident"; return SWM_E_STATE; }
  out->kps = h->last_kps;
  out->desc = h->last_desc;
  out->n = h->last_n;
  out->cap = h->last_cap;
  out->batch = h->last_batch;
  out->device = h->device;
  out->stream = h->last_stream;
  return SWM_OK;
}
}  // namespace swm

