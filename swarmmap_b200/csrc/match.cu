// match.cu -- B200 (sm_100a) Hamming matchers behind the ORBmatcher API (include/swm_orb.h).
//
// Reference behaviour restated (paths relative to /root/reference/code/):
//   ORBmatcher::DescriptorDistance        src/ORBmatcher.cc:1511-1525
//   ORBmatcher::SearchForInitialization   src/ORBmatcher.cc:375-479
//   ORBmatcher::SearchByProjection x4     src/ORBmatcher.cc:44-121, 264-373, 1223-1354, 1356-1473
//   ORBmatcher::SearchByBoW x2            src/ORBmatcher.cc:150-262, 481-597
//   ComputeThreeMaxima                    src/ORBmatcher.cc:1475-1506
//   Frame grid                            src/Frame.cc:277-292 (AssignFeaturesToGrid), :377-442
//
// Structure: every Search* is "for each source in order: enumerate candidates in a fixed order,
// take best / second best Hamming distance among candidates that are still free, accept under a
// threshold + ratio rule, mutate the free-state".  The enumeration and all distances are
// embarrassingly parallel (one warp per source row, LOP3+POPC on the CUDA cores); only the greedy
// accept/steal state is order dependent, and that is replayed over the pre-computed candidate rows
// by resolve_kernel (speculative batches of 32 rows, in-order commit), which keeps match indices
// bit-exact.  The place-recognition shard scan uses the u8 tensor-core MMA (db_top2_mma_kernel).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <vector>

#include "swm_internal.cuh"
#include "db_umma.cuh"

namespace swm {

constexpr int kThLow = 50;      // ORBmatcher.cc:38
constexpr int kHistoLen = 30;   // ORBmatcher.cc:39
constexpr int kGridCols = SWM_GRID_COLS, kGridRows = SWM_GRID_ROWS, kCells = kGridCols * kGridRows;

__device__ __forceinline__ int ham256(const uint4 a0, const uint4 a1, const uint4* __restrict__ b) {
  const uint4 b0 = __ldg(b), b1 = __ldg(b + 1);
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
         __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// ---------------------------------------------------------------------------------------------
// DescriptorDistance in bulk
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) hamming_matrix_kernel(const uint4* __restrict__ a, int na,
                                                             const uint4* __restrict__ b, int nb,
                                                             uint16_t* __restrict__ out) {
  const int j = blockIdx.x * 32 + (threadIdx.x & 31);
  const int i0 = (blockIdx.y * 8 + (threadIdx.x >> 5)) * 4;
  if (j >= nb) return;
  const uint4 b0 = __ldg(b + 2 * j), b1 = __ldg(b + 2 * j + 1);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int i = i0 + k;
    if (i < na) out[(size_t)i * nb + j] = (uint16_t)ham256(b0, b1, a + 2 * i);
  }
}

__global__ void hamming_pairs_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, int n,
                                     int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = ham256(__ldg(a + 2 * i), __ldg(a + 2 * i + 1), b + 2 * i);
}

// ---------------------------------------------------------------------------------------------
// Frame grid (Frame.cc:277-292, PosInGrid :432-442 uses round()).  One CTA; cell lists keep
// ascending keypoint index, cell index = ix*48+iy so a column's cells are contiguous in `items`
// (GetFeaturesInArea's "for ix, for iy, for j" order = a few contiguous spans).
// ---------------------------------------------------------------------------------------------
struct FrameDev {
  int n;
  const float* x;
  const float* y;
  const int32_t* octave;
  const float* angle;
  const uint4* desc;
  float min_x, min_y, max_x, max_y, inv_w, inv_h;
  const int32_t* starts;  // kCells + 1
  const int32_t* items;
};

__device__ __forceinline__ void grid_build_body(const FrameDev& f, int32_t* __restrict__ starts,
                                                int32_t* __restrict__ items, int32_t* __restrict__ cell_of) {
  __shared__ int s_cnt[kCells + 1];
  __shared__ int s_part[1024];
  const int tid = threadIdx.x;
  for (int c = tid; c <= kCells; c += 1024) s_cnt[c] = 0;
  __syncthreads();
  for (int i = tid; i < f.n; i += 1024) {
    const int px = (int)roundf((f.x[i] - f.min_x) * f.inv_w);
    const int py = (int)roundf((f.y[i] - f.min_y) * f.inv_h);
    int cell = -1;
    if (px >= 0 && px < kGridCols && py >= 0 && py < kGridRows) {
      cell = px * kGridRows + py;
      atomicAdd(&s_cnt[cell], 1);
    }
    cell_of[i] = cell;
  }
  __syncthreads();
  // exclusive scan over 3072 cells: 3 per thread
  const int c0 = tid * 3;
  int local = 0;
  for (int k = 0; k < 3; k++) local += s_cnt[c0 + k];
  s_part[tid] = local;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int v = tid >= o ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int run = s_part[tid] - local;
  for (int k = 0; k < 3; k++) {
    const int v = s_cnt[c0 + k];
    starts[c0 + k] = run;
    s_cnt[c0 + k] = run;  // becomes the scatter cursor
    run += v;
  }
  if (tid == 1023) starts[kCells] = run;
  __syncthreads();
  for (int i = tid; i < f.n; i += 1024) {
    const int cell = cell_of[i];
    if (cell >= 0) items[atomicAdd(&s_cnt[cell], 1)] = i;
  }
  __syncthreads();
  // restore ascending index order inside each cell (insertion sort; cells hold a handful of items)
  for (int c = tid; c < kCells; c += 1024) {
    const int b = starts[c], e = s_cnt[c];
    for (int i = b + 1; i < e; i++) {
      const int v = items[i];
      int j = i - 1;
      while (j >= b && items[j] > v) {
        items[j + 1] = items[j];
        j--;
      }
      items[j + 1] = v;
    }
  }
}

__global__ void __launch_bounds__(1024) grid_build_kernel(FrameDev f, int32_t* __restrict__ starts,
                                                          int32_t* __restrict__ items, int32_t* __restrict__ cell_of) {
  grid_build_body(f, starts, items, cell_of);
}

// ---------------------------------------------------------------------------------------------
// Candidate rows by window query (Frame::GetFeaturesInArea, Frame.cc:377-430), one warp per
// source.  pass 0 counts, pass 1 writes (index, level<<16 | distance) in the reference's order.
// ---------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------
// Resident frames (SURVEY section 8(f) rank 1): Frame::UndistortKeyPoints (Frame.cc:454-484) + SoA split of the
// extractor's cv::KeyPoint records, so that extract -> grid -> match never leaves the GPU.
// cv::undistortPoints(pts, pts, K, D, Mat(), K): 5 fixed-point iterations in double (OpenCV's default criteria),
// float in/out; every operation is an explicit round-to-nearest intrinsic so that nothing is contracted into an
// FMA and the result is bit-identical to OpenCV's scalar code (and to oracle/orc_undistort_points).
// ---------------------------------------------------------------------------------------------
struct CameraDev {
  float fx, fy, cx, cy, k1, k2, p1, p2, k3;
  int distorted;  // mDistCoef.at<float>(0) != 0
};

__device__ __forceinline__ void undistort_point(const CameraDev& c, float px, float py, float* ox, float* oy) {
  const double fx = c.fx, fy = c.fy, cx = c.cx, cy = c.cy, k1 = c.k1, k2 = c.k2, p1 = c.p1, p2 = c.p2, k3 = c.k3;
  const double ifx = __ddiv_rn(1.0, fx), ify = __ddiv_rn(1.0, fy);
  const double u = px, v = py;
  double x = __dmul_rn(__dsub_rn(u, cx), ifx), y = __dmul_rn(__dsub_rn(v, cy), ify);
  const double x0 = x, y0 = y;
  for (int j = 0; j < 5; j++) {
    const double r2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
    const double poly = __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k3, r2), k2), r2), k1), r2);
    const double icdist = __ddiv_rn(1.0, __dadd_rn(1.0, poly));
    if (icdist < 0) {
      x = __dmul_rn(__dsub_rn(u, cx), ifx);
      y = __dmul_rn(__dsub_rn(v, cy), ify);
      break;
    }
    // deltaX = 2 p1 x y + p2 (r2 + 2 x x);  deltaY = p1 (r2 + 2 y y) + 2 p2 x y   (left to right)
    const double dx = __dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, p1), x), y),
                                __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, x), x))));
    const double dy = __dadd_rn(__dmul_rn(p1, __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, y), y))),
                                __dmul_rn(__dmul_rn(__dmul_rn(2.0, p2), x), y));
    x = __dmul_rn(__dsub_rn(x0, dx), icdist);
    y = __dmul_rn(__dsub_rn(y0, dy), icdist);
  }
  *ox = (float)__dadd_rn(__dmul_rn(fx, x), cx);
  *oy = (float)__dadd_rn(__dmul_rn(fy, y), cy);
}

__global__ void __launch_bounds__(256) frame_from_kps_kernel(const swm_keypoint* __restrict__ kps,
                                                             const uint4* __restrict__ desc_in, int n, CameraDev cam,
                                                             float* __restrict__ x, float* __restrict__ y,
                                                             int32_t* __restrict__ octave, float* __restrict__ angle,
                                                             uint4* __restrict__ desc_out) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const swm_keypoint kp = kps[i];
  float ux = kp.x, uy = kp.y;
  if (cam.distorted) undistort_point(cam, kp.x, kp.y, &ux, &uy);
  x[i] = ux;
  y[i] = uy;
  octave[i] = kp.octave;
  angle[i] = kp.angle;
  desc_out[2 * i] = desc_in[2 * i];
  desc_out[2 * i + 1] = desc_in[2 * i + 1];
}

__global__ void undistort_points_kernel(const float* __restrict__ in_xy, int n, CameraDev cam, float* __restrict__ out_xy) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float ux = in_xy[2 * i], uy = in_xy[2 * i + 1];
  if (cam.distorted) undistort_point(cam, ux, uy, &ux, &uy);
  out_xy[2 * i] = ux;
  out_xy[2 * i + 1] = uy;
}

// SearchForInitialization's source rows (ORBmatcher.cc:390-396): F1 keypoints of octave 0, window centre =
// vbPrevMatched, levels (0, 0).
__global__ void init_query_kernel(const int32_t* __restrict__ octave1, const float* __restrict__ prev_xy, int n1,
                                  float window, float* __restrict__ u, float* __restrict__ v, float* __restrict__ rad,
                                  int32_t* __restrict__ lv, uint8_t* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n1) return;
  u[i] = prev_xy[2 * i];
  v[i] = prev_xy[2 * i + 1];
  rad[i] = window;
  lv[i] = octave1[i];
  valid[i] = octave1[i] > 0 ? 0 : 1;
}

struct WindowDev {
  int m;
  const uint4* desc;
  const float* u;
  const float* v;
  const float* radius;
  const int32_t* min_level;
  const int32_t* max_level;
  const uint8_t* valid;
};

__device__ __forceinline__ void window_rows_body(const FrameDev& f, const WindowDev& q, int pass,
                                                 int32_t* __restrict__ row_count, const int32_t* __restrict__ row_start,
                                                 int32_t* __restrict__ cand_idx, uint32_t* __restrict__ cand_val) {
  const int s = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (s >= q.m) return;
  int total = 0;
  if (q.valid[s]) {
    const float x = q.u[s], y = q.v[s], r = q.radius[s];
    const int min_level = q.min_level[s], max_level = q.max_level[s];
    // Frame.cc:382-396
    const int min_cx = max(0, (int)floorf((x - f.min_x - r) * f.inv_w));
    const int max_cx = min(kGridCols - 1, (int)ceilf((x - f.min_x + r) * f.inv_w));
    const int min_cy = max(0, (int)floorf((y - f.min_y - r) * f.inv_h));
    const int max_cy = min(kGridRows - 1, (int)ceilf((y - f.min_y + r) * f.inv_h));
    if (min_cx < kGridCols && max_cx >= 0 && min_cy < kGridRows && max_cy >= 0) {
      const bool check_levels = (min_level > 0) || (max_level >= 0);
      uint4 d0 = make_uint4(0, 0, 0, 0), d1 = d0;
      int base = 0;
      if (pass) {
        d0 = __ldg(q.desc + 2 * s);
        d1 = __ldg(q.desc + 2 * s + 1);
        base = row_start[s];
      }
      for (int ix = min_cx; ix <= max_cx; ix++) {
        const int b = f.starts[ix * kGridRows + min_cy], e = f.starts[ix * kGridRows + max_cy + 1];
        for (int c0 = b; c0 < e; c0 += 32) {
          const int c = c0 + lane;
          bool ok = false;
          int j = 0, oct = 0;
          if (c < e) {
            j = f.items[c];
            oct = f.octave[j];
            ok = true;
            if (check_levels) {
              if (oct < min_level) ok = false;
              if (max_level >= 0 && oct > max_level) ok = false;
            }
            const float dx = f.x[j] - x, dy = f.y[j] - y;
            ok = ok && fabsf(dx) < r && fabsf(dy) < r;
          }
          const unsigned mask = __ballot_sync(0xffffffffu, ok);
          if (pass && ok) {
            const int pos = base + total + __popc(mask & ((1u << lane) - 1));
            cand_idx[pos] = j;
            cand_val[pos] = ((uint32_t)oct << 16) | (uint32_t)ham256(d0, d1, f.desc + 2 * j);
          }
          total += __popc(mask);
        }
      }
    }
  }
  if (!pass && lane == 0) row_count[s] = total;
}

__global__ void __launch_bounds__(256) window_rows_kernel(FrameDev f, WindowDev q, int pass,
                                                          int32_t* __restrict__ row_count,
                                                          const int32_t* __restrict__ row_start,
                                                          int32_t* __restrict__ cand_idx, uint32_t* __restrict__ cand_val) {
  window_rows_body(f, q, pass, row_count, row_start, cand_idx, cand_val);
}

// BoW rows: candidate indices come from the shared vocabulary nodes (host-built spans); fill distances.
__global__ void __launch_bounds__(256) list_rows_kernel(const uint4* __restrict__ desc1, const uint4* __restrict__ desc2,
                                                        const int32_t* __restrict__ octave2, int rows,
                                                        const int32_t* __restrict__ row_src,
                                                        const int32_t* __restrict__ row_start,
                                                        const int32_t* __restrict__ cand_idx,
                                                        uint32_t* __restrict__ cand_val) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const int s = row_src[r];
  const uint4 d0 = __ldg(desc1 + 2 * s), d1 = __ldg(desc1 + 2 * s + 1);
  for (int c = row_start[r] + lane; c < row_start[r + 1]; c += 32) {
    const int j = cand_idx[c];
    cand_val[c] = ((uint32_t)octave2[j] << 16) | (uint32_t)ham256(d0, d1, desc2 + 2 * j);
  }
}

// single-CTA exclusive scan of row counts -> row_start[0..m]
__global__ void __launch_bounds__(1024) scan_rows_kernel(const int32_t* __restrict__ count, int m,
                                                         int32_t* __restrict__ start) {
  __shared__ int s_part[1024];
  const int tid = threadIdx.x;
  const int per = (m + 1023) / 1024;
  const int b = tid * per, e = min(b + per, m);
  int local = 0;
  for (int i = b; i < e; i++) local += count[i];
  s_part[tid] = local;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int v = tid >= o ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int run = s_part[tid] - local;
  for (int i = b; i < e; i++) {
    start[i] = run;
    run += count[i];
  }
  if (tid == 1023) start[m] = s_part[1023];
}

// ---------------------------------------------------------------------------------------------
// Sequential resolve by one warp.
// ---------------------------------------------------------------------------------------------
enum ResolveMode { kModeInit = 0, kModeWindow = 1, kModeBowFrame = 2, kModeBowKf = 3 };

struct ResolveArgs {
  int mode;
  int rows;                 // rows to replay, in order
  const int32_t* row_src;   // row -> source index (NULL: identity)
  const uint8_t* row_valid; // per source (NULL: all valid)
  const int32_t* row_start;
  const int32_t* cand_idx;
  const uint32_t* cand_val;
  int32_t* row_list;        // scratch, `rows` entries: the valid, non-empty rows in order (built by the kernel)
  int n1, n2;
  const float* angle1;      // per source
  const float* angle2;      // per target
  const uint8_t* blocks;    // window mode: per source
  const uint8_t* valid2;    // BowKf: per target validity
  int th_dist;
  int ratio_mode;
  float nnratio;
  int check_ori;
  // state / outputs (global memory, single warp)
  uint8_t* blocked;         // n2 (pre-initialised by the host for window mode)
  int32_t* out;             // init: matches12[n1]; window: assignment[n2]; bowFrame: n2; bowKf: n1
  int32_t* ev_bin;          // per source: histogram bin of its accepted match (-1 none)
  int32_t* ev_tgt;          // per source: index stored in rotHist (what gets pruned)
  float* prev_xy;           // init mode: vbPrevMatched
  const float* x2;
  const float* y2;
  int32_t* nmatches;
};

// rot = a1 - a2; if (rot < 0) rot += 360; bin = round(rot * (1/30)); if (bin == 30) bin = 0
__device__ __forceinline__ int rot_bin(float a1, float a2) {
  const float factor = 1.0f / kHistoLen;
  float rot = __fsub_rn(a1, a2);
  if (rot < 0.0f) rot = __fadd_rn(rot, 360.0f);
  int bin = (int)roundf(__fmul_rn(rot, factor));
  if (bin == kHistoLen) bin = 0;
  return bin;
}

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w < v ? w : v;
  }
  return v;
}

// The greedy state a row reads: "is candidate j still available" (per mode).
__device__ __forceinline__ bool cand_skip(const ResolveArgs& a, const int* matched_dist, const uint8_t* blocked, int j,
                                          unsigned dist) {
  if (a.mode == kModeInit) return matched_dist[j] <= (int)dist;       // :414-415
  if (a.mode == kModeBowKf) return blocked[j] || !a.valid2[j];        // :531-535
  return blocked[j] != 0;                                             // :67-69,:196-197,:306,:1291,:1413
}

// Replays the reference's greedy loop.  Within a call the state only ever REMOVES candidates
// (blocked[] gets set, vMatchedDistance[] only decreases), and removing candidate t changes a row's
// outcome only if t is that row's best or (when a ratio test is used) second-best candidate.  So the
// block evaluates a batch of consecutive rows speculatively (one warp per row, against the state at
// batch start), marks the target each accepted row takes, and commits rows in order up to the first
// row whose best / second-best target is taken by an earlier row of the batch; that row starts the
// next batch.  Every committed row decided exactly as the serial loop would: indices stay bit-exact.
constexpr int kResolveWarps = 32;

__device__ __forceinline__ void resolve_body(const ResolveArgs& a) {
  extern __shared__ __align__(16) uint8_t dsm[];
  __shared__ int s_row[kResolveWarps], s_accept[kResolveWarps], s_best_idx[kResolveWarps], s_best_dist[kResolveWarps];
  __shared__ int s_second_idx[kResolveWarps];
  __shared__ int s_rb[kResolveWarps], s_re[kResolveWarps];  // candidate span of each row of the batch
  __shared__ int s_src[kResolveWarps], s_blk[kResolveWarps];
  __shared__ int s_cursor, s_nmatches, s_batches, s_nlist;
  __shared__ int s_wsum[kResolveWarps];
  __shared__ int s_hist[kHistoLen];
  __shared__ int s_keep[3];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned long long kNone = ~0ull;
  const int n2 = a.n2;
  // greedy state lives in shared memory
  int* matched_dist = reinterpret_cast<int*>(dsm);
  int* matches21 = matched_dist + (a.mode == kModeInit ? n2 : 0);
  uint8_t* blocked = reinterpret_cast<uint8_t*>(matches21 + (a.mode == kModeInit ? n2 : 0));
  int* mark = reinterpret_cast<int*>(blocked + ((n2 + 3) & ~3));
  for (int j = tid; j < n2; j += blockDim.x) {
    if (a.mode == kModeInit) {
      matched_dist[j] = 0x7FFFFFFF;
      matches21[j] = -1;
    }
    blocked[j] = a.mode == kModeInit ? 0 : a.blocked[j];
    mark[j] = 0x7FFFFFFF;
  }
  if (tid == 0) {
    s_cursor = 0;
    s_nmatches = 0;
    s_batches = 0;
    s_nlist = 0;
  }
  __syncthreads();

  // ---- 0. the valid, non-empty rows in order, compacted once: a batch is then 32 consecutive list entries and the
  // commit step can assemble the next batch from registers (no dependent global loads between batches)
  for (int r0 = 0; r0 < a.rows; r0 += blockDim.x) {
    const int r = r0 + tid;
    bool ok = false;
    if (r < a.rows) {
      const int s = a.row_src ? a.row_src[r] : r;
      ok = (!a.row_valid || a.row_valid[s]) && a.row_start[r] != a.row_start[r + 1];
    }
    const unsigned bm = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) s_wsum[wid] = __popc(bm);
    __syncthreads();
    int off = s_nlist;
    for (int w = 0; w < wid; w++) off += s_wsum[w];
    if (ok) a.row_list[off + __popc(bm & ((1u << lane) - 1))] = r;
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < kResolveWarps; w++) tot += s_wsum[w];
      s_nlist += tot;
    }
    __syncthreads();
  }
  const int n_list = s_nlist;
  __threadfence_block();
  if (wid == 0) {
    const int r = lane < n_list ? a.row_list[lane] : -1;
    s_row[lane] = r;
    s_rb[lane] = r >= 0 ? a.row_start[r] : 0;
    s_re[lane] = r >= 0 ? a.row_start[r + 1] : 0;
  }
  __syncthreads();

  while (true) {
    const int cursor = s_cursor;
    const int nb = min(kResolveWarps, n_list - cursor);
    if (nb <= 0) break;
    // the 32 list entries after this batch, fetched by warp 0 while the batch is evaluated (used by the commit
    // step to assemble the next batch)
    int pre = -1, pre_b = 0, pre_e = 0;
    if (wid == 0 && cursor + kResolveWarps + lane < n_list) {
      pre = a.row_list[cursor + kResolveWarps + lane];
      pre_b = a.row_start[pre];
      pre_e = a.row_start[pre + 1];
    }

    // ---- 1. speculative evaluation, one warp per row
    if (wid < nb) {
      int b, e, best_pos = -1;
      const int r = s_row[wid];
      b = s_rb[wid];
      e = s_re[wid];
      const bool small = e - b <= 32;  // the common case: one candidate per lane, loaded once
      // what the in-order commit needs from global memory, requested before the candidate scan (uniform address)
      const int src_s = a.row_src ? a.row_src[r] : r;
      const int src_blk = a.mode == kModeWindow ? a.blocks[src_s] : 1;
      int rj = 0;
      uint32_t rval = 0;
      bool rok = false;
      unsigned long long best = kNone;  // key = dist << 32 | position: smallest distance, first in enumeration order
      if (small) {
        if (b + lane < e) {
          rj = a.cand_idx[b + lane];
          rval = a.cand_val[b + lane];
          rok = !cand_skip(a, matched_dist, blocked, rj, rval & 0xFFFFu);
        }
        // one hardware warp reduction on a 32-bit key (distance << 8 | lane) instead of ten shuffles
        const unsigned k32 = __reduce_min_sync(0xffffffffu, rok ? (((rval & 0xFFFFu) << 8) | (unsigned)lane) : 0xFFFFFFFFu);
        if (k32 != 0xFFFFFFFFu) best = ((unsigned long long)(k32 >> 8) << 32) | (k32 & 31u);
      } else {
        for (int c = b + lane; c < e; c += 32) {
          const int j = a.cand_idx[c];
          const unsigned dist = a.cand_val[c] & 0xFFFFu;
          if (!cand_skip(a, matched_dist, blocked, j, dist)) {
            const unsigned long long key = ((unsigned long long)dist << 32) | (unsigned)(c - b);
            best = key < best ? key : best;
          }
        }
        best = warp_min_u64(best);
      }
      bool accept = false;
      int best_idx = -1, best_dist = 0, second_idx = -1;
      if (best != kNone) {
        best_pos = (int)(best & 0xFFFFFFFFu);
        best_dist = (int)(best >> 32);
        best_idx = small ? __shfl_sync(0xffffffffu, rj, best_pos) : a.cand_idx[b + best_pos];
        const bool need_second = !(a.mode == kModeWindow && a.ratio_mode == 0);
        int second_dist = a.mode == kModeInit ? 0x7FFFFFFF : 256, second_level = -1;  // INT_MAX (:404) vs 256 (:57,:190)
        if (need_second) {
          // second best: P = first minimum before the winner, Q = first minimum after it; the running
          // "bestDist2" of the reference ends as P if P <= Q else Q (see DESIGN.md, matcher section).
          unsigned long long p = kNone, q = kNone;
          if (small) {
            const unsigned kk = (rok && lane != best_pos) ? (((rval & 0xFFFFu) << 8) | (unsigned)lane) : 0xFFFFFFFFu;
            const unsigned p32 = __reduce_min_sync(0xffffffffu, lane < best_pos ? kk : 0xFFFFFFFFu);
            const unsigned q32 = __reduce_min_sync(0xffffffffu, lane > best_pos ? kk : 0xFFFFFFFFu);
            if (p32 != 0xFFFFFFFFu) p = ((unsigned long long)(p32 >> 8) << 32) | (p32 & 31u);
            if (q32 != 0xFFFFFFFFu) q = ((unsigned long long)(q32 >> 8) << 32) | (q32 & 31u);
          } else {
            for (int c = b + lane; c < e; c += 32) {
              if (c - b == best_pos) continue;
              const int j = a.cand_idx[c];
              const unsigned dist = a.cand_val[c] & 0xFFFFu;
              if (!cand_skip(a, matched_dist, blocked, j, dist)) {
                const unsigned long long key = ((unsigned long long)dist << 32) | (unsigned)(c - b);
                if (c - b < best_pos) p = key < p ? key : p;
                else q = key < q ? key : q;
              }
            }
            p = warp_min_u64(p);
            q = warp_min_u64(q);
          }
          const unsigned long long sec = (p >> 32) <= (q >> 32) ? p : q;
          if (sec != kNone) {
            const int sp = (int)(sec & 0xFFFFFFFFu);
            second_dist = (int)(sec >> 32);
            second_level = (int)((small ? __shfl_sync(0xffffffffu, rval, sp) : a.cand_val[b + sp]) >> 16);
            second_idx = small ? __shfl_sync(0xffffffffu, rj, sp) : a.cand_idx[b + sp];
          }
        }
        const int best_level = (int)((small ? __shfl_sync(0xffffffffu, rval, best_pos) : a.cand_val[b + best_pos]) >> 16);
        if (a.mode == kModeInit) {
          accept = best_dist <= kThLow && (float)best_dist < __fmul_rn((float)second_dist, a.nnratio);  // :426-427
        } else if (a.mode == kModeWindow) {
          accept = best_dist <= a.th_dist;                                                             // :111,:365,:1316,:1428
          if (accept && a.ratio_mode == 1 && best_level == second_level &&
              (float)best_dist > __fmul_rn(a.nnratio, (float)second_dist))                             // :112
            accept = false;
        } else if (a.mode == kModeBowFrame) {
          accept = best_dist <= kThLow && (float)best_dist < __fmul_rn(a.nnratio, (float)second_dist);  // :212-213
        } else {
          accept = best_dist < kThLow && (float)best_dist < __fmul_rn(a.nnratio, (float)second_dist);   // :550-551
        }
      }
      if (lane == 0) {
        s_accept[wid] = accept;
        s_best_idx[wid] = best_idx;
        s_best_dist[wid] = best_dist;
        s_second_idx[wid] = second_idx;
        // everything the in-order commit needs from global memory is fetched here, in parallel
        s_src[wid] = src_s;
        s_blk[wid] = (a.mode == kModeWindow && accept) ? src_blk : 1;
        if (accept) atomicMin(mark + best_idx, wid);
      }
    }
    if (wid == 0 && pre >= 0) {
      // warm L1 with the candidate lists of the rows that can enter the next batch (first and last line of each)
      asm volatile("prefetch.global.L1 [%0];" ::"l"(a.cand_idx + pre_b));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(a.cand_val + pre_b));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(a.cand_idx + pre_e - 1));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(a.cand_val + pre_e - 1));
    }
    __syncthreads();

    // ---- 3. commit, by the lanes of warp 0 (lane k = row k of the batch).  A row conflicts if an earlier
    // row of this batch removes its best (or, when a ratio test is in play, second-best) candidate; rows
    // before the first conflict touch pairwise different targets, so their commits are independent.
    if (wid == 0) {
      const bool uses_second = !(a.mode == kModeWindow && a.ratio_mode == 0);
      const int k = lane;
      bool conflict = false, acc = false;
      int bi = -1;
      if (k < nb) {
        bi = s_best_idx[k];
        const int si = s_second_idx[k];
        acc = s_accept[k] != 0;
        conflict = bi >= 0 && (uses_second || acc) && (mark[bi] < k || (si >= 0 && mark[si] < k));
      }
      const unsigned cm = __ballot_sync(0xffffffffu, conflict);
      const int first = cm ? __ffs(cm) - 1 : nb;
      int delta = 0;
      if (k < first && acc) {
        const int s = s_src[k];
        int ev_tgt = bi;
        if (a.mode == kModeInit) {
          const int prev_owner = matches21[bi];
          if (prev_owner >= 0) {  // steal (:428-431)
            a.out[prev_owner] = -1;
            delta--;
          }
          a.out[s] = bi;
          matches21[bi] = s;
          matched_dist[bi] = s_best_dist[k];
          ev_tgt = s;
        } else if (a.mode == kModeWindow) {
          a.out[bi] = s;
          if (s_blk[k]) blocked[bi] = 1;
        } else if (a.mode == kModeBowFrame) {
          a.out[bi] = s;
          blocked[bi] = 1;
        } else {
          a.out[s] = bi;
          blocked[bi] = 1;
          ev_tgt = s;
        }
        delta++;
        if (a.check_ori) {
          a.ev_bin[s] = bi;  // the partner; turned into its histogram bin after the loop (keeps two dependent
          a.ev_tgt[s] = ev_tgt;  // global loads out of every batch)
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) delta += __shfl_xor_sync(0xffffffffu, delta, o);
      __syncwarp();
      if (k < nb && acc) mark[bi] = 0x7FFFFFFF;
      // next batch = the uncommitted tail of this one followed by the prefetched list entries
      const int keep = first + lane;
      const bool old = keep < kResolveWarps;
      const int old_row = old ? s_row[keep] : -1, old_b = old ? s_rb[keep] : 0, old_e = old ? s_re[keep] : 0;
      const int src_lane = (lane - (kResolveWarps - first)) & 31;
      const int from_pre = __shfl_sync(0xffffffffu, pre, src_lane);
      const int from_b = __shfl_sync(0xffffffffu, pre_b, src_lane), from_e = __shfl_sync(0xffffffffu, pre_e, src_lane);
      __syncwarp();
      s_row[lane] = old ? old_row : from_pre;
      s_rb[lane] = old ? old_b : from_b;
      s_re[lane] = old ? old_e : from_e;
      if (lane == 0) {
        s_nmatches += delta;
        s_batches++;
        s_cursor = cursor + first;
      }
    }
    __syncthreads();
  }

  // ---- rotation-consistency pruning (e.g. :229-246): histogram of accepted events, keep the top three bins
  if (a.check_ori) {
    if (tid < kHistoLen) s_hist[tid] = 0;
    __syncthreads();
    for (int s = tid; s < a.n1; s += blockDim.x) {
      const int partner = a.ev_bin[s];
      if (partner >= 0) {
        const int bin = rot_bin(a.angle1[s], a.angle2[partner]);
        a.ev_bin[s] = bin;
        atomicAdd(&s_hist[bin], 1);
      }
    }
    __syncthreads();
    if (tid == 0) {  // ComputeThreeMaxima, :1475-1506
      int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
      for (int i = 0; i < kHistoLen; i++) {
        const int c = s_hist[i];
        if (c > max1) {
          max3 = max2; max2 = max1; max1 = c;
          ind3 = ind2; ind2 = ind1; ind1 = i;
        } else if (c > max2) {
          max3 = max2; max2 = c;
          ind3 = ind2; ind2 = i;
        } else if (c > max3) {
          max3 = c;
          ind3 = i;
        }
      }
      if ((float)max2 < 0.1f * (float)max1) {
        ind2 = -1;
        ind3 = -1;
      } else if ((float)max3 < 0.1f * (float)max1) {
        ind3 = -1;
      }
      s_keep[0] = ind1; s_keep[1] = ind2; s_keep[2] = ind3;
    }
    __syncthreads();
    int dropped = 0;
    for (int s = tid; s < a.n1; s += blockDim.x) {
      const int bin = a.ev_bin[s];
      if (bin < 0 || bin == s_keep[0] || bin == s_keep[1] || bin == s_keep[2]) continue;
      const int t = a.ev_tgt[s];
      if (a.mode == kModeInit) {
        if (a.out[t] >= 0) {  // :462-465 (only live matches are counted down)
          a.out[t] = -1;
          dropped++;
        }
      } else {
        a.out[t] = -1;  // idempotent store; every event counts down (:240-243,:1345-1348)
        dropped++;
      }
    }
    if (dropped) atomicSub(&s_nmatches, dropped);
  }
  __syncthreads();
  if (a.mode == kModeInit) {  // :474-476
    for (int s = tid; s < a.n1; s += blockDim.x) {
      const int j = a.out[s];
      if (j >= 0) {
        a.prev_xy[2 * s] = a.x2[j];
        a.prev_xy[2 * s + 1] = a.y2[j];
      }
    }
  }
  if (tid == 0) {
    a.nmatches[0] = s_nmatches;
    a.nmatches[1] = s_batches;  // diagnostics: speculative batches executed
  }
}

__global__ void __launch_bounds__(kResolveWarps * 32) resolve_kernel(ResolveArgs a) { resolve_body(a); }

// ---------------------------------------------------------------------------------------------
// SearchForTriangulation (ORBmatcher.cc:599-749, monocular) with CheckDistEpipolarLine (:131-148).  The reference
// never sets vbMatched2, so the rows are independent: warp per row, the winner is the candidate of smallest distance
// among those that pass the epipole and epipolar-line tests, the LAST one on ties ("dist > bestDist -> continue").
// Float expressions are evaluated left to right with explicit round-to-nearest operations (no FMA contraction).
// ---------------------------------------------------------------------------------------------
struct TriDev {
  float F[9];
  float ex, ey;
  const float* sf2;     // pKF2->mvScaleFactors
  const float* sigma2;  // pKF2->mvLevelSigma2
  int nlevels;          // entries in the two tables; candidates of a higher octave are skipped
};

__global__ void __launch_bounds__(256) tri_rows_kernel(FrameDev f1, FrameDev f2, const uint8_t* __restrict__ valid2, int rows,
                                                       const int32_t* __restrict__ row_src,
                                                       const int32_t* __restrict__ row_start,
                                                       const int32_t* __restrict__ cand_idx, TriDev t, int check_ori,
                                                       int32_t* __restrict__ out, int32_t* __restrict__ ev_bin) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const int s = row_src[r];
  const uint4 d0 = __ldg(f1.desc + 2 * s), d1 = __ldg(f1.desc + 2 * s + 1);
  const float x1 = f1.x[s], y1 = f1.y[s];
  // l = x1' F12 = [a b c]  (:134-136)
  const float a = __fadd_rn(__fadd_rn(__fmul_rn(x1, t.F[0]), __fmul_rn(y1, t.F[3])), t.F[6]);
  const float b = __fadd_rn(__fadd_rn(__fmul_rn(x1, t.F[1]), __fmul_rn(y1, t.F[4])), t.F[7]);
  const float c = __fadd_rn(__fadd_rn(__fmul_rn(x1, t.F[2]), __fmul_rn(y1, t.F[5])), t.F[8]);
  const float den = __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b));
  unsigned long long best = ~0ull;
  const int c0 = row_start[r];
  for (int ci = c0 + lane; ci < row_start[r + 1]; ci += 32) {
    const int j = cand_idx[ci];
    if (!valid2[j]) continue;  // pMP2 (:662-666)
    const int dist = ham256(d0, d1, f2.desc + 2 * j);
    if (dist > kThLow) continue;  // :674
    const float x2 = f2.x[j], y2 = f2.y[j];
    const int oct = f2.octave[j];
    if ((unsigned)oct >= (unsigned)t.nlevels) continue;                // outside the caller's tables
    const float dex = __fsub_rn(t.ex, x2), dey = __fsub_rn(t.ey, y2);  // :679-683
    if (__fadd_rn(__fmul_rn(dex, dex), __fmul_rn(dey, dey)) < __fmul_rn(100.0f, t.sf2[oct])) continue;
    const float num = __fadd_rn(__fadd_rn(__fmul_rn(a, x2), __fmul_rn(b, y2)), c);
    if (den == 0.0f) continue;
    const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
    if (!((double)dsqr < __dmul_rn(3.84, (double)t.sigma2[oct]))) continue;  // :147
    const unsigned long long key = ((unsigned long long)dist << 32) | (unsigned)(0x7FFFFFFF - (ci - c0));
    best = best < key ? best : key;
  }
  best = warp_min_u64(best);
  if (lane == 0) {
    int j = -1, bin = -1;
    if (best != ~0ull) {
      j = cand_idx[c0 + (0x7FFFFFFF - (int)(unsigned)best)];
      if (check_ori) bin = rot_bin(f1.angle[s], f2.angle[j]);
    }
    out[s] = j;
    ev_bin[s] = bin;
  }
}

// nmatches, rotation histogram, ComputeThreeMaxima, pruning (:724-738).  One CTA.
__global__ void __launch_bounds__(1024) tri_finalize_kernel(int n1, int32_t* __restrict__ out, const int32_t* __restrict__ ev_bin,
                                                            int check_ori, int32_t* __restrict__ nmatches) {
  __shared__ int s_hist[kHistoLen];
  __shared__ int s_keep[3];
  __shared__ int s_n;
  const int tid = threadIdx.x;
  if (tid < kHistoLen) s_hist[tid] = 0;
  if (tid == 0) s_n = 0;
  __syncthreads();
  int mine = 0;
  for (int s = tid; s < n1; s += 1024) {
    if (out[s] >= 0) mine++;
    if (check_ori && ev_bin[s] >= 0) atomicAdd(&s_hist[ev_bin[s]], 1);
  }
  if (mine) atomicAdd(&s_n, mine);
  __syncthreads();
  if (check_ori) {
    if (tid == 0) {  // ComputeThreeMaxima, :1475-1506
      int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
      for (int i = 0; i < kHistoLen; i++) {
        const int cnt = s_hist[i];
        if (cnt > max1) {
          max3 = max2; max2 = max1; max1 = cnt;
          ind3 = ind2; ind2 = ind1; ind1 = i;
        } else if (cnt > max2) {
          max3 = max2; max2 = cnt;
          ind3 = ind2; ind2 = i;
        } else if (cnt > max3) {
          max3 = cnt;
          ind3 = i;
        }
      }
      if ((float)max2 < 0.1f * (float)max1) {
        ind2 = -1;
        ind3 = -1;
      } else if ((float)max3 < 0.1f * (float)max1) {
        ind3 = -1;
      }
      s_keep[0] = ind1; s_keep[1] = ind2; s_keep[2] = ind3;
    }
    __syncthreads();
    int dropped = 0;
    for (int s = tid; s < n1; s += 1024) {
      const int bin = ev_bin[s];
      if (bin < 0 || bin == s_keep[0] || bin == s_keep[1] || bin == s_keep[2]) continue;
      out[s] = -1;
      dropped++;
    }
    if (dropped) atomicSub(&s_n, dropped);
    __syncthreads();
  }
  if (tid == 0) nmatches[0] = s_n;
}

// ---------------------------------------------------------------------------------------------
// Best keypoint inside a window, independent rows: the inner loop of ORBmatcher::Fuse (ORBmatcher.cc:824-870,
// :962-999) and SearchBySim3 (:1098-1134, :1178-1214).  Candidates come from window_rows_kernel in
// GetFeaturesInArea's order with the level filter applied; the optional monocular reprojection gate
// (e2 * mvInvLevelSigma2[level] > 5.99 -> skip, :857-864) is evaluated here; "dist < bestDist" = smallest distance,
// first candidate on ties.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) best_rows_kernel(FrameDev tgt, int rows, const float* __restrict__ u,
                                                        const float* __restrict__ v, const int32_t* __restrict__ row_start,
                                                        const int32_t* __restrict__ cand_idx,
                                                        const uint32_t* __restrict__ cand_val,
                                                        const float* __restrict__ inv_sigma2, int nlevels, float chi2,
                                                        int32_t* __restrict__ best_idx, int32_t* __restrict__ best_dist) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float pu = u[r], pv = v[r];
  const int c0 = row_start[r];
  unsigned long long best = ~0ull;
  for (int ci = c0 + lane; ci < row_start[r + 1]; ci += 32) {
    const int j = cand_idx[ci];
    const uint32_t val = cand_val[ci];
    if (chi2 > 0.0f) {
      if ((int)(val >> 16) >= nlevels) continue;  // outside the caller's mvInvLevelSigma2
      const float ex = __fsub_rn(pu, tgt.x[j]), ey = __fsub_rn(pv, tgt.y[j]);
      const float e2 = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
      if ((double)__fmul_rn(e2, inv_sigma2[val >> 16]) > (double)chi2) continue;
    }
    const unsigned long long key = ((unsigned long long)(val & 0xFFFFu) << 32) | (unsigned)(ci - c0);
    best = best < key ? best : key;
  }
  best = warp_min_u64(best);
  if (lane == 0) {
    best_idx[r] = best == ~0ull ? -1 : cand_idx[c0 + (int)(unsigned)best];
    best_dist[r] = best == ~0ull ? 256 : (int)(best >> 32);
  }
}

// ---------------------------------------------------------------------------------------------
// MapPoint::ComputeDistinctiveDescriptors (code/src/MapPoint.cc:361-391) for a batch of MapPoints: N x N Hamming
// distances between a point's observed descriptors, per row the median sorted[int(0.5 * (N - 1))], the row with the
// least median wins (first one on ties).  One CTA per point, descriptors in shared memory, thread per row; the
// order statistic is found by bisection on the distance value (count(d <= v) >= k + 1), so no sort is needed.
// ---------------------------------------------------------------------------------------------
constexpr int kDistinctMax = 1024;  // observations per MapPoint served by one CTA (32 KB of shared memory)

__global__ void __launch_bounds__(128) distinctive_kernel(const uint4* __restrict__ desc, const int32_t* __restrict__ offsets,
                                                          int32_t* __restrict__ best_idx, int32_t* __restrict__ best_median) {
  extern __shared__ __align__(16) uint4 s_desc[];
  __shared__ unsigned long long s_best[4];
  const int p = blockIdx.x, tid = threadIdx.x;
  const int o = offsets[p], N = offsets[p + 1] - o;
  if (N <= 0) {
    if (tid == 0) { best_idx[p] = -1; best_median[p] = -1; }
    return;
  }
  for (int i = tid; i < 2 * N; i += 128) s_desc[i] = __ldg(desc + 2 * (size_t)o + i);
  __syncthreads();
  const int k = (int)(0.5 * (N - 1));  // vDists[0.5 * (N - 1)]
  unsigned long long best = ~0ull;
  for (int i = tid; i < N; i += 128) {
    const uint4 a0 = s_desc[2 * i], a1 = s_desc[2 * i + 1];
    int lo = 0, hi = 256;  // smallest v with #{j : d(i, j) <= v} >= k + 1
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      int cnt = 0;
      for (int j = 0; j < N; j++) {  // shared-memory operands: plain loads (ham256 uses the read-only global path)
        const uint4 b0 = s_desc[2 * j], b1 = s_desc[2 * j + 1];
        const int d = __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
                      __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
        cnt += d <= mid;
      }
      if (cnt >= k + 1) hi = mid; else lo = mid + 1;
    }
    const unsigned long long key = ((unsigned long long)lo << 32) | (unsigned)i;  // median < BestMedian: first wins
    best = best < key ? best : key;
  }
  best = warp_min_u64(best);
  if ((tid & 31) == 0) s_best[tid >> 5] = best;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < 4; w++) best = best < s_best[w] ? best : s_best[w];
    best_idx[p] = (int)(unsigned)best;
    best_median[p] = (int)(best >> 32);
  }
}

// ---------------------------------------------------------------------------------------------
// Place-recognition shard (BASELINE config 5): brute-force top-2 of each query over the shard.
// Each thread owns one query (descriptor in registers); the CTA streams database tiles through
// shared memory (broadcast reads), keeping a running top-2 of packed keys dist<<48 | global index.
// Per-CTA partials are merged by a second kernel (deterministic: ties -> lower index).
// ---------------------------------------------------------------------------------------------
constexpr int kDbTile = 256;     // database descriptors per smem tile
constexpr int kDbQPerCta = 128;  // queries per CTA (one per thread)

__global__ void __launch_bounds__(kDbQPerCta) db_top2_kernel(const uint4* __restrict__ db, long long ndb,
                                                             long long first_index, const uint4* __restrict__ q, int nq,
                                                             int tiles_per_cta, unsigned long long* __restrict__ partial) {
  __shared__ uint4 s_db[kDbTile * 2];
  const int qi = blockIdx.y * kDbQPerCta + threadIdx.x;
  uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0;
  if (qi < nq) {
    q0 = __ldg(q + 2 * qi);
    q1 = __ldg(q + 2 * qi + 1);
  }
  unsigned long long k0 = ~0ull, k1 = ~0ull;
  const long long tile0 = (long long)blockIdx.x * tiles_per_cta;
  for (int t = 0; t < tiles_per_cta; t++) {
    const long long base = (tile0 + t) * kDbTile;
    if (base >= ndb) break;
    const int cnt = (int)min((long long)kDbTile, ndb - base);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * 2; i += kDbQPerCta) s_db[i] = __ldg(db + 2 * base + i);
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < cnt; j++) {
      const uint4 b0 = s_db[2 * j], b1 = s_db[2 * j + 1];
      const unsigned d = __popc(q0.x ^ b0.x) + __popc(q0.y ^ b0.y) + __popc(q0.z ^ b0.z) + __popc(q0.w ^ b0.w) +
                         __popc(q1.x ^ b1.x) + __popc(q1.y ^ b1.y) + __popc(q1.z ^ b1.z) + __popc(q1.w ^ b1.w);
      const unsigned long long key = ((unsigned long long)d << 48) | (unsigned long long)(first_index + base + j);
      if (key < k1) {
        if (key < k0) {
          k1 = k0;
          k0 = key;
        } else {
          k1 = key;
        }
      }
    }
  }
  if (qi < nq) {
    partial[((size_t)blockIdx.x * nq + qi) * 2] = k0;
    partial[((size_t)blockIdx.x * nq + qi) * 2 + 1] = k1;
  }
}

// ---------------------------------------------------------------------------------------------
// Tensor-core variant of the shard scan.  With descriptors expanded to 0/1 bytes,
//     hamming(q, d) = popc(q) + popc(d) - 2 * dot(q, d),
// and dot() over 256 dimensions is eight m16n8k32 u8 x u8 -> s32 MMAs per 16 x 8 block of pairs
// (north_star's "popc(a)+popc(b)-2*popc(a&b)" identity; the b1 AND/XOR-popc MMA it mentions is not native
// on sm_100a -- it compiles to IMMA plus bit expansion -- so the expansion is done once per CTA tile here).
// One warp owns 32 queries (A fragments for all 256 dimensions stay in 64 registers); the CTA streams the
// database in tiles of 128 descriptors, expanded to bytes in shared memory in fragment order (one 64-bit
// load per B fragment, row stride 288 B -> conflict-free).  Per thread a running top-2 of (dist << 20 | index in
// this CTA's slice) for its two query rows; quads are merged by shuffles at the end.  Output format and
// the cross-slice merge are those of the POPC kernel, results are identical (ties -> lower index).
// ---------------------------------------------------------------------------------------------
constexpr int kMmaTile = 128;          // database descriptors per smem tile
constexpr int kMmaRow = 288;           // bytes per expanded descriptor row: 36 x 8 B = 4 mod 16 -> 64-bit fragment loads are conflict-free
constexpr int kMmaQPerCta = 256;       // 8 warps x 32 queries

__device__ __forceinline__ uint32_t expand_nibble(uint32_t w, int shift) {
  return (((w >> shift) & 0xFu) * 0x00204081u) & 0x01010101u;  // 4 bits -> 4 bytes of 0/1
}

__device__ __forceinline__ void top2_insert(uint32_t key, uint32_t& k0, uint32_t& k1) {
  k1 = min(k1, max(k0, key));  // branch-free: second smallest of {k0, k1, key}
  k0 = min(k0, key);
}

__device__ __forceinline__ void mma_u8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(256, 2) db_top2_mma_kernel(const uint4* __restrict__ db, long long ndb, long long first_index,
                                                             const uint32_t* __restrict__ q, int nq, int tiles_per_cta,
                                                             unsigned long long* __restrict__ partial) {
  __shared__ __align__(16) uint8_t s_exp[kMmaTile * kMmaRow];
  __shared__ __align__(8) uint32_t s_cb[kMmaTile];  // per column: (popc + 256) << 20 | index in slice
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  // ---- A fragments: this warp's 32 queries = two 16-row blocks (rows g, g+8 of each), all 8 k-steps,
  // expanded from bits.  Every B fragment read from shared memory then feeds two MMAs (the kernel is
  // otherwise bound by shared-memory bandwidth: 256 B of B operand per MMA).
  const int qrow0 = blockIdx.y * kMmaQPerCta + wid * 32 + g;  // rows of this thread: qrow0 + 8 r, r = 0..3
  uint32_t a[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; mt++) {
    const int r0 = qrow0 + 16 * mt, r1 = r0 + 8;
#pragma unroll
    for (int ks = 0; ks < 8; ks++) {
      const uint32_t w0 = r0 < nq ? __ldg(q + (size_t)r0 * 8 + ks) : 0u;
      const uint32_t w1 = r1 < nq ? __ldg(q + (size_t)r1 * 8 + ks) : 0u;
      a[mt][ks][0] = expand_nibble(w0, 4 * t);
      a[mt][ks][1] = expand_nibble(w1, 4 * t);
      a[mt][ks][2] = expand_nibble(w0, 16 + 4 * t);
      a[mt][ks][3] = expand_nibble(w1, 16 + 4 * t);
    }
  }
  // running top-2 keys of the 4 rows.  Inside the scan a key is (popc(d) + 256 - 2 dot) << 20 | index: the
  // query's own popcount is the same for every column of a row, so it is added only when the key is widened.
  uint32_t k0[4] = {~0u, ~0u, ~0u, ~0u}, k1[4] = {~0u, ~0u, ~0u, ~0u};
  const long long tile0 = (long long)blockIdx.x * tiles_per_cta;
  // thread = (descriptor n of the tile, half of its 8 words); the next tile's bits are fetched into
  // registers before the MMA loop of the current one, so the DRAM latency is off the critical path
  const int xn = tid >> 1, xhalf = tid & 1;
  uint4 w_next = make_uint4(0, 0, 0, 0);
  if (tile0 * kMmaTile + xn < ndb) w_next = __ldg(db + 2 * (tile0 * kMmaTile + xn) + xhalf);
  for (int tile = 0; tile < tiles_per_cta; tile++) {
    const long long base = (tile0 + tile) * kMmaTile;
    if (base >= ndb) break;
    __syncthreads();
    {  // expand this tile to 0/1 bytes, in fragment order: k-step ks, lane t -> 8 bytes (b0 | b1) at 32 ks + 8 t
      const uint4 w = w_next;
      const bool live = base + xn < ndb;
      int pc = __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
      pc += __shfl_xor_sync(0xffffffffu, pc, 1);
      // padding rows can never win (dot = 0 and the key still fits 32 bits)
      if (xhalf == 0) s_cb[xn] = ((uint32_t)((live ? pc : 1000) + 256) << 20) | (uint32_t)(tile * kMmaTile + xn);
      uint4* dst = reinterpret_cast<uint4*>(s_exp + xn * kMmaRow + 128 * xhalf);
      const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        dst[2 * k] = make_uint4(expand_nibble(ww[k], 0), expand_nibble(ww[k], 16), expand_nibble(ww[k], 4), expand_nibble(ww[k], 20));
        dst[2 * k + 1] = make_uint4(expand_nibble(ww[k], 8), expand_nibble(ww[k], 24), expand_nibble(ww[k], 12), expand_nibble(ww[k], 28));
      }
      const long long nb = base + kMmaTile + xn;
      w_next = (tile + 1 < tiles_per_cta && nb < ndb) ? __ldg(db + 2 * nb + xhalf) : make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    for (int nt = 0; nt < kMmaTile / 8; nt += 2) {  // 2 column blocks x 2 row blocks per step: 4 independent MMAs
      int c[2][2][4] = {};
      const uint8_t* brow = s_exp + (nt * 8 + g) * kMmaRow + 8 * t;
      const uint8_t* drow = brow + 8 * kMmaRow;
#pragma unroll
      for (int ks = 0; ks < 8; ks++) {
        const uint2 b = *reinterpret_cast<const uint2*>(brow + 32 * ks);
        const uint2 e = *reinterpret_cast<const uint2*>(drow + 32 * ks);
        mma_u8(c[0][0], a[0][ks], b.x, b.y);
        mma_u8(c[0][1], a[0][ks], e.x, e.y);
        mma_u8(c[1][0], a[1][ks], b.x, b.y);
        mma_u8(c[1][1], a[1][ks], e.x, e.y);
      }
      // c[.][.][0]:(row g, col 2t) [1]:(row g, col 2t+1) [2]:(row g+8, col 2t) [3]:(row g+8, col 2t+1)
      const int n0 = nt * 8 + 2 * t;
      const uint2 cb[2] = {*reinterpret_cast<const uint2*>(s_cb + n0), *reinterpret_cast<const uint2*>(s_cb + n0 + 8)};
      constexpr uint32_t kNeg2 = 0u - (2u << 20);  // key = column base - (2 dot) << 20: one multiply-add per element
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int nb = 0; nb < 2; nb++) {
          top2_insert((uint32_t)c[mt][nb][0] * kNeg2 + cb[nb].x, k0[2 * mt], k1[2 * mt]);
          top2_insert((uint32_t)c[mt][nb][1] * kNeg2 + cb[nb].y, k0[2 * mt], k1[2 * mt]);
          top2_insert((uint32_t)c[mt][nb][2] * kNeg2 + cb[nb].x, k0[2 * mt + 1], k1[2 * mt + 1]);
          top2_insert((uint32_t)c[mt][nb][3] * kNeg2 + cb[nb].y, k0[2 * mt + 1], k1[2 * mt + 1]);
        }
    }
  }
  // ---- merge the four lanes of a quad (they hold different columns of the same rows)
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1)
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const uint32_t o0 = __shfl_xor_sync(0xffffffffu, k0[r], o), o1 = __shfl_xor_sync(0xffffffffu, k1[r], o);
      top2_insert(o0, k0[r], k1[r]);
      top2_insert(o1, k0[r], k1[r]);
    }
  if (t == 0) {
    const unsigned long long slice_base = (unsigned long long)(first_index + tile0 * kMmaTile);
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int row = qrow0 + 8 * r;
      if (row >= nq) continue;
      int pq = 0;
#pragma unroll
      for (int ks = 0; ks < 8; ks++) pq += __popc(__ldg(q + (size_t)row * 8 + ks));
      auto widen = [&](uint32_t key) -> unsigned long long {
        const int d = (int)(key >> 20) + pq - 256;
        if (key == ~0u || d > 256) return ~0ull;
        return ((unsigned long long)d << 48) | (slice_base + (key & 0xFFFFFu));
      };
      partial[((size_t)blockIdx.x * nq + row) * 2] = widen(k0[r]);
      partial[((size_t)blockIdx.x * nq + row) * 2 + 1] = widen(k1[r]);
    }
  }
}

// partial: [nparts][nq][kin] keys (kin = 2 for the slices of one shard scan; the all-gathered (world, nq, k) block of
// the multi-GPU query has the same layout with kin = k).
__global__ void db_merge_kernel(const unsigned long long* __restrict__ partial, int nparts, int nq, int kin, int k,
                                unsigned long long* __restrict__ topk, int32_t* __restrict__ votes, int th_votes,
                                long long first_kf, int desc_per_kf, long long first_index, long long n_kf) {
  const int qi = blockIdx.x * blockDim.x + threadIdx.x;
  if (qi >= nq) return;
  unsigned long long k0 = ~0ull, k1 = ~0ull;
  for (int p = 0; p < nparts; p++) {
    for (int e = 0; e < kin; e++) {
      const unsigned long long key = partial[((size_t)p * nq + qi) * kin + e];
      if (key < k1) {
        if (key < k0) {
          k1 = k0;
          k0 = key;
        } else {
          k1 = key;
        }
      }
    }
  }
  topk[(size_t)qi * k] = k0;
  if (k > 1) topk[(size_t)qi * k + 1] = k1;
  if (votes && k0 != ~0ull && (int)(k0 >> 48) <= th_votes) {
    const long long idx = (long long)(k0 & 0xFFFFFFFFFFFFull) - first_index;  // < 0: another shard's keyframe
    const long long kf = idx / desc_per_kf;
    if (idx >= 0 && kf < n_kf) atomicAdd(votes + kf, 1);
  }
  (void)first_kf;
}


// ---- Sharded place query, exchange over PEER MEMORY (NVLink / NVSwitch) inside the merge kernel.
// Every rank owns a window that its peers write into: keys[2][world][nq_max][2] (u64) followed by flags[2][world][kPeerBlocks]
// (u32), the leading 2 = parity of the query sequence number (a rank can be at most one query ahead of a peer: it
// cannot finish query s + 1 before that peer has pushed s + 1, which it does after it finished reading s).
// One launch per rank does what swm_db_query_sharded needs three enqueues for (slice merge, all-gather, final merge):
//   1. merge this shard's slice results for my queries (as db_merge_kernel);
//   2. store the (nq, k) keys into slot `rank` of EVERY rank's window -- remote stores over NVLink --, fence, then
//      publish flag[rank][block] = seq in each window (release, system scope);
//   3. wait until my own window holds flag[r][block] == seq for every r (acquire), merge the world key blocks with
//      L1-bypassing loads, write the global top-k and cast this shard's votes.
// CTAs only wait for the SAME block index of the other ranks and the whole grid (ceil(nq / 128) CTAs) is resident at
// once, so the launch behaves like a collective: every rank must enqueue it with the same nq, k and seq.
constexpr int kPeerBlocks = 64;  // CTAs of 128 queries: nq <= 8192 per call
constexpr int kPeerMaxWorld = 16;
struct PeerWindows {
  unsigned long long* keys[kPeerMaxWorld];  // window base of rank r as mapped in THIS process
};
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__global__ void __launch_bounds__(128) db_merge_peers_kernel(const unsigned long long* __restrict__ partial, int nparts, int nq, int k,
                                                             PeerWindows win, int rank, int world, int nq_max, unsigned int seq,
                                                             unsigned long long* __restrict__ topk, int32_t* __restrict__ votes,
                                                             int th_votes, int desc_per_kf, long long first_index, long long n_kf) {
  const int qi = blockIdx.x * blockDim.x + threadIdx.x;
  const int par = (int)(seq & 1u);
  const size_t keys_per_par = (size_t)world * nq_max * 2;
  const size_t flag_base = 2 * keys_per_par;  // in u64 units; flags follow the keys
  // 1. this shard's top-2 of my query
  unsigned long long k0 = ~0ull, k1 = ~0ull;
  if (qi < nq) {
    for (int p = 0; p < nparts; p++)
      for (int e = 0; e < 2; e++) {
        const unsigned long long key = partial[((size_t)p * nq + qi) * 2 + e];
        if (key < k1) {
          if (key < k0) { k1 = k0; k0 = key; }
          else k1 = key;
        }
      }
    // 2a. push into slot `rank` of every window
    const size_t slot = (size_t)par * keys_per_par + ((size_t)rank * nq_max + qi) * 2;
    for (int r = 0; r < world; r++) {
      unsigned long long* w = win.keys[r] + slot;
      w[0] = k0;
      w[1] = k1;
    }
  }
  __threadfence_system();
  __syncthreads();
  // 2b. publish: one flag per (writer rank, block) in every window
  if (threadIdx.x < world) {
    unsigned int* flags = reinterpret_cast<unsigned int*>(win.keys[threadIdx.x] + flag_base);
    st_release_sys(flags + ((size_t)par * world + rank) * kPeerBlocks + blockIdx.x, seq);
  }
  // 3. wait for every rank's block in MY window
  if (threadIdx.x < world) {
    const unsigned int* flags = reinterpret_cast<const unsigned int*>(win.keys[rank] + flag_base);
    const unsigned int* f = flags + ((size_t)par * world + threadIdx.x) * kPeerBlocks + blockIdx.x;
    long long spins = 0;
    while (ld_acquire_sys(f) != seq)
      if (++spins > (1ll << 28)) __trap();  // minutes: a rank that never arrives must abort, not hang the GPU for ever
  }
  __syncthreads();
  if (qi >= nq) return;
  k0 = k1 = ~0ull;
  const unsigned long long* mine = win.keys[rank] + (size_t)par * keys_per_par;
  for (int r = 0; r < world; r++)
    for (int e = 0; e < k; e++) {
      const unsigned long long key = __ldcg(mine + ((size_t)r * nq_max + qi) * 2 + e);  // written by a peer: not through L1
      if (key < k1) {
        if (key < k0) { k1 = k0; k0 = key; }
        else k1 = key;
      }
    }
  topk[(size_t)qi * k] = k0;
  if (k > 1) topk[(size_t)qi * k + 1] = k1;
  if (votes && k0 != ~0ull && (int)(k0 >> 48) <= th_votes) {
    const long long idx = (long long)(k0 & 0xFFFFFFFFFFFFull) - first_index;  // < 0: another shard's keyframe
    const long long kf = idx / desc_per_kf;
    if (idx >= 0 && kf < n_kf) atomicAdd(votes + kf, 1);
  }
}

}  // namespace swm

// =================================================================================================
// Host side
// =================================================================================================
using namespace swm;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  bool owned = true;
  void view(void* ptr) {  // point into the upload arena (non-owning)
    if (owned && p) cudaFree(p);
    p = ptr;
    cap = 0;
    owned = false;
  }
  cudaError_t ensure(size_t bytes) {
    if (owned && bytes <= cap) return cudaSuccess;
    if (owned && p) cudaFree(p);
    owned = true;
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 2 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (owned && p) cudaFree(p);
    p = nullptr;
    cap = 0;
    owned = true;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct swm_matcher {
  int device = 0;
  std::string err;
  cudaStream_t stream = nullptr;
  // frame uploads (two frames), query uploads, rows, state
  DevBuf f[2][6];  // x, y, octave, angle, desc, (grid starts+items+cell_of)
  DevBuf q[10];
  DevBuf iq[5];    // SearchForInitialization's source rows, built on the device (owned)
  DevBuf rowlist;  // resolve_kernel's compacted row list
  DevBuf rows[5];  // row_count, row_start, cand_idx, cand_val, row_src
  DevBuf state[5]; // blocked, out, ev_bin / best_dist, ev_tgt, nmatches
  // batch calls (match_batch.cuh): per-call scratch and the shared candidate buffers (index, level | distance),
  // grow-only, sized from earlier calls
  DevBuf bscratch;
  DevBuf bcand[2];
  size_t bcand_cap = 0;
  cudaEvent_t bev[2] = {nullptr, nullptr};  // around the kernels of the last batch call (swm_matcher_last_device_ms)
  float last_device_ms = 0.f;
  // PredictScale's level thresholds of the last scale table a projection call used (swm_predict_scale_thresholds)
  float thr_lsf = 0.f;
  int thr_n = 0;
  float thr[SWM_MAX_LEVELS] = {};
  // upload arena: every host array of a call is packed into one pinned buffer and sent with ONE copy
  uint8_t* h_arena = nullptr;
  uint8_t* d_arena = nullptr;
  size_t arena_cap = 0, arena_used = 0;
  // results come back through one pinned staging buffer (pageable destinations make every D2H copy a staged,
  // synchronising transfer); filled by down_copy, handed to the caller's arrays by down_finish
  uint8_t* h_down = nullptr;
  size_t down_cap = 0, down_used = 0;
  struct Down { void* dst; size_t off, bytes; };
  std::vector<Down> downs;
  void free_all() {
    if (h_arena) cudaFreeHost(h_arena);
    if (d_arena) cudaFree(d_arena);
    if (h_down) cudaFreeHost(h_down);
    h_arena = d_arena = h_down = nullptr;
    arena_cap = arena_used = down_cap = down_used = 0;
    for (auto& a : f) for (auto& b : a) b.release();
    for (auto& b : q) b.release();
    for (auto& b : iq) b.release();
    rowlist.release();
    for (auto& b : rows) b.release();
    for (auto& b : state) b.release();
    bscratch.release();
    for (auto& b : bcand) b.release();
    bcand_cap = 0;
    for (auto& e : bev) {
      if (e) cudaEventDestroy(e);
      e = nullptr;
    }
  }
};

// A frame's features resident on the device: undistorted keypoints (SoA), descriptors, grid CSR.
struct swm_frame {
  int device = 0;
  std::string err;
  int n = 0;
  DevBuf b[6];  // x, y, octave, angle, desc, grid (starts | items | cell_of)
  FrameDev dev{};
  cudaStream_t stream = nullptr;  // uploads; frames built from the extractor use the extractor's stream
  cudaEvent_t ready = nullptr;    // recorded after the last kernel that writes the frame
  // swm_frames_from_extractor: the first frame of a batch carries the build table and the pinned count read-back
  DevBuf bstage;
  int32_t* h_counts = nullptr;
  size_t h_counts_cap = 0;
};

namespace {

thread_local std::string g_match_create_error;
thread_local std::string g_frame_create_error;

// A matcher operand: host arrays (uploaded per call) or a resident frame.
struct FrameSrc {
  const swm_frame_view* host;
  const swm_frame* dev;
  int n() const { return dev ? dev->n : host->n; }
};

#define MCK(m, call)                                   \
  do {                                                 \
    cudaError_t e_ = (call);                           \
    if (e_ != cudaSuccess) {                           \
      (m)->err = cuda_err(#call, e_);                  \
      return SWM_E_CUDA;                               \
    }                                                  \
  } while (0)

// Reserve the upload arena for one call (upper bound on the packed bytes); previous views die here.
int arena_begin(swm_matcher* m, size_t bytes) {
  bytes += 4096;
  if (bytes > m->arena_cap) {
    MCK(m, cudaStreamSynchronize(m->stream));
    if (m->h_arena) cudaFreeHost(m->h_arena);
    if (m->d_arena) cudaFree(m->d_arena);
    m->h_arena = m->d_arena = nullptr;
    m->arena_cap = 0;
    const size_t want = bytes + bytes / 2;
    MCK(m, cudaMallocHost(&m->h_arena, want));
    MCK(m, cudaMalloc(&m->d_arena, want));
    m->arena_cap = want;
  }
  m->arena_used = 0;
  return SWM_OK;
}

// Packs a host array into the arena; `b` becomes a view of its device copy (valid after arena_flush).
int upload(swm_matcher* m, DevBuf& b, const void* src, size_t bytes) {
  const size_t off = (m->arena_used + 255) & ~(size_t)255;
  if (off + bytes > m->arena_cap) { m->err = "internal: upload arena overflow"; return SWM_E_CAPACITY; }
  if (bytes) memcpy(m->h_arena + off, src, bytes);
  b.view(m->d_arena + off);
  m->arena_used = off + bytes;
  return SWM_OK;
}

int arena_flush(swm_matcher* m) {
  if (m->arena_used)
    MCK(m, cudaMemcpyAsync(m->d_arena, m->h_arena, m->arena_used, cudaMemcpyHostToDevice, m->stream));
  return SWM_OK;
}

// Result download through the pinned staging buffer: down_begin(total) once, down_copy per array, down_finish
// synchronises the stream and copies into the caller's (pageable) arrays.
int down_begin(swm_matcher* m, size_t bytes) {
  bytes += 1024;
  if (bytes > m->down_cap) {
    MCK(m, cudaStreamSynchronize(m->stream));
    if (m->h_down) cudaFreeHost(m->h_down);
    m->h_down = nullptr;
    m->down_cap = 0;
    MCK(m, cudaMallocHost(&m->h_down, bytes + bytes / 2));
    m->down_cap = bytes + bytes / 2;
  }
  m->down_used = 0;
  m->downs.clear();
  return SWM_OK;
}
int down_copy(swm_matcher* m, void* dst, const void* d_src, size_t bytes) {
  const size_t off = (m->down_used + 63) & ~(size_t)63;
  if (off + bytes > m->down_cap) { m->err = "internal: download buffer overflow"; return SWM_E_CAPACITY; }
  if (bytes) MCK(m, cudaMemcpyAsync(m->h_down + off, d_src, bytes, cudaMemcpyDeviceToHost, m->stream));
  m->downs.push_back({dst, off, bytes});
  m->down_used = off + bytes;
  return SWM_OK;
}
int down_finish(swm_matcher* m) {
  MCK(m, cudaStreamSynchronize(m->stream));
  for (const auto& d : m->downs)
    if (d.bytes) memcpy(d.dst, m->h_down + d.off, d.bytes);
  m->downs.clear();
  return SWM_OK;
}

size_t frame_bytes(const swm_frame_view* f) { return (size_t)f->n * 48 + 5 * 256; }

// The keypoint arrays are caller-supplied (a keyframe slab may come off the wire): octave[] indexes the per-level
// tables inside the kernels and is packed into 16 bits next to the distance, so it must lie in [0, SWM_MAX_LEVELS);
// coordinates must be finite (they are turned into grid cells).
bool payload_ok(const swm_frame_view* f) {
  for (int i = 0; i < f->n; i++) {
    if ((uint32_t)f->octave[i] >= (uint32_t)SWM_MAX_LEVELS) return false;
    if (!std::isfinite(f->x[i]) || !std::isfinite(f->y[i])) return false;
  }
  return true;
}

bool frame_ok(const swm_frame_view* f) {
  return f && f->n >= 0 && (f->n == 0 || (f->x && f->y && f->octave && f->angle && f->desc)) && f->max_x > f->min_x &&
         f->max_y > f->min_y && payload_ok(f);
}

// Packs a frame's arrays into the upload arena (device views valid after arena_flush).
int upload_frame(swm_matcher* m, int slot, const swm_frame_view* f, FrameDev* out) {
  const size_t n = (size_t)f->n;
  int rc;
  if ((rc = upload(m, m->f[slot][0], f->x, n * 4))) return rc;
  if ((rc = upload(m, m->f[slot][1], f->y, n * 4))) return rc;
  if ((rc = upload(m, m->f[slot][2], f->octave, n * 4))) return rc;
  if ((rc = upload(m, m->f[slot][3], f->angle, n * 4))) return rc;
  if ((rc = upload(m, m->f[slot][4], f->desc, n * 32))) return rc;
  FrameDev d;
  d.n = f->n;
  d.x = m->f[slot][0].as<float>();
  d.y = m->f[slot][1].as<float>();
  d.octave = m->f[slot][2].as<int32_t>();
  d.angle = m->f[slot][3].as<float>();
  d.desc = m->f[slot][4].as<uint4>();
  d.min_x = f->min_x; d.min_y = f->min_y; d.max_x = f->max_x; d.max_y = f->max_y;
  d.inv_w = (float)kGridCols / (float)(f->max_x - f->min_x);  // Frame.cc:259-260
  d.inv_h = (float)kGridRows / (float)(f->max_y - f->min_y);
  d.starts = nullptr;
  d.items = nullptr;
  *out = d;
  return SWM_OK;
}

// Builds the frame grid on the device (after arena_flush).
int build_grid(swm_matcher* m, int slot, FrameDev* d) {
  const size_t n = (size_t)d->n;
  MCK(m, m->f[slot][5].ensure(((size_t)kCells + 1 + 2 * n + 8) * 4));
  int32_t* starts = m->f[slot][5].as<int32_t>();
  int32_t* items = starts + kCells + 1;
  int32_t* cell_of = items + n + 4;
  grid_build_kernel<<<1, 1024, 0, m->stream>>>(*d, starts, items, cell_of);
  MCK(m, cudaGetLastError());
  d->starts = starts;
  d->items = items;
  return SWM_OK;
}

// Operand -> device views.  Host arrays are packed into the arena (valid after arena_flush); a resident frame is
// used in place once its producer's event has been waited for on the matcher stream.
int acquire_frame(swm_matcher* m, int slot, const FrameSrc& f, FrameDev* out) {
  if (!f.dev) return upload_frame(m, slot, f.host, out);
  if (f.dev->device != m->device) { m->err = "resident frame lives on another device"; return SWM_E_INVALID; }
  MCK(m, cudaStreamWaitEvent(m->stream, f.dev->ready, 0));
  *out = f.dev->dev;
  return SWM_OK;
}
int acquire_grid(swm_matcher* m, int slot, const FrameSrc& f, FrameDev* d) {
  if (f.dev) return SWM_OK;  // built with the frame
  return build_grid(m, slot, d);
}
size_t src_bytes(const FrameSrc& f) { return f.dev ? 0 : frame_bytes(f.host); }

CameraDev camera_dev(const swm_camera* cam) {
  CameraDev c{};
  if (cam) {
    c.fx = cam->fx; c.fy = cam->fy; c.cx = cam->cx; c.cy = cam->cy;
    c.k1 = cam->k1; c.k2 = cam->k2; c.p1 = cam->p1; c.p2 = cam->p2; c.k3 = cam->k3;
    c.distorted = cam->k1 != 0.0f;  // Frame.cc:456
  }
  return c;
}

#define FCK(f, call)                                   \
  do {                                                 \
    cudaError_t e_ = (call);                           \
    if (e_ != cudaSuccess) {                           \
      (f)->err = cuda_err(#call, e_);                  \
      return SWM_E_CUDA;                               \
    }                                                  \
  } while (0)

// Allocates the SoA arrays + grid for n keypoints and points f->dev at them.
int frame_reserve(swm_frame* f, int n, const float* bounds4) {
  const size_t nn = (size_t)(n > 0 ? n : 1);
  FCK(f, f->b[0].ensure(nn * 4));
  FCK(f, f->b[1].ensure(nn * 4));
  FCK(f, f->b[2].ensure(nn * 4));
  FCK(f, f->b[3].ensure(nn * 4));
  FCK(f, f->b[4].ensure(nn * 32));
  FCK(f, f->b[5].ensure(((size_t)kCells + 1 + 2 * nn + 8) * 4));
  FrameDev d{};
  d.n = n;
  d.x = f->b[0].as<float>();
  d.y = f->b[1].as<float>();
  d.octave = f->b[2].as<int32_t>();
  d.angle = f->b[3].as<float>();
  d.desc = f->b[4].as<uint4>();
  d.min_x = bounds4[0]; d.max_x = bounds4[1]; d.min_y = bounds4[2]; d.max_y = bounds4[3];
  d.inv_w = (float)kGridCols / (float)(d.max_x - d.min_x);  // Frame.cc:259-260
  d.inv_h = (float)kGridRows / (float)(d.max_y - d.min_y);
  d.starts = f->b[5].as<int32_t>();
  d.items = f->b[5].as<int32_t>() + kCells + 1;
  f->dev = d;
  f->n = n;
  return SWM_OK;
}

int frame_grid(swm_frame* f, cudaStream_t st) {
  int32_t* starts = f->b[5].as<int32_t>();
  int32_t* items = starts + kCells + 1;
  int32_t* cell_of = items + (f->n > 0 ? f->n : 1) + 4;
  grid_build_kernel<<<1, 1024, 0, st>>>(f->dev, starts, items, cell_of);
  FCK(f, cudaGetLastError());
  FCK(f, cudaEventRecord(f->ready, st));
  return SWM_OK;
}

int launch_resolve(swm_matcher* m, const ResolveArgs& a) {
  const size_t n2 = (size_t)a.n2;
  const size_t bytes = (a.mode == kModeInit ? 8 * n2 : 0) + ((n2 + 3) & ~(size_t)3) + 4 * n2 + 16;
  if (bytes > 200 * 1024) {
    m->err = "target frame too large for the matcher's shared-memory state (n2 limit ~15000 keypoints)";
    return SWM_E_CAPACITY;
  }
  static bool attr_set[64] = {};
  if (!attr_set[m->device & 63]) {
    MCK(m, cudaFuncSetAttribute(resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set[m->device & 63] = true;
  }
  MCK(m, m->rowlist.ensure(((size_t)a.rows + 64) * 4));
  ResolveArgs ra = a;
  ra.row_list = m->rowlist.as<int32_t>();
  resolve_kernel<<<1, kResolveWarps * 32, bytes, m->stream>>>(ra);
  MCK(m, cudaGetLastError());
  return SWM_OK;
}

// window rows: count -> scan -> fill.  Returns total candidates through *total.
int build_window_rows(swm_matcher* m, const FrameDev& tgt, const WindowDev& q, int* total) {
  const int M = q.m;
  MCK(m, m->rows[0].ensure((size_t)(M + 1) * 4));
  MCK(m, m->rows[1].ensure((size_t)(M + 2) * 4));
  int32_t* row_count = m->rows[0].as<int32_t>();
  int32_t* row_start = m->rows[1].as<int32_t>();
  const int grid = (M + 7) / 8;
  window_rows_kernel<<<grid, 256, 0, m->stream>>>(tgt, q, 0, row_count, nullptr, nullptr, nullptr);
  scan_rows_kernel<<<1, 1024, 0, m->stream>>>(row_count, M, row_start);
  int tot = 0;
  MCK(m, cudaMemcpyAsync(&tot, row_start + M, 4, cudaMemcpyDeviceToHost, m->stream));
  MCK(m, cudaStreamSynchronize(m->stream));
  MCK(m, m->rows[2].ensure((size_t)(tot + 1) * 4));
  MCK(m, m->rows[3].ensure((size_t)(tot + 1) * 4));
  window_rows_kernel<<<grid, 256, 0, m->stream>>>(tgt, q, 1, row_count, row_start, m->rows[2].as<int32_t>(),
                                                  m->rows[3].as<uint32_t>());
  MCK(m, cudaGetLastError());
  *total = tot;
  return SWM_OK;
}

}  // namespace

extern "C" {

int swm_matcher_create(int device, swm_matcher** out) {
  if (!out) return SWM_E_INVALID;
  *out = nullptr;
  int rc = check_device(device, &g_match_create_error);
  if (rc != SWM_OK) return rc;
  swm_matcher* m = new swm_matcher;
  m->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    g_match_create_error = cuda_err("swm_matcher_create", e);
    delete m;
    return SWM_E_CUDA;
  }
  *out = m;
  return SWM_OK;
}

void swm_matcher_destroy(swm_matcher* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  m->free_all();
  if (m->stream) cudaStreamDestroy(m->stream);
  delete m;
}

const char* swm_matcher_last_error(const swm_matcher* m) { return m ? m->err.c_str() : g_match_create_error.c_str(); }

int swm_hamming_matrix_device(const uint8_t* d_a, int na, const uint8_t* d_b, int nb, uint16_t* d_out, void* stream) {
  if (!d_a || !d_b || !d_out || na < 0 || nb < 0) return SWM_E_INVALID;
  if (na == 0 || nb == 0) return SWM_OK;
  dim3 grid((nb + 31) / 32, (na + 31) / 32);
  hamming_matrix_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)d_a, na, (const uint4*)d_b, nb, d_out);
  return cudaGetLastError() == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

// Device scratch of the handle-less entry points below (swm_hamming_matrix / _pairs, swm_distinctive_descriptors,
// swm_camera_bounds): one grow-only arena per device, allocated on first use and kept, so that no call on the path
// allocates or frees device memory.  A call holds the arena's mutex from upload to download (these entry points
// run on the default stream and return host results, so they were serialised per device already).
namespace {
struct StaticScratch {
  std::mutex mu;
  uint8_t* p = nullptr;
  size_t cap = 0;
  uint8_t* reserve(size_t bytes) {
    if (bytes > cap) {
      if (p) cudaFree(p);
      p = nullptr; cap = 0;
      const size_t want = (std::max(bytes, (size_t)1 << 20) + 255) & ~(size_t)255;
      if (cudaMalloc(&p, want) != cudaSuccess) return nullptr;
      cap = want;
    }
    return p;
  }
};
StaticScratch g_static_scratch[64];
inline size_t up256(size_t n) { return (n + 255) & ~(size_t)255; }
}  // namespace

int swm_hamming_matrix(const uint8_t* a, int na, const uint8_t* b, int nb, uint16_t* out, int device) {
  if (!a || !b || !out || na < 0 || nb < 0) return SWM_E_INVALID;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (na == 0 || nb == 0) return SWM_OK;
  if (device < 0 || device >= 64 || cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  StaticScratch& sc = g_static_scratch[device];
  std::lock_guard<std::mutex> lock(sc.mu);
  const size_t oa = 0, ob = up256((size_t)na * 32), oo = ob + up256((size_t)nb * 32);
  uint8_t* base = sc.reserve(oo + (size_t)na * nb * 2);
  if (!base) return SWM_E_CUDA;
  uint8_t *da = base + oa, *db = base + ob;
  uint16_t* dout = (uint16_t*)(base + oo);
  cudaError_t e = cudaMemcpy(da, a, (size_t)na * 32, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(db, b, (size_t)nb * 32, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) rc = swm_hamming_matrix_device(da, na, db, nb, dout, nullptr);
  if (e == cudaSuccess && rc == SWM_OK) e = cudaMemcpy(out, dout, (size_t)na * nb * 2, cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? rc : SWM_E_CUDA;
}

int swm_hamming_pairs(const uint8_t* a, const uint8_t* b, int n, int32_t* out, int device) {
  if (!a || !b || !out || n < 0) return SWM_E_INVALID;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (n == 0) return SWM_OK;
  if (device < 0 || device >= 64 || cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  StaticScratch& sc = g_static_scratch[device];
  std::lock_guard<std::mutex> lock(sc.mu);
  const size_t ob = up256((size_t)n * 32), oo = 2 * ob;
  uint8_t* base = sc.reserve(oo + (size_t)n * 4);
  if (!base) return SWM_E_CUDA;
  uint8_t *da = base, *db = base + ob;
  int32_t* dout = (int32_t*)(base + oo);
  cudaError_t e = cudaMemcpy(da, a, (size_t)n * 32, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(db, b, (size_t)n * 32, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    hamming_pairs_kernel<<<(n + 255) / 256, 256>>>((const uint4*)da, (const uint4*)db, n, dout);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, dout, (size_t)n * 4, cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

int swm_distinctive_descriptors(const uint8_t* desc, const int32_t* offsets, int npoints, int32_t* best_idx,
                                int32_t* best_median, int device) {
  if (!offsets || npoints < 0 || !best_idx) return SWM_E_INVALID;
  if (npoints == 0) return SWM_OK;
  const long long total = offsets[npoints];
  int max_n = 0;
  for (int p = 0; p < npoints; p++) {
    const int n = offsets[p + 1] - offsets[p];
    if (n < 0) return SWM_E_INVALID;
    max_n = std::max(max_n, n);
  }
  if (total < 0 || offsets[0] != 0 || (total > 0 && !desc)) return SWM_E_INVALID;
  if (max_n > kDistinctMax) return SWM_E_CAPACITY;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (device < 0 || device >= 64 || cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  StaticScratch& sc = g_static_scratch[device];
  std::lock_guard<std::mutex> lock(sc.mu);
  const size_t o_off = up256((size_t)std::max<long long>(total, 1) * 32), o_out = o_off + up256(((size_t)npoints + 1) * 4);
  uint8_t* base = sc.reserve(o_out + 2 * (size_t)npoints * 4);
  if (!base) return SWM_E_CUDA;
  uint8_t* d_desc = base;
  int32_t *d_off = (int32_t*)(base + o_off), *d_out = (int32_t*)(base + o_out);
  std::vector<int32_t> out(2 * (size_t)npoints);
  bool ok = true;
  if (ok && total) ok = cudaMemcpy(d_desc, desc, (size_t)total * 32, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(d_off, offsets, ((size_t)npoints + 1) * 4, cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok) {
    distinctive_kernel<<<npoints, 128, (size_t)std::max(max_n, 1) * 32>>>((const uint4*)d_desc, d_off, d_out, d_out + npoints);
    ok = cudaGetLastError() == cudaSuccess &&
         cudaMemcpy(out.data(), d_out, out.size() * 4, cudaMemcpyDeviceToHost) == cudaSuccess;
  }
  if (!ok) return SWM_E_CUDA;
  for (int p = 0; p < npoints; p++) {
    best_idx[p] = out[p];
    if (best_median) best_median[p] = out[(size_t)npoints + p];
  }
  return SWM_OK;
}

int swm_grid_build(swm_matcher* m, const swm_frame_view* f, int32_t* starts, int32_t* items) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(f) || !starts || !items) { m->err = "bad argument"; return SWM_E_INVALID; }
  MCK(m, cudaSetDevice(m->device));
  FrameDev d;
  int rc;
  if ((rc = arena_begin(m, frame_bytes(f)))) return rc;
  if ((rc = upload_frame(m, 0, f, &d))) return rc;
  if ((rc = arena_flush(m))) return rc;
  if ((rc = build_grid(m, 0, &d))) return rc;
  MCK(m, cudaMemcpyAsync(starts, d.starts, ((size_t)kCells + 1) * 4, cudaMemcpyDeviceToHost, m->stream));
  MCK(m, cudaStreamSynchronize(m->stream));
  const int total = starts[kCells];
  if (total) MCK(m, cudaMemcpy(items, d.items, (size_t)total * 4, cudaMemcpyDeviceToHost));
  return SWM_OK;
}

}  // extern "C"

namespace {

int match_init_impl(swm_matcher* m, const FrameSrc& f1, const FrameSrc& f2, float* prev_xy, int32_t* matches12,
                    int window, float nnratio, int check_ori, int* nmatches) {
  *nmatches = 0;
  const int n1 = f1.n(), n2 = f2.n();
  for (int i = 0; i < n1; i++) matches12[i] = -1;
  if (n1 == 0 || n2 == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  FrameDev d1, d2;
  int rc;
  if ((rc = arena_begin(m, src_bytes(f1) + src_bytes(f2) + (size_t)n1 * 8 + 8 * 256))) return rc;
  if ((rc = acquire_frame(m, 0, f1, &d1))) return rc;
  if ((rc = acquire_frame(m, 1, f2, &d2))) return rc;
  if ((rc = upload(m, m->q[5], prev_xy, (size_t)n1 * 8))) return rc;
  if ((rc = arena_flush(m))) return rc;
  if ((rc = acquire_grid(m, 1, f2, &d2))) return rc;
  // sources = F1 keypoints at octave 0 (:390-392), window centre = vbPrevMatched, levels (0,0) (:394-396)
  for (int i = 0; i < 4; i++) MCK(m, m->iq[i].ensure((size_t)n1 * 4));
  MCK(m, m->iq[4].ensure((size_t)n1));
  init_query_kernel<<<(n1 + 255) / 256, 256, 0, m->stream>>>(d1.octave, m->q[5].as<float>(), n1, (float)window,
                                                             m->iq[0].as<float>(), m->iq[1].as<float>(),
                                                             m->iq[2].as<float>(), m->iq[3].as<int32_t>(),
                                                             m->iq[4].as<uint8_t>());
  MCK(m, cudaGetLastError());
  WindowDev q;
  q.m = n1;
  q.desc = d1.desc;
  q.u = m->iq[0].as<float>();
  q.v = m->iq[1].as<float>();
  q.radius = m->iq[2].as<float>();
  q.min_level = m->iq[3].as<int32_t>();
  q.max_level = m->iq[3].as<int32_t>();
  q.valid = m->iq[4].as<uint8_t>();
  int total = 0;
  if ((rc = build_window_rows(m, d2, q, &total))) return rc;
  // state
  MCK(m, m->state[1].ensure((size_t)n1 * 4));
  MCK(m, m->state[2].ensure((size_t)n1 * 4));
  MCK(m, m->state[3].ensure((size_t)n1 * 4));
  MCK(m, m->state[4].ensure(16));
  MCK(m, cudaMemsetAsync(m->state[1].p, 0xFF, (size_t)n1 * 4, m->stream));
  MCK(m, cudaMemsetAsync(m->state[2].p, 0xFF, (size_t)n1 * 4, m->stream));
  ResolveArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = kModeInit;
  a.rows = n1;
  a.row_valid = q.valid;
  a.row_start = m->rows[1].as<int32_t>();
  a.cand_idx = m->rows[2].as<int32_t>();
  a.cand_val = m->rows[3].as<uint32_t>();
  a.n1 = n1; a.n2 = n2;
  a.angle1 = d1.angle; a.angle2 = d2.angle;
  a.nnratio = nnratio;
  a.check_ori = check_ori;
  a.out = m->state[1].as<int32_t>();
  a.ev_bin = m->state[2].as<int32_t>();
  a.ev_tgt = m->state[3].as<int32_t>();
  a.prev_xy = m->q[5].as<float>();
  a.x2 = d2.x; a.y2 = d2.y;
  a.nmatches = m->state[4].as<int32_t>();
  if ((rc = launch_resolve(m, a))) return rc;
  MCK(m, cudaGetLastError());
  if ((rc = down_begin(m, (size_t)n1 * 12 + 256))) return rc;
  if ((rc = down_copy(m, matches12, a.out, (size_t)n1 * 4))) return rc;
  if ((rc = down_copy(m, prev_xy, a.prev_xy, (size_t)n1 * 8))) return rc;
  if ((rc = down_copy(m, nmatches, a.nmatches, 4))) return rc;
  return down_finish(m);
}

bool window_query_ok(const swm_window_query* wq, int check_ori) {
  return wq && wq->m >= 0 &&
         (wq->m == 0 || (wq->desc && wq->u && wq->v && wq->radius && wq->min_level && wq->max_level && wq->valid &&
                         wq->blocks && (!check_ori || wq->angle)));
}

// Resident operands as every matcher entry point checks them: both on the matcher's device, and `built` (when not NULL)
// holding its grid.
int resident_ok(swm_matcher* m, const swm_frame* a, const swm_frame* b, const swm_frame* built) {
  if (a->device != m->device || b->device != m->device) { m->err = "resident frame lives on another device"; return SWM_E_INVALID; }
  if (built && !built->dev.starts) { m->err = "resident frame has not been built"; return SWM_E_STATE; }
  return SWM_OK;
}

bool featvec_ok(const swm_featvec* fv) {
  if (!fv || fv->n_nodes < 0) return false;
  if (fv->n_nodes == 0) return true;
  if (!fv->node_ids || !fv->offsets || !fv->feats || fv->offsets[0] < 0) return false;
  for (int a = 0; a < fv->n_nodes; a++) {
    if (fv->offsets[a + 1] < fv->offsets[a]) return false;
    if (a && fv->node_ids[a] <= fv->node_ids[a - 1]) return false;  // strictly ascending node ids (std::map order)
  }
  return true;
}

int match_window_impl(swm_matcher* m, const FrameSrc& tgt, const swm_window_query* wq, const uint8_t* tgt_blocked,
                      int th_dist, int ratio_mode, float nnratio, int check_ori, int32_t* assignment, int* nmatches) {
  *nmatches = 0;
  const int M = wq->m, n2 = tgt.n();
  if (M == 0 || n2 == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  FrameDev d2;
  int rc;
  if ((rc = arena_begin(m, src_bytes(tgt) + (size_t)M * 64 + (size_t)n2 * 8 + 16 * 256))) return rc;
  if ((rc = acquire_frame(m, 1, tgt, &d2))) return rc;
  if ((rc = upload(m, m->q[0], wq->u, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[1], wq->v, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[2], wq->radius, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[3], wq->min_level, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[6], wq->max_level, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[4], wq->valid, (size_t)M))) return rc;
  if ((rc = upload(m, m->q[7], wq->desc, (size_t)M * 32))) return rc;
  if ((rc = upload(m, m->q[8], wq->blocks, (size_t)M))) return rc;
  if (check_ori && (rc = upload(m, m->q[9], wq->angle, (size_t)M * 4))) return rc;
  // initial greedy state travels in the same packed upload
  std::vector<uint8_t> zero_blocked;
  if (!tgt_blocked) zero_blocked.assign((size_t)n2, 0);
  if ((rc = upload(m, m->state[0], tgt_blocked ? tgt_blocked : zero_blocked.data(), (size_t)n2))) return rc;
  if ((rc = upload(m, m->state[1], assignment, (size_t)n2 * 4))) return rc;
  if ((rc = arena_flush(m))) return rc;
  if ((rc = acquire_grid(m, 1, tgt, &d2))) return rc;
  WindowDev q;
  q.m = M;
  q.desc = m->q[7].as<uint4>();
  q.u = m->q[0].as<float>();
  q.v = m->q[1].as<float>();
  q.radius = m->q[2].as<float>();
  q.min_level = m->q[3].as<int32_t>();
  q.max_level = m->q[6].as<int32_t>();
  q.valid = m->q[4].as<uint8_t>();
  int total = 0;
  if ((rc = build_window_rows(m, d2, q, &total))) return rc;
  MCK(m, m->state[2].ensure((size_t)M * 4));
  MCK(m, m->state[3].ensure((size_t)M * 4));
  MCK(m, m->state[4].ensure(16));
  MCK(m, cudaMemsetAsync(m->state[2].p, 0xFF, (size_t)M * 4, m->stream));
  ResolveArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = kModeWindow;
  a.rows = M;
  a.row_valid = q.valid;
  a.row_start = m->rows[1].as<int32_t>();
  a.cand_idx = m->rows[2].as<int32_t>();
  a.cand_val = m->rows[3].as<uint32_t>();
  a.n1 = M; a.n2 = n2;
  a.angle1 = m->q[9].as<float>();
  a.angle2 = d2.angle;
  a.blocks = m->q[8].as<uint8_t>();
  a.th_dist = th_dist;
  a.ratio_mode = ratio_mode;
  a.nnratio = nnratio;
  a.check_ori = check_ori;
  a.blocked = m->state[0].as<uint8_t>();
  a.out = m->state[1].as<int32_t>();
  a.ev_bin = m->state[2].as<int32_t>();
  a.ev_tgt = m->state[3].as<int32_t>();
  a.nmatches = m->state[4].as<int32_t>();
  if ((rc = launch_resolve(m, a))) return rc;
  if ((rc = down_begin(m, (size_t)n2 * 4 + 256))) return rc;
  if ((rc = down_copy(m, assignment, a.out, (size_t)n2 * 4))) return rc;
  if ((rc = down_copy(m, nmatches, a.nmatches, 4))) return rc;
  return down_finish(m);
}

// Merge-walk of two sorted FeatureVectors (ORBmatcher.cc:166-241, :507-581, :629-722): rows = the valid side-1
// features of shared nodes in visiting order, candidates = the side-2 features of the node.
int node_rows(swm_matcher* m, const swm_featvec* fv1, const uint8_t* valid1, int n1, const swm_featvec* fv2, int n2,
              std::vector<int32_t>& row_src, std::vector<int32_t>& row_start, std::vector<int32_t>& cand) {
  row_src.clear();
  cand.clear();
  row_start.assign(1, 0);
  for (const swm_featvec* fv : {fv1, fv2})  // offsets[] is caller-supplied: non-negative and non-decreasing
    for (int a = 0; a < fv->n_nodes; a++)
      if (fv->offsets[a] < 0 || fv->offsets[a + 1] < fv->offsets[a]) { m->err = "feature vector offsets not monotonic"; return SWM_E_INVALID; }
  int a = 0, b = 0;
  while (a < fv1->n_nodes && b < fv2->n_nodes) {
    const uint32_t ia = fv1->node_ids[a], ib = fv2->node_ids[b];
    if (ia == ib) {
      for (int i1 = fv1->offsets[a]; i1 < fv1->offsets[a + 1]; i1++) {
        const uint32_t idx1 = fv1->feats[i1];
        if (idx1 >= (uint32_t)n1) { m->err = "feature index out of range"; return SWM_E_INVALID; }
        if (!valid1[idx1]) continue;
        row_src.push_back((int32_t)idx1);
        for (int i2 = fv2->offsets[b]; i2 < fv2->offsets[b + 1]; i2++) {
          if (fv2->feats[i2] >= (uint32_t)n2) { m->err = "feature index out of range"; return SWM_E_INVALID; }
          cand.push_back((int32_t)fv2->feats[i2]);
        }
        row_start.push_back((int32_t)cand.size());
      }
      a++;
      b++;
    } else if (ia < ib) {
      a = (int)(std::lower_bound(fv1->node_ids, fv1->node_ids + fv1->n_nodes, ib) - fv1->node_ids);
    } else {
      b = (int)(std::lower_bound(fv2->node_ids, fv2->node_ids + fv2->n_nodes, ia) - fv2->node_ids);
    }
  }
  return SWM_OK;
}

int match_bow_impl(swm_matcher* m, const FrameSrc& f1, const swm_featvec* fv1, const uint8_t* valid1, const FrameSrc& f2,
                   const swm_featvec* fv2, const uint8_t* valid2, int mode, float nnratio, int check_ori, int32_t* matches,
                   int* nmatches) {
  *nmatches = 0;
  const int n1 = f1.n(), n2 = f2.n();
  const int n_out = mode == 0 ? n2 : n1;
  for (int i = 0; i < n_out; i++) matches[i] = -1;
  if (n1 == 0 || n2 == 0) return SWM_OK;
  std::vector<int32_t> row_src, row_start, cand;
  {
    const int wrc = node_rows(m, fv1, valid1, n1, fv2, n2, row_src, row_start, cand);
    if (wrc != SWM_OK) return wrc;
  }
  const int R = (int)row_src.size();
  if (R == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  FrameDev d1, d2;
  int rc;
  if ((rc = arena_begin(m, src_bytes(f1) + src_bytes(f2) + (size_t)R * 8 + cand.size() * 4 + (size_t)n2 + 8 * 256))) return rc;
  if ((rc = acquire_frame(m, 0, f1, &d1))) return rc;
  if ((rc = acquire_frame(m, 1, f2, &d2))) return rc;
  if ((rc = upload(m, m->rows[4], row_src.data(), (size_t)R * 4))) return rc;
  if ((rc = upload(m, m->rows[1], row_start.data(), (size_t)(R + 1) * 4))) return rc;
  if ((rc = upload(m, m->rows[2], cand.data(), cand.size() * 4))) return rc;
  if (mode == 1 && (rc = upload(m, m->q[4], valid2, (size_t)n2))) return rc;
  if ((rc = arena_flush(m))) return rc;
  MCK(m, m->rows[3].ensure((cand.size() + 1) * 4));
  list_rows_kernel<<<(R + 7) / 8, 256, 0, m->stream>>>(d1.desc, d2.desc, d2.octave, R, m->rows[4].as<int32_t>(),
                                                      m->rows[1].as<int32_t>(), m->rows[2].as<int32_t>(),
                                                      m->rows[3].as<uint32_t>());
  MCK(m, cudaGetLastError());
  MCK(m, m->state[0].ensure((size_t)n2));
  MCK(m, m->state[1].ensure((size_t)n_out * 4));
  MCK(m, m->state[2].ensure((size_t)n1 * 4));
  MCK(m, m->state[3].ensure((size_t)n1 * 4));
  MCK(m, m->state[4].ensure(16));
  MCK(m, cudaMemsetAsync(m->state[0].p, 0, (size_t)n2, m->stream));
  MCK(m, cudaMemsetAsync(m->state[1].p, 0xFF, (size_t)n_out * 4, m->stream));
  MCK(m, cudaMemsetAsync(m->state[2].p, 0xFF, (size_t)n1 * 4, m->stream));
  ResolveArgs ra;
  memset(&ra, 0, sizeof(ra));
  ra.mode = mode == 0 ? kModeBowFrame : kModeBowKf;
  ra.rows = R;
  ra.row_src = m->rows[4].as<int32_t>();
  ra.row_start = m->rows[1].as<int32_t>();
  ra.cand_idx = m->rows[2].as<int32_t>();
  ra.cand_val = m->rows[3].as<uint32_t>();
  ra.n1 = n1; ra.n2 = n2;
  ra.angle1 = d1.angle; ra.angle2 = d2.angle;
  ra.valid2 = m->q[4].as<uint8_t>();
  ra.nnratio = nnratio;
  ra.check_ori = check_ori;
  ra.blocked = m->state[0].as<uint8_t>();
  ra.out = m->state[1].as<int32_t>();
  ra.ev_bin = m->state[2].as<int32_t>();
  ra.ev_tgt = m->state[3].as<int32_t>();
  ra.nmatches = m->state[4].as<int32_t>();
  if ((rc = launch_resolve(m, ra))) return rc;
  MCK(m, cudaGetLastError());
  if ((rc = down_begin(m, (size_t)n_out * 4 + 256))) return rc;
  if ((rc = down_copy(m, matches, ra.out, (size_t)n_out * 4))) return rc;
  if ((rc = down_copy(m, nmatches, ra.nmatches, 4))) return rc;
  return down_finish(m);
}

int match_triangulation_impl(swm_matcher* m, const FrameSrc& f1, const swm_featvec* fv1, const uint8_t* valid1,
                             const FrameSrc& f2, const swm_featvec* fv2, const uint8_t* valid2,
                             const swm_triangulation_query* q, int check_ori, int32_t* matches12, int* nmatches) {
  *nmatches = 0;
  const int n1 = f1.n(), n2 = f2.n();
  for (int i = 0; i < n1; i++) matches12[i] = -1;
  if (n1 == 0 || n2 == 0) return SWM_OK;
  std::vector<int32_t> row_src, row_start, cand;
  int rc = node_rows(m, fv1, valid1, n1, fv2, n2, row_src, row_start, cand);
  if (rc != SWM_OK) return rc;
  const int R = (int)row_src.size();
  if (R == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  FrameDev d1, d2;
  const size_t nl = (size_t)q->nlevels;
  if ((rc = arena_begin(m, src_bytes(f1) + src_bytes(f2) + (size_t)R * 8 + cand.size() * 4 + (size_t)n2 + nl * 8 + 10 * 256))) return rc;
  if ((rc = acquire_frame(m, 0, f1, &d1))) return rc;
  if ((rc = acquire_frame(m, 1, f2, &d2))) return rc;
  if ((rc = upload(m, m->rows[4], row_src.data(), (size_t)R * 4))) return rc;
  if ((rc = upload(m, m->rows[1], row_start.data(), (size_t)(R + 1) * 4))) return rc;
  if ((rc = upload(m, m->rows[2], cand.data(), cand.size() * 4))) return rc;
  if ((rc = upload(m, m->q[4], valid2, (size_t)n2))) return rc;
  if ((rc = upload(m, m->q[0], q->scale_factors2, nl * 4))) return rc;
  if ((rc = upload(m, m->q[1], q->level_sigma2, nl * 4))) return rc;
  if ((rc = arena_flush(m))) return rc;
  MCK(m, m->state[1].ensure((size_t)n1 * 4));
  MCK(m, m->state[2].ensure((size_t)n1 * 4));
  MCK(m, m->state[4].ensure(16));
  MCK(m, cudaMemsetAsync(m->state[1].p, 0xFF, (size_t)n1 * 4, m->stream));
  MCK(m, cudaMemsetAsync(m->state[2].p, 0xFF, (size_t)n1 * 4, m->stream));
  TriDev t;
  for (int i = 0; i < 9; i++) t.F[i] = q->F12[i];
  t.ex = q->ex;
  t.ey = q->ey;
  t.sf2 = m->q[0].as<float>();
  t.sigma2 = m->q[1].as<float>();
  t.nlevels = q->nlevels;
  tri_rows_kernel<<<(R + 7) / 8, 256, 0, m->stream>>>(d1, d2, m->q[4].as<uint8_t>(), R, m->rows[4].as<int32_t>(),
                                                      m->rows[1].as<int32_t>(), m->rows[2].as<int32_t>(), t, check_ori,
                                                      m->state[1].as<int32_t>(), m->state[2].as<int32_t>());
  MCK(m, cudaGetLastError());
  tri_finalize_kernel<<<1, 1024, 0, m->stream>>>(n1, m->state[1].as<int32_t>(), m->state[2].as<int32_t>(), check_ori,
                                                 m->state[4].as<int32_t>());
  MCK(m, cudaGetLastError());
  if ((rc = down_begin(m, (size_t)n1 * 4 + 256))) return rc;
  if ((rc = down_copy(m, matches12, m->state[1].p, (size_t)n1 * 4))) return rc;
  if ((rc = down_copy(m, nmatches, m->state[4].p, 4))) return rc;
  return down_finish(m);
}

int window_best_impl(swm_matcher* m, const FrameSrc& tgt, const swm_best_query* bq, int32_t* best_idx, int32_t* best_dist) {
  const int M = bq->m, n2 = tgt.n();
  for (int i = 0; i < M; i++) { best_idx[i] = -1; best_dist[i] = 256; }
  if (M == 0 || n2 == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  FrameDev d2;
  int rc;
  const bool gate = bq->chi2 > 0.0f;
  if ((rc = arena_begin(m, src_bytes(tgt) + (size_t)M * 64 + (size_t)SWM_MAX_LEVELS * 4 + 12 * 256))) return rc;
  if ((rc = acquire_frame(m, 1, tgt, &d2))) return rc;
  if ((rc = upload(m, m->q[0], bq->u, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[1], bq->v, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[2], bq->radius, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[3], bq->min_level, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[6], bq->max_level, (size_t)M * 4))) return rc;
  if ((rc = upload(m, m->q[4], bq->valid, (size_t)M))) return rc;
  if ((rc = upload(m, m->q[7], bq->desc, (size_t)M * 32))) return rc;
  if (gate && (rc = upload(m, m->q[9], bq->inv_level_sigma2, (size_t)bq->nlevels * 4))) return rc;
  if ((rc = arena_flush(m))) return rc;
  if ((rc = acquire_grid(m, 1, tgt, &d2))) return rc;
  WindowDev q;
  q.m = M;
  q.desc = m->q[7].as<uint4>();
  q.u = m->q[0].as<float>();
  q.v = m->q[1].as<float>();
  q.radius = m->q[2].as<float>();
  q.min_level = m->q[3].as<int32_t>();
  q.max_level = m->q[6].as<int32_t>();
  q.valid = m->q[4].as<uint8_t>();
  int total = 0;
  if ((rc = build_window_rows(m, d2, q, &total))) return rc;
  MCK(m, m->state[1].ensure((size_t)M * 4));
  MCK(m, m->state[2].ensure((size_t)M * 4));
  best_rows_kernel<<<(M + 7) / 8, 256, 0, m->stream>>>(d2, M, q.u, q.v, m->rows[1].as<int32_t>(), m->rows[2].as<int32_t>(),
                                                       m->rows[3].as<uint32_t>(), gate ? m->q[9].as<float>() : nullptr,
                                                       gate ? bq->nlevels : 0, gate ? bq->chi2 : 0.0f, m->state[1].as<int32_t>(),
                                                       m->state[2].as<int32_t>());
  MCK(m, cudaGetLastError());
  if ((rc = down_begin(m, (size_t)M * 8 + 256))) return rc;
  if ((rc = down_copy(m, best_idx, m->state[1].p, (size_t)M * 4))) return rc;
  if ((rc = down_copy(m, best_dist, m->state[2].p, (size_t)M * 4))) return rc;
  return down_finish(m);
}

bool best_query_ok(const swm_best_query* q) {
  return q && q->m >= 0 &&
         (q->m == 0 || (q->desc && q->u && q->v && q->radius && q->min_level && q->max_level && q->valid)) &&
         (q->chi2 <= 0.0f || (q->inv_level_sigma2 && q->nlevels > 0 && q->nlevels <= SWM_MAX_LEVELS));
}

bool tri_query_ok(const swm_triangulation_query* q) {
  return q && q->F12 && q->scale_factors2 && q->level_sigma2 && q->nlevels > 0 && q->nlevels <= SWM_MAX_LEVELS;
}

}  // namespace

extern "C" {

int swm_match_init(swm_matcher* m, const swm_frame_view* f1, const swm_frame_view* f2, float* prev_xy,
                   int32_t* matches12, int window, float nnratio, int check_ori, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(f1) || !frame_ok(f2) || !prev_xy || !matches12 || !nmatches || window < 0) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  return match_init_impl(m, FrameSrc{f1, nullptr}, FrameSrc{f2, nullptr}, prev_xy, matches12, window, nnratio, check_ori,
                         nmatches);
}

int swm_match_init_resident(swm_matcher* m, const swm_frame* f1, const swm_frame* f2, float* prev_xy, int32_t* matches12,
                            int window, float nnratio, int check_ori, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!f1 || !f2 || !prev_xy || !matches12 || !nmatches || window < 0) { m->err = "bad argument"; return SWM_E_INVALID; }
  if (int rc = resident_ok(m, f1, f2, f2)) return rc;
  return match_init_impl(m, FrameSrc{nullptr, f1}, FrameSrc{nullptr, f2}, prev_xy, matches12, window, nnratio, check_ori,
                         nmatches);
}

int swm_match_window(swm_matcher* m, const swm_frame_view* tgt, const swm_window_query* wq,
                     const uint8_t* tgt_blocked, int th_dist, int ratio_mode, float nnratio, int check_ori,
                     int32_t* assignment, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(tgt) || !window_query_ok(wq, check_ori) || !assignment || !nmatches ||
      (ratio_mode != 0 && ratio_mode != 1)) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  return match_window_impl(m, FrameSrc{tgt, nullptr}, wq, tgt_blocked, th_dist, ratio_mode, nnratio, check_ori, assignment,
                           nmatches);
}

int swm_match_window_resident(swm_matcher* m, const swm_frame* tgt, const swm_window_query* wq,
                              const uint8_t* tgt_blocked, int th_dist, int ratio_mode, float nnratio, int check_ori,
                              int32_t* assignment, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!tgt || !window_query_ok(wq, check_ori) || !assignment || !nmatches || (ratio_mode != 0 && ratio_mode != 1)) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  if (int rc = resident_ok(m, tgt, tgt, tgt)) return rc;
  return match_window_impl(m, FrameSrc{nullptr, tgt}, wq, tgt_blocked, th_dist, ratio_mode, nnratio, check_ori, assignment,
                           nmatches);
}

int swm_match_bow(swm_matcher* m, const swm_frame_view* f1, const swm_featvec* fv1, const uint8_t* valid1,
                  const swm_frame_view* f2, const swm_featvec* fv2, const uint8_t* valid2, int mode, float nnratio,
                  int check_ori, int32_t* matches, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(f1) || !frame_ok(f2) || !featvec_ok(fv1) || !featvec_ok(fv2) || !valid1 || (mode == 1 && !valid2) ||
      !matches || !nmatches || (mode != 0 && mode != 1)) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  return match_bow_impl(m, FrameSrc{f1, nullptr}, fv1, valid1, FrameSrc{f2, nullptr}, fv2, valid2, mode, nnratio, check_ori,
                        matches, nmatches);
}

int swm_match_bow_resident(swm_matcher* m, const swm_frame* f1, const swm_featvec* fv1, const uint8_t* valid1,
                           const swm_frame* f2, const swm_featvec* fv2, const uint8_t* valid2, int mode, float nnratio,
                           int check_ori, int32_t* matches, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!f1 || !f2 || !featvec_ok(fv1) || !featvec_ok(fv2) || !valid1 || (mode == 1 && !valid2) || !matches || !nmatches ||
      (mode != 0 && mode != 1)) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  if (int rc = resident_ok(m, f1, f2, nullptr)) return rc;
  return match_bow_impl(m, FrameSrc{nullptr, f1}, fv1, valid1, FrameSrc{nullptr, f2}, fv2, valid2, mode, nnratio, check_ori,
                        matches, nmatches);
}

int swm_window_best(swm_matcher* m, const swm_frame_view* tgt, const swm_best_query* q, int32_t* best_idx, int32_t* best_dist) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(tgt) || !best_query_ok(q) || !best_idx || !best_dist) { m->err = "bad argument"; return SWM_E_INVALID; }
  return window_best_impl(m, FrameSrc{tgt, nullptr}, q, best_idx, best_dist);
}

int swm_window_best_resident(swm_matcher* m, const swm_frame* tgt, const swm_best_query* q, int32_t* best_idx,
                             int32_t* best_dist) {
  if (!m) return SWM_E_INVALID;
  if (!tgt || !best_query_ok(q) || !best_idx || !best_dist) { m->err = "bad argument"; return SWM_E_INVALID; }
  return window_best_impl(m, FrameSrc{nullptr, tgt}, q, best_idx, best_dist);
}

int swm_match_triangulation(swm_matcher* m, const swm_frame_view* f1, const swm_featvec* fv1, const uint8_t* valid1,
                            const swm_frame_view* f2, const swm_featvec* fv2, const uint8_t* valid2,
                            const swm_triangulation_query* q, int check_ori, int32_t* matches12, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!frame_ok(f1) || !frame_ok(f2) || !fv1 || !fv2 || !valid1 || !valid2 || !tri_query_ok(q) || !matches12 || !nmatches) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  return match_triangulation_impl(m, FrameSrc{f1, nullptr}, fv1, valid1, FrameSrc{f2, nullptr}, fv2, valid2, q, check_ori,
                                  matches12, nmatches);
}

int swm_match_triangulation_resident(swm_matcher* m, const swm_frame* f1, const swm_featvec* fv1, const uint8_t* valid1,
                                     const swm_frame* f2, const swm_featvec* fv2, const uint8_t* valid2,
                                     const swm_triangulation_query* q, int check_ori, int32_t* matches12, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!f1 || !f2 || !fv1 || !fv2 || !valid1 || !valid2 || !tri_query_ok(q) || !matches12 || !nmatches) {
    m->err = "bad argument";
    return SWM_E_INVALID;
  }
  return match_triangulation_impl(m, FrameSrc{nullptr, f1}, fv1, valid1, FrameSrc{nullptr, f2}, fv2, valid2, q, check_ori,
                                  matches12, nmatches);
}

// ------------------------------------------------------------------------------ resident frames
int swm_frame_create(int device, swm_frame** out) {
  if (!out) return SWM_E_INVALID;
  *out = nullptr;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) { g_frame_create_error = err; return rc; }
  swm_frame* f = new swm_frame();
  f->device = device;
  if (cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&f->ready, cudaEventDisableTiming) != cudaSuccess) {
    g_frame_create_error = "cudaStreamCreate / cudaEventCreate failed";
    delete f;
    return SWM_E_CUDA;
  }
  *out = f;
  return SWM_OK;
}

void swm_frame_destroy(swm_frame* f) {
  if (!f) return;
  cudaSetDevice(f->device);
  if (f->ready) cudaEventSynchronize(f->ready);
  for (auto& b : f->b) b.release();
  f->bstage.release();
  if (f->h_counts) cudaFreeHost(f->h_counts);
  if (f->ready) cudaEventDestroy(f->ready);
  if (f->stream) cudaStreamDestroy(f->stream);
  delete f;
}

const char* swm_frame_last_error(const swm_frame* f) { return f ? f->err.c_str() : g_frame_create_error.c_str(); }

int32_t swm_frame_size(const swm_frame* f) { return f ? f->n : 0; }

int swm_camera_bounds(int device, const swm_camera* cam, int cols, int rows, float* bounds4) {
  if (!cam || !bounds4 || cols <= 0 || rows <= 0) return SWM_E_INVALID;
  if (cam->k1 == 0.0f) {  // Frame.cc:507-513
    bounds4[0] = 0.0f; bounds4[1] = (float)cols; bounds4[2] = 0.0f; bounds4[3] = (float)rows;
    return SWM_OK;
  }
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (device < 0 || device >= 64 || cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  const float corners[8] = {0.f, 0.f, (float)cols, 0.f, 0.f, (float)rows, (float)cols, (float)rows};  // Frame.cc:490-494
  StaticScratch& sc = g_static_scratch[device];
  std::lock_guard<std::mutex> lock(sc.mu);
  float* d = (float*)sc.reserve(64);
  if (!d) return SWM_E_CUDA;
  float m[8];
  bool ok = cudaMemcpy(d, corners, 32, cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok) {
    undistort_points_kernel<<<1, 32>>>(d, 4, camera_dev(cam), d + 8);
    ok = cudaMemcpy(m, d + 8, 32, cudaMemcpyDeviceToHost) == cudaSuccess;
  }
  if (!ok) return SWM_E_CUDA;
  bounds4[0] = std::min(m[0], m[4]);  // mnMinX = min(mat(0,0), mat(2,0))   Frame.cc:501-504
  bounds4[1] = std::max(m[2], m[6]);
  bounds4[2] = std::min(m[1], m[3]);
  bounds4[3] = std::max(m[5], m[7]);
  return SWM_OK;
}

int swm_frame_from_extractor(swm_frame* f, swm_orb* h, int index, const swm_camera* cam, const float* bounds4) {
  if (!f) return SWM_E_INVALID;
  if (!h || !bounds4 || !(bounds4[1] > bounds4[0]) || !(bounds4[3] > bounds4[2])) { f->err = "bad argument"; return SWM_E_INVALID; }
  OrbDeviceView v;
  int rc = orb_device_view(h, &v);
  if (rc != SWM_OK) { f->err = "the extractor holds no resident batch"; return rc; }
  if (index < 0 || index >= v.batch) { f->err = "frame index outside the extractor's last batch"; return SWM_E_INVALID; }
  if (v.device != f->device) { f->err = "extractor and frame live on different devices"; return SWM_E_INVALID; }
  FCK(f, cudaSetDevice(f->device));
  // the keypoint count is the only thing read back: it sizes the frame's arrays and later kernel grids
  int n = 0;
  FCK(f, cudaMemcpyAsync(&n, v.n + index, 4, cudaMemcpyDeviceToHost, v.stream));
  FCK(f, cudaStreamSynchronize(v.stream));
  if (n > v.cap) n = v.cap;
  if ((rc = frame_reserve(f, n, bounds4))) return rc;
  if (n > 0) {
    frame_from_kps_kernel<<<(n + 255) / 256, 256, 0, v.stream>>>(
        v.kps + (size_t)index * v.cap, reinterpret_cast<const uint4*>(v.desc + (size_t)index * v.cap * 32), n,
        camera_dev(cam), f->b[0].as<float>(), f->b[1].as<float>(), f->b[2].as<int32_t>(), f->b[3].as<float>(),
        f->b[4].as<uint4>());
    FCK(f, cudaGetLastError());
  }
  return frame_grid(f, v.stream);
}

int swm_frame_upload(swm_frame* f, const swm_frame_view* v) {
  if (!f) return SWM_E_INVALID;
  if (!frame_ok(v)) { f->err = "bad argument"; return SWM_E_INVALID; }
  FCK(f, cudaSetDevice(f->device));
  FCK(f, cudaEventSynchronize(f->ready));  // a previous build of this frame may still be in flight
  const float bounds[4] = {v->min_x, v->max_x, v->min_y, v->max_y};
  int rc;
  if ((rc = frame_reserve(f, v->n, bounds))) return rc;
  const size_t n = (size_t)v->n;
  if (n) {
    FCK(f, cudaMemcpyAsync(f->b[0].p, v->x, n * 4, cudaMemcpyHostToDevice, f->stream));
    FCK(f, cudaMemcpyAsync(f->b[1].p, v->y, n * 4, cudaMemcpyHostToDevice, f->stream));
    FCK(f, cudaMemcpyAsync(f->b[2].p, v->octave, n * 4, cudaMemcpyHostToDevice, f->stream));
    FCK(f, cudaMemcpyAsync(f->b[3].p, v->angle, n * 4, cudaMemcpyHostToDevice, f->stream));
    FCK(f, cudaMemcpyAsync(f->b[4].p, v->desc, n * 32, cudaMemcpyHostToDevice, f->stream));
  }
  if ((rc = frame_grid(f, f->stream))) return rc;
  FCK(f, cudaStreamSynchronize(f->stream));  // the host arrays may be pageable / reused by the caller
  return SWM_OK;
}

// Binary keyframe-feature slab (SURVEY section 8(f) rank 4): what travels instead of the Boost text archive of
// mvKeysUn + mDescriptors (code/src/MapUpdater.cc:192-230, code/include/KeyFrame.h:309-404).  Little-endian:
//   uint32 magic 'SWKF', uint32 version 1, int32 n, float min_x, max_x, min_y, max_y, uint32 reserved,
//   float x[n], float y[n], int32 octave[n], float angle[n], uint8 desc[n][32]        = 32 + 48 n bytes
// i.e. the resident frame's own arrays, so export is five device-to-host copies into the caller's buffer and import
// five host-to-device copies plus the grid kernel.
namespace {
struct SlabHeader {
  uint32_t magic, version;
  int32_t n;
  float min_x, max_x, min_y, max_y;
  uint32_t reserved;
};
static_assert(sizeof(SlabHeader) == 32, "slab header layout");
constexpr uint32_t kSlabMagic = 0x464B5753u;  // "SWKF"
}  // namespace

size_t swm_frame_slab_bytes(int32_t n) { return n < 0 ? 0 : sizeof(SlabHeader) + (size_t)n * 48; }

int swm_frame_export(swm_frame* f, uint8_t* buf, size_t cap, size_t* bytes) {
  if (!f) return SWM_E_INVALID;
  if (!buf || !bytes) { f->err = "bad argument"; return SWM_E_INVALID; }
  if (!f->dev.starts) { f->err = "frame has not been built"; return SWM_E_STATE; }
  const size_t n = (size_t)f->n, need = swm_frame_slab_bytes(f->n);
  *bytes = need;
  if (cap < need) { f->err = "slab buffer too small"; return SWM_E_CAPACITY; }
  FCK(f, cudaSetDevice(f->device));
  FCK(f, cudaEventSynchronize(f->ready));
  SlabHeader h{kSlabMagic, 1u, f->n, f->dev.min_x, f->dev.max_x, f->dev.min_y, f->dev.max_y, 0u};
  memcpy(buf, &h, sizeof(h));
  uint8_t* p = buf + sizeof(h);
  if (n) {
    FCK(f, cudaMemcpyAsync(p, f->b[0].p, n * 4, cudaMemcpyDeviceToHost, f->stream));
    FCK(f, cudaMemcpyAsync(p + n * 4, f->b[1].p, n * 4, cudaMemcpyDeviceToHost, f->stream));
    FCK(f, cudaMemcpyAsync(p + n * 8, f->b[2].p, n * 4, cudaMemcpyDeviceToHost, f->stream));
    FCK(f, cudaMemcpyAsync(p + n * 12, f->b[3].p, n * 4, cudaMemcpyDeviceToHost, f->stream));
    FCK(f, cudaMemcpyAsync(p + n * 16, f->b[4].p, n * 32, cudaMemcpyDeviceToHost, f->stream));
    FCK(f, cudaStreamSynchronize(f->stream));
  }
  return SWM_OK;
}

int swm_frame_import(swm_frame* f, const uint8_t* buf, size_t bytes) {
  if (!f) return SWM_E_INVALID;
  SlabHeader h;
  if (!buf || bytes < sizeof(h)) { f->err = "slab too short"; return SWM_E_INVALID; }
  memcpy(&h, buf, sizeof(h));
  if (h.magic != kSlabMagic || h.version != 1 || h.n < 0 || bytes < swm_frame_slab_bytes(h.n) || !(h.max_x > h.min_x) ||
      !(h.max_y > h.min_y)) {
    f->err = "not a version-1 keyframe slab";
    return SWM_E_INVALID;
  }
  const size_t n = (size_t)h.n;
  const uint8_t* p = buf + sizeof(h);
  swm_frame_view v;
  v.n = h.n;
  v.x = reinterpret_cast<const float*>(p);
  v.y = reinterpret_cast<const float*>(p + n * 4);
  v.octave = reinterpret_cast<const int32_t*>(p + n * 8);
  v.angle = reinterpret_cast<const float*>(p + n * 12);
  v.desc = p + n * 16;
  v.min_x = h.min_x; v.max_x = h.max_x; v.min_y = h.min_y; v.max_y = h.max_y;
  return swm_frame_upload(f, &v);
}

int swm_frame_download(swm_frame* f, float* x, float* y, int32_t* octave, float* angle, uint8_t* desc,
                       int32_t* grid_starts, int32_t* grid_items) {
  if (!f) return SWM_E_INVALID;
  FCK(f, cudaSetDevice(f->device));
  FCK(f, cudaEventSynchronize(f->ready));
  const size_t n = (size_t)f->n;
  if (n) {
    if (x) FCK(f, cudaMemcpy(x, f->b[0].p, n * 4, cudaMemcpyDeviceToHost));
    if (y) FCK(f, cudaMemcpy(y, f->b[1].p, n * 4, cudaMemcpyDeviceToHost));
    if (octave) FCK(f, cudaMemcpy(octave, f->b[2].p, n * 4, cudaMemcpyDeviceToHost));
    if (angle) FCK(f, cudaMemcpy(angle, f->b[3].p, n * 4, cudaMemcpyDeviceToHost));
    if (desc) FCK(f, cudaMemcpy(desc, f->b[4].p, n * 32, cudaMemcpyDeviceToHost));
  }
  if (grid_starts || grid_items) {
    if (!f->dev.starts) { f->err = "frame has not been built"; return SWM_E_STATE; }
    std::vector<int32_t> st((size_t)kCells + 1);
    FCK(f, cudaMemcpy(st.data(), f->dev.starts, st.size() * 4, cudaMemcpyDeviceToHost));
    if (grid_starts) memcpy(grid_starts, st.data(), st.size() * 4);
    if (grid_items && st[kCells] > 0)
      FCK(f, cudaMemcpy(grid_items, f->dev.items, (size_t)st[kCells] * 4, cudaMemcpyDeviceToHost));
  }
  return SWM_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Place-recognition shard
// ---------------------------------------------------------------------------------------------
struct swm_db {
  int device = 0;
  uint8_t* d_desc = nullptr;
  bool owns = false;
  long long ndesc = 0;
  int desc_per_kf = 1;
  long long first_kf = 0;
  unsigned long long* d_partial = nullptr;
  size_t partial_cap = 0;
  int n_sm = 148;
  // swm_db_query_sharded: this shard's (nq, k) key block and the all-gathered (world, nq, k) blocks, grow-only
  unsigned long long* d_exchange = nullptr;
  size_t exchange_cap = 0;
  // swm_db_query_peers: my exchange window (peers write into it) and the peers' windows as mapped here
  unsigned long long* d_window = nullptr;
  size_t window_bytes = 0;
  int peer_world = 0, peer_rank = -1, peer_nq_max = 0;
  unsigned int peer_seq = 0;
  unsigned long long* peer_win[16] = {};
  bool peer_ipc[16] = {};  // opened with cudaIpcOpenMemHandle (to be closed), as opposed to a same-process pointer
};

extern "C" {

int swm_db_create_device(int device, const uint8_t* d_desc, int64_t ndesc, int32_t desc_per_kf, int64_t first_kf_id,
                         swm_db** out) {
  if (!out || !d_desc || ndesc <= 0 || desc_per_kf <= 0) return SWM_E_INVALID;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  swm_db* db = new swm_db;
  db->device = device;
  db->d_desc = const_cast<uint8_t*>(d_desc);
  db->ndesc = ndesc;
  db->desc_per_kf = desc_per_kf;
  db->first_kf = first_kf_id;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) db->n_sm = prop.multiProcessorCount;
  *out = db;
  return SWM_OK;
}

int swm_db_create(int device, const uint8_t* desc, int64_t ndesc, int32_t desc_per_kf, int64_t first_kf_id,
                  swm_db** out) {
  if (!out || !desc || ndesc <= 0 || desc_per_kf <= 0) return SWM_E_INVALID;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  uint8_t* d = nullptr;
  if (cudaMalloc(&d, (size_t)ndesc * 32) != cudaSuccess) return SWM_E_CUDA;
  if (cudaMemcpy(d, desc, (size_t)ndesc * 32, cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(d);
    return SWM_E_CUDA;
  }
  rc = swm_db_create_device(device, d, ndesc, desc_per_kf, first_kf_id, out);
  if (rc != SWM_OK) {
    cudaFree(d);
    return rc;
  }
  (*out)->owns = true;
  return SWM_OK;
}

void swm_db_destroy(swm_db* db) {
  if (!db) return;
  cudaSetDevice(db->device);
  if (db->owns) cudaFree(db->d_desc);
  cudaFree(db->d_partial);
  cudaFree(db->d_exchange);
  for (int r = 0; r < 16; r++)
    if (db->peer_ipc[r] && db->peer_win[r]) cudaIpcCloseMemHandle(db->peer_win[r]);
  cudaFree(db->d_window);
  delete db;
}

int64_t swm_db_size(const swm_db* db) { return db ? db->ndesc : 0; }

// Measured int8 rate of the tensor pipe: `iters` back-to-back tcgen05 kind::i8 MMAs per SM (see umma::i8_peak_kernel).
int swm_i8_peak(int device, int mode, int iters, double* tops) {
  if (!tops || iters < 16 || (mode != 0 && mode != 1)) return SWM_E_INVALID;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) return rc;
  if (cudaSetDevice(device) != cudaSuccess) return SWM_E_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return SWM_E_CUDA;
  const int ctas = prop.multiProcessorCount;
  cudaEvent_t e0, e1;
  if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return SWM_E_CUDA;
  umma::i8_peak_kernel<<<ctas, 128, umma::kPeakSmem>>>(mode, 64, nullptr);  // warm-up
  cudaEventRecord(e0);
  umma::i8_peak_kernel<<<ctas, 128, umma::kPeakSmem>>>(mode, iters, nullptr);
  cudaEventRecord(e1);
  const bool ok = cudaEventSynchronize(e1) == cudaSuccess && cudaGetLastError() == cudaSuccess;
  float ms = 0.f;
  if (ok) cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (!ok || ms <= 0.f) return SWM_E_CUDA;
  const double n = mode == 0 ? 64.0 : 256.0;
  *tops = (double)ctas * iters * 2.0 * 128.0 * n * 32.0 / (ms * 1e-3) / 1e12;
  return SWM_OK;
}

}  // extern "C"

// The shard scan: slices x query blocks of one of the three top-2 kernels into db->d_partial ([parts][nq][2] keys).
static int db_scan(swm_db* db, const uint8_t* d_q, int nq, cudaStream_t st, long long* parts_out) {
  // Three kernels produce identical keys.  Default: tcgen05 int8 (db_umma.cuh).  SWM_DB_KERNEL=imma selects the
  // legacy mma.sync kernel, SWM_DB_KERNEL=popc the CUDA-core LOP3+POPC kernel; both are kept as A/B baselines for
  // profiles/ and as independent implementations the parity tests cross-check.
  const int kind = [] {  // read per call so that one process can cross-check the three kernels
    const char* e = getenv("SWM_DB_KERNEL");
    if (e && !strcmp(e, "popc")) return 2;
    if (e && !strcmp(e, "imma")) return 1;
    return 0;
  }();
  const int tile = kind == 2 ? kDbTile : kind == 1 ? kMmaTile : umma::kTileN;
  const int qper = kind == 2 ? kDbQPerCta : kind == 1 ? kMmaQPerCta : umma::kQPerCta;
  const long long tiles = (db->ndesc + tile - 1) / tile;
  const int qblocks = (nq + qper - 1) / qper;
  // enough database slices that slices x query blocks fills the machine a few times over
  long long parts = std::max<long long>(1, (long long)db->n_sm * (kind == 0 ? 2 : 8) / qblocks);
  parts = std::min<long long>(parts, tiles);
  int tiles_per_cta = (int)((tiles + parts - 1) / parts);
  if (kind != 2) tiles_per_cta = std::min(tiles_per_cta, (1 << 20) / tile);  // 20-bit in-slice index
  parts = (tiles + tiles_per_cta - 1) / tiles_per_cta;
  const size_t need = (size_t)parts * nq * 2 * sizeof(unsigned long long);
  if (need > db->partial_cap) {
    cudaFree(db->d_partial);
    db->d_partial = nullptr;
    db->partial_cap = 0;
    if (cudaMalloc(&db->d_partial, need) != cudaSuccess) return SWM_E_CUDA;
    db->partial_cap = need;
  }
  const long long first_index = db->first_kf * db->desc_per_kf;
  dim3 grid((unsigned)parts, qblocks);
  if (kind == 2) {
    db_top2_kernel<<<grid, kDbQPerCta, 0, st>>>((const uint4*)db->d_desc, db->ndesc, first_index, (const uint4*)d_q, nq,
                                                tiles_per_cta, db->d_partial);
  } else if (kind == 1) {
    db_top2_mma_kernel<<<grid, 256, 0, st>>>((const uint4*)db->d_desc, db->ndesc, first_index, (const uint32_t*)d_q, nq,
                                             tiles_per_cta, db->d_partial);
  } else {
    if (cudaFuncSetAttribute(umma::db_top2_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             umma::kSmemBytes) != cudaSuccess)
      return SWM_E_CUDA;
    umma::db_top2_umma_kernel<<<grid, umma::kThreads, umma::kSmemBytes, st>>>(
        (const uint4*)db->d_desc, db->ndesc, first_index, (const uint4*)d_q, nq, tiles_per_cta, db->d_partial);
  }
  *parts_out = parts;
  return cudaGetLastError() == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

extern "C" {

int swm_db_query_device(swm_db* db, const uint8_t* d_q, int nq, int k, uint64_t* d_topk, int32_t* d_votes,
                        int th_votes, void* stream) {
  if (!db || !d_q || nq <= 0 || k < 1 || k > 2 || !d_topk) return SWM_E_INVALID;
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  cudaStream_t st = (cudaStream_t)stream;
  long long parts = 0;
  const int rc = db_scan(db, d_q, nq, st, &parts);
  if (rc != SWM_OK) return rc;
  const long long first_index = db->first_kf * db->desc_per_kf;
  const long long n_kf = (db->ndesc + db->desc_per_kf - 1) / db->desc_per_kf;
  db_merge_kernel<<<(nq + 127) / 128, 128, 0, st>>>(db->d_partial, (int)parts, nq, 2, k, (unsigned long long*)d_topk,
                                                    d_votes, th_votes, db->first_kf, db->desc_per_kf, first_index, n_kf);
  return cudaGetLastError() == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

// ---- peer-memory exchange (see db_merge_peers_kernel)
static size_t peer_window_bytes(int world, int nq_max) {
  return (size_t)2 * world * nq_max * 2 * sizeof(unsigned long long) + (size_t)2 * world * kPeerBlocks * sizeof(unsigned int);
}

int swm_db_peer_window(swm_db* db, int world, int nq_max, void* ipc_handle64, void** window) {
  if (!db || world < 1 || world > kPeerMaxWorld || nq_max < 1 || nq_max > 128 * kPeerBlocks) return SWM_E_INVALID;
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  for (int r = 0; r < 16; r++) {
    if (db->peer_ipc[r] && db->peer_win[r]) cudaIpcCloseMemHandle(db->peer_win[r]);
    db->peer_win[r] = nullptr;
    db->peer_ipc[r] = false;
  }
  cudaFree(db->d_window);
  db->d_window = nullptr;
  db->peer_world = 0;
  db->peer_rank = -1;
  const size_t bytes = peer_window_bytes(world, nq_max);
  if (cudaMalloc(&db->d_window, bytes) != cudaSuccess) return SWM_E_CUDA;
  if (cudaMemset(db->d_window, 0, bytes) != cudaSuccess) return SWM_E_CUDA;  // flags start at 0; sequence numbers start at 1
  db->window_bytes = bytes;
  db->peer_nq_max = nq_max;
  db->peer_world = world;
  db->peer_seq = 0;
  if (ipc_handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the handle is exchanged as 64 opaque bytes");
    cudaIpcMemHandle_t hdl;
    if (cudaIpcGetMemHandle(&hdl, db->d_window) != cudaSuccess) return SWM_E_CUDA;
    memcpy(ipc_handle64, &hdl, 64);
  }
  if (window) *window = db->d_window;
  return SWM_OK;
}

int swm_db_peer_open(swm_db* db, int rank, const void* ipc_handles, void* const* windows) {
  if (!db || !db->d_window || rank < 0 || rank >= db->peer_world || (!ipc_handles && !windows)) return SWM_E_INVALID;
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  for (int r = 0; r < db->peer_world; r++) {
    if (r == rank) {
      db->peer_win[r] = db->d_window;
    } else if (windows) {  // same process (tests, a server that drives several GPUs from one process)
      db->peer_win[r] = static_cast<unsigned long long*>(windows[r]);
    } else {
      cudaIpcMemHandle_t hdl;
      memcpy(&hdl, static_cast<const char*>(ipc_handles) + 64 * (size_t)r, 64);
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, hdl, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) return SWM_E_CUDA;
      db->peer_win[r] = static_cast<unsigned long long*>(p);
      db->peer_ipc[r] = true;
    }
    if (!db->peer_win[r]) return SWM_E_INVALID;
  }
  db->peer_rank = rank;
  return SWM_OK;
}

int swm_db_query_peers(swm_db* db, const uint8_t* d_q, int nq, int k, uint64_t* d_topk, int32_t* d_votes, int th_votes,
                       void* stream) {
  if (!db || !d_q || nq <= 0 || k < 1 || k > 2 || !d_topk) return SWM_E_INVALID;
  if (db->peer_rank < 0 || nq > db->peer_nq_max) return SWM_E_STATE;
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  cudaStream_t st = (cudaStream_t)stream;
  long long parts = 0;
  const int rc = db_scan(db, d_q, nq, st, &parts);
  if (rc != SWM_OK) return rc;
  PeerWindows win;
  for (int r = 0; r < kPeerMaxWorld; r++) win.keys[r] = r < db->peer_world ? db->peer_win[r] : nullptr;
  const long long first_index = db->first_kf * db->desc_per_kf;
  const long long n_kf = (db->ndesc + db->desc_per_kf - 1) / db->desc_per_kf;
  db->peer_seq++;
  db_merge_peers_kernel<<<(nq + 127) / 128, 128, 0, st>>>(db->d_partial, (int)parts, nq, k, win, db->peer_rank, db->peer_world,
                                                          db->peer_nq_max, db->peer_seq, (unsigned long long*)d_topk, d_votes,
                                                          th_votes, db->desc_per_kf, first_index, n_kf);
  return cudaGetLastError() == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

int swm_db_merge_gathered(swm_db* db, const uint64_t* d_gathered, int world, int nq, int k, uint64_t* d_topk,
                          int32_t* d_votes, int th_votes, void* stream) {
  if (!db || !d_gathered || world < 1 || nq <= 0 || k < 1 || k > 2 || !d_topk) return SWM_E_INVALID;
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  const long long first_index = db->first_kf * db->desc_per_kf;
  const long long n_kf = (db->ndesc + db->desc_per_kf - 1) / db->desc_per_kf;
  db_merge_kernel<<<(nq + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_gathered, world, nq, k, k,
                                                                      (unsigned long long*)d_topk, d_votes, th_votes,
                                                                      db->first_kf, db->desc_per_kf, first_index, n_kf);
  return cudaGetLastError() == cudaSuccess ? SWM_OK : SWM_E_CUDA;
}

}  // extern "C"

// ---- NCCL, bound at first use: libswm_orb.so does not link libnccl (a host process -- SwarmMap's server, or a
// PyTorch rank -- has its own copy loaded; binding to that one avoids two NCCL runtimes in one process).
namespace {
using nccl_allgather_fn = int (*)(const void*, void*, size_t, int, void*, cudaStream_t);
constexpr int kNcclUint64 = 5;  // ncclDataType_t::ncclUint64 (nccl.h)
nccl_allgather_fn bind_nccl_allgather() {
  static nccl_allgather_fn fn = [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // already in the process?
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    void* sym = h ? dlsym(h, "ncclAllGather") : dlsym(RTLD_DEFAULT, "ncclAllGather");
    return reinterpret_cast<nccl_allgather_fn>(sym);
  }();
  return fn;
}
}  // namespace

extern "C" {

// Config 5 end to end on one rank, callable from a C++ server (the role of AgentMediator::CheckOverlapCandidates,
// code/src/AgentMediator.cc:140-202): brute-force top-k of the queries against this shard, ONE ncclAllGather of the
// fixed-size (nq, k) key blocks over NVLink, and the merge kernel that also casts this shard's votes from the GLOBAL
// best matches -- three enqueues on `stream`, no host synchronisation.  nccl_comm is an ncclComm_t whose rank owns
// this shard; world = its size.  d_topk: (nq, k) merged keys, identical on every rank.
int swm_db_query_sharded(swm_db* db, void* nccl_comm, int world, const uint8_t* d_q, int nq, int k, uint64_t* d_topk,
                         int32_t* d_votes, int th_votes, void* stream) {
  if (!db || !d_q || nq <= 0 || k < 1 || k > 2 || !d_topk || world < 1 || (world > 1 && !nccl_comm)) return SWM_E_INVALID;
  if (world == 1) return swm_db_query_device(db, d_q, nq, k, d_topk, d_votes, th_votes, stream);
  if (cudaSetDevice(db->device) != cudaSuccess) return SWM_E_CUDA;
  const size_t block = (size_t)nq * k;
  const size_t need = block * ((size_t)world + 1) * sizeof(unsigned long long);
  if (need > db->exchange_cap) {
    cudaFree(db->d_exchange);
    db->d_exchange = nullptr;
    db->exchange_cap = 0;
    if (cudaMalloc(&db->d_exchange, need) != cudaSuccess) return SWM_E_CUDA;
    db->exchange_cap = need;
  }
  nccl_allgather_fn allgather = bind_nccl_allgather();
  if (!allgather) return SWM_E_STATE;  // no NCCL in this process and none on the library path
  unsigned long long* local = db->d_exchange;
  unsigned long long* gathered = db->d_exchange + block;
  int rc = swm_db_query_device(db, d_q, nq, k, (uint64_t*)local, nullptr, th_votes, stream);
  if (rc != SWM_OK) return rc;
  if (allgather(local, gathered, block, kNcclUint64, nccl_comm, (cudaStream_t)stream) != 0) return SWM_E_CUDA;
  return swm_db_merge_gathered(db, (const uint64_t*)gathered, world, nq, k, d_topk, d_votes, th_votes, stream);
}

}  // extern "C"

namespace swm {
int frame_device_view(const swm_frame* f, FrameDeviceView* out) {
  if (!f || !out) return SWM_E_INVALID;
  out->desc = f->dev.desc;
  out->n = f->n;
  out->device = f->device;
  out->ready = f->ready;
  return SWM_OK;
}
}  // namespace swm

#include "mappoints.cuh"
#include "match_batch.cuh"
