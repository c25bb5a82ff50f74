// match_batch.cuh -- throughput form of the matchers: P independent matching problems ("jobs") per call.
// Included at the end of match.cu (same translation unit: it reuses the row / resolve device bodies).
//
// One agent's tracking thread calls a Search* once per frame; a GPU serving many agents (or replaying recorded
// streams) has hundreds of such problems in flight.  A batch call packs the host arrays of ALL jobs into one pinned
// arena (one H2D copy), runs SIX launches whatever the number of jobs --
//   prepare   (CTA per job: target grid if the frame came as host arrays; SearchForInitialization's source rows;
//              SearchByBoW's merge-walk of the two FeatureVectors and its row layout, ORBmatcher.cc:166-241,:507-581)
//   count     (warp per source row: size of its GetFeaturesInArea window)
//   scan      (CTA per job: row starts)
//   offsets   (one CTA: where each job's candidates start in the shared candidate buffer)
//   fill      (warp per row: candidate index + Hamming distance, in the reference's enumeration order)
//   resolve   (CTA per job: the greedy accept / steal / overwrite order replayed, rotation histogram, pruning)
// -- and brings every result back with one D2H copy and one synchronisation.  The candidate buffer is sized from
// earlier calls; if a batch needs more, the device raises a flag instead of writing, and the call is repeated once
// with a larger buffer (no host synchronisation in the middle of a call in the steady state).
// Results are identical to the single-job entry points (same device bodies) and to the oracle.
#pragma once

namespace swm {

enum { kJobWindow = 0, kJobInit = 1, kJobBowFrame = 2, kJobBowKf = 3 };

struct BatchJob {
  int kind;
  int n1, n2;
  FrameDev f1;          // source frame (init, bow)
  FrameDev f2;          // target frame; starts / items point at grid2 when that is set
  int32_t* grid2;       // != NULL: build the target's grid here first (starts | items | cell_of)
  WindowDev q;          // window: uploaded; init: views of the iq_* arrays below
  float *iq_u, *iq_v, *iq_r;
  int32_t* iq_l;
  uint8_t* iq_valid;
  const float* prev_in;
  float window;
  const uint32_t *ids1, *feats1, *ids2, *feats2;  // bow: the two FeatureVectors as CSR
  const int32_t *off1, *off2;
  int nn1, nn2;
  const uint8_t* valid1;
  int32_t* node_scratch;  // 2 * (nn1 + 1)
  int rows_cap;
  int32_t* row_count;     // rows_cap + 1
  int32_t* row_start;     // rows_cap + 2, relative to the job's candidate base
  int32_t* row_src;       // bow
  int32_t* row_aux;       // bow: start of the row's candidate span in feats2
  ResolveArgs ra;
};

struct BatchCtl {
  int32_t cand_cap, cand_total, overflow, bad_index;
};

// Exclusive block scan of v[0..n) (n arbitrary) by 1024 threads, in place; returns the total to every thread.
__device__ __forceinline__ int block_exscan_1024(int32_t* v, int n, int* s_part) {
  const int tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int b = min(tid * per, n), e = min(b + per, n);
  int local = 0;
  for (int i = b; i < e; i++) local += v[i];
  s_part[tid] = local;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int x = tid >= o ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += x;
    __syncthreads();
  }
  int run = s_part[tid] - local;
  for (int i = b; i < e; i++) {
    const int x = v[i];
    v[i] = run;
    run += x;
  }
  const int total = s_part[1023];
  __syncthreads();
  return total;
}

// SearchByBoW's walk over the two sorted FeatureVectors, per job: a node of fv1 contributes rows iff fv2 has the same
// node id; rows = its valid features in list order; every row's candidates = the node's features in fv2.
__device__ __forceinline__ void bow_rows_body(const BatchJob& J, int32_t* job_total, int32_t* job_rows, BatchCtl* ctl,
                                              int* s_part) {
  const int tid = threadIdx.x;
  int32_t* nrows = J.node_scratch;            // rows per node, then their exclusive scan
  int32_t* ncand = J.node_scratch + J.nn1 + 1;  // candidates per node (rows * len2), then their exclusive scan
  for (int a = tid; a < J.nn1; a += 1024) {
    const uint32_t id = J.ids1[a];
    int lo = 0, hi = J.nn2 - 1, b = -1;
    while (lo <= hi) {
      const int mid = (lo + hi) >> 1;
      const uint32_t v = J.ids2[mid];
      if (v == id) { b = mid; break; }
      if (v < id) lo = mid + 1; else hi = mid - 1;
    }
    int nv = 0;
    if (b >= 0) {
      for (int k = J.off1[a]; k < J.off1[a + 1]; k++) {
        const uint32_t i1 = J.feats1[k];
        if (i1 >= (uint32_t)J.n1) { ctl->bad_index = 1; continue; }
        nv += J.valid1[i1] ? 1 : 0;
      }
    }
    nrows[a] = nv;
    ncand[a] = b >= 0 ? nv * (J.off2[b + 1] - J.off2[b]) : 0;
  }
  __syncthreads();
  const int R = block_exscan_1024(nrows, J.nn1, s_part);
  const int T = block_exscan_1024(ncand, J.nn1, s_part);
  for (int a = tid; a < J.nn1; a += 1024) {
    const int r_end = a + 1 < J.nn1 ? nrows[a + 1] : R;
    int r = nrows[a];
    if (r == r_end) continue;
    const uint32_t id = J.ids1[a];
    int lo = 0, hi = J.nn2 - 1, b = -1;
    while (lo <= hi) {
      const int mid = (lo + hi) >> 1;
      const uint32_t v = J.ids2[mid];
      if (v == id) { b = mid; break; }
      if (v < id) lo = mid + 1; else hi = mid - 1;
    }
    const int len2 = J.off2[b + 1] - J.off2[b];
    int c = ncand[a];
    for (int k = J.off1[a]; k < J.off1[a + 1]; k++) {
      const uint32_t i1 = J.feats1[k];
      if (i1 >= (uint32_t)J.n1 || !J.valid1[i1]) continue;
      J.row_src[r] = (int32_t)i1;
      J.row_start[r] = c;
      J.row_aux[r] = J.off2[b];
      r++;
      c += len2;
    }
  }
  if (tid == 0) {
    J.row_start[R] = T;
    job_rows[blockIdx.x] = R;
    job_total[blockIdx.x] = T;
  }
}

__global__ void __launch_bounds__(1024) bq_prepare_kernel(const BatchJob* __restrict__ jobs, int32_t* job_total,
                                                          int32_t* job_rows, BatchCtl* ctl) {
  __shared__ int s_part[1024];
  const BatchJob& J = jobs[blockIdx.x];
  const int tid = threadIdx.x;
  if (J.grid2) {
    const int nn = J.n2 > 0 ? J.n2 : 1;
    grid_build_body(J.f2, J.grid2, J.grid2 + kCells + 1, J.grid2 + kCells + 1 + nn + 4);
    __syncthreads();
  }
  if (J.kind == kJobInit) {  // ORBmatcher.cc:390-396
    for (int i = tid; i < J.n1; i += 1024) {
      const int oct = J.f1.octave[i];
      J.iq_u[i] = J.prev_in[2 * i];
      J.iq_v[i] = J.prev_in[2 * i + 1];
      J.iq_r[i] = J.window;
      J.iq_l[i] = oct;
      J.iq_valid[i] = oct > 0 ? 0 : 1;
    }
  }
  if (J.kind >= kJobBowFrame) bow_rows_body(J, job_total, job_rows, ctl, s_part);
  else if (tid == 0) job_rows[blockIdx.x] = J.q.m;
}

__global__ void __launch_bounds__(256) bq_count_kernel(const BatchJob* __restrict__ jobs) {
  const BatchJob& J = jobs[blockIdx.y];
  if (J.kind >= kJobBowFrame) return;
  window_rows_body(J.f2, J.q, 0, J.row_count, nullptr, nullptr, nullptr);
}

__global__ void __launch_bounds__(1024) bq_scan_kernel(const BatchJob* __restrict__ jobs, int32_t* job_total) {
  __shared__ int s_part[1024];
  const BatchJob& J = jobs[blockIdx.x];
  if (J.kind >= kJobBowFrame) return;
  const int m = J.q.m;
  for (int i = threadIdx.x; i < m; i += 1024) J.row_start[i] = J.row_count[i];
  __syncthreads();
  const int total = block_exscan_1024(J.row_start, m, s_part);
  if (threadIdx.x == 0) {
    J.row_start[m] = total;
    job_total[blockIdx.x] = total;
  }
}

__global__ void __launch_bounds__(1024) bq_offsets_kernel(const int32_t* __restrict__ job_total, int njobs,
                                                          int32_t* job_base, BatchCtl* ctl) {
  __shared__ int s_part[1024];
  for (int i = threadIdx.x; i < njobs; i += 1024) job_base[i] = job_total[i];
  __syncthreads();
  const int total = block_exscan_1024(job_base, njobs, s_part);
  if (threadIdx.x == 0) {
    job_base[njobs] = total;
    ctl->cand_total = total;
    ctl->overflow = total > ctl->cand_cap ? 1 : 0;
  }
}

__global__ void __launch_bounds__(256) bq_fill_kernel(const BatchJob* __restrict__ jobs, const int32_t* __restrict__ job_base,
                                                      const int32_t* __restrict__ job_rows, BatchCtl* ctl,
                                                      int32_t* __restrict__ cand_idx, uint32_t* __restrict__ cand_val) {
  if (ctl->overflow) return;
  const BatchJob& J = jobs[blockIdx.y];
  const int base = job_base[blockIdx.y];
  if (J.kind < kJobBowFrame) {
    window_rows_body(J.f2, J.q, 1, J.row_count, J.row_start, cand_idx + base, cand_val + base);
    return;
  }
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= job_rows[blockIdx.y]) return;
  const int s = J.row_src[r];
  const uint4 d0 = __ldg(J.f1.desc + 2 * s), d1 = __ldg(J.f1.desc + 2 * s + 1);
  const int c0 = J.row_start[r], len = J.row_start[r + 1] - c0, src = J.row_aux[r];
  for (int c = lane; c < len; c += 32) {
    uint32_t j = J.feats2[src + c];
    if (j >= (uint32_t)J.n2) { ctl->bad_index = 1; j = 0; }
    cand_idx[base + c0 + c] = (int32_t)j;
    cand_val[base + c0 + c] = ((uint32_t)J.f2.octave[j] << 16) | (uint32_t)ham256(d0, d1, J.f2.desc + 2 * j);
  }
}

__global__ void __launch_bounds__(kResolveWarps * 32) bq_resolve_kernel(const BatchJob* __restrict__ jobs,
                                                                       const int32_t* __restrict__ job_base,
                                                                       const int32_t* __restrict__ job_rows,
                                                                       const BatchCtl* __restrict__ ctl,
                                                                       const int32_t* __restrict__ cand_idx,
                                                                       const uint32_t* __restrict__ cand_val) {
  __shared__ ResolveArgs s_a;
  if (ctl->overflow || ctl->bad_index) return;
  const int tid = threadIdx.x;
  const int* src = reinterpret_cast<const int*>(&jobs[blockIdx.x].ra);
  for (int i = tid; i < (int)(sizeof(ResolveArgs) / 4); i += blockDim.x) reinterpret_cast<int*>(&s_a)[i] = src[i];
  __syncthreads();
  if (tid == 0) {
    s_a.cand_idx = cand_idx + job_base[blockIdx.x];
    s_a.cand_val = cand_val + job_base[blockIdx.x];
    s_a.rows = job_rows[blockIdx.x];
  }
  if (s_a.check_ori)
    for (int i = tid; i < s_a.n1; i += blockDim.x) s_a.ev_bin[i] = -1;
  __syncthreads();
  resolve_body(s_a);
}

// Resident frames for a whole extractor batch: Frame::UndistortKeyPoints + SoA split + AssignFeaturesToGrid, one
// launch each for all frames; the keypoint counts stay on the device until the single read-back at the end.
struct FrameBuildDev {
  const swm_keypoint* kps;
  const uint4* desc_in;
  const int32_t* n_ptr;
  int cap;
  float *x, *y, *angle;
  int32_t* octave;
  uint4* desc_out;
  FrameDev dev;     // n filled on the device
  int32_t* grid;    // starts | items | cell_of
};

__global__ void __launch_bounds__(256) frames_from_kps_kernel(const FrameBuildDev* __restrict__ fb, CameraDev cam) {
  const FrameBuildDev& F = fb[blockIdx.y];
  const int n = min(*F.n_ptr, F.cap);
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const swm_keypoint kp = F.kps[i];
  float ux = kp.x, uy = kp.y;
  if (cam.distorted) undistort_point(cam, kp.x, kp.y, &ux, &uy);
  F.x[i] = ux;
  F.y[i] = uy;
  F.octave[i] = kp.octave;
  F.angle[i] = kp.angle;
  F.desc_out[2 * i] = F.desc_in[2 * i];
  F.desc_out[2 * i + 1] = F.desc_in[2 * i + 1];
}

__global__ void __launch_bounds__(1024) frames_grid_kernel(const FrameBuildDev* __restrict__ fb) {
  const FrameBuildDev& F = fb[blockIdx.x];
  FrameDev f = F.dev;
  f.n = min(*F.n_ptr, F.cap);
  grid_build_body(f, F.grid, F.grid + kCells + 1, F.grid + kCells + 1 + F.cap + 4);
}

}  // namespace swm

namespace {

using namespace swm;

// A projection job (swm_match_local_map*): the caller's job, its table and the level thresholds of its scale table.
// `wq` carries only the number of sources; lm_project_kernel writes the query rows on the device.
struct LocalMapHost {
  swm_localmap_job* job;
  swm_mappoints* table;
  swm_window_query wq;
  float thr[SWM_MAX_LEVELS];
  size_t off_track = 0;
};

// One matching problem as the entry points hand it over.
struct HostJob {
  int kind = kJobWindow;
  FrameSrc f1{nullptr, nullptr}, f2{nullptr, nullptr};
  const swm_window_query* wq = nullptr;
  const uint8_t* tgt_blocked = nullptr;
  int th_dist = 0, ratio_mode = 0;
  float* prev_xy = nullptr;
  int window = 0;
  const swm_featvec *fv1 = nullptr, *fv2 = nullptr;
  const uint8_t *valid1 = nullptr, *valid2 = nullptr;
  float nnratio = 0.f;
  int check_ori = 0;
  int32_t* out = nullptr;
  int32_t* nmatches = nullptr;
  LocalMapHost* lm = nullptr;
  // filled by run_batch
  size_t off_out = 0, off_n = 0, off_prev = 0;
  int n_out = 0;
};

struct Packer {  // bump allocator over the matcher's upload arena: host copy in, device address out
  // (Spreading the copies over helper threads was measured: spawning them costs more than the ~1 ms of memcpy a
  // 128-job batch needs -- 2.3 ms vs 1.4 ms per call -- so packing stays on the calling thread.)
  swm_matcher* m;
  bool overflow = false;
  size_t reserve(size_t bytes) {
    const size_t off = (m->arena_used + 255) & ~(size_t)255;
    if (off + bytes > m->arena_cap) { overflow = true; return 0; }
    m->arena_used = off + bytes;
    return off;
  }
  template <typename T>
  T* put(const void* src, size_t bytes) {
    const size_t off = reserve(bytes);
    if (overflow) return nullptr;
    if (bytes && src) memcpy(m->h_arena + off, src, bytes);
    return reinterpret_cast<T*>(m->d_arena + off);
  }
};

struct Carver {  // bump allocator over device scratch
  uint8_t* base;
  size_t used = 0;
  template <typename T>
  T* take(size_t count) {
    used = (used + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
    used += count * sizeof(T);
    return p;
  }
};

size_t up256b(size_t n) { return (n + 255) & ~(size_t)255; }

FrameDev frame_dev_from_host(Packer& pk, const swm_frame_view* f) {
  FrameDev d{};
  const size_t n = (size_t)f->n;
  d.n = f->n;
  d.x = pk.put<float>(f->x, n * 4);
  d.y = pk.put<float>(f->y, n * 4);
  d.octave = pk.put<int32_t>(f->octave, n * 4);
  d.angle = pk.put<float>(f->angle, n * 4);
  d.desc = pk.put<uint4>(f->desc, n * 32);
  d.min_x = f->min_x; d.min_y = f->min_y; d.max_x = f->max_x; d.max_y = f->max_y;
  d.inv_w = (float)kGridCols / (float)(f->max_x - f->min_x);
  d.inv_h = (float)kGridRows / (float)(f->max_y - f->min_y);
  return d;
}

size_t featvec_bytes(const swm_featvec* fv) {
  const size_t nn = (size_t)fv->n_nodes;
  return up256b(nn * 4) + up256b((nn + 1) * 4) + up256b((size_t)(nn ? fv->offsets[nn] : 0) * 4) + 256;
}

// A projection job's device record: its operands packed into the arena, its query rows carved from the scratch (the
// projection kernel writes them), its tracking fields pointed into the in/out region that comes back with the results.
LocalMapDev lm_dev(swm_matcher* m, Packer& pk, Carver& cv, const LocalMapHost& h, int n2, int check_ori, size_t off_n) {
  const swm_localmap_job& w = *h.job;
  const size_t M = (size_t)h.wq.m;
  LocalMapDev L;
  memset(&L, 0, sizeof(L));
  L.mode = w.mode;
  L.m = (int)M;
  L.n2 = n2;
  L.nlevels = w.proj->nlevels;
  L.rows = pk.put<int32_t>(w.rows, M * 4);
  L.frame_rows = w.frame_rows ? pk.put<int32_t>(w.frame_rows, (size_t)n2 * 4) : nullptr;
  L.nwords = (h.table->size + 31) / 32;
  L.seen = w.mode == SWM_LOCALMAP_POINTS ? cv.take<uint32_t>((size_t)L.nwords) : nullptr;
  L.t = h.table->view();
  memcpy(L.T, w.proj->Tcw, sizeof(L.T));
  L.fx = w.proj->fx; L.fy = w.proj->fy; L.cx = w.proj->cx; L.cy = w.proj->cy;
  const FrameDev& d = w.tgt->dev;
  L.min_x = d.min_x; L.max_x = d.max_x; L.min_y = d.min_y; L.max_y = d.max_y;
  L.th = w.th;
  for (int k = 0; k < L.nlevels; k++) L.sf[k] = w.proj->scale_factors[k];
  for (int k = 0; k + 1 < L.nlevels; k++) L.thr[k] = h.thr[k];
  if (w.mode == SWM_LOCALMAP_LAST) {
    L.last_octave = w.last->dev.octave;
    L.last_angle = w.last->dev.angle;
  }
  L.u = cv.take<float>(M); L.v = cv.take<float>(M); L.radius = cv.take<float>(M);
  L.min_level = cv.take<int32_t>(M); L.max_level = cv.take<int32_t>(M);
  L.valid = cv.take<uint8_t>(M); L.blocks = cv.take<uint8_t>(M);
  L.desc = cv.take<uint4>(2 * M);
  L.angle = check_ori ? cv.take<float>(M) : nullptr;
  L.tgt_blocked = cv.take<uint8_t>((size_t)n2);
  if (w.track) {
    uint8_t* base = m->d_arena + h.off_track;
    const size_t o1 = up256b(M), o4 = up256b(M * 4);
    L.t_in_view = w.track->in_view ? base : nullptr;
    L.t_u = w.track->u ? reinterpret_cast<float*>(base + o1) : nullptr;
    L.t_v = w.track->v ? reinterpret_cast<float*>(base + o1 + o4) : nullptr;
    L.t_cos = w.track->view_cos ? reinterpret_cast<float*>(base + o1 + 2 * o4) : nullptr;
    L.t_level = w.track->level ? reinterpret_cast<int32_t*>(base + o1 + 3 * o4) : nullptr;
  }
  L.n_to_match = reinterpret_cast<int32_t*>(m->d_arena + off_n) + 2;
  return L;
}

void lm_finish(const LocalMapHost& h, const uint8_t* down, size_t off_n) {
  swm_localmap_job& w = *h.job;
  w.n_to_match = reinterpret_cast<const int32_t*>(down + off_n)[2];
  const swm_track_out* tr = w.track;
  if (!tr) return;
  const size_t M = (size_t)h.wq.m, o1 = up256b(M), o4 = up256b(M * 4);
  const uint8_t* base = down + h.off_track;
  if (tr->in_view) memcpy(tr->in_view, base, M);
  if (tr->u) memcpy(tr->u, base + o1, M * 4);
  if (tr->v) memcpy(tr->v, base + o1 + o4, M * 4);
  if (tr->view_cos) memcpy(tr->view_cos, base + o1 + 2 * o4, M * 4);
  if (tr->level) memcpy(tr->level, base + o1 + 3 * o4, M * 4);
}

// Runs the jobs that need the device (the callers have already answered the trivial ones).
int run_batch(swm_matcher* m, std::vector<HostJob>& jobs) {
  const int P = (int)jobs.size();
  if (P == 0) return SWM_OK;
  MCK(m, cudaSetDevice(m->device));
  // ---- sizes
  size_t arena = 0, scratch = 0, max_smem = 0, zero_bytes = 0;
  int max_rows = 0;
  for (auto& j : jobs) {
    const size_t n1 = j.kind == kJobWindow ? (size_t)j.wq->m : (size_t)j.f1.n(), n2 = (size_t)j.f2.n();
    j.n_out = j.kind == kJobWindow || j.kind == kJobBowFrame ? (int)n2 : (int)n1;
    if (j.kind == kJobWindow) j.n_out = (int)n2;
    arena += up256b((size_t)j.n_out * 4) + 256 + (j.kind == kJobInit ? 2 * up256b(n1 * 8) : 0);
    if (!j.f2.dev) arena += (size_t)n2 * 48 + 6 * 256;
    if (j.kind != kJobWindow && !j.f1.dev) arena += n1 * 48 + 6 * 256;
    if (!j.f2.dev) scratch += up256b(((size_t)kCells + 1 + 2 * std::max<size_t>(n2, 1) + 8) * 4);
    size_t rows = 0;
    if (j.kind == kJobWindow) {
      const size_t M = (size_t)j.wq->m;
      rows = M;
      arena += M * 58 + 10 * 256 + up256b(n2);
      scratch += 2 * up256b(M * 4);  // ev_bin, ev_tgt
      if (j.lm) {  // rows, frame rows, tracking fields, the LocalMapDev; device-written query rows, seen stamps
        arena += n2 * 4 + 17 * M + sizeof(LocalMapDev) + 8 * 256;
        scratch += 58 * M + n2 + up256b((size_t)(j.lm->table->size + 31) / 32 * 4) + 12 * 256;
      }
    } else if (j.kind == kJobInit) {
      rows = n1;
      scratch += 4 * up256b(n1 * 4) + up256b(n1) + 2 * up256b(n1 * 4);
    } else {
      rows = n1;
      arena += featvec_bytes(j.fv1) + featvec_bytes(j.fv2) + up256b(n1) + up256b(n2) + 512;
      scratch += 2 * up256b(((size_t)j.fv1->n_nodes + 1) * 4) + 2 * up256b(n1 * 4) + 2 * up256b(n1 * 4);
      zero_bytes = std::max(zero_bytes, n2);
    }
    scratch += up256b((rows + 1) * 4) + up256b((rows + 2) * 4) + up256b((rows + 64) * 4) + 16 * 256;  // + alignment of every carve
    max_rows = std::max(max_rows, (int)rows);
    const size_t smem = (j.kind == kJobInit ? 8 * n2 : 0) + ((n2 + 3) & ~(size_t)3) + 4 * n2 + 16;
    max_smem = std::max(max_smem, smem);
  }
  if (max_smem > 200 * 1024) {
    m->err = "target frame too large for the matcher's shared-memory state (n2 limit ~15000 keypoints)";
    return SWM_E_CAPACITY;
  }
  arena += up256b((size_t)P * sizeof(BatchJob)) + 4096;
  scratch += up256b(zero_bytes) + 3 * up256b(((size_t)P + 1) * 4) + 4096;
  int rc;
  if ((rc = arena_begin(m, arena))) return rc;
  MCK(m, m->bscratch.ensure(scratch));
  if (m->bcand_cap == 0) {
    m->bcand_cap = (size_t)1 << 22;
    MCK(m, m->bcand[0].ensure(m->bcand_cap * 4));
    MCK(m, m->bcand[1].ensure(m->bcand_cap * 4));
  }

  // ---- pack
  Packer pk{m};
  Carver cv{m->bscratch.as<uint8_t>()};
  uint8_t* zeros = cv.take<uint8_t>(zero_bytes);
  BatchCtl* ctl = cv.take<BatchCtl>(1);
  int32_t* job_total = cv.take<int32_t>((size_t)P + 1);
  int32_t* job_base = cv.take<int32_t>((size_t)P + 1);
  int32_t* job_rows = cv.take<int32_t>((size_t)P + 1);
  std::vector<BatchJob> bj((size_t)P);
  // in/out region first: one contiguous span comes back with a single copy
  for (auto& j : jobs) {
    j.off_out = pk.reserve((size_t)j.n_out * 4);
    if (j.kind == kJobWindow) memcpy(m->h_arena + j.off_out, j.out, (size_t)j.n_out * 4);
    else memset(m->h_arena + j.off_out, 0xFF, (size_t)j.n_out * 4);
    j.off_n = pk.reserve(16);  // nmatches, resolve batches, n_to_match
    memset(m->h_arena + j.off_n, 0, 16);
    if (j.lm && j.lm->job->track) j.lm->off_track = pk.reserve(17 * (size_t)j.wq->m + 5 * 256);
    if (j.kind == kJobInit) {
      j.off_prev = pk.reserve((size_t)j.f1.n() * 8);
      memcpy(m->h_arena + j.off_prev, j.prev_xy, (size_t)j.f1.n() * 8);
    }
  }
  const size_t inout_bytes = m->arena_used;
  std::vector<const swm_frame*> waits;
  std::vector<LocalMapDev> lms;
  std::vector<swm_mappoints*> tables;
  for (int p = 0; p < P; p++) {
    HostJob& j = jobs[p];
    BatchJob& b = bj[p];
    memset(&b, 0, sizeof(b));
    b.kind = j.kind;
    const int n1 = j.kind == kJobWindow ? j.wq->m : j.f1.n(), n2 = j.f2.n();
    b.n1 = n1;
    b.n2 = n2;
    if (j.f2.dev) {
      b.f2 = j.f2.dev->dev;
      waits.push_back(j.f2.dev);
    } else {
      b.f2 = frame_dev_from_host(pk, j.f2.host);
      b.grid2 = cv.take<int32_t>((size_t)kCells + 1 + 2 * std::max(n2, 1) + 8);
      b.f2.starts = b.grid2;
      b.f2.items = b.grid2 ? b.grid2 + kCells + 1 : nullptr;
    }
    if (j.kind != kJobWindow) {
      if (j.f1.dev) {
        b.f1 = j.f1.dev->dev;
        waits.push_back(j.f1.dev);
      } else {
        b.f1 = frame_dev_from_host(pk, j.f1.host);
      }
    }
    ResolveArgs& a = b.ra;
    a.n2 = n2;
    a.nnratio = j.nnratio;
    a.check_ori = j.check_ori;
    a.out = reinterpret_cast<int32_t*>(m->d_arena + j.off_out);
    a.nmatches = reinterpret_cast<int32_t*>(m->d_arena + j.off_n);
    a.angle2 = b.f2.angle;
    if (j.kind == kJobWindow) {
      const swm_window_query* wq = j.wq;
      const size_t M = (size_t)wq->m;
      b.rows_cap = wq->m;
      b.q.m = wq->m;
      if (j.lm) {
        lms.push_back(lm_dev(m, pk, cv, *j.lm, n2, j.check_ori, j.off_n));
        const LocalMapDev& L = lms.back();
        b.q.u = L.u; b.q.v = L.v; b.q.radius = L.radius;
        b.q.min_level = L.min_level; b.q.max_level = L.max_level;
        b.q.valid = L.valid; b.q.desc = L.desc;
        a.blocks = L.blocks;
        a.angle1 = L.angle;
        a.blocked = L.tgt_blocked;
        if (std::find(tables.begin(), tables.end(), j.lm->table) == tables.end()) tables.push_back(j.lm->table);
        if (j.lm->job->mode == SWM_LOCALMAP_LAST) waits.push_back(j.lm->job->last);
      } else {
        b.q.u = pk.put<float>(wq->u, M * 4);
        b.q.v = pk.put<float>(wq->v, M * 4);
        b.q.radius = pk.put<float>(wq->radius, M * 4);
        b.q.min_level = pk.put<int32_t>(wq->min_level, M * 4);
        b.q.max_level = pk.put<int32_t>(wq->max_level, M * 4);
        b.q.valid = pk.put<uint8_t>(wq->valid, M);
        b.q.desc = pk.put<uint4>(wq->desc, M * 32);
        a.blocks = pk.put<uint8_t>(wq->blocks, M);
        a.angle1 = j.check_ori ? pk.put<float>(wq->angle, M * 4) : nullptr;
        uint8_t* blk = pk.put<uint8_t>(j.tgt_blocked, (size_t)n2);
        if (!j.tgt_blocked && blk) memset(m->h_arena + (reinterpret_cast<uint8_t*>(blk) - m->d_arena), 0, (size_t)n2);
        a.blocked = blk;
      }
      a.mode = kModeWindow;
      a.rows = wq->m;
      a.row_valid = b.q.valid;
      a.n1 = wq->m;
      a.th_dist = j.th_dist;
      a.ratio_mode = j.ratio_mode;
      a.ev_bin = cv.take<int32_t>(M);
      a.ev_tgt = cv.take<int32_t>(M);
    } else if (j.kind == kJobInit) {
      b.rows_cap = n1;
      b.iq_u = cv.take<float>((size_t)n1);
      b.iq_v = cv.take<float>((size_t)n1);
      b.iq_r = cv.take<float>((size_t)n1);
      b.iq_l = cv.take<int32_t>((size_t)n1);
      b.iq_valid = cv.take<uint8_t>((size_t)n1);
      b.prev_in = pk.put<float>(j.prev_xy, (size_t)n1 * 8);  // read-only copy: the in/out one is rewritten by resolve
      b.window = (float)j.window;
      b.q.m = n1;
      b.q.desc = b.f1.desc;
      b.q.u = b.iq_u; b.q.v = b.iq_v; b.q.radius = b.iq_r;
      b.q.min_level = b.iq_l; b.q.max_level = b.iq_l;
      b.q.valid = b.iq_valid;
      a.mode = kModeInit;
      a.rows = n1;
      a.row_valid = b.iq_valid;
      a.n1 = n1;
      a.angle1 = b.f1.angle;
      a.prev_xy = reinterpret_cast<float*>(m->d_arena + j.off_prev);
      a.x2 = b.f2.x; a.y2 = b.f2.y;
      a.ev_bin = cv.take<int32_t>((size_t)n1);
      a.ev_tgt = cv.take<int32_t>((size_t)n1);
    } else {
      b.rows_cap = n1;
      const swm_featvec *f1v = j.fv1, *f2v = j.fv2;
      b.nn1 = f1v->n_nodes; b.nn2 = f2v->n_nodes;
      b.ids1 = pk.put<uint32_t>(f1v->node_ids, (size_t)b.nn1 * 4);
      b.off1 = pk.put<int32_t>(f1v->offsets, ((size_t)b.nn1 + 1) * 4);
      b.feats1 = pk.put<uint32_t>(f1v->feats, (size_t)(b.nn1 ? f1v->offsets[b.nn1] : 0) * 4);
      b.ids2 = pk.put<uint32_t>(f2v->node_ids, (size_t)b.nn2 * 4);
      b.off2 = pk.put<int32_t>(f2v->offsets, ((size_t)b.nn2 + 1) * 4);
      b.feats2 = pk.put<uint32_t>(f2v->feats, (size_t)(b.nn2 ? f2v->offsets[b.nn2] : 0) * 4);
      b.valid1 = pk.put<uint8_t>(j.valid1, (size_t)n1);
      b.node_scratch = cv.take<int32_t>(2 * ((size_t)b.nn1 + 1));
      b.row_src = cv.take<int32_t>((size_t)n1);
      b.row_aux = cv.take<int32_t>((size_t)n1);
      a.mode = j.kind == kJobBowFrame ? kModeBowFrame : kModeBowKf;
      a.row_src = b.row_src;
      a.n1 = n1;
      a.angle1 = b.f1.angle;
      a.valid2 = j.kind == kJobBowKf ? pk.put<uint8_t>(j.valid2, (size_t)n2) : nullptr;
      a.blocked = zeros;
      a.ev_bin = cv.take<int32_t>((size_t)n1);
      a.ev_tgt = cv.take<int32_t>((size_t)n1);
    }
    b.row_count = cv.take<int32_t>((size_t)b.rows_cap + 1);
    b.row_start = cv.take<int32_t>((size_t)b.rows_cap + 2);
    a.row_start = b.row_start;
    a.row_list = cv.take<int32_t>((size_t)b.rows_cap + 64);
  }
  BatchJob* d_jobs = pk.put<BatchJob>(bj.data(), (size_t)P * sizeof(BatchJob));
  LocalMapDev* d_lm = lms.empty() ? nullptr : pk.put<LocalMapDev>(lms.data(), lms.size() * sizeof(LocalMapDev));
  if (pk.overflow || cv.used > m->bscratch.cap) { m->err = "internal: batch arena overflow"; return SWM_E_CAPACITY; }
  for (const swm_frame* f : waits) MCK(m, cudaStreamWaitEvent(m->stream, f->ready, 0));
  for (swm_mappoints* t : tables) MCK(m, cudaStreamWaitEvent(m->stream, t->written, 0));
  if ((rc = arena_flush(m))) return rc;
  static bool attr_set[64] = {};
  if (!attr_set[m->device & 63]) {
    MCK(m, cudaFuncSetAttribute(bq_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set[m->device & 63] = true;
  }
  if ((rc = down_begin(m, inout_bytes + 256))) return rc;
  if (zero_bytes) MCK(m, cudaMemsetAsync(zeros, 0, zero_bytes, m->stream));
  if (!m->bev[0]) {
    MCK(m, cudaEventCreate(&m->bev[0]));
    MCK(m, cudaEventCreate(&m->bev[1]));
  }

  for (int attempt = 0; attempt < 2; attempt++) {
    BatchCtl h_ctl{(int32_t)std::min<size_t>(m->bcand_cap, 0x7FFFFFFF), 0, 0, 0};
    MCK(m, cudaMemcpyAsync(ctl, &h_ctl, sizeof(h_ctl), cudaMemcpyHostToDevice, m->stream));
    MCK(m, cudaMemsetAsync(job_total, 0, ((size_t)P + 1) * 4, m->stream));
    const dim3 rows_grid((unsigned)((max_rows + 7) / 8), (unsigned)P);
    MCK(m, cudaEventRecord(m->bev[0], m->stream));
    if (d_lm) {
      lm_project_kernel<<<(unsigned)lms.size(), kLmThreads, 0, m->stream>>>(d_lm);
      for (swm_mappoints* t : tables) MCK(m, cudaEventRecord(t->read_done, m->stream));
    }
    bq_prepare_kernel<<<P, 1024, 0, m->stream>>>(d_jobs, job_total, job_rows, ctl);
    bq_count_kernel<<<rows_grid, 256, 0, m->stream>>>(d_jobs);
    bq_scan_kernel<<<P, 1024, 0, m->stream>>>(d_jobs, job_total);
    bq_offsets_kernel<<<1, 1024, 0, m->stream>>>(job_total, P, job_base, ctl);
    bq_fill_kernel<<<rows_grid, 256, 0, m->stream>>>(d_jobs, job_base, job_rows, ctl, m->bcand[0].as<int32_t>(),
                                                     m->bcand[1].as<uint32_t>());
    bq_resolve_kernel<<<P, kResolveWarps * 32, max_smem, m->stream>>>(d_jobs, job_base, job_rows, ctl,
                                                                      m->bcand[0].as<int32_t>(), m->bcand[1].as<uint32_t>());
    MCK(m, cudaGetLastError());
    MCK(m, cudaEventRecord(m->bev[1], m->stream));
    MCK(m, cudaMemcpyAsync(m->h_down, m->d_arena, inout_bytes, cudaMemcpyDeviceToHost, m->stream));
    MCK(m, cudaMemcpyAsync(m->h_down + up256b(inout_bytes), ctl, sizeof(BatchCtl), cudaMemcpyDeviceToHost, m->stream));
    MCK(m, cudaStreamSynchronize(m->stream));
    memcpy(&h_ctl, m->h_down + up256b(inout_bytes), sizeof(h_ctl));
    MCK(m, cudaEventElapsedTime(&m->last_device_ms, m->bev[0], m->bev[1]));
    if (h_ctl.bad_index) { m->err = "feature index out of range"; return SWM_E_INVALID; }
    if (!h_ctl.overflow) break;
    if (attempt == 1) { m->err = "internal: candidate buffer overflow after regrowth"; return SWM_E_CAPACITY; }
    m->bcand_cap = (size_t)h_ctl.cand_total + (size_t)h_ctl.cand_total / 2 + 1024;
    MCK(m, m->bcand[0].ensure(m->bcand_cap * 4));
    MCK(m, m->bcand[1].ensure(m->bcand_cap * 4));
  }
  for (auto& j : jobs) {
    memcpy(j.out, m->h_down + j.off_out, (size_t)j.n_out * 4);
    *j.nmatches = *reinterpret_cast<const int32_t*>(m->h_down + j.off_n);
    if (j.kind == kJobInit) memcpy(j.prev_xy, m->h_down + j.off_prev, (size_t)j.f1.n() * 8);
    if (j.lm) lm_finish(*j.lm, m->h_down, j.off_n);
  }
  return SWM_OK;
}

}  // namespace

extern "C" {

float swm_matcher_last_device_ms(const swm_matcher* m) { return m ? m->last_device_ms : 0.f; }

int swm_match_window_batch(swm_matcher* m, swm_window_job* jobs, int njobs) {
  if (!m) return SWM_E_INVALID;
  if (njobs < 0 || (njobs && !jobs)) { m->err = "bad argument"; return SWM_E_INVALID; }
  std::vector<HostJob> hj;
  hj.reserve((size_t)njobs);
  for (int p = 0; p < njobs; p++) {
    swm_window_job& w = jobs[p];
    const bool have = (w.tgt != nullptr) != (w.tgt_resident != nullptr);
    if (!have || (w.tgt && !frame_ok(w.tgt)) || !window_query_ok(w.q, w.check_ori) || !w.assignment ||
        (w.ratio_mode != 0 && w.ratio_mode != 1)) {
      m->err = "bad argument in window job";
      return SWM_E_INVALID;
    }
    if (w.tgt_resident) {
      if (int rc = resident_ok(m, w.tgt_resident, w.tgt_resident, w.tgt_resident)) return rc;
    }
    w.nmatches = 0;
    HostJob j;
    j.kind = kJobWindow;
    j.f2 = FrameSrc{w.tgt, w.tgt_resident};
    if (w.q->m == 0 || j.f2.n() == 0) continue;
    j.wq = w.q;
    j.tgt_blocked = w.tgt_blocked;
    j.th_dist = w.th_dist;
    j.ratio_mode = w.ratio_mode;
    j.nnratio = w.nnratio;
    j.check_ori = w.check_ori;
    j.out = w.assignment;
    j.nmatches = &w.nmatches;
    hj.push_back(j);
  }
  return run_batch(m, hj);
}

int swm_match_init_batch(swm_matcher* m, swm_init_job* jobs, int njobs) {
  if (!m) return SWM_E_INVALID;
  if (njobs < 0 || (njobs && !jobs)) { m->err = "bad argument"; return SWM_E_INVALID; }
  std::vector<HostJob> hj;
  hj.reserve((size_t)njobs);
  for (int p = 0; p < njobs; p++) {
    swm_init_job& w = jobs[p];
    const bool res = w.r1 && w.r2 && !w.f1 && !w.f2, host = w.f1 && w.f2 && !w.r1 && !w.r2;
    if ((!res && !host) || (host && (!frame_ok(w.f1) || !frame_ok(w.f2))) || !w.prev_xy || !w.matches12 || w.window < 0) {
      m->err = "bad argument in initialization job";
      return SWM_E_INVALID;
    }
    if (res) {
      if (int rc = resident_ok(m, w.r1, w.r2, w.r2)) return rc;
    }
    w.nmatches = 0;
    HostJob j;
    j.kind = kJobInit;
    j.f1 = FrameSrc{w.f1, w.r1};
    j.f2 = FrameSrc{w.f2, w.r2};
    for (int i = 0; i < j.f1.n(); i++) w.matches12[i] = -1;
    if (j.f1.n() == 0 || j.f2.n() == 0) continue;
    j.prev_xy = w.prev_xy;
    j.window = w.window;
    j.nnratio = w.nnratio;
    j.check_ori = w.check_ori;
    j.out = w.matches12;
    j.nmatches = &w.nmatches;
    hj.push_back(j);
  }
  return run_batch(m, hj);
}

int swm_match_bow_batch(swm_matcher* m, swm_bow_job* jobs, int njobs) {
  if (!m) return SWM_E_INVALID;
  if (njobs < 0 || (njobs && !jobs)) { m->err = "bad argument"; return SWM_E_INVALID; }
  std::vector<HostJob> hj;
  hj.reserve((size_t)njobs);
  for (int p = 0; p < njobs; p++) {
    swm_bow_job& w = jobs[p];
    const bool res = w.r1 && w.r2 && !w.f1 && !w.f2, host = w.f1 && w.f2 && !w.r1 && !w.r2;
    if ((!res && !host) || (host && (!frame_ok(w.f1) || !frame_ok(w.f2))) || !featvec_ok(w.fv1) || !featvec_ok(w.fv2) ||
        !w.valid1 || !w.matches || (w.mode != 0 && w.mode != 1) || (w.mode == 1 && !w.valid2)) {
      m->err = "bad argument in BoW job";
      return SWM_E_INVALID;
    }
    if (res) {
      if (int rc = resident_ok(m, w.r1, w.r2, nullptr)) return rc;
    }
    w.nmatches = 0;
    HostJob j;
    j.kind = w.mode == 0 ? kJobBowFrame : kJobBowKf;
    j.f1 = FrameSrc{w.f1, w.r1};
    j.f2 = FrameSrc{w.f2, w.r2};
    const int n_out = w.mode == 0 ? j.f2.n() : j.f1.n();
    for (int i = 0; i < n_out; i++) w.matches[i] = -1;
    if (j.f1.n() == 0 || j.f2.n() == 0 || w.fv1->n_nodes == 0 || w.fv2->n_nodes == 0) continue;
    j.fv1 = w.fv1; j.fv2 = w.fv2;
    j.valid1 = w.valid1; j.valid2 = w.valid2;
    j.nnratio = w.nnratio;
    j.check_ori = w.check_ori;
    j.out = w.matches;
    j.nmatches = &w.nmatches;
    hj.push_back(j);
  }
  return run_batch(m, hj);
}

int swm_frames_from_extractor(swm_frame** frames, int count, swm_orb* h, const int32_t* indices, const swm_camera* cam,
                              const float* bounds4) {
  if (!frames || count <= 0 || !frames[0]) return SWM_E_INVALID;
  swm_frame* f0 = frames[0];
  if (!h || !bounds4 || !(bounds4[1] > bounds4[0]) || !(bounds4[3] > bounds4[2])) { f0->err = "bad argument"; return SWM_E_INVALID; }
  OrbDeviceView v;
  int rc = orb_device_view(h, &v);
  if (rc != SWM_OK) { f0->err = "the extractor holds no resident batch"; return rc; }
  if (count > v.batch && !indices) { f0->err = "more frames than the extractor's last batch holds"; return SWM_E_INVALID; }
  FCK(f0, cudaSetDevice(f0->device));
  std::vector<FrameBuildDev> fb((size_t)count);
  for (int b = 0; b < count; b++) {
    swm_frame* f = frames[b];
    const int index = indices ? indices[b] : b;
    if (!f || f->device != v.device) { f0->err = "frame missing or on another device than the extractor"; return SWM_E_INVALID; }
    if (index < 0 || index >= v.batch) { f0->err = "frame index outside the extractor's last batch"; return SWM_E_INVALID; }
    FCK(f, cudaEventSynchronize(f->ready));
    if ((rc = frame_reserve(f, v.cap, bounds4))) return rc;  // capacity for the largest possible count
    FrameBuildDev& d = fb[b];
    d.kps = v.kps + (size_t)index * v.cap;
    d.desc_in = reinterpret_cast<const uint4*>(v.desc + (size_t)index * v.cap * 32);
    d.n_ptr = v.n + index;
    d.cap = v.cap;
    d.x = f->b[0].as<float>(); d.y = f->b[1].as<float>(); d.octave = f->b[2].as<int32_t>();
    d.angle = f->b[3].as<float>(); d.desc_out = f->b[4].as<uint4>();
    d.dev = f->dev;
    d.grid = f->b[5].as<int32_t>();
  }
  // the descriptor table and the counts travel through the first frame's grow-only staging buffers
  FCK(f0, f0->bstage.ensure((size_t)count * sizeof(FrameBuildDev)));
  if ((size_t)v.batch * 4 > f0->h_counts_cap) {
    if (f0->h_counts) cudaFreeHost(f0->h_counts);
    f0->h_counts = nullptr;
    f0->h_counts_cap = 0;
    FCK(f0, cudaMallocHost(&f0->h_counts, (size_t)v.batch * 4 + 1024));
    f0->h_counts_cap = (size_t)v.batch * 4 + 1024;
  }
  FCK(f0, cudaMemcpyAsync(f0->bstage.p, fb.data(), fb.size() * sizeof(FrameBuildDev), cudaMemcpyHostToDevice, v.stream));
  const FrameBuildDev* d_fb = f0->bstage.as<FrameBuildDev>();
  frames_from_kps_kernel<<<dim3((unsigned)((v.cap + 255) / 256), (unsigned)count), 256, 0, v.stream>>>(d_fb, camera_dev(cam));
  frames_grid_kernel<<<count, 1024, 0, v.stream>>>(d_fb);
  FCK(f0, cudaGetLastError());
  FCK(f0, cudaMemcpyAsync(f0->h_counts, v.n, (size_t)v.batch * 4, cudaMemcpyDeviceToHost, v.stream));
  FCK(f0, cudaStreamSynchronize(v.stream));  // fb (host) and the counts are done with here
  for (int b = 0; b < count; b++) {
    swm_frame* f = frames[b];
    const int n = std::min(f0->h_counts[indices ? indices[b] : b], v.cap);
    f->n = n;
    f->dev.n = n;
    FCK(f, cudaEventRecord(f->ready, v.stream));
  }
  return SWM_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------ projection from the MapPoint table
namespace {

bool rows_ok(const int32_t* r, int n, int32_t size, bool allow_none) {
  for (int i = 0; i < n; i++)
    if (r[i] >= size || r[i] < (allow_none ? -1 : 0)) return false;
  return true;
}

// Validates one job and prepares its host record; a job with nothing to match is answered here (*skip = true).
int lm_prepare(swm_matcher* m, swm_localmap_job& w, LocalMapHost& h, bool* skip) {
  w.nmatches = 0;
  w.n_to_match = 0;
  *skip = true;
  const bool last = w.mode == SWM_LOCALMAP_LAST;
  if ((w.mode != SWM_LOCALMAP_POINTS && !last) || !w.tgt || !w.table || !w.proj || !w.assignment ||
      (last && !w.last) || (!last && (w.n_rows < 0 || (w.n_rows > 0 && !w.rows))) || !w.proj->scale_factors ||
      w.proj->nlevels < 1 || w.proj->nlevels > SWM_MAX_LEVELS) {
    m->err = "bad argument in local-map job";
    return SWM_E_INVALID;
  }
  for (const swm_frame* f : {w.tgt, w.last})
    if (f && f->device != m->device) { m->err = "resident frame lives on another device"; return SWM_E_INVALID; }
  if (w.table->device != m->device) { m->err = "MapPoint table lives on another device"; return SWM_E_INVALID; }
  if (!w.tgt->dev.starts || (last && !w.last->dev.starts)) { m->err = "resident frame has not been built"; return SWM_E_STATE; }
  const int M = last ? w.last->n : w.n_rows, n2 = w.tgt->n;
  if (M > 0 && !w.rows) { m->err = "bad argument in local-map job"; return SWM_E_INVALID; }
  const int32_t size = w.table->size;
  if (!rows_ok(w.rows, M, size, last) || (w.frame_rows && !rows_ok(w.frame_rows, n2, size, true))) {
    m->err = "row outside the MapPoint table";
    return SWM_E_INVALID;
  }
  if (m->thr_n != w.proj->nlevels || m->thr_lsf != w.proj->log_scale_factor) {
    if (swm_predict_scale_thresholds(w.proj->log_scale_factor, w.proj->nlevels, m->thr) != SWM_OK) {
      m->err = "bad scale table";
      return SWM_E_INVALID;
    }
    m->thr_n = w.proj->nlevels;
    m->thr_lsf = w.proj->log_scale_factor;
  }
  memcpy(h.thr, m->thr, sizeof(h.thr));
  h.job = &w;
  h.table = w.table;
  memset(&h.wq, 0, sizeof(h.wq));
  h.wq.m = M;
  *skip = M == 0 || (last && n2 == 0);
  return SWM_OK;
}

int run_local_map(swm_matcher* m, swm_localmap_job* jobs, int njobs) {
  if (njobs < 0 || (njobs && !jobs)) { m->err = "bad argument"; return SWM_E_INVALID; }
  // every table the batch reads stays locked from the size check in lm_prepare until the results are back (see
  // swm_mappoints); address order, so two batches over the same tables cannot deadlock
  std::vector<swm_mappoints*> tables;
  for (int p = 0; p < njobs; p++)
    if (jobs[p].table) tables.push_back(jobs[p].table);
  std::sort(tables.begin(), tables.end());
  tables.erase(std::unique(tables.begin(), tables.end()), tables.end());
  std::vector<std::unique_lock<std::mutex>> locks;
  locks.reserve(tables.size());
  for (swm_mappoints* t : tables) locks.emplace_back(t->mu);
  std::vector<LocalMapHost> lh((size_t)njobs);
  std::vector<HostJob> hj;
  hj.reserve((size_t)njobs);
  for (int p = 0; p < njobs; p++) {
    swm_localmap_job& w = jobs[p];
    bool skip;
    int rc = lm_prepare(m, w, lh[p], &skip);
    if (rc) return rc;
    if (skip) continue;
    const bool last = w.mode == SWM_LOCALMAP_LAST;
    HostJob j;
    j.kind = kJobWindow;
    j.f2 = FrameSrc{nullptr, w.tgt};
    j.wq = &lh[p].wq;
    j.th_dist = 100;                                   // TH_HIGH, ORBmatcher.cc:111 / :1316
    j.ratio_mode = last ? 0 : 1;
    j.nnratio = w.nnratio;
    j.check_ori = last ? (w.check_ori != 0) : 0;
    j.out = w.assignment;
    j.nmatches = &w.nmatches;
    j.lm = &lh[p];
    hj.push_back(j);
  }
  return run_batch(m, hj);
}

}  // namespace

extern "C" {

int swm_match_local_map_batch(swm_matcher* m, swm_localmap_job* jobs, int njobs) {
  if (!m) return SWM_E_INVALID;
  return run_local_map(m, jobs, njobs);
}

int swm_match_local_map(swm_matcher* m, const swm_frame* tgt, swm_mappoints* t, const swm_projection* proj,
                        const int32_t* rows, int n_rows, const int32_t* frame_rows, float th, float nnratio,
                        const swm_track_out* track, int32_t* assignment, int* nmatches, int* n_to_match) {
  if (!m) return SWM_E_INVALID;
  if (!nmatches) { m->err = "bad argument"; return SWM_E_INVALID; }
  swm_localmap_job j;
  memset(&j, 0, sizeof(j));
  j.mode = SWM_LOCALMAP_POINTS;
  j.tgt = tgt; j.table = t; j.proj = proj; j.rows = rows; j.n_rows = n_rows; j.frame_rows = frame_rows;
  j.th = th; j.nnratio = nnratio; j.track = track; j.assignment = assignment;
  const int rc = run_local_map(m, &j, 1);
  *nmatches = j.nmatches;
  if (n_to_match) *n_to_match = j.n_to_match;
  return rc;
}

int swm_match_last_frame(swm_matcher* m, const swm_frame* cur, const swm_frame* last, swm_mappoints* t,
                         const swm_projection* proj, const int32_t* last_rows, const int32_t* cur_rows, float th,
                         int check_ori, int32_t* assignment, int* nmatches) {
  if (!m) return SWM_E_INVALID;
  if (!nmatches) { m->err = "bad argument"; return SWM_E_INVALID; }
  swm_localmap_job j;
  memset(&j, 0, sizeof(j));
  j.mode = SWM_LOCALMAP_LAST;
  j.tgt = cur; j.last = last; j.table = t; j.proj = proj; j.rows = last_rows; j.frame_rows = cur_rows;
  j.th = th; j.check_ori = check_ori; j.assignment = assignment;
  const int rc = run_local_map(m, &j, 1);
  *nmatches = j.nmatches;
  return rc;
}

}  // extern "C"
