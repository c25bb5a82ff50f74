// mappoints.cuh -- the resident MapPoint table (swm_mappoints_*) and the projection step of the two tracking
// SearchByProjection calls run from it (swm_match_local_map*, swm_match_last_frame).  Included by match.cu before
// match_batch.cuh: a projection job is a window job whose query rows are written on the device by lm_project_kernel;
// the six batch launches that follow it are the existing ones.
//
// Reference behaviour restated (paths relative to /root/reference/code/):
//   Tracking::SearchLocalPoints            src/Tracking.cc:964-1006 (the mnLastFrameSeen stamp, isInFrustum per point)
//   Frame::isInFrustum                     src/Frame.cc:316-375
//   MapPoint::PredictScale                 src/MapPoint.cc:476-485
//   SearchByProjection(F, vpMapPoints, th) src/ORBmatcher.cc:44-121 (RadiusByViewingCos :123-128)
//   SearchByProjection(cur, last, th, bMono = true)  src/ORBmatcher.cc:1223-1354
// Every rounding the reference does is an explicit round-to-nearest intrinsic, so nothing is contracted into an FMA;
// the numerics are those of DESIGN.md section 2.
#pragma once

// ---- PredictScale without libm on the device.  The level is clamp(ceil(logf(max / dist) / logScaleFactor), 0,
// nlevels - 1): non-decreasing in the ratio, so it equals the number of boundaries thr[k] (k = 0 .. nlevels - 2, the
// largest ratio whose level is <= k) that the ratio exceeds.  The host finds the boundaries once per scale table by
// bisection over float bit patterns with the reference's own expression; the device only divides and compares, which
// is exact on both sides.  (CUDA's logf and glibc's may differ by an ulp, which would move a level at a boundary.)
namespace {

int predict_level_host(float ratio, float log_sf, int nlevels) {
  const float q = std::ceil(std::log(ratio) / log_sf);
  if (std::isnan(q) || q < 0.0f) return 0;
  if (q >= (float)nlevels) return nlevels - 1;
  return (int)q;
}

}  // namespace

extern "C" int swm_predict_scale_thresholds(float log_scale_factor, int32_t nlevels, float* thresholds) {
  if (!thresholds || nlevels < 1 || nlevels > SWM_MAX_LEVELS || !(log_scale_factor > 0.0f) ||
      !std::isfinite(log_scale_factor))
    return SWM_E_INVALID;
  for (int k = 1; k < nlevels; k++) {
    uint32_t lo = 0, hi = 0x7F7FFFFFu;  // level(+0) = 0 < k <= nlevels - 1 = level(FLT_MAX)
    while (hi - lo > 1) {
      const uint32_t mid = lo + (hi - lo) / 2;
      float r;
      memcpy(&r, &mid, 4);
      if (predict_level_host(r, log_scale_factor, nlevels) < k) lo = mid;
      else hi = mid;
    }
    memcpy(&thresholds[k - 1], &lo, 4);
  }
  return SWM_OK;
}

// ---- the table: structure-of-arrays rows on one device
namespace swm {

struct TableDev {
  const float *px, *py, *pz, *nx, *ny, *nz, *min_d, *max_d;
  const uint4* desc;
  const uint8_t *has_obs, *bad;
};

__global__ void __launch_bounds__(256) mp_scatter_kernel(const uint8_t* __restrict__ stage, int n, float* __restrict__ cols,
                                                         size_t cap, uint4* __restrict__ desc, uint8_t* __restrict__ has_obs,
                                                         uint8_t* __restrict__ bad) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  // stage: rows[n] | 8 float columns [8][n] | desc[n][32] | has_obs[n] | bad[n] (each section 256-byte aligned)
  const size_t sn = ((size_t)n * 4 + 255) & ~(size_t)255;
  const int32_t row = reinterpret_cast<const int32_t*>(stage)[i];
  const float* f = reinterpret_cast<const float*>(stage + sn);
  const size_t fs = (((size_t)n * 4 + 255) & ~(size_t)255) / 4;
  for (int c = 0; c < 8; c++) cols[(size_t)c * cap + row] = f[(size_t)c * fs + i];
  const uint4* d = reinterpret_cast<const uint4*>(stage + sn + 8 * fs * 4);
  desc[2 * (size_t)row] = d[2 * i];
  desc[2 * (size_t)row + 1] = d[2 * i + 1];
  const uint8_t* b = stage + sn + 8 * fs * 4 + (((size_t)n * 32 + 255) & ~(size_t)255);
  has_obs[row] = b[i];
  bad[row] = b[(((size_t)n + 255) & ~(size_t)255) + i];
}

// One projection job: SearchLocalPoints' list (mode 0) or the last frame's keypoints (mode 1).
struct LocalMapDev {
  int mode, m, n2, nwords, nlevels;
  const int32_t* rows;        // m: table row per source (mode 1: -1 = no point / outlier)
  const int32_t* frame_rows;  // n2 or NULL: the table row held by each keypoint of the current frame
  uint32_t* seen;             // nwords: mode 0, rows stamped by the current frame (mnLastFrameSeen)
  TableDev t;
  float T[12];
  float fx, fy, cx, cy, min_x, max_x, min_y, max_y, th;
  float sf[SWM_MAX_LEVELS], thr[SWM_MAX_LEVELS];
  const int32_t* last_octave;  // mode 1
  const float* last_angle;
  // the window query the six batch launches read
  float *u, *v, *radius, *angle;
  int32_t *min_level, *max_level;
  uint8_t *valid, *blocks, *tgt_blocked;
  uint4* desc;
  // tracking fields (mode 0; each may be NULL) and the number of points in view
  uint8_t* t_in_view;
  float *t_u, *t_v, *t_cos;
  int32_t *t_level, *n_to_match;
};

// Pc = Rcw * P + tcw (cv::gemm's small-matrix path: float products and sums, left to right, then + t)
__device__ __forceinline__ float gemm_row(const float* T, int r, float x, float y, float z) {
  float acc = __fmul_rn(T[4 * r], x);
  acc = __fadd_rn(acc, __fmul_rn(T[4 * r + 1], y));
  acc = __fadd_rn(acc, __fmul_rn(T[4 * r + 2], z));
  return __fadd_rn(acc, T[4 * r + 3]);
}

constexpr int kLmThreads = 512;  // one CTA per job; 1024 threads would cap the kernel at 64 registers and spill

__global__ void __launch_bounds__(kLmThreads, 1) lm_project_kernel(const LocalMapDev* __restrict__ jobs) {
  __shared__ int s_count;
  const LocalMapDev& J = jobs[blockIdx.x];
  const int tid = threadIdx.x;
  const TableDev& t = J.t;
  if (tid == 0) s_count = 0;
  if (J.mode == 0)
    for (int w = tid; w < J.nwords; w += kLmThreads) J.seen[w] = 0;
  __syncthreads();
  // the current frame's points: stamped as seen and, when they have observations, unavailable (Tracking.cc:970-979,
  // ORBmatcher.cc:78-80; SearchLocalPoints NULLs a bad point first, so it neither stamps nor blocks) -- resp. the
  // current frame's points of the last-frame overload (:1291-1293)
  for (int j = tid; j < J.n2; j += kLmThreads) {
    const int r = J.frame_rows ? J.frame_rows[j] : -1;
    bool blk = false;
    if (r >= 0) {
      const bool live = J.mode == 1 || !t.bad[r];
      blk = live && t.has_obs[r];
      if (J.mode == 0 && live) atomicOr(&J.seen[r >> 5], 1u << (r & 31));
    }
    J.tgt_blocked[j] = blk ? 1 : 0;
  }
  __syncthreads();
  // Ow = -Rcw.t() * tcw (generic path: double products and sums, left to right)
  float Ow[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 3; k++) acc = __dadd_rn(acc, __dmul_rn((double)J.T[4 * k + c], (double)J.T[4 * k + 3]));
    Ow[c] = __double2float_rn(__dmul_rn(-1.0, acc));
  }
  int count = 0;
  for (int s = tid; s < J.m; s += kLmThreads) {
    const int row = J.rows[s];
    bool ok = false, in_view = false;
    float u = 0.f, v = 0.f, vc = 0.f, radius = 0.f;
    int lvl = 0, lo = -1, hi = -1;
    if (J.mode == 0) {
      if (!t.bad[row] && !((J.seen[row >> 5] >> (row & 31)) & 1u)) {  // Tracking.cc:985-990
        // Frame::isInFrustum(pMP, 0.5), Frame.cc:316-375
        const float X = t.px[row], Y = t.py[row], Z = t.pz[row];
        const float PcX = gemm_row(J.T, 0, X, Y, Z), PcY = gemm_row(J.T, 1, X, Y, Z), PcZ = gemm_row(J.T, 2, X, Y, Z);
        if (!(PcZ < 0.0f)) {
          const float invz = __fdiv_rn(1.0f, PcZ);
          const float pu = __fadd_rn(__fmul_rn(__fmul_rn(J.fx, PcX), invz), J.cx);
          const float pv = __fadd_rn(__fmul_rn(__fmul_rn(J.fy, PcY), invz), J.cy);
          if (!(pu < J.min_x || pu > J.max_x) && !(pv < J.min_y || pv > J.max_y)) {
            const float maxD = __fmul_rn(1.2f, t.max_d[row]), minD = __fmul_rn(0.8f, t.min_d[row]);
            const float PO0 = __fsub_rn(X, Ow[0]), PO1 = __fsub_rn(Y, Ow[1]), PO2 = __fsub_rn(Z, Ow[2]);
            double ss = 0.0;
            ss = __dadd_rn(ss, __dmul_rn((double)PO0, (double)PO0));
            ss = __dadd_rn(ss, __dmul_rn((double)PO1, (double)PO1));
            ss = __dadd_rn(ss, __dmul_rn((double)PO2, (double)PO2));
            const float dist = __double2float_rn(__dsqrt_rn(ss));
            if (!(dist < minD || dist > maxD)) {
              double dot = 0.0;
              dot = __dadd_rn(dot, __dmul_rn((double)PO0, (double)t.nx[row]));
              dot = __dadd_rn(dot, __dmul_rn((double)PO1, (double)t.ny[row]));
              dot = __dadd_rn(dot, __dmul_rn((double)PO2, (double)t.nz[row]));
              const float cosv = __double2float_rn(__ddiv_rn(dot, (double)dist));
              if (!(cosv < 0.5f)) {
                const float ratio = __fdiv_rn(t.max_d[row], dist);  // PredictScale
                for (int k = 0; k + 1 < J.nlevels; k++) lvl += ratio > J.thr[k] ? 1 : 0;
                in_view = true;
                u = pu; v = pv; vc = cosv;
              }
            }
          }
        }
      }
      if (in_view) {  // ORBmatcher.cc:62-66: RadiusByViewingCos compares with the double 0.998
        float r = (double)vc > 0.998 ? 2.5f : 4.0f;
        if (J.th != 1.0f) r = __fmul_rn(r, J.th);
        radius = __fmul_rn(r, J.sf[lvl]);
        lo = lvl - 1;
        hi = lvl;
        ok = true;
        count++;
      }
      if (J.t_in_view) J.t_in_view[s] = in_view ? 1 : 0;
      if (J.t_u) J.t_u[s] = u;
      if (J.t_v) J.t_v[s] = v;
      if (J.t_cos) J.t_cos[s] = vc;
      if (J.t_level) J.t_level[s] = lvl;
    } else if (row >= 0) {  // ORBmatcher.cc:1247-1282
      const float X = t.px[row], Y = t.py[row], Z = t.pz[row];
      const float xc = gemm_row(J.T, 0, X, Y, Z), yc = gemm_row(J.T, 1, X, Y, Z), zc = gemm_row(J.T, 2, X, Y, Z);
      const float invzc = __double2float_rn(__ddiv_rn(1.0, (double)zc));
      if (!(invzc < 0.0f)) {
        u = __fadd_rn(__fmul_rn(__fmul_rn(J.fx, xc), invzc), J.cx);
        v = __fadd_rn(__fmul_rn(__fmul_rn(J.fy, yc), invzc), J.cy);
        if (!(u < J.min_x || u > J.max_x) && !(v < J.min_y || v > J.max_y)) {
          const int oct = J.last_octave[s];
          radius = __fmul_rn(J.th, J.sf[oct]);
          lo = oct - 1;
          hi = oct + 1;
          ok = true;
        }
      }
      if (J.angle) J.angle[s] = J.last_angle[s];
    }
    J.valid[s] = ok ? 1 : 0;
    J.u[s] = ok ? u : 0.f;
    J.v[s] = ok ? v : 0.f;
    J.radius[s] = radius;
    J.min_level[s] = lo;
    J.max_level[s] = hi;
    J.blocks[s] = row >= 0 ? t.has_obs[row] : 1;
    if (ok) {
      J.desc[2 * s] = t.desc[2 * (size_t)row];
      J.desc[2 * s + 1] = t.desc[2 * (size_t)row + 1];
    }
  }
  if (count) atomicAdd(&s_count, count);
  __syncthreads();
  if (tid == 0 && J.n_to_match) *J.n_to_match = s_count;
}

}  // namespace swm

// One device's MapPoint table.  Ordering: an upsert waits (on the table's stream) for `read_done`, recorded by the last
// query that read the table, and records `written`; a query waits for `written` before its projection kernel and
// records `read_done` after it.  `mu` makes those two steps atomic with respect to each other across host threads: an
// upsert holds it from its size check to its `written` record (a growing upsert frees the old block inside), a query
// from reading the table's size and pointers until its results are back, so a query never launches on a block an upsert
// has freed and never waits on an event that a concurrent call has not recorded yet.
struct swm_mappoints {
  std::mutex mu;
  int device = 0;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t written = nullptr, read_done = nullptr, staged = nullptr;
  int32_t size = 0;
  size_t cap = 0;
  uint8_t* block = nullptr;  // float cols[8][cap] | desc[cap][32] | has_obs[cap] | bad[cap]
  uint8_t* h_stage = nullptr;
  size_t stage_cap = 0;
  DevBuf d_stage;
  TableDev view() const {
    TableDev t{};
    const float* f = reinterpret_cast<const float*>(block);
    t.px = f; t.py = f + cap; t.pz = f + 2 * cap; t.nx = f + 3 * cap; t.ny = f + 4 * cap; t.nz = f + 5 * cap;
    t.min_d = f + 6 * cap; t.max_d = f + 7 * cap;
    t.desc = reinterpret_cast<const uint4*>(block + 32 * cap);
    t.has_obs = block + 64 * cap;
    t.bad = block + 65 * cap;
    return t;
  }
};

namespace {

thread_local std::string g_mappoints_create_error;

#define TCK(t, call)                                   \
  do {                                                 \
    cudaError_t e_ = (call);                           \
    if (e_ != cudaSuccess) {                           \
      (t)->err = cuda_err(#call, e_);                  \
      return SWM_E_CUDA;                               \
    }                                                  \
  } while (0)

// Grows the table to hold `need` rows; the contents move along.  New rows are all zero (position, normal, distances,
// descriptor) with no observations and the bad flag set, so an unwritten row is defined in both projection modes.
int mp_reserve(swm_mappoints* t, size_t need) {
  if (need <= t->cap) return SWM_OK;
  const size_t cap = std::max<size_t>({need, 2 * t->cap, 1024});
  uint8_t* nb = nullptr;
  TCK(t, cudaMalloc(&nb, 66 * cap));
  TCK(t, cudaStreamWaitEvent(t->stream, t->read_done, 0));
  if (t->cap) {
    for (int c = 0; c < 8; c++)
      TCK(t, cudaMemcpyAsync(nb + 4 * c * cap, t->block + 4 * c * t->cap, 4 * t->cap, cudaMemcpyDeviceToDevice, t->stream));
    TCK(t, cudaMemcpyAsync(nb + 32 * cap, t->block + 32 * t->cap, 32 * t->cap, cudaMemcpyDeviceToDevice, t->stream));
    TCK(t, cudaMemcpyAsync(nb + 64 * cap, t->block + 64 * t->cap, t->cap, cudaMemcpyDeviceToDevice, t->stream));
    TCK(t, cudaMemcpyAsync(nb + 65 * cap, t->block + 65 * t->cap, t->cap, cudaMemcpyDeviceToDevice, t->stream));
  }
  const size_t fresh = cap - t->cap;
  for (int c = 0; c < 8; c++) TCK(t, cudaMemsetAsync(nb + 4 * c * cap + 4 * t->cap, 0, 4 * fresh, t->stream));
  TCK(t, cudaMemsetAsync(nb + 32 * cap + 32 * t->cap, 0, 32 * fresh, t->stream));
  TCK(t, cudaMemsetAsync(nb + 64 * cap + t->cap, 0, fresh, t->stream));
  TCK(t, cudaMemsetAsync(nb + 65 * cap + t->cap, 1, fresh, t->stream));
  TCK(t, cudaStreamSynchronize(t->stream));  // no query reads the old block any more (read_done was waited for)
  if (t->block) cudaFree(t->block);
  t->block = nb;
  t->cap = cap;
  return SWM_OK;
}

}  // namespace

extern "C" {

int swm_mappoints_create(int device, int capacity, swm_mappoints** out) {
  if (!out) return SWM_E_INVALID;
  *out = nullptr;
  if (capacity < 0) { g_mappoints_create_error = "negative capacity"; return SWM_E_INVALID; }
  int rc = check_device(device, &g_mappoints_create_error);
  if (rc != SWM_OK) return rc;
  swm_mappoints* t = new swm_mappoints;
  t->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->written, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->read_done, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->staged, cudaEventDisableTiming);
  if (e == cudaSuccess && capacity > 0 && mp_reserve(t, (size_t)capacity) != SWM_OK) e = cudaErrorMemoryAllocation;
  if (e != cudaSuccess) {
    g_mappoints_create_error = cuda_err("swm_mappoints_create", e);
    swm_mappoints_destroy(t);
    return SWM_E_CUDA;
  }
  *out = t;
  return SWM_OK;
}

void swm_mappoints_destroy(swm_mappoints* t) {
  if (!t) return;
  cudaSetDevice(t->device);
  {
    std::lock_guard<std::mutex> lock(t->mu);  // no query or upsert of another thread is inside
  }
  if (t->stream) cudaStreamSynchronize(t->stream);
  if (t->read_done) cudaEventSynchronize(t->read_done);
  if (t->block) cudaFree(t->block);
  if (t->h_stage) cudaFreeHost(t->h_stage);
  t->d_stage.release();
  for (cudaEvent_t e : {t->written, t->read_done, t->staged})
    if (e) cudaEventDestroy(e);
  if (t->stream) cudaStreamDestroy(t->stream);
  delete t;
}

const char* swm_mappoints_last_error(const swm_mappoints* t) { return t ? t->err.c_str() : g_mappoints_create_error.c_str(); }

int32_t swm_mappoints_size(const swm_mappoints* t) {
  if (!t) return 0;
  std::lock_guard<std::mutex> lock(const_cast<swm_mappoints*>(t)->mu);
  return t->size;
}

int swm_mappoints_upsert(swm_mappoints* t, int n, const int32_t* rows, const float* pos, const float* normal,
                         const float* min_d, const float* max_d, const uint8_t* desc, const uint8_t* has_obs,
                         const uint8_t* bad) {
  if (!t) return SWM_E_INVALID;
  if (n < 0 || (n > 0 && (!rows || !pos || !normal || !min_d || !max_d || !desc || !has_obs || !bad))) {
    t->err = "bad argument";
    return SWM_E_INVALID;
  }
  int32_t max_row = -1;
  for (int i = 0; i < n; i++) {
    if (rows[i] < 0) { t->err = "negative row in upsert"; return SWM_E_INVALID; }
    max_row = std::max(max_row, rows[i]);
  }
  if (n == 0) return SWM_OK;
  std::lock_guard<std::mutex> lock(t->mu);
  // a row given twice: the last entry wins (the scatter kernel writes every kept entry exactly once)
  std::vector<int32_t> order((size_t)n);
  for (int i = 0; i < n; i++) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rows[a] < rows[b]; });
  std::vector<int32_t> keep;
  keep.reserve((size_t)n);
  for (int k = 0; k < n; k++)
    if (k + 1 == n || rows[order[k + 1]] != rows[order[k]]) keep.push_back(order[k]);
  const int nk = (int)keep.size();
  TCK(t, cudaSetDevice(t->device));
  int rc;
  if ((rc = mp_reserve(t, (size_t)max_row + 1))) return rc;
  auto a256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t fs = a256((size_t)nk * 4);
  const size_t bytes = fs + 8 * fs + a256((size_t)nk * 32) + 2 * a256((size_t)nk);
  TCK(t, cudaEventSynchronize(t->staged));  // the previous upload out of the pinned buffer has been made
  if (bytes > t->stage_cap) {
    if (t->h_stage) cudaFreeHost(t->h_stage);
    t->h_stage = nullptr;
    t->stage_cap = 0;
    TCK(t, cudaMallocHost(&t->h_stage, bytes + bytes / 2));
    t->stage_cap = bytes + bytes / 2;
  }
  TCK(t, t->d_stage.ensure(bytes));
  uint8_t* h = t->h_stage;
  int32_t* hr = reinterpret_cast<int32_t*>(h);
  float* hf = reinterpret_cast<float*>(h + fs);
  const size_t fn = fs / 4;
  uint8_t* hd = h + 9 * fs;
  uint8_t* hb = hd + a256((size_t)nk * 32);
  for (int k = 0; k < nk; k++) {
    const int i = keep[k];
    hr[k] = rows[i];
    for (int c = 0; c < 3; c++) {
      hf[c * fn + k] = pos[3 * i + c];
      hf[(3 + c) * fn + k] = normal[3 * i + c];
    }
    hf[6 * fn + k] = min_d[i];
    hf[7 * fn + k] = max_d[i];
    memcpy(hd + (size_t)k * 32, desc + (size_t)i * 32, 32);
    hb[k] = has_obs[i] ? 1 : 0;
    hb[a256((size_t)nk) + k] = bad[i] ? 1 : 0;
  }
  TCK(t, cudaStreamWaitEvent(t->stream, t->read_done, 0));  // a write never overtakes a query that still reads
  TCK(t, cudaMemcpyAsync(t->d_stage.p, h, bytes, cudaMemcpyHostToDevice, t->stream));
  TCK(t, cudaEventRecord(t->staged, t->stream));
  mp_scatter_kernel<<<(nk + 255) / 256, 256, 0, t->stream>>>(t->d_stage.as<uint8_t>(), nk, reinterpret_cast<float*>(t->block),
                                                             t->cap, reinterpret_cast<uint4*>(t->block + 32 * t->cap),
                                                             t->block + 64 * t->cap, t->block + 65 * t->cap);
  TCK(t, cudaGetLastError());
  TCK(t, cudaEventRecord(t->written, t->stream));
  t->size = std::max(t->size, max_row + 1);
  return SWM_OK;
}

}  // extern "C"
