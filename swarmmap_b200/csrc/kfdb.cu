// kfdb.cu -- KeyFrameDatabase on the device: DetectRelocalizationCandidates / DetectLoopCandidates with DBoW2's L1
// score (ORB-SLAM2 KeyFrameDatabase.cc as SwarmMap carries it; Thirdparty/DBoW2/DBoW2/ScoringObject.cpp).  The rules
// and the three frozen definitions are in DESIGN.md section 2; results equal the CPU oracle's (tests/test_gpu_kfdb.py).
//
// Storage (grow-only): a pool of the keyframes' BowVectors (word ids + doubles, appended by add), one slot per
// keyframe id ever added (the id -> slot map lives on the host and is never shrunk, so the persistent reloc score of
// an id survives erase / re-add / clear), and the inverted file in CSR order: per word, the live slots sorted by add
// sequence number -- the reference's list order.  The inverted file is rebuilt on the device by the first query
// after a change: (word << 32 | add_seq, slot) pairs of the live keyframes, one radix sort, word offsets.
//
// A query call (nq queries, dense [nq][slots] work arrays):
//   kfdb_walk_kernel      a warp per (query, word) walks the word's list: word count by atomicAdd, and the first
//                         meeting key (position of the word in the query) << 32 | add_seq by 64-bit atomicMin.  Sorting
//                         the listed keyframes by that key gives lKFsSharingWords' order without replaying it;
//   kfdb_exclude_kernel   loop mode: connected keyframes are never listed (their count is cleared);
//   kfdb_max_kernel       maxCommonWords per query, minCommonWords = int(max * 0.8f);
//   kfdb_compact_kernel   the keyframes with count > minCommonWords, keyed (query << 48 | first-meeting key), then
//                         one radix sort over all queries and per-query offsets (after one count read-back);
//   kfdb_score_kernel     a warp per scored keyframe: the word lists are intersected in parallel (binary search), the
//                         terms of the common words summed by one running double in ascending word order, exactly
//                         as L1Scoring::score rounds; float si;
//   kfdb_persist_kernel   reloc mode: the persistent score of every slot becomes that of the batch's last scorer
//                         (the previous values are kept for finish's stale lookups).
// Finish (kfdb_finish_kernel, a CTA per query): covisibility accumulation over the caller's neighbour slots in float,
// stale lookups (latest earlier scorer in the batch, then the persistent state), bestAccScore, the 0.75 retain test,
// first-occurrence de-duplication (atomicMin of the entry index per best slot) and an ordered compaction.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "swm_internal.cuh"

using namespace swm;

namespace {

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    release();
    const size_t want = bytes + bytes / 2 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // grow keeping the first `used` bytes (stream-ordered copy); new bytes are zero
  cudaError_t grow(size_t bytes, size_t used, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    const size_t want = bytes + bytes / 2 + 256;
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(q, 0, want, st)) != cudaSuccess) return e;
    if (used && (e = cudaMemcpyAsync(q, p, used, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (p) cudaFree(p);
    p = q;
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kMaxQueryWords = 65535;  // first-meeting key: 16-bit word position
constexpr int kMaxBatch = 65535;       // compaction key: 16-bit query index
constexpr int kFinishThreads = 256;

// L1Scoring::score(a, b): the common words' terms fabs(vi - wi) - fabs(vi) - fabs(wi) (vi from a, wi from b) added
// to one running double in ascending word order, then -score / 2.0.  The warp walks the shorter list 32 words at a
// time and binary-searches the longer; the terms of a chunk are added in lane order, which is ascending word order.
__device__ double l1_score_warp(const uint32_t* aw, const double* av, int na, const uint32_t* bw, const double* bv,
                                int nb) {
  const int lane = threadIdx.x & 31;
  const bool a_short = na <= nb;
  const uint32_t* sw = a_short ? aw : bw;
  const double* sv = a_short ? av : bv;
  const uint32_t* lw = a_short ? bw : aw;
  const double* lv = a_short ? bv : av;
  const int ns = a_short ? na : nb, nl = a_short ? nb : na;
  double score = 0.0;
  for (int base = 0; base < ns; base += 32) {
    const int i = base + lane;
    double t = 0.0;
    bool hit = false;
    if (i < ns) {
      const uint32_t w = sw[i];
      int lo = 0, hi = nl;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (lw[mid] < w) lo = mid + 1;
        else hi = mid;
      }
      if (lo < nl && lw[lo] == w) {
        const double vi = a_short ? sv[i] : lv[lo], wi = a_short ? lv[lo] : sv[i];
        t = __dsub_rn(__dsub_rn(fabs(__dsub_rn(vi, wi)), fabs(vi)), fabs(wi));
        hit = true;
      }
    }
    unsigned m = __ballot_sync(kFull, hit);
    while (m) {
      const int l = __ffs(m) - 1;
      m &= m - 1;
      score = __dadd_rn(score, __shfl_sync(kFull, t, l));
    }
  }
  return __ddiv_rn(-score, 2.0);
}

__global__ void __launch_bounds__(256) l1_score_pairs_kernel(int npairs, const int32_t* __restrict__ a_off,
                                                             const uint32_t* __restrict__ aw, const double* __restrict__ av,
                                                             const int32_t* __restrict__ b_off,
                                                             const uint32_t* __restrict__ bw, const double* __restrict__ bv,
                                                             double* __restrict__ out) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (i >= npairs) return;
  const int a0 = a_off[i], b0 = b_off[i];
  const double s = l1_score_warp(aw + a0, av + a0, a_off[i + 1] - a0, bw + b0, bv + b0, b_off[i + 1] - b0);
  if ((threadIdx.x & 31) == 0) out[i] = s;
}

// ---- inverted file rebuild
__global__ void kfdb_postings_kernel(int n_live, const int32_t* __restrict__ live, const int64_t* __restrict__ pstart,
                                     const int64_t* __restrict__ slot_off, const int32_t* __restrict__ slot_len,
                                     const uint32_t* __restrict__ add_seq, const uint32_t* __restrict__ pool_words,
                                     unsigned long long* __restrict__ keys, int32_t* __restrict__ vals) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= n_live) return;
  const int s = live[i];
  const int64_t o = slot_off[s], p = pstart[i];
  for (int j = lane; j < slot_len[s]; j += 32) {
    keys[p + j] = ((unsigned long long)pool_words[o + j] << 32) | add_seq[s];
    vals[p + j] = s;
  }
}

// offsets[x] = first position whose group (key >> shift) is >= x, for x in [0, n_groups]
__global__ void group_offsets_kernel(const unsigned long long* __restrict__ keys, int64_t n, int shift, int n_groups,
                                     int32_t* __restrict__ offsets) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const long long g = i < n ? (long long)(keys[i] >> shift) : n_groups;
  const long long prev = i > 0 ? (long long)(keys[i - 1] >> shift) : -1;
  for (long long x = prev + 1; x <= g && x <= n_groups; x++) offsets[x] = (int32_t)i;
}

// ---- query
__global__ void kfdb_walk_kernel(int total, const uint32_t* __restrict__ q_words, const int32_t* __restrict__ q_of,
                                 const int32_t* __restrict__ q_off, const int32_t* __restrict__ inv_off,
                                 const int32_t* __restrict__ inv_slot, const uint32_t* __restrict__ add_seq, int S,
                                 int32_t* __restrict__ count, unsigned long long* __restrict__ key) {
  const int lane = threadIdx.x & 31;
  const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
  for (int j = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); j < total; j += nwarps) {
    const int q = q_of[j];
    const unsigned long long pos = (unsigned long long)(j - q_off[q]) << 32;
    const uint32_t w = q_words[j];
    const int b = inv_off[w], e = inv_off[w + 1];
    for (int p = b + lane; p < e; p += 32) {
      const int s = inv_slot[p];
      const size_t idx = (size_t)q * S + s;
      atomicAdd(count + idx, 1);
      atomicMin(key + idx, pos | add_seq[s]);
    }
  }
}

__global__ void kfdb_exclude_kernel(int n, const int32_t* __restrict__ q_of, const int32_t* __restrict__ slot, int S,
                                    int32_t* __restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && slot[i] >= 0) count[(size_t)q_of[i] * S + slot[i]] = 0;
}

__global__ void __launch_bounds__(256) kfdb_max_kernel(const int32_t* __restrict__ count, int S,
                                                       int32_t* __restrict__ min_common) {
  __shared__ int s_max[8];
  const int q = blockIdx.x;
  int m = 0;
  for (int s = threadIdx.x; s < S; s += 256) m = max(m, count[(size_t)q * S + s]);
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; w++) m = max(m, s_max[w]);
    min_common[q] = (int)__fmul_rn((float)m, 0.8f);  // int minCommonWords = maxCommonWords * 0.8f
  }
}

__global__ void kfdb_compact_kernel(int nq, int S, const int32_t* __restrict__ count,
                                    const unsigned long long* __restrict__ key, const int32_t* __restrict__ min_common,
                                    int32_t* __restrict__ n_out, unsigned long long* __restrict__ out_key,
                                    int32_t* __restrict__ out_slot) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)nq * S) return;
  const int q = (int)(i / S), s = (int)(i % S);
  if (count[i] > min_common[q]) {
    const int k = atomicAdd(n_out, 1);
    out_key[k] = ((unsigned long long)q << 48) | key[i];
    out_slot[k] = s;
  }
}

__global__ void __launch_bounds__(256) kfdb_score_kernel(int n, const unsigned long long* __restrict__ e_key,
                                                         const int32_t* __restrict__ e_slot,
                                                         const int32_t* __restrict__ q_off,
                                                         const uint32_t* __restrict__ q_words,
                                                         const double* __restrict__ q_values,
                                                         const int64_t* __restrict__ slot_off,
                                                         const int32_t* __restrict__ slot_len,
                                                         const uint32_t* __restrict__ pool_words,
                                                         const double* __restrict__ pool_values, int S,
                                                         float* __restrict__ e_score, float* __restrict__ dscore) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (i >= n) return;
  const int q = (int)(e_key[i] >> 48), s = e_slot[i];
  const int a0 = q_off[q];
  const int64_t b0 = slot_off[s];
  const double sc = l1_score_warp(q_words + a0, q_values + a0, q_off[q + 1] - a0, pool_words + b0, pool_values + b0,
                                  slot_len[s]);
  if ((threadIdx.x & 31) == 0) {
    const float si = __double2float_rn(sc);  // float si = mpVoc->score(...)
    e_score[i] = si;
    dscore[(size_t)q * S + s] = si;
  }
}

__global__ void kfdb_persist_kernel(int nq, int S, const int32_t* __restrict__ count,
                                    const int32_t* __restrict__ min_common, const float* __restrict__ dscore,
                                    float* __restrict__ persist) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  for (int q = nq - 1; q >= 0; q--)
    if (count[(size_t)q * S + s] > min_common[q]) {
      persist[s] = dscore[(size_t)q * S + s];
      return;
    }
}

// ---- finish: a CTA per query over its listed entries [e_off[q], e_off[q+1])
__device__ int block_exclusive_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  int before = 0, sum = 0;
  for (int w = 0; w < kFinishThreads / 32; w++) {
    if (w < wid) before += s_warp[w];
    sum += s_warp[w];
  }
  __syncthreads();
  *total = sum;
  return before + incl - v;
}

__global__ void __launch_bounds__(kFinishThreads) kfdb_finish_kernel(
    int mode, int S, const int32_t* __restrict__ e_off, const int32_t* __restrict__ e_slot,
    const float* __restrict__ e_score, const int32_t* __restrict__ nb_off, const int32_t* __restrict__ nb_slot,
    const int32_t* __restrict__ count, const int32_t* __restrict__ min_common, const float* __restrict__ dscore,
    const float* __restrict__ prev_persist, const float* __restrict__ min_score, float* __restrict__ acc_out,
    int32_t* __restrict__ best_out, uint32_t* __restrict__ first, int32_t* __restrict__ cand_out,
    int32_t* __restrict__ n_cand) {
  __shared__ float s_max[kFinishThreads / 32];
  __shared__ int s_warp[kFinishThreads / 32];
  const int q = blockIdx.x, b = e_off[q], e = e_off[q + 1];
  const int mc = min_common[q];
  float m = mode == 0 ? 0.0f : min_score[q];  // bestAccScore's initial value
  for (int i = b + threadIdx.x; i < e; i += kFinishThreads) {
    const float si = e_score[i];
    float acc = si, best_score = si;
    int best = e_slot[i];
    for (int k = nb_off[i]; k < nb_off[i + 1]; k++) {
      const int n = nb_slot[k];
      if (n < 0) continue;
      const int c = count[(size_t)q * S + n];
      float ns;
      if (c > mc) {
        ns = dscore[(size_t)q * S + n];  // scored by this query
      } else if (mode == 0 && c > 0) {   // shares a word, not scored: the stale mRelocScore
        ns = prev_persist[n];
        for (int qq = q - 1; qq >= 0; qq--)
          if (count[(size_t)qq * S + n] > min_common[qq]) {
            ns = dscore[(size_t)qq * S + n];
            break;
          }
      } else {
        continue;
      }
      acc = __fadd_rn(acc, ns);
      if (ns > best_score) {
        best = n;
        best_score = ns;
      }
    }
    acc_out[i] = acc;
    best_out[i] = best;
    m = fmaxf(m, acc);
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
  __syncthreads();
  float best_acc = s_max[0];
  for (int w = 1; w < kFinishThreads / 32; w++) best_acc = fmaxf(best_acc, s_max[w]);
  const float keep = __fmul_rn(0.75f, best_acc);  // minScoreToRetain
  for (int i = b + threadIdx.x; i < e; i += kFinishThreads)
    if (acc_out[i] > keep) atomicMin(first + (size_t)q * S + best_out[i], (uint32_t)(i - b));
  __syncthreads();
  int written = 0;
  for (int base = b; base < e; base += kFinishThreads) {
    const int i = base + threadIdx.x;
    const bool keep_i = i < e && acc_out[i] > keep && first[(size_t)q * S + best_out[i]] == (uint32_t)(i - b);
    int total;
    const int rank = block_exclusive_scan(keep_i ? 1 : 0, s_warp, &total);
    if (keep_i) cand_out[b + written + rank] = best_out[i];
    written += total;
  }
  if (threadIdx.x == 0) n_cand[q] = written;
}

thread_local std::string g_kfdb_create_error;

unsigned blocks_for(long long threads, int per_block = 256) { return (unsigned)((threads + per_block - 1) / per_block); }

}  // namespace

namespace swm {
cudaError_t launch_l1_score_pairs(int npairs, const int32_t* a_off, const uint32_t* a_words, const double* a_values,
                                  const int32_t* b_off, const uint32_t* b_words, const double* b_values, double* out,
                                  cudaStream_t stream) {
  if (npairs <= 0) return cudaSuccess;
  l1_score_pairs_kernel<<<blocks_for((long long)npairs * 32), 256, 0, stream>>>(npairs, a_off, a_words, a_values, b_off,
                                                                                b_words, b_values, out);
  return cudaGetLastError();
}
}  // namespace swm

struct swm_kfdb {
  int device = 0, n_words = 0;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // query begin / end, finish begin / end
  PinnedArena arena;
  // host: id -> slot (never shrinks), per slot its pool range, add sequence and liveness
  std::unordered_map<uint64_t, int> slot_of;
  std::vector<uint64_t> id_of;
  std::vector<int64_t> slot_off;
  std::vector<int32_t> slot_len;
  std::vector<uint32_t> add_seq;
  std::vector<uint8_t> live;
  int64_t n_live = 0, pool_used = 0;
  uint32_t next_seq = 1;
  bool dirty = true;
  uint64_t version = 0;  // bumped by add / erase / clear
  // device
  Buf pool_words, pool_values, persist, prev_persist;
  Buf d_slot_off, d_slot_len, d_add_seq, inv_off, inv_slot;
  Buf pkeys[2], pvals[2], sort_tmp;
  Buf count, key, dscore, min_common, n_out, ekeys[2], eslot[2], e_off, e_score;
  Buf f_acc, f_best, f_cand, f_ncand;
  // the last query, for finish
  bool pending = false;
  uint64_t pending_version = 0;
  int q_mode = 0, q_nq = 0, q_S = 0;
  std::vector<int32_t> q_listed_off;  // per query, listed entries (lScoreAndMatch)
  std::vector<int32_t> q_listed_slot;
  std::vector<float> q_listed_score, q_min_score;
  float last_ms[2] = {0.f, 0.f};

  void free_all() {
    for (Buf* x : {&pool_words, &pool_values, &persist, &prev_persist, &d_slot_off, &d_slot_len, &d_add_seq, &inv_off,
                   &inv_slot, &pkeys[0], &pkeys[1], &pvals[0], &pvals[1], &sort_tmp, &count, &key, &dscore,
                   &min_common, &n_out, &ekeys[0], &ekeys[1], &eslot[0], &eslot[1], &e_off, &e_score, &f_acc, &f_best,
                   &f_cand, &f_ncand})
      x->release();
    arena.release();
    for (auto& e : ev)
      if (e) cudaEventDestroy(e);
  }
};

#define KCK(db, call)                \
  do {                               \
    cudaError_t e_ = (call);         \
    if (e_ != cudaSuccess) {         \
      (db)->err = cuda_err(#call, e_); \
      return SWM_E_CUDA;             \
    }                                \
  } while (0)

namespace {

// CSR sanity: offsets from 0, non-decreasing, words strictly ascending inside each vector and < n_words.
bool csr_ok(int n, const int32_t* off, const uint32_t* words, int n_words, int max_len, std::string* err) {
  if (off[0] != 0) { *err = "offsets[0] must be 0"; return false; }
  for (int i = 0; i < n; i++) {
    const int len = off[i + 1] - off[i];
    if (len < 0 || len > max_len) { *err = "bad BowVector length"; return false; }
    for (int j = off[i]; j < off[i + 1]; j++) {
      if (words[j] >= (uint32_t)n_words) { *err = "word id >= the vocabulary's size"; return false; }
      if (j > off[i] && words[j] <= words[j - 1]) { *err = "word ids not strictly ascending"; return false; }
    }
  }
  return true;
}

int sort_pairs(swm_kfdb* db, Buf* keys, Buf* vals, int64_t n, int end_bit, int* which) {
  cub::DoubleBuffer<unsigned long long> k(keys[0].as<unsigned long long>(), keys[1].as<unsigned long long>());
  cub::DoubleBuffer<int32_t> v(vals[0].as<int32_t>(), vals[1].as<int32_t>());
  size_t tmp = 0;
  KCK(db, cub::DeviceRadixSort::SortPairs(nullptr, tmp, k, v, n, 0, end_bit, db->stream));
  KCK(db, db->sort_tmp.ensure(tmp));
  KCK(db, cub::DeviceRadixSort::SortPairs(db->sort_tmp.p, tmp, k, v, n, 0, end_bit, db->stream));
  *which = k.selector;
  return SWM_OK;
}

int bits_for(uint64_t x) {
  int b = 0;
  while (b < 64 && (x >> b)) b++;
  return std::max(b, 1);
}

int rebuild(swm_kfdb* db) {
  const int S = (int)db->id_of.size();
  std::vector<int32_t> live;
  std::vector<int64_t> pstart;
  int64_t total = 0;
  for (int s = 0; s < S; s++)
    if (db->live[s]) {
      live.push_back(s);
      pstart.push_back(total);
      total += db->slot_len[s];
    }
  if (total > INT32_MAX) { db->err = "inverted file exceeds 2^31 postings"; return SWM_E_CAPACITY; }
  KCK(db, db->arena.begin((size_t)S * 16 + live.size() * 12 + 2048, db->stream));
  const int64_t* d_off = db->arena.put(db->slot_off.data(), S);
  const int32_t* d_len = db->arena.put(db->slot_len.data(), S);
  const uint32_t* d_seq = db->arena.put(db->add_seq.data(), S);
  const int32_t* d_live = db->arena.put(live.data(), live.size());
  const int64_t* d_pstart = db->arena.put(pstart.data(), pstart.size());
  KCK(db, db->arena.flush(db->stream));
  KCK(db, db->d_slot_off.ensure((size_t)S * 8 + 8));
  KCK(db, db->d_slot_len.ensure((size_t)S * 4 + 4));
  KCK(db, db->d_add_seq.ensure((size_t)S * 4 + 4));
  KCK(db, cudaMemcpyAsync(db->d_slot_off.p, d_off, (size_t)S * 8, cudaMemcpyDeviceToDevice, db->stream));
  KCK(db, cudaMemcpyAsync(db->d_slot_len.p, d_len, (size_t)S * 4, cudaMemcpyDeviceToDevice, db->stream));
  KCK(db, cudaMemcpyAsync(db->d_add_seq.p, d_seq, (size_t)S * 4, cudaMemcpyDeviceToDevice, db->stream));
  KCK(db, db->inv_off.ensure(((size_t)db->n_words + 1) * 4));
  KCK(db, db->inv_slot.ensure((size_t)total * 4 + 4));
  if (total == 0) {
    KCK(db, cudaMemsetAsync(db->inv_off.p, 0, ((size_t)db->n_words + 1) * 4, db->stream));
  } else {
    for (int i = 0; i < 2; i++) {
      KCK(db, db->pkeys[i].ensure((size_t)total * 8));
      KCK(db, db->pvals[i].ensure((size_t)total * 4));
    }
    kfdb_postings_kernel<<<blocks_for((long long)live.size() * 32), 256, 0, db->stream>>>(
        (int)live.size(), d_live, d_pstart, db->d_slot_off.as<int64_t>(), db->d_slot_len.as<int32_t>(),
        db->d_add_seq.as<uint32_t>(), db->pool_words.as<uint32_t>(), db->pkeys[0].as<unsigned long long>(),
        db->pvals[0].as<int32_t>());
    KCK(db, cudaGetLastError());
    int which = 0;
    int rc = sort_pairs(db, db->pkeys, db->pvals, total, 32 + bits_for((uint64_t)db->n_words), &which);
    if (rc != SWM_OK) return rc;
    group_offsets_kernel<<<blocks_for(total + 1), 256, 0, db->stream>>>(db->pkeys[which].as<unsigned long long>(), total,
                                                                         32, db->n_words, db->inv_off.as<int32_t>());
    KCK(db, cudaGetLastError());
    KCK(db, cudaMemcpyAsync(db->inv_slot.p, db->pvals[which].p, (size_t)total * 4, cudaMemcpyDeviceToDevice, db->stream));
  }
  // the arena is reused by the caller right after: its copies must have been consumed
  KCK(db, cudaStreamSynchronize(db->stream));
  db->dirty = false;
  return SWM_OK;
}

}  // namespace

extern "C" {

int swm_kfdb_create(swm_vocab* v, swm_kfdb** out) {
  if (!out) return SWM_E_INVALID;
  *out = nullptr;
  VocabProps vp;
  if (!v || vocab_props(v, &vp) != SWM_OK) { g_kfdb_create_error = "no vocabulary"; return SWM_E_INVALID; }
  if (vp.scoring != 0) {
    g_kfdb_create_error = "the vocabulary's scoring type is not L1_NORM: only DBoW2's L1 score is implemented";
    return SWM_E_INVALID;
  }
  std::string err;
  int rc = check_device(vp.device, &err);
  if (rc != SWM_OK) { g_kfdb_create_error = err; return rc; }
  swm_kfdb* db = new swm_kfdb();
  db->device = vp.device;
  db->n_words = vp.n_words;
  bool ok = cudaSetDevice(vp.device) == cudaSuccess &&
            cudaStreamCreateWithFlags(&db->stream, cudaStreamNonBlocking) == cudaSuccess;
  for (auto& e : db->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
  if (!ok) {
    g_kfdb_create_error = cuda_err("swm_kfdb_create", cudaGetLastError());
    db->free_all();
    if (db->stream) cudaStreamDestroy(db->stream);
    delete db;
    return SWM_E_CUDA;
  }
  *out = db;
  return SWM_OK;
}

void swm_kfdb_destroy(swm_kfdb* db) {
  if (!db) return;
  cudaSetDevice(db->device);
  if (db->stream) cudaStreamSynchronize(db->stream);
  db->free_all();
  if (db->stream) cudaStreamDestroy(db->stream);
  delete db;
}

const char* swm_kfdb_last_error(const swm_kfdb* db) { return db ? db->err.c_str() : g_kfdb_create_error.c_str(); }

int64_t swm_kfdb_size(const swm_kfdb* db) { return db ? db->n_live : 0; }

float swm_kfdb_last_device_ms(const swm_kfdb* db) { return db ? db->last_ms[0] + db->last_ms[1] : 0.f; }

int swm_kfdb_add(swm_kfdb* db, int n, const uint64_t* kf_ids, const int32_t* offsets, const uint32_t* word_ids,
                 const double* values) {
  if (!db) return SWM_E_INVALID;
  if (n < 0 || (n > 0 && (!kf_ids || !offsets || (offsets[n] > 0 && (!word_ids || !values))))) {
    db->err = "bad argument";
    return SWM_E_INVALID;
  }
  if (n == 0) return SWM_OK;
  if (!csr_ok(n, offsets, word_ids, db->n_words, INT32_MAX, &db->err)) return SWM_E_INVALID;
  {
    std::unordered_map<uint64_t, int> seen;
    for (int i = 0; i < n; i++) {
      auto it = db->slot_of.find(kf_ids[i]);
      if ((it != db->slot_of.end() && db->live[it->second]) || !seen.emplace(kf_ids[i], i).second) {
        db->err = "keyframe id " + std::to_string(kf_ids[i]) + " is already in the database";
        return SWM_E_INVALID;
      }
    }
  }
  if ((uint64_t)db->next_seq + n >= 0xFFFFFFFFull) { db->err = "add sequence numbers exhausted"; return SWM_E_CAPACITY; }
  KCK(db, cudaSetDevice(db->device));
  const int64_t nw = offsets[n];
  // slots first (the persistent score of a new slot starts at 0.0f: frozen definition 2)
  int S = (int)db->id_of.size();
  int new_slots = 0;
  for (int i = 0; i < n; i++) new_slots += db->slot_of.count(kf_ids[i]) ? 0 : 1;
  KCK(db, db->persist.grow((size_t)(S + new_slots) * 4, (size_t)S * 4, db->stream));
  KCK(db, db->prev_persist.grow((size_t)(S + new_slots) * 4, (size_t)S * 4, db->stream));
  KCK(db, db->pool_words.grow((size_t)(db->pool_used + nw) * 4, (size_t)db->pool_used * 4, db->stream));
  KCK(db, db->pool_values.grow((size_t)(db->pool_used + nw) * 8, (size_t)db->pool_used * 8, db->stream));
  KCK(db, db->arena.begin((size_t)nw * 12 + 512, db->stream));
  const uint32_t* dw = db->arena.put(word_ids, nw);
  const double* dv = db->arena.put(values, nw);
  KCK(db, db->arena.flush(db->stream));
  KCK(db, cudaMemcpyAsync(db->pool_words.as<uint32_t>() + db->pool_used, dw, nw * 4, cudaMemcpyDeviceToDevice, db->stream));
  KCK(db, cudaMemcpyAsync(db->pool_values.as<double>() + db->pool_used, dv, nw * 8, cudaMemcpyDeviceToDevice, db->stream));
  for (int i = 0; i < n; i++) {
    auto it = db->slot_of.find(kf_ids[i]);
    int s;
    if (it == db->slot_of.end()) {
      s = S++;
      db->slot_of.emplace(kf_ids[i], s);
      db->id_of.push_back(kf_ids[i]);
      db->slot_off.push_back(0);
      db->slot_len.push_back(0);
      db->add_seq.push_back(0);
      db->live.push_back(0);
    } else {
      s = it->second;
    }
    db->slot_off[s] = db->pool_used + offsets[i];
    db->slot_len[s] = offsets[i + 1] - offsets[i];
    db->add_seq[s] = db->next_seq++;
    db->live[s] = 1;
    db->n_live++;
  }
  db->pool_used += nw;
  // the arena is reused by the next call: its copy has to be consumed first
  KCK(db, cudaStreamSynchronize(db->stream));
  db->dirty = true;
  db->version++;
  return SWM_OK;
}

int swm_kfdb_erase(swm_kfdb* db, int n, const uint64_t* kf_ids) {
  if (!db) return SWM_E_INVALID;
  if (n < 0 || (n > 0 && !kf_ids)) { db->err = "bad argument"; return SWM_E_INVALID; }
  for (int i = 0; i < n; i++) {
    auto it = db->slot_of.find(kf_ids[i]);
    if (it != db->slot_of.end() && db->live[it->second]) {
      db->live[it->second] = 0;
      db->n_live--;
    }
  }
  db->dirty = true;
  db->version++;
  return SWM_OK;
}

int swm_kfdb_clear(swm_kfdb* db) {
  if (!db) return SWM_E_INVALID;
  std::fill(db->live.begin(), db->live.end(), 0);
  db->n_live = 0;
  db->pool_used = 0;  // every BowVector is dead; the slots and their persistent scores stay
  db->dirty = true;
  db->version++;
  return SWM_OK;
}

int swm_kfdb_query(swm_kfdb* db, int mode, int nq, const int32_t* q_offsets, const uint32_t* q_words,
                   const double* q_values, const float* min_score, const int32_t* conn_offsets,
                   const uint64_t* conn_ids, int32_t* scored_offsets, uint64_t* scored_ids, float* scored_scores,
                   int32_t scored_cap) {
  if (!db) return SWM_E_INVALID;
  if ((mode != SWM_KFDB_RELOC && mode != SWM_KFDB_LOOP) || nq < 1 || nq > kMaxBatch || !q_offsets || !scored_offsets ||
      scored_cap < 0 || (scored_cap > 0 && (!scored_ids || !scored_scores)) ||
      (q_offsets[nq] > 0 && (!q_words || !q_values)) || (mode == SWM_KFDB_LOOP && !min_score) ||
      (conn_offsets && conn_offsets[nq] > 0 && !conn_ids)) {
    db->err = "bad argument";
    return SWM_E_INVALID;
  }
  if (!csr_ok(nq, q_offsets, q_words, db->n_words, kMaxQueryWords, &db->err)) return SWM_E_INVALID;
  const bool loop = mode == SWM_KFDB_LOOP;
  if (loop && conn_offsets) {
    bool ok = conn_offsets[0] == 0;
    for (int q = 0; q < nq; q++) ok = ok && conn_offsets[q + 1] >= conn_offsets[q];
    if (!ok) { db->err = "bad connected-keyframe offsets"; return SWM_E_INVALID; }
  }
  KCK(db, cudaSetDevice(db->device));
  db->pending = false;
  KCK(db, cudaEventRecord(db->ev[0], db->stream));
  if (db->dirty) {
    int rc = rebuild(db);
    if (rc != SWM_OK) return rc;
  }
  const int S = (int)db->id_of.size();
  const int total = q_offsets[nq];
  std::vector<int32_t> q_of(total);
  for (int q = 0; q < nq; q++)
    for (int j = q_offsets[q]; j < q_offsets[q + 1]; j++) q_of[j] = q;
  std::vector<int32_t> ex_q, ex_slot;  // loop mode: (query, slot) of connected keyframes in the database
  if (loop && conn_offsets)
    for (int q = 0; q < nq; q++)
      for (int j = conn_offsets[q]; j < conn_offsets[q + 1]; j++) {
        auto it = db->slot_of.find(conn_ids[j]);
        if (it != db->slot_of.end()) {
          ex_q.push_back(q);
          ex_slot.push_back(it->second);
        }
      }
  KCK(db, db->arena.begin((size_t)total * 16 + (size_t)nq * 4 + ex_q.size() * 8 + 2048, db->stream));
  const int32_t* d_qoff = db->arena.put(q_offsets, nq + 1);
  const uint32_t* d_qw = db->arena.put(q_words, total);
  const double* d_qv = db->arena.put(q_values, total);
  const int32_t* d_qof = db->arena.put(q_of.data(), total);
  const int32_t* d_exq = db->arena.put(ex_q.data(), ex_q.size());
  const int32_t* d_exs = db->arena.put(ex_slot.data(), ex_slot.size());
  KCK(db, db->arena.flush(db->stream));

  const size_t dense = (size_t)nq * std::max(S, 1);
  KCK(db, db->count.ensure(dense * 4));
  KCK(db, db->key.ensure(dense * 8));
  KCK(db, db->dscore.ensure(dense * 4));
  KCK(db, db->min_common.ensure((size_t)nq * 4));
  KCK(db, db->n_out.ensure(4));
  KCK(db, db->e_off.ensure((size_t)(nq + 1) * 4));
  KCK(db, cudaMemsetAsync(db->count.p, 0, dense * 4, db->stream));
  KCK(db, cudaMemsetAsync(db->key.p, 0xFF, dense * 8, db->stream));
  KCK(db, cudaMemsetAsync(db->n_out.p, 0, 4, db->stream));
  if (total > 0 && db->n_live > 0) {
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, db->device);
    const long long warps = std::min<long long>(total, (long long)n_sm * 64);
    kfdb_walk_kernel<<<blocks_for(warps * 32), 256, 0, db->stream>>>(
        total, d_qw, d_qof, d_qoff, db->inv_off.as<int32_t>(), db->inv_slot.as<int32_t>(), db->d_add_seq.as<uint32_t>(),
        S, db->count.as<int32_t>(), db->key.as<unsigned long long>());
    KCK(db, cudaGetLastError());
  }
  if (!ex_q.empty()) {
    kfdb_exclude_kernel<<<blocks_for((long long)ex_q.size()), 256, 0, db->stream>>>((int)ex_q.size(), d_exq, d_exs, S,
                                                                                  db->count.as<int32_t>());
    KCK(db, cudaGetLastError());
  }
  kfdb_max_kernel<<<nq, 256, 0, db->stream>>>(db->count.as<int32_t>(), S, db->min_common.as<int32_t>());
  KCK(db, cudaGetLastError());
  int n_scored = 0;
  if (S > 0) {
    KCK(db, db->ekeys[0].ensure(dense * 8));
    KCK(db, db->eslot[0].ensure(dense * 4));
    kfdb_compact_kernel<<<blocks_for((long long)nq * S), 256, 0, db->stream>>>(
        nq, S, db->count.as<int32_t>(), db->key.as<unsigned long long>(), db->min_common.as<int32_t>(),
        db->n_out.as<int32_t>(), db->ekeys[0].as<unsigned long long>(), db->eslot[0].as<int32_t>());
    KCK(db, cudaGetLastError());
    KCK(db, cudaMemcpyAsync(db->arena.h, db->n_out.p, 4, cudaMemcpyDeviceToHost, db->stream));
    KCK(db, cudaStreamSynchronize(db->stream));
    memcpy(&n_scored, db->arena.h, 4);
  }
  int which = 0;
  if (n_scored > 0) {
    KCK(db, db->ekeys[1].ensure((size_t)n_scored * 8));
    KCK(db, db->eslot[1].ensure((size_t)n_scored * 4));
    KCK(db, db->e_score.ensure((size_t)n_scored * 4));
    int rc = sort_pairs(db, db->ekeys, db->eslot, n_scored, 48 + bits_for((uint64_t)nq), &which);
    if (rc != SWM_OK) return rc;
    group_offsets_kernel<<<blocks_for((long long)n_scored + 1), 256, 0, db->stream>>>(
        db->ekeys[which].as<unsigned long long>(), n_scored, 48, nq, db->e_off.as<int32_t>());
    KCK(db, cudaGetLastError());
    kfdb_score_kernel<<<blocks_for((long long)n_scored * 32), 256, 0, db->stream>>>(
        n_scored, db->ekeys[which].as<unsigned long long>(), db->eslot[which].as<int32_t>(), d_qoff, d_qw, d_qv,
        db->d_slot_off.as<int64_t>(), db->d_slot_len.as<int32_t>(), db->pool_words.as<uint32_t>(),
        db->pool_values.as<double>(), S, db->e_score.as<float>(), db->dscore.as<float>());
    KCK(db, cudaGetLastError());
  } else {
    KCK(db, cudaMemsetAsync(db->e_off.p, 0, (size_t)(nq + 1) * 4, db->stream));
  }
  // read back: per-query offsets, slots and scores of the scored entries (through the pinned arena, after its inputs)
  const size_t h_off = (db->arena.used + 255) & ~(size_t)255;
  const size_t need = h_off + (size_t)(nq + 1) * 4 + (size_t)n_scored * 8 + 512;
  if (need > db->arena.cap) {  // grow keeping the device inputs the score kernel has read: synchronise first
    KCK(db, cudaStreamSynchronize(db->stream));
    PinnedArena bigger;
    KCK(db, bigger.begin(need, db->stream));
    std::swap(bigger, db->arena);
    bigger.release();
  }
  int32_t* h_eoff = reinterpret_cast<int32_t*>(db->arena.h + h_off);
  int32_t* h_slot = h_eoff + (nq + 1);
  float* h_score = reinterpret_cast<float*>(h_slot + n_scored);
  KCK(db, cudaMemcpyAsync(h_eoff, db->e_off.p, (size_t)(nq + 1) * 4, cudaMemcpyDeviceToHost, db->stream));
  if (n_scored > 0) {
    KCK(db, cudaMemcpyAsync(h_slot, db->eslot[which].p, (size_t)n_scored * 4, cudaMemcpyDeviceToHost, db->stream));
    KCK(db, cudaMemcpyAsync(h_score, db->e_score.p, (size_t)n_scored * 4, cudaMemcpyDeviceToHost, db->stream));
  }
  KCK(db, cudaEventRecord(db->ev[1], db->stream));
  KCK(db, cudaStreamSynchronize(db->stream));
  // lScoreAndMatch: every scored keyframe (reloc), those with si >= minScore (loop)
  db->q_listed_off.assign(nq + 1, 0);
  db->q_listed_slot.clear();
  db->q_listed_score.clear();
  for (int q = 0; q < nq; q++) {
    for (int i = h_eoff[q]; i < h_eoff[q + 1]; i++)
      if (!loop || h_score[i] >= min_score[q]) {
        db->q_listed_slot.push_back(h_slot[i]);
        db->q_listed_score.push_back(h_score[i]);
      }
    db->q_listed_off[q + 1] = (int32_t)db->q_listed_slot.size();
  }
  const int n_listed = (int)db->q_listed_slot.size();
  memcpy(scored_offsets, db->q_listed_off.data(), (size_t)(nq + 1) * 4);
  if (n_listed > scored_cap) {
    db->err = "scored capacity " + std::to_string(scored_cap) + " < " + std::to_string(n_listed);
    return SWM_E_CAPACITY;
  }
  for (int i = 0; i < n_listed; i++) {
    scored_ids[i] = db->id_of[db->q_listed_slot[i]];
    scored_scores[i] = db->q_listed_score[i];
  }
  if (!loop && S > 0) {  // mRelocScore of this batch's scored keyframes; finish reads the values from before it
    KCK(db, cudaMemcpyAsync(db->prev_persist.p, db->persist.p, (size_t)S * 4, cudaMemcpyDeviceToDevice, db->stream));
    kfdb_persist_kernel<<<blocks_for(S), 256, 0, db->stream>>>(nq, S, db->count.as<int32_t>(),
                                                                db->min_common.as<int32_t>(), db->dscore.as<float>(),
                                                                db->persist.as<float>());
    KCK(db, cudaGetLastError());
  }
  cudaEventElapsedTime(&db->last_ms[0], db->ev[0], db->ev[1]);
  db->last_ms[1] = 0.f;
  db->q_mode = mode;
  db->q_nq = nq;
  db->q_S = S;
  db->q_min_score.assign(nq, 0.f);
  if (loop) std::copy(min_score, min_score + nq, db->q_min_score.begin());
  db->pending = true;
  db->pending_version = db->version;
  return SWM_OK;
}

int swm_kfdb_finish(swm_kfdb* db, const int32_t* neigh_offsets, const uint64_t* neigh_ids, int32_t* cand_offsets,
                    uint64_t* cand_ids, int32_t cand_cap) {
  if (!db) return SWM_E_INVALID;
  if (!db->pending || db->pending_version != db->version) {
    db->err = "swm_kfdb_finish needs a swm_kfdb_query with no add / erase / clear after it";
    return SWM_E_STATE;
  }
  const int nq = db->q_nq, S = db->q_S, n_listed = (int)db->q_listed_slot.size();
  if (!cand_offsets || cand_cap < 0 || (cand_cap > 0 && !cand_ids) || (n_listed > 0 && !neigh_offsets)) {
    db->err = "bad argument";
    return SWM_E_INVALID;
  }
  std::vector<int32_t> nb_off(n_listed + 1, 0), nb_slot;
  if (n_listed > 0) {
    if (neigh_offsets[0] != 0) { db->err = "neigh_offsets[0] must be 0"; return SWM_E_INVALID; }
    for (int i = 0; i < n_listed; i++)
      if (neigh_offsets[i + 1] < neigh_offsets[i]) { db->err = "bad neighbour offsets"; return SWM_E_INVALID; }
    if (neigh_offsets[n_listed] > 0 && !neigh_ids) { db->err = "bad argument"; return SWM_E_INVALID; }
    nb_slot.resize(neigh_offsets[n_listed]);
    for (int j = 0; j < neigh_offsets[n_listed]; j++) {
      auto it = db->slot_of.find(neigh_ids[j]);
      nb_slot[j] = it == db->slot_of.end() ? -1 : it->second;
    }
    memcpy(nb_off.data(), neigh_offsets, (size_t)(n_listed + 1) * 4);
  }
  KCK(db, cudaSetDevice(db->device));
  KCK(db, cudaEventRecord(db->ev[2], db->stream));
  KCK(db, db->arena.begin((size_t)n_listed * 12 + nb_slot.size() * 4 + (size_t)nq * 12 + 4096, db->stream));
  const int32_t* d_eoff = db->arena.put(db->q_listed_off.data(), nq + 1);
  const int32_t* d_eslot = db->arena.put(db->q_listed_slot.data(), n_listed);
  const float* d_escore = db->arena.put(db->q_listed_score.data(), n_listed);
  const int32_t* d_nboff = db->arena.put(nb_off.data(), n_listed + 1);
  const int32_t* d_nbslot = db->arena.put(nb_slot.data(), nb_slot.size());
  const float* d_ms = db->arena.put(db->q_min_score.data(), nq);
  KCK(db, db->arena.flush(db->stream));
  KCK(db, db->f_acc.ensure((size_t)n_listed * 4 + 4));
  KCK(db, db->f_best.ensure((size_t)n_listed * 4 + 4));
  KCK(db, db->f_cand.ensure((size_t)n_listed * 4 + 4));
  KCK(db, db->f_ncand.ensure((size_t)nq * 4));
  // first-occurrence marks, [nq][S] uint32, in the first-meeting key array (dead after the query's compaction)
  KCK(db, cudaMemsetAsync(db->key.p, 0xFF, (size_t)nq * std::max(S, 1) * 4, db->stream));
  kfdb_finish_kernel<<<nq, kFinishThreads, 0, db->stream>>>(
      db->q_mode, S, d_eoff, d_eslot, d_escore, d_nboff, d_nbslot, db->count.as<int32_t>(), db->min_common.as<int32_t>(),
      db->dscore.as<float>(), db->prev_persist.as<float>(), d_ms, db->f_acc.as<float>(), db->f_best.as<int32_t>(),
      db->key.as<uint32_t>(), db->f_cand.as<int32_t>(), db->f_ncand.as<int32_t>());
  KCK(db, cudaGetLastError());
  const size_t h_off = (db->arena.used + 255) & ~(size_t)255;
  int32_t* h_ncand = reinterpret_cast<int32_t*>(db->arena.h + h_off);
  int32_t* h_cand = h_ncand + nq;
  if (h_off + (size_t)(nq + n_listed) * 4 > db->arena.cap) { db->err = "internal: arena overflow"; return SWM_E_CAPACITY; }
  KCK(db, cudaMemcpyAsync(h_ncand, db->f_ncand.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, db->stream));
  if (n_listed) KCK(db, cudaMemcpyAsync(h_cand, db->f_cand.p, (size_t)n_listed * 4, cudaMemcpyDeviceToHost, db->stream));
  KCK(db, cudaEventRecord(db->ev[3], db->stream));
  KCK(db, cudaStreamSynchronize(db->stream));
  cudaEventElapsedTime(&db->last_ms[1], db->ev[2], db->ev[3]);
  cand_offsets[0] = 0;
  for (int q = 0; q < nq; q++) cand_offsets[q + 1] = cand_offsets[q] + h_ncand[q];
  if (cand_offsets[nq] > cand_cap) {
    db->err = "candidate capacity " + std::to_string(cand_cap) + " < " + std::to_string(cand_offsets[nq]);
    return SWM_E_CAPACITY;
  }
  for (int q = 0; q < nq; q++)
    for (int k = 0; k < h_ncand[q]; k++)
      cand_ids[cand_offsets[q] + k] = db->id_of[h_cand[db->q_listed_off[q] + k]];
  return SWM_OK;
}

}  // extern "C"
