// bow.cu -- DBoW2 TemplatedVocabulary<FORB>::transform on the device (SURVEY.md section 8(f) rank 2).
//
// Reference: code/Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1151-1218 (features -> BowVector + FeatureVector),
// :1242-1283 (one feature down the tree), :1478-1522 (binary vocabulary layout), FORB.cpp:82-102 (distance),
// BowVector.cpp:33-90 (addWeight / addIfNotExist / normalize), FeatureVector.cpp:31-45 (addFeature); callers
// Frame::ComputeBoW (code/src/Frame.cc:445-452) and KeyFrame::ComputeBoW (code/src/KeyFrame.cc:126-133), levelsup = 4,
// and the server's recomputation for every received keyframe (code/src/Map.cc:372-385).
//
// Two kernels per batch of frames:
//   bow_descend_kernel   16 lanes per descriptor walk the tree: each lane takes children lane, lane + 16, ... of the
//                        current node (k = 10 in ORBvoc), the minimum of (distance << 20 | child position) over the
//                        16 lanes picks the reference's winner (strict <, first child wins ties);
//   bow_assemble_kernel  one CTA per frame turns the per-feature (word, node, weight) triples into the two ordered
//                        containers: bitonic sort of (key << 32 | feature index) in shared memory, run heads by a
//                        block scan, TF sums as the reference's repeated additions, L1 / L2 norm accumulated
//                        sequentially in ascending word order (the std::map iteration order), IEEE division.
// Results are bit-identical to the oracle's std::map implementation (tests/test_gpu_bow.py).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "swm_internal.cuh"

using namespace swm;

namespace {

struct VocabDev {
  const uint4* desc;        // 2 x uint4 per node
  const int32_t* child_off; // n_nodes + 1
  const int32_t* child;     // child ids, file order
  const int32_t* word;      // word id of a leaf
  const float* weight;      // node weight as stored in the file
  int L;
};

__device__ __forceinline__ int hamming256(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) +
         __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// desc: [batch][cap] descriptors; n: keypoints per frame.  Per feature: word id, node id at level L - levelsup, weight.
__global__ void __launch_bounds__(256) bow_descend_kernel(const uint4* __restrict__ desc, const int32_t* __restrict__ n,
                                                          int cap, int batch, VocabDev v, int levelsup,
                                                          int32_t* __restrict__ word_of, int32_t* __restrict__ node_of,
                                                          float* __restrict__ w_of) {
  const long long g = ((long long)blockIdx.x * 256 + threadIdx.x) >> 4;
  const int sub = threadIdx.x & 15;
  const int b = (int)(g / cap), i = (int)(g % cap);
  if (b >= batch || i >= n[b]) return;  // uniform over the 16 lanes of a group
  const unsigned mask = 0xFFFFu << (threadIdx.x & 16);
  const uint4 q0 = __ldg(desc + 2 * g), q1 = __ldg(desc + 2 * g + 1);
  const int nid_level = v.L - levelsup;
  int final_id = 0, level = 0, nid = nid_level <= 0 ? 0 : -1;
  for (;;) {
    const int off = __ldg(v.child_off + final_id), cnt = __ldg(v.child_off + final_id + 1) - off;
    if (cnt == 0) break;  // isLeaf()
    level++;
    unsigned best = 0xFFFFFFFFu;
    for (int c = sub; c < cnt; c += 16) {
      const int id = __ldg(v.child + off + c);
      const int d = hamming256(q0, q1, __ldg(v.desc + 2 * id), __ldg(v.desc + 2 * id + 1));
      best = min(best, ((unsigned)d << 20) | (unsigned)c);  // d < best_d, first child wins ties (:1262-1271)
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(mask, best, o, 16));
    final_id = __ldg(v.child + off + (int)(best & 0xFFFFFu));
    if (level == nid_level) nid = final_id;  // :1275-1276
  }
  if (sub == 0) {
    // a leaf above nid_level leaves *nid unset in the reference (uninitialised in the caller): defined as the leaf
    word_of[g] = __ldg(v.word + final_id);
    node_of[g] = nid < 0 ? final_id : nid;
    w_of[g] = __ldg(v.weight + final_id);
  }
}

constexpr int kAsmThreads = 1024;

// ascending bitonic sort of P (power of two) 64-bit keys in shared memory
__device__ void bitonic_sort(unsigned long long* s, int P) {
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int idx = threadIdx.x; idx < P; idx += kAsmThreads) {
        const int ixj = idx ^ j;
        if (ixj > idx) {
          const unsigned long long a = s[idx], b = s[ixj];
          if (((idx & k) == 0) == (a > b)) {
            s[idx] = b;
            s[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
}

// Exclusive scan of one flag per position over P positions (each thread owns P / kAsmThreads consecutive ones).
// Returns the total; rank_out(p) is delivered through the callback for flagged positions.
template <class Flag, class Emit>
__device__ int scan_heads(int P, int* s_warp, Flag flag, Emit emit) {
  const int per = (P + kAsmThreads - 1) / kAsmThreads;
  const int p0 = threadIdx.x * per;
  int local = 0;
  for (int p = p0; p < p0 + per && p < P; p++) local += flag(p) ? 1 : 0;
  int incl = local;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xFFFFFFFFu, w, o);
      if (lane >= o) w += t;
    }
    s_warp[32 + lane] = w;  // inclusive over warps
  }
  __syncthreads();
  const int total = s_warp[32 + 31];
  int rank = incl - local + (wid ? s_warp[32 + wid - 1] : 0);
  for (int p = p0; p < p0 + per && p < P; p++)
    if (flag(p)) emit(p, rank++);
  __syncthreads();
  return total;
}

struct BowOutDev {
  uint32_t* word_ids;   // [batch][cap]
  double* word_values;  // [batch][cap]
  int32_t* n_words;     // [batch]
  uint32_t* node_ids;   // [batch][cap]
  int32_t* offsets;     // [batch][cap + 1]
  uint32_t* feats;      // [batch][cap]
  int32_t* n_nodes;     // [batch]
};

// One CTA per frame.  weighting: 0 TF_IDF, 1 TF, 2 IDF, 3 BINARY; norm: 0 none, 1 L1, 2 L2 (scoring object).
__global__ void __launch_bounds__(kAsmThreads) bow_assemble_kernel(const int32_t* __restrict__ n_per_frame, int cap, int P,
                                                                   const int32_t* __restrict__ word_of,
                                                                   const int32_t* __restrict__ node_of,
                                                                   const float* __restrict__ w_of, int weighting, int norm,
                                                                   BowOutDev out) {
  extern __shared__ __align__(16) unsigned long long s_keys[];  // P keys
  __shared__ int s_warp[64];
  __shared__ int s_nv;
  __shared__ double s_norm;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = min(n_per_frame[b], cap);
  const long long base = (long long)b * cap;
  const bool tf = weighting == 0 || weighting == 1;
  uint32_t* word_ids = out.word_ids + base;
  double* values = out.word_values + base;
  uint32_t* node_ids = out.node_ids + base;
  int32_t* offsets = out.offsets + (long long)b * (cap + 1);
  uint32_t* feats = out.feats + base;

  // ---- BowVector: (word << 32 | feature) ascending; features of stopped words (w <= 0) are dropped (:1181)
  if (tid == 0) s_nv = 0;
  __syncthreads();
  int mine = 0;
  for (int i = tid; i < P; i += kAsmThreads) {
    const bool ok = i < n && w_of[base + i] > 0.0f;
    s_keys[i] = ok ? (((unsigned long long)(uint32_t)word_of[base + i] << 32) | (uint32_t)i) : ~0ull;
    mine += ok;
  }
  if (mine) atomicAdd(&s_nv, mine);
  __syncthreads();
  const int nv = s_nv;
  bitonic_sort(s_keys, P);
  auto word_head = [&](int p) { return p < nv && (p == 0 || (s_keys[p] >> 32) != (s_keys[p - 1] >> 32)); };
  const int nw = scan_heads(P, s_warp, word_head, [&](int p, int rank) {
    int e = p + 1;
    while (e < nv && (s_keys[e] >> 32) == (s_keys[p] >> 32)) e++;
    const double w = (double)w_of[base + (uint32_t)s_keys[p]];  // WordValue = the file's float widened (:1507)
    double sum = w;
    if (tf)
      for (int c = 1; c < e - p; c++) sum = __dadd_rn(sum, w);  // addWeight: vit->second += v
    word_ids[rank] = (uint32_t)(s_keys[p] >> 32);
    values[rank] = sum;
  });
  __syncthreads();
  if (tid == 0) {
    out.n_words[b] = nw;
    double nr = 0.0;
    if (norm == 1) {
      for (int i = 0; i < nw; i++) nr = __dadd_rn(nr, fabs(values[i]));  // ascending word id = std::map order
    } else if (norm == 2) {
      for (int i = 0; i < nw; i++) nr = __dadd_rn(nr, __dmul_rn(values[i], values[i]));
      nr = sqrt(nr);
    }
    s_norm = nr;
  }
  __syncthreads();
  if (norm == 0) {
    if (tf && nw > 0)  // "unnecessary when normalizing" (:1189-1195)
      for (int i = tid; i < nw; i += kAsmThreads) values[i] = __ddiv_rn(values[i], (double)nw);
  } else if (s_norm > 0.0) {
    const double nr = s_norm;
    for (int i = tid; i < nw; i += kAsmThreads) values[i] = __ddiv_rn(values[i], nr);
  }
  __syncthreads();

  // ---- FeatureVector: (node << 32 | feature) ascending -> CSR
  for (int i = tid; i < P; i += kAsmThreads) {
    const bool ok = i < n && w_of[base + i] > 0.0f;
    s_keys[i] = ok ? (((unsigned long long)(uint32_t)node_of[base + i] << 32) | (uint32_t)i) : ~0ull;
  }
  __syncthreads();
  bitonic_sort(s_keys, P);
  for (int p = tid; p < nv; p += kAsmThreads) feats[p] = (uint32_t)s_keys[p];
  auto node_head = [&](int p) { return p < nv && (p == 0 || (s_keys[p] >> 32) != (s_keys[p - 1] >> 32)); };
  const int nn = scan_heads(P, s_warp, node_head, [&](int p, int rank) {
    node_ids[rank] = (uint32_t)(s_keys[p] >> 32);
    offsets[rank] = p;
  });
  if (tid == 0) {
    offsets[nn] = nv;
    out.n_nodes[b] = nn;
  }
}

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

thread_local std::string g_vocab_create_error;

}  // namespace

struct swm_vocab {
  int device = 0;
  std::string err;
  int k = 0, L = 0, scoring = 0, weighting = 0, n_nodes = 0, n_words = 0;
  Buf desc, child_off, child, word, weight;
  Buf in_desc, in_n, word_of, node_of, w_of;
  Buf o_word_ids, o_values, o_n_words, o_node_ids, o_offsets, o_feats, o_n_nodes;
  PinnedArena score_arena;  // swm_bow_score: operands in, scores out
  Buf score_out;
  cudaStream_t stream = nullptr;
  void free_all() {
    for (Buf* b : {&desc, &child_off, &child, &word, &weight, &in_desc, &in_n, &word_of, &node_of, &w_of, &o_word_ids,
                   &o_values, &o_n_words, &o_node_ids, &o_offsets, &o_feats, &o_n_nodes, &score_out})
      b->release();
    score_arena.release();
  }
};

#define VCK(v, call)                                   \
  do {                                                 \
    cudaError_t e_ = (call);                           \
    if (e_ != cudaSuccess) {                           \
      (v)->err = cuda_err(#call, e_);                  \
      return SWM_E_CUDA;                               \
    }                                                  \
  } while (0)

namespace {

// d_desc: device [batch][cap][32]; d_n: device [batch].  Runs both kernels and copies the slabs to the host.
int bow_run(swm_vocab* v, const uint4* d_desc, const int32_t* d_n, int batch, int cap, int levelsup, const swm_bow_out* out) {
  int P = 1024;
  while (P < cap) P <<= 1;
  const size_t tot = (size_t)batch * cap;
  VCK(v, v->word_of.ensure(tot * 4));
  VCK(v, v->node_of.ensure(tot * 4));
  VCK(v, v->w_of.ensure(tot * 4));
  VCK(v, v->o_word_ids.ensure(tot * 4));
  VCK(v, v->o_values.ensure(tot * 8));
  VCK(v, v->o_node_ids.ensure(tot * 4));
  VCK(v, v->o_feats.ensure(tot * 4));
  VCK(v, v->o_offsets.ensure((size_t)batch * (cap + 1) * 4));
  VCK(v, v->o_n_words.ensure((size_t)batch * 4));
  VCK(v, v->o_n_nodes.ensure((size_t)batch * 4));
  VocabDev vd{v->desc.as<uint4>(), v->child_off.as<int32_t>(), v->child.as<int32_t>(), v->word.as<int32_t>(),
              v->weight.as<float>(), v->L};
  const long long groups = (long long)tot;
  const unsigned blocks = (unsigned)((groups * 16 + 255) / 256);
  bow_descend_kernel<<<blocks, 256, 0, v->stream>>>(d_desc, d_n, cap, batch, vd, levelsup, v->word_of.as<int32_t>(),
                                                    v->node_of.as<int32_t>(), v->w_of.as<float>());
  VCK(v, cudaGetLastError());
  BowOutDev od{v->o_word_ids.as<uint32_t>(), v->o_values.as<double>(), v->o_n_words.as<int32_t>(),
               v->o_node_ids.as<uint32_t>(), v->o_offsets.as<int32_t>(), v->o_feats.as<uint32_t>(),
               v->o_n_nodes.as<int32_t>()};
  // scoring object -> (mustNormalize, norm): ScoringObject.h:76-91
  const int norm = v->scoring == 5 ? 0 : (v->scoring == 1 ? 2 : 1);
  const size_t smem = (size_t)P * 8;
  VCK(v, cudaFuncSetAttribute(bow_assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bow_assemble_kernel<<<batch, kAsmThreads, smem, v->stream>>>(d_n, cap, P, v->word_of.as<int32_t>(),
                                                               v->node_of.as<int32_t>(), v->w_of.as<float>(),
                                                               v->weighting, norm, od);
  VCK(v, cudaGetLastError());
  VCK(v, cudaMemcpyAsync(out->word_ids, od.word_ids, tot * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->word_values, od.word_values, tot * 8, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->n_words, od.n_words, (size_t)batch * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->node_ids, od.node_ids, tot * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->node_offsets, od.offsets, (size_t)batch * (cap + 1) * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->feats, od.feats, tot * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaMemcpyAsync(out->n_nodes, od.n_nodes, (size_t)batch * 4, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaStreamSynchronize(v->stream));
  return SWM_OK;
}

bool out_ok(const swm_bow_out* o) {
  return o && o->word_ids && o->word_values && o->n_words && o->node_ids && o->node_offsets && o->feats && o->n_nodes;
}

}  // namespace

extern "C" {

int swm_vocab_create(int device, const uint8_t* blob, size_t bytes, swm_vocab** out) {
  if (!out) return SWM_E_INVALID;
  *out = nullptr;
  if (!blob || bytes < 24) { g_vocab_create_error = "vocabulary blob too short"; return SWM_E_INVALID; }
  uint32_t nb_nodes, size_node;
  int32_t hdr[4];
  memcpy(&nb_nodes, blob, 4);
  memcpy(&size_node, blob + 4, 4);
  memcpy(hdr, blob + 8, 16);
  if (size_node != 41) { g_vocab_create_error = "node record size is not 4 + 32 + 4 + 1 (not an ORB vocabulary)"; return SWM_E_INVALID; }
  if (hdr[2] < 0 || hdr[2] > 5 || hdr[3] < 0 || hdr[3] > 3) { g_vocab_create_error = "unknown scoring / weighting type"; return SWM_E_INVALID; }
  const size_t n_rec = (bytes - 24) / size_node;
  const size_t n_nodes = n_rec + 1;
  if (n_rec == 0 || n_nodes > (1u << 30)) { g_vocab_create_error = "bad node count"; return SWM_E_INVALID; }
  // children lists in file order (:1504), word ids = leaves in file order (:1509-1512)
  std::vector<int32_t> parent(n_nodes, 0), cnt(n_nodes + 1, 0), word(n_nodes, 0);
  std::vector<float> weight(n_nodes, 0.f);
  std::vector<uint8_t> desc(n_nodes * 32, 0);
  int n_words = 0;
  for (size_t r = 0; r < n_rec; r++) {
    const uint8_t* buf = blob + 24 + r * size_node;
    const size_t nid = r + 1;
    int32_t p;
    memcpy(&p, buf, 4);
    if (p < 0 || (size_t)p >= n_nodes || (size_t)p == nid) { g_vocab_create_error = "node with an invalid parent"; return SWM_E_INVALID; }
    parent[nid] = p;
    cnt[p]++;
    memcpy(&desc[nid * 32], buf + 4, 32);
    memcpy(&weight[nid], buf + 36, 4);
    if (buf[40]) word[nid] = n_words++;
  }
  std::vector<int32_t> off(n_nodes + 1, 0), child(n_rec), cur(n_nodes);
  for (size_t i = 0; i < n_nodes; i++) off[i + 1] = off[i] + cnt[i];
  for (size_t i = 0; i < n_nodes; i++) cur[i] = off[i];
  for (size_t nid = 1; nid < n_nodes; nid++) child[cur[parent[nid]]++] = (int32_t)nid;
  std::string err;
  int rc = check_device(device, &err);
  if (rc != SWM_OK) { g_vocab_create_error = err; return rc; }
  swm_vocab* v = new swm_vocab();
  v->device = device;
  v->k = hdr[0]; v->L = hdr[1]; v->scoring = hdr[2]; v->weighting = hdr[3];
  v->n_nodes = (int)n_nodes;
  v->n_words = n_words;
  bool ok = cudaSetDevice(device) == cudaSuccess &&
            cudaStreamCreateWithFlags(&v->stream, cudaStreamNonBlocking) == cudaSuccess &&
            v->desc.ensure(n_nodes * 32) == cudaSuccess && v->child_off.ensure((n_nodes + 1) * 4) == cudaSuccess &&
            v->child.ensure(n_rec * 4) == cudaSuccess && v->word.ensure(n_nodes * 4) == cudaSuccess &&
            v->weight.ensure(n_nodes * 4) == cudaSuccess &&
            cudaMemcpy(v->desc.p, desc.data(), n_nodes * 32, cudaMemcpyHostToDevice) == cudaSuccess &&
            cudaMemcpy(v->child_off.p, off.data(), (n_nodes + 1) * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
            cudaMemcpy(v->child.p, child.data(), n_rec * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
            cudaMemcpy(v->word.p, word.data(), n_nodes * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
            cudaMemcpy(v->weight.p, weight.data(), n_nodes * 4, cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) {
    g_vocab_create_error = cuda_err("vocabulary upload", cudaGetLastError());
    v->free_all();
    if (v->stream) cudaStreamDestroy(v->stream);
    delete v;
    return SWM_E_CUDA;
  }
  *out = v;
  return SWM_OK;
}

void swm_vocab_destroy(swm_vocab* v) {
  if (!v) return;
  cudaSetDevice(v->device);
  if (v->stream) cudaStreamSynchronize(v->stream);
  v->free_all();
  if (v->stream) cudaStreamDestroy(v->stream);
  delete v;
}

const char* swm_vocab_last_error(const swm_vocab* v) { return v ? v->err.c_str() : g_vocab_create_error.c_str(); }

int swm_vocab_info(const swm_vocab* v, int32_t* k, int32_t* L, int32_t* n_nodes, int32_t* n_words) {
  if (!v) return SWM_E_INVALID;
  if (k) *k = v->k;
  if (L) *L = v->L;
  if (n_nodes) *n_nodes = v->n_nodes;
  if (n_words) *n_words = v->n_words;
  return SWM_OK;
}

int swm_bow_transform(swm_vocab* v, const uint8_t* desc, const int32_t* n, int batch, int cap, int levelsup,
                      const swm_bow_out* out) {
  if (!v) return SWM_E_INVALID;
  if (!desc || !n || batch < 1 || cap < 1 || !out_ok(out)) { v->err = "bad argument"; return SWM_E_INVALID; }
  if (cap > SWM_BOW_MAX_FEATURES) { v->err = "cap exceeds SWM_BOW_MAX_FEATURES"; return SWM_E_CAPACITY; }
  for (int b = 0; b < batch; b++)
    if (n[b] < 0 || n[b] > cap) { v->err = "n[b] outside [0, cap]"; return SWM_E_INVALID; }
  VCK(v, cudaSetDevice(v->device));
  const size_t tot = (size_t)batch * cap;
  VCK(v, v->in_desc.ensure(tot * 32));
  VCK(v, v->in_n.ensure((size_t)batch * 4));
  VCK(v, cudaMemcpyAsync(v->in_desc.p, desc, tot * 32, cudaMemcpyHostToDevice, v->stream));
  VCK(v, cudaMemcpyAsync(v->in_n.p, n, (size_t)batch * 4, cudaMemcpyHostToDevice, v->stream));
  return bow_run(v, v->in_desc.as<uint4>(), v->in_n.as<int32_t>(), batch, cap, levelsup, out);
}

int swm_bow_transform_frame(swm_vocab* v, const swm_frame* f, int levelsup, const swm_bow_out* out) {
  if (!v) return SWM_E_INVALID;
  if (!f || !out_ok(out)) { v->err = "bad argument"; return SWM_E_INVALID; }
  FrameDeviceView fv;
  if (frame_device_view(f, &fv) != SWM_OK || fv.device != v->device) { v->err = "frame is not resident on the vocabulary's device"; return SWM_E_INVALID; }
  out->n_words[0] = 0;
  out->n_nodes[0] = 0;
  out->node_offsets[0] = 0;
  if (fv.n == 0) return SWM_OK;
  if (fv.n > SWM_BOW_MAX_FEATURES) { v->err = "frame exceeds SWM_BOW_MAX_FEATURES"; return SWM_E_CAPACITY; }
  VCK(v, cudaSetDevice(v->device));
  VCK(v, cudaStreamWaitEvent(v->stream, fv.ready, 0));
  VCK(v, v->in_n.ensure(4));
  VCK(v, cudaMemcpyAsync(v->in_n.p, &fv.n, 4, cudaMemcpyHostToDevice, v->stream));
  return bow_run(v, fv.desc, v->in_n.as<int32_t>(), 1, fv.n, levelsup, out);
}

int swm_bow_score(swm_vocab* v, int npairs, const int32_t* a_offsets, const uint32_t* a_words, const double* a_values,
                  const int32_t* b_offsets, const uint32_t* b_words, const double* b_values, double* out) {
  if (!v) return SWM_E_INVALID;
  if (v->scoring != 0) { v->err = "swm_bow_score: the vocabulary's scoring type is not L1_NORM"; return SWM_E_INVALID; }
  if (npairs < 0 || (npairs > 0 && (!a_offsets || !b_offsets || !out))) { v->err = "bad argument"; return SWM_E_INVALID; }
  if (npairs == 0) return SWM_OK;
  for (const int32_t* off : {a_offsets, b_offsets}) {
    const uint32_t* w = off == a_offsets ? a_words : b_words;
    if (off[0] != 0) { v->err = "offsets[0] must be 0"; return SWM_E_INVALID; }
    for (int i = 0; i < npairs; i++) {
      if (off[i + 1] < off[i]) { v->err = "offsets not non-decreasing"; return SWM_E_INVALID; }
      for (int j = off[i] + 1; j < off[i + 1]; j++)
        if (w[j] <= w[j - 1]) { v->err = "word ids not strictly ascending"; return SWM_E_INVALID; }
    }
    if (off[npairs] > 0 && (!w || !(off == a_offsets ? a_values : b_values))) { v->err = "bad argument"; return SWM_E_INVALID; }
  }
  VCK(v, cudaSetDevice(v->device));
  const size_t na = (size_t)a_offsets[npairs], nb = (size_t)b_offsets[npairs];
  const size_t bytes = (na + nb) * 12 + (size_t)(npairs + 1) * 8 + (size_t)npairs * 8 + 2048;
  VCK(v, v->score_arena.begin(bytes, v->stream));
  const int32_t* da = v->score_arena.put(a_offsets, npairs + 1);
  const uint32_t* daw = v->score_arena.put(a_words, na);
  const double* dav = v->score_arena.put(a_values, na);
  const int32_t* db = v->score_arena.put(b_offsets, npairs + 1);
  const uint32_t* dbw = v->score_arena.put(b_words, nb);
  const double* dbv = v->score_arena.put(b_values, nb);
  VCK(v, v->score_arena.flush(v->stream));
  VCK(v, v->score_out.ensure((size_t)npairs * 8));
  VCK(v, launch_l1_score_pairs(npairs, da, daw, dav, db, dbw, dbv, v->score_out.as<double>(), v->stream));
  double* h = v->score_arena.put(out, 0);  // device address of the read-back slot; its host twin follows
  uint8_t* h_host = v->score_arena.h + (reinterpret_cast<uint8_t*>(h) - v->score_arena.d);
  VCK(v, cudaMemcpyAsync(h_host, v->score_out.p, (size_t)npairs * 8, cudaMemcpyDeviceToHost, v->stream));
  VCK(v, cudaStreamSynchronize(v->stream));
  memcpy(out, h_host, (size_t)npairs * 8);
  return SWM_OK;
}

}  // extern "C"

namespace swm {
int vocab_props(const swm_vocab* v, VocabProps* out) {
  if (!v || !out) return SWM_E_INVALID;
  out->device = v->device;
  out->scoring = v->scoring;
  out->n_words = v->n_words;
  return SWM_OK;
}
}  // namespace swm
