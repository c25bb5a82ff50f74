// swm_internal.cuh -- shared declarations of the libswm_orb translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>
#include <string>

#include "../../include/swm_orb.h"
#include "swm_core.cuh"

namespace swm {

// Geometry of one pyramid level inside a frame slab.  Every plane (un-blurred, blurred, score)
// uses the same layout: rows = h + 2*kEdge, row pitch a multiple of 128 bytes, ROI pixel (0,0)
// at byte kEdge*pitch + kPadX from the plane start.
struct LevelGeom {
  int w, h;            // level size (cvRound(cols * invScale), ORBextractor.cc:825-826)
  int pitch;           // bytes per plane row
  int rows;            // h + 38
  long long plane_off; // byte offset of the plane inside a frame slab
  int xtab_off, ytab_off;  // offsets into the resize tap tables (levels >= 1)
  int tiles_x, tiles_y;    // 32x32 FAST tiles (Fast_gpu.cu:374-375)
  int tile_off;            // offset of this level's tiles in the per-frame retry-flag array
  int fblk_x, fblk_off;    // FAST kernel blocks (two tiles wide) per row / offset of this level in the grid
  int cand_off, cand_cap;  // per-frame candidate array slice (FAST survivors, pre-quadtree)
  int sel_off, sel_cap;    // per-frame selection slice (post-quadtree)
  int quota;               // mnFeaturesPerLevel[level]
  int kp_size;             // int(31 * scale)
  float scale;             // mvScaleFactor[level]
};

struct FrameLayout {
  int nlevels;
  int w, h;
  long long slab_bytes;  // bytes per frame of one plane set
  int tiles_total;       // FAST tiles per frame (all levels)
  int fblk_total;        // FAST kernel blocks per frame (all levels)
  int cand_total;        // candidate slots per frame
  int sel_total;         // selection slots per frame
  LevelGeom lv[SWM_MAX_LEVELS];
};

inline std::string cuda_err(const char* what, cudaError_t e) {
  return std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
}

// Verifies a usable sm_100 device; fills err on failure.  No CPU fallback exists.
int check_device(int device, std::string* err);

// Device-resident outputs of the extractor's most recent batch (extract.cu), for consumers inside the library
// that continue on the GPU (swm_frame_from_extractor in match.cu).
struct OrbDeviceView {
  const swm_keypoint* kps;  // [batch][cap]
  const uint8_t* desc;      // [batch][cap][32]
  const int32_t* n;         // [batch]
  int cap, batch, device;
  cudaStream_t stream;      // the stream the batch was enqueued on
};
int orb_device_view(swm_orb* h, OrbDeviceView* out);

// Descriptors of a resident frame (match.cu) for the vocabulary transform (bow.cu).
struct FrameDeviceView {
  const uint4* desc;  // n x 2
  int n, device;
  cudaEvent_t ready;  // recorded after the frame's last write
};
int frame_device_view(const swm_frame* f, FrameDeviceView* out);

// Vocabulary properties for the keyframe database (kfdb.cu); scoring is DBoW2's ScoringType (0 = L1_NORM).
struct VocabProps {
  int device, scoring, n_words;
};
int vocab_props(const swm_vocab* v, VocabProps* out);

// Host operands of a call packed into one pinned buffer and sent with one copy; results come back through the
// same buffer.  Grow-only; growing synchronises `stream` first because earlier copies may still read the buffer.
struct PinnedArena {
  uint8_t* h = nullptr;
  uint8_t* d = nullptr;
  size_t cap = 0, used = 0;
  cudaError_t begin(size_t bytes, cudaStream_t stream) {
    bytes += 4096;
    used = 0;
    if (bytes <= cap) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return e;
    release();
    const size_t want = bytes + bytes / 2;
    if ((e = cudaMallocHost(&h, want)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&d, want)) != cudaSuccess) return e;
    cap = want;
    return cudaSuccess;
  }
  // copies `bytes` of src into the arena; returns the device address its copy will have after flush()
  template <class T>
  T* put(const T* src, size_t count) {
    const size_t off = (used + 255) & ~(size_t)255, bytes = count * sizeof(T);
    if (bytes) memcpy(h + off, src, bytes);
    used = off + bytes;
    return reinterpret_cast<T*>(d + off);
  }
  cudaError_t flush(cudaStream_t stream) {
    return used ? cudaMemcpyAsync(d, h, used, cudaMemcpyHostToDevice, stream) : cudaSuccess;
  }
  void release() {
    if (h) cudaFreeHost(h);
    if (d) cudaFree(d);
    h = d = nullptr;
    cap = used = 0;
  }
};

// DBoW2 L1Scoring::score of npairs pairs (a[i], b[i]) of BowVectors in CSR form, one warp per pair (kfdb.cu).
cudaError_t launch_l1_score_pairs(int npairs, const int32_t* a_off, const uint32_t* a_words, const double* a_values,
                                  const int32_t* b_off, const uint32_t* b_words, const double* b_values, double* out,
                                  cudaStream_t stream);

}  // namespace swm
