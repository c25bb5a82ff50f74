// ORBVocabulary.h -- drop-in for the part of DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB> that SwarmMap's hot
// path uses (reference code/include/ORBVocabulary.h:30-31 typedefs it as ORB_SLAM2::ORBVocabulary):
//   loadFromBinaryFile(filename)                      TemplatedVocabulary.h:1478-1522 (swarm_map.cc loads ORBvoc.bin)
//   transform(features, BowVector&, FeatureVector&, levelsup)   :1151-1218, called by Frame::ComputeBoW
//                                                     (Frame.cc:445-452), KeyFrame::ComputeBoW (KeyFrame.cc:126-133)
// The tree walk and the assembly of both containers run on the GPU (swm_bow_transform); BowVector / FeatureVector
// below have DBoW2's container types (std::map<WordId, WordValue>, std::map<NodeId, std::vector<unsigned>>), so the
// callers' code (SearchByBoW's merge walk) compiles unchanged.
//   score(a, b)                                       L1Scoring::score (ScoringObject.cpp), on the GPU (swm_bow_score);
//                                                     LoopClosing::DetectLoop's minScore; L1_NORM vocabularies only
// KeyFrameDatabase (KeyFrameDatabase.h) runs on the GPU too.  The rest of the vocabulary API stays with DBoW2
// (DESIGN.md section 8).
#pragma once
#include <cstdio>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef SWM_HAVE_OPENCV
#include <opencv2/core/core.hpp>
#else
#include "cv_shim.h"
#endif
#include "../../include/swm_orb.h"

namespace DBoW2 {
typedef unsigned int WordId;
typedef double WordValue;
typedef unsigned int NodeId;
#ifndef SWM_HAVE_DBOW2  // with the real DBoW2 headers on the include path these come from BowVector.h / FeatureVector.h
class BowVector : public std::map<WordId, WordValue> {};
class FeatureVector : public std::map<NodeId, std::vector<unsigned int>> {};
#endif
}  // namespace DBoW2

namespace ORB_SLAM2 {

class ORBVocabulary {
 public:
  explicit ORBVocabulary(int device = 0) : device_(device) {}
  ~ORBVocabulary() { swm_vocab_destroy(v_); }
  ORBVocabulary(const ORBVocabulary&) = delete;
  ORBVocabulary& operator=(const ORBVocabulary&) = delete;

  bool loadFromBinaryFile(const std::string& filename) {
    FILE* f = std::fopen(filename.c_str(), "rb");
    if (!f) return false;
    std::vector<uint8_t> blob;
    uint8_t buf[1 << 16];
    size_t got;
    while ((got = std::fread(buf, 1, sizeof(buf), f)) > 0) blob.insert(blob.end(), buf, buf + got);
    std::fclose(f);
    return loadFromMemory(blob.data(), blob.size());
  }
  bool loadFromMemory(const uint8_t* blob, size_t bytes) {
    swm_vocab_destroy(v_);
    v_ = nullptr;
    return swm_vocab_create(device_, blob, bytes, &v_) == SWM_OK;
  }
  bool empty() const { return v_ == nullptr; }
  unsigned int size() const {
    int32_t nw = 0;
    if (v_) swm_vocab_info(v_, nullptr, nullptr, nullptr, &nw);
    return (unsigned)nw;
  }

  // features: one 1 x 32 CV_8U row per keypoint (Converter::toDescriptorVector(mDescriptors))
  void transform(const std::vector<cv::Mat>& features, DBoW2::BowVector& v, DBoW2::FeatureVector& fv, int levelsup) const {
    v.clear();
    fv.clear();
    if (empty() || features.empty()) return;  // :1157-1160
    const int n = (int)features.size();
    std::vector<uint8_t> desc((size_t)n * 32);
    for (int i = 0; i < n; i++) std::memcpy(&desc[(size_t)i * 32], features[i].ptr(0), 32);
    transform(desc.data(), n, v, fv, levelsup);
  }
  // the same from the N x 32 descriptor matrix itself (saves the per-row cv::Mat vector)
  void transform(const uint8_t* desc, int n, DBoW2::BowVector& v, DBoW2::FeatureVector& fv, int levelsup) const {
    v.clear();
    fv.clear();
    if (empty() || n <= 0) return;
    std::vector<uint32_t> word_ids(n), node_ids(n), feats(n);
    std::vector<double> values(n);
    std::vector<int32_t> offsets(n + 1);
    int32_t nw = 0, nn = 0;
    swm_bow_out out = {word_ids.data(), values.data(), &nw, node_ids.data(), offsets.data(), feats.data(), &nn};
    const int32_t cnt = n;
    if (swm_bow_transform(v_, desc, &cnt, 1, n, levelsup, &out) != SWM_OK)
      throw std::runtime_error(std::string("ORBVocabulary::transform: ") + swm_vocab_last_error(v_));
    for (int i = 0; i < nw; i++) v.insert(v.end(), std::make_pair(word_ids[i], values[i]));  // ascending: O(1) hinted
    for (int j = 0; j < nn; j++)
      fv.insert(fv.end(), std::make_pair(node_ids[j], std::vector<unsigned int>(feats.begin() + offsets[j],
                                                                                feats.begin() + offsets[j + 1])));
  }
  double score(const DBoW2::BowVector& a, const DBoW2::BowVector& b) const {
    std::vector<uint32_t> w;
    std::vector<double> x;
    for (const auto& e : a) { w.push_back(e.first); x.push_back(e.second); }
    for (const auto& e : b) { w.push_back(e.first); x.push_back(e.second); }
    const int32_t ao[2] = {0, (int32_t)a.size()}, bo[2] = {0, (int32_t)b.size()};
    double out = 0.0;
    if (swm_bow_score(v_, 1, ao, w.data(), x.data(), bo, w.data() + a.size(), x.data() + a.size(), &out) != SWM_OK)
      throw std::runtime_error(std::string("ORBVocabulary::score: ") + swm_vocab_last_error(v_));
    return out;
  }
  swm_vocab* handle() const { return v_; }

 private:
  int device_;
  swm_vocab* v_ = nullptr;
};

}  // namespace ORB_SLAM2
