// KeyFrameDatabase.h -- drop-in for ORB_SLAM2::KeyFrameDatabase (KeyFrameDatabase.cc as SwarmMap carries it):
//   add(pKF), erase(pKF), clear()                         the inverted file, kept on the GPU
//   DetectRelocalizationCandidates(F)                     Tracking::Relocalization
//   DetectLoopCandidates(pKF, minScore)                   LoopClosing::DetectLoop, AgentMediator::CheckOverlapCandidates
// on top of swm_kfdb_* (csrc/kfdb.cu), with DBoW2's L1 score.  The members are templates on the keyframe / frame
// types, like ORBmatcher.h: they read mnId, mBowVec, GetConnectedKeyFrames() and GetBestCovisibilityKeyFrames(10), and
// map the ids the device returns back to the pointers given to add().  The candidate lists convert to
// std::vector<KeyFrame*>, so `vector<KeyFrame*> v = mpKeyFrameDB->DetectRelocalizationCandidates(&mCurrentFrame);`
// compiles unchanged.  Results equal the reference's under the definitions of DESIGN.md section 2.
#pragma once
#include <mutex>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "ORBVocabulary.h"

namespace ORB_SLAM2 {

class KeyFrameDatabase {
 public:
  // Converts to std::vector<KF*> for the keyframe type the caller names.
  struct Candidates {
    std::vector<void*> p;
    template <class KF>
    operator std::vector<KF*>() const {
      std::vector<KF*> v;
      v.reserve(p.size());
      for (void* x : p) v.push_back(static_cast<KF*>(x));
      return v;
    }
    bool empty() const { return p.empty(); }
    size_t size() const { return p.size(); }
  };

  explicit KeyFrameDatabase(const ORBVocabulary& voc) {
    if (swm_kfdb_create(voc.handle(), &db_) != SWM_OK)
      throw std::runtime_error(std::string("KeyFrameDatabase: ") + swm_kfdb_last_error(nullptr));
  }
  ~KeyFrameDatabase() { swm_kfdb_destroy(db_); }
  KeyFrameDatabase(const KeyFrameDatabase&) = delete;
  KeyFrameDatabase& operator=(const KeyFrameDatabase&) = delete;

  template <class KF>
  void add(KF* pKF) {
    std::unique_lock<std::mutex> lock(mMutex);
    std::vector<uint32_t> w;
    std::vector<double> x;
    for (const auto& e : pKF->mBowVec) { w.push_back(e.first); x.push_back(e.second); }
    const uint64_t id = (uint64_t)pKF->mnId;
    const int32_t off[2] = {0, (int32_t)w.size()};
    check(swm_kfdb_add(db_, 1, &id, off, w.data(), x.data()), "add");
    ptr_[id] = pKF;
    neigh_fn_ = &finish_as<KF>;
  }

  template <class KF>
  void erase(KF* pKF) {
    std::unique_lock<std::mutex> lock(mMutex);
    const uint64_t id = (uint64_t)pKF->mnId;
    check(swm_kfdb_erase(db_, 1, &id), "erase");
    ptr_.erase(id);
  }

  void clear() {
    std::unique_lock<std::mutex> lock(mMutex);
    check(swm_kfdb_clear(db_), "clear");
    ptr_.clear();
  }

  template <class KF>
  Candidates DetectLoopCandidates(KF* pKF, float minScore) {
    std::unique_lock<std::mutex> lock(mMutex);
    std::vector<uint64_t> conn;
    for (KF* k : pKF->GetConnectedKeyFrames()) conn.push_back((uint64_t)k->mnId);
    const int32_t coff[2] = {0, (int32_t)conn.size()};
    query(SWM_KFDB_LOOP, pKF->mBowVec, &minScore, coff, conn.data());
    return finish<KF>();
  }

  template <class F>
  Candidates DetectRelocalizationCandidates(F* pF) {
    std::unique_lock<std::mutex> lock(mMutex);
    query(SWM_KFDB_RELOC, pF->mBowVec, nullptr, nullptr, nullptr);
    return finish_any();
  }

  swm_kfdb* handle() const { return db_; }

 private:
  void check(int rc, const char* what) const {
    if (rc != SWM_OK) throw std::runtime_error(std::string("KeyFrameDatabase::") + what + ": " + swm_kfdb_last_error(db_));
  }

  void query(int mode, const DBoW2::BowVector& bow, const float* min_score, const int32_t* coff, const uint64_t* conn) {
    std::vector<uint32_t> w;
    std::vector<double> x;
    for (const auto& e : bow) { w.push_back(e.first); x.push_back(e.second); }
    const int32_t qoff[2] = {0, (int32_t)w.size()};
    int32_t soff[2] = {0, 0};
    for (;;) {
      scored_.resize(std::max<size_t>(scored_.size(), 1));
      scores_.resize(scored_.size());
      const int rc = swm_kfdb_query(db_, mode, 1, qoff, w.data(), x.data(), min_score, coff, conn, soff,
                                    scored_.data(), scores_.data(), (int32_t)scored_.size());
      if (rc == SWM_E_CAPACITY && soff[1] > (int32_t)scored_.size()) {  // nothing changed: repeat with the size needed
        scored_.resize(soff[1]);
        continue;
      }
      check(rc, "query");
      break;
    }
    n_scored_ = soff[1];
  }

  // The reference calls GetBestCovisibilityKeyFrames(10) on the scored keyframes only: so does this.
  template <class KF>
  Candidates finish() {
    std::vector<int32_t> noff(1, 0);
    std::vector<uint64_t> nids;
    for (int i = 0; i < n_scored_; i++) {
      KF* k = static_cast<KF*>(ptr_.at(scored_[i]));
      for (KF* n : k->GetBestCovisibilityKeyFrames(10)) nids.push_back((uint64_t)n->mnId);
      noff.push_back((int32_t)nids.size());
    }
    std::vector<uint64_t> cand(std::max(n_scored_, 1));
    int32_t coff[2] = {0, 0};
    check(swm_kfdb_finish(db_, noff.data(), nids.data(), coff, cand.data(), (int32_t)cand.size()), "finish");
    Candidates out;
    for (int i = 0; i < coff[1]; i++) out.p.push_back(ptr_.at(cand[i]));
    return out;
  }
  // Relocalisation knows only the frame type: the scored keyframes have the type add() was last given (SwarmMap adds
  // one keyframe type); before any add nothing can be scored.
  Candidates finish_any() { return neigh_fn_ ? neigh_fn_(this) : finish_none(); }
  Candidates finish_none() {
    std::vector<int32_t> noff(n_scored_ + 1, 0);
    std::vector<uint64_t> cand(std::max(n_scored_, 1));
    int32_t coff[2] = {0, 0};
    check(swm_kfdb_finish(db_, noff.data(), nullptr, coff, cand.data(), (int32_t)cand.size()), "finish");
    Candidates out;
    for (int i = 0; i < coff[1]; i++) out.p.push_back(ptr_.at(cand[i]));
    return out;
  }

  template <class KF>
  static Candidates finish_as(KeyFrameDatabase* self) { return self->finish<KF>(); }

  swm_kfdb* db_ = nullptr;
  std::mutex mMutex;
  std::unordered_map<uint64_t, void*> ptr_;
  std::vector<uint64_t> scored_;
  std::vector<float> scores_;
  int n_scored_ = 0;
  Candidates (*neigh_fn_)(KeyFrameDatabase*) = nullptr;
};

}  // namespace ORB_SLAM2
