// The C++ drop-ins ORB_SLAM2::KeyFrameDatabase and ORBVocabulary::score on small KeyFrame / Frame doubles, against
// the CPU oracle (oracle/liborb_oracle_kfdb.so).  Tracking::Relocalization's and LoopClosing::DetectLoop's calls are
// written as the reference writes them.  Prints KFDB_WRAPPER_OK.
#include <cstdio>
#include <random>
#include <set>
#include <vector>

#include "../oracle/orb_oracle_kfdb.h"
#include "../swarmmap_b200/host/KeyFrameDatabase.h"

using namespace ORB_SLAM2;

struct KeyFrame {
  long unsigned int mnId;
  DBoW2::BowVector mBowVec;
  std::vector<KeyFrame*> best;
  std::set<KeyFrame*> connected;
  std::vector<KeyFrame*> GetBestCovisibilityKeyFrames(const int& N) {
    return std::vector<KeyFrame*>(best.begin(), best.begin() + std::min<size_t>(N, best.size()));
  }
  std::set<KeyFrame*> GetConnectedKeyFrames() { return connected; }
};
struct Frame {
  long unsigned int mnId;
  DBoW2::BowVector mBowVec;
};

static int fails = 0;
#define EXPECT(c)                                              \
  do {                                                         \
    if (!(c)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); fails++; } \
  } while (0)

static void split(const DBoW2::BowVector& b, std::vector<uint32_t>& w, std::vector<double>& v) {
  w.clear();
  v.clear();
  for (const auto& e : b) { w.push_back(e.first); v.push_back(e.second); }
}

int main() {
  // a k=10, L=2 vocabulary blob (L1_NORM, TF_IDF): 110 nodes, 100 words
  std::vector<uint8_t> blob(24 + 110 * 41, 0);
  const int32_t hdr[4] = {10, 2, 0, 0};
  const uint32_t nb_nodes = 111, size_node = 41;
  memcpy(blob.data(), &nb_nodes, 4);
  memcpy(blob.data() + 4, &size_node, 4);
  memcpy(blob.data() + 8, hdr, 16);
  for (int r = 0; r < 110; r++) {
    uint8_t* rec = blob.data() + 24 + r * 41;
    const int32_t parent = r < 10 ? 0 : 1 + (r - 10) / 10;
    const float weight = 1.0f;
    memcpy(rec, &parent, 4);
    rec[4] = (uint8_t)r;
    memcpy(rec + 36, &weight, 4);
    rec[40] = r >= 10;
  }
  ORBVocabulary voc;
  EXPECT(voc.loadFromMemory(blob.data(), blob.size()));
  EXPECT(voc.size() == 100);

  std::mt19937 rng(7);
  std::vector<KeyFrame> kfs(60);
  for (int i = 0; i < 60; i++) {
    kfs[i].mnId = 1000 + i;
    double sum = 0;
    for (int w = 0; w < 100; w++)
      if (rng() % 4 == 0) { kfs[i].mBowVec[w] = 1.0 + rng() % 100; sum += kfs[i].mBowVec[w]; }
    for (auto& e : kfs[i].mBowVec) e.second /= sum;
  }
  for (int i = 0; i < 60; i++)
    for (int d = 1; d <= 5; d++) {
      if (i + d < 60) kfs[i].best.push_back(&kfs[i + d]);
      if (i - d >= 0) kfs[i].best.push_back(&kfs[i - d]);
      if (d <= 2 && i + d < 60) kfs[i].connected.insert(&kfs[i + d]);
    }
  KeyFrameDatabase* mpKeyFrameDB = new KeyFrameDatabase(voc);
  orc_kfdb* o = orc_kfdb_create(100);
  std::vector<uint64_t> ids, nbs;
  std::vector<int32_t> noff(1, 0);
  std::vector<uint32_t> w;
  std::vector<double> v;
  for (auto& k : kfs) {
    mpKeyFrameDB->add(&k);
    split(k.mBowVec, w, v);
    orc_kfdb_add(o, k.mnId, (int)w.size(), w.data(), v.data());
    ids.push_back(k.mnId);
    for (KeyFrame* n : k.best) nbs.push_back(n->mnId);
    noff.push_back((int32_t)nbs.size());
  }
  orc_kfdb_set_neighbours(o, (int)ids.size(), ids.data(), noff.data(), nbs.data());
  mpKeyFrameDB->erase(&kfs[3]);
  orc_kfdb_erase(o, kfs[3].mnId);
  mpKeyFrameDB->add(&kfs[3]);
  split(kfs[3].mBowVec, w, v);
  orc_kfdb_add(o, kfs[3].mnId, (int)w.size(), w.data(), v.data());

  std::vector<uint64_t> sid(64), cid(64);
  std::vector<float> ssc(64);
  int ns = 0, checked = 0;
  for (int t = 0; t < 40; t++) {
    KeyFrame& src = kfs[rng() % 60];
    Frame mCurrentFrame{(long unsigned)t, src.mBowVec};
    if (t % 3 == 0) mCurrentFrame.mBowVec.erase(mCurrentFrame.mBowVec.begin());
    // Tracking::Relocalization
    std::vector<KeyFrame*> vpCandidateKFs = mpKeyFrameDB->DetectRelocalizationCandidates(&mCurrentFrame);
    split(mCurrentFrame.mBowVec, w, v);
    int nc = orc_kfdb_query(o, 0, (int)w.size(), w.data(), v.data(), 0.f, 0, nullptr, sid.data(), ssc.data(), 64, &ns,
                            cid.data(), 64);
    EXPECT((int)vpCandidateKFs.size() == nc);
    for (int i = 0; i < nc && i < (int)vpCandidateKFs.size(); i++) EXPECT(vpCandidateKFs[i]->mnId == cid[i]);
    // LoopClosing::DetectLoop: minScore from ORBVocabulary::score over the covisible keyframes
    KeyFrame* mpCurrentKF = &src;
    const DBoW2::BowVector& CurrentBowVec = mpCurrentKF->mBowVec;
    float minScore = 1;
    for (KeyFrame* pKF : mpCurrentKF->GetBestCovisibilityKeyFrames(10)) {
      float score = voc.score(CurrentBowVec, pKF->mBowVec);
      std::vector<uint32_t> w2;
      std::vector<double> v2;
      split(CurrentBowVec, w, v);
      split(pKF->mBowVec, w2, v2);
      EXPECT(voc.score(CurrentBowVec, pKF->mBowVec) ==
             orc_l1_score((int)w.size(), w.data(), v.data(), (int)w2.size(), w2.data(), v2.data()));
      if (score < minScore) minScore = score;
    }
    std::vector<KeyFrame*> vpLoop = mpKeyFrameDB->DetectLoopCandidates(mpCurrentKF, minScore);
    std::vector<uint64_t> conn;
    for (KeyFrame* c : mpCurrentKF->GetConnectedKeyFrames()) conn.push_back(c->mnId);
    split(CurrentBowVec, w, v);
    nc = orc_kfdb_query(o, 1, (int)w.size(), w.data(), v.data(), minScore, (int)conn.size(), conn.data(), sid.data(),
                        ssc.data(), 64, &ns, cid.data(), 64);
    EXPECT((int)vpLoop.size() == nc);
    for (int i = 0; i < nc && i < (int)vpLoop.size(); i++) EXPECT(vpLoop[i]->mnId == cid[i]);
    checked += nc + (int)vpCandidateKFs.size();
  }
  mpKeyFrameDB->clear();
  Frame empty{999, kfs[0].mBowVec};
  std::vector<KeyFrame*> none = mpKeyFrameDB->DetectRelocalizationCandidates(&empty);
  EXPECT(none.empty());
  delete mpKeyFrameDB;
  orc_kfdb_destroy(o);
  EXPECT(checked > 0);
  if (fails) return 1;
  std::printf("KFDB_WRAPPER_OK %d candidates\n", checked);
  return 0;
}
