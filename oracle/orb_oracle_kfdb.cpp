// orb_oracle_kfdb.cpp -- CPU oracle of KeyFrameDatabase (test infrastructure; see orb_oracle_kfdb.h).
//
// A literal restatement of ORB-SLAM2's KeyFrameDatabase.cc as SwarmMap carries it, with the reference's own
// containers: one std::list<KF*> per word with push_back on add, std::list<pair<float, KF*>> for the scored and the
// accumulated lists, a std::set for de-duplication, and the per-keyframe members mnRelocQuery / mnRelocWords /
// mRelocScore and mnLoopQuery / mnLoopWords / mLoopScore.
//
//   L1 score (ScoringObject.cpp, L1Scoring::score): merge walk of the two ascending word lists; over the common words,
//     in ascending word order, score += fabs(vi - wi) - fabs(vi) - fabs(wi) in double; return -score / 2.0.  The
//     database stores it as float si.
//   Shared-word walk: for each word of the query in ascending order, walk that word's inverted list in list order.
//     The first time a keyframe is met it is appended to lKFsSharingWords; every meeting increments its word count.
//     The list order is therefore "first common word, then add order"; erase + re-add moves a keyframe to the back
//     of every list.
//   Thresholds: int minCommonWords = maxCommonWords * 0.8f (int truncation); a keyframe is scored iff words > it.
//   Reloc: every scored keyframe enters lScoreAndMatch.
//   Loop: keyframes in the query's GetConnectedKeyFrames() are never listed; a keyframe is scored if it passes the
//     word test and enters lScoreAndMatch only if si >= minScore.
//   Covisibility accumulation: per entry, in list order, walk the candidate's GetBestCovisibilityKeyFrames(10) in the
//     given order; accScore starts at si, summed in float; pBestKF changes only on a strictly greater score.  Reloc
//     counts every neighbour that shares a word with this query (mnRelocQuery == F->mnId), scored or not; loop counts
//     a neighbour only if mnLoopQuery == id && mnLoopWords > minCommonWords.  bestAccScore starts at 0 (reloc) and
//     at minScore (loop).
//   Retain: keep an entry if accScore > 0.75f * bestAccScore; output pBestKF in list order, first occurrence only.
//
// Frozen definitions (DESIGN.md section 2):
//   1. Stale reloc scores are reproduced: a sharing but unscored reloc neighbour contributes the mRelocScore of the
//      most recent earlier query that scored it.  The state lives per keyframe id for the database's lifetime and
//      survives erase, re-add and clear.
//   2. mRelocScore / mLoopScore start at 0.0f (uninitialised in the reference).
//   3. Every query is a fresh query: it gets a query id no earlier query had, so word counts never carry over.
//      This equals the reference whenever query ids do not repeat (Tracking and LoopClosing never repeat them).
#include "orb_oracle_kfdb.h"

#include <chrono>
#include <cmath>
#include <list>
#include <map>
#include <set>
#include <unordered_map>
#include <utility>
#include <vector>

namespace {

typedef std::map<uint32_t, double> BowVector;  // DBoW2::BowVector: std::map<WordId, WordValue>

struct KF {
  uint64_t mnId = 0;
  BowVector mBowVec;
  bool live = false;
  long unsigned int mnRelocQuery = 0;
  int mnRelocWords = 0;
  float mRelocScore = 0.0f;  // frozen definition 2
  long unsigned int mnLoopQuery = 0;
  int mnLoopWords = 0;
  float mLoopScore = 0.0f;
};

double l1_score(const BowVector& v1, const BowVector& v2) {
  BowVector::const_iterator v1_it = v1.begin(), v2_it = v2.begin();
  const BowVector::const_iterator v1_end = v1.end(), v2_end = v2.end();
  double score = 0;
  while (v1_it != v1_end && v2_it != v2_end) {
    const double& vi = v1_it->second;
    const double& wi = v2_it->second;
    if (v1_it->first == v2_it->first) {
      score += fabs(vi - wi) - fabs(vi) - fabs(wi);
      ++v1_it;
      ++v2_it;
    } else if (v1_it->first < v2_it->first) {
      v1_it = v1.lower_bound(v2_it->first);
    } else {
      v2_it = v2.lower_bound(v1_it->first);
    }
  }
  score = -score / 2.0;
  return score;
}

BowVector make_bow(int n, const uint32_t* words, const double* values) {
  BowVector v;
  for (int i = 0; i < n; i++) v.insert(v.end(), std::make_pair(words[i], values[i]));
  return v;
}

}  // namespace

struct orc_kfdb {
  std::vector<std::list<KF*>> mvInvertedFile;
  std::map<uint64_t, KF*> kfs;  // every keyframe ever added: the reference's KeyFrame objects outlive erase / clear
  std::map<uint64_t, std::vector<uint64_t>> neigh;
  long unsigned int next_query = 1;  // frozen definition 3

  std::vector<KF*> best_covisibility(const KF* k) {
    std::vector<KF*> out;
    auto it = neigh.find(k->mnId);
    if (it == neigh.end()) return out;
    for (uint64_t id : it->second) {
      auto f = kfs.find(id);
      if (f != kfs.end()) out.push_back(f->second);  // an id never added shares no word with any query
    }
    return out;
  }

  std::vector<KF*> reloc(const BowVector& bow, const long unsigned int mnId, std::list<std::pair<float, KF*>>& lScoreAndMatch) {
    std::list<KF*> lKFsSharingWords;
    for (BowVector::const_iterator vit = bow.begin(), vend = bow.end(); vit != vend; vit++) {
      std::list<KF*>& lKFs = mvInvertedFile[vit->first];
      for (std::list<KF*>::iterator lit = lKFs.begin(), lend = lKFs.end(); lit != lend; lit++) {
        KF* pKFi = *lit;
        if (pKFi->mnRelocQuery != mnId) {
          pKFi->mnRelocWords = 0;
          pKFi->mnRelocQuery = mnId;
          lKFsSharingWords.push_back(pKFi);
        }
        pKFi->mnRelocWords++;
      }
    }
    if (lKFsSharingWords.empty()) return std::vector<KF*>();
    int maxCommonWords = 0;
    for (std::list<KF*>::iterator lit = lKFsSharingWords.begin(), lend = lKFsSharingWords.end(); lit != lend; lit++)
      if ((*lit)->mnRelocWords > maxCommonWords) maxCommonWords = (*lit)->mnRelocWords;
    int minCommonWords = maxCommonWords * 0.8f;
    for (std::list<KF*>::iterator lit = lKFsSharingWords.begin(), lend = lKFsSharingWords.end(); lit != lend; lit++) {
      KF* pKFi = *lit;
      if (pKFi->mnRelocWords > minCommonWords) {
        float si = l1_score(bow, pKFi->mBowVec);
        pKFi->mRelocScore = si;
        lScoreAndMatch.push_back(std::make_pair(si, pKFi));
      }
    }
    if (lScoreAndMatch.empty()) return std::vector<KF*>();
    std::list<std::pair<float, KF*>> lAccScoreAndMatch;
    float bestAccScore = 0;
    for (auto it = lScoreAndMatch.begin(), itend = lScoreAndMatch.end(); it != itend; it++) {
      KF* pKFi = it->second;
      std::vector<KF*> vpNeighs = best_covisibility(pKFi);
      float bestScore = it->first;
      float accScore = bestScore;
      KF* pBestKF = pKFi;
      for (std::vector<KF*>::iterator vit = vpNeighs.begin(), vend = vpNeighs.end(); vit != vend; vit++) {
        KF* pKF2 = *vit;
        if (pKF2->mnRelocQuery != mnId) continue;
        accScore += pKF2->mRelocScore;
        if (pKF2->mRelocScore > bestScore) {
          pBestKF = pKF2;
          bestScore = pKF2->mRelocScore;
        }
      }
      lAccScoreAndMatch.push_back(std::make_pair(accScore, pBestKF));
      if (accScore > bestAccScore) bestAccScore = accScore;
    }
    return retain(lAccScoreAndMatch, bestAccScore);
  }

  std::vector<KF*> loop(const BowVector& bow, const long unsigned int mnId, const std::set<KF*>& spConnectedKeyFrames,
                        float minScore, std::list<std::pair<float, KF*>>& lScoreAndMatch) {
    std::list<KF*> lKFsSharingWords;
    for (BowVector::const_iterator vit = bow.begin(), vend = bow.end(); vit != vend; vit++) {
      std::list<KF*>& lKFs = mvInvertedFile[vit->first];
      for (std::list<KF*>::iterator lit = lKFs.begin(), lend = lKFs.end(); lit != lend; lit++) {
        KF* pKFi = *lit;
        if (pKFi->mnLoopQuery != mnId) {
          pKFi->mnLoopWords = 0;
          if (!spConnectedKeyFrames.count(pKFi)) {
            pKFi->mnLoopQuery = mnId;
            lKFsSharingWords.push_back(pKFi);
          }
        }
        pKFi->mnLoopWords++;
      }
    }
    if (lKFsSharingWords.empty()) return std::vector<KF*>();
    int maxCommonWords = 0;
    for (std::list<KF*>::iterator lit = lKFsSharingWords.begin(), lend = lKFsSharingWords.end(); lit != lend; lit++)
      if ((*lit)->mnLoopWords > maxCommonWords) maxCommonWords = (*lit)->mnLoopWords;
    int minCommonWords = maxCommonWords * 0.8f;
    for (std::list<KF*>::iterator lit = lKFsSharingWords.begin(), lend = lKFsSharingWords.end(); lit != lend; lit++) {
      KF* pKFi = *lit;
      if (pKFi->mnLoopWords > minCommonWords) {
        float si = l1_score(bow, pKFi->mBowVec);
        pKFi->mLoopScore = si;
        if (si >= minScore) lScoreAndMatch.push_back(std::make_pair(si, pKFi));
      }
    }
    if (lScoreAndMatch.empty()) return std::vector<KF*>();
    std::list<std::pair<float, KF*>> lAccScoreAndMatch;
    float bestAccScore = minScore;
    for (auto it = lScoreAndMatch.begin(), itend = lScoreAndMatch.end(); it != itend; it++) {
      KF* pKFi = it->second;
      std::vector<KF*> vpNeighs = best_covisibility(pKFi);
      float bestScore = it->first;
      float accScore = it->first;
      KF* pBestKF = pKFi;
      for (std::vector<KF*>::iterator vit = vpNeighs.begin(), vend = vpNeighs.end(); vit != vend; vit++) {
        KF* pKF2 = *vit;
        if (pKF2->mnLoopQuery == mnId && pKF2->mnLoopWords > minCommonWords) {
          accScore += pKF2->mLoopScore;
          if (pKF2->mLoopScore > bestScore) {
            pBestKF = pKF2;
            bestScore = pKF2->mLoopScore;
          }
        }
      }
      lAccScoreAndMatch.push_back(std::make_pair(accScore, pBestKF));
      if (accScore > bestAccScore) bestAccScore = accScore;
    }
    return retain(lAccScoreAndMatch, bestAccScore);
  }

  static std::vector<KF*> retain(std::list<std::pair<float, KF*>>& lAccScoreAndMatch, float bestAccScore) {
    float minScoreToRetain = 0.75f * bestAccScore;
    std::set<KF*> spAlreadyAddedKF;
    std::vector<KF*> vpCandidates;
    vpCandidates.reserve(lAccScoreAndMatch.size());
    for (auto it = lAccScoreAndMatch.begin(), itend = lAccScoreAndMatch.end(); it != itend; it++) {
      if (it->first > minScoreToRetain) {
        KF* pKFi = it->second;
        if (!spAlreadyAddedKF.count(pKFi)) {
          vpCandidates.push_back(pKFi);
          spAlreadyAddedKF.insert(pKFi);
        }
      }
    }
    return vpCandidates;
  }

  std::vector<KF*> query(int mode, const BowVector& bow, float min_score, int n_conn, const uint64_t* conn,
                         std::list<std::pair<float, KF*>>& scored) {
    const long unsigned int id = next_query++;
    if (mode == 0) return reloc(bow, id, scored);
    std::set<KF*> connected;
    for (int i = 0; i < n_conn; i++) {
      auto f = kfs.find(conn[i]);
      if (f != kfs.end()) connected.insert(f->second);
    }
    return loop(bow, id, connected, min_score, scored);
  }
};

extern "C" {

double orc_l1_score(int na, const uint32_t* aw, const double* av, int nb, const uint32_t* bw, const double* bv) {
  return l1_score(make_bow(na, aw, av), make_bow(nb, bw, bv));
}

orc_kfdb* orc_kfdb_create(int n_words) {
  orc_kfdb* db = new orc_kfdb();
  db->mvInvertedFile.resize(n_words);
  return db;
}

void orc_kfdb_destroy(orc_kfdb* db) {
  if (!db) return;
  for (auto& kv : db->kfs) delete kv.second;
  delete db;
}

int orc_kfdb_add(orc_kfdb* db, uint64_t id, int n, const uint32_t* words, const double* values) {
  for (int i = 0; i < n; i++)
    if (words[i] >= db->mvInvertedFile.size() || (i && words[i] <= words[i - 1])) return -1;
  KF*& k = db->kfs[id];
  if (!k) {
    k = new KF();
    k->mnId = id;
  } else if (k->live) {
    return -1;
  }
  k->mBowVec = make_bow(n, words, values);
  k->live = true;
  for (BowVector::const_iterator vit = k->mBowVec.begin(), vend = k->mBowVec.end(); vit != vend; vit++)
    db->mvInvertedFile[vit->first].push_back(k);
  return 0;
}

void orc_kfdb_erase(orc_kfdb* db, uint64_t id) {
  auto f = db->kfs.find(id);
  if (f == db->kfs.end() || !f->second->live) return;
  KF* pKF = f->second;
  for (BowVector::const_iterator vit = pKF->mBowVec.begin(), vend = pKF->mBowVec.end(); vit != vend; vit++) {
    std::list<KF*>& lKFs = db->mvInvertedFile[vit->first];
    for (std::list<KF*>::iterator lit = lKFs.begin(), lend = lKFs.end(); lit != lend; lit++) {
      if (pKF == *lit) {
        lKFs.erase(lit);
        break;
      }
    }
  }
  pKF->live = false;
}

void orc_kfdb_clear(orc_kfdb* db) {
  const size_t n = db->mvInvertedFile.size();
  db->mvInvertedFile.clear();
  db->mvInvertedFile.resize(n);
  for (auto& kv : db->kfs) kv.second->live = false;
}

int orc_kfdb_size(const orc_kfdb* db) {
  int n = 0;
  for (const auto& kv : db->kfs) n += kv.second->live;
  return n;
}

void orc_kfdb_set_neighbours(orc_kfdb* db, int n, const uint64_t* ids, const int32_t* offsets, const uint64_t* neigh) {
  db->neigh.clear();
  for (int i = 0; i < n; i++) db->neigh[ids[i]] = std::vector<uint64_t>(neigh + offsets[i], neigh + offsets[i + 1]);
}

int orc_kfdb_query(orc_kfdb* db, int mode, int n, const uint32_t* words, const double* values, float min_score,
                   int n_conn, const uint64_t* conn, uint64_t* scored_ids, float* scored_scores, int scored_cap,
                   int* n_scored, uint64_t* cand_ids, int cand_cap) {
  std::list<std::pair<float, KF*>> scored;
  const std::vector<KF*> cand = db->query(mode, make_bow(n, words, values), min_score, n_conn, conn, scored);
  int i = 0;
  for (const auto& e : scored) {
    if (i < scored_cap) {
      scored_ids[i] = e.second->mnId;
      scored_scores[i] = e.first;
    }
    i++;
  }
  *n_scored = i;
  for (size_t j = 0; j < cand.size() && (int)j < cand_cap; j++) cand_ids[j] = cand[j]->mnId;
  return (int)cand.size();
}

double orc_kfdb_time_queries(orc_kfdb* db, int mode, int nq, const int32_t* q_off, const uint32_t* q_words,
                             const double* q_values, const float* min_score, int iters) {
  std::vector<BowVector> q(nq);
  for (int i = 0; i < nq; i++) q[i] = make_bow(q_off[i + 1] - q_off[i], q_words + q_off[i], q_values + q_off[i]);
  size_t sink = 0;
  const auto t0 = std::chrono::steady_clock::now();
  for (int it = 0; it < iters; it++)
    for (int i = 0; i < nq; i++) {
      std::list<std::pair<float, KF*>> scored;
      sink += db->query(mode, q[i], mode ? min_score[i] : 0.f, 0, nullptr, scored).size();
    }
  const auto t1 = std::chrono::steady_clock::now();
  if (sink == (size_t)-1) return -1.0;
  return std::chrono::duration<double>(t1 - t0).count();
}

}  // extern "C"
