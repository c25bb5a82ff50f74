// ORBmatcher.h -- drop-in ORB_SLAM2::ORBmatcher on top of libswm_orb.so (include/swm_orb.h).
//
// Same constructor, constants and member signatures as the reference
// (/root/reference/code/include/ORBmatcher.h:37-102) for the entry points on the hot path:
//   DescriptorDistance, SearchForInitialization, SearchByProjection(Frame&, const Frame&, th, bMono),
//   SearchByProjection(Frame&, const vector<MapPoint*>&, th), SearchByBoW(KeyFrame*, Frame&, ...),
//   SearchByBoW(KeyFrame*, KeyFrame*, ...).
// The member functions are templates over the Frame / KeyFrame / MapPoint types so this header
// compiles both against the reference's own headers (instantiate with ORB_SLAM2::Frame etc.) and
// against small test doubles; they only touch the members the reference's implementation touches
// (file:line cited at each gather).  MapPoint pointers never cross the C ABI: the wrapper gathers
// flat arrays, calls swm_match_*, and scatters the indices back into mvpMapPoints / vpMatches.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef SWM_HAVE_OPENCV
#include <opencv2/core.hpp>
#else
#include "cv_shim.h"
#endif
#include "../../include/swm_orb.h"
#include "MapPointTable.h"

namespace ORB_SLAM2 {

class ORBmatcher {
 public:
  static const int TH_LOW = 50;        // ORBmatcher.cc:38
  static const int TH_HIGH = 100;      // ORBmatcher.cc:37
  static const int HISTO_LENGTH = 30;  // ORBmatcher.cc:39

  ORBmatcher(float nnratio = 0.6, bool checkOri = true, int device = 0)
      : mfNNratio(nnratio), mbCheckOrientation(checkOri), device_(device) {
    if (swm_matcher_create(device, &m_) != SWM_OK)
      throw std::runtime_error(std::string("ORBmatcher: ") + swm_matcher_last_error(nullptr));
  }
  ~ORBmatcher() { swm_matcher_destroy(m_); }
  ORBmatcher(const ORBmatcher&) = delete;
  ORBmatcher& operator=(const ORBmatcher&) = delete;

  // Hamming distance between two ORB descriptors (ORBmatcher.cc:1511-1525).  ONE 32-byte pair is host glue, not the
  // hot path: the reference's callers use it inside scalar loops (MapPoint.cc:368, Frame.cc:589), where a device
  // round trip per pair would cost four orders of magnitude more than the eight popcounts below, which give the same
  // integer as the reference's SWAR bit trick.  Everything batched -- DescriptorDistanceMatrix, DescriptorDistancePairs,
  // DistinctiveDescriptor, all Search* -- runs on the GPU and has no host path.
  static int DescriptorDistance(const cv::Mat& a, const cv::Mat& b) {
    uint32_t pa[8], pb[8];
    std::memcpy(pa, a.ptr(0), 32);
    std::memcpy(pb, b.ptr(0), 32);
    int dist = 0;
    for (int i = 0; i < 8; i++) dist += __builtin_popcount(pa[i] ^ pb[i]);
    return dist;
  }
  // n pairs in one device call (a, b: n x 32 bytes).
  static void DescriptorDistancePairs(const unsigned char* a, const unsigned char* b, int n, std::vector<int32_t>& out,
                                      int device = 0) {
    out.resize((size_t)n);
    if (swm_hamming_pairs(a, b, n, out.data(), device) != SWM_OK)
      throw std::runtime_error("ORBmatcher::DescriptorDistancePairs: no CUDA device (there is no CPU fallback)");
  }
  static void DescriptorDistanceMatrix(const unsigned char* a, int na, const unsigned char* b, int nb,
                                       std::vector<uint16_t>& out, int device = 0) {
    out.resize((size_t)na * nb);
    if (swm_hamming_matrix(a, na, b, nb, out.data(), device) != SWM_OK)
      throw std::runtime_error("ORBmatcher::DescriptorDistanceMatrix failed");
  }

  // MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:361-391): index of the observed descriptor with the least
  // median distance to the others.  In MapPoint.cc replace the N x N loop and the median scan by
  //   const int BestIdx = ORBmatcher::DistinctiveDescriptor(vDescriptors);
  // (many MapPoints at once: swm_distinctive_descriptors takes a CSR batch).
  static int DistinctiveDescriptor(const std::vector<cv::Mat>& vDescriptors, int device = 0) {
    const int n = (int)vDescriptors.size();
    if (n == 0) return -1;
    std::vector<uint8_t> d((size_t)n * 32);
    for (int i = 0; i < n; i++) std::memcpy(&d[(size_t)i * 32], vDescriptors[i].ptr(0), 32);
    const int32_t off[2] = {0, n};
    int32_t best = -1;
    if (swm_distinctive_descriptors(d.data(), off, 1, &best, nullptr, device) != SWM_OK)
      throw std::runtime_error("ORBmatcher::DistinctiveDescriptor failed (no CUDA device? there is no CPU fallback)");
    return best;
  }

  // ---- Matching for the Map Initialization (ORBmatcher.cc:375-479)
  template <class FrameT, class Point2fT>
  int SearchForInitialization(FrameT& F1, FrameT& F2, std::vector<Point2fT>& vbPrevMatched,
                              std::vector<int>& vnMatches12, int windowSize = 10) {
    FlatFrame a, b;
    const bool res = resident_of(F1, 0) && resident_of(F2, 0);  // both on the device, or both gathered
    gather(F1, a, res);
    gather(F2, b, res);
    std::vector<float> prev(2 * a.n);
    for (int i = 0; i < a.n; i++) { prev[2 * i] = vbPrevMatched[i].x; prev[2 * i + 1] = vbPrevMatched[i].y; }
    vnMatches12.assign(a.n, -1);
    int n = 0;
    swm_frame_view va = a.view(), vb = b.view();
    check(res ? swm_match_init_resident(m_, resident_of(F1, 0), resident_of(F2, 0), prev.data(), vnMatches12.data(),
                                        windowSize, mfNNratio, mbCheckOrientation, &n)
              : swm_match_init(m_, &va, &vb, prev.data(), vnMatches12.data(), windowSize, mfNNratio, mbCheckOrientation, &n));
    for (int i = 0; i < a.n; i++) { vbPrevMatched[i].x = prev[2 * i]; vbPrevMatched[i].y = prev[2 * i + 1]; }
    return n;
  }

  // ---- Project MapPoints tracked in last frame into the current frame (ORBmatcher.cc:1223-1354), monocular.
  // The stereo-only forward/backward branches (:1243-1244,:1274-1277) need bMono == false and are not served.
  template <class FrameT>
  int SearchByProjection(FrameT& CurrentFrame, const FrameT& LastFrame, const float th, const bool bMono) {
    if (!bMono) throw std::runtime_error("ORBmatcher::SearchByProjection: stereo/RGB-D branch not supported (monocular SwarmMap)");
    FlatFrame cur;
    gather(CurrentFrame, cur);
    const int M = LastFrame.N;
    Query q(M);
    float R[9], t[3];
    pose(CurrentFrame.mTcw, R, t);
    for (int i = 0; i < M; i++) {
      auto* pMP = LastFrame.mvpMapPoints[i];
      if (!pMP || LastFrame.mvbOutlier[i]) continue;                       // :1247-1250
      float xw[3];
      world_pos(pMP->GetWorldPos(), xw);
      float xc[3];
      transform(R, t, xw, xc);                                              // :1252-1253
      const float invzc = 1.0 / xc[2];                                      // :1257
      if (invzc < 0) continue;
      const float u = CurrentFrame.fx * xc[0] * invzc + CurrentFrame.cx;    // :1262-1263
      const float v = CurrentFrame.fy * xc[1] * invzc + CurrentFrame.cy;
      if (u < CurrentFrame.mnMinX || u > CurrentFrame.mnMaxX) continue;
      if (v < CurrentFrame.mnMinY || v > CurrentFrame.mnMaxY) continue;
      const int oct = LastFrame.mvKeys[i].octave;                           // :1270
      q.valid[i] = 1;
      q.u[i] = u; q.v[i] = v;
      q.radius[i] = th * CurrentFrame.mvScaleFactors[oct];                  // :1273
      q.min_level[i] = oct - 1; q.max_level[i] = oct + 1;                   // :1282
      q.angle[i] = LastFrame.mvKeysUn[i].angle;
      q.blocks[i] = pMP->Observations() > 0;                                // :1291-1293
      std::memcpy(&q.desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);  // :1287
    }
    std::vector<uint8_t> blocked(cur.n, 0);
    for (int j = 0; j < cur.n; j++)
      blocked[j] = CurrentFrame.mvpMapPoints[j] && CurrentFrame.mvpMapPoints[j]->Observations() > 0;
    // assignment is in/out: untouched slots keep the sentinel, accepted slots get the source index,
    // slots assigned and then pruned by the rotation histogram come back as -1 (NULL, :1345-1348)
    const int32_t kUntouched = -3;
    std::vector<int32_t> asg(cur.n, kUntouched);
    int n = 0;
    swm_frame_view vc = cur.view();
    swm_window_query wq = q.view();
    check(window_call(resident_of(CurrentFrame, 0), &vc, &wq, blocked.data(), TH_HIGH, 0, mbCheckOrientation, asg.data(), &n));
    for (int j = 0; j < cur.n; j++) {
      if (asg[j] >= 0) CurrentFrame.mvpMapPoints[j] = LastFrame.mvpMapPoints[asg[j]];  // :1317
      else if (asg[j] == -1) CurrentFrame.mvpMapPoints[j] = nullptr;
    }
    return n;
  }

  // ---- Search matches between Frame keypoints and projected MapPoints (ORBmatcher.cc:44-121).
  template <class FrameT, class MapPointT>
  int SearchByProjection(FrameT& F, const std::vector<MapPointT*>& vpMapPoints, const float th = 3) {
    FlatFrame f;
    gather(F, f);
    const int M = (int)vpMapPoints.size();
    Query q(M);
    const bool bFactor = th != 1.0;
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = vpMapPoints[i];
      if (!pMP->mbTrackInView || pMP->isBad()) continue;                    // :51-55
      const int lvl = pMP->mnTrackScaleLevel;
      float r = pMP->mTrackViewCos > 0.998 ? 2.5f : 4.0f;                   // RadiusByViewingCos :123-128
      if (bFactor) r *= th;
      q.valid[i] = 1;
      q.u[i] = pMP->mTrackProjX; q.v[i] = pMP->mTrackProjY;
      q.radius[i] = r * F.mvScaleFactors[lvl];                              // :66
      q.min_level[i] = lvl - 1; q.max_level[i] = lvl;
      q.blocks[i] = pMP->Observations() > 0;
      std::memcpy(&q.desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    std::vector<uint8_t> blocked(f.n, 0);
    for (int j = 0; j < f.n; j++) blocked[j] = F.mvpMapPoints[j] && F.mvpMapPoints[j]->Observations() > 0;  // :78-80
    std::vector<int32_t> asg(f.n, -1);
    int n = 0;
    swm_frame_view vf = f.view();
    swm_window_query wq = q.view();
    check(window_call(resident_of(F, 0), &vf, &wq, blocked.data(), TH_HIGH, 1, 0, asg.data(), &n));
    for (int j = 0; j < f.n; j++)
      if (asg[j] >= 0) F.mvpMapPoints[j] = vpMapPoints[asg[j]];             // :115
    return n;
  }

  // ---- Tracking::SearchLocalPoints (Tracking.cc:964-1006) with the MapPoints resident in `table`: the frame's own
  // points (bad ones NULLed, the others IncreaseVisible, mnLastFrameSeen, mbTrackInView = false), then isInFrustum(pMP,
  // 0.5) + PredictScale and SearchByProjection(F, vpMapPoints, th) in one GPU call, then isInFrustum's writes
  // (mbTrackInView, mTrackProjX/Y, mTrackViewCos, mnTrackScaleLevel) and IncreaseVisible in list order.  F must be
  // resident (host/ResidentFrame.h); points the table does not hold yet are upserted first.  *nToMatch (may be NULL):
  // the points found in view.  Monocular: mTrackProjXR is not written.
  template <class FrameT, class MapPointT>
  int SearchByProjection(FrameT& F, const std::vector<MapPointT*>& vpMapPoints, const float th,
                         MapPointTable<MapPointT>& table, int* nToMatch = nullptr) {
    const swm_frame* res = resident_of(F, 0);
    if (!res) throw std::runtime_error("ORBmatcher::SearchByProjection(F, vpMapPoints, th, table): F must be resident");
    for (auto& pMP : F.mvpMapPoints) {  // :970-979
      if (!pMP) continue;
      if (pMP->isBad()) {
        pMP = nullptr;
        continue;
      }
      pMP->IncreaseVisible();
      pMP->mnLastFrameSeen = F.mnId;
      pMP->mbTrackInView = false;
    }
    std::vector<MapPointT*> missing;
    for (MapPointT* p : F.mvpMapPoints)
      if (p && table.Row(p) < 0) missing.push_back(p);
    for (MapPointT* p : vpMapPoints)
      if (table.Row(p) < 0) missing.push_back(p);
    table.Upsert(missing);
    const int M = (int)vpMapPoints.size(), N = F.N;
    std::vector<int32_t> rows(M), frame_rows(N, -1), asg(N, -1), level(M);
    for (int i = 0; i < M; i++) rows[i] = table.Row(vpMapPoints[i]);
    for (int j = 0; j < N; j++)
      if (F.mvpMapPoints[j]) frame_rows[j] = table.Row(F.mvpMapPoints[j]);
    std::vector<uint8_t> in_view(M);
    std::vector<float> u(M), v(M), view_cos(M);
    swm_track_out tr = {in_view.data(), u.data(), v.data(), view_cos.data(), level.data()};
    swm_projection proj = projection(F);
    int n = 0, ntm = 0;
    check(swm_match_local_map(m_, res, table.get(), &proj, rows.data(), M, frame_rows.data(), th, mfNNratio, &tr,
                              asg.data(), &n, &ntm));
    for (int i = 0; i < M; i++) {  // :985-996, in list order
      MapPointT* pMP = vpMapPoints[i];
      if (pMP->mnLastFrameSeen == F.mnId || pMP->isBad()) continue;
      pMP->mbTrackInView = in_view[i] != 0;
      if (!in_view[i]) continue;
      pMP->mTrackProjX = u[i];
      pMP->mTrackProjY = v[i];
      pMP->mTrackViewCos = view_cos[i];
      pMP->mnTrackScaleLevel = level[i];
      pMP->IncreaseVisible();
    }
    if (nToMatch) *nToMatch = ntm;
    for (int j = 0; j < N; j++)
      if (asg[j] >= 0) F.mvpMapPoints[j] = vpMapPoints[asg[j]];  // ORBmatcher.cc:115
    return n;
  }

  // ---- SearchByProjection(CurrentFrame, LastFrame, th, bMono) (ORBmatcher.cc:1223-1354) with the last frame's points
  // projected on the GPU from `table`.  Both frames must be resident; points the table does not hold yet are upserted.
  template <class FrameT, class MapPointT>
  int SearchByProjection(FrameT& CurrentFrame, const FrameT& LastFrame, const float th, const bool bMono,
                         MapPointTable<MapPointT>& table) {
    if (!bMono) throw std::runtime_error("ORBmatcher::SearchByProjection: stereo/RGB-D branch not supported (monocular SwarmMap)");
    const swm_frame *cur = resident_of(CurrentFrame, 0), *last = resident_of(LastFrame, 0);
    if (!cur || !last) throw std::runtime_error("ORBmatcher::SearchByProjection(cur, last, th, bMono, table): both frames must be resident");
    std::vector<MapPointT*> missing;
    for (int i = 0; i < LastFrame.N; i++) {
      MapPointT* p = LastFrame.mvpMapPoints[i];
      if (p && !LastFrame.mvbOutlier[i] && table.Row(p) < 0) missing.push_back(p);
    }
    for (MapPointT* p : CurrentFrame.mvpMapPoints)
      if (p && table.Row(p) < 0) missing.push_back(p);
    table.Upsert(missing);
    std::vector<int32_t> last_rows(LastFrame.N, -1), cur_rows(CurrentFrame.N, -1);
    for (int i = 0; i < LastFrame.N; i++) {  // :1247-1250
      MapPointT* p = LastFrame.mvpMapPoints[i];
      if (p && !LastFrame.mvbOutlier[i]) last_rows[i] = table.Row(p);
    }
    for (int j = 0; j < CurrentFrame.N; j++)
      if (CurrentFrame.mvpMapPoints[j]) cur_rows[j] = table.Row(CurrentFrame.mvpMapPoints[j]);
    const int32_t kUntouched = -3;
    std::vector<int32_t> asg(CurrentFrame.N, kUntouched);
    swm_projection proj = projection(CurrentFrame);
    int n = 0;
    check(swm_match_last_frame(m_, cur, last, table.get(), &proj, last_rows.data(), cur_rows.data(), th,
                               mbCheckOrientation, asg.data(), &n));
    for (int j = 0; j < CurrentFrame.N; j++) {
      if (asg[j] >= 0) CurrentFrame.mvpMapPoints[j] = LastFrame.mvpMapPoints[asg[j]];  // :1317
      else if (asg[j] == -1) CurrentFrame.mvpMapPoints[j] = nullptr;
    }
    return n;
  }

  // ---- Project MapPoints seen in a KeyFrame into the Frame (relocalisation), ORBmatcher.cc:1356-1473.
  template <class FrameT, class KeyFrameT, class MapPointT>
  int SearchByProjection(FrameT& CurrentFrame, KeyFrameT* pKF, const std::set<MapPointT*>& sAlreadyFound, const float th,
                         const int ORBdist, const bool bGlobal = false) {
    FlatFrame cur;
    gather(CurrentFrame, cur);
    const std::vector<MapPointT*> vpMPs = pKF->GetMapPointMatches();
    const int M = (int)vpMPs.size();
    Query q(M);
    float R[9], t[3];
    pose(CurrentFrame.mTcw, R, t);
    float Ow[3];
    centre(R, t, Ow);                                                     // :1362
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = vpMPs[i];
      if (!pMP || pMP->isBad() || sAlreadyFound.count(pMP)) continue;     // :1379
      float xw[3];
      world_pos(bGlobal ? pMP->GetGlobalPos() : pMP->GetWorldPos(), xw);  // :1382
      float xc[3];
      transform(R, t, xw, xc);
      const float invzc = 1.0 / xc[2];
      const float u = FrameT::fx * xc[0] * invzc + FrameT::cx;            // :1389-1390
      const float v = FrameT::fy * xc[1] * invzc + FrameT::cy;
      if (u < FrameT::mnMinX || u > FrameT::mnMaxX) continue;
      if (v < FrameT::mnMinY || v > FrameT::mnMaxY) continue;
      const float PO[3] = {xw[0] - Ow[0], xw[1] - Ow[1], xw[2] - Ow[2]};
      const float dist3D = norm3(PO);                                     // cv::norm(PO), :1399
      if (dist3D < pMP->GetMinDistanceInvariance() || dist3D > pMP->GetMaxDistanceInvariance()) continue;
      const int lvl = pMP->PredictScale(dist3D, CurrentFrame.mfLogScaleFactor, CurrentFrame.mnScaleLevels);
      q.valid[i] = 1;
      q.u[i] = u; q.v[i] = v;
      q.radius[i] = th * CurrentFrame.mvScaleFactors[lvl];                // :1413
      q.min_level[i] = lvl - 1; q.max_level[i] = lvl + 1;
      q.angle[i] = pKF->mvKeysUn[i].angle;
      q.blocks[i] = 1;
      std::memcpy(&q.desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    std::vector<uint8_t> blocked(cur.n, 0);
    for (int j = 0; j < cur.n; j++) blocked[j] = CurrentFrame.mvpMapPoints[j] != nullptr;  // :1425
    const int32_t kUntouched = -3;
    std::vector<int32_t> asg(cur.n, kUntouched);
    int n = 0;
    swm_frame_view vc = cur.view();
    swm_window_query wq = q.view();
    check(window_call(resident_of(CurrentFrame, 0), &vc, &wq, blocked.data(), ORBdist, 0, mbCheckOrientation, asg.data(), &n));
    for (int j = 0; j < cur.n; j++) {
      if (asg[j] >= 0) CurrentFrame.mvpMapPoints[j] = vpMPs[asg[j]];
      else if (asg[j] == -1) CurrentFrame.mvpMapPoints[j] = nullptr;
    }
    return n;
  }

  // ---- Project MapPoints with a Sim3 into a KeyFrame (loop closing), ORBmatcher.cc:264-373.
  template <class KeyFrameT, class MatT, class MapPointT>
  int SearchByProjection(KeyFrameT* pKF, const MatT& Scw, const std::vector<MapPointT*>& vpPoints,
                         std::vector<MapPointT*>& vpMatched, int th) {
    FlatFrame kf;
    gather(*pKF, kf);
    // decompose Scw (:273-277)
    float R[9], t[3], Ow[3];
    sim3_decompose(Scw, R, t, Ow);
    std::set<MapPointT*> found(vpMatched.begin(), vpMatched.end());
    found.erase(static_cast<MapPointT*>(nullptr));
    const int M = (int)vpPoints.size();
    Query q(M);
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = vpPoints[i];
      if (pMP->isBad() || found.count(pMP)) continue;                     // :291
      float xw[3], xc[3];
      world_pos(pMP->GetWorldPos(), xw);
      transform(R, t, xw, xc);
      if (xc[2] < 0.0) continue;                                          // :301
      const float invz = 1 / xc[2];
      const float u = pKF->fx * (xc[0] * invz) + pKF->cx;
      const float v = pKF->fy * (xc[1] * invz) + pKF->cy;
      if (!pKF->IsInImage(u, v)) continue;                                // :314
      const float PO[3] = {xw[0] - Ow[0], xw[1] - Ow[1], xw[2] - Ow[2]};
      const float dist = norm3(PO);                                       // :319
      if (dist < pMP->GetMinDistanceInvariance() || dist > pMP->GetMaxDistanceInvariance()) continue;
      float pn[3];
      world_pos(pMP->GetNormal(), pn);
      if (dot3(PO, pn) < 0.5 * dist) continue;                            // :327
      const int lvl = pMP->PredictScale(dist, pKF->mfLogScaleFactor, pKF->mnScaleLevels);
      q.valid[i] = 1;
      q.u[i] = u; q.v[i] = v;
      q.radius[i] = th * pKF->mvScaleFactors[lvl];                        // :334
      q.min_level[i] = lvl - 1; q.max_level[i] = lvl;                     // :351
      q.blocks[i] = 1;
      std::memcpy(&q.desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    std::vector<uint8_t> blocked(kf.n, 0);
    for (int j = 0; j < kf.n; j++) blocked[j] = vpMatched[j] != nullptr;  // :346
    std::vector<int32_t> asg(kf.n, -1);
    int n = 0;
    swm_frame_view vk = kf.view();
    swm_window_query wq = q.view();
    check(window_call(resident_of(*pKF, 0), &vk, &wq, blocked.data(), TH_LOW, 0, 0, asg.data(), &n));
    for (int j = 0; j < kf.n; j++)
      if (asg[j] >= 0) vpMatched[j] = vpPoints[asg[j]];                   // :366
    return n;
  }

  // ---- Search matches between MapPoints in a KeyFrame and ORB in a Frame (ORBmatcher.cc:150-262).
  template <class KeyFrameT, class FrameT, class MapPointT>
  int SearchByBoW(KeyFrameT* pKF, FrameT& F, std::vector<MapPointT*>& vpMapPointMatches) {
    const std::vector<MapPointT*> vpMapPointsKF = pKF->GetMapPointMatches();
    FlatFrame a, b;
    const bool res = resident_of(*pKF, 0) && resident_of(F, 0);
    gather(*pKF, a, res);
    gather(F, b, res);
    std::vector<uint8_t> valid(a.n, 0);
    for (int i = 0; i < a.n; i++) valid[i] = vpMapPointsKF[i] && !vpMapPointsKF[i]->isBad();  // :182-188
    FlatFeatVec fa(pKF->mFeatVec), fb(F.mFeatVec);
    std::vector<int32_t> out(b.n, -1);
    int n = 0;
    swm_frame_view va = a.view(), vb = b.view();
    swm_featvec ga = fa.view(), gb = fb.view();
    check(res ? swm_match_bow_resident(m_, resident_of(*pKF, 0), &ga, valid.data(), resident_of(F, 0), &gb, nullptr, 0,
                                       mfNNratio, mbCheckOrientation, out.data(), &n)
              : swm_match_bow(m_, &va, &ga, valid.data(), &vb, &gb, nullptr, 0, mfNNratio, mbCheckOrientation, out.data(), &n));
    vpMapPointMatches.assign(b.n, static_cast<MapPointT*>(nullptr));
    for (int j = 0; j < b.n; j++)
      if (out[j] >= 0) vpMapPointMatches[j] = vpMapPointsKF[out[j]];
    return n;
  }

  // ---- KeyFrame <-> KeyFrame (loop / merge candidates), ORBmatcher.cc:481-597.
  template <class KeyFrameT, class MapPointT>
  int SearchByBoW(KeyFrameT* pKF1, KeyFrameT* pKF2, std::vector<MapPointT*>& vpMatches12) {
    const std::vector<MapPointT*> mp1 = pKF1->GetMapPointMatches(), mp2 = pKF2->GetMapPointMatches();
    FlatFrame a, b;
    const bool res = resident_of(*pKF1, 0) && resident_of(*pKF2, 0);
    gather(*pKF1, a, res);
    gather(*pKF2, b, res);
    std::vector<uint8_t> v1(a.n, 0), v2(b.n, 0);
    for (int i = 0; i < a.n; i++) v1[i] = mp1[i] && !mp1[i]->isBad();
    for (int i = 0; i < b.n; i++) v2[i] = mp2[i] && !mp2[i]->isBad();
    FlatFeatVec fa(pKF1->mFeatVec), fb(pKF2->mFeatVec);
    std::vector<int32_t> out(a.n, -1);
    int n = 0;
    swm_frame_view va = a.view(), vb = b.view();
    swm_featvec ga = fa.view(), gb = fb.view();
    check(res ? swm_match_bow_resident(m_, resident_of(*pKF1, 0), &ga, v1.data(), resident_of(*pKF2, 0), &gb, v2.data(), 1,
                                       mfNNratio, mbCheckOrientation, out.data(), &n)
              : swm_match_bow(m_, &va, &ga, v1.data(), &vb, &gb, v2.data(), 1, mfNNratio, mbCheckOrientation, out.data(), &n));
    vpMatches12.assign(a.n, static_cast<MapPointT*>(nullptr));
    for (int i = 0; i < a.n; i++)
      if (out[i] >= 0) vpMatches12[i] = mp2[out[i]];
    return n;
  }

  // ---- Project MapPoints into a KeyFrame and search for duplicated MapPoints (ORBmatcher.cc:751-880), monocular.
  // Pass 1 (host): the reference's visibility tests and projection per MapPoint.  GPU: best keypoint in the window
  // (swm_window_best, levels [pred - 1, pred], reprojection gate 5.99).  Pass 2 (host, in list order): the
  // Replace / AddObservation bookkeeping, re-checking isBad() / IsInKeyFrame() at commit time because an earlier
  // Replace can retire a later point of the list (the reference tests them at the top of each iteration).
  template <class KeyFrameT, class MapPointT>
  int Fuse(KeyFrameT* pKF, const std::vector<MapPointT*>& vpMapPoints, const float th = 3.0) {
    float R[9], t[3], Ow[3];
    {
      const auto Rcw = pKF->GetRotation();
      const auto tcw = pKF->GetTranslation();
      for (int r = 0; r < 3; r++) {
        for (int c = 0; c < 3; c++) R[3 * r + c] = Rcw.template at<float>(r, c);
        t[r] = tcw.template at<float>(r);
      }
      world_pos(pKF->GetCameraCenter(), Ow);
    }
    const int M = (int)vpMapPoints.size();
    std::vector<uint8_t> desc((size_t)M * 32, 0), valid(M, 0);
    std::vector<float> u(M, 0.f), v(M, 0.f), radius(M, 0.f);
    std::vector<int32_t> lo(M, -1), hi(M, -1);
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = vpMapPoints[i];
      if (!pMP) continue;
      if (pMP->isBad() || pMP->IsInKeyFrame(pKF)) continue;
      float Pw[3], Pc[3];
      world_pos(pMP->GetWorldPos(), Pw);
      transform(R, t, Pw, Pc);
      if (Pc[2] < 0.0f) continue;                                          // :779-780
      const float invz = 1 / Pc[2];
      const float pu = pKF->fx * (Pc[0] * invz) + pKF->cx, pv = pKF->fy * (Pc[1] * invz) + pKF->cy;
      if (!pKF->IsInImage(pu, pv)) continue;                                // :790-791
      const float PO[3] = {Pw[0] - Ow[0], Pw[1] - Ow[1], Pw[2] - Ow[2]};
      const float dist3D = norm3(PO);                                      // cv::norm
      if (dist3D < pMP->GetMinDistanceInvariance() || dist3D > pMP->GetMaxDistanceInvariance()) continue;
      float Pn[3];
      world_pos(pMP->GetNormal(), Pn);
      if (dot3(PO, Pn) < 0.5 * dist3D) continue;                           // :808-809
      const int pred = pMP->PredictScale(dist3D, pKF->mfLogScaleFactor, pKF->mnScaleLevels);
      valid[i] = 1;
      u[i] = pu; v[i] = pv;
      radius[i] = th * pKF->mvScaleFactors[pred];                          // :814
      lo[i] = pred - 1; hi[i] = pred;                                       // :840-842
      std::memcpy(&desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    swm_best_query q;
    q.m = M; q.desc = desc.data(); q.u = u.data(); q.v = v.data(); q.radius = radius.data();
    q.min_level = lo.data(); q.max_level = hi.data(); q.valid = valid.data();
    q.inv_level_sigma2 = pKF->mvInvLevelSigma2.data();
    q.nlevels = (int32_t)pKF->mvInvLevelSigma2.size();
    q.chi2 = 5.99f;
    std::vector<int32_t> best_idx(M, -1), best_dist(M, 256);
    FlatFrame kf;
    gather(*pKF, kf);
    swm_frame_view vk = kf.view();
    check(resident_of(*pKF, 0) ? swm_window_best_resident(m_, resident_of(*pKF, 0), &q, best_idx.data(), best_dist.data())
                               : swm_window_best(m_, &vk, &q, best_idx.data(), best_dist.data()));
    int nFused = 0;
    for (int i = 0; i < M; i++) {
      if (!valid[i] || best_idx[i] < 0 || best_dist[i] > TH_LOW) continue;  // :873
      MapPointT* pMP = vpMapPoints[i];
      if (pMP->isBad() || pMP->IsInKeyFrame(pKF)) continue;                 // state may have changed since pass 1
      MapPointT* pMPinKF = pKF->GetMapPoint(best_idx[i]);
      if (pMPinKF) {
        if (!pMPinKF->isBad()) {
          if (pMPinKF->Observations() > pMP->Observations()) pMP->Replace(pMPinKF);
          else pMPinKF->Replace(pMP);
        }
      } else {
        pMP->AddObservation(pKF, best_idx[i]);
        pKF->AddMapPoint(pMP, best_idx[i]);
      }
      nFused++;
    }
    return nFused;
  }

  // ---- Project MapPoints into a KeyFrame using a given Sim3 and search for duplicated MapPoints (loop closing,
  // ORBmatcher.cc:891-1009).  Same split as the other Fuse: host projection, one swm_window_best call (no
  // reprojection gate), then the in-order bookkeeping (vpReplacePoint / AddObservation).
  template <class KeyFrameT, class MapPointT, class MatT>
  int Fuse(KeyFrameT* pKF, const MatT& Scw, const std::vector<MapPointT*>& vpPoints, float th,
           std::vector<MapPointT*>& vpReplacePoint) {
    // Decompose Scw (:899-904): scw = |row 0 of sRcw|, Rcw = sRcw / scw, tcw = Scw[0:3, 3] / scw, Ow = -Rcw' tcw
    float R[9], t[3], Ow[3];
    sim3_decompose(Scw, R, t, Ow);
    const auto spAlreadyFound = pKF->GetMapPoints();
    const int M = (int)vpPoints.size();
    std::vector<uint8_t> desc((size_t)M * 32, 0), valid(M, 0);
    std::vector<float> u(M, 0.f), v(M, 0.f), radius(M, 0.f);
    std::vector<int32_t> lo(M, -1), hi(M, -1);
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = vpPoints[i];
      if (pMP->isBad() || spAlreadyFound.count(pMP)) continue;             // :918-919
      float Pw[3], Pc[3];
      world_pos(pMP->GetGlobalPos(), Pw);
      transform(R, t, Pw, Pc);
      if (Pc[2] < 0.0f) continue;
      const float invz = (float)(1.0 / Pc[2]);
      const float pu = pKF->fx * (Pc[0] * invz) + pKF->cx, pv = pKF->fy * (Pc[1] * invz) + pKF->cy;
      if (!pKF->IsInImage(pu, pv)) continue;
      const float PO[3] = {Pw[0] - Ow[0], Pw[1] - Ow[1], Pw[2] - Ow[2]};
      const float dist3D = norm3(PO);
      if (dist3D < pMP->GetMinDistanceInvariance() || dist3D > pMP->GetMaxDistanceInvariance()) continue;
      float Pn[3];
      world_pos(pMP->GetNormal(), Pn);
      if (dot3(PO, Pn) < 0.5 * dist3D) continue;
      const int pred = pMP->PredictScale(dist3D, pKF->mfLogScaleFactor, pKF->mnScaleLevels);
      valid[i] = 1;
      u[i] = pu; v[i] = pv;
      radius[i] = th * pKF->mvScaleFactors[pred];
      lo[i] = pred - 1; hi[i] = pred;
      std::memcpy(&desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    swm_best_query q;
    q.m = M; q.desc = desc.data(); q.u = u.data(); q.v = v.data(); q.radius = radius.data();
    q.min_level = lo.data(); q.max_level = hi.data(); q.valid = valid.data();
    q.inv_level_sigma2 = nullptr; q.nlevels = 0; q.chi2 = 0.0f;
    std::vector<int32_t> best_idx(M, -1), best_dist(M, 256);
    FlatFrame kf;
    gather(*pKF, kf);
    swm_frame_view vk = kf.view();
    check(resident_of(*pKF, 0) ? swm_window_best_resident(m_, resident_of(*pKF, 0), &q, best_idx.data(), best_dist.data())
                               : swm_window_best(m_, &vk, &q, best_idx.data(), best_dist.data()));
    int nFused = 0;
    for (int i = 0; i < M; i++) {
      if (!valid[i] || best_idx[i] < 0 || best_dist[i] > TH_LOW) continue;  // :991
      MapPointT* pMP = vpPoints[i];
      MapPointT* pMPinKF = pKF->GetMapPoint(best_idx[i]);
      if (pMPinKF) {
        if (!pMPinKF->isBad()) vpReplacePoint[i] = pMPinKF;
      } else {
        pMP->AddObservation(pKF, best_idx[i]);
        pKF->AddMapPoint(pMP, best_idx[i]);
      }
      nFused++;
    }
    return nFused;
  }

  // ---- Search matches between MapPoints seen in KF1 and KF2 transforming by a Sim3 [s12*R12|t12]
  // (ORBmatcher.cc:1011-1221).  Host: the two projection loops; GPU: two swm_window_best calls (levels [pred - 1,
  // pred], no reprojection gate, accept at TH_HIGH); host: the mutual-agreement check.
  template <class KeyFrameT, class MapPointT, class MatT>
  int SearchBySim3(KeyFrameT* pKF1, KeyFrameT* pKF2, std::vector<MapPointT*>& vpMatches12, const float& s12, const MatT& R12,
                   const MatT& t12, const float th) {
    float R1w[9], t1w[3], R2w[9], t2w[3], sR12[9], sR21[9], T12[3], t21[3];
    load_pose(pKF1->GetRotation(), pKF1->GetTranslation(), R1w, t1w);
    load_pose(pKF2->GetRotation(), pKF2->GetTranslation(), R2w, t2w);
    for (int r = 0; r < 3; r++) {
      T12[r] = t12.template at<float>(r);
      for (int c = 0; c < 3; c++) {
        sR12[3 * r + c] = fmul(R12.template at<float>(r, c), s12);                              // s12 * R12
        sR21[3 * r + c] = fmul(R12.template at<float>(c, r), (float)(1.0 / (double)s12));       // (1.0 / s12) * R12.t()
      }
    }
    transform(sR21, nullptr, T12, t21, -1.0);  // t21 = -sR21 * t12
    const std::vector<MapPointT*> mp1 = pKF1->GetMapPointMatches(), mp2 = pKF2->GetMapPointMatches();
    const int N1 = (int)mp1.size(), N2 = (int)mp2.size();
    std::vector<uint8_t> already1(N1, 0), already2(N2, 0);
    for (int i = 0; i < N1; i++) {
      MapPointT* pMP = vpMatches12[i];
      if (pMP) {
        already1[i] = 1;
        const int idx2 = pMP->GetIndexInKeyFrame(pKF2);
        if (idx2 >= 0 && idx2 < N2) already2[idx2] = 1;
      }
    }
    std::vector<int32_t> match1, match2;
    sim3_direction(pKF1, pKF2, mp1, already1, R1w, t1w, sR21, t21, th, match1);  // KF1's points into KF2
    sim3_direction(pKF2, pKF1, mp2, already2, R2w, t2w, sR12, T12, th, match2);  // KF2's points into KF1
    int nFound = 0;
    for (int i1 = 0; i1 < N1; i1++) {  // :1207-1217
      const int idx2 = match1[i1];
      if (idx2 >= 0 && match2[idx2] == i1) {
        vpMatches12[i1] = mp2[idx2];
        nFound++;
      }
    }
    return nFound;
  }

  // ---- Matching to triangulate new MapPoints, with the epipolar constraint (ORBmatcher.cc:599-749), monocular.
  // F12 is the 3x3 CV_32F fundamental matrix LocalMapping::ComputeF12 builds.  The stereo branches need mvuRight >= 0
  // and are not served (bOnlyStereo must be false; SwarmMap is monocular).
  template <class KeyFrameT, class MatT>
  int SearchForTriangulation(KeyFrameT* pKF1, KeyFrameT* pKF2, const MatT& F12,
                             std::vector<std::pair<size_t, size_t>>& vMatchedPairs, const bool bOnlyStereo) {
    if (bOnlyStereo) throw std::runtime_error("ORBmatcher::SearchForTriangulation: stereo-only mode not supported (monocular SwarmMap)");
    // epipole in the second image (:605-611): C2 = R2w * Cw + t2w
    float Cw[3], R2w[9], t2w[3], C2[3];
    world_pos(pKF1->GetCameraCenter(), Cw);
    const auto R = pKF2->GetRotation();
    const auto t = pKF2->GetTranslation();
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) R2w[3 * r + c] = R.template at<float>(r, c);
      t2w[r] = t.template at<float>(r);
    }
    transform(R2w, t2w, Cw, C2);
    const float invz = 1.0f / C2[2];
    swm_triangulation_query q;
    float F[9];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) F[3 * r + c] = F12.template at<float>(r, c);
    q.F12 = F;
    q.ex = pKF2->fx * C2[0] * invz + pKF2->cx;
    q.ey = pKF2->fy * C2[1] * invz + pKF2->cy;
    q.scale_factors2 = pKF2->mvScaleFactors.data();
    q.level_sigma2 = pKF2->mvLevelSigma2.data();
    q.nlevels = (int32_t)pKF2->mvScaleFactors.size();
    FlatFrame a, b;
    const bool res = resident_of(*pKF1, 0) && resident_of(*pKF2, 0);
    gather(*pKF1, a, res);
    gather(*pKF2, b, res);
    std::vector<uint8_t> v1(a.n, 0), v2(b.n, 0);
    for (int i = 0; i < a.n; i++) v1[i] = pKF1->GetMapPoint(i) == nullptr;  // :640-643
    for (int i = 0; i < b.n; i++) v2[i] = pKF2->GetMapPoint(i) == nullptr;  // :662-666
    FlatFeatVec fa(pKF1->mFeatVec), fb(pKF2->mFeatVec);
    std::vector<int32_t> out(a.n, -1);
    int n = 0;
    swm_frame_view va = a.view(), vb = b.view();
    swm_featvec ga = fa.view(), gb = fb.view();
    check(res ? swm_match_triangulation_resident(m_, resident_of(*pKF1, 0), &ga, v1.data(), resident_of(*pKF2, 0), &gb,
                                                 v2.data(), &q, mbCheckOrientation, out.data(), &n)
              : swm_match_triangulation(m_, &va, &ga, v1.data(), &vb, &gb, v2.data(), &q, mbCheckOrientation, out.data(), &n));
    vMatchedPairs.clear();
    vMatchedPairs.reserve(n);
    for (int i = 0; i < a.n; i++)
      if (out[i] >= 0) vMatchedPairs.push_back(std::make_pair((size_t)i, (size_t)out[i]));  // :743-747
    return n;
  }

 protected:
  struct FlatFrame {
    int n = 0;
    std::vector<float> x, y, angle;
    std::vector<int32_t> octave;
    std::vector<uint8_t> desc;
    float min_x = 0, min_y = 0, max_x = 1, max_y = 1;
    swm_frame_view view() const {
      swm_frame_view v;
      v.n = n; v.x = x.data(); v.y = y.data(); v.octave = octave.data(); v.angle = angle.data(); v.desc = desc.data();
      v.min_x = min_x; v.min_y = min_y; v.max_x = max_x; v.max_y = max_y;
      return v;
    }
  };
  struct Query {
    std::vector<uint8_t> desc, valid, blocks;
    std::vector<float> u, v, radius, angle;
    std::vector<int32_t> min_level, max_level;
    explicit Query(int m) : desc((size_t)m * 32), valid(m, 0), blocks(m, 1), u(m), v(m), radius(m), angle(m),
                            min_level(m, -1), max_level(m, -1) {}
    swm_window_query view() const {
      swm_window_query q;
      q.m = (int)valid.size(); q.desc = desc.data(); q.u = u.data(); q.v = v.data(); q.radius = radius.data();
      q.min_level = min_level.data(); q.max_level = max_level.data(); q.valid = valid.data();
      q.angle = angle.data(); q.blocks = blocks.data();
      return q;
    }
  };
  // DBoW2::FeatureVector (std::map<NodeId, std::vector<unsigned>>) -> CSR in map order
  struct FlatFeatVec {
    std::vector<uint32_t> node_ids, feats;
    std::vector<int32_t> offsets;
    template <class FeatVecT>
    explicit FlatFeatVec(const FeatVecT& fv) {
      offsets.push_back(0);
      for (auto it = fv.begin(); it != fv.end(); ++it) {
        node_ids.push_back((uint32_t)it->first);
        for (unsigned idx : it->second) feats.push_back(idx);
        offsets.push_back((int32_t)feats.size());
      }
    }
    swm_featvec view() const {
      swm_featvec v;
      v.n_nodes = (int)node_ids.size(); v.node_ids = node_ids.data(); v.offsets = offsets.data(); v.feats = feats.data();
      return v;
    }
  };

  // A Frame / KeyFrame that carries `const swm_frame* mpResident` (built by ORB_SLAM2::ResidentFrame from the
  // extractor's device output, host/ResidentFrame.h) is matched in place on the GPU; otherwise its arrays are
  // gathered and uploaded per call.
  template <class FrameT>
  static auto resident_of(const FrameT& F, int) -> decltype(F.mpResident) { return F.mpResident; }
  template <class FrameT>
  static const swm_frame* resident_of(const FrameT&, long) { return nullptr; }
  int window_call(const swm_frame* res, const swm_frame_view* v, const swm_window_query* q, const uint8_t* blocked,
                  int th, int ratio_mode, int check_ori, int32_t* asg, int* n) {
    return res ? swm_match_window_resident(m_, res, q, blocked, th, ratio_mode, mfNNratio, check_ori, asg, n)
               : swm_match_window(m_, v, q, blocked, th, ratio_mode, mfNNratio, check_ori, asg, n);
  }

  // Frame / KeyFrame members read by every matcher: N, mvKeysUn, mDescriptors, image bounds.
  template <class FrameT>
  static void gather(const FrameT& F, FlatFrame& o, bool use_resident = true) {
    o.n = F.N;
    o.min_x = F.mnMinX; o.min_y = F.mnMinY; o.max_x = F.mnMaxX; o.max_y = F.mnMaxY;
    if (use_resident && resident_of(F, 0)) return;  // the arrays already live on the device
    o.x.resize(o.n); o.y.resize(o.n); o.angle.resize(o.n); o.octave.resize(o.n); o.desc.resize((size_t)o.n * 32);
    for (int i = 0; i < o.n; i++) {
      o.x[i] = F.mvKeysUn[i].pt.x; o.y[i] = F.mvKeysUn[i].pt.y;
      o.angle[i] = F.mvKeysUn[i].angle; o.octave[i] = F.mvKeysUn[i].octave;
      std::memcpy(&o.desc[(size_t)i * 32], F.mDescriptors.ptr(i), 32);
    }
  }
  template <class MatR, class MatTr>
  static void load_pose(const MatR& Rm, const MatTr& tm, float R[9], float t[3]) {
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) R[3 * r + c] = Rm.template at<float>(r, c);
      t[r] = tm.template at<float>(r);
    }
  }
  // One direction of SearchBySim3 (:1055-1129 / :1132-1204): the source keyframe's MapPoints, moved into the target
  // camera by (Rsw, tsw) then (sR, tt), searched in the target keyframe.  match[i] = target index or -1.
  template <class KeyFrameT, class MapPointT>
  void sim3_direction(KeyFrameT* pSrc, KeyFrameT* pTgt, const std::vector<MapPointT*>& mps, const std::vector<uint8_t>& already,
                      const float Rsw[9], const float tsw[3], const float sR[9], const float tt[3], float th,
                      std::vector<int32_t>& match) {
    (void)pSrc;
    const int M = (int)mps.size();
    match.assign(M, -1);
    std::vector<uint8_t> desc((size_t)M * 32, 0), valid(M, 0);
    std::vector<float> u(M, 0.f), v(M, 0.f), radius(M, 0.f);
    std::vector<int32_t> lo(M, -1), hi(M, -1);
    for (int i = 0; i < M; i++) {
      MapPointT* pMP = mps[i];
      if (!pMP || already[i]) continue;
      if (pMP->isBad()) continue;
      float Pw[3], Pa[3], Pb[3];
      world_pos(pMP->GetWorldPos(), Pw);
      transform(Rsw, tsw, Pw, Pa);
      transform(sR, tt, Pa, Pb);
      if (Pb[2] < 0.0) continue;
      const float invz = (float)(1.0 / Pb[2]);
      const float pu = pTgt->fx * (Pb[0] * invz) + pTgt->cx, pv = pTgt->fy * (Pb[1] * invz) + pTgt->cy;
      if (!pTgt->IsInImage(pu, pv)) continue;
      const float dist3D = norm3(Pb);
      if (dist3D < pMP->GetMinDistanceInvariance() || dist3D > pMP->GetMaxDistanceInvariance()) continue;
      const int pred = pMP->PredictScale(dist3D, pTgt->mfLogScaleFactor, pTgt->mnScaleLevels);
      valid[i] = 1;
      u[i] = pu; v[i] = pv;
      radius[i] = th * pTgt->mvScaleFactors[pred];
      lo[i] = pred - 1; hi[i] = pred;
      std::memcpy(&desc[(size_t)i * 32], descriptor_of(pMP).ptr(0), 32);
    }
    swm_best_query q;
    q.m = M; q.desc = desc.data(); q.u = u.data(); q.v = v.data(); q.radius = radius.data();
    q.min_level = lo.data(); q.max_level = hi.data(); q.valid = valid.data();
    q.inv_level_sigma2 = nullptr; q.nlevels = 0; q.chi2 = 0.0f;
    std::vector<int32_t> best_idx(M, -1), best_dist(M, 256);
    FlatFrame kf;
    gather(*pTgt, kf);
    swm_frame_view vk = kf.view();
    check(resident_of(*pTgt, 0) ? swm_window_best_resident(m_, resident_of(*pTgt, 0), &q, best_idx.data(), best_dist.data())
                                : swm_window_best(m_, &vk, &q, best_idx.data(), best_dist.data()));
    for (int i = 0; i < M; i++)
      if (valid[i] && best_idx[i] >= 0 && best_dist[i] <= TH_HIGH) match[i] = best_idx[i];  // :1125-1128
  }
  template <class MapPointT>
  static cv::Mat descriptor_of(MapPointT* p) { return p->GetDescriptor(); }
  // ---- cv::Mat arithmetic of the reference's projections, as OpenCV evaluates it for these shapes (pinned against
  // cv2 in tests/test_ref_orbmatcher.py::test_cv_shim_numerics_match_cv2, and against the reference's ORBmatcher.cc
  // compiled on a cv::Mat stand-in with the same rules in tests/ref_vs_product_test.cpp):
  //   R * x + t      (3x3 * 3x1, no transpose): cv::gemm's small-matrix path -- FLOAT products and sums, left to
  //                  right, then (float)(acc * alpha + t * beta) in double;
  //   -R.t() * t     (transposed operand): generic path, accumulation in DOUBLE, (float)(alpha * acc);
  //   Mat::dot, cv::norm: accumulation in double;  Mat * s, Mat / s: float product with (float)s resp. (float)(1.0 / s).
  template <class MatT>
  static void pose(const MatT& Tcw, float R[9], float t[3]) {
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 3; c++) R[3 * r + c] = Tcw.template at<float>(r, c);
      t[r] = Tcw.template at<float>(r, 3);
    }
  }
  // The frame's pose, camera and scale table as the tracking projections take them.
  template <class FrameT>
  static swm_projection projection(const FrameT& F) {
    swm_projection p;
    std::memset(&p, 0, sizeof(p));
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) p.Tcw[4 * r + c] = F.mTcw.template at<float>(r, c);
    p.fx = F.fx; p.fy = F.fy; p.cx = F.cx; p.cy = F.cy;
    p.scale_factors = F.mvScaleFactors.data();
    p.log_scale_factor = F.mfLogScaleFactor;
    p.nlevels = (int32_t)F.mvScaleFactors.size();
    return p;
  }
  template <class MatT>
  static void world_pos(const MatT& p, float x[3]) { for (int i = 0; i < 3; i++) x[i] = p.template at<float>(i); }
  static void transform(const float R[9], const float t[3], const float x[3], float out[3], double alpha = 1.0) {
    for (int r = 0; r < 3; r++) {
      float acc = fmul(R[3 * r], x[0]);
      acc = fadd(acc, fmul(R[3 * r + 1], x[1]));
      acc = fadd(acc, fmul(R[3 * r + 2], x[2]));
      out[r] = t ? (float)((double)acc * alpha + (double)t[r]) : (float)((double)acc * alpha);
    }
  }
  // volatile stores keep the compiler from contracting a * b + c into an FMA whatever -ffp-contract says
  static float fmul(float a, float b) { volatile float r = a * b; return r; }
  static float fadd(float a, float b) { volatile float r = a + b; return r; }
  static void centre(const float R[9], const float t[3], float Ow[3]) {  // -R.t() * t
    for (int c = 0; c < 3; c++)
      Ow[c] = (float)(-1.0 * ((double)R[c] * (double)t[0] + (double)R[3 + c] * (double)t[1] + (double)R[6 + c] * (double)t[2]));
  }
  static double dot3(const float a[3], const float b[3]) {
    return (double)a[0] * (double)b[0] + (double)a[1] * (double)b[1] + (double)a[2] * (double)b[2];
  }
  static float norm3(const float a[3]) { return (float)std::sqrt(dot3(a, a)); }
  // Decompose a Sim3 (:272-276, :899-903): scw = sqrt(row0 . row0), Rcw = sRcw / scw, tcw = Scw[0:3, 3] / scw
  template <class MatT>
  static void sim3_decompose(const MatT& Scw, float R[9], float t[3], float Ow[3]) {
    float sR[9], st[3];
    pose(Scw, sR, st);
    const float scw = (float)std::sqrt(dot3(sR, sR));
    const float inv = (float)(1.0 / (double)scw);
    for (int i = 0; i < 9; i++) R[i] = fmul(sR[i], inv);
    for (int i = 0; i < 3; i++) t[i] = fmul(st[i], inv);
    centre(R, t, Ow);
  }
  void check(int rc) {
    if (rc != SWM_OK) throw std::runtime_error(std::string("ORBmatcher: ") + swm_matcher_last_error(m_));
  }

  float mfNNratio;
  bool mbCheckOrientation;
  int device_;
  swm_matcher* m_ = nullptr;
};

}  // namespace ORB_SLAM2
