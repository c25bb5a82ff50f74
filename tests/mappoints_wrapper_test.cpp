// The C++ drop-ins for the two tracking projections from MapPoints resident on the GPU (host/MapPointTable.h and the
// MapPointTable overloads of ORBmatcher::SearchByProjection), on Frame / MapPoint doubles, against the host path: the
// reference's Tracking::SearchLocalPoints (Tracking.cc:964-1006) written as the reference writes it -- isInFrustum on
// the CPU (Frame.cc:316-375, cv::Mat arithmetic as DESIGN.md section 2 freezes it) and the host-array
// SearchByProjection(F, vpMapPoints, th) -- and the host-array SearchByProjection(cur, last, th, true).  The two runs
// start from identical copies of the scene; mvpMapPoints, nmatches, nToMatch and every MapPoint's mnVisible,
// mbTrackInView and tracking fields must come out the same.  Prints MAPPOINTS_WRAPPER_OK.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "../swarmmap_b200/host/ORBmatcher.h"

using namespace ORB_SLAM2;

struct Mat4 {  // stand-in for the CV_32F cv::Mat pose / 3-vectors
  float v[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  template <typename T> T at(int r, int c) const { return v[r * 4 + c]; }
  template <typename T> T at(int i) const { return v[i]; }
};

struct MapPoint {
  Mat4 pos, normal;
  float mind = 0, maxd = 0;
  cv::Mat desc;
  int nobs = 1;
  bool bad = false;
  bool mbTrackInView = false;
  float mTrackProjX = 0, mTrackProjY = 0, mTrackViewCos = 0;
  int mnTrackScaleLevel = 0;
  long unsigned int mnLastFrameSeen = 0;
  int mnVisible = 1;
  Mat4 GetWorldPos() { return pos; }
  Mat4 GetNormal() { return normal; }
  float GetMinDistance() { return mind; }
  float GetMaxDistance() { return maxd; }
  float GetMinDistanceInvariance() { return 0.8f * mind; }
  float GetMaxDistanceInvariance() { return 1.2f * maxd; }
  cv::Mat GetDescriptor() { return desc; }
  int Observations() { return nobs; }
  bool isBad() { return bad; }
  void IncreaseVisible(int n = 1) { mnVisible += n; }
  int PredictScale(const float& currentDist, const float& logScaleFactor, const int nLevels) {  // MapPoint.cc:476-485
    const float ratio = maxd / currentDist;
    int nScale = (int)std::ceil(std::log(ratio) / logScaleFactor);
    if (nScale < 0) nScale = 0;
    else if (nScale >= nLevels) nScale = nLevels - 1;
    return nScale;
  }
};

static float fmul(float a, float b) { volatile float r = a * b; return r; }
static float fadd(float a, float b) { volatile float r = a + b; return r; }

struct Frame {
  int N = 0;
  long unsigned int mnId = 7;
  std::vector<cv::KeyPoint> mvKeys, mvKeysUn;
  cv::Mat mDescriptors;
  std::vector<MapPoint*> mvpMapPoints;
  std::vector<bool> mvbOutlier;
  Mat4 mTcw;
  float fx = 458.654f, fy = 457.296f, cx = 367.215f, cy = 248.375f;
  float mnMinX = 0, mnMinY = 0, mnMaxX = 752, mnMaxY = 480;
  float mfLogScaleFactor = 0;
  int mnScaleLevels = 8;
  std::vector<float> mvScaleFactors;
  const swm_frame* mpResident = nullptr;

  // Frame::isInFrustum, Frame.cc:316-375 (gemm small path in float, Ow / norm / dot in double)
  bool isInFrustum(MapPoint* pMP, float viewingCosLimit) {
    pMP->mbTrackInView = false;
    const float* P = pMP->pos.v;
    float Pc[3];
    for (int r = 0; r < 3; r++) {
      float acc = fmul(mTcw.v[4 * r], P[0]);
      acc = fadd(acc, fmul(mTcw.v[4 * r + 1], P[1]));
      acc = fadd(acc, fmul(mTcw.v[4 * r + 2], P[2]));
      Pc[r] = fadd(acc, mTcw.v[4 * r + 3]);
    }
    if (Pc[2] < 0.0f) return false;
    const float invz = 1.0f / Pc[2];
    const float u = fadd(fmul(fmul(fx, Pc[0]), invz), cx);
    const float v = fadd(fmul(fmul(fy, Pc[1]), invz), cy);
    if (u < mnMinX || u > mnMaxX) return false;
    if (v < mnMinY || v > mnMaxY) return false;
    const float maxDistance = pMP->GetMaxDistanceInvariance(), minDistance = pMP->GetMinDistanceInvariance();
    float Ow[3], PO[3];
    for (int c = 0; c < 3; c++) {
      double acc = 0.0;
      for (int k = 0; k < 3; k++) acc += (double)mTcw.v[4 * k + c] * (double)mTcw.v[4 * k + 3];
      Ow[c] = (float)(-1.0 * acc);
      PO[c] = P[c] - Ow[c];
    }
    double s = 0.0, dot = 0.0;
    for (int k = 0; k < 3; k++) s += (double)PO[k] * (double)PO[k];
    const float dist = (float)std::sqrt(s);
    if (dist < minDistance || dist > maxDistance) return false;
    for (int k = 0; k < 3; k++) dot += (double)PO[k] * (double)pMP->normal.v[k];
    const float viewCos = (float)(dot / (double)dist);
    if (viewCos < viewingCosLimit) return false;
    const int nPredictedLevel = pMP->PredictScale(dist, mfLogScaleFactor, mnScaleLevels);
    pMP->mbTrackInView = true;
    pMP->mTrackProjX = u;
    pMP->mTrackProjY = v;
    pMP->mnTrackScaleLevel = nPredictedLevel;
    pMP->mTrackViewCos = viewCos;
    return true;
  }
};

static int fails = 0;
#define EXPECT(c)                                                                   \
  do {                                                                              \
    if (!(c)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); fails++; } \
  } while (0)

static std::mt19937 rng(11);
static float uni(float a, float b) { return std::uniform_real_distribution<float>(a, b)(rng); }

struct Scene {
  std::vector<MapPoint> pts;
  Frame F, last;
  std::vector<int> list;  // local map, indices into pts (with duplicates)
};

// A local map seen from a camera and a frame whose keypoints are noisy projections of 60 % of the points in view.
static Scene make_scene(int npts) {
  Scene S;
  Frame& F = S.F;
  F.mvScaleFactors.resize(8);
  F.mvScaleFactors[0] = 1.0f;
  for (int i = 1; i < 8; i++) F.mvScaleFactors[i] = F.mvScaleFactors[i - 1] * 1.2f;
  F.mfLogScaleFactor = std::log(1.2f);
  const float a = 0.03f;  // small rotation about y, translation
  F.mTcw.v[0] = std::cos(a); F.mTcw.v[2] = std::sin(a); F.mTcw.v[8] = -std::sin(a); F.mTcw.v[10] = std::cos(a);
  F.mTcw.v[3] = 0.1f; F.mTcw.v[7] = -0.05f; F.mTcw.v[11] = 0.2f;
  S.pts.resize(npts);
  for (int i = 0; i < npts; i++) {
    MapPoint& p = S.pts[i];
    const double z = uni(0.5f, 20.f) * (uni(0, 1) < 0.05f ? -1 : 1);
    const double px = uni(-60, 812), py = uni(-60, 540);
    const double pc[3] = {(px - F.cx) / F.fx * z, (py - F.cy) / F.fy * z, z};
    double d[3];
    for (int c = 0; c < 3; c++) d[c] = pc[c] - F.mTcw.v[4 * c + 3];
    for (int c = 0; c < 3; c++) p.pos.v[c] = (float)(F.mTcw.v[c] * d[0] + F.mTcw.v[4 + c] * d[1] + F.mTcw.v[8 + c] * d[2]);
    const double dist = std::sqrt(pc[0] * pc[0] + pc[1] * pc[1] + pc[2] * pc[2]);
    double n[3] = {p.pos.v[0] + uni(-0.6f, 0.6f) * dist, p.pos.v[1] + uni(-0.6f, 0.6f) * dist, p.pos.v[2] + uni(-0.6f, 0.6f) * dist};
    const double nn = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    for (int c = 0; c < 3; c++) p.normal.v[c] = (float)(n[c] / nn);
    p.maxd = (float)(dist * uni(0.7f, 6.f));
    p.mind = p.maxd / uni(2.f, 30.f);
    p.desc = cv::Mat(1, 32, 0);
    for (int k = 0; k < 32; k++) p.desc.ptr(0)[k] = (uint8_t)(rng() & 255);
    p.nobs = uni(0, 1) < 0.9f ? 2 : 0;
    p.bad = uni(0, 1) < 0.03f;
  }
  // keypoints: projections of in-view points (level = predicted level), plus unrelated ones
  std::vector<int> owner;
  for (int i = 0; i < npts; i++) {
    MapPoint probe = S.pts[i];
    if (!F.isInFrustum(&probe, 0.5f) || uni(0, 1) > 0.6f) continue;
    cv::KeyPoint kp;
    kp.pt.x = std::min(std::max(probe.mTrackProjX + uni(-1, 1), 0.f), 751.9f);
    kp.pt.y = std::min(std::max(probe.mTrackProjY + uni(-1, 1), 0.f), 479.9f);
    kp.octave = probe.mnTrackScaleLevel;
    kp.angle = uni(0, 360);
    F.mvKeysUn.push_back(kp);
    owner.push_back(i);
  }
  for (int k = 0; k < 300; k++) {
    cv::KeyPoint kp;
    kp.pt.x = uni(0, 751.9f); kp.pt.y = uni(0, 479.9f); kp.octave = (int)(rng() % 8); kp.angle = uni(0, 360);
    F.mvKeysUn.push_back(kp);
    owner.push_back(-1);
  }
  F.N = (int)F.mvKeysUn.size();
  F.mvKeys = F.mvKeysUn;
  F.mDescriptors = cv::Mat(F.N, 32, 0);
  for (int j = 0; j < F.N; j++) {
    uint8_t* d = F.mDescriptors.ptr(j);
    for (int k = 0; k < 32; k++) d[k] = owner[j] >= 0 ? S.pts[owner[j]].desc.ptr(0)[k] : (uint8_t)(rng() & 255);
    if (owner[j] >= 0) d[rng() % 32] ^= (uint8_t)(1u << (rng() % 8));
  }
  F.mvpMapPoints.assign(F.N, nullptr);
  F.mvbOutlier.assign(F.N, false);
  for (int j = 0; j < F.N; j++)
    if (owner[j] >= 0 && uni(0, 1) < 0.15f) F.mvpMapPoints[j] = &S.pts[owner[j]];
  for (int i = 0; i < npts; i++) S.list.push_back(i);
  std::shuffle(S.list.begin(), S.list.end(), rng);
  for (int k = 0; k < 40; k++) S.list.push_back(S.list[k]);  // duplicates: IncreaseVisible twice, list order kept
  // the last frame: the same keypoints moved a little, holding their points (some outliers); the current frame empty
  S.last = F;
  for (auto& kp : S.last.mvKeysUn) { kp.pt.x = std::min(kp.pt.x + 1.5f, 751.9f); kp.pt.y = std::max(kp.pt.y - 0.5f, 0.f); }
  S.last.mvKeys = S.last.mvKeysUn;
  for (int j = 0; j < F.N; j++) {
    S.last.mvpMapPoints[j] = owner[j] >= 0 && uni(0, 1) < 0.9f ? &S.pts[owner[j]] : nullptr;
    S.last.mvbOutlier[j] = uni(0, 1) < 0.05f;
  }
  return S;
}

// Re-points a copy of the scene's frames at the copy's own points.
static void rebase(Scene& dst, const Scene& src) {
  for (Frame* f : {&dst.F, &dst.last})
    for (auto& p : f->mvpMapPoints)
      if (p) p = &dst.pts[p - &src.pts[0]];
}

static swm_frame* upload(const Frame& F) {
  swm_frame* f = nullptr;
  if (swm_frame_create(0, &f) != SWM_OK) return nullptr;
  std::vector<float> x(F.N), y(F.N), ang(F.N);
  std::vector<int32_t> oct(F.N);
  for (int j = 0; j < F.N; j++) { x[j] = F.mvKeysUn[j].pt.x; y[j] = F.mvKeysUn[j].pt.y; ang[j] = F.mvKeysUn[j].angle; oct[j] = F.mvKeysUn[j].octave; }
  swm_frame_view v;
  v.n = F.N; v.x = x.data(); v.y = y.data(); v.octave = oct.data(); v.angle = ang.data(); v.desc = F.mDescriptors.ptr(0);
  v.min_x = F.mnMinX; v.min_y = F.mnMinY; v.max_x = F.mnMaxX; v.max_y = F.mnMaxY;
  if (swm_frame_upload(f, &v) != SWM_OK) { swm_frame_destroy(f); return nullptr; }
  return f;
}

static void compare_points(const Scene& a, const Scene& b) {
  int diff = 0;
  for (size_t i = 0; i < a.pts.size(); i++) {
    const MapPoint &p = a.pts[i], &q = b.pts[i];
    bool same = p.mnVisible == q.mnVisible && p.mbTrackInView == q.mbTrackInView;
    if (p.mbTrackInView && q.mbTrackInView)
      same = same && !std::memcmp(&p.mTrackProjX, &q.mTrackProjX, 4) && !std::memcmp(&p.mTrackProjY, &q.mTrackProjY, 4) &&
             !std::memcmp(&p.mTrackViewCos, &q.mTrackViewCos, 4) && p.mnTrackScaleLevel == q.mnTrackScaleLevel;
    diff += !same;
  }
  EXPECT(diff == 0);
}

static void compare_frames(const Frame& a, const Scene& sa, const Frame& b, const Scene& sb) {
  int diff = 0;
  for (int j = 0; j < a.N; j++) {
    const long ia = a.mvpMapPoints[j] ? a.mvpMapPoints[j] - &sa.pts[0] : -1;
    const long ib = b.mvpMapPoints[j] ? b.mvpMapPoints[j] - &sb.pts[0] : -1;
    diff += ia != ib;
  }
  EXPECT(diff == 0);
}

int main() {
  ORBmatcher matcher(0.8f, true);
  for (float th : {1.0f, 3.0f}) {
    Scene host = make_scene(2000);
    Scene gpu = host;
    rebase(gpu, host);
    // host path: Tracking::SearchLocalPoints as the reference writes it
    int nToMatch = 0;
    for (auto& pMP : host.F.mvpMapPoints) {
      if (!pMP) continue;
      if (pMP->isBad()) { pMP = nullptr; continue; }
      pMP->IncreaseVisible();
      pMP->mnLastFrameSeen = host.F.mnId;
      pMP->mbTrackInView = false;
    }
    std::vector<MapPoint*> vh, vg;
    for (int i : host.list) vh.push_back(&host.pts[i]);
    for (int i : gpu.list) vg.push_back(&gpu.pts[i]);
    for (MapPoint* pMP : vh) {
      if (pMP->mnLastFrameSeen == host.F.mnId || pMP->isBad()) continue;
      if (host.F.isInFrustum(pMP, 0.5f)) { pMP->IncreaseVisible(); nToMatch++; }
    }
    const int n_host = nToMatch > 0 ? matcher.SearchByProjection(host.F, vh, th) : 0;
    // GPU path: the table and one call
    MapPointTable<MapPoint> table(0, 16);  // grows while the points are written
    std::vector<MapPoint*> all;
    for (auto& p : gpu.pts) all.push_back(&p);
    table.Upsert(all);
    swm_frame* rf = upload(gpu.F);
    EXPECT(rf != nullptr);
    gpu.F.mpResident = rf;
    int ntm_gpu = -1;
    const int n_gpu = matcher.SearchByProjection(gpu.F, vg, th, table, &ntm_gpu);
    std::printf("local map th %.0f: %d matches, %d in view\n", th, n_gpu, ntm_gpu);
    EXPECT(n_host == n_gpu && nToMatch == ntm_gpu && n_gpu > 100);
    compare_frames(host.F, host, gpu.F, gpu);
    compare_points(host, gpu);

    // SearchByProjection(cur, last, 15, true): the current frame starts empty (Tracking.cc:715-737)
    Frame hc = host.F, gc = gpu.F;
    hc.mvpMapPoints.assign(hc.N, nullptr);
    gc.mvpMapPoints.assign(gc.N, nullptr);
    hc.mpResident = nullptr;
    swm_frame* rl = upload(gpu.last);
    gpu.last.mpResident = rl;
    const int l_host = matcher.SearchByProjection(hc, host.last, 15.0f, true);
    const int l_gpu = matcher.SearchByProjection(gc, gpu.last, 15.0f, true, table);
    std::printf("last frame: %d matches\n", l_gpu);
    EXPECT(l_host == l_gpu && l_gpu > 100);
    compare_frames(hc, host, gc, gpu);
    // Erase returns the row; a new point reuses it
    MapPoint* gone = &gpu.pts[0];
    const int32_t r = table.Row(gone);
    table.Erase(gone);
    EXPECT(table.Row(gone) == -1);
    table.Upsert({&gpu.pts[0]});
    EXPECT(table.Row(&gpu.pts[0]) == r);
    swm_frame_destroy(rf);
    swm_frame_destroy(rl);
  }
  if (fails) return 1;
  std::printf("MAPPOINTS_WRAPPER_OK\n");
  return 0;
}
