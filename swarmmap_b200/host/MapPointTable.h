// MapPointTable.h -- MapPoints resident on the GPU (swm_mappoints_*, include/swm_orb.h) for the two per-frame tracking
// projections: ORBmatcher::SearchByProjection(F, vpMapPoints, th, table) (Tracking::SearchLocalPoints) and
// SearchByProjection(CurrentFrame, LastFrame, th, bMono, table).  The table maps MapPoint* to a row; rows of erased
// points go to a free list.  A template over the MapPoint type: it reads GetWorldPos(), GetNormal(), GetMinDistance(),
// GetMaxDistance() (the two getters INTEGRATION.md adds to MapPoint.h), GetDescriptor(), Observations() and isBad().
//
// Where SwarmMap changes a point, Upsert it again (INTEGRATION.md section 9): LocalMapping::CreateNewMapPoints,
// SearchInNeighbors, after LocalBundleAdjustment, UpdateNormalAndDepth, ComputeDistinctiveDescriptors, MapPointCulling /
// SetBadFlag.  Erase a point only once no frame refers to it: the last-frame projection projects a point whatever its
// bad flag, as the reference does, so its row must not stand in for another point before then.
#pragma once
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/swm_orb.h"

namespace ORB_SLAM2 {

template <class MapPointT>
class MapPointTable {
 public:
  explicit MapPointTable(int device = 0, int capacity = 0) {
    if (swm_mappoints_create(device, capacity, &t_) != SWM_OK)
      throw std::runtime_error(std::string("MapPointTable: ") + swm_mappoints_last_error(nullptr));
  }
  ~MapPointTable() { swm_mappoints_destroy(t_); }
  MapPointTable(const MapPointTable&) = delete;
  MapPointTable& operator=(const MapPointTable&) = delete;

  swm_mappoints* get() const { return t_; }

  // The point's row, or -1 when it is not in the table.
  int32_t Row(MapPointT* p) const {
    auto it = row_.find(p);
    return it == row_.end() ? -1 : it->second;
  }

  // Writes the current state of every point (new points get a row) in one upload.
  void Upsert(const std::vector<MapPointT*>& points) {
    const size_t n = points.size();
    if (n == 0) return;
    std::vector<int32_t> rows(n);
    std::vector<float> pos(3 * n), normal(3 * n), mind(n), maxd(n);
    std::vector<uint8_t> desc(32 * n), obs(n), bad(n);
    for (size_t i = 0; i < n; i++) {
      MapPointT* p = points[i];
      rows[i] = RowFor(p);
      const auto P = p->GetWorldPos();
      const auto N = p->GetNormal();
      for (int c = 0; c < 3; c++) {
        pos[3 * i + c] = P.template at<float>(c);
        normal[3 * i + c] = N.template at<float>(c);
      }
      mind[i] = p->GetMinDistance();
      maxd[i] = p->GetMaxDistance();
      std::memcpy(&desc[32 * i], p->GetDescriptor().ptr(0), 32);
      obs[i] = p->Observations() > 0;
      bad[i] = p->isBad();
    }
    check(swm_mappoints_upsert(t_, (int)n, rows.data(), pos.data(), normal.data(), mind.data(), maxd.data(), desc.data(),
                               obs.data(), bad.data()));
  }

  // Marks the point's row bad and returns it to the free list.
  void Erase(MapPointT* p) {
    auto it = row_.find(p);
    if (it == row_.end()) return;
    const int32_t r = it->second;
    const float zero3[3] = {0, 0, 0}, zero = 0;
    const uint8_t zdesc[32] = {0}, no = 0, yes = 1;
    check(swm_mappoints_upsert(t_, 1, &r, zero3, zero3, &zero, &zero, zdesc, &no, &yes));
    row_.erase(it);
    free_.push_back(r);
  }

 private:
  int32_t RowFor(MapPointT* p) {
    auto it = row_.find(p);
    if (it != row_.end()) return it->second;
    int32_t r;
    if (!free_.empty()) {
      r = free_.back();
      free_.pop_back();
    } else {
      r = next_++;
    }
    row_.emplace(p, r);
    return r;
  }
  void check(int rc) {
    if (rc != SWM_OK) throw std::runtime_error(std::string("MapPointTable: ") + swm_mappoints_last_error(t_));
  }

  swm_mappoints* t_ = nullptr;
  std::unordered_map<MapPointT*, int32_t> row_;
  std::vector<int32_t> free_;
  int32_t next_ = 0;
};

}  // namespace ORB_SLAM2
