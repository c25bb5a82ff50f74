// orb_oracle_frustum.cpp -- CPU ORACLE of Frame::isInFrustum (Frame.cc:316-375), MapPoint::PredictScale
// (MapPoint.cc:476-485) and the projection step of SearchByProjection(Frame&, const Frame&, th, bMono)
// (ORBmatcher.cc:1247-1268), on flat arrays.  TEST INFRASTRUCTURE ONLY (see orb_oracle.h); built as a library of its
// own (tests/oracle_frustum_lib.py) so that the matcher oracle is unchanged.  Paths relative to /root/reference/code/.
//
// cv::Mat arithmetic as DESIGN.md section 2 freezes it (compiled with -ffp-contract=off, so nothing is fused):
//   Pc = Rcw * P + tcw   cv::gemm's small-matrix path: float products and sums, left to right, then
//                        (float)(acc * 1.0 + t) in double, which is the float sum acc + t;
//   Ow = -Rcw.t() * tcw  generic path: products and sums in double, left to right, then (float)(-1.0 * acc);
//   cv::norm(PO)         squares summed in double, sqrt, then float;
//   PO.dot(Pn)           products and sums in double.
// `log` of a float is std::log(float) (logf): the reference's headers leak `using namespace std`.
#include <cmath>
#include <cstdint>

namespace {

float gemm_row(const float* T, int r, const float* x) {
  float acc = T[4 * r] * x[0];
  acc = acc + T[4 * r + 1] * x[1];
  acc = acc + T[4 * r + 2] * x[2];
  return (float)((double)acc * 1.0 + (double)T[4 * r + 3]);
}

// Rows of the 3x4 pose (row-major, Tcw rows 0..2) to the camera centre Ow = -Rcw.t() * tcw (Frame::UpdatePoseMatrices).
void centre(const float* T, float* Ow) {
  for (int c = 0; c < 3; c++) {
    double acc = 0.0;
    for (int k = 0; k < 3; k++) acc += (double)T[4 * k + c] * (double)T[4 * k + 3];
    Ow[c] = (float)(-1.0 * acc);
  }
}

}  // namespace

extern "C" {

// MapPoint::PredictScale, MapPoint.cc:476-485: ratio = mfMaxDistance / currentDist (float), nScale =
// ceil(log(ratio) / logScaleFactor) in float, clamped to [0, nScaleLevels - 1].  The reference converts the float to
// int first, which is undefined for a non-finite quotient; here +inf gives the top level and NaN gives level 0.
int orc_predict_scale(float max_distance, float current_dist, float log_scale_factor, int nlevels) {
  const float ratio = max_distance / current_dist;
  const float q = std::ceil(std::log(ratio) / log_scale_factor);
  if (std::isnan(q)) return 0;
  if (q < 0.0f) return 0;
  if (q >= (float)nlevels) return nlevels - 1;
  return (int)q;
}

void orc_predict_scale_many(int n, const float* max_distance, const float* current_dist, float log_scale_factor,
                            int nlevels, int32_t* out) {
  for (int i = 0; i < n; i++) out[i] = orc_predict_scale(max_distance[i], current_dist[i], log_scale_factor, nlevels);
}

// Frame::isInFrustum(pMP, viewingCosLimit), Frame.cc:316-375, for n points.  T: mTcw rows 0..2 (12 floats,
// row-major); bounds4: mnMinX, mnMaxX, mnMinY, mnMaxY.  Outputs are written for every point; u, v, view_cos and level
// hold the tracking fields only where in_view = 1 and are 0 elsewhere.
void orc_is_in_frustum(const float* T, float fx, float fy, float cx, float cy, const float* bounds4, int n,
                       const float* pos, const float* normal, const float* min_d, const float* max_d,
                       float viewing_cos_limit, float log_scale_factor, int nlevels, uint8_t* in_view, float* u_out,
                       float* v_out, float* view_cos, int32_t* level) {
  float Ow[3];
  centre(T, Ow);
  for (int i = 0; i < n; i++) {
    in_view[i] = 0;
    u_out[i] = v_out[i] = view_cos[i] = 0.0f;
    level[i] = 0;
    const float* P = pos + 3 * i;
    const float PcX = gemm_row(T, 0, P), PcY = gemm_row(T, 1, P), PcZ = gemm_row(T, 2, P);
    if (PcZ < 0.0f) continue;                                           // :327-328
    const float invz = 1.0f / PcZ;                                      // :331
    const float u = fx * PcX * invz + cx;                               // :332-333
    const float v = fy * PcY * invz + cy;
    if (u < bounds4[0] || u > bounds4[1]) continue;                     // :335-338
    if (v < bounds4[2] || v > bounds4[3]) continue;
    const float maxDistance = 1.2f * max_d[i];                          // GetMaxDistanceInvariance, MapPoint.cc:472-474
    const float minDistance = 0.8f * min_d[i];                          // GetMinDistanceInvariance, :466-470
    const float PO[3] = {P[0] - Ow[0], P[1] - Ow[1], P[2] - Ow[2]};
    double s = 0.0;
    for (int k = 0; k < 3; k++) s += (double)PO[k] * (double)PO[k];
    const float dist = (float)std::sqrt(s);                             // cv::norm, :344
    if (dist < minDistance || dist > maxDistance) continue;             // :346-347
    const float* Pn = normal + 3 * i;
    double dot = 0.0;
    for (int k = 0; k < 3; k++) dot += (double)PO[k] * (double)Pn[k];
    const float viewCos = (float)(dot / (double)dist);                  // :351
    if (viewCos < viewing_cos_limit) continue;                          // :353-354
    level[i] = orc_predict_scale(max_d[i], dist, log_scale_factor, nlevels);  // :357
    in_view[i] = 1;                                                     // :360-367
    u_out[i] = u;
    v_out[i] = v;
    view_cos[i] = viewCos;
  }
}

// The projection of SearchByProjection(CurrentFrame, LastFrame, th, bMono = true), ORBmatcher.cc:1252-1268, for n
// world points: invzc = 1.0 / z in double, then float; valid = invzc >= 0 and (u, v) inside the bounds.
void orc_project_last(const float* T, float fx, float fy, float cx, float cy, const float* bounds4, int n,
                      const float* pos, uint8_t* valid, float* u_out, float* v_out) {
  for (int i = 0; i < n; i++) {
    valid[i] = 0;
    u_out[i] = v_out[i] = 0.0f;
    const float* P = pos + 3 * i;
    const float xc = gemm_row(T, 0, P), yc = gemm_row(T, 1, P), zc = gemm_row(T, 2, P);
    const float invzc = 1.0 / zc;                                       // :1257
    if (invzc < 0) continue;                                            // :1259-1260
    const float u = fx * xc * invzc + cx;                               // :1262-1263
    const float v = fy * yc * invzc + cy;
    if (u < bounds4[0] || u > bounds4[1]) continue;                     // :1265-1268
    if (v < bounds4[2] || v > bounds4[3]) continue;
    valid[i] = 1;
    u_out[i] = u;
    v_out[i] = v;
  }
}

}  // extern "C"
