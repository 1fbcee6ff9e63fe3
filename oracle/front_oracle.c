/* ORACLE (test infrastructure - never linked into, or called by, the product library).
 *
 * Plain-C restatement of the two host-side stages either side of the level-0 tracker that SURVEY.md section 8(f)
 * ranks "next" (n2, n1):
 *   make_images      FrameHessian::makeImages            tandem/src/FullSystem/HessianBlocks.cpp:128-191
 *                    (grey pyramid by 2x2 means, central-difference gradients over the FLAT index range
 *                    [w, w*(h-1)), non-finite gradients -> 0; absSquaredGrad without the gamma weighting, which
 *                    needs the photometric calibration object and is not consumed by the tracker)
 *   dense_reference  CoarseTracker::setCoarseTrackingRef tandem/src/FullSystem/CoarseTracker.cpp:655-732
 *                    (forward-warp of the rendered dense depth into the reference keyframe with a nearest-depth
 *                    test, then raster-order append behind the sparse points, INCLUDING the pre-increment quirk of
 *                    :717-722: slot n_before keeps its stale content and the last appended point is not counted)
 * PINNED (round 2): the reference ships no test or golden for either function and CoarseTracker.cpp / HessianBlocks.cpp
 * as a whole need Eigen + Sophus (absent from the build container), but the two function BODIES only touch Eigen as
 * 3-vectors / 3x3 matrices.  oracle/ref_build.mk cuts them out of the files where they lie (HessianBlocks.cpp:128-191,
 * CoarseTracker.cpp:655-725) and compiles them, unmodified, against a stand-in Eigen (tests/cpp/eigen_stub) and the harness
 * oracle/ref_wrap_front.cpp into oracle/_ref/libfront_ref.so; tests/test_oracle_cpu.py::test_front_oracle_*_pinned_* compare
 * this restatement with that library bit for bit (pyramid incl. a non-finite pixel; pc_n and all four point arrays for
 * steps 1-3, with and without sparse points, up to 640x480); what that library returned is stored in
 * tests/golden/ref_front.npz (oracle/ref_golden.py), so the tests run without the reference.  Deliberate, documented deviations:
 *   * rows 0 and h-1 of (dx, dy, absSquaredGrad) are uninitialised memory in the reference (`new Eigen::Vector3f[]`);
 *     here they are 0.  The tracker never reads them (2 < Kv < h-3).
 *   * a warped depth <= 0 (point behind the reference camera) is ignored; in the reference its effect depends on the
 *     raster order of later arrivals at the same pixel (CoarseTracker.cpp:699-703).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* dI: levels concatenated, level l holds wl*hl float3 (I,dx,dy); wl = w >> l, hl = h >> l (globalCalib.cpp:62-66).
 * absgrad: levels concatenated, wl*hl floats. */
void front_oracle_make_images(const float* color, int w, int h, int levels, float* dI, float* absgrad) {
  size_t off = 0, off_prev = 0;
  int wprev = 0;
  for (int lvl = 0; lvl < levels; ++lvl) {
    const int wl = w >> lvl, hl = h >> lvl;
    float* d = dI + 3 * off;
    float* a = absgrad + off;
    memset(d, 0, sizeof(float) * 3 * (size_t)wl * hl);
    memset(a, 0, sizeof(float) * (size_t)wl * hl);
    if (lvl == 0) {
      for (int i = 0; i < wl * hl; ++i) d[3 * i] = color[i];
    } else {
      const float* p = dI + 3 * off_prev;
      for (int y = 0; y < hl; ++y)
        for (int x = 0; x < wl; ++x)
          d[3 * (x + y * wl)] = 0.25f * (p[3 * (2 * x + 2 * y * wprev)] + p[3 * (2 * x + 1 + 2 * y * wprev)] +
                                         p[3 * (2 * x + 2 * y * wprev + wprev)] + p[3 * (2 * x + 1 + 2 * y * wprev + wprev)]);
    }
    for (int idx = wl; idx < wl * (hl - 1); ++idx) {
      float dx = 0.5f * (d[3 * (idx + 1)] - d[3 * (idx - 1)]);
      float dy = 0.5f * (d[3 * (idx + wl)] - d[3 * (idx - wl)]);
      if (!isfinite(dx)) dx = 0;
      if (!isfinite(dy)) dy = 0;
      d[3 * idx + 1] = dx;
      d[3 * idx + 2] = dy;
      a[idx] = dx * dx + dy * dy;
    }
    off_prev = off;
    wprev = wl;
    off += (size_t)wl * hl;
  }
}

/* KRKi = (K * R) * Ki and Kt = K * t in float, products accumulated k = 0,1,2 (CoarseTracker.cpp:676-677).
 * T is the 4x4 row-major double transform depth-frame -> reference keyframe. */
void front_oracle_krki(const double* T, float fx, float fy, float cx, float cy, float KRKi[9], float Kt[3]) {
  const float K[9] = {fx, 0, cx, 0, fy, cy, 0, 0, 1};
  const float Ki[9] = {1.0f / fx, 0, -cx / fx, 0, 1.0f / fy, -cy / fy, 0, 0, 1};
  float R[9], t[3], KR[9];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) R[3 * r + c] = (float)T[4 * r + c];
    t[r] = (float)T[4 * r + 3];
  }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      float s = 0;
      for (int k = 0; k < 3; ++k) s += K[3 * r + k] * R[3 * k + c];
      KR[3 * r + c] = s;
    }
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) {
      float s = 0;
      for (int k = 0; k < 3; ++k) s += KR[3 * r + k] * Ki[3 * k + c];
      KRKi[3 * r + c] = s;
    }
    float s = 0;
    for (int k = 0; k < 3; ++k) s += K[3 * r + k] * t[k];
    Kt[r] = s;
  }
}

/* pc_* : capacity >= n_before + 1 + (w*h); entries [0, n_before] are inputs (slot n_before = the stale slot).
 * idepth0 may be NULL (treated as all <= 0).  Returns the new pc_n. proj (w*h floats, -1 = invalid) is an output for
 * inspection. */
int front_oracle_dense_reference(const float* depth, int w, int h, int step, const float KRKi[9], const float Kt[3],
                                 int dense_only, int n_before, const float* idepth0, const float* ref_gray,
                                 float* pc_u, float* pc_v, float* pc_idepth, float* pc_color, float* proj) {
  for (int i = 0; i < w * h; ++i) proj[i] = -1.f;
  for (int y = 0; y < h; y += step)
    for (int x = 0; x < w; x += step) {
      const size_t i = (size_t)x + (size_t)y * w;
      const float z = depth[i];
      if (z <= 0.f) continue;
      const float ox = x * z, oy = y * z;
      float p[3];
      for (int r = 0; r < 3; ++r) p[r] = (KRKi[3 * r] * ox + KRKi[3 * r + 1] * oy + KRKi[3 * r + 2] * z) + Kt[r];
      if (!(p[2] > 0.f)) continue;                       /* documented deviation, see header */
      const int pu = (int)(p[0] / p[2] + 0.5f), pv = (int)(p[1] / p[2] + 0.5f);
      if (pu > w - 4 || pv > h - 4 || pu < 3 || pv < 3) continue;
      float* q = proj + pu + (size_t)pv * w;
      if (*q < 0 || p[2] < *q) *q = p[2];
    }
  int n = n_before;
  for (int y = 2; y < h - 2; ++y)
    for (int x = 2; x < w - 2; ++x) {
      const int i = x + y * w;
      const float d = proj[i];
      if (d <= 0) continue;
      if (dense_only || !idepth0 || idepth0[i] <= 0) {
        ++n;
        pc_u[n] = (float)x;
        pc_v[n] = (float)y;
        pc_idepth[n] = 1.f / d;
        pc_color[n] = ref_gray[i];
      }
    }
  return n;
}
