// ilsm::IterativeClosestPoint (include/ilsm.hpp) against the C ABI it wraps: the same pair through both must give the
// same bytes.  Exit codes: 0 pass, 1 mismatch, 100 ilsm::Error (ILSM_ERR_NO_DEVICE without a GPU, printed as -3).
#include <cstdio>
#include <cstring>

#include "ilsm.hpp"

namespace {
unsigned g_seed = 12345u;
float frand(float lo, float hi) {  // seeded LCG: the same clouds on every machine
  g_seed = g_seed * 1664525u + 1013904223u;
  return lo + (hi - lo) * (float)((g_seed >> 8) & 0xFFFFFF) / 16777216.0f;
}
}  // namespace

int main() {
  try {
    ilsm::PointCloud<ilsm::PointXYZI> target, source, out;
    for (int i = 0; i < 6000; ++i) {  // three walls and a floor
      ilsm::PointXYZI p;
      const int face = i % 4;
      const float a = frand(-8.f, 8.f), b = frand(0.f, 4.f);
      p.x = face == 0 ? -8.f : face == 1 ? 8.f : a;
      p.y = face == 2 ? 6.f : face == 3 ? frand(-6.f, 6.f) : a * 0.75f;
      p.z = face == 3 ? 0.f : b;
      target.push_back(p);
    }
    const float c = 0.9950042f, s = 0.0998334f;  // yaw 0.1 rad, shift (0.4, -0.3, 0.05): source = T^-1 target
    for (size_t i = 0; i < target.size(); i += 3) {
      const ilsm::PointXYZI& t = target.points[i];
      ilsm::PointXYZI p;
      const float x = t.x - 0.4f, y = t.y + 0.3f;
      p.x = c * x + s * y, p.y = -s * x + c * y, p.z = t.z - 0.05f;
      source.push_back(p);
    }
    ilsm::Matrix4f guess;
    guess(0, 0) = 0.9987503f, guess(0, 1) = -0.0499792f, guess(1, 0) = 0.0499792f, guess(1, 1) = 0.9987503f;  // yaw 0.05
    guess(0, 3) = 0.3f, guess(1, 3) = -0.2f;

    ilsm::IterativeClosestPoint<ilsm::PointXYZI, ilsm::PointXYZI> icp;
    icp.setMaxCorrespondenceDistance(2.0);
    icp.setMaximumIterations(30);
    icp.setTransformationEpsilon(1e-10);
    icp.setEuclideanFitnessEpsilon(1e-8);
    icp.setRANSACIterations(0);
    icp.setInputSource(source);
    icp.setInputTarget(target);
    icp.align(out, guess);

    // the same pair through the C ABI
    ilsm::ContextPtr ctx = ilsm::Context::shared();
    ilsm_map* map = nullptr;
    ilsm::check(ilsm_map_create(ctx->get(), &map), "ilsm_map_create");
    ilsm::check(ilsm_map_build(map, ilsm::cloud_ptr(target), (int)target.size(), 32, 0.f), "ilsm_map_build");
    ilsm_icp_opts o;
    ilsm_icp_opts_default(&o);
    o.max_correspondence_distance = 2.0, o.max_iterations = 30, o.transformation_epsilon = 1e-10, o.euclidean_fitness_epsilon = 1e-8;
    double g[7];
    ilsm::matrix_to_pose7(guess, g);
    const int offs[2] = {0, (int)source.size()};
    ilsm_icp_result r;
    ilsm::check(ilsm_icp_align_batch(ctx->get(), &map, 1, ilsm::cloud_ptr(source), offs, 32, g, &o, &r), "ilsm_icp_align_batch");
    ilsm_map_destroy(map);

    const ilsm_icp_result& m = icp.lastResult();
    const bool same = std::memcmp(&m, &r, sizeof(r)) == 0;
    std::printf("icp mirror: converged %d state %d iterations %d fitness %.9g t (%.6f %.6f %.6f) -- %s\n", m.converged, m.state,
                m.iterations, m.fitness, m.t[0], m.t[1], m.t[2], same ? "identical to the C ABI" : "DIFFERS from the C ABI");
    const ilsm::Matrix4f T = icp.getFinalTransformation();
    const bool ok = same && icp.hasConverged() && icp.getFitnessScore() < 1e-6 && std::fabs(T(0, 3) - 0.4f) < 1e-3f &&
                    std::fabs(T(1, 3) + 0.3f) < 1e-3f && out.size() == source.size();
    std::printf(ok ? "icp mirror checks passed\n" : "icp mirror checks FAILED\n");
    return ok ? 0 : 1;
  } catch (const ilsm::Error& e) {
    std::printf("ilsm::Error %d: %s\n", e.code, e.what());
    return 100;
  }
}
