// ilsm::LoopClosure (include/ilsm.hpp) against the C ABI it wraps: the same keyframes through both must give the same
// bytes, and a revisit must be accepted.  Input: a keyframe file (int32 count; per keyframe int32 n, double q[4], t[3],
// float xyz[n][3]).  Exit codes: 0 pass, 1 mismatch or no accepted revisit, 2 unreadable input, the ilsm_status of an
// ilsm::Error otherwise (ILSM_ERR_NO_DEVICE without a GPU).
#include <cstdio>
#include <cstring>
#include <vector>

#include "ilsm.hpp"

int main(int argc, char** argv) {
  try {
    ilsm::ContextPtr ctx = ilsm::Context::shared();  // first: without a GPU this throws ILSM_ERR_NO_DEVICE
    FILE* f = argc > 1 ? std::fopen(argv[1], "rb") : nullptr;
    if (!f) return 2;
    int32_t count = 0;
    if (std::fread(&count, 4, 1, f) != 1) return 2;
    ilsm_loop_opts o;
    ilsm_loop_opts_default(&o);
    o.exclude_recent = 6, o.tree_period = 1, o.sc_dist_threshold = 0.3;
    ilsm::LoopClosure lc(ctx, &o);
    ilsm_loop* raw = nullptr;
    ilsm::check(ilsm_loop_create(ctx->get(), &o, &raw), "ilsm_loop_create");
    int accepted = 0, same = 0;
    for (int k = 0; k < count; ++k) {
      int32_t n = 0;
      double q[4], t[3];
      if (std::fread(&n, 4, 1, f) != 1 || std::fread(q, 8, 4, f) != 4 || std::fread(t, 8, 3, f) != 3) return 2;
      std::vector<float> xyz((size_t)n * 3);
      if (n && std::fread(xyz.data(), 4, xyz.size(), f) != xyz.size()) return 2;
      ilsm::PointCloud<ilsm::PointXYZI> cloud;
      for (int i = 0; i < n; ++i) {
        ilsm::PointXYZI p;
        p.x = xyz[3 * i], p.y = xyz[3 * i + 1], p.z = xyz[3 * i + 2];
        cloud.push_back(p);
      }
      ilsm_loop_result a, b;
      accepted += lc.addKeyframe(cloud, q, t, &a);
      ilsm::check(ilsm_loop_add_keyframe(raw, ilsm::cloud_ptr(cloud), n, 32, q, t, &b), "ilsm_loop_add_keyframe");
      same += std::memcmp(&a, &b, sizeof(a)) == 0;
      if (a.accepted)
        std::printf("keyframe %d: loop %d, distance %.4f, shift %d, fitness %.4f\n", a.keyframe_id, a.loop_id, a.sc_dist, a.shift,
                    a.icp.fitness);
    }
    std::fclose(f);
    ilsm_loop_destroy(raw);
    const bool ok = same == count && accepted > 0 && lc.size() == count;
    std::printf("loop mirror: %d keyframes, %d accepted, %d identical to the C ABI -- %s\n", count, accepted, same,
                ok ? "loop mirror checks passed" : "loop mirror checks FAILED");
    return ok ? 0 : 1;
  } catch (const ilsm::Error& e) {
    std::printf("ilsm::Error %d: %s\n", e.code, e.what());
    return e.code;
  }
}
