// ilsm::StagedLoamPipeline with loop closure (include/ilsm.hpp) against the C ABI it wraps: the same frames through the
// mirror and through a raw ilsm_slam_create_staged handle must give the same loop events byte for byte, and a revisit
// must be accepted.  Input: a frame file (int32 frame count, int32 points per frame, then the frames as float x y z i).
// Exit codes: 0 pass, 1 mismatch or no accepted revisit, 2 unreadable input, the ilsm_status of an ilsm::Error otherwise
// (ILSM_ERR_NO_DEVICE without a GPU).
#include <cstdio>
#include <cstring>
#include <vector>

#include "ilsm.hpp"

int main(int argc, char** argv) {
  try {
    ilsm::ContextPtr ctx = ilsm::Context::shared();  // first: without a GPU this throws ILSM_ERR_NO_DEVICE
    FILE* f = argc > 1 ? std::fopen(argv[1], "rb") : nullptr;
    if (!f) return 2;
    int32_t count = 0, n = 0;
    if (std::fread(&count, 4, 1, f) != 1 || std::fread(&n, 4, 1, f) != 1 || count < 1 || n < 1) return 2;
    ilsm_slam_loop_opts o;
    ilsm_slam_loop_opts_default(&o);
    o.loop.exclude_recent = 20, o.loop.tree_period = 1, o.loop.sc_dist_threshold = 0.3;
    ilsm::StagedLoamPipeline mirror(0.6f, 0.8f, 0.3f, 16384, ctx);
    mirror.enableLoopClosure(o);
    ilsm_slam* raw = nullptr;
    ilsm::check(ilsm_slam_create_staged(ctx->get(), 0.6f, 0.8f, 0.3f, 16384, &raw), "ilsm_slam_create_staged");
    ilsm::check(ilsm_slam_enable_loop(raw, &o), "ilsm_slam_enable_loop");
    std::vector<ilsm_slam_loop_event> got;
    std::vector<float> xyzi((size_t)n * 4);
    ilsm::PointCloud<ilsm::PointXYZI> held[2];  // the raw handle reads a frame until the next call returns
    double q[4], t[3], qm[4], tm[3];
    int fo, fm;
    for (int k = 0; k < count + 2; ++k) {
      if (k < count) {
        ilsm::PointCloud<ilsm::PointXYZI>& cloud = held[k & 1];
        if (std::fread(xyzi.data(), 4, xyzi.size(), f) != xyzi.size()) return 2;
        cloud.resize(n);
        for (int i = 0; i < n; ++i) {
          ilsm::PointXYZI& p = cloud[i];
          p.x = xyzi[4 * i], p.y = xyzi[4 * i + 1], p.z = xyzi[4 * i + 2], p.intensity = xyzi[4 * i + 3];
        }
        mirror.push(cloud);
        ilsm::check(ilsm_slam_frame_staged(raw, ilsm::cloud_ptr(cloud), n, 32, 1, q, t, &fo, qm, tm, &fm, nullptr), "ilsm_slam_frame_staged");
      } else {
        mirror.drain();
        ilsm::check(ilsm_slam_frame_staged(raw, nullptr, -1, 16, 1, q, t, &fo, qm, tm, &fm, nullptr), "ilsm_slam_frame_staged");
      }
      if (k % 16 == 0) mirror.loopResults(got, false);  // collect on the way, as a caller would
    }
    std::fclose(f);
    mirror.loopResults(got, true);
    std::vector<ilsm_slam_loop_event> want(got.size() + 8);
    int n_want = 0;
    ilsm::check(ilsm_slam_loop_results(raw, 1, want.data(), (int)want.size(), &n_want), "ilsm_slam_loop_results");
    ilsm_slam_destroy(raw);
    int same = 0, accepted = 0;
    for (size_t i = 0; i < got.size() && (int)i < n_want; ++i) {
      same += std::memcmp(&got[i], &want[i], sizeof(ilsm_slam_loop_event)) == 0;
      if (got[i].result.accepted) {
        ++accepted;
        std::printf("frame %lld: loop with keyframe %d, distance %.4f, fitness %.4f\n", (long long)got[i].frame,
                    got[i].result.loop_id, got[i].result.sc_dist, got[i].result.icp.fitness);
      }
    }
    const bool ok = n_want == (int)got.size() && same == n_want && accepted > 0;
    std::printf("slam loop mirror: %d frames, %d keyframes, %d accepted, %d identical to the C ABI -- %s\n", count, (int)got.size(),
                accepted, same, ok ? "slam loop mirror checks passed" : "slam loop mirror checks FAILED");
    return ok ? 0 : 1;
  } catch (const ilsm::Error& e) {
    std::printf("ilsm::Error %d: %s\n", e.code, e.what());
    return e.code;
  }
}
