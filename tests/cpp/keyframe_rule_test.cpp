// The full loop's keyframe rule (csrc/ilsm_keyframe.hpp) on poses read from stdin, one case per line as 16 hex floats:
// q_kf[4] t_kf[3] q[4] t[3] keyframe_dist keyframe_angle_rad.  Prints 1 (keyframe) or 0 per line.
#include <cstdio>
#include <cstdlib>

#include "ilsm_keyframe.hpp"

int main() {
  double v[16];
  for (;;) {
    for (int i = 0; i < 16; ++i) {
      char tok[64];
      if (std::scanf("%63s", tok) != 1) return 0;
      v[i] = std::strtod(tok, nullptr);
    }
    std::printf("%d\n", ilsm::keyframe_due(v, v + 4, v + 7, v + 11, v[14], v[15]) ? 1 : 0);
  }
}
