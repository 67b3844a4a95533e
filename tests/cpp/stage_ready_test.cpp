// ilsm::Stage::ready() (csrc/ilsm_stage.hpp), the non-blocking check ilsm_slam_loop_results(wait = 0) uses: false while
// the oldest job runs or nothing is posted, true once its result waits, unchanged by later jobs, and it never blocks or
// changes the in-flight count.  Built with -fsanitize=thread.  Exit code 0: every check passed.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <string>
#include <thread>

#include "ilsm_stage.hpp"

namespace {
thread_local std::string t_error;
const char* last_error() { return t_error.c_str(); }
int fail(int code, const char* text) {
  t_error = text;
  return code;
}

int g_failures = 0;
#define CHECK(cond)                                                 \
  do {                                                              \
    if (!(cond)) {                                                  \
      std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      ++g_failures;                                                 \
    }                                                               \
  } while (0)

struct Job {
  int id = -1;
  bool gated = false;  // waits for the test to open the gate
};
using Stage = ilsm::Stage<Job, int>;

// polls ready() until it is true or ~5 s have passed
bool becomes_ready(const Stage& s) {
  for (int i = 0; i < 5000; ++i) {
    if (s.ready()) return true;
    std::this_thread::sleep_for(std::chrono::milliseconds(1));
  }
  return false;
}
}  // namespace

int main() {
  {  // never started, and started with nothing posted
    Stage s(last_error, fail);
    CHECK(!s.ready());
    s.start([] {}, [](const Job& j, int& r) { return r = j.id, 0; });
    CHECK(!s.ready());
  }
  {  // the oldest job still running: not ready, however long one waits
    std::atomic<bool> gate{false};
    Stage s(last_error, fail);
    s.start([] {}, [&gate](const Job& j, int& r) {
      while (j.gated && !gate.load()) std::this_thread::sleep_for(std::chrono::microseconds(200));
      r = j.id;
      return 0;
    });
    s.post({0, true});
    s.post({1, false});
    std::this_thread::sleep_for(std::chrono::milliseconds(50));
    CHECK(!s.ready());
    CHECK(s.in_flight() == 2);
    gate.store(true);
    CHECK(becomes_ready(s));
    CHECK(s.in_flight() == 2);  // ready() takes nothing
    int r = -1;
    CHECK(s.take(r) == 0 && r == 0);
    CHECK(becomes_ready(s));
    CHECK(s.take(r) == 0 && r == 1);
    CHECK(!s.ready() && s.in_flight() == 0);
  }
  {  // a failed job is ready too; take() carries its status
    Stage s(last_error, fail);
    s.start([] {}, [](const Job& j, int& r) { return r = j.id, fail(-7, "job failed"); });
    s.post({3, false});
    CHECK(becomes_ready(s));
    int r = -1;
    CHECK(s.take(r) == -7 && r == 3 && t_error == "job failed");
    CHECK(!s.ready());
  }
  {  // poll-and-take until every posted job is answered, the pattern of ilsm_slam_loop_results
    Stage s(last_error, fail);
    s.start([] {}, [](const Job& j, int& r) {
      std::this_thread::sleep_for(std::chrono::microseconds(100 * (j.id % 3)));
      return r = j.id, 0;
    });
    for (int i = 0; i < 50; ++i) s.post({i, false});
    int next = 0;
    for (int spins = 0; s.in_flight() > 0 && spins < 1000000; ++spins) {
      if (!s.ready()) continue;
      int r = -1;
      CHECK(s.take(r) == 0 && r == next);
      ++next;
    }
    CHECK(next == 50);
  }
  std::printf("%s\n", g_failures ? "stage ready checks FAILED" : "stage ready checks passed");
  return g_failures ? 1 : 0;
}
