// ilsm::Stage (csrc/ilsm_stage.hpp) on its own, without CUDA: results in FIFO order, the in-flight count, shutdown with
// and without posted jobs, and a failed job's status and error text reaching the thread that takes it.  Built with
// -fsanitize=thread.  Exit code 0: every check passed.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <string>
#include <thread>

#include "ilsm_stage.hpp"

namespace {
// the library's thread-local error text, as this test supplies it
thread_local std::string t_error;
const char* last_error() { return t_error.c_str(); }
int fail(int code, const char* text) {
  t_error = text;
  return code;
}

int g_failures = 0;
#define CHECK(cond)                                                      \
  do {                                                                   \
    if (!(cond)) {                                                       \
      std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond);      \
      ++g_failures;                                                      \
    }                                                                    \
  } while (0)

struct Job {
  int id = -1;
  int delay_us = 0;
  int fail_code = 0;
};
struct Result {
  int id = -1;
  std::thread::id thread;
};
using Stage = ilsm::Stage<Job, Result>;

// the job body: echoes the id, records the thread it ran on and fails on request
struct Counters {
  std::atomic<int> ran{0}, entered{0};
  std::thread::id enter_thread;  // written by `enter`, read after the stage has been stopped
};
void start(Stage& st, Counters& c) {
  st.start([&c] { c.enter_thread = std::this_thread::get_id(), c.entered++; },
           [&c](const Job& j, Result& r) {
             if (j.delay_us) std::this_thread::sleep_for(std::chrono::microseconds(j.delay_us));
             r.id = j.id, r.thread = std::this_thread::get_id();
             c.ran++;
             return j.fail_code ? fail(j.fail_code, ("job " + std::to_string(j.id) + " failed on the stage's thread").c_str()) : 0;
           });
}

double seconds_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// queued jobs come back in order: a burst, then the mapping stage's pattern (post frame k, take frame k - 1)
void fifo_queue() {
  Counters c;
  Stage st(last_error, fail);
  start(st, c);
  for (int i = 0; i < 5; ++i) st.post({i, 200 * (5 - i), 0});  // the first jobs are the slowest
  CHECK(st.in_flight() == 5);
  Result r;
  for (int i = 0; i < 5; ++i) {
    CHECK(st.take(r) == 0 && r.id == i);
    CHECK(st.in_flight() == 4 - i);
    CHECK(r.thread != std::this_thread::get_id() && r.thread == c.enter_thread);
  }
  st.post({100, 0, 0});
  for (int k = 101; k < 300; ++k) {
    st.post({k, k % 3 ? 0 : 50, 0});
    CHECK(st.in_flight() == 2);
    CHECK(st.take(r) == 0 && r.id == k - 1);
  }
  CHECK(st.take(r) == 0 && r.id == 299 && st.in_flight() == 0);
  st.stop();
  CHECK(c.entered == 1 && c.ran == 205);
}

// the front-end stage's one-slot pattern: post, take, post, ...
void one_slot() {
  Counters c;
  Stage st(last_error, fail);
  start(st, c);
  Result r;
  for (int k = 0; k < 200; ++k) {
    st.post({k, k % 7 ? 0 : 100, 0});
    CHECK(st.in_flight() == 1);
    CHECK(st.take(r) == 0 && r.id == k && st.in_flight() == 0);
  }
  st.stop();
  CHECK(c.entered == 1 && c.ran == 200);
}

// a stage destroyed with jobs posted and not taken runs them all, then joins
void destroy_with_jobs() {
  Counters c;
  {
    Stage st(last_error, fail);
    start(st, c);
    for (int i = 0; i < 20; ++i) st.post({i, 1000, 0});
    CHECK(st.in_flight() == 20);
  }
  CHECK(c.ran == 20);
}

// a stage destroyed with no job posted joins at once: asleep on its condition variable, just started, or never started
void destroy_idle() {
  Counters c;
  auto t0 = std::chrono::steady_clock::now();
  {
    Stage st(last_error, fail);
    start(st, c);
    std::this_thread::sleep_for(std::chrono::milliseconds(50));  // past the spin: the thread sleeps
    t0 = std::chrono::steady_clock::now();
  }
  CHECK(seconds_since(t0) < 1.0);
  t0 = std::chrono::steady_clock::now();
  {
    Stage st(last_error, fail);
    start(st, c);
  }
  CHECK(seconds_since(t0) < 1.0);
  { Stage st(last_error, fail); }
  Stage st(last_error, fail);
  start(st, c);
  st.stop();
  st.stop();  // a second stop, and the destructor's, do nothing
  CHECK(c.entered == 3 && c.ran == 0);
}

// a failed job's status and error text reach take() on the caller's thread; the jobs after it still run
void failed_job() {
  Counters c;
  Stage st(last_error, fail);
  start(st, c);
  st.post({0, 0, 0});
  st.post({1, 300, 7});
  st.post({2, 0, 0});
  Result r;
  CHECK(st.take(r) == 0 && r.id == 0);
  CHECK(t_error.empty());
  CHECK(st.take(r) == 7 && r.id == 1);
  CHECK(t_error == "job 1 failed on the stage's thread");
  t_error.clear();
  CHECK(st.take(r) == 0 && r.id == 2 && t_error.empty());
  CHECK(st.in_flight() == 0);
}
}  // namespace

int main() {
  fifo_queue();
  one_slot();
  destroy_with_jobs();
  destroy_idle();
  failed_job();
  if (g_failures) return 1;
  std::printf("stage checks passed\n");
  return 0;
}
