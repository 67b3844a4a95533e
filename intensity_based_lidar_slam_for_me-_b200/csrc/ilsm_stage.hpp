// ilsm_stage.hpp -- one pipeline stage on its own host thread: jobs go in and results come out in FIFO order.  Plain
// C++17 with no CUDA or library headers, so that a CPU test can build it on its own.
#pragma once
#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <utility>

namespace ilsm {

// post(), take() and stop() are for one caller thread; the job body runs on the stage's thread.  Status 0 is success.
template <typename Job, typename Result>
class Stage {
 public:
  // last_error: the calling thread's error text after a failed call; fail(code, text): makes `text` the calling
  // thread's error text and returns `code`.  Together they carry a failed job's error to the thread that takes it.
  Stage(const char* (*last_error)(), int (*fail)(int code, const char* text)) : last_error_(last_error), fail_(fail) {}
  ~Stage() { stop(); }

  // Starts the thread: `enter` runs once on it, then `body(job, result)` once per posted job, in posting order.
  void start(std::function<void()> enter, std::function<int(const Job&, Result&)> body) {
    body_ = std::move(body);
    thread_ = std::thread([this, enter] {
      enter();
      for (Job job; pop(jobs_, n_jobs_, job, true);) {
        Done d;
        d.rc = body_(job, d.r);
        if (d.rc) d.err = last_error_();  // the error text is thread-local: carry it over
        push(results_, n_results_, std::move(d));
      }
    });
  }

  void post(Job job) {
    push(jobs_, n_jobs_, std::move(job));
    in_flight_++;
  }

  // Waits for the result of the oldest job not yet taken into `out` and returns that job's status.
  int take(Result& out) {
    Done d;
    pop(results_, n_results_, d, false);
    in_flight_--;
    out = std::move(d.r);
    return d.rc ? fail_(d.rc, d.err.c_str()) : 0;
  }

  int in_flight() const { return in_flight_; }  // jobs posted and not yet taken

  // Whether take() would return at once: the oldest job not yet taken has finished.  Does not wait.
  bool ready() const { return n_results_.load(std::memory_order_acquire) > 0; }

  // Lets the thread run every job posted so far, then joins it.  Results not taken are dropped.
  void stop() {
    if (!thread_.joinable()) return;
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_.store(true, std::memory_order_release);
    }
    cv_.notify_all();
    thread_.join();
  }

 private:
  struct Done {
    Result r;
    int rc = 0;
    std::string err;
  };

  template <typename T>
  void push(std::deque<T>& q, std::atomic<int>& n, T v) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      q.push_back(std::move(v));
      n.fetch_add(1, std::memory_order_release);
    }
    cv_.notify_all();
  }

  // Takes the front of `q` into `out`; false when `stoppable` and the stage stops with `q` empty.  An empty queue is
  // first SPUN on (its atomic length, up to ~100 us), then slept on: a futex wake-up costs 10-50 us, a third of a
  // stage's time per frame.
  template <typename T>
  bool pop(std::deque<T>& q, std::atomic<int>& n, T& out, bool stoppable) {
    for (int i = 0; i < 4000 && n.load(std::memory_order_acquire) == 0 && !(stoppable && stop_.load(std::memory_order_acquire)); ++i) {
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
    }
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&] { return !q.empty() || (stoppable && stop_.load(std::memory_order_relaxed)); });
    if (q.empty()) return false;
    out = std::move(q.front());
    q.pop_front();
    n.fetch_sub(1, std::memory_order_relaxed);
    return true;
  }

  const char* (*last_error_)();
  int (*fail_)(int, const char*);
  std::function<int(const Job&, Result&)> body_;
  std::thread thread_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<Job> jobs_;
  std::deque<Done> results_;
  std::atomic<int> n_jobs_{0}, n_results_{0};  // the queues' lengths, for the spin outside the lock
  std::atomic<bool> stop_{false};
  int in_flight_ = 0;  // the caller's thread only
};

}  // namespace ilsm
