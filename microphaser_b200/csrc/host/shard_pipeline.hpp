// shard_pipeline.hpp — the ordered shard pipeline of the file drivers: a pool of workers packs each submitted shard of
// genes, phases it on a device and writes the results in submission order. The device work comes in as callables, so
// the threading, ordering and error rules live here once and are tested without a GPU (tests/units/shard_pipeline.cpp).
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <exception>
#include <functional>
#include <map>
#include <mutex>
#include <optional>
#include <thread>
#include <vector>

namespace mph {

// Rules:
//  - shard k is written once shards 0 .. k-1 are out, so the output is the concatenation in submission order;
//  - once an error is recorded nothing more is written, and shards not yet started are skipped before packing;
//  - a shard's genes are freed as soon as it is packed, a result as soon as it is written (or passed over after an error);
//  - with a limit L, submit() waits while L shards are submitted but not yet written, which bounds the memory held.
template <class Shard, class Batch, class Result, class Timing>
class ShardPipeline {
 public:
  static constexpr size_t kAnyDevice = size_t(-1);
  using PackFn = std::function<Batch(Shard&)>;                           // runs without a device lock
  using PhaseFn = std::function<Result(size_t, Batch&, Timing& dev_sum)>;  // under that device's lock: a context is not re-entrant
  using WriteFn = std::function<void(Result&)>;                          // under the output lock, in shard order
  struct Totals { std::vector<Timing> per_dev; uint64_t pack_us = 0, write_us = 0; };  // per_dev: what phase() added up

  ShardPipeline(size_t n_dev, size_t n_workers, size_t max_pending, PackFn pack, PhaseFn phase, WriteFn write)
      : n_dev_(n_dev), max_pending_(max_pending), pack_(std::move(pack)), phase_(std::move(phase)), write_(std::move(write)),
        dev_mu_(n_dev), dev_sum_(n_dev, Timing{}) {
    for (size_t w = 0; w < n_workers; ++w) pool_.emplace_back([this, w] { work(w); });
  }
  ~ShardPipeline() { join(); }

  // Queues a shard for `device` (kAnyDevice: the first device whose lock is free, else worker % devices). Blocks while
  // the limit is reached. Returns false without taking the shard once an error has stopped the pipeline.
  bool submit(Shard&& shard, size_t device) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&] { return max_pending_ == 0 || n_submitted_ - next_out_ < max_pending_ || err_; });
    if (err_) return false;
    queue_.push_back(Job{n_submitted_++, std::move(shard), device});
    cv_.notify_all();
    return true;
  }

  bool failed() {
    std::lock_guard<std::mutex> lk(mu_);
    return err_ != nullptr;
  }

  // Joins the workers and fills `out`, then rethrows the first pack, phase or write error. `out` is filled either way:
  // the shards phased before a failure still count.
  void finish(Totals& out) {
    join();
    out = Totals{dev_sum_, pack_us_, write_us_};
    if (err_) std::rethrow_exception(err_);
  }

 private:
  struct Job { size_t k; Shard shard; size_t device; };

  static uint64_t us_since(std::chrono::steady_clock::time_point t0) {
    return uint64_t(std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count());
  }

  void join() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      closing_ = true;
    }
    cv_.notify_all();
    for (auto& t : pool_) t.join();
    pool_.clear();
  }

  // locks the device the shard goes to and returns its index
  size_t lock_device(size_t want, size_t worker) {
    if (want == kAnyDevice) {
      for (size_t d = 0; d < n_dev_; ++d)
        if (dev_mu_[d].try_lock()) return d;
      want = worker % n_dev_;
    }
    dev_mu_[want].lock();
    return want;
  }

  void work(size_t worker) {
    for (;;) {
      Job job;
      bool skip;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !queue_.empty() || closing_; });
        if (queue_.empty()) return;
        job = std::move(queue_.front());
        queue_.pop_front();
        skip = err_ != nullptr;
      }
      std::optional<Result> res;
      std::exception_ptr err;
      if (!skip) {
        try {
          const auto tp0 = std::chrono::steady_clock::now();
          Batch batch = pack_(job.shard);
          job.shard = Shard();  // what the genes hold is in the batch now
          pack_us_ += us_since(tp0);
          const size_t dv = lock_device(job.device, worker);
          std::lock_guard<std::mutex> dl(dev_mu_[dv], std::adopt_lock);
          res.emplace(phase_(dv, batch, dev_sum_[dv]));
        } catch (...) {
          err = std::current_exception();
        }
      }
      finished(job.k, std::move(res), err);
    }
  }

  void finished(size_t k, std::optional<Result>&& res, std::exception_ptr err) {
    std::lock_guard<std::mutex> lk(mu_);
    if (err && !err_) err_ = err;
    done_.emplace(k, std::move(res));
    for (auto it = done_.find(next_out_); it != done_.end(); it = done_.find(next_out_)) {
      if (it->second && !err_) {
        const auto tw0 = std::chrono::steady_clock::now();
        try {
          write_(*it->second);
        } catch (...) {
          err_ = std::current_exception();
        }
        write_us_ += us_since(tw0);
      }
      done_.erase(it);
      ++next_out_;
    }
    cv_.notify_all();
  }

  const size_t n_dev_, max_pending_;
  const PackFn pack_;
  const PhaseFn phase_;
  const WriteFn write_;
  std::mutex mu_;  // the queue, the shards waiting to be written, the error and the output
  std::condition_variable cv_;
  std::deque<Job> queue_;
  std::map<size_t, std::optional<Result>> done_;  // finished shards waiting for their turn; empty when skipped or failed
  size_t n_submitted_ = 0, next_out_ = 0;
  bool closing_ = false;
  std::exception_ptr err_;
  std::vector<std::mutex> dev_mu_;
  std::vector<Timing> dev_sum_;  // dev_sum_[d] is guarded by dev_mu_[d]
  std::atomic<uint64_t> pack_us_{0}, write_us_{0};
  std::vector<std::thread> pool_;
};

}  // namespace mph
