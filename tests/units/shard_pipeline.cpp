// TEST INFRASTRUCTURE ONLY — the ordered shard pipeline of the file drivers (csrc/host/shard_pipeline.hpp) with fake
// pack / phase / write steps that sleep for random times: write order, device choice and exclusion, the pending-shard
// limit, failures in each step and the destruction of results that are never written.
#include <atomic>
#include <cstdio>
#include <memory>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../microphaser_b200/csrc/host/shard_pipeline.hpp"

static std::atomic<int> g_fail{0};
#define CHECK(c) do { if (!(c)) { fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); ++g_fail; } } while (0)

static void jitter() {
  thread_local std::mt19937 rng(std::hash<std::thread::id>()(std::this_thread::get_id()));
  std::this_thread::sleep_for(std::chrono::microseconds(rng() % 300));
}

std::atomic<int> g_live{0};  // results alive
struct Tracked {
  size_t k;
  explicit Tracked(size_t k_) : k(k_) { ++g_live; }
  ~Tracked() { --g_live; }
};

struct Shard {
  size_t k = 0;
  size_t device = 0;  // the device it was submitted for, or kAnyDevice
  std::vector<int> genes;
};
struct Count {
  size_t shards = 0;
};
using Pipe = mph::ShardPipeline<Shard, Shard, std::unique_ptr<Tracked>, Count>;
constexpr size_t kAny = Pipe::kAnyDevice;

struct Run {
  size_t n_dev = 1, n_workers = 1, limit = 0, n = 40;
  bool fixed_device = false;
  size_t fail_pack = size_t(-1), fail_phase = size_t(-1), fail_write = size_t(-1);
  bool wait_for_failure = false;  // after submitting the failing shard, wait until the pipeline has stopped

  std::mutex mu;
  std::vector<size_t> written, packed;
  std::vector<std::atomic<int>> busy = std::vector<std::atomic<int>>(4);
  std::atomic<size_t> n_written{0};
  size_t submitted = 0, refused = 0, submitted_after_stop = 0;
  std::string error;
  Pipe::Totals totals;

  void go() {
    Pipe pipe(
        n_dev, n_workers, limit,
        [&](Shard& s) {
          jitter();
          {
            std::lock_guard<std::mutex> lk(mu);
            packed.push_back(s.k);
          }
          CHECK(s.genes.size() == s.k % 5);
          if (s.k == fail_pack) throw std::runtime_error("pack " + std::to_string(s.k));
          return std::move(s);
        },
        [&](size_t dv, Shard& b, Count& sum) {
          CHECK(dv < n_dev);
          if (b.device != kAny) CHECK(dv == b.device);
          CHECK(++busy[dv] == 1);  // one phase call at a time on a device
          jitter();
          --busy[dv];
          ++sum.shards;
          if (b.k == fail_phase) throw std::runtime_error("phase " + std::to_string(b.k));
          return std::unique_ptr<Tracked>(new Tracked(b.k));
        },
        [&](std::unique_ptr<Tracked>& r) {
          jitter();
          if (r->k == fail_write) throw std::runtime_error("write " + std::to_string(r->k));
          std::lock_guard<std::mutex> lk(mu);
          written.push_back(r->k);
          ++n_written;
        });
    const size_t fail_at = std::min(fail_pack, std::min(fail_phase, fail_write));
    for (size_t k = 0; k < n; ++k) {
      const bool stopped = pipe.failed();
      Shard s;
      s.k = k;
      s.device = fixed_device ? k * n_dev / n : kAny;
      s.genes.assign(k % 5, int(k));
      const size_t device = s.device;
      if (!pipe.submit(std::move(s), device)) {
        ++refused;
        continue;
      }
      ++submitted;
      if (stopped) ++submitted_after_stop;
      if (limit) CHECK(submitted - n_written.load() <= limit);
      if (k == fail_at && wait_for_failure)
        while (!pipe.failed()) std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
    try {
      pipe.finish(totals);
    } catch (const std::exception& e) {
      error = e.what();
    }
  }
};

static void check_in_order(const Run& r, size_t n_out) {
  CHECK(r.written.size() == n_out);
  for (size_t i = 0; i < r.written.size(); ++i) CHECK(r.written[i] == i);
}

static void ordering() {
  for (size_t n_dev : {1, 2})
    for (size_t n_workers : {1, 3, 8})
      for (bool fixed : {false, true}) {
        Run r;
        r.n_dev = n_dev;
        r.n_workers = n_workers;
        r.fixed_device = fixed;
        r.go();
        CHECK(r.error.empty());
        check_in_order(r, r.n);
        CHECK(r.totals.per_dev.size() == n_dev);
        size_t phased = 0;
        for (size_t d = 0; d < n_dev; ++d) phased += r.totals.per_dev[d].shards;
        CHECK(phased == r.n);
        if (fixed)
          for (size_t d = 0; d < n_dev; ++d) CHECK(r.totals.per_dev[d].shards == r.n / n_dev);
        CHECK(g_live == 0);
      }
}

static void limit() {
  for (size_t lim : {1, 2, 4}) {
    Run r;
    r.n_dev = 2;
    r.n_workers = 8;
    r.limit = lim;
    r.go();
    CHECK(r.error.empty());
    check_in_order(r, r.n);
  }
}

static void failures() {
  for (int step = 0; step < 3; ++step)
    for (size_t n_workers : {1, 3, 8}) {
      const size_t k = 10;
      Run r;
      r.n_dev = 2;
      r.n_workers = n_workers;
      r.wait_for_failure = true;
      (step == 0 ? r.fail_pack : step == 1 ? r.fail_phase : r.fail_write) = k;
      r.go();
      const char* what[] = {"pack ", "phase ", "write "};
      CHECK(r.error == what[step] + std::to_string(k));
      // shards before k may be left unwritten when a later one failed first; none from k on is written
      CHECK(r.written.size() <= k);
      check_in_order(r, r.written.size());
      CHECK(r.refused > 0 && r.submitted_after_stop == 0);
      for (size_t p : r.packed) CHECK(p <= k);  // nothing submitted after the failure was packed
      CHECK(g_live == 0);
    }
  // one worker: the shards queued behind the failing one were not started yet and are skipped before packing
  Run r;
  r.n_workers = 1;
  r.fail_phase = 5;
  r.go();
  CHECK(r.error == "phase 5");
  check_in_order(r, 5);
  for (size_t p : r.packed) CHECK(p <= 5);
  CHECK(g_live == 0);
  // the first write fails: every later result is destroyed unwritten
  Run w;
  w.n_workers = 8;
  w.n_dev = 2;
  w.fail_write = 0;
  w.go();
  CHECK(w.error == "write 0");
  CHECK(w.written.empty());
  CHECK(w.totals.per_dev[0].shards + w.totals.per_dev[1].shards > 1);
  CHECK(g_live == 0);
}

int main() {
  ordering();
  limit();
  failures();
  if (g_fail) return 1;
  printf("shard pipeline ok\n");
  return 0;
}
