// chain_batcher.hpp -- many host threads prepare chaining problems, ONE kernel launch solves what they have ready.
//
// The Anchorer's fill-in pass (reference: include/centrolign/anchorer.hpp:655-693) chains the matches inside every gap of
// the main chain separately: thousands of independent subproblems of a few dozen matches, each of which builds its own
// reachability structures and match bank on the host and then needs the DP result at once for its traceback.  Solved one
// after the other, every subproblem pays a staging copy, a launch on ONE SM and a read-back, and the host work between the
// launches keeps the GPU idle.  Here the subproblems run on a pool of worker threads (many more than cores: a worker spends
// most of its time blocked).  A worker that reaches the DP lays its problem out itself (clb_chain_job_create) and blocks in
// ChainBatcher::solve; when every worker of the pool is blocked (or enough jobs are waiting) one of them takes all waiting
// jobs to the device in one clb_chain_jobs_run -- a CTA per problem -- and wakes the others.  Results do not depend on
// which jobs share a launch, so the output is the one the serial loop produces.  Given several devices, the pool keeps
// one batcher per device and binds every worker to one of them: the subproblems are independent, so they spread over the
// GPUs like the windows of a stitch.
#ifndef CENTROLIGN_B200_CHAIN_BATCHER_HPP
#define CENTROLIGN_B200_CHAIN_BATCHER_HPP

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <exception>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "centrolign_b200.h"
#include "devices.hpp"

namespace centrolign_b200 {

class ChainBatcher {
public:
    // `run` takes a batch of jobs to the device (clb_chain_jobs_run; the unit test passes a stand-in that needs no GPU)
    typedef int (*RunJobs)(int device, int64_t n_jobs, clb_chain_job* const* jobs);
    ChainBatcher(int device, int workers, size_t max_batch, RunJobs run = clb_chain_jobs_run)
        : device_(device), active_(workers), max_batch_(max_batch), run_(run) {}

    // the device every job of this batcher is created for and run on
    int device() const { return device_; }

    // the batcher of the pool the calling thread works for, or nullptr: ChainProblem::solve asks
    static ChainBatcher*& current() {
        static thread_local ChainBatcher* b = nullptr;
        return b;
    }

    // Called by a worker with a job from clb_chain_job_create: returns when the job has run (its outputs are filled).
    void solve(clb_chain_job* job) {
        Waiting me{job, false, CLB_OK, std::string()};
        std::unique_lock<std::mutex> lk(mu_);
        waiting_.push_back(&me);
        while (!me.done) {
            if (!flushing_ && !waiting_.empty() && (waiting_.size() + in_flight_ >= (size_t)active_ || waiting_.size() >= max_batch_)) {
                // everybody who could still add a job is blocked here (or the batch is large enough): take it to the device
                std::vector<Waiting*> batch;
                batch.swap(waiting_);
                in_flight_ = batch.size();
                flushing_ = true;
                lk.unlock();
                std::vector<clb_chain_job*> jobs(batch.size());
                for (size_t k = 0; k < batch.size(); ++k) jobs[k] = batch[k]->job;
                const int rc = run_(device_, (int64_t)jobs.size(), jobs.data());
                const std::string err = rc == CLB_OK ? std::string() : std::string(clb_last_error());
                lk.lock();
                for (Waiting* w : batch) {
                    w->rc = rc;
                    w->error = err;
                    w->done = true;
                }
                in_flight_ = 0;
                flushing_ = false;
                cv_.notify_all();
            } else {
                cv_.wait(lk);
            }
        }
        if (me.rc != CLB_OK) throw std::runtime_error("centrolign_b200: " + me.error);
    }

    // a worker has left the pool: the others must not wait for it
    void worker_done() {
        std::lock_guard<std::mutex> lk(mu_);
        --active_;
        cv_.notify_all();
    }

private:
    struct Waiting {
        clb_chain_job* job;
        bool done;
        int rc;
        std::string error;
    };
    const int device_;
    int active_;
    const size_t max_batch_;
    const RunJobs run_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::vector<Waiting*> waiting_;
    size_t in_flight_ = 0;
    bool flushing_ = false;
};

// body(i) for every i in [0, n), on a pool of workers whose ChainProblem::solve calls share launches.  With several
// devices, worker t works for the batcher of devices[t % D] (D = the number of devices, at most the number of workers):
// its jobs are created for that device and run there, in launches that carry that device's jobs only.
// CLB_FILL_IN_THREADS sets the pool size (default 4 per hardware thread, 16..128); 1 = the serial loop, no batching.
template <class Body>
void batched_parallel_for(size_t n, const std::vector<int>& devices, Body&& body, ChainBatcher::RunJobs run = clb_chain_jobs_run,
                          int pool_size = 0) {
    static const int configured = getenv("CLB_FILL_IN_THREADS") ? atoi(getenv("CLB_FILL_IN_THREADS")) : 0;
    const unsigned hw = std::thread::hardware_concurrency();
    size_t threads = pool_size > 0 ? (size_t)pool_size
                     : configured > 0 ? (size_t)configured : std::min<size_t>(128, std::max<size_t>(16, 4 * (size_t)(hw ? hw : 4)));
    threads = std::min(threads, n);
    if (threads <= 1 || ChainBatcher::current()) {  // nothing to share, or already inside a pool
        for (size_t i = 0; i < n; ++i) body(i);
        return;
    }
    const size_t n_dev = std::max<size_t>(1, std::min(devices.size(), threads));
    std::vector<std::unique_ptr<ChainBatcher>> batchers;
    for (size_t d = 0; d < n_dev; ++d) {
        const size_t workers = threads / n_dev + (d < threads % n_dev ? 1 : 0);  // the t < threads with t % n_dev == d
        batchers.emplace_back(new ChainBatcher(devices.empty() ? 0 : devices[d], (int)workers, 4 * 148, run));
    }
    std::atomic<size_t> next(0);
    std::mutex err_mu;
    std::exception_ptr first_error;
    std::vector<std::thread> pool;
    pool.reserve(threads);
    for (size_t t = 0; t < threads; ++t)
        pool.emplace_back([&, t] {
            ChainBatcher& batcher = *batchers[t % n_dev];
            ChainBatcher::current() = &batcher;
            try {
                for (size_t i = next.fetch_add(1); i < n; i = next.fetch_add(1)) body(i);
            } catch (...) {
                std::lock_guard<std::mutex> lk(err_mu);
                if (!first_error) first_error = std::current_exception();
                next.store(n);  // the others finish what they have and stop
            }
            ChainBatcher::current() = nullptr;
            batcher.worker_done();
        });
    for (std::thread& th : pool) th.join();
    if (first_error) std::rethrow_exception(first_error);
}

// The pool on one device.
template <class Body>
void batched_parallel_for(size_t n, int device, Body&& body, ChainBatcher::RunJobs run = clb_chain_jobs_run, int pool_size = 0) {
    batched_parallel_for(n, std::vector<int>(1, device), std::forward<Body>(body), run, pool_size);
}

}  // namespace centrolign_b200

#endif
