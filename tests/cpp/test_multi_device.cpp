// The multi-device parts of the C++ drop-in layer without a device: the fill-in pool over several devices
// (hostcpp/chain_batcher.hpp) with a stand-in run function, and the CLB_DEVICES parsing (hostcpp/devices.hpp).
//   --pool     the pool over devices {0, 1} and {0}
//   --solve    ChainProblem::solve inside the pool over devices {0, 1}: the device each job is created for
//   --devices  prints default_devices() and chain_device() for the CLB_DEVICES of the environment
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <stdexcept>
#include <thread>
#include <vector>

#include "chain_b200.hpp"
#include "chain_batcher.hpp"
#include "devices.hpp"

namespace {

// A job is an integer in disguise: (device << 32) | (k + 1), device = the device of the worker's batcher.
clb_chain_job* make_job(int device, size_t k) { return reinterpret_cast<clb_chain_job*>((uint64_t(device) << 32) | uint64_t(k + 1)); }
int job_device(clb_chain_job* j) { return (int)(reinterpret_cast<uint64_t>(j) >> 32); }
size_t job_index(clb_chain_job* j) { return (size_t)((reinterpret_cast<uint64_t>(j) & 0xffffffffu) - 1); }

std::mutex mu;
std::vector<int> runs_of;       // how often job k was run
std::vector<int> ran_on;        // the device job k was run on
std::map<int, int> launches;    // launches per device
int mixed_launches = 0;         // launches that carried a job created for another device
int fail_device = -1;           // a launch on this device reports an error

int fake_run(int device, int64_t n, clb_chain_job* const* jobs) {
    std::lock_guard<std::mutex> lk(mu);
    launches[device] += 1;
    bool mixed = false;
    for (int64_t i = 0; i < n; ++i) {
        const size_t k = job_index(jobs[i]);
        mixed |= job_device(jobs[i]) != device;
        runs_of[k] += 1;
        ran_on[k] = device;
    }
    mixed_launches += mixed ? 1 : 0;
    return device == fail_device ? CLB_ECUDA : CLB_OK;
}

int run(const std::vector<int>& devices, int n_items, int pool, int failing_device) {
    runs_of.assign((size_t)n_items, 0);
    ran_on.assign((size_t)n_items, -1);
    launches.clear();
    mixed_launches = 0;
    fail_device = failing_device;
    std::vector<std::thread::id> worker_of((size_t)n_items);
    std::vector<int> device_of((size_t)n_items, -1);
    bool threw = false;
    try {
        centrolign_b200::batched_parallel_for((size_t)n_items, devices, [&](size_t k) {
            if (k % 7 == 3) return;  // a gap without matches: no chaining call at all
            if (k % 5 == 0) std::this_thread::sleep_for(std::chrono::microseconds(100 + 37 * (k % 11)));
            centrolign_b200::ChainBatcher* b = centrolign_b200::ChainBatcher::current();
            const int dev = b ? b->device() : devices[0];
            worker_of[k] = std::this_thread::get_id();
            device_of[k] = dev;
            clb_chain_job* job = make_job(dev, k);
            if (b) b->solve(job);
            else if (fake_run(dev, 1, &job) != CLB_OK) throw std::runtime_error("serial call failed");
        }, fake_run, pool);
    } catch (const std::runtime_error&) {
        threw = true;
    }
    int bad = 0;
    const bool expect_throw = failing_device >= 0;
    if (threw != expect_throw) { std::fprintf(stderr, "FAILED: exception %d, expected %d\n", (int)threw, (int)expect_throw); ++bad; }
    if (mixed_launches) { std::fprintf(stderr, "FAILED: %d launches carried jobs of another device\n", mixed_launches); ++bad; }
    if (!expect_throw) {
        std::map<std::thread::id, int> device_of_worker;
        for (int k = 0; k < n_items; ++k) {
            const bool skipped = k % 7 == 3;
            if (runs_of[(size_t)k] != (skipped ? 0 : 1)) {
                std::fprintf(stderr, "FAILED: job %d ran %d times\n", k, runs_of[(size_t)k]);
                ++bad;
                break;
            }
            if (skipped) continue;
            if (ran_on[(size_t)k] != device_of[(size_t)k]) {
                std::fprintf(stderr, "FAILED: job %d was created for device %d and ran on %d\n", k, device_of[(size_t)k], ran_on[(size_t)k]);
                ++bad;
                break;
            }
            auto it = device_of_worker.find(worker_of[(size_t)k]);
            if (it == device_of_worker.end()) device_of_worker[worker_of[(size_t)k]] = device_of[(size_t)k];
            else if (it->second != device_of[(size_t)k]) {
                std::fprintf(stderr, "FAILED: one worker created jobs for devices %d and %d\n", it->second, device_of[(size_t)k]);
                ++bad;
                break;
            }
        }
        const bool busy = pool > 1 && n_items >= 1000;  // enough work that every worker takes some
        for (int d : devices)
            if (busy && launches[d] == 0) { std::fprintf(stderr, "FAILED: no launch on device %d\n", d); ++bad; }
        if (launches.size() > devices.size()) { std::fprintf(stderr, "FAILED: launches on %zu devices\n", launches.size()); ++bad; }
    }
    std::printf("pool over %zu device(s): %d items, %d workers%s:", devices.size(), n_items, pool, expect_throw ? ", failing launch" : "");
    for (const auto& kv : launches) std::printf(" device %d %d launches", kv.first, kv.second);
    std::printf("\n");
    return bad;
}

// ---- ChainProblem::solve in the pool: which device does it create its job for? ----
std::mutex solve_mu;
std::map<std::thread::id, std::vector<int>> created_on;  // per worker thread, the device of every job it created
std::atomic<size_t> n_created(0), n_run(0), n_foreign(0);

int solve_run(int device, int64_t n, clb_chain_job* const* jobs) {
    for (int64_t i = 0; i < n; ++i)
        if (job_device(jobs[i]) != device) ++n_foreign;
    n_run += (size_t)n;
    return CLB_OK;
}

int solve_test() {
    const int kArgumentDevice = 7;  // the device argument of solve(): inside a pool it must not be used
    const size_t n_items = 600;
    centrolign_b200::batched_parallel_for(n_items, std::vector<int>{0, 1}, [&](size_t) {
        centrolign_b200::ChainProblem p;  // what it holds does not matter: the stand-in job calls below never read it
        p.solve(kArgumentDevice);
    }, solve_run, 16);
    int bad = 0;
    std::map<int, size_t> per_device;
    for (const auto& kv : created_on) {
        for (int d : kv.second) per_device[d] += 1;
        for (int d : kv.second)
            if (d != kv.second[0]) { std::fprintf(stderr, "FAILED: one worker created jobs for devices %d and %d\n", kv.second[0], d); ++bad; break; }
    }
    if (n_created != n_items || n_run != n_items) { std::fprintf(stderr, "FAILED: %zu jobs created, %zu run, %zu items\n", n_created.load(), n_run.load(), n_items); ++bad; }
    if (n_foreign) { std::fprintf(stderr, "FAILED: %zu jobs ran on another device than the one they were created for\n", n_foreign.load()); ++bad; }
    if (per_device.count(kArgumentDevice)) { std::fprintf(stderr, "FAILED: %zu jobs were created for the device argument of solve()\n", per_device[kArgumentDevice]); ++bad; }
    if (per_device[0] == 0 || per_device[1] == 0) { std::fprintf(stderr, "FAILED: jobs per device: %zu on 0, %zu on 1\n", per_device[0], per_device[1]); ++bad; }
    std::printf("solve in the pool: %zu jobs on device 0, %zu on device 1\n", per_device[0], per_device[1]);
    std::printf(bad ? "FAILED\n" : "solve passed all tests!\n");
    return bad ? 1 : 0;
}

}  // namespace

// Stand-ins for the library's job calls; the linker resolves this program's calls to them rather than to
// libcentrolign_b200.so.  A job records the device it was created for, and there is nothing to solve.
extern "C" int clb_chain_job_create(int device, const clb_chain_problem*, float*, int64_t*, int64_t*, int64_t* chain_len, float*,
                                    clb_chain_job** job) {
    std::lock_guard<std::mutex> lk(solve_mu);
    *chain_len = 0;
    *job = make_job(device, n_created++);
    created_on[std::this_thread::get_id()].push_back(device);
    return CLB_OK;
}
extern "C" void clb_chain_job_destroy(clb_chain_job*) {}

int main(int argc, char** argv) {
    if (argc > 1 && !std::strcmp(argv[1], "--devices")) {
        std::printf("default_devices");
        for (int d : centrolign_b200::default_devices()) std::printf(" %d", d);
        std::printf("\nchain_device %d\n", centrolign_b200::chain_device());
        return 0;
    }
    if (argc > 1 && !std::strcmp(argv[1], "--pool")) {
        int bad = 0;
        bad += run({0, 1}, 2000, 32, -1);
        bad += run({0, 1}, 300, 7, -1);   // an odd pool: the devices get 4 and 3 workers
        bad += run({0}, 2000, 32, -1);    // one device: the single-device pool
        bad += run({0, 1}, 3, 64, -1);    // more workers than items
        bad += run({0, 1}, 300, 1, -1);   // serial loop: no batcher at all
        bad += run({0, 1}, 400, 16, 1);   // an error in one device's launch comes back as an exception
        std::printf(bad ? "FAILED\n" : "multi-device pool passed all tests!\n");
        return bad ? 1 : 0;
    }
    if (argc > 1 && !std::strcmp(argv[1], "--solve")) return solve_test();
    std::fprintf(stderr, "usage: %s --pool | --solve | --devices\n", argv[0]);
    return 2;
}
