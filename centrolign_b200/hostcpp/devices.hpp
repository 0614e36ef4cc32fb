// devices.hpp -- the GPUs the C++ drop-in layer uses, read from CLB_DEVICES.
#ifndef CENTROLIGN_B200_DEVICES_HPP
#define CENTROLIGN_B200_DEVICES_HPP

#include <algorithm>
#include <cstdlib>
#include <vector>

namespace centrolign_b200 {

// Device list of the process: CLB_DEVICES="0,1,..." (ordinals; a repeated ordinal counts once, first-seen order is kept),
// else device 0.  The Stitcher recorder spreads every stitch over these GPUs and the fill-in chaining pool deals its
// subproblems to them, so a reference binary built with the shadow headers uses the listed GPUs without a source change.
inline std::vector<int> default_devices() {
    std::vector<int> out;
    if (const char* e = std::getenv("CLB_DEVICES")) {
        int cur = -1;
        for (const char* c = e;; ++c) {
            if (*c >= '0' && *c <= '9') cur = (cur < 0 ? 0 : cur * 10) + (*c - '0');
            else {
                if (cur >= 0 && std::find(out.begin(), out.end(), cur) == out.end()) out.push_back(cur);
                cur = -1;
                if (!*c) break;
            }
        }
    }
    if (out.empty()) out.push_back(0);
    return out;
}

// Device of the chaining calls that do not shard (one problem runs on one device): the first of default_devices().
inline int chain_device() { return default_devices()[0]; }

}  // namespace centrolign_b200

#endif
