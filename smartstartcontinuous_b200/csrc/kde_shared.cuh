// kde_shared.cuh -- what both KDE selection paths use: the result block the finish kernels count in, the host slots
// they hand the selection back through, and the padded state dimensions the pair kernels are built for.
#pragma once

#include "common.cuh"

namespace {

struct KdeResult {
    double best_ucb;
    long long best_j;
    unsigned int blocks_done;
    int n_rescued;
    unsigned int moments_ticket;      // last-block election of kde_moments_kernel
    int pad;
};

// what a selection hands back to the host, written by the last block of the finish kernel straight
// into mapped pinned host memory (flag last, release at system scope): the call ends without a
// device->host copy and without a stream synchronisation
// the selection result in mapped pinned host memory: three tagged slots (common.cuh host_slot_put)
constexpr int KDE_HOST_SLOTS = 3;     // best_ucb | best_j | (status, max_norm2_bits)

int pad_dim(int d) {
    const int opts[] = {1, 2, 3, 4, 6, 8, 12, 16, 24, 32};
    for (int o : opts)
        if (d <= o) return o;
    return -1;
}

}  // namespace
