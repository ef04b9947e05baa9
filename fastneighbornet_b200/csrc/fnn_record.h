// fnn_record.h — the digest of the per-iteration strategy record (fnn_ctx_strategy_record, include/fastnn.h).
//
// One record row per agglomeration iteration holds what the Random or Relaxed strategy did in findNodes, plus a 64-bit
// digest of every position it produced.  The digest is a sum mod 2^64 of independent terms, so its value does not depend
// on the order in which the device's blocks add them.  Each term mixes the item's index (draw index, scan index, tie
// rank) with its positions: a draw or tie that is wrong, swapped with another or shifted by one changes the digest.
//
// Plain C++ with host/device qualifiers: fnn_modes.cuh accumulates it on the GPU, oracle/nnet_oracle.cpp compiles the same
// code for the CPU, and oracle/pyref.py restates rec_mix independently for the Random rows.
#pragma once
#include <stdint.h>

#ifndef FNN_HD
#if defined(__CUDACC__)
#define FNN_HD __host__ __device__
#else
#define FNN_HD
#endif
#endif

namespace rec {

constexpr int COLS = 4;   // Random: draws, rejected draws, remapped draws, digest.  Relaxed: scans, ties, look-aheads, digest.

// splitmix64's output function (Steele, Lea, Flood: "Fast splittable pseudorandom number generators", 2014)
FNN_HD inline uint64_t rec_mix(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
FNN_HD inline uint64_t rec_pack(int a, int b) { return ((uint64_t)(uint32_t)a << 32) | (uint64_t)(uint32_t)b; }

// Random: draw k of the iteration (0-based) went from position i to position j
FNN_HD inline uint64_t draw_term(int64_t k, int i, int j) { return rec_mix(rec_mix((uint64_t)k) ^ rec_pack(i, j)); }

// Relaxed: row scan s of the findNodes call (0-based) of position `row`; rank -1 stands for the scan itself, rank r >= 0 for
// its r-th tie (position order) at position `tie`
FNN_HD inline uint64_t scan_term(int s, int row, int rank, int tie) {
    return rec_mix(rec_mix(rec_pack(s, rank)) ^ rec_pack(row, tie));
}

}  // namespace rec
