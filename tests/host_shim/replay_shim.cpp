// tests/host_shim/replay_shim.cpp - TEST INFRASTRUCTURE ONLY.
//
// Host build of the replay sampler's index function (sdc_gym_b200/csrc/replay_index.cuh), the header
// csrc/replay.cu includes, so that the CPU suite can check it against the numpy restatement in
// sdc_gym_b200/replay.py.  Build: g++ -O1 -std=c++17 -fPIC -shared replay_shim.cpp
#include <cstdint>

#include "../../sdc_gym_b200/csrc/replay_index.cuh"

// rows/envs of samples j = 0 .. count-1 of one sample call
extern "C" void shim_replay_indices(uint64_t seed, uint32_t call, int64_t count, uint32_t upper, uint32_t n_envs,
                                    uint32_t* rows, uint32_t* envs) {
    for (int64_t j = 0; j < count; j++) sdcgym::replay_index(seed, call, (uint64_t)j, upper, n_envs, rows + j, envs + j);
}
