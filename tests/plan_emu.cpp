// plan_emu.cpp — compiles the pruned walker's slice builder (garlic_b200/csrc/bound.cuh:plan_slice) for the CPU so that
// tests/test_plan_walk.py can check it against the column gather without a GPU.  TEST HARNESS ONLY: on the GPU the same
// source runs inside kernels.cu:walk_units_kernel.
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
#include "../garlic_b200/csrc/common.cuh"
#include "../garlic_b200/csrc/bound.cuh"

using namespace garlic;

extern "C" {

// compacted words [wlo, wlo + n) of every row → out [n_ind][n], from the uncompacted rows and the gather list src
void emu_plan_slice(const uint64_t* rows_in, int64_t in_words, const int32_t* src, long long L, int n_ind, long long wlo, int n,
                    uint64_t* out)
{
    const long long n_q = 2 * (wlo + n);
    std::vector<uint4> head(n_q), segs(n_q * kPlanSegMax);
    for (long long q = 0; q < n_q; ++q) plan_half(src, L, q, &head[q], &segs[q * kPlanSegMax]);
    for (int i = 0; i < n_ind; ++i)
        plan_slice(head.data(), segs.data(), L, reinterpret_cast<const uint32_t*>(rows_in + (int64_t)i * in_words), wlo, n,
                   out + (int64_t)i * n);
}

}  // extern "C"
