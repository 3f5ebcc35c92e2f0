// bed_select_emu.cpp — compiles the gather rule of a .bed column selection (garlic_b200/csrc/bed_select.cuh:
// bed_gather_byte) for the CPU so that tests/test_by_pop.py can check it against a numpy gather without a GPU.  TEST
// HARNESS ONLY: on the GPU the same source runs inside bed.cu:bed_select_kernel.
#include <cstdint>
#include "../garlic_b200/csrc/common.cuh"
#include "../garlic_b200/csrc/bed_select.cuh"

extern "C" {

// rows [n_snp][in_stride] → out [n_snp][ceil(n_ind/4)], the fields of columns cols[n_ind] from bit 0
void emu_bed_select(const uint8_t* rows, int64_t in_stride, int n_snp, const int32_t* cols, int n_ind, uint8_t* out)
{
    const int64_t out_bytes = (n_ind + 3) / 4;
    for (int s = 0; s < n_snp; ++s)
        for (int64_t ob = 0; ob < out_bytes; ++ob)
            out[s * out_bytes + ob] = garlic::bed_gather_byte(rows + s * in_stride, cols, n_ind, ob);
}

}  // extern "C"
