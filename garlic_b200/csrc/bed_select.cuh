// bed_select.cuh — the gather rule of a column selection on .bed rows.  __host__ __device__ so that
// tests/bed_select_emu.cpp runs on the CPU the code that bed.cu:bed_select_kernel runs on the GPU.
//
// A .bed row holds input column c at bits 2(c%4) of byte c/4.  The selected row holds the handle's individual i (input
// column cols[i], cols ascending) at bits 2(i%4) of byte i/4, so byte ob is made of cols[4ob .. 4ob+3]; the fields of a
// ragged last byte beyond n_ind are 0.
#pragma once
#include "common.cuh"

namespace garlic {

GHD uint8_t bed_gather_byte(const uint8_t* row, const int32_t* cols, int n_ind, long long ob)
{
    uint32_t v = 0;
    for (int f = 0; f < 4; ++f) {
        const long long i = 4 * ob + f;
        if (i >= n_ind) break;
        const int c = cols[i];
        v |= (uint32_t)((row[c >> 2] >> (2 * (c & 3))) & 3u) << (2 * f);
    }
    return (uint8_t)v;
}

}  // namespace garlic
