// Supersampled frames (DESIGN.md "Supersampling").  Sample pass k = j*N + i renders the part in F64 with the
// ray-space offset (i, j) of FrameParams; pass 0 writes the accumulator itself, every later pass is folded into it
// here, in pass order, one IEEE addition per channel.  The fold of the last pass also resolves: it divides by N*N
// and writes the requested format with the quantisation rule of pix_store (colour_store).
#pragma once

#include "ert_device.cuh"

namespace ert {

template <bool RESOLVE>
__global__ void __launch_bounds__(256)
ss_fold(const double *__restrict__ pass, double *__restrict__ acc, size_t n_px, int nn, int format, void *out)
{
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n_px; i += (size_t)gridDim.x * 256) {
        const size_t k = 3 * i;
        const d3 a = mk(acc[k] + pass[k], acc[k + 1] + pass[k + 1], acc[k + 2] + pass[k + 2]);
        if constexpr (RESOLVE) {
            const double d = (double)nn;
            colour_store(out, format, k, mk(a.x / d, a.y / d, a.z / d));
        } else {
            acc[k] = a.x; acc[k + 1] = a.y; acc[k + 2] = a.z;
        }
    }
}

}  // namespace ert
