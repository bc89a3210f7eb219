// fs_post.cuh -- antialias + palette colouring and min/max/sum reduction (row a7, SURVEY.md section 8).
//
// What: FractalSharkGpuLib/AntialiasingKernel.cuh:3-71 (box filter over AAxAA iteration cells, palette
// index (iters >> aux_depth) % palIters, in-set cells contribute 0, alpha 65535, colour index NOT padded)
// and ReductionKernels.cuh:73-142 (Min/Max/Sum over the width x height cells; Min starts at the
// IterType maximum).
//
// How: the reference runs two kernels that each stream the iteration buffer from HBM; here ONE pass
// reads every cell once, produces the colour and feeds a warp-shuffle reduction finished with native
// 64-bit atomics (HBM-bound: sizeof(IterType) read + 8/AA^2 written per cell).
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace fs {

struct Color16 { uint16_t r, g, b, a; };                 // GPU_Types.h:14-16
struct Reduction { unsigned long long Min, Max, Sum; };   // GPU_Types.h:40-50

template <class IterT> __global__ void __launch_bounds__(256) reduction_init_kernel(Reduction *out) {
    if (threadIdx.x != 0) return;
    out->Min = (unsigned long long)(IterT)~(IterT)0;
    out->Max = 0;
    out->Sum = 0;
}

// Colors = false: the caller asked for no colour buffer (RenderCurrent with color_buffer == NULL): the same pass without the
// palette gathers and the 8-byte colour stores, i.e. the reduction alone (4K frame: 47 -> 12 us).
template <class IterT, int AA, bool Colors = true>
__global__ void __launch_bounds__(256) post_kernel(const IterT *__restrict__ iters, int pitch,
                                                   Color16 *__restrict__ colors, const Color16 *__restrict__ pal,
                                                   uint32_t pal_iters, uint32_t aux_depth, int color_w, int color_h,
                                                   IterT n_iterations, Reduction *out, int shard_count, int shard_index) {
    unsigned long long vmin = ~0ull, vmax = 0, vsum = 0;
    const size_t total = (size_t)color_w * (size_t)color_h;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (size_t)gridDim.x * blockDim.x) {
        const int ox = (int)(o % (size_t)color_w);
        const int oy = (int)(o / (size_t)color_w);
        // multi-GPU: a shard colours and reduces the cells of its own 4-row bands only (AA in {1,2,4} divides the band
        // height, so a cell never straddles two bands; the host refuses AA 3 with more than one shard)
        if (shard_count > 1 && ((oy * AA) >> 2) % shard_count != shard_index) continue;
        unsigned long long ar = 0, ag = 0, ab = 0;
#pragma unroll
        for (int sx = 0; sx < AA; sx++) {
#pragma unroll
            for (int sy = 0; sy < AA; sy++) {
                const IterT n = iters[(size_t)(oy * AA + sy) * pitch + (ox * AA + sx)];
                vmin = n < vmin ? n : vmin;
                vmax = n > vmax ? n : vmax;
                vsum += n;
                if (Colors && n < n_iterations) {
                    const Color16 c = pal[(n >> aux_depth) % pal_iters];
                    ar += c.r; ag += c.g; ab += c.b;
                }
            }
        }
        if (Colors) {
            Color16 c;
            c.r = (uint16_t)(ar / (AA * AA));
            c.g = (uint16_t)(ag / (AA * AA));
            c.b = (uint16_t)(ab / (AA * AA));
            c.a = 65535;
            colors[o] = c;
        }
    }
    for (int s = 16; s > 0; s >>= 1) {
        const unsigned long long omin = __shfl_down_sync(0xffffffffu, vmin, s);
        const unsigned long long omax = __shfl_down_sync(0xffffffffu, vmax, s);
        vsum += __shfl_down_sync(0xffffffffu, vsum, s);
        vmin = omin < vmin ? omin : vmin;
        vmax = omax > vmax ? omax : vmax;
    }
    __shared__ unsigned long long smin[8], smax[8], ssum[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { smin[warp] = vmin; smax[warp] = vmax; ssum[warp] = vsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) {
            vmin = smin[w] < vmin ? smin[w] : vmin;
            vmax = smax[w] > vmax ? smax[w] : vmax;
            vsum += ssum[w];
        }
        atomicMin(&out->Min, vmin);
        atomicMax(&out->Max, vmax);
        atomicAdd(&out->Sum, vsum);
    }
}

// Device groups: the frame's Min/Max/Sum from the members' reductions of their own bands, on the lead device, so the
// result call stays enqueue-only.  A member that owns no cell contributes the neutral {IterT max, 0, 0}.
__global__ void __launch_bounds__(256) reduction_combine_kernel(const Reduction *__restrict__ parts, int n, Reduction *out) {
    if (threadIdx.x != 0) return;
    Reduction r = parts[0];
    for (int i = 1; i < n; i++) {
        r.Min = parts[i].Min < r.Min ? parts[i].Min : r.Min;
        r.Max = parts[i].Max > r.Max ? parts[i].Max : r.Max;
        r.Sum += parts[i].Sum;
    }
    *out = r;
}

} // namespace fs
