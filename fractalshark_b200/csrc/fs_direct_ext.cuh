// fs_direct_ext.cuh -- direct (non-perturbed) escape-time kernels in the extended-precision types, the rest of
// row a6 of SURVEY.md section 8:
//   Gpu2x32   mandel_2x_float<P>   LowPrecisionKernels.cuh:383-553   (2x32 double-float, P = 1/4/8/16 steps per test)
//   Gpu2x64   mandel_2x_double     LowPrecisionKernels.cuh:171-287   (double-double)
//   Gpu4x32   mandel_4x_float      LowPrecisionKernels.cuh:5-74      (four-float expansion)
//   Gpu4x64   mandel_4x_double     LowPrecisionKernels.cuh:76-144    (four-double expansion)
//   GpuHDRx32 mandel_hdr_float<P>  LowPrecisionKernels.cuh:554-678   (float+exponent wrapper over 2x32)
// Each pixel policy below states the reference's step in its own arithmetic; none of these kernels shortens
// n_iterations by P-1 (only the 1x kernels do), the output row is flipped (Y -> height-Y-1) as there.
// Execution: the persistent warp-tile queue shared by every render kernel of this library.
#pragma once
#include "fs_df32.cuh"
#include "fs_direct.cuh"
#include "fs_qd.cuh"

namespace fs {

template <class C, class IterT> struct DirectExtArgs {
    IterT *out;
    int width, height, pitch;
    int shard_count, shard_index;
    C cx, cy, dx, dy;
    IterT n_iterations;
    TileQueue queue;
    unsigned long long *step_counter;
};

// ---- Gpu2x32 -----------------------------------------------------------------------------------------------------
// mul_dblflt2x  dblflt.cuh:180-193: product, renormalise, then both halves times 2
FS_D df32 df_mul2x(df32 a, df32 b) {
    df32 z = df_mul(a, b);
    z.tail = __fmul_rn(z.tail, 2.0f);
    z.head = __fmul_rn(z.head, 2.0f);
    return z;
}
template <int P> struct Pixel2x32 {
    using Coord = df32;
    template <class IterT> FS_D static IterT run(const DirectExtArgs<df32, IterT> &A, int X, int Y) {
        const df32 cx = df_two_sum(A.cx.head, A.cx.tail), cy = df_two_sum(A.cy.head, A.cy.tail);
        const df32 dx = df_two_sum(A.dx.head, A.dx.tail), dy = df_two_sum(A.dy.head, A.dy.tail);
        const df32 x0 = df_add(cx, df_mul(dx, df_two_sum((float)X, 0.0f)));
        const df32 y0 = df_add(cy, df_mul(dy, df_two_sum((float)Y, 0.0f)));
        df32 x = df_make(0, 0), y = x, zr = x, zi = x;
        IterT iter = 0;
        while (__fadd_rn(zr.head, zi.head) < 4.0f && iter < A.n_iterations) {
#pragma unroll
            for (int p = 0; p < P; p++) {
                y = df_add(df_mul2x(x, y), y0);
                x = df_add(df_sub(zr, zi), x0);
                zr = df_sqr(x);
                zi = df_sqr(y);
            }
            iter += P;
        }
        return iter;
    }
};

// ---- Gpu2x64 -----------------------------------------------------------------------------------------------------
struct Pixel2x64 {
    using Coord = dd64;
    template <class IterT> FS_D static IterT run(const DirectExtArgs<dd64, IterT> &A, int X, int Y) {
        const dd64 cx = dd_two_sum(A.cx.head, A.cx.tail), cy = dd_two_sum(A.cy.head, A.cy.tail);
        const dd64 dx = dd_two_sum(A.dx.head, A.dx.tail), dy = dd_two_sum(A.dy.head, A.dy.tail);
        const dd64 x0 = dd_add(cx, dd_mul(dx, dd_two_sum((double)X, 0.0)));
        const dd64 y0 = dd_add(cy, dd_mul(dy, dd_two_sum((double)Y, 0.0)));
        const dd64 two = dd_two_sum(2.0, 0.0);
        dd64 x = dd_two_sum(0.0, 0.0), y = x;
        dd64 zr = dd_mul(x, x), zi = dd_mul(y, y);
        IterT iter = 0;
        while (__dadd_rn(zr.head, zi.head) < 4.0 && iter < A.n_iterations) {
            const dd64 xt = dd_add(dd_sub(zr, zi), x0);
            y = dd_add(dd_mul(two, dd_mul(x, y)), y0);
            x = xt;
            zr = dd_mul(x, x);
            zi = dd_mul(y, y);
            iter++;
        }
        return iter;
    }
};

// ---- Gpu4x32 / Gpu4x64 -------------------------------------------------------------------------------------------
// the step loop is quad_escape_count (fs_qd.cuh), shared with the host build of the oracle
template <class F> struct PixelQuad {
    using Coord = Quad<F>;
    template <class IterT> FS_D static IterT run(const DirectExtArgs<Coord, IterT> &A, int X, int Y) {
        return quad_escape_count<F, IterT>(A.cx, A.cy, A.dx, A.dy, X, Y, A.n_iterations);
    }
};
using Pixel4x32 = PixelQuad<float>;
using Pixel4x64 = PixelQuad<double>;

// ---- GpuHDRx32 (float+exponent over 2x32) ------------------------------------------------------------------------
template <int P> struct PixelHdr2x32 {
    using Coord = Hdr<df32>;
    template <class IterT> FS_D static IterT run(const DirectExtArgs<Coord, IterT> &A, int X, int Y) {
        const Coord X2 = reduced(hd_from_float((float)X)), Y2 = reduced(hd_from_float((float)Y));
        const Coord x0 = reduced(add(A.cx, mul(A.dx, X2)));
        const Coord y0 = reduced(add(A.cy, mul(A.dy, Y2)));
        Coord x = hd_zero(), y = hd_zero(), zr = hd_zero(), zi = hd_zero(), zs = hd_zero();
        const Coord Two = hd_from_float(2.0f), Four = hd_from_float(4.0f);
        IterT iter = 0;
        while (cmp_pr(zs, Four) < 0 && iter < A.n_iterations) {
#pragma unroll 1
            for (int p = 0; p < P; p++) {
                reduce(y);
                reduce(x);
                y = add(mul(mul(x, y), Two), y0);
                x = add(sub(zr, zi), x0);
                zr = reduced(mul(x, x));
                zi = reduced(mul(y, y));
                zs = reduced(add(zr, zi));
            }
            iter += P;
        }
        return iter;
    }
};

template <class Pixel, class IterT>
__global__ void __launch_bounds__(256) direct_ext_kernel(const DirectExtArgs<typename Pixel::Coord, IterT> A) {
    const int lane = threadIdx.x & 31;
    const int tiles_x = (A.width + 7) >> 3;
    const int tiles_y = (((A.height + 3) >> 2) - A.shard_index + A.shard_count - 1) / A.shard_count;
    const unsigned int n_tiles = (unsigned int)tiles_x * (unsigned int)tiles_y;
    unsigned long long steps = 0;
    TileCursor cursor;
    tile_queue_begin(cursor);
    for (;;) {
        unsigned int tile;
        if (!next_tile(A.queue, cursor, n_tiles, tile)) break;
        // bands are dealt over the output rows; the kernels' own Y is flipped (LowPrecisionKernels.cuh:309)
        int X, Yout;
        tile_origin(tile, tiles_x, tiles_y, A.shard_count, A.shard_index, X, Yout);
        X += lane & 7;
        Yout += lane >> 3;
        if (X < A.width && Yout < A.height) {
            const IterT iter = Pixel::template run<IterT>(A, X, A.height - 1 - Yout);
            steps += iter;
            A.out[(size_t)Yout * A.pitch + X] = iter;
        }
        __syncwarp();
    }
    if (A.step_counter) {
        for (int o = 16; o > 0; o >>= 1) steps += __shfl_down_sync(0xffffffffu, steps, o);
        if (lane == 0 && steps) atomicAdd(A.step_counter, steps);
    }
}

} // namespace fs
