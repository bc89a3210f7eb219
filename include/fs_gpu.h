/* fs_gpu.h -- C-ABI of the B200-native per-pixel render path (libfsgpu.so).
 *
 * Drop-in boundary for the reference class `GPURenderer`
 * (FractalSharkLib/GPU_Render.h:20-227, implemented in FractalSharkGpuLib/GPU_Render.cu:92-1823).
 * Every C++ template of that class collapses to a runtime tag here; all numeric arguments cross as the
 * raw bytes of the reference PODs:
 *     float | double | {float head,tail} | {float m; int32 e} | {double m; int32 e; pad} | {float h,t; int32 e}
 * Orbit elements, LA records, LA stages, ATInfo and BLA records cross in the reference's own memory
 * layout (GPU_ReferenceIter.h:119-125, LAInfoDeep.h:33-39, LAInfoI.h:5-35, ATInfo.h:80-89, BLA.h:7-14),
 * so the reference host code can hand over `GetOrbitData()`, `GetLAs().GetData()` ... unchanged.
 *
 * Conventions (GPU_Render.cu:33-43, 626-628, 1007-1022): every call returns uint32_t, 0 = success,
 * else a cudaError_t value or a FractalSharkError (10000..10008).  Host pointers are borrowed for the
 * duration of the call; device copies are owned by the renderer and cached by generation number.
 * Render calls only enqueue work on the renderer's low-priority compute stream.
 * No C++ exceptions cross this boundary.  There is no CPU fallback: without a CUDA device every call
 * fails with the CUDA error.
 */
#ifndef FS_GPU_H
#define FS_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fs_renderer fs_renderer;

/* GPU_Types.h:14-16, 40-50 */
typedef struct { uint16_t r, g, b, a; } fs_color16;
typedef struct { uint64_t Min, Max, Sum; } fs_reduction;

/* numeric tag = the template argument T of the reference entry points */
enum fs_numeric {
    FS_NUM_F32 = 0,      /* float                                  */
    FS_NUM_F64 = 1,      /* double                                 */
    FS_NUM_2X32 = 2,     /* CudaDblflt<MattDblflt>  {head,tail}    */
    FS_NUM_HDR32 = 3,    /* HDRFloat<float>                        */
    FS_NUM_HDR64 = 4,    /* HDRFloat<double>                       */
    FS_NUM_HDR2X32 = 5,  /* HDRFloat<CudaDblflt<MattDblflt>>       */
    FS_NUM_2X64 = 6,     /* MattDbldbl   (direct kernels only)     */
    FS_NUM_4X32 = 7,     /* MattQFltflt  (direct kernels only)     */
    FS_NUM_4X64 = 8      /* MattQDbldbl  (direct kernels only)     */
};

/* PerturbExtras (HpSharkFloatLib/HighPrecision.h) */
enum fs_pextras { FS_PEXTRAS_DISABLE = 0, FS_PEXTRAS_BAD = 1, FS_PEXTRAS_SIMPLE_COMPRESSION = 2 };

/* LAv2Mode (FractalSharkLib/RenderAlgorithm.h:12-17) */
enum fs_lav2_mode { FS_LAV2_FULL = 1, FS_LAV2_PO = 2, FS_LAV2_LAO = 3 };

/* FractalSharkError (GPU_Render.cu:33-43) */
enum fs_error {
    FS_ERROR_1 = 10000, FS_ERROR_2, FS_ERROR_3_BAD_ANTIALIASING, FS_ERROR_4_WIDTH_NOT_MULTIPLE_OF_AA,
    FS_ERROR_5_HEIGHT_NOT_MULTIPLE_OF_AA, FS_ERROR_6_NO_ORBIT, FS_ERROR_7_NO_LA, FS_ERROR_8, FS_ERROR_9,
    FS_ERROR_UNSUPPORTED = 10100 /* tag combination the reference does not instantiate either */
};

/* replaces GPUPerturbResults<IterType,T,PExtras> (GPU_Types.h:83-175) */
typedef struct {
    const void *elements;        /* GPUReferenceIter<T,PExtras>[compressed_count], reference layout */
    uint64_t compressed_count;   /* GetCompressedSize()                                             */
    uint64_t uncompressed_count; /* GetUncompressedSize() == GetCountOrbitEntries()                 */
    uint64_t period_maybe_zero;  /* GetPeriodMaybeZero()                                            */
    const void *orbit_x_low;     /* T, may be NULL unless PExtras == SimpleCompression              */
    const void *orbit_y_low;
} fs_orbit;

/* replaces the accessors of LAReference<IterType,T,SubType,PExtras> read by the upload
 * (GPU_LAReference.h:78-162) */
typedef struct {
    const void *las;        /* LAInfoDeep<IterType,T,SubType,PExtras>[num_las], reference layout */
    uint64_t num_las;
    const void *stages;     /* LAStageInfo<IterType>[num_stages]                                 */
    uint64_t num_stages;
    const void *at;         /* ATInfo<IterType,T,SubType>                                        */
    uint64_t la_stage_count;/* GetLAStageCount()                                                 */
    int32_t use_at;         /* UseAT()                                                           */
    int32_t is_valid;       /* IsValid()                                                         */
} fs_la_reference;

/* replaces BLAS<IterType,T> as read by GPU_BLAS (BLA.cuh:123-160, GPU_BLAS.h:9-50) */
typedef struct {
    const void *const *levels;    /* levels[i] -> BLA<T>[level_counts[i]] (BLA.h:7-14), NULL for i < first_level */
    const uint64_t *level_counts;
    uint32_t num_levels;          /* LM2 + 2                                                     */
    uint32_t first_level;         /* BLAS::m_FirstLevel (= 2)                                    */
    int32_t lm2;                  /* compile-time LM2 of the reference instantiation (0..30)     */
} fs_blas;

/* ---- lifecycle ------------------------------------------------------------------------------ */
uint32_t fs_test_cuda_is_working(void);                        /* GPURenderer::TestCudaIsWorking  GPU_Render.h:25   */
fs_renderer *fs_create(int32_t device);                        /* GPURenderer()  (reference: always device 0)       */
void fs_destroy(fs_renderer *r);                               /* ~GPURenderer()                                    */

/* Device group (no reference counterpart): one handle that renders every frame on n devices.  Member i runs on
 * devices[i] and renders the 4-row bands b % n == i (the fs_set_shard rule); ids may repeat ({0, 0, 0} is three shards
 * on one GPU).  Every entry accepts the handle: uploads, clears, setters and render calls go to every member (render calls
 * enqueue on all of them from the calling thread; status = the first non-zero member status), fs_render_current
 * returns the same bytes a single renderer returns (iteration cells, colours at every antialiasing, Min/Max/Sum) and
 * stays enqueue-only (result calls may follow each other without a synchronise), the done callback runs once after
 * every member's render, step counters and launch counts are summed, fs_last_render_ms is the slowest member's, fs_get_width/height and fs_device_iter_buffer are member 0's.
 * fs_set_shard and fs_render_current_shard return FS_ERROR_UNSUPPORTED.  NULL for n == 0, an id outside
 * [0, device count) or an allocation failure; n == 1 is fs_create(devices[0]). */
fs_renderer *fs_create_group(const int32_t *devices, uint32_t n);
/* fs_create(0) when the environment variable FS_GPU_DEVICES is unset; else the group on the listed devices (decimal ids
 * separated by commas, e.g. "0,1,2,3").  NULL, before any CUDA call, for a malformed list: an empty item, a character
 * other than a digit or a comma, or more than 64 ids. */
fs_renderer *fs_create_default(void);
/* 1 for handles of fs_create, n for groups. */
uint32_t fs_device_count(const fs_renderer *r);

/* GPURenderer::InitializeMemory<IterType>  GPU_Render.h:91-100 ; iter_bytes = sizeof(IterType) (4|8) */
uint32_t fs_initialize_memory(fs_renderer *r, uint32_t iter_bytes, uint32_t w, uint32_t h, uint32_t antialiasing,
                              const fs_color16 *pal_interleaved, uint32_t pal_iters, uint32_t palette_aux_depth,
                              uint64_t palette_generation, int32_t expected_reuse);

/* GPURenderer::InitializePerturb<IterType,T1,SubType,PExtras,T2>  GPU_Render.h:102-108.
 * perturb2 / la may be NULL exactly as in the reference.  The uploads are queued on the compute stream: pageable
 * sources are consumed before the call returns (as with the reference's cudaMemcpy); PAGE-LOCKED sources are read
 * asynchronously and must stay unchanged until the stream has passed the upload (fs_sync_compute_stream, or the
 * result call of the render that follows). */
uint32_t fs_initialize_perturb(fs_renderer *r, uint32_t iter_bytes, int32_t numeric1, int32_t pextras,
                               uint64_t generation1, const fs_orbit *perturb1, int32_t numeric2, uint64_t generation2,
                               const fs_orbit *perturb2, const fs_la_reference *la);

/* GPURenderer::ClearMemory<IterType>  GPU_Render.h:110-111 */
void fs_clear_memory(fs_renderer *r);

/* ---- render calls (enqueue only) -------------------------------------------------------------- */
/* GPURenderer::Render<IterType,T>  GPU_Render.h:27-35 */
uint32_t fs_render(fs_renderer *r, uint32_t algorithm, int32_t numeric, const void *cx, const void *cy,
                   const void *dx, const void *dy, uint64_t n_iterations, int32_t iteration_precision);

/* GPURenderer::RenderPerturbLAv2<IterType,T,SubType,Mode,PExtras>  GPU_Render.h:79-88 */
uint32_t fs_render_perturb_lav2(fs_renderer *r, uint32_t algorithm, int32_t numeric, int32_t mode, int32_t pextras,
                                const void *cx, const void *cy, const void *dx, const void *dy, const void *center_x,
                                const void *center_y, uint64_t n_iterations);

/* Zoom batch (no reference counterpart): n_frames frames of the uploaded orbit and LA table in one launch -- the frames
 * of a zoom sequence share the view centre, hence the reference orbit.  Each coordinate pointer holds n_frames PODs of
 * `numeric` back to back (frame f at byte offset f * sizeof(POD)); algorithm, numeric, mode, pextras and n_iterations
 * are the same for every frame.  Enqueue only; the arrays are read before the call returns.  fs_set_shard applies to
 * every frame; the frames of a device group are sharded over its members like a single frame.  Frame 0 renders into the
 * iteration buffer, frames 1..n_frames-1 into a frame stack the renderer grows on demand; fs_select_frame picks the one
 * the result calls read.  The batch always runs the fused LAv2 tile kernel: fs_set_split_at, fs_set_pool_kernel and the
 * small-shard probe order do not apply (they change scheduling, never results).  The result sink is not written and is
 * left unfilled, so the next fs_render_current copies.  fs_last_render_ms and the step counters cover the whole batch.
 * n_frames outside [1, FS_MAX_FRAMES], a NULL renderer or a NULL dx/dy/center pointer: FS_ERROR_UNSUPPORTED, before any
 * CUDA call.  Frames that differ in scale need nothing extra: the AT shortcut's usability test is per pixel. */
#define FS_MAX_FRAMES 64
uint32_t fs_render_perturb_lav2_frames(fs_renderer *r, uint32_t algorithm, int32_t numeric, int32_t mode, int32_t pextras,
                                       uint32_t n_frames, const void *cx, const void *cy, const void *dx, const void *dy,
                                       const void *center_x, const void *center_y, uint64_t n_iterations);
/* Subsequent fs_render_current / fs_render_current_shard / fs_device_iter_buffer read frame k of the last render
 * (colours and Min/Max/Sum are computed from that frame).  Every render call selects frame 0; a single-frame render
 * counts as one frame.  k >= the last render's frame count (any k before the first render): FS_ERROR_UNSUPPORTED and
 * the selection is unchanged.  A device group selects the frame on every member. */
uint32_t fs_select_frame(fs_renderer *r, uint32_t k);

/* GPURenderer::RenderPerturbBLA<IterType,T>  GPU_Render.h:51-77 */
uint32_t fs_render_perturb_bla(fs_renderer *r, uint32_t algorithm, int32_t numeric, const fs_orbit *results,
                               const fs_blas *blas, const void *cx, const void *cy, const void *dx, const void *dy,
                               const void *center_x, const void *center_y, uint64_t n_iterations,
                               int32_t iteration_precision);

/* GPURenderer::RenderPerturbBLAScaled<IterType,T>  GPU_Render.h:37-49 (orbits carry the Bad field) */
uint32_t fs_render_perturb_bla_scaled(fs_renderer *r, uint32_t algorithm, int32_t numeric,
                                      const fs_orbit *double_perturb, const fs_orbit *float_perturb, const void *cx,
                                      const void *cy, const void *dx, const void *dy, const void *center_x,
                                      const void *center_y, uint64_t n_iterations, int32_t iteration_precision);

/* ---- results ---------------------------------------------------------------------------------- */
/* GPURenderer::RenderCurrent<IterType>  GPU_Render.h:123-129.  iter_buffer holds
 * roundup16(w)*roundup8(h) IterType cells, color_buffer roundup16(w/aa)*roundup8(h/aa) cells; any may be NULL. */
uint32_t fs_render_current(fs_renderer *r, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                           fs_reduction *reduction_results, int32_t progressive);

/* Sharded form of RenderCurrent (no reference counterpart: the reference drives one GPU, GPU_Render.h:123-129 is the
 * whole-frame call).  After fs_set_shard(n, i) it copies only the 4-row bands shard i rendered -- iteration cells and,
 * when color_buffer is given, the Color16 cells computed from them -- into the same positions of whole-frame host
 * buffers (layouts as in fs_render_current), so n processes can fill one host frame without a collective.  Colours and
 * the reduction cover this shard's cells only (frame reduction = min / max / sum of the shards').  Antialiasing 3 with
 * n > 1 and a colour buffer is refused (FS_ERROR_UNSUPPORTED): 3x3 cells straddle the 4-row bands.  With one shard it
 * is fs_render_current. */
uint32_t fs_render_current_shard(fs_renderer *r, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                                 fs_reduction *reduction_results, int32_t progressive);

/* Result sink (no reference counterpart; the reference copies the frame after the render, GPU_Render.cu:1768-1788).
 * Once set, the LAv2 render kernels store every finished pixel into `host_iter_buffer` (page-locked, or registered
 * here) as well as into the device buffer, so the frame crosses PCIe during the render; a following
 * fs_render_current / fs_render_current_shard given the same pointer skips its copy.  Rows a shard does not own are
 * not written.  Other render entries ignore the sink (their RenderCurrent copies as usual).  NULL removes it;
 * fs_initialize_memory and fs_destroy drop it. */
uint32_t fs_set_result_sink(fs_renderer *r, void *host_iter_buffer, uint64_t bytes);

uint32_t fs_sync_compute_stream(fs_renderer *r);   /* GPU_Render.h:131 */
uint32_t fs_sync_display_stream(fs_renderer *r);   /* GPU_Render.h:132 */
uint32_t fs_query_compute_stream(fs_renderer *r);  /* GPU_Render.h:133 */
/* GPU_Render.h:134-155: the callback replaces SignalComputeDone(); it runs on a CUDA host-func thread */
typedef void (*fs_done_callback)(void *user);
uint32_t fs_enqueue_compute_done_callback(fs_renderer *r, fs_done_callback fn, void *user);

const char *fs_convert_error_to_string(uint32_t err); /* GPU_Render.h:113 */
uint32_t fs_get_width(const fs_renderer *r);          /* GPU_Render.h:157 */
uint32_t fs_get_height(const fs_renderer *r);         /* GPU_Render.h:158 */

/* ---- additions with no reference counterpart (measurement + multi-GPU sharding) --------------- */
/* Multi-GPU sharding: subsequent render calls compute only the 4-row tile bands b with
 * b % shard_count == shard_index (1,0 = whole image). Cells of other shards are left untouched. */
uint32_t fs_set_shard(fs_renderer *r, uint32_t shard_count, uint32_t shard_index);
/* Measured FP32 issue peak of `device` (FFMA thread-instructions per second, micro-kernel with 16
 * independent chains per thread): the denominator of the roofline fraction reported by bench.py. */
uint32_t fs_measure_fp32_issue_peak(int32_t device, double *ffma_per_second);
/* Same probe with DFMA chains: the denominator for the FP64 kernels (Gpu1x64 direct, FP64 perturbation). */
uint32_t fs_measure_fp64_issue_peak(int32_t device, double *dfma_per_second);
/* Device time (CUDA events on the compute stream) of the most recent render kernel, in ms. Syncs. */
uint32_t fs_last_render_ms(fs_renderer *r, float *ms);
/* Count executed steps (perturbation + LA + AT) of subsequent renders into a device counter. */
uint32_t fs_enable_step_counter(fs_renderer *r, int32_t enable);
uint32_t fs_read_step_counter(fs_renderer *r, uint64_t *steps);
/* Same, split: counters3[0] = all executed steps, [1] = AT passes, [2] = LA steps (the LAv2 kernel fills 1 and 2;
 * perturbation steps = [0] - [1] - [2]). */
uint32_t fs_read_step_counters(fs_renderer *r, uint64_t *counters3);
/* HDRx32 perturbation: 1 (default) = scaled plain-float chunks with float+exponent fallback
 * (fs_scaled_loop.cuh), 0 = pure float+exponent loop.  Results are identical; takes effect at the next
 * InitializePerturb upload.  A/B switch for tests and profiling. */
uint32_t fs_set_scaled_steps(fs_renderer *r, int32_t enable);
/* HDRx32 LAv2 with an AT block: 1 = the AT shortcut runs in its own launch ahead of the LA/perturbation launch;
 * 0 (default) = one fused launch as in the reference.  Results are identical; the fused form measured faster. */
uint32_t fs_set_split_at(fs_renderer *r, int32_t enable);
/* Cycle detection: 1 (default) = a pixel whose state has entered an exactly periodic sequence (interior pixels) skips
 * whole periods instead of executing them -- in the AT shortcut of the LAv2 kernels (state after every 16 passes of
 * ATInfo::PerformAT) and in the BLA kernels (state at rebase events); 0 = every pass / period is executed, as the
 * reference does.  Results are identical bit for bit. */
uint32_t fs_set_at_cycle_detection(fs_renderer *r, int32_t enable);
/* Select-free forms of the HDRx32 kernels: 1 (default) = the LAv2 LA walk (32-bit iteration counts) runs on step-shaped
 * records derived on the device at upload (fs_la_step2.cuh) and the BLA loop evaluates its float+exponent sums without
 * operand selects (fs_bla.cuh bla_pixel_hdr32); 0 = the reference-shaped records / operators.  Results are identical bit
 * for bit. */
uint32_t fs_set_la_step2(fs_renderer *r, int32_t enable);
/* HDRx32 LAv2: 1 = the lane-refill kernel (every warp keeps pools of pixels waiting for the LA walk and for
 * perturbation steps and refills idle lanes from them, fs_lav2_pool.cuh); 0 (default: measured faster) = one 8x4 tile
 * per warp from start to finish.  Results are identical.  A/B switch for tests and profiling. */
uint32_t fs_set_pool_kernel(fs_renderer *r, int32_t enable);
/* Self-test: evaluates one operation of the device numeric types (the functions the render kernels call) on n operand
 * pairs from host arrays and writes n results to a host array.  op: 0-6 HDRFloat<float> add, sub, mul, square, Reduce,
 * divide, compareToBothPositiveReduced (result in .exp); 10-14 HDRFloatComplex<float> add, mul, Reduce, chebychevNorm,
 * times HDRFloat; 20-23 dblflt add, sub, mul, sqr; 30-32 dbldbl add, sub, mul; 40 the HDRx32 perturbation step (a = {dX, dY, Zx},
 * b = {Zy, cX, cY}, out = {dX', dY', 0}: 24 B each); 50-56 HDRFloat<double> add, sub, mul, square, Reduce, divide, compare
 * ({double mantissa; int32 exp; int32 pad}, 16 B).  Elements: {float mantissa; int32 exp}
 * (8 B), {float re, im; int32 exp} (12 B), {float head, tail} (8 B), {double head, tail} (16 B).  Reference: HDRFloat.h,
 * HDRFloatComplex.h, dblflt.cuh, dbldbl.cuh (the per-type operator tables SURVEY.md section 8 row a8 lists). */
uint32_t fs_selftest_numeric_op(int32_t device, uint32_t op, const void *a, const void *b, void *out, uint64_t n);
/* Device pointer of the iteration buffer (for NCCL gather by the host plumbing). */
void *fs_device_iter_buffer(fs_renderer *r);
/* Number of kernels this renderer has launched so far. */
uint64_t fs_kernel_launch_count(const fs_renderer *r);

#ifdef __cplusplus
}
#endif
#endif /* FS_GPU_H */
