// fs_capi.cu -- C-ABI (include/fs_gpu.h) over the sm_100a kernels: renderer lifecycle, table upload
// with generation-number caching, kernel dispatch from runtime tags, result extraction.
//
// Mirrors the host half of the reference boundary (row a9 of SURVEY.md section 8):
//   InitializeMemory  GPU_Render.cu:232-407      InitializePerturb  GPU_Render.cu:431-501
//   ClearMemory       GPU_Render.cu:212-225      Render             GPU_Render.cu:617-847
//   RenderPerturbLAv2 GPU_Render.cu:995-1188     RenderCurrent      GPU_Render.cu:556-581
//   RunAntialiasing   GPU_Render.cu:1695-1757    ExtractItersAndColors GPU_Render.cu:1759-1805
//   table upload      Perturb.cuh:20-80, GPU_LAReference.h:78-162
#include "../../include/fs_gpu.h"

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <new>
#include <vector>

#include "fs_bla.cuh"
#include "fs_direct.cuh"
#include "fs_direct_ext.cuh"
#include "fs_lav2.cuh"
#include "fs_lav2_pool.cuh"
#include "fs_orbit_rc.cuh"
#include "fs_post.cuh"
#include "fs_scaled_kernel.cuh"

using namespace fs;

namespace {

constexpr uint32_t NB_THREADS_W = 16; // GPU_Render.h:116-120
constexpr uint32_t NB_THREADS_H = 8;

// ---- reference wire layouts (natural alignment reproduces the reference structs; sizes asserted) ----
template <class Num, class IterT> struct WireLA {
    typename Num::Cplx Ref, ZCoeff, CCoeff;
    typename Num::Real LAThreshold, LAThresholdC, MinMag;
    IterT StepLength, NextStageLAIndex;
};
template <class Num, class IterT> struct WireAT {
    IterT StepLength;
    typename Num::Real ThresholdC, SqrEscapeRadius;
    typename Num::Cplx RefC, ZCoeff, CCoeff, InvZCoeff, CCoeffSqrInvZCoeff, CCoeffInvZCoeff;
    typename Num::Real CCoeffNormSqr, RefCNormSqr, factor;
};
// sizes measured from the reference headers with nvcc 12.9 (SURVEY.md section 2.2)
static_assert(sizeof(WireLA<NumHdr<float>, uint32_t>) == 68 && sizeof(WireLA<NumHdr<float>, uint64_t>) == 80, "LAInfoDeep");
static_assert(sizeof(WireLA<NumPlain<float>, uint32_t>) == 44 && sizeof(WireLA<NumPlain<float>, uint64_t>) == 56, "LAInfoDeep");
static_assert(sizeof(WireLA<NumPlain<double>, uint32_t>) == 80 && sizeof(WireLA<NumPlain<double>, uint64_t>) == 88, "LAInfoDeep");
static_assert(sizeof(WireLA<NumHdr<double>, uint32_t>) == 128 && sizeof(WireLA<NumHdr<double>, uint64_t>) == 136, "LAInfoDeep");
static_assert(sizeof(WireAT<NumHdr<float>, uint32_t>) == 116 && sizeof(WireAT<NumHdr<float>, uint64_t>) == 120, "ATInfo");
static_assert(sizeof(WireAT<NumPlain<float>, uint32_t>) == 72 && sizeof(WireAT<NumPlain<float>, uint64_t>) == 80, "ATInfo");
static_assert(sizeof(WireAT<NumPlain<double>, uint32_t>) == 144 && sizeof(WireAT<NumHdr<double>, uint32_t>) == 232, "ATInfo");
// 2x32 types (sizes from the reference headers, nvcc 12.9)
static_assert(sizeof(WireLA<Num2x32, uint32_t>) == 80 && sizeof(WireLA<Num2x32, uint64_t>) == 88, "LAInfoDeep 2x32");
static_assert(sizeof(WireLA<NumHdr2x32, uint32_t>) == 104 && sizeof(WireLA<NumHdr2x32, uint64_t>) == 112, "LAInfoDeep HDRx2x32");
static_assert(sizeof(WireAT<Num2x32, uint32_t>) == 140 && sizeof(WireAT<Num2x32, uint64_t>) == 144, "ATInfo 2x32");
static_assert(sizeof(WireAT<NumHdr2x32, uint32_t>) == 184 && sizeof(WireAT<NumHdr2x32, uint64_t>) == 192, "ATInfo HDRx2x32");

struct DeviceBlob {
    void *ptr = nullptr;
    size_t bytes = 0;
    bool host = false; // page-locked host memory read over PCIe: the reference's fallback when device memory runs out
};

struct OrbitDev {
    DeviceBlob data;
    DeviceBlob fast; // HDRx32: scaled::FastElem[compressed] derived on the device after the upload
    uint64_t compressed = 0, uncompressed = 0, period = 0;
    int numeric = -1, pextras = 0;
    uint64_t generation = 0;
    bool valid = false;
};

struct LaDev {
    DeviceBlob las, stages;
    DeviceBlob las2, stages2; // HDRx32 / 32-bit counts: step-shaped records of fs_la_step2.cuh, derived on the device
    uint64_t num_las = 0, num_stages = 0, stage_count = 0;
    int use_at = 0, is_valid = 0;
    int numeric = -1;
    uint32_t iter_bytes = 0;
    alignas(16) unsigned char at[256]; // AtDev<Num,IterT> image
    bool present = false;
};

} // namespace

struct fs_renderer {
    int device = 0;
    cudaStream_t compute = nullptr, display = nullptr;
    void *iter_buf = nullptr;
    Reduction *red_dev = nullptr;
    Color16 *color_buf = nullptr;
    Color16 *pal_dev = nullptr;
    uint32_t pal_iters = 0, aux_depth = 0;
    const void *cached_pal_host = nullptr;
    uint64_t cached_pal_gen = 0;
    uint32_t width = 0, height = 0, aa = 0, iter_bytes = 0;
    uint32_t w_block = 0, h_block = 0, color_w = 0, color_h = 0;
    size_t n_cu = 0, n_color_cu = 0;
    uint32_t shard_count = 1, shard_index = 0;
    unsigned int *tile_counter = nullptr;
    int *yield_quota = nullptr;          // device word next to the counter (TileQueue::yield_quota)
    int *yield_src = nullptr;            // page-locked constant the display stream copies into it
    bool yield_requested = false;        // a progressive RenderCurrent already freed SM slots during the current render
    cudaEvent_t ev_alloc = nullptr;      // orders display-stream work after (re)allocations made on the compute stream
    unsigned long long *step_counter = nullptr;
    bool count_steps = false;
    // result sink (fs_set_result_sink): a page-locked host frame the LAv2 kernels store finished pixels into while they
    // run, so the device->host transfer of the frame overlaps the render instead of following it
    void *sink_host = nullptr, *sink_dev = nullptr;
    bool sink_registered = false, sink_filled = false;
    int carveout_pct = -1;   // explicit shared-memory carve-out preference for every kernel (% of 228 KB), -1 = the driver's choice; FS_CARVEOUT
    bool force_host_tables = false; // FS_FORCE_HOST_TABLES: take the page-locked fallback of alloc_table (test hook)
    int ctas_per_sm_cap = 0; // FS_CTAS_PER_SM: experiment switch, caps the persistent grid below full occupancy
    bool split_at = false;  // HDRx32 + AT: AT shortcut in its own launch ahead of the LA/perturbation launch (fs_lav2.cuh AtPhase);
                            // measured slower than the fused launch (View 14: 9.7 vs 8.5 ms), kept as an A/B switch
    DeviceBlob at_state;    // float4 per iteration-buffer cell, allocated on first use
    bool at_cycle = true;   // AT shortcut: cycle detection (fs_lav2.cuh CycleWatch); FS_AT_CYCLE=0 / fs_set_at_cycle_detection executes every pass
    int probe_passes = 0;    // small shards: AT passes the cost probe runs per tile corner (lav2_probe_kernel); 0 = no probe; FS_PROBE_PASSES
    DeviceBlob tile_order;   // queue position -> tile ticket, plus two counters behind it
    bool use_la2 = true;    // HDRx32 / 32-bit counts: LA walk on step-shaped records (fs_la_step2.cuh); FS_LA_STEP2=0: reference-shaped records
    bool use_pool = false;  // HDRx32 LAv2: the lane-refill kernel of fs_lav2_pool.cuh (FS_LAV2_POOL=0 / fs_set_pool_kernel: one tile per warp)
    bool use_scaled = true; // HDRx32: scaled plain-float chunks (fs_scaled_loop.cuh); off = pure float+exponent loop
    OrbitDev orbit1, orbit2;
    OrbitDev bla_orbit;                  // RenderPerturbBLA uploads its orbit and table per call (GPU_Render.cu:1462-1483)
    OrbitDev scaled_orbit_f;             // RenderPerturbBLAScaled: binary32 orbit, per call (GPU_Render.cu:1324-1350)
    DeviceBlob bla_raw, bla_heads, bla_coefs;
    LaDev la;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    bool timed = false;
    uint64_t launches = 0;
    int num_sms = 148;
    fs_done_callback cb = nullptr;
    void *cb_user = nullptr;
    // device group (fs_create_group): member i renders shard (n, i) on its own device and every entry forwards to the
    // members; member 0 is the lead.  Empty for handles of fs_create.
    std::vector<fs_renderer *> members;
    std::vector<cudaEvent_t> joins; // one per member, on its device: joins the member's stream into the lead's
    Reduction *red_parts = nullptr; // on the lead: n member reductions + the frame's, for the compute and the display stream
    // AA 3: the whole frame's iteration cells gathered on the lead, one buffer for the compute and one for the display
    // stream.  cudaMalloc, not the stream-ordered pool: peer access (cudaDeviceEnablePeerAccess) covers it, so the members
    // write their bands into it directly.  Allocated only while the group's antialiasing is 3.
    void *gather[2] = {nullptr, nullptr};
    size_t gather_bytes = 0;
    cudaEvent_t lead_marks[2] = {nullptr, nullptr}; // on the lead's compute / display stream: what the lead has read so far
    // zoom batches (fs_render_perturb_lav2_frames): frame 0 renders into iter_buf, frames 1..n-1 into the frame stack, which
    // has iter_buf's layout per frame and comes from the same allocator, so every result path treats a stack frame as it
    // treats iter_buf.  Result calls read frame `selected` (fs_select_frame) of the last render's `n_frames`.
    void *frame_stack = nullptr;
    uint32_t stack_frames = 0;
    uint32_t n_frames = 0, selected = 0; // n_frames = 0: nothing rendered since the buffers were allocated
    DeviceBlob frame_recs;               // the batch's Lav2Frame records
    DeviceBlob expmap_tables;            // fs_render_perturb_lav2_expmap: radius[height], dir_x[width], dir_y[width]
};

namespace {

struct DeviceGuard {
    int prev = 0;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

void free_blob(fs_renderer *r, DeviceBlob &b) {
    if (b.ptr && b.host) {
        cudaStreamSynchronize(r->compute); // cudaFreeHost is not stream-ordered
        cudaFreeHost(b.ptr);
    } else if (b.ptr) {
        cudaFreeAsync(b.ptr, r->compute);
    }
    b.ptr = nullptr;
    b.bytes = 0;
    b.host = false;
}

// Table memory (orbit, LA records, LA stages): device memory, else page-locked host memory the kernels read through the
// unified address space -- the reference's own fallback for orbits that do not fit (Perturb.cuh:50-61,
// GPU_LAReference.h:90-113).  FS_FORCE_HOST_TABLES=1 takes the fallback unconditionally (test hook).
cudaError_t alloc_table(fs_renderer *r, DeviceBlob &b, size_t bytes) {
    b = DeviceBlob{};
    cudaError_t err = r->force_host_tables ? cudaErrorMemoryAllocation : cudaMallocAsync(&b.ptr, bytes, r->compute);
    if (err != cudaSuccess) {
        (void)cudaGetLastError();
        b.ptr = nullptr;
        err = cudaMallocHost(&b.ptr, bytes);
        if (err != cudaSuccess) return err;
        b.host = true;
    }
    b.bytes = bytes;
    return cudaSuccess;
}

void reset_perturb(fs_renderer *r) {
    free_blob(r, r->bla_orbit.data);
    free_blob(r, r->bla_orbit.fast);
    r->bla_orbit = OrbitDev{};
    free_blob(r, r->scaled_orbit_f.data);
    r->scaled_orbit_f = OrbitDev{};
    free_blob(r, r->bla_raw);
    free_blob(r, r->bla_heads);
    free_blob(r, r->bla_coefs);
    free_blob(r, r->orbit1.data);
    free_blob(r, r->orbit2.data);
    free_blob(r, r->orbit1.fast);
    free_blob(r, r->orbit2.fast);
    r->orbit1 = OrbitDev{};
    r->orbit2 = OrbitDev{};
    free_blob(r, r->la.las);
    free_blob(r, r->la.stages);
    free_blob(r, r->la.las2);
    free_blob(r, r->la.stages2);
    free_blob(r, r->tile_order);
    r->la = LaDev{};
}

void drop_sink(fs_renderer *r) {
    if (r->sink_registered) cudaHostUnregister(r->sink_host);
    r->sink_host = r->sink_dev = nullptr;
    r->sink_registered = r->sink_filled = false;
}

void reset_buffers(fs_renderer *r) {
    drop_sink(r);
    free_blob(r, r->at_state);
    free_blob(r, r->frame_recs);
    free_blob(r, r->expmap_tables);
    if (r->frame_stack) cudaFreeAsync(r->frame_stack, r->compute);
    r->frame_stack = nullptr;
    r->stack_frames = 0;
    r->n_frames = r->selected = 0;
    if (r->iter_buf) cudaFreeAsync(r->iter_buf, r->compute);
    if (r->red_dev) cudaFreeAsync(r->red_dev, r->compute);
    if (r->color_buf) cudaFreeAsync(r->color_buf, r->compute);
    r->iter_buf = nullptr;
    r->red_dev = nullptr;
    r->color_buf = nullptr;
}

bool memory_initialized(const fs_renderer *r) { return r->iter_buf && r->red_dev && r->color_buf; }

// The iteration cells every result call reads: frame `selected` of the last render (frame 0 = iter_buf).
void *selected_iter_buf(const fs_renderer *r) {
    if (r->selected == 0) return r->iter_buf;
    return static_cast<char *>(r->frame_stack) + (size_t)(r->selected - 1) * r->n_cu * r->iter_bytes;
}

template <class T> T load_pod_early(const void *p) {
    T v;
    memcpy(&v, p, sizeof(T));
    return v;
}

size_t orbit_elem_bytes(int numeric, int pextras) {
    size_t base;
    switch (numeric) {
    case FS_NUM_F32: base = 8; break;
    case FS_NUM_F64: base = 16; break;
    case FS_NUM_2X32: base = 16; break;
    case FS_NUM_HDR32: base = 16; break;
    case FS_NUM_HDR64: base = 32; break;
    case FS_NUM_HDR2X32: base = 24; break;
    default: return 0;
    }
    // Bad / CompressionIndex prefix is 8 bytes (GPU_ReferenceIter.h:10-49)
    return pextras == FS_PEXTRAS_DISABLE ? base : base + 8;
}

// Derives the plain-float step table (fs_scaled_loop.cuh) from an uploaded HDRx32 orbit.
__global__ void __launch_bounds__(256) build_fast_table_kernel(const uint4 *__restrict__ orbit, uint64_t count,
                                                               scaled::FastElem *__restrict__ tab) {
    for (uint64_t n = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; n < count; n += (uint64_t)gridDim.x * blockDim.x) {
        const uint4 v = orbit[n];
        tab[n] = scaled::make_fast_elem(__uint_as_float(v.x), (int)v.y, __uint_as_float(v.w), (int)v.z, n, n + 1 >= count);
    }
}

// Expands an uploaded waypoint list into the uncompressed layout (fs_orbit_rc.cuh)
template <class Num>
uint32_t expand_orbit(fs_renderer *r, const void *wire, uint64_t n_way, uint64_t n_full, const void *x_low, const void *y_low,
                      void *out) {
    using Real = typename Num::Real;
    const Real X = load_pod_early<Real>(x_low), Y = load_pod_early<Real>(y_low);
    const uint64_t want = (n_way + 127) / 128;
    const unsigned grid = (unsigned)(want < (uint64_t)r->num_sms * 16 ? (want ? want : 1) : (uint64_t)r->num_sms * 16);
    orbit_expand_kernel<Num><<<grid, 128, 0, r->compute>>>(static_cast<const unsigned char *>(wire), n_way, n_full, X, Y, out);
    r->launches++;
    return cudaGetLastError();
}

uint32_t upload_orbit(fs_renderer *r, OrbitDev &dst, int numeric, int pextras, uint64_t generation, const fs_orbit *src) {
    const size_t eb = orbit_elem_bytes(numeric, pextras);
    if (eb == 0) return FS_ERROR_UNSUPPORTED;
    free_blob(r, dst.data);
    free_blob(r, dst.fast);
    dst = OrbitDev{};
    if (pextras == FS_PEXTRAS_SIMPLE_COMPRESSION) {
        // waypoints -> device -> full orbit in the Disable layout; the staging copy is freed in stream order
        if (!src->orbit_x_low || !src->orbit_y_low || src->compressed_count == 0 ||
            src->uncompressed_count < src->compressed_count)
            return FS_ERROR_6_NO_ORBIT;
        const size_t full_eb = orbit_elem_bytes(numeric, FS_PEXTRAS_DISABLE);
        const size_t full_bytes = full_eb * src->uncompressed_count;
        void *wire = nullptr;
        cudaError_t e = cudaMallocAsync(&wire, eb * src->compressed_count, r->compute);
        if (e != cudaSuccess) return e;
        e = cudaMemcpyAsync(wire, src->elements, eb * src->compressed_count, cudaMemcpyDefault, r->compute);
        if (e != cudaSuccess) return e;
        e = alloc_table(r, dst.data, full_bytes + 64);
        if (e != cudaSuccess) return e;
        dst.data.bytes = full_bytes;
        e = cudaMemsetAsync(static_cast<char *>(dst.data.ptr) + full_bytes, 0, 64, r->compute);
        if (e != cudaSuccess) return e;
        uint32_t rc;
        switch (numeric) {
        case FS_NUM_F32: rc = expand_orbit<NumPlain<float>>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        case FS_NUM_F64: rc = expand_orbit<NumPlain<double>>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        case FS_NUM_2X32: rc = expand_orbit<Num2x32>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        case FS_NUM_HDR32: rc = expand_orbit<NumHdr<float>>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        case FS_NUM_HDR64: rc = expand_orbit<NumHdr<double>>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        case FS_NUM_HDR2X32: rc = expand_orbit<NumHdr2x32>(r, wire, src->compressed_count, src->uncompressed_count, src->orbit_x_low, src->orbit_y_low, dst.data.ptr); break;
        default: rc = FS_ERROR_UNSUPPORTED; break;
        }
        cudaFreeAsync(wire, r->compute);
        if (rc) return rc;
        if (numeric == FS_NUM_HDR32 && src->uncompressed_count > 1 && src->uncompressed_count <= scaled::kMaxElems && r->use_scaled) {
            const size_t fbytes = sizeof(scaled::FastElem) * src->uncompressed_count;
            e = cudaMallocAsync(&dst.fast.ptr, fbytes, r->compute);
            if (e != cudaSuccess) return e;
            dst.fast.bytes = fbytes;
            const uint64_t want = (src->uncompressed_count + 255) / 256;
            const unsigned grid = (unsigned)(want < (uint64_t)r->num_sms * 8 ? want : (uint64_t)r->num_sms * 8);
            build_fast_table_kernel<<<grid, 256, 0, r->compute>>>(static_cast<const uint4 *>(dst.data.ptr), src->uncompressed_count,
                                                                  static_cast<scaled::FastElem *>(dst.fast.ptr));
            r->launches++;
            e = cudaGetLastError();
            if (e != cudaSuccess) return e;
        }
        dst.compressed = src->compressed_count;
        dst.uncompressed = src->uncompressed_count;
        dst.period = src->period_maybe_zero;
        dst.numeric = numeric;
        dst.pextras = pextras;
        dst.generation = generation;
        dst.valid = true;
        return 0;
    }
    const size_t bytes = eb * src->compressed_count;
    // one zeroed element of padding: the reference's FP64 BLA kernel can read one element past the end after an
    // escaping skip (BLAKernels.cuh:128-134, its own TODO); the value there does not reach the output
    cudaError_t err = alloc_table(r, dst.data, bytes + 64);
    if (err != cudaSuccess) return err;
    dst.data.bytes = bytes;
    err = cudaMemsetAsync(static_cast<char *>(dst.data.ptr) + bytes, 0, 64, r->compute);
    if (err != cudaSuccess) return err;
    err = cudaMemcpyAsync(dst.data.ptr, src->elements, bytes, cudaMemcpyDefault, r->compute);
    if (err != cudaSuccess) return err;
    if (numeric == FS_NUM_HDR32 && pextras == FS_PEXTRAS_DISABLE && src->compressed_count > 1 &&
        src->compressed_count <= scaled::kMaxElems && r->use_scaled) {
        const size_t fbytes = sizeof(scaled::FastElem) * src->compressed_count;
        err = cudaMallocAsync(&dst.fast.ptr, fbytes, r->compute);
        if (err != cudaSuccess) return err;
        dst.fast.bytes = fbytes;
        const uint64_t want = (src->compressed_count + 255) / 256;
        const unsigned grid = (unsigned)(want < (uint64_t)r->num_sms * 8 ? want : (uint64_t)r->num_sms * 8);
        build_fast_table_kernel<<<grid, 256, 0, r->compute>>>(static_cast<const uint4 *>(dst.data.ptr), src->compressed_count,
                                                              static_cast<scaled::FastElem *>(dst.fast.ptr));
        r->launches++;
        err = cudaGetLastError();
        if (err != cudaSuccess) return err;
    }
    dst.compressed = src->compressed_count;
    dst.uncompressed = src->uncompressed_count;
    dst.period = src->period_maybe_zero;
    dst.numeric = numeric;
    dst.pextras = pextras;
    dst.generation = generation;
    dst.valid = true;
    return 0;
}

// Repack LAInfoDeep[] (reference layout) into 16-byte-aligned LaRec[] and ATInfo into AtDev.  The wire records are
// copied to the device as they are and repacked there, so the call never waits for the stream: with page-locked
// sources the whole upload is asynchronous and the render launch queues right behind it.
template <class Num, class IterT>
__global__ void __launch_bounds__(256) la_repack_kernel(const WireLA<Num, IterT> *wire, LaRec<Num, IterT> *out, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const WireLA<Num, IterT> w = wire[i];
        LaRec<Num, IterT> d;
        memset(&d, 0, sizeof(d));
        d.Ref = w.Ref; d.ZCoeff = w.ZCoeff; d.CCoeff = w.CCoeff;
        d.LAThreshold = w.LAThreshold; d.LAThresholdC = w.LAThresholdC;
        d.StepLength = w.StepLength; d.NextStageLAIndex = w.NextStageLAIndex;
        out[i] = d;
    }
}

// LaRec[] -> la2::Rec[] (fs_la_step2.cuh): 2*Ref's exponent, the next record's Ref, threshold beside the operands.
// A record whose LAThreshold mantissa is not in [1, 2) (never produced by the reference's builder: thresholds are
// reduced, LAInfoDeep.h:109-502) gets Ref = NaN, which makes la2::step refuse every step on it.
__global__ void __launch_bounds__(256) la2_pack_kernel(const LaRec<NumHdr<float>, uint32_t> *las, la2::Rec *out, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const LaRec<NumHdr<float>, uint32_t> a = las[i];
        const bool has_next = i + 1 < n;
        HdrC<float> next_ref = hc_zero<float>();
        if (has_next) next_ref = las[i + 1].Ref;
        const la2::Rec d = la2::pack(a.Ref, a.ZCoeff, a.CCoeff, a.LAThreshold, a.StepLength, a.NextStageLAIndex, has_next, next_ref);
        out[i] = d;
    }
}
__global__ void __launch_bounds__(256) la2_stage_kernel(const LaRec<NumHdr<float>, uint32_t> *las, uint64_t n_las,
                                                        const StageRec<uint32_t> *stages, uint4 *out, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const StageRec<uint32_t> s = stages[i];
        Hdr<float> thc = hdr_zero<float>();
        if (s.LAIndex < n_las) thc = las[s.LAIndex].LAThresholdC;
        out[i] = make_uint4(s.LAIndex, s.MacroItCount, __float_as_uint(thc.m), (uint32_t)thc.e);
    }
}

template <class Num, class IterT> uint32_t upload_la_typed(fs_renderer *r, const fs_la_reference *src) {
    using W = WireLA<Num, IterT>;
    using D = LaRec<Num, IterT>;
    LaDev &la = r->la;
    const size_t n = src->num_las;
    cudaError_t err = alloc_table(r, la.las, (n ? n : 1) * sizeof(D));
    if (err != cudaSuccess) return err;
    if (n) {
        void *wire = nullptr;
        err = cudaMallocAsync(&wire, n * sizeof(W), r->compute);
        if (err != cudaSuccess) return err;
        err = cudaMemcpyAsync(wire, src->las, n * sizeof(W), cudaMemcpyHostToDevice, r->compute);
        if (err != cudaSuccess) return err;
        const unsigned int grid = (unsigned int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
        la_repack_kernel<Num, IterT><<<grid, 256, 0, r->compute>>>(static_cast<const W *>(wire), static_cast<D *>(la.las.ptr), n);
        cudaFreeAsync(wire, r->compute);
    }
    const size_t sbytes = (src->num_stages ? src->num_stages : 1) * sizeof(StageRec<IterT>);
    err = alloc_table(r, la.stages, sbytes);
    if (err != cudaSuccess) return err;
    if (src->num_stages) {
        err = cudaMemcpyAsync(la.stages.ptr, src->stages, src->num_stages * sizeof(StageRec<IterT>), cudaMemcpyHostToDevice, r->compute);
        if (err != cudaSuccess) return err;
    }
    if constexpr (std::is_same<Num, NumHdr<float>>::value && sizeof(IterT) == 4) {
        if (n && src->num_stages) {
            err = alloc_table(r, la.las2, n * sizeof(la2::Rec));
            if (err != cudaSuccess) return err;
            err = alloc_table(r, la.stages2, src->num_stages * sizeof(uint4));
            if (err != cudaSuccess) return err;
            const unsigned int grid = (unsigned int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
            la2_pack_kernel<<<grid, 256, 0, r->compute>>>(static_cast<const D *>(la.las.ptr), static_cast<la2::Rec *>(la.las2.ptr), n);
            la2_stage_kernel<<<(unsigned int)((src->num_stages + 255) / 256), 256, 0, r->compute>>>(
                static_cast<const D *>(la.las.ptr), n, static_cast<const StageRec<IterT> *>(la.stages.ptr),
                static_cast<uint4 *>(la.stages2.ptr), src->num_stages);
        }
    }
    AtDev<Num, IterT> at;
    memset(&at, 0, sizeof(at));
    if (src->at) {
        WireAT<Num, IterT> w;
        memcpy(&w, src->at, sizeof(w));
        at.StepLength = w.StepLength; at.ThresholdC = w.ThresholdC; at.SqrEscapeRadius = w.SqrEscapeRadius;
        at.RefC = w.RefC; at.CCoeff = w.CCoeff; at.InvZCoeff = w.InvZCoeff;
    }
    static_assert(sizeof(at) <= sizeof(la.at), "AT image");
    memcpy(la.at, &at, sizeof(at));
    la.num_las = src->num_las;
    la.num_stages = src->num_stages;
    la.stage_count = src->la_stage_count;
    la.use_at = src->use_at && src->at;
    la.is_valid = src->is_valid;
    la.present = true;
    return 0;
}

template <class F> uint32_t dispatch_num_iter(int numeric, uint32_t iter_bytes, F &&f, bool allow_2x32 = true) {
    const bool u64 = iter_bytes == 8;
    if (!allow_2x32 && (numeric == FS_NUM_2X32 || numeric == FS_NUM_HDR2X32)) return FS_ERROR_UNSUPPORTED;
    switch (numeric) {
    case FS_NUM_F32: return u64 ? f(NumPlain<float>{}, uint64_t{}) : f(NumPlain<float>{}, uint32_t{});
    case FS_NUM_F64: return u64 ? f(NumPlain<double>{}, uint64_t{}) : f(NumPlain<double>{}, uint32_t{});
    case FS_NUM_HDR32: return u64 ? f(NumHdr<float>{}, uint64_t{}) : f(NumHdr<float>{}, uint32_t{});
    case FS_NUM_HDR64: return u64 ? f(NumHdr<double>{}, uint64_t{}) : f(NumHdr<double>{}, uint32_t{});
    case FS_NUM_2X32: return u64 ? f(Num2x32{}, uint64_t{}) : f(Num2x32{}, uint32_t{});
    case FS_NUM_HDR2X32: return u64 ? f(NumHdr2x32{}, uint64_t{}) : f(NumHdr2x32{}, uint32_t{});
    default: return FS_ERROR_UNSUPPORTED;
    }
}

uint32_t upload_la(fs_renderer *r, int numeric, uint32_t iter_bytes, const fs_la_reference *src) {
    free_blob(r, r->la.las);
    free_blob(r, r->la.stages);
    free_blob(r, r->la.las2);
    free_blob(r, r->la.stages2);
    r->la = LaDev{};
    const uint32_t rc = dispatch_num_iter(numeric, iter_bytes, [&](auto num, auto it) -> uint32_t {
        return upload_la_typed<decltype(num), decltype(it)>(r, src);
    });
    if (rc == 0) {
        r->la.numeric = numeric;
        r->la.iter_bytes = iter_bytes;
    }
    return rc;
}

// persistent grid: one 256-thread CTA per resident slot -- minus kDisplaySlots.  The render kernels never give an SM
// slot back before their queue is empty, and one warp-tile can last as long as the frame (interior pixels at a
// multi-million iteration limit), so a progressive RenderCurrent (high-priority display stream, called by the
// reference's pool once a second while the frame renders: RenderThreadPool.cpp:915-959, 1923-1948) would otherwise
// wait for the end of the render.  Two CTA slots (of 592 for the HDRx32 kernels: 0.3 % of the throughput) stay free
// for it at all times; more are freed on request where tiles turn over quickly (TileQueue::yield_quota).
constexpr int kDisplaySlots = 2;
// Kernels of two streams share an SM only if they agree on its shared-memory carve-out (it cannot change while CTAs are
// resident; measured with tools/concurrency_probe.cu: a launch whose carve-out differs waits until the SMs have drained,
// i.e. until the render is over).  The driver sizes the carve-out from the launch's occupancy -- 1 KB is reserved per
// resident CTA, so a <<<1, 1>>> launch (up to 32 CTAs per SM) asks for four times the carve-out of a 256-thread one.
// Every kernel of this library is therefore launched with 256-thread CTAs and a few bytes of static shared memory at
// most, which puts all of them in the same class; FS_CARVEOUT (a percentage) forces an explicit preference instead.
template <class K> void same_carveout(fs_renderer *r, K kernel) {
    if (r->carveout_pct >= 0) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, r->carveout_pct);
}
template <class K> int resident_ctas(fs_renderer *r, K kernel) {
    same_carveout(r, kernel);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    if (r->ctas_per_sm_cap > 0 && per_sm > r->ctas_per_sm_cap) per_sm = r->ctas_per_sm_cap;
    const int slots = per_sm * r->num_sms;
    return slots > 8 * kDisplaySlots ? slots - kDisplaySlots : slots;
}

// Grid of the LAv2 kernels: full occupancy.  (Round 1 cut the grid to 3/4 of the occupancy for shards with fewer than 8
// tiles per resident warp; with the AT cycle watch and the la2 records the full grid is faster there too: View 14 8-way
// shard 0.699 ms at 4 CTAs/SM, 0.719 at 3, 0.918 at 2; whole frame 4.23 / 4.97 / 6.68 ms.)
template <class K> int lav2_grid(fs_renderer *r, K kernel) { return resident_ctas(r, kernel); }

// Grid of the lane-refill LAv2 kernel (fs_lav2_pool.cuh): full occupancy with its per-warp pools in shared memory.
template <class K> int pool_grid(fs_renderer *r, K kernel, size_t smem) {
    same_carveout(r, kernel);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    if (r->ctas_per_sm_cap > 0 && per_sm > r->ctas_per_sm_cap) per_sm = r->ctas_per_sm_cap;
    const int slots = per_sm * r->num_sms;
    return slots > 8 * kDisplaySlots ? slots - kDisplaySlots : slots;
}

// CTAs a progressive RenderCurrent asks to leave a running persistent grid (of num_sms x 2..8 CTAs): enough slots for
// the post kernel to stream the frame in well under a millisecond, ~1 % of the render's throughput
constexpr int kYieldCtas = 8;

TileQueue render_queue(fs_renderer *r) {
    TileQueue q;
    q.counter = r->tile_counter;
    q.yield_quota = r->yield_quota;
    q.grab = 1;
    return q;
}

void begin_render(fs_renderer *r, bool streams_to_sink = false) {
    r->sink_filled = streams_to_sink && r->sink_dev != nullptr; // any other render makes the host copy stale
    r->n_frames = 1; // a zoom batch sets its own count after this
    r->selected = 0;
    // tile counter and yield quota are adjacent words: one memset
    cudaMemsetAsync(r->tile_counter, 0, 2 * sizeof(unsigned int), r->compute);
    r->yield_requested = false;
    cudaEventRecord(r->ev_start, r->compute);
}
uint32_t end_render(fs_renderer *r) {
    cudaEventRecord(r->ev_stop, r->compute);
    r->timed = true;
    r->launches++;
    return cudaGetLastError();
}

template <class T> T load_pod(const void *p) {
    T v;
    memcpy(&v, p, sizeof(T));
    return v;
}

// Arguments of the LAv2 kernels for r's orbit, tables, geometry and switches; `have_la`: the LA table matches the orbit.
template <class Num, class IterT>
Lav2Args<Num, IterT> lav2_args(fs_renderer *r, const void *dx, const void *dy, const void *cx, const void *cy, uint64_t n_iter,
                               bool &have_la) {
    using Real = typename Num::Real;
    Lav2Args<Num, IterT> A;
    memset(&A, 0, sizeof(A));
    A.out = static_cast<IterT *>(r->iter_buf);
    A.orbit = r->orbit1.data.ptr;
    A.orbit_fast = r->use_scaled ? r->orbit1.fast.ptr : nullptr;
    A.orbit_count = (IterT)r->orbit1.uncompressed;
    have_la = r->la.present && r->la.numeric == r->orbit1.numeric && r->la.iter_bytes == sizeof(IterT);
    if (have_la) {
        A.las = static_cast<const LaRec<Num, IterT> *>(r->la.las.ptr);
        A.stages = static_cast<const StageRec<IterT> *>(r->la.stages.ptr);
        memcpy(&A.at, r->la.at, sizeof(A.at));
        A.las2 = r->use_la2 ? r->la.las2.ptr : nullptr;
        A.stages2 = r->la.stages2.ptr;
        A.la_stage_count = (IterT)r->la.stage_count;
        A.la_valid = r->la.is_valid;
        A.use_at = r->la.use_at;
    }
    A.width = (int)r->width;
    A.height = (int)r->height;
    A.pitch = (int)(r->w_block * NB_THREADS_W);
    A.shard_count = (int)r->shard_count;
    A.shard_index = (int)r->shard_index;
    A.dx = load_pod<Real>(dx);
    A.dy = load_pod<Real>(dy);
    A.centerX = load_pod<Real>(cx);
    A.centerY = load_pod<Real>(cy);
    A.n_iterations = (IterT)n_iter;
    A.sink = static_cast<IterT *>(r->sink_dev);
    A.at_cycle = r->at_cycle ? 1 : 0;
    A.queue = render_queue(r);
    A.step_counter = r->count_steps ? r->step_counter : nullptr;
    return A;
}

template <class Num, class IterT>
uint32_t launch_lav2(fs_renderer *r, int mode, const void *dx, const void *dy, const void *cx, const void *cy, uint64_t n_iter) {
    bool have_la = false;
    Lav2Args<Num, IterT> A = lav2_args<Num, IterT>(r, dx, dy, cx, cy, n_iter, have_la);
    const bool count = r->count_steps;
    // two-launch form (AT, then everything else) for the float+exponent binary32 type when the table has an AT block
    if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) {
        if (r->split_at && have_la && A.la_valid && A.use_at && (mode == FS_LAV2_FULL || mode == FS_LAV2_LAO)) {
            const size_t need = r->n_cu * sizeof(float4);
            if (r->at_state.bytes < need) {
                free_blob(r, r->at_state);
                cudaError_t e = cudaMallocAsync(&r->at_state.ptr, need, r->compute);
                if (e != cudaSuccess) return e;
                r->at_state.bytes = need;
            }
            A.at_state = static_cast<float4 *>(r->at_state.ptr);
            begin_render(r, true);
#define FS_LAUNCH_SPLIT(MODE, COUNT)                                                                                   \
    {                                                                                                                  \
        auto ka = lav2_kernel<Num, IterT, MODE, COUNT, AtPhase::AtOnly>;                                               \
        ka<<<lav2_grid(r, ka), 256, 0, r->compute>>>(A);                                                           \
        cudaMemsetAsync(r->tile_counter, 0, sizeof(unsigned int), r->compute);                                        \
        auto kb = lav2_kernel<Num, IterT, MODE, COUNT, AtPhase::AfterAt>;                                              \
        kb<<<lav2_grid(r, kb), 256, 0, r->compute>>>(A);                                                           \
    }
            if (mode == FS_LAV2_FULL) { if (count) FS_LAUNCH_SPLIT(Lav2Mode::Full, true) else FS_LAUNCH_SPLIT(Lav2Mode::Full, false) }
            else { if (count) FS_LAUNCH_SPLIT(Lav2Mode::LAO, true) else FS_LAUNCH_SPLIT(Lav2Mode::LAO, false) }
#undef FS_LAUNCH_SPLIT
            r->launches++;
            return end_render(r);
        }
    }
    // float+exponent binary32: the lane-refill kernel (fs_lav2_pool.cuh); pixel coordinates travel as 16 + 16 bits
    if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) {
        if (r->use_pool && r->width < 65536u && r->height < 65536u) {
            begin_render(r, true);
            const size_t smem = pool::Layout<IterT>::kCtaBytes;
#define FS_LAUNCH_POOL(MODE)                                                                                           \
    if (count) { auto k = lav2_pool_kernel<IterT, MODE, true>; k<<<pool_grid(r, k, smem), 256, smem, r->compute>>>(A); } \
    else { auto k = lav2_pool_kernel<IterT, MODE, false>; k<<<pool_grid(r, k, smem), 256, smem, r->compute>>>(A); }
            switch (mode) {
            case FS_LAV2_FULL: FS_LAUNCH_POOL(Lav2Mode::Full) break;
            case FS_LAV2_PO: FS_LAUNCH_POOL(Lav2Mode::PO) break;
            case FS_LAV2_LAO: FS_LAUNCH_POOL(Lav2Mode::LAO) break;
            default: return FS_ERROR_UNSUPPORTED;
            }
#undef FS_LAUNCH_POOL
            return end_render(r);
        }
    }
    begin_render(r, true);
    // small shards of the float+exponent binary32 path: cost probe + expensive-tiles-first queue order (lav2_probe_kernel)
    if constexpr (Num::kHdr && !Num::kDf && sizeof(typename Num::Mant) == 4) {
        const uint64_t tiles_x = (r->width + 7) / 8;
        const uint64_t bands = ((r->height + 3) / 4 + r->shard_count - 1 - r->shard_index) / r->shard_count;
        const uint64_t n_tiles = tiles_x * bands;
        const uint64_t warps = (uint64_t)resident_ctas(r, lav2_kernel<Num, IterT, Lav2Mode::Full, false>) * 8;
        const uint64_t at_step = have_la && A.la_valid && A.use_at ? (uint64_t)A.at.StepLength : 0;
        if (r->probe_passes > 0 && at_step > 0 && (mode == FS_LAV2_FULL || mode == FS_LAV2_LAO) && n_tiles < 16 * warps &&
            n_tiles <= 64ull * 1024ull && n_iter / at_step > 4ull * (uint64_t)r->probe_passes) {
            const size_t need = (2 * n_tiles + 2) * sizeof(unsigned int);
            cudaError_t e = cudaSuccess;
            if (r->tile_order.bytes < need) {
                free_blob(r, r->tile_order);
                e = cudaMallocAsync(&r->tile_order.ptr, need, r->compute);
                if (e == cudaSuccess) r->tile_order.bytes = need;
            }
            if (e == cudaSuccess) {
                unsigned int *order = static_cast<unsigned int *>(r->tile_order.ptr);
                unsigned int *heads = order + 2 * n_tiles;
                cudaMemsetAsync(heads, 0, 2 * sizeof(unsigned int), r->compute);
                Lav2Args<Num, IterT> P = A;
                P.n_iterations = (IterT)((uint64_t)r->probe_passes * at_step);
                P.at_cycle = 1;
                P.step_counter = nullptr;
                auto kp = lav2_probe_kernel<IterT>;
                same_carveout(r, kp);
                kp<<<(unsigned int)((n_tiles * 4 + 255) / 256), 256, 0, r->compute>>>(P, order, heads);
                lav2_order_kernel<<<1, 1024, 0, r->compute>>>(order, heads, (unsigned int)n_tiles);
                r->launches += 2;
                A.order = order;
            }
        }
    }
#define FS_LAUNCH_LAV2(MODE)                                                                                           \
    if (count) { auto k = lav2_kernel<Num, IterT, MODE, true>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); }         \
    else { auto k = lav2_kernel<Num, IterT, MODE, false>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); }
    switch (mode) {
    case FS_LAV2_FULL: FS_LAUNCH_LAV2(Lav2Mode::Full) break;
    case FS_LAV2_PO: FS_LAUNCH_LAV2(Lav2Mode::PO) break;
    case FS_LAV2_LAO: FS_LAUNCH_LAV2(Lav2Mode::LAO) break;
    default: return FS_ERROR_UNSUPPORTED;
    }
#undef FS_LAUNCH_LAV2
    return end_render(r);
}

// A zoom batch: n_frames frames of r's orbit and tables in one launch of lav2_kernel<..., Lav2Layout::Frames>.  `dx` ... `cy`
// hold n_frames PODs each.  The batch always runs the fused tile kernel: the split-AT, lane-refill and probe-order
// switches of launch_lav2 only change how a single frame is scheduled, never its cells, so a batch ignores them.
template <class Num, class IterT>
uint32_t launch_lav2_frames(fs_renderer *r, int mode, uint32_t n_frames, const void *dx, const void *dy, const void *cx,
                            const void *cy, uint64_t n_iter) {
    using Real = typename Num::Real;
    using Frame = Lav2Frame<Num, IterT>;
    if (mode != FS_LAV2_FULL && mode != FS_LAV2_PO && mode != FS_LAV2_LAO) return FS_ERROR_UNSUPPORTED;
    const uint64_t bands = ((r->height + 3) / 4 + r->shard_count - 1 - r->shard_index) / r->shard_count;
    if ((r->width + 7) / 8 * bands * n_frames >= (1ull << 31)) return FS_ERROR_UNSUPPORTED; // tickets are 32-bit
    const size_t frame_bytes = r->n_cu * r->iter_bytes;
    if (r->stack_frames < n_frames - 1) {
        // a progressive RenderCurrent may still be reading a frame of the old stack on the display stream
        cudaStreamSynchronize(r->display);
        if (r->frame_stack) cudaFreeAsync(r->frame_stack, r->compute);
        r->frame_stack = nullptr;
        r->stack_frames = 0;
        cudaError_t err = cudaMallocAsync(&r->frame_stack, (n_frames - 1) * frame_bytes, r->compute);
        if (err != cudaSuccess) return err;
        err = cudaMemsetAsync(r->frame_stack, 0, (n_frames - 1) * frame_bytes, r->compute);
        if (err != cudaSuccess) return err;
        r->stack_frames = n_frames - 1;
        cudaEventRecord(r->ev_alloc, r->compute);
        cudaStreamWaitEvent(r->display, r->ev_alloc, 0);
    }
    const size_t recs_bytes = (size_t)FS_MAX_FRAMES * sizeof(Frame);
    if (r->frame_recs.bytes < recs_bytes) {
        free_blob(r, r->frame_recs);
        cudaError_t err = cudaMallocAsync(&r->frame_recs.ptr, recs_bytes, r->compute);
        if (err != cudaSuccess) return err;
        r->frame_recs.bytes = recs_bytes;
    }
    Frame recs[FS_MAX_FRAMES];
    for (uint32_t f = 0; f < n_frames; f++) {
        recs[f].dx = load_pod<Real>(static_cast<const char *>(dx) + f * sizeof(Real));
        recs[f].dy = load_pod<Real>(static_cast<const char *>(dy) + f * sizeof(Real));
        recs[f].centerX = load_pod<Real>(static_cast<const char *>(cx) + f * sizeof(Real));
        recs[f].centerY = load_pod<Real>(static_cast<const char *>(cy) + f * sizeof(Real));
        recs[f].out = static_cast<IterT *>(f == 0 ? r->iter_buf : static_cast<char *>(r->frame_stack) + (f - 1) * frame_bytes);
    }
    cudaError_t err = cudaMemcpyAsync(r->frame_recs.ptr, recs, n_frames * sizeof(Frame), cudaMemcpyHostToDevice, r->compute);
    if (err != cudaSuccess) return err;
    bool have_la = false;
    Lav2Args<Num, IterT> A = lav2_args<Num, IterT>(r, dx, dy, cx, cy, n_iter, have_la);
    A.out = nullptr;
    A.sink = nullptr;
    A.frames = static_cast<const Frame *>(r->frame_recs.ptr);
    A.n_frames = n_frames;
    begin_render(r);
    r->n_frames = n_frames;
    const bool count = r->count_steps;
#define FS_LAUNCH_FRAMES(MODE)                                                                                         \
    if (count) { auto k = lav2_kernel<Num, IterT, MODE, true, AtPhase::Fused, Lav2Layout::Frames>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); } \
    else { auto k = lav2_kernel<Num, IterT, MODE, false, AtPhase::Fused, Lav2Layout::Frames>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); }
    switch (mode) {
    case FS_LAV2_FULL: FS_LAUNCH_FRAMES(Lav2Mode::Full) break;
    case FS_LAV2_PO: FS_LAUNCH_FRAMES(Lav2Mode::PO) break;
    default: FS_LAUNCH_FRAMES(Lav2Mode::LAO) break;
    }
#undef FS_LAUNCH_FRAMES
    return end_render(r);
}

// An exponential map: one frame of lav2_kernel<..., Lav2Layout::ExpMap>, pixel (X, Y) at dc = expmap_dc(radius[Y],
// dir_x[X], dir_y[X]).  The tables are copied into renderer-owned device memory before the call returns.  Like a zoom
// batch it always runs the fused tile kernel (the split-AT, lane-refill and probe-order switches change scheduling, never
// cells); otherwise it is a single-frame render: frame 0, the result sink, the shard rule.
template <class Num, class IterT>
uint32_t launch_lav2_expmap(fs_renderer *r, int mode, const void *radius, const void *dir_x, const void *dir_y,
                            uint64_t n_iter) {
    using Real = typename Num::Real;
    const uint64_t bands = ((r->height + 3) / 4 + r->shard_count - 1 - r->shard_index) / r->shard_count;
    if ((r->width + 7) / 8 * bands >= (1ull << 31)) return FS_ERROR_UNSUPPORTED; // tickets are 32-bit
    const size_t h_bytes = (size_t)r->height * sizeof(Real), w_bytes = (size_t)r->width * sizeof(Real);
    const size_t need = h_bytes + 2 * w_bytes;
    if (r->expmap_tables.bytes < need) {
        free_blob(r, r->expmap_tables);
        cudaError_t err = cudaMallocAsync(&r->expmap_tables.ptr, need, r->compute);
        if (err != cudaSuccess) return err;
        r->expmap_tables.bytes = need;
    }
    // one staging copy in pageable memory: cudaMemcpyAsync has consumed it when it returns, whatever memory the caller's
    // tables are in, so the caller may reuse them at once
    std::vector<unsigned char> host(need);
    memcpy(host.data(), radius, h_bytes);
    memcpy(host.data() + h_bytes, dir_x, w_bytes);
    memcpy(host.data() + h_bytes + w_bytes, dir_y, w_bytes);
    cudaError_t err = cudaMemcpyAsync(r->expmap_tables.ptr, host.data(), need, cudaMemcpyHostToDevice, r->compute);
    if (err != cudaSuccess) return err;
    bool have_la = false;
    Real unused;
    memset(&unused, 0, sizeof(unused));
    Lav2Args<Num, IterT> A = lav2_args<Num, IterT>(r, &unused, &unused, &unused, &unused, n_iter, have_la);
    const unsigned char *tables = static_cast<const unsigned char *>(r->expmap_tables.ptr);
    A.exp_radius = reinterpret_cast<const Real *>(tables);
    A.exp_dir_x = reinterpret_cast<const Real *>(tables + h_bytes);
    A.exp_dir_y = reinterpret_cast<const Real *>(tables + h_bytes + w_bytes);
    begin_render(r, true);
    const bool count = r->count_steps;
#define FS_LAUNCH_EXPMAP(MODE)                                                                                         \
    if (count) { auto k = lav2_kernel<Num, IterT, MODE, true, AtPhase::Fused, Lav2Layout::ExpMap>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); } \
    else { auto k = lav2_kernel<Num, IterT, MODE, false, AtPhase::Fused, Lav2Layout::ExpMap>; k<<<lav2_grid(r, k), 256, 0, r->compute>>>(A); }
    switch (mode) {
    case FS_LAV2_FULL: FS_LAUNCH_EXPMAP(Lav2Mode::Full) break;
    case FS_LAV2_PO: FS_LAUNCH_EXPMAP(Lav2Mode::PO) break;
    default: FS_LAUNCH_EXPMAP(Lav2Mode::LAO) break;
    }
#undef FS_LAUNCH_EXPMAP
    return end_render(r);
}

// GPU_BLAS upload (BLA.cuh:123-160) + launch (GPU_Render.cu:1462-1570).  The wire records are copied level by
// level into one device buffer and repacked there into the aligned head/coefficient arrays of fs_bla.cuh.
template <class Num, class IterT>
uint32_t launch_bla(fs_renderer *r, const fs_blas *blas, const void *dx, const void *dy, const void *cx, const void *cy,
                    uint64_t n_iter) {
    using Real = typename Num::Real;
    using Wire = BlaWire<Num>;
    if (blas->num_levels > (uint32_t)kBlaMaxLevels || blas->lm2 < 0 || blas->lm2 > 30) return FS_ERROR_UNSUPPORTED;
    BlaArgs<Num, IterT> A;
    memset(&A, 0, sizeof(A));
    uint64_t total = 0;
    for (uint32_t i = 0; i < blas->num_levels; i++) {
        A.level_off[i] = total;
        if (blas->levels[i]) total += blas->level_counts[i];
    }
    free_blob(r, r->bla_raw);
    free_blob(r, r->bla_heads);
    free_blob(r, r->bla_coefs);
    const uint64_t alloc_n = total ? total : 1;
    cudaError_t err = cudaMallocAsync(&r->bla_raw.ptr, alloc_n * sizeof(Wire), r->compute);
    if (err != cudaSuccess) return err;
    err = cudaMallocAsync(&r->bla_heads.ptr, alloc_n * sizeof(BlaHead<Num>), r->compute);
    if (err != cudaSuccess) return err;
    err = cudaMallocAsync(&r->bla_coefs.ptr, alloc_n * sizeof(BlaCoef<Num>), r->compute);
    if (err != cudaSuccess) return err;
    for (uint32_t i = 0; i < blas->num_levels; i++) {
        if (!blas->levels[i] || !blas->level_counts[i]) continue;
        err = cudaMemcpyAsync(static_cast<Wire *>(r->bla_raw.ptr) + A.level_off[i], blas->levels[i],
                              blas->level_counts[i] * sizeof(Wire), cudaMemcpyDefault, r->compute);
        if (err != cudaSuccess) return err;
    }
    if (total) {
        const uint64_t want = (total + 255) / 256;
        const unsigned grid = (unsigned)(want < (uint64_t)r->num_sms * 8 ? want : (uint64_t)r->num_sms * 8);
        bla_repack_kernel<Num><<<grid, 256, 0, r->compute>>>(static_cast<const Wire *>(r->bla_raw.ptr), total,
                                                            static_cast<BlaHead<Num> *>(r->bla_heads.ptr),
                                                            static_cast<BlaCoef<Num> *>(r->bla_coefs.ptr));
        r->launches++;
    }
    A.out = static_cast<IterT *>(r->iter_buf);
    A.orbit = r->bla_orbit.data.ptr;
    A.orbit_count = (IterT)r->bla_orbit.uncompressed;
    A.heads = static_cast<const BlaHead<Num> *>(r->bla_heads.ptr);
    A.coefs = static_cast<const BlaCoef<Num> *>(r->bla_coefs.ptr);
    A.lm2 = blas->lm2;
    A.width = (int)r->width;
    A.height = (int)r->height;
    A.pitch = (int)(r->w_block * NB_THREADS_W);
    A.shard_count = (int)r->shard_count;
    A.shard_index = (int)r->shard_index;
    A.dx = load_pod<Real>(dx);
    A.dy = load_pod<Real>(dy);
    A.centerX = load_pod<Real>(cx);
    A.centerY = load_pod<Real>(cy);
    A.n_iterations = (IterT)n_iter;
    A.queue = render_queue(r);
    A.step_counter = r->count_steps ? r->step_counter : nullptr;
    A.cycle_watch = r->at_cycle ? 1 : 0;
    A.fast = r->use_la2 ? 1 : 0; // the A/B switch of the select-free forms (fs_set_la_step2) covers this loop too
    begin_render(r);
    if (r->count_steps) { auto k = bla_kernel<Num, IterT, true>; k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A); }
    else { auto k = bla_kernel<Num, IterT, false>; k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A); }
    return end_render(r);
}

// RenderPerturbBLAScaled launch (GPU_Render.cu:1352-1375); both orbits were uploaded by the caller below
template <class Num, class IterT>
uint32_t launch_scaled(fs_renderer *r, const void *dx, const void *dy, const void *cx, const void *cy, uint64_t n_iter) {
    using Real = typename Num::Real;
    ScaledArgs<Num, IterT> A;
    memset(&A, 0, sizeof(A));
    A.out = static_cast<IterT *>(r->iter_buf);
    A.orbit_f = static_cast<const ScaledElemF *>(r->scaled_orbit_f.data.ptr);
    A.orbit_t = static_cast<const unsigned char *>(r->bla_orbit.data.ptr);
    A.orbit_count = (IterT)r->scaled_orbit_f.uncompressed;
    A.width = (int)r->width;
    A.height = (int)r->height;
    A.pitch = (int)(r->w_block * NB_THREADS_W);
    A.shard_count = (int)r->shard_count;
    A.shard_index = (int)r->shard_index;
    A.dx = load_pod<Real>(dx);
    A.dy = load_pod<Real>(dy);
    A.centerX = load_pod<Real>(cx);
    A.centerY = load_pod<Real>(cy);
    A.n_iterations = (IterT)n_iter;
    A.queue = render_queue(r);
    A.step_counter = r->count_steps ? r->step_counter : nullptr;
    begin_render(r);
    if (r->count_steps) { auto k = scaled_kernel<Num, IterT, true>; k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A); }
    else { auto k = scaled_kernel<Num, IterT, false>; k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A); }
    return end_render(r);
}

template <class M, class IterT, int P>
void launch_direct_p(fs_renderer *r, const DirectArgs<M, IterT> &A) {
    auto k = direct_kernel<M, IterT, P>;
    k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A);
}

template <class M, class IterT>
uint32_t launch_direct(fs_renderer *r, const void *cx, const void *cy, const void *dx, const void *dy, uint64_t n_iter, int prec) {
    // the reference launches nothing for precisions other than 1/4/8/16 (GPU_Render.cu:633-668)
    if (prec != 1 && prec != 4 && prec != 8 && prec != 16) return 0;
    DirectArgs<M, IterT> A;
    memset(&A, 0, sizeof(A));
    A.out = static_cast<IterT *>(r->iter_buf);
    A.width = (int)r->width;
    A.height = (int)r->height;
    A.pitch = (int)(r->w_block * NB_THREADS_W);
    A.shard_count = (int)r->shard_count;
    A.shard_index = (int)r->shard_index;
    A.cx = load_pod<M>(cx); A.cy = load_pod<M>(cy); A.dx = load_pod<M>(dx); A.dy = load_pod<M>(dy);
    A.n_iterations = (IterT)n_iter;
    A.queue = render_queue(r);
    A.step_counter = r->count_steps ? r->step_counter : nullptr;
    begin_render(r);
    switch (prec) {
    case 1: launch_direct_p<M, IterT, 1>(r, A); break;
    case 4: launch_direct_p<M, IterT, 4>(r, A); break;
    case 8: launch_direct_p<M, IterT, 8>(r, A); break;
    default: launch_direct_p<M, IterT, 16>(r, A); break;
    }
    return end_render(r);
}

template <class Pixel, class IterT>
uint32_t launch_direct_ext(fs_renderer *r, const typename Pixel::Coord &cx, const typename Pixel::Coord &cy,
                           const typename Pixel::Coord &dx, const typename Pixel::Coord &dy, uint64_t n_iter) {
    DirectExtArgs<typename Pixel::Coord, IterT> A;
    memset(&A, 0, sizeof(A));
    A.out = static_cast<IterT *>(r->iter_buf);
    A.width = (int)r->width;
    A.height = (int)r->height;
    A.pitch = (int)(r->w_block * NB_THREADS_W);
    A.shard_count = (int)r->shard_count;
    A.shard_index = (int)r->shard_index;
    A.cx = cx; A.cy = cy; A.dx = dx; A.dy = dy;
    A.n_iterations = (IterT)n_iter;
    A.queue = render_queue(r);
    A.step_counter = r->count_steps ? r->step_counter : nullptr;
    begin_render(r);
    auto k = direct_ext_kernel<Pixel, IterT>;
    k<<<resident_ctas(r, k), 256, 0, r->compute>>>(A);
    return end_render(r);
}

// HDRFloat<CudaDblflt>(const HDRFloat<double>&): mantissa through MattDblflt(double) (dblflt.h:37-52), exponent kept.
// Host-side, as in GPURenderer::Render (GPU_Render.cu:799-803).
Hdr<df32> hdr2x32_from_hdr64(const void *p) {
    const Hdr<double> v = load_pod<Hdr<double>>(p);
    const float a = (float)v.m;
    const float b = (float)(v.m - (double)a);
    Hdr<df32> r;
    volatile float head = a + b;
    volatile float t1 = head - a;
    volatile float t2 = head - t1;
    t1 = b - t1;
    t2 = a - t2;
    r.m.head = head;
    r.m.tail = t1 + t2;
    r.e = v.e;
    return r;
}

template <class Pixel> uint32_t launch_direct_ext_pods(fs_renderer *r, const void *cx, const void *cy, const void *dx,
                                                       const void *dy, uint64_t n_iter) {
    using Cd = typename Pixel::Coord;
    return r->iter_bytes == 8
               ? launch_direct_ext<Pixel, uint64_t>(r, load_pod<Cd>(cx), load_pod<Cd>(cy), load_pod<Cd>(dx), load_pod<Cd>(dy), n_iter)
               : launch_direct_ext<Pixel, uint32_t>(r, load_pod<Cd>(cx), load_pod<Cd>(cy), load_pod<Cd>(dx), load_pod<Cd>(dy), n_iter);
}

// Colours and Min/Max/Sum of the 4-row bands b % shard_count == shard_index (1, 0: the whole frame) of r's buffers, or of
// the iteration cells at `iters` (r's geometry) when given.
template <class IterT>
uint32_t run_post(fs_renderer *r, uint64_t n_iter, cudaStream_t stream, bool colors, uint32_t shard_count, uint32_t shard_index,
                  const void *iters = nullptr) {
    same_carveout(r, reduction_init_kernel<IterT>);
    same_carveout(r, post_kernel<IterT, 1>);
    same_carveout(r, post_kernel<IterT, 2>);
    same_carveout(r, post_kernel<IterT, 3>);
    same_carveout(r, post_kernel<IterT, 4>);
    reduction_init_kernel<IterT><<<1, 256, 0, stream>>>(r->red_dev); // 256 threads: same carve-out class as the render kernels
    const int pitch = (int)(r->w_block * NB_THREADS_W);
    const int grid = r->num_sms * 8;
    const IterT *it = static_cast<const IterT *>(iters ? iters : selected_iter_buf(r));
#define FS_POST_ARGS (it, pitch, r->color_buf, r->pal_dev, r->pal_iters, r->aux_depth, (int)r->color_w, (int)r->color_h, (IterT)n_iter, r->red_dev, (int)shard_count, (int)shard_index)
#define FS_POST(AA)                                                                                                    \
    if (colors) post_kernel<IterT, AA, true><<<grid, 256, 0, stream>>> FS_POST_ARGS;                                    \
    else { same_carveout(r, post_kernel<IterT, AA, false>); post_kernel<IterT, AA, false><<<grid, 256, 0, stream>>> FS_POST_ARGS; }
    switch (r->aa) {
    case 1: FS_POST(1); break;
    case 2: FS_POST(2); break;
    case 3: FS_POST(3); break;
    default: FS_POST(4); break;
    }
#undef FS_POST
#undef FS_POST_ARGS
    r->launches += 2;
    return cudaGetLastError();
}

template <class IterT> void preload_post_kernels_typed() {
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, reduction_init_kernel<IterT>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 1>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 2>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 3>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 4>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 1, false>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 2, false>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 3, false>);
    cudaFuncGetAttributes(&fa, post_kernel<IterT, 4, false>);
}
void preload_post_kernels(fs_renderer *r) {
    if (r->iter_bytes == 8) preload_post_kernels_typed<uint64_t>();
    else preload_post_kernels_typed<uint32_t>();
}

// FP32 issue-rate probe: 16 independent FFMA chains per thread, no memory traffic.
__global__ void __launch_bounds__(256) ffma_peak_kernel(float *sink, int iters, float seed) {
    float a[16];
#pragma unroll
    for (int k = 0; k < 16; k++) a[k] = seed + (float)(threadIdx.x + k);
    const float m = 0.999f, c = 0.001f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) a[k] = __fmaf_rn(a[k], m, c);
    }
    float s = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) s += a[k];
    if (s == 12345.678f) *sink = s;
}

// FP64 issue-rate probe: the same shape with DFMA chains.
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *sink, int iters, double seed) {
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; k++) a[k] = seed + (double)(threadIdx.x + k);
    const double m = 0.999, c = 0.001;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) a[k] = __fma_rn(a[k], m, c);
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) s += a[k];
    if (s == 12345.678) *sink = s;
}

void CUDART_CB done_trampoline(void *p) {
    fs_renderer *r = static_cast<fs_renderer *>(p);
    if (r->cb) r->cb(r->cb_user);
}

bool is_group(const fs_renderer *r) { return r && !r->members.empty(); }

// Runs f on every member in order; the first non-zero status is the group's.
template <class F> uint32_t each_member(fs_renderer *grp, F &&f) {
    uint32_t first = 0;
    for (fs_renderer *m : grp->members) {
        const uint32_t rc = f(m);
        if (rc && !first) first = rc;
    }
    return first;
}

// Makes `to`'s stream wait for everything enqueued so far on member i's stream `from`.
cudaError_t join_member(fs_renderer *grp, size_t i, cudaStream_t from, cudaStream_t to) {
    fs_renderer *m = grp->members[i];
    DeviceGuard g(m->device);
    cudaError_t err = cudaEventRecord(grp->joins[i], from);
    if (err != cudaSuccess) return err;
    return cudaStreamWaitEvent(to, grp->joins[i], 0);
}


void sync_members(fs_renderer *grp, bool display_too = false) {
    for (fs_renderer *m : grp->members) {
        if (!m->compute) continue;
        DeviceGuard g(m->device);
        cudaStreamSynchronize(m->compute);
        if (display_too) cudaStreamSynchronize(m->display);
    }
}

// Group state that needs the members' streams: the join events, the reduction parts on the lead and, at AA 3, the gather
// buffers.  The combine kernel is loaded here for the reason preload_post_kernels gives.
cudaError_t prepare_group(fs_renderer *grp) {
    fs_renderer *lead = grp->members[0];
    const size_t n = grp->members.size();
    if (!grp->red_parts) {
        grp->joins.assign(n, nullptr);
        for (size_t i = 0; i < n; i++) {
            DeviceGuard g(grp->members[i]->device);
            cudaError_t err = cudaEventCreateWithFlags(&grp->joins[i], cudaEventDisableTiming);
            if (err != cudaSuccess) return err;
        }
        DeviceGuard g(lead->device);
        for (cudaEvent_t &e : grp->lead_marks) {
            cudaError_t err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            if (err != cudaSuccess) return err;
        }
        cudaFuncAttributes fa;
        cudaFuncGetAttributes(&fa, reduction_combine_kernel);
        cudaError_t err = cudaMalloc(&grp->red_parts, 2 * (n + 1) * sizeof(Reduction));
        if (err != cudaSuccess) return err;
    }
    const size_t want = lead->aa == 3 ? lead->n_cu * lead->iter_bytes : 0;
    if (grp->gather_bytes == want) return cudaSuccess;
    sync_members(grp, true); // no member may still be writing into the old buffers
    DeviceGuard g(lead->device);
    for (void *&b : grp->gather) {
        if (b) cudaFree(b);
        b = nullptr;
    }
    grp->gather_bytes = 0;
    for (void *&b : grp->gather) {
        if (!want) break;
        cudaError_t err = cudaMalloc(&b, want);
        if (err != cudaSuccess) return err;
    }
    grp->gather_bytes = want;
    return cudaSuccess;
}

} // namespace

// ---- per-operation self-test (fs_selftest_numeric_op) -------------------------------------------------------------
// One operation of the device numeric types on arrays of operands, evaluated with the functions the render kernels
// call (fs_types.cuh, fs_df32.cuh, fs_qd.cuh).  tests/test_gpu_parity.py compares the results with the oracle's
// restatement of the reference's HDRFloat / HDRFloatComplex / dblflt / dbldbl routines, bit for bit; the Quad<F> ops
// (60-67, 70-77) have no restatement and are compared with the host build of fs_qd.cuh and with exact arithmetic
// (tests/test_exact_escape.py).
namespace {
struct SelfHf { float m; int32_t e; };
struct SelfHc { float re, im; int32_t e; };
__global__ void numeric_op_kernel(uint32_t op, const void *a_, const void *b_, void *out_, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    auto hf = [](const void *p, uint64_t k) { const SelfHf v = static_cast<const SelfHf *>(p)[k]; return hdr_make<float>(v.e, v.m); };
    auto hc = [](const void *p, uint64_t k) { const SelfHc v = static_cast<const SelfHc *>(p)[k]; HdrC<float> c; c.re = v.re; c.im = v.im; c.e = v.e; return c; };
    auto put_hf = [&](Hdr<float> v) { static_cast<SelfHf *>(out_)[i] = SelfHf{v.m, v.e}; };
    auto put_hc = [&](HdrC<float> v) { static_cast<SelfHc *>(out_)[i] = SelfHc{v.re, v.im, v.e}; };
    const df32 *da = static_cast<const df32 *>(a_), *db = static_cast<const df32 *>(b_);
    const dd64 *qa = static_cast<const dd64 *>(a_), *qb = static_cast<const dd64 *>(b_);
    switch (op) {
    case 0: put_hf(add(hf(a_, i), hf(b_, i))); break;
    case 1: put_hf(sub(hf(a_, i), hf(b_, i))); break;
    case 2: put_hf(mul(hf(a_, i), hf(b_, i))); break;
    case 3: put_hf(square(hf(a_, i))); break;
    case 4: { Hdr<float> v = hf(a_, i); reduce(v); put_hf(v); break; }
    case 5: put_hf(div(hf(a_, i), hf(b_, i))); break;
    case 6: put_hf(hdr_make<float>(cmp_pr(hf(a_, i), hf(b_, i)), 0.0f)); break;
    case 10: put_hc(add(hc(a_, i), hc(b_, i))); break;
    case 11: put_hc(mul(hc(a_, i), hc(b_, i))); break;
    case 12: { HdrC<float> v = hc(a_, i); reduce(v); put_hc(v); break; }
    case 13: { const Hdr<float> c = cheb(hc(a_, i)); HdrC<float> v; v.re = c.m; v.im = 0.0f; v.e = c.e; put_hc(v); break; }
    case 14: { const HdrC<float> f = hc(b_, i); put_hc(mul(hc(a_, i), hdr_make<float>(f.e, f.re))); break; }
    case 20: static_cast<df32 *>(out_)[i] = df_add(da[i], db[i]); break;
    case 21: static_cast<df32 *>(out_)[i] = df_sub(da[i], db[i]); break;
    case 22: static_cast<df32 *>(out_)[i] = df_mul(da[i], db[i]); break;
    case 23: static_cast<df32 *>(out_)[i] = df_sqr(da[i]); break;
    case 40: { // the perturbation step of the HDRx32 kernels: a = {dX, dY, Zx}, b = {Zy, cX, cY}
        Hdr<float> dx = hf(a_, 3 * i), dy = hf(a_, 3 * i + 1);
        NumHdr<float>::perturb(dx, dy, hf(a_, 3 * i + 2), hf(b_, 3 * i), hf(b_, 3 * i + 1), hf(b_, 3 * i + 2));
        SelfHf *o = static_cast<SelfHf *>(out_) + 3 * i;
        o[0] = SelfHf{dx.m, dx.e}; o[1] = SelfHf{dy.m, dy.e}; o[2] = SelfHf{0.0f, 0};
        break;
    }
    case 50: case 51: case 52: case 53: case 54: case 55: case 56: { // HDRFloat<double>: {double mantissa; int32 exp; pad}
        struct Wire { double m; int32_t e; int32_t pad; };
        const Wire wa = static_cast<const Wire *>(a_)[i], wb = static_cast<const Wire *>(b_)[i];
        const Hdr<double> x = hdr_make<double>(wa.e, wa.m), y = hdr_make<double>(wb.e, wb.m);
        Hdr<double> r = hdr_make<double>(0, 0.0);
        switch (op) {
        case 50: r = add(x, y); break;
        case 51: r = sub(x, y); break;
        case 52: r = mul(x, y); break;
        case 53: r = square(x); break;
        case 54: r = x; reduce(r); break;
        case 55: r = div(x, y); break;
        default: r = hdr_make<double>(cmp_pr(x, y), 0.0); break;
        }
        static_cast<Wire *>(out_)[i] = Wire{r.m, r.e, 0};
        break;
    }
    case 80: case 81: case 82: case 83: case 84: case 85: { // perturbation policies, 128-byte records (fs_num.cuh)
        const unsigned char *in = static_cast<const unsigned char *>(a_) + (size_t)kPerturbRecordBytes * i;
        unsigned char *o = static_cast<unsigned char *>(out_) + (size_t)kPerturbRecordBytes * i;
        switch (op) {
        case 80: perturb_selftest<NumPlain<float>>(in, o); break;
        case 81: perturb_selftest<NumPlain<double>>(in, o); break;
        case 82: perturb_selftest<NumHdr<float>>(in, o); break;
        case 83: perturb_selftest<NumHdr<double>>(in, o); break;
        case 84: perturb_selftest<Num2x32>(in, o); break;
        default: perturb_selftest<NumHdr2x32>(in, o); break;
        }
        break;
    }
    case 86: case 87: case 88: case 89: case 90: case 91: { // exp-map pixel -> dc (fs_num.cuh expmap_dc), 32-byte elements
        const size_t at = (size_t)kExpmapRecordBytes * i;
        const unsigned char *a = static_cast<const unsigned char *>(a_) + at, *b = static_cast<const unsigned char *>(b_) + at;
        unsigned char *o = static_cast<unsigned char *>(out_) + at;
        switch (op) {
        case 86: expmap_selftest<NumPlain<float>>(a, b, o); break;
        case 87: expmap_selftest<NumPlain<double>>(a, b, o); break;
        case 88: expmap_selftest<NumHdr<float>>(a, b, o); break;
        case 89: expmap_selftest<NumHdr<double>>(a, b, o); break;
        case 90: expmap_selftest<Num2x32>(a, b, o); break;
        default: expmap_selftest<NumHdr2x32>(a, b, o); break;
        }
        break;
    }
    case 30: static_cast<dd64 *>(out_)[i] = dd_add(qa[i], qb[i]); break;
    case 31: static_cast<dd64 *>(out_)[i] = dd_sub(qa[i], qb[i]); break;
    case 32: static_cast<dd64 *>(out_)[i] = dd_mul(qa[i], qb[i]); break;
    case 60: case 61: case 62: case 63: case 64: case 65: case 66: case 67:
        static_cast<Quad<double> *>(out_)[i] = quad_selftest_op<double>(op - 60, static_cast<const Quad<double> *>(a_)[i],
                                                                        static_cast<const Quad<double> *>(b_)[i]);
        break;
    case 70: case 71: case 72: case 73: case 74: case 75: case 76: case 77:
        static_cast<Quad<float> *>(out_)[i] = quad_selftest_op<float>(op - 70, static_cast<const Quad<float> *>(a_)[i],
                                                                      static_cast<const Quad<float> *>(b_)[i]);
        break;
    default: break;
    }
}
uint32_t numeric_op_elem_bytes(uint32_t op) {
    if (op <= 6) return 8;
    if (op >= 10 && op <= 14) return 12;
    if (op >= 20 && op <= 23) return 8;
    if (op >= 30 && op <= 32) return 16;
    if (op == 40) return 24;
    if (op >= 50 && op <= 56) return 16;
    if (op >= 60 && op <= 67) return 32;
    if (op >= 70 && op <= 77) return 16;
    if (op >= 80 && op <= 85) return kPerturbRecordBytes;
    if (op >= 86 && op <= 91) return kExpmapRecordBytes;
    return 0;
}
} // namespace

extern "C" {

uint32_t fs_test_cuda_is_working(void) {
    // GPU_Render.cu:100-123 (returns a bool-like value: 1 = working)
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return 0;
    if (cudaSetDevice(0) != cudaSuccess) return 0;
    if (cudaFree(nullptr) != cudaSuccess) return 0;
    return 1;
}

fs_renderer *fs_create(int32_t device) {
    fs_renderer *r = new (std::nothrow) fs_renderer();
    if (r) {
        r->device = device;
        // development switches (profiling under ncu without touching the caller): FS_SPLIT_AT=1, FS_SCALED_STEPS=0
        if (const char *e = getenv("FS_SPLIT_AT")) r->split_at = atoi(e) != 0;
        if (const char *e = getenv("FS_CTAS_PER_SM")) r->ctas_per_sm_cap = atoi(e);
        if (const char *e = getenv("FS_CARVEOUT")) r->carveout_pct = atoi(e);
        if (const char *e = getenv("FS_FORCE_HOST_TABLES")) r->force_host_tables = atoi(e) != 0;
        if (const char *e = getenv("FS_SCALED_STEPS")) r->use_scaled = atoi(e) != 0;
        if (const char *e = getenv("FS_LAV2_POOL")) r->use_pool = atoi(e) != 0;
        if (const char *e = getenv("FS_AT_CYCLE")) r->at_cycle = atoi(e) != 0;
        if (const char *e = getenv("FS_LA_STEP2")) r->use_la2 = atoi(e) != 0;
        if (const char *e = getenv("FS_PROBE_PASSES")) r->probe_passes = atoi(e);
    }
    return r;
}

fs_renderer *fs_create_group(const int32_t *devices, uint32_t n) {
    if (!devices || n == 0) return nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    for (uint32_t i = 0; i < n; i++)
        if (devices[i] < 0 || devices[i] >= count) return nullptr;
    if (n == 1) return fs_create(devices[0]);
    fs_renderer *grp = new (std::nothrow) fs_renderer();
    if (!grp) return nullptr;
    grp->device = devices[0];
    for (uint32_t i = 0; i < n; i++) {
        fs_renderer *m = fs_create(devices[i]);
        if (!m) { for (fs_renderer *k : grp->members) fs_destroy(k); grp->members.clear(); delete grp; return nullptr; }
        m->shard_count = n;
        m->shard_index = i;
        grp->members.push_back(m);
    }
    // the members' bands meet on the lead (AA-3 colours, the reduction parts): direct over NVLink where the pair allows it.
    // Peer access is per process and other groups may rely on it, so it is never disabled.
    for (uint32_t i = 1; i < n; i++) {
        const int a = devices[0], b = devices[i];
        if (a == b) continue;
        int ok = 0;
        for (int k = 0; k < 2; k++) {
            const int from = k ? b : a, to = k ? a : b;
            if (cudaDeviceCanAccessPeer(&ok, from, to) != cudaSuccess || !ok) continue;
            DeviceGuard g(from);
            if (cudaDeviceEnablePeerAccess(to, 0) != cudaSuccess) (void)cudaGetLastError(); // e.g. already enabled
        }
    }
    return grp;
}

fs_renderer *fs_create_default(void) {
    const char *list = getenv("FS_GPU_DEVICES");
    if (!list) return fs_create(0);
    int32_t ids[64];
    uint32_t n = 0;
    const char *p = list;
    for (;;) { // one or more digits per item, items separated by single commas
        if (*p < '0' || *p > '9' || n == 64) return nullptr;
        int64_t v = 0;
        while (*p >= '0' && *p <= '9') {
            v = v * 10 + (*p++ - '0');
            if (v > INT32_MAX) return nullptr;
        }
        ids[n++] = (int32_t)v;
        if (*p == '\0') break;
        if (*p++ != ',') return nullptr;
    }
    return fs_create_group(ids, n);
}

uint32_t fs_device_count(const fs_renderer *r) { return !r ? 0 : is_group(r) ? (uint32_t)r->members.size() : 1; }

void fs_destroy(fs_renderer *r) {
    if (!r) return;
    if (is_group(r)) {
        sync_members(r, true);
        for (size_t i = 0; i < r->joins.size(); i++) {
            DeviceGuard g(r->members[i]->device);
            if (r->joins[i]) cudaEventDestroy(r->joins[i]);
        }
        {
            DeviceGuard g(r->device);
            for (cudaEvent_t e : r->lead_marks)
                if (e) cudaEventDestroy(e);
            for (void *b : r->gather)
                if (b) cudaFree(b);
            if (r->red_parts) cudaFree(r->red_parts);
        }
        // member 0 registered a result sink the others only map: it lets go of it last
        for (size_t i = r->members.size(); i-- > 0;) fs_destroy(r->members[i]);
        delete r;
        return;
    }
    DeviceGuard g(r->device);
    if (r->compute) {
        if (r->display) cudaStreamSynchronize(r->display);
        reset_perturb(r);
        reset_buffers(r);
        if (r->pal_dev) cudaFreeAsync(r->pal_dev, r->compute);
        if (r->tile_counter) cudaFreeAsync(r->tile_counter, r->compute);
        if (r->step_counter) cudaFreeAsync(r->step_counter, r->compute);
        cudaStreamSynchronize(r->compute);
        cudaStreamDestroy(r->compute);
        if (r->display) cudaStreamDestroy(r->display);
        if (r->ev_start) cudaEventDestroy(r->ev_start);
        if (r->ev_stop) cudaEventDestroy(r->ev_stop);
        if (r->ev_alloc) cudaEventDestroy(r->ev_alloc);
        if (r->yield_src) cudaFreeHost(r->yield_src);
    }
    delete r;
}

uint32_t fs_initialize_memory(fs_renderer *r, uint32_t iter_bytes, uint32_t w, uint32_t h, uint32_t antialiasing,
                              const fs_color16 *pal, uint32_t pal_iters, uint32_t aux_depth, uint64_t pal_gen,
                              int32_t expected_reuse) {
    if (is_group(r)) {
        // a geometry change drops the result sink member 0 registered: no member may still be writing into it
        if (r->members[0]->sink_dev) sync_members(r);
        const uint32_t rc = each_member(r, [&](fs_renderer *m) {
            return fs_initialize_memory(m, iter_bytes, w, h, antialiasing, pal, pal_iters, aux_depth, pal_gen, expected_reuse);
        });
        return rc ? rc : (uint32_t)prepare_group(r);
    }
    if (!r || (iter_bytes != 4 && iter_bytes != 8)) return FS_ERROR_UNSUPPORTED;
    cudaError_t err = cudaSetDevice(r->device);
    if (err != cudaSuccess) return err;
    r->aux_depth = aux_depth;
    if (!r->compute) {
        int lo, hi;
        err = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (err != cudaSuccess) return err;
        err = cudaStreamCreateWithPriority(&r->compute, cudaStreamNonBlocking, lo);
        if (err != cudaSuccess) return err;
        err = cudaStreamCreateWithPriority(&r->display, cudaStreamNonBlocking, hi);
        if (err != cudaSuccess) return err;
        cudaEventCreate(&r->ev_start);
        cudaEventCreate(&r->ev_stop);
        cudaDeviceGetAttribute(&r->num_sms, cudaDevAttrMultiProcessorCount, r->device);
        cudaEventCreateWithFlags(&r->ev_alloc, cudaEventDisableTiming);
        err = cudaMallocAsync(&r->tile_counter, 2 * sizeof(unsigned int), r->compute);
        if (err != cudaSuccess) return err;
        r->yield_quota = reinterpret_cast<int *>(r->tile_counter + 1);
        cudaMemsetAsync(r->tile_counter, 0, 2 * sizeof(unsigned int), r->compute);
        err = cudaMallocHost(&r->yield_src, sizeof(int));
        if (err != cudaSuccess) return err;
        *r->yield_src = kYieldCtas;
        err = cudaMallocAsync(&r->step_counter, 4 * sizeof(unsigned long long), r->compute);
        if (err != cudaSuccess) return err;
        cudaMemsetAsync(r->step_counter, 0, 4 * sizeof(unsigned long long), r->compute);
    }
    bool allocated = false;
    if (r->cached_pal_host != pal || r->cached_pal_gen != pal_gen) {
        // a progressive RenderCurrent may still be reading the old palette on the display stream
        if (r->pal_dev) { cudaStreamSynchronize(r->display); cudaFreeAsync(r->pal_dev, r->compute); }
        allocated = true;
        r->pal_dev = nullptr;
        r->pal_iters = pal_iters;
        r->cached_pal_host = pal;
        err = cudaMallocAsync(&r->pal_dev, (pal_iters ? pal_iters : 1) * sizeof(Color16), r->compute);
        if (err != cudaSuccess) return err;
        if (pal && pal_iters) {
            err = cudaMemcpyAsync(r->pal_dev, pal, pal_iters * sizeof(Color16), cudaMemcpyHostToDevice, r->compute);
            if (err != cudaSuccess) return err;
        }
        r->cached_pal_gen = pal_gen;
    }
    if (r->width == w && r->height == h && r->aa == antialiasing && r->iter_bytes == iter_bytes && expected_reuse) {
        if (allocated) { cudaEventRecord(r->ev_alloc, r->compute); cudaStreamWaitEvent(r->display, r->ev_alloc, 0); }
        return 0;
    }
    if (antialiasing > 4 || antialiasing < 1) return FS_ERROR_3_BAD_ANTIALIASING;
    if (w % antialiasing != 0) return FS_ERROR_4_WIDTH_NOT_MULTIPLE_OF_AA;
    if (h % antialiasing != 0) return FS_ERROR_5_HEIGHT_NOT_MULTIPLE_OF_AA;

    r->w_block = w / NB_THREADS_W + (w % NB_THREADS_W != 0);
    r->h_block = h / NB_THREADS_H + (h % NB_THREADS_H != 0);
    r->width = w;
    r->height = h;
    r->aa = antialiasing;
    r->iter_bytes = iter_bytes;
    r->n_cu = (size_t)r->w_block * NB_THREADS_W * r->h_block * NB_THREADS_H;
    r->color_w = w / antialiasing;
    r->color_h = h / antialiasing;
    const uint32_t wcb = r->color_w / NB_THREADS_W + (r->color_w % NB_THREADS_W != 0);
    const uint32_t hcb = r->color_h / NB_THREADS_H + (r->color_h % NB_THREADS_H != 0);
    r->n_color_cu = (size_t)wcb * NB_THREADS_W * hcb * NB_THREADS_H;

    // geometry change drops cached orbit/LA uploads (ResetPerturb::Yes, GPU_Render.cu:358).  The buffers are freed and
    // allocated in compute-stream order; display-stream work (progressive RenderCurrent) is fenced on both sides.
    cudaStreamSynchronize(r->display);
    reset_perturb(r);
    reset_buffers(r);
    err = cudaMallocAsync(&r->iter_buf, r->n_cu * iter_bytes, r->compute);
    if (err != cudaSuccess) return err;
    err = cudaMallocAsync(&r->red_dev, sizeof(Reduction), r->compute);
    if (err != cudaSuccess) return err;
    err = cudaMallocAsync(&r->color_buf, r->n_color_cu * sizeof(Color16), r->compute);
    if (err != cudaSuccess) return err;
    fs_clear_memory(r);
    cudaEventRecord(r->ev_alloc, r->compute);
    cudaStreamWaitEvent(r->display, r->ev_alloc, 0);
    // With lazy module loading a kernel's first launch loads it, and that waits for running kernels: the result
    // kernels are loaded here so the first progressive RenderCurrent does not sit out the render it was meant to show.
    preload_post_kernels(r);
    return 0;
}

uint32_t fs_initialize_perturb(fs_renderer *r, uint32_t iter_bytes, int32_t numeric1, int32_t pextras,
                               uint64_t generation1, const fs_orbit *perturb1, int32_t numeric2, uint64_t generation2,
                               const fs_orbit *perturb2, const fs_la_reference *la) {
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_initialize_perturb(m, iter_bytes, numeric1, pextras, generation1, perturb1, numeric2, generation2, perturb2, la);
        });
    if (!r || !r->compute) return FS_ERROR_6_NO_ORBIT;
    DeviceGuard g(r->device);
    bool install_la = false;
    const uint64_t have1 = r->orbit1.valid ? r->orbit1.generation : 0;
    const uint64_t have2 = r->orbit2.valid ? r->orbit2.generation : 0;
    if (generation1 != have1 || generation2 != have2) reset_perturb(r);
    if (generation1 != (r->orbit1.valid ? r->orbit1.generation : 0)) {
        if (!perturb1) return FS_ERROR_6_NO_ORBIT;
        const uint32_t rc = upload_orbit(r, r->orbit1, numeric1, pextras, generation1, perturb1);
        if (rc) return rc;
        install_la = true;
    }
    if (generation2 != (r->orbit2.valid ? r->orbit2.generation : 0)) {
        if (!perturb2) return FS_ERROR_6_NO_ORBIT;
        const uint32_t rc = upload_orbit(r, r->orbit2, numeric2, pextras, generation2, perturb2);
        if (rc) return rc;
        install_la = true;
    }
    if (install_la && la) {
        const uint32_t rc = upload_la(r, numeric1, iter_bytes, la);
        if (rc) return rc;
    }
    return 0;
}

void fs_clear_memory(fs_renderer *r) {
    if (is_group(r)) { each_member(r, [](fs_renderer *m) { fs_clear_memory(m); return 0u; }); return; }
    if (!r || !r->compute) return;
    r->sink_filled = false;
    DeviceGuard g(r->device);
    if (r->iter_buf) cudaMemsetAsync(r->iter_buf, 0, r->n_cu * r->iter_bytes, r->compute);
    if (r->frame_stack) cudaMemsetAsync(r->frame_stack, 0, r->stack_frames * r->n_cu * r->iter_bytes, r->compute);
    if (r->red_dev) cudaMemsetAsync(r->red_dev, 0, r->iter_bytes, r->compute);
    if (r->color_buf) cudaMemsetAsync(r->color_buf, 0, r->n_color_cu * sizeof(Color16), r->compute);
}

uint32_t fs_render(fs_renderer *r, uint32_t algorithm, int32_t numeric, const void *cx, const void *cy,
                   const void *dx, const void *dy, uint64_t n_iterations, int32_t iteration_precision) {
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render(m, algorithm, numeric, cx, cy, dx, dy, n_iterations, iteration_precision);
        });
    (void)algorithm;
    if (!r || !memory_initialized(r)) return 0; // GPU_Render.cu:626-628
    DeviceGuard g(r->device);
    const bool u64 = r->iter_bytes == 8;
    switch (numeric) {
    case FS_NUM_F32:
        return u64 ? launch_direct<float, uint64_t>(r, cx, cy, dx, dy, n_iterations, iteration_precision)
                   : launch_direct<float, uint32_t>(r, cx, cy, dx, dy, n_iterations, iteration_precision);
    case FS_NUM_F64:
        return u64 ? launch_direct<double, uint64_t>(r, cx, cy, dx, dy, n_iterations, iteration_precision)
                   : launch_direct<double, uint32_t>(r, cx, cy, dx, dy, n_iterations, iteration_precision);
    case FS_NUM_2X32: // Gpu2x32: MattDblflt {head, tail}; 1/4/8/16 steps per bailout test (GPU_Render.cu:733-771)
        switch (iteration_precision) {
        case 1: return launch_direct_ext_pods<Pixel2x32<1>>(r, cx, cy, dx, dy, n_iterations);
        case 4: return launch_direct_ext_pods<Pixel2x32<4>>(r, cx, cy, dx, dy, n_iterations);
        case 8: return launch_direct_ext_pods<Pixel2x32<8>>(r, cx, cy, dx, dy, n_iterations);
        case 16: return launch_direct_ext_pods<Pixel2x32<16>>(r, cx, cy, dx, dy, n_iterations);
        default: return 0;
        }
    case FS_NUM_2X64: return launch_direct_ext_pods<Pixel2x64>(r, cx, cy, dx, dy, n_iterations); // MattDbldbl {head, tail}
    case FS_NUM_4X32: return launch_direct_ext_pods<Pixel4x32>(r, cx, cy, dx, dy, n_iterations); // MattQFltflt {x,y,z,w}
    case FS_NUM_4X64: return launch_direct_ext_pods<Pixel4x64>(r, cx, cy, dx, dy, n_iterations); // MattQDbldbl {x,y,z,w}
    case FS_NUM_HDR64: { // GpuHDRx32: HDRFloat<double> in, float+exponent over 2x32 inside (GPU_Render.cu:797-841)
        const Hdr<df32> vcx = hdr2x32_from_hdr64(cx), vcy = hdr2x32_from_hdr64(cy), vdx = hdr2x32_from_hdr64(dx),
                        vdy = hdr2x32_from_hdr64(dy);
#define FS_HDRD(P) (u64 ? launch_direct_ext<PixelHdr2x32<P>, uint64_t>(r, vcx, vcy, vdx, vdy, n_iterations)             \
                        : launch_direct_ext<PixelHdr2x32<P>, uint32_t>(r, vcx, vcy, vdx, vdy, n_iterations))
        switch (iteration_precision) {
        case 1: return FS_HDRD(1);
        case 4: return FS_HDRD(4);
        case 8: return FS_HDRD(8);
        case 16: return FS_HDRD(16);
        default: return 0;
        }
#undef FS_HDRD
    }
    default: return FS_ERROR_UNSUPPORTED;
    }
}

uint32_t fs_render_perturb_lav2(fs_renderer *r, uint32_t algorithm, int32_t numeric, int32_t mode, int32_t pextras,
                                const void *cx, const void *cy, const void *dx, const void *dy, const void *center_x,
                                const void *center_y, uint64_t n_iterations) {
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render_perturb_lav2(m, algorithm, numeric, mode, pextras, cx, cy, dx, dy, center_x, center_y, n_iterations);
        });
    (void)algorithm; (void)cx; (void)cy;
    if (!r || !memory_initialized(r)) return 0; // GPU_Render.cu:1007-1009
    DeviceGuard g(r->device);
    if (!r->orbit1.valid || r->orbit1.numeric != numeric || r->orbit1.pextras != pextras) return FS_ERROR_6_NO_ORBIT;
    // compressed orbits were expanded at upload (fs_orbit_rc.cuh): the same kernels serve both layouts
    if (pextras != FS_PEXTRAS_DISABLE && pextras != FS_PEXTRAS_SIMPLE_COMPRESSION) return FS_ERROR_UNSUPPORTED;
    return dispatch_num_iter(numeric, r->iter_bytes, [&](auto num, auto it) -> uint32_t {
        return launch_lav2<decltype(num), decltype(it)>(r, mode, dx, dy, center_x, center_y, n_iterations);
    });
}

uint32_t fs_render_perturb_lav2_frames(fs_renderer *r, uint32_t algorithm, int32_t numeric, int32_t mode, int32_t pextras,
                                       uint32_t n_frames, const void *cx, const void *cy, const void *dx, const void *dy,
                                       const void *center_x, const void *center_y, uint64_t n_iterations) {
    if (!r || n_frames == 0 || n_frames > FS_MAX_FRAMES || !dx || !dy || !center_x || !center_y) return FS_ERROR_UNSUPPORTED;
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render_perturb_lav2_frames(m, algorithm, numeric, mode, pextras, n_frames, cx, cy, dx, dy, center_x,
                                                 center_y, n_iterations);
        });
    (void)algorithm; (void)cx; (void)cy;
    if (!memory_initialized(r)) return 0; // as fs_render_perturb_lav2
    DeviceGuard g(r->device);
    if (!r->orbit1.valid || r->orbit1.numeric != numeric || r->orbit1.pextras != pextras) return FS_ERROR_6_NO_ORBIT;
    if (pextras != FS_PEXTRAS_DISABLE && pextras != FS_PEXTRAS_SIMPLE_COMPRESSION) return FS_ERROR_UNSUPPORTED;
    return dispatch_num_iter(numeric, r->iter_bytes, [&](auto num, auto it) -> uint32_t {
        return launch_lav2_frames<decltype(num), decltype(it)>(r, mode, n_frames, dx, dy, center_x, center_y, n_iterations);
    });
}

uint32_t fs_render_perturb_lav2_expmap(fs_renderer *r, uint32_t algorithm, int32_t numeric, int32_t mode, int32_t pextras,
                                       const void *radius, const void *dir_x, const void *dir_y, uint64_t n_iterations) {
    if (!r || !radius || !dir_x || !dir_y) return FS_ERROR_UNSUPPORTED;
    if (mode != FS_LAV2_FULL && mode != FS_LAV2_PO && mode != FS_LAV2_LAO) return FS_ERROR_UNSUPPORTED;
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render_perturb_lav2_expmap(m, algorithm, numeric, mode, pextras, radius, dir_x, dir_y, n_iterations);
        });
    (void)algorithm;
    if (!memory_initialized(r)) return FS_ERROR_UNSUPPORTED; // the tables' sizes are the initialized frame's
    DeviceGuard g(r->device);
    if (!r->orbit1.valid || r->orbit1.numeric != numeric || r->orbit1.pextras != pextras) return FS_ERROR_6_NO_ORBIT;
    if (pextras != FS_PEXTRAS_DISABLE && pextras != FS_PEXTRAS_SIMPLE_COMPRESSION) return FS_ERROR_UNSUPPORTED;
    return dispatch_num_iter(numeric, r->iter_bytes, [&](auto num, auto it) -> uint32_t {
        return launch_lav2_expmap<decltype(num), decltype(it)>(r, mode, radius, dir_x, dir_y, n_iterations);
    });
}

uint32_t fs_select_frame(fs_renderer *r, uint32_t k) {
    if (is_group(r)) {
        for (fs_renderer *m : r->members) // all members rendered the same batch: refuse before any of them changes
            if (k >= m->n_frames) return FS_ERROR_UNSUPPORTED;
        return each_member(r, [&](fs_renderer *m) { return fs_select_frame(m, k); });
    }
    if (!r || k >= r->n_frames) return FS_ERROR_UNSUPPORTED;
    r->selected = k;
    return 0;
}

uint32_t fs_render_perturb_bla(fs_renderer *r, uint32_t algorithm, int32_t numeric, const fs_orbit *results,
                               const fs_blas *blas, const void *cx, const void *cy, const void *dx, const void *dy,
                               const void *center_x, const void *center_y, uint64_t n_iterations,
                               int32_t iteration_precision) {
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render_perturb_bla(m, algorithm, numeric, results, blas, cx, cy, dx, dy, center_x, center_y, n_iterations,
                                         iteration_precision);
        });
    (void)algorithm; (void)cx; (void)cy; (void)iteration_precision;
    if (!r || !memory_initialized(r)) return 0; // GPU_Render.cu:1454-1456
    if (!results || !blas) return FS_ERROR_6_NO_ORBIT;
    // the reference instantiates HDRFloat<float>, HDRFloat<double> and double (GPU_Render.cu:1610-1692)
    if (numeric != FS_NUM_HDR32 && numeric != FS_NUM_HDR64 && numeric != FS_NUM_F64) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    const bool saved_scaled = r->use_scaled;
    r->use_scaled = false; // no plain-float step table for this kernel
    const uint32_t rc = upload_orbit(r, r->bla_orbit, numeric, FS_PEXTRAS_DISABLE, 0, results);
    r->use_scaled = saved_scaled;
    if (rc) return rc;
    const bool u64 = r->iter_bytes == 8;
    switch (numeric) {
    case FS_NUM_HDR32:
        return u64 ? launch_bla<NumHdr<float>, uint64_t>(r, blas, dx, dy, center_x, center_y, n_iterations)
                   : launch_bla<NumHdr<float>, uint32_t>(r, blas, dx, dy, center_x, center_y, n_iterations);
    case FS_NUM_HDR64:
        return u64 ? launch_bla<NumHdr<double>, uint64_t>(r, blas, dx, dy, center_x, center_y, n_iterations)
                   : launch_bla<NumHdr<double>, uint32_t>(r, blas, dx, dy, center_x, center_y, n_iterations);
    default:
        return u64 ? launch_bla<NumPlain<double>, uint64_t>(r, blas, dx, dy, center_x, center_y, n_iterations)
                   : launch_bla<NumPlain<double>, uint32_t>(r, blas, dx, dy, center_x, center_y, n_iterations);
    }
}

uint32_t fs_render_perturb_bla_scaled(fs_renderer *r, uint32_t algorithm, int32_t numeric,
                                      const fs_orbit *double_perturb, const fs_orbit *float_perturb, const void *cx,
                                      const void *cy, const void *dx, const void *dy, const void *center_x,
                                      const void *center_y, uint64_t n_iterations, int32_t iteration_precision) {
    if (is_group(r))
        return each_member(r, [&](fs_renderer *m) {
            return fs_render_perturb_bla_scaled(m, algorithm, numeric, double_perturb, float_perturb, cx, cy, dx, dy, center_x,
                                                center_y, n_iterations, iteration_precision);
        });
    (void)algorithm; (void)cx; (void)cy; (void)iteration_precision;
    if (!r || !memory_initialized(r)) return 0; // GPU_Render.cu:1317-1319
    if (!double_perturb || !float_perturb) return FS_ERROR_6_NO_ORBIT;
    // the reference instantiates T = double and T = HDRFloat<float> (GPU_Render.cu:1381-1436)
    if (numeric != FS_NUM_F64 && numeric != FS_NUM_HDR32) return FS_ERROR_UNSUPPORTED;
    if (double_perturb->compressed_count != float_perturb->compressed_count) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    uint32_t rc = upload_orbit(r, r->scaled_orbit_f, FS_NUM_F32, FS_PEXTRAS_BAD, 0, float_perturb);
    if (rc) return rc;
    rc = upload_orbit(r, r->bla_orbit, numeric, FS_PEXTRAS_BAD, 0, double_perturb);
    if (rc) return rc;
    const bool u64 = r->iter_bytes == 8;
    if (numeric == FS_NUM_F64)
        return u64 ? launch_scaled<NumPlain<double>, uint64_t>(r, dx, dy, center_x, center_y, n_iterations)
                   : launch_scaled<NumPlain<double>, uint32_t>(r, dx, dy, center_x, center_y, n_iterations);
    return u64 ? launch_scaled<NumHdr<float>, uint64_t>(r, dx, dy, center_x, center_y, n_iterations)
               : launch_scaled<NumHdr<float>, uint32_t>(r, dx, dy, center_x, center_y, n_iterations);
}

// A progressive frame asked for while a render kernel holds every SM slot: the display stream raises the yield quota
// (a 4-byte copy, no SM needed), kYieldCtas CTAs of the persistent grid retire at their next tile boundary, and the
// high-priority post kernel launched right after takes their slots.  Asked once per render: the slots stay free.
static void request_yield_if_rendering(fs_renderer *r) {
    if (r->yield_requested) return;
    if (cudaStreamQuery(r->compute) != cudaErrorNotReady) return;
    (void)cudaGetLastError();
    r->yield_requested = true;
    cudaMemcpyAsync(r->yield_quota, r->yield_src, sizeof(int), cudaMemcpyHostToDevice, r->display);
}

static cudaError_t copy_shard_bands(fs_renderer *r, void *iter_buffer, fs_color16 *color_buffer, cudaStream_t stream);
static uint32_t group_render_current(fs_renderer *grp, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                                     fs_reduction *reduction_results, int32_t progressive);

uint32_t fs_render_current(fs_renderer *r, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                           fs_reduction *reduction_results, int32_t progressive) {
    if (is_group(r)) return group_render_current(r, n_iterations, iter_buffer, color_buffer, reduction_results, progressive);
    if (!r || !memory_initialized(r)) return 0; // GPU_Render.cu:563-565
    DeviceGuard g(r->device);
    cudaStream_t stream = progressive ? r->display : r->compute;
    if (progressive) request_yield_if_rendering(r);
    // no colour buffer asked for: the reduction alone (the colour buffer on the device is then stale until a call that asks)
    const bool colors = color_buffer != nullptr;
    uint32_t rc = r->iter_bytes == 8 ? run_post<uint64_t>(r, n_iterations, stream, colors, r->shard_count, r->shard_index)
                                     : run_post<uint32_t>(r, n_iterations, stream, colors, r->shard_count, r->shard_index);
    if (rc) return rc;
    cudaError_t err = cudaSuccess;
    if (iter_buffer && !(r->sink_filled && iter_buffer == r->sink_host)) { // a filled sink already holds the frame
        err = cudaMemcpyAsync(iter_buffer, selected_iter_buf(r), r->n_cu * r->iter_bytes, cudaMemcpyDefault, stream);
        if (err != cudaSuccess) return err;
    }
    if (color_buffer) {
        err = cudaMemcpyAsync(color_buffer, r->color_buf, r->n_color_cu * sizeof(Color16), cudaMemcpyDefault, stream);
        if (err != cudaSuccess) return err;
    }
    if (reduction_results) {
        err = cudaMemcpyAsync(reduction_results, r->red_dev, sizeof(Reduction), cudaMemcpyDefault, stream);
        if (err != cudaSuccess) return err;
    }
    return 0;
}

// Multi-GPU result path: only the 4-row bands this shard rendered leave the device (one strided 2-D copy each for the
// iteration cells and, when asked for, their colours), so N ranks writing into one host frame (e.g. a registered
// shared-memory mapping) assemble it with no collective and 1/N of the PCIe bytes each.  Colours and Min/Max/Sum cover this
// shard's cells only (post_kernel skips the others): the frame's reduction is min / max / sum over the shards'.
uint32_t fs_render_current_shard(fs_renderer *r, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                                 fs_reduction *reduction_results, int32_t progressive) {
    if (is_group(r)) return FS_ERROR_UNSUPPORTED; // a group already is the sharding
    if (!r || !memory_initialized(r)) return 0;
    if (r->shard_count <= 1) return fs_render_current(r, n_iterations, iter_buffer, color_buffer, reduction_results, progressive);
    // an antialiasing cell must lie inside one 4-row band: 3x3 cells straddle bands, their colours would need other shards' rows
    if (color_buffer && r->aa == 3) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    cudaStream_t stream = progressive ? r->display : r->compute;
    if (progressive) request_yield_if_rendering(r);
    const bool colors = color_buffer != nullptr;
    uint32_t rc = r->iter_bytes == 8 ? run_post<uint64_t>(r, n_iterations, stream, colors, r->shard_count, r->shard_index)
                                     : run_post<uint32_t>(r, n_iterations, stream, colors, r->shard_count, r->shard_index);
    if (rc) return rc;
    cudaError_t err = copy_shard_bands(r, iter_buffer, color_buffer, stream);
    if (err != cudaSuccess) return err;
    if (reduction_results) {
        err = cudaMemcpyAsync(reduction_results, r->red_dev, sizeof(Reduction), cudaMemcpyDefault, stream);
        if (err != cudaSuccess) return err;
    }
    return 0;
}

// The shard's own 4-row bands of the iteration cells into the same positions of a whole-frame buffer (host, or another
// renderer's device buffer): one strided 2-D copy.
static cudaError_t copy_iter_bands(const fs_renderer *r, void *dst, cudaStream_t stream) {
    const size_t row_bytes = (size_t)r->w_block * NB_THREADS_W * r->iter_bytes;
    const size_t bands = (size_t)r->h_block * NB_THREADS_H / 4; // padded height is a multiple of 8
    const size_t owned = (bands - r->shard_index + r->shard_count - 1) / r->shard_count;
    const size_t first = (size_t)r->shard_index * 4 * row_bytes, stride = (size_t)r->shard_count * 4 * row_bytes;
    if (!owned) return cudaSuccess;
    return cudaMemcpy2DAsync((char *)dst + first, stride, (const char *)selected_iter_buf(r) + first, stride, 4 * row_bytes, owned,
                             cudaMemcpyDefault, stream);
}

// The shard's own 4-row bands of the iteration cells (unless a filled sink already holds them) and, when color_buffer is
// given, of the Color16 cells, into the same positions of whole-frame host buffers.
static cudaError_t copy_shard_bands(fs_renderer *r, void *iter_buffer, fs_color16 *color_buffer, cudaStream_t stream) {
    cudaError_t err = cudaSuccess;
    if (iter_buffer && !(r->sink_filled && iter_buffer == r->sink_host)) {
        err = copy_iter_bands(r, iter_buffer, stream);
        if (err != cudaSuccess) return err;
    }
    if (color_buffer) {
        // colour cells are stored un-padded (index oy * color_w + ox, AntialiasingKernel.cuh:3-71): the colour rows of one
        // band, 4 / AA of them, are contiguous; band b of this shard sits at row (b * shard_count + shard_index) * 4 / AA
        const size_t rows_per_band = 4 / r->aa;
        const size_t band_bytes = rows_per_band * (size_t)r->color_w * sizeof(Color16);
        const size_t total_bands = ((size_t)r->color_h + rows_per_band - 1) / rows_per_band;
        const size_t full_rows_bands = (size_t)r->color_h / rows_per_band; // bands with all their rows inside the frame
        size_t owned_full = 0;
        if (full_rows_bands > r->shard_index) owned_full = (full_rows_bands - r->shard_index + r->shard_count - 1) / r->shard_count;
        const size_t first = (size_t)r->shard_index * band_bytes, stride = (size_t)r->shard_count * band_bytes;
        if (owned_full) {
            err = cudaMemcpy2DAsync((char *)color_buffer + first, stride, (const char *)r->color_buf + first, stride, band_bytes,
                                    owned_full, cudaMemcpyDefault, stream);
            if (err != cudaSuccess) return err;
        }
        if (total_bands > full_rows_bands && (total_bands - 1) % r->shard_count == r->shard_index) {
            // the frame's last band is cut short by the frame edge and belongs to this shard
            const size_t off = (total_bands - 1) * band_bytes;
            const size_t rest = ((size_t)r->color_h - full_rows_bands * rows_per_band) * (size_t)r->color_w * sizeof(Color16);
            err = cudaMemcpyAsync((char *)color_buffer + off, (const char *)r->color_buf + off, rest, cudaMemcpyDefault, stream);
            if (err != cudaSuccess) return err;
        }
    }
    return cudaSuccess;
}

// RenderCurrent of a device group: the bytes one renderer returns, assembled without a host synchronise.  Every member
// copies its own iteration bands to the host over its own link.  AA 1/2/4: every member colours and reduces its own bands
// (a cell never straddles two bands) and copies its colour bands; the members' reductions meet on the lead, where
// reduction_combine_kernel makes the frame's.  AA 3: 3x3 cells straddle bands, so every member copies its iteration bands
// into the lead's gather buffer (peer to peer) and the lead colours and reduces the whole frame from there.
// Members write into lead-owned memory (reduction parts, gather buffer) only after the lead's stream has passed what it
// had been given before this call, so result calls may follow each other without a synchronise in between.
static uint32_t group_render_current(fs_renderer *grp, uint64_t n_iterations, void *iter_buffer, fs_color16 *color_buffer,
                                     fs_reduction *reduction_results, int32_t progressive) {
    fs_renderer *lead = grp->members[0];
    if (!memory_initialized(lead) || !grp->red_parts) return 0;
    const size_t n = grp->members.size();
    const bool colors = color_buffer != nullptr;
    const bool on_lead = lead->aa == 3;
    const bool to_lead = colors || reduction_results; // anything beyond the iteration cells, which need no meeting point
    const int slot = progressive ? 1 : 0;
    auto stream_of = [&](fs_renderer *m) { return progressive ? m->display : m->compute; };
    Reduction *parts = grp->red_parts + slot * (n + 1), *frame_red = parts + n;
    void *gather = grp->gather[slot];
    // fs_initialize_memory sizes the gather buffers; a call that failed on some member may have left them behind
    if (on_lead && to_lead && (!gather || grp->gather_bytes != lead->n_cu * lead->iter_bytes)) return FS_ERROR_UNSUPPORTED;
    cudaError_t err = cudaSuccess;
    { // what the lead's stream has been given so far, including the reads of the previous result call on this stream
        DeviceGuard g(lead->device);
        err = cudaEventRecord(grp->lead_marks[slot], stream_of(lead));
        if (err != cudaSuccess) return err;
    }
    for (size_t i = 0; i < n; i++) {
        fs_renderer *m = grp->members[i];
        DeviceGuard g(m->device);
        const cudaStream_t s = stream_of(m);
        if (progressive) request_yield_if_rendering(m);
        if (!on_lead) {
            const uint32_t rc = m->iter_bytes == 8 ? run_post<uint64_t>(m, n_iterations, s, colors, m->shard_count, m->shard_index)
                                                   : run_post<uint32_t>(m, n_iterations, s, colors, m->shard_count, m->shard_index);
            if (rc) return rc;
        }
        err = copy_shard_bands(m, iter_buffer, on_lead ? nullptr : color_buffer, s);
        if (err != cudaSuccess) return err;
        const bool writes_lead = on_lead ? to_lead : reduction_results != nullptr;
        if (!writes_lead) continue;
        if (i > 0) { // write only after the lead has read what the previous result call left there
            err = cudaStreamWaitEvent(s, grp->lead_marks[slot], 0);
            if (err != cudaSuccess) return err;
        }
        err = on_lead ? copy_iter_bands(m, gather, s)
                      : cudaMemcpyPeerAsync(parts + i, lead->device, m->red_dev, m->device, sizeof(Reduction), s);
        if (err != cudaSuccess) return err;
        if (i > 0) {
            err = join_member(grp, i, s, stream_of(lead));
            if (err != cudaSuccess) return err;
        }
    }
    DeviceGuard g(lead->device);
    const cudaStream_t s = stream_of(lead);
    if (on_lead) {
        if (!to_lead) return 0;
        const uint32_t rc = lead->iter_bytes == 8 ? run_post<uint64_t>(lead, n_iterations, s, colors, 1, 0, gather)
                                                  : run_post<uint32_t>(lead, n_iterations, s, colors, 1, 0, gather);
        if (rc) return rc;
        if (color_buffer) {
            err = cudaMemcpyAsync(color_buffer, lead->color_buf, lead->n_color_cu * sizeof(Color16), cudaMemcpyDefault, s);
            if (err != cudaSuccess) return err;
        }
        if (reduction_results) {
            err = cudaMemcpyAsync(reduction_results, lead->red_dev, sizeof(Reduction), cudaMemcpyDefault, s);
            if (err != cudaSuccess) return err;
        }
        return 0;
    }
    if (color_buffer) { // the padding behind the colour cells, as fs_render_current copies it
        const size_t cells = (size_t)lead->color_w * lead->color_h;
        err = cudaMemcpyAsync(color_buffer + cells, lead->color_buf + cells, (lead->n_color_cu - cells) * sizeof(Color16),
                              cudaMemcpyDefault, s);
        if (err != cudaSuccess) return err;
    }
    if (reduction_results) {
        auto k = reduction_combine_kernel;
        same_carveout(lead, k);
        k<<<1, 256, 0, s>>>(parts, (int)n, frame_red);
        lead->launches++;
        err = cudaGetLastError();
        if (err != cudaSuccess) return err;
        err = cudaMemcpyAsync(reduction_results, frame_red, sizeof(Reduction), cudaMemcpyDefault, s);
        if (err != cudaSuccess) return err;
    }
    return 0;
}

uint32_t fs_sync_compute_stream(fs_renderer *r) {
    if (is_group(r)) return each_member(r, [](fs_renderer *m) { return fs_sync_compute_stream(m); });
    DeviceGuard g(r->device);
    return cudaStreamSynchronize(r->compute);
}
uint32_t fs_sync_display_stream(fs_renderer *r) {
    if (is_group(r)) return each_member(r, [](fs_renderer *m) { return fs_sync_display_stream(m); });
    DeviceGuard g(r->device);
    return cudaStreamSynchronize(r->display);
}
uint32_t fs_query_compute_stream(fs_renderer *r) {
    if (is_group(r)) {
        uint32_t first = 0;
        for (fs_renderer *m : r->members) {
            const uint32_t rc = fs_query_compute_stream(m);
            if (rc == cudaErrorNotReady) return rc;
            if (rc && !first) first = rc;
        }
        return first;
    }
    DeviceGuard g(r->device);
    return cudaStreamQuery(r->compute);
}

uint32_t fs_enqueue_compute_done_callback(fs_renderer *r, fs_done_callback fn, void *user) {
    if (is_group(r)) { // once, after every member's render: the lead's compute stream joins the others, then calls back
        if (!r->red_parts) return FS_ERROR_UNSUPPORTED;
        fs_renderer *lead = r->members[0];
        for (size_t i = 1; i < r->members.size(); i++) {
            const cudaError_t err = join_member(r, i, r->members[i]->compute, lead->compute);
            if (err != cudaSuccess) return err;
        }
        return fs_enqueue_compute_done_callback(lead, fn, user);
    }
    DeviceGuard g(r->device);
    r->cb = fn;
    r->cb_user = user;
    return cudaLaunchHostFunc(r->compute, done_trampoline, r);
}

const char *fs_convert_error_to_string(uint32_t err) {
    // GPU_Render.cu:1820-1823 forwards everything to cudaGetErrorString; FractalSharkError values get names here.
    switch (err) {
    case FS_ERROR_3_BAD_ANTIALIASING: return "FractalSharkError 10002: antialiasing must be 1..4";
    case FS_ERROR_4_WIDTH_NOT_MULTIPLE_OF_AA: return "FractalSharkError 10003: width not a multiple of antialiasing";
    case FS_ERROR_5_HEIGHT_NOT_MULTIPLE_OF_AA: return "FractalSharkError 10004: height not a multiple of antialiasing";
    case FS_ERROR_6_NO_ORBIT: return "FractalSharkError 10005: no reference orbit uploaded for this type";
    case FS_ERROR_7_NO_LA: return "FractalSharkError 10006: no LA reference uploaded for this type";
    case FS_ERROR_UNSUPPORTED: return "fs_gpu: unsupported numeric/extras/iteration-width combination";
    default: return cudaGetErrorString(static_cast<cudaError_t>(err));
    }
}

uint32_t fs_get_width(const fs_renderer *r) { return is_group(r) ? r->members[0]->width : r->width; }
uint32_t fs_get_height(const fs_renderer *r) { return is_group(r) ? r->members[0]->height : r->height; }

uint32_t fs_set_shard(fs_renderer *r, uint32_t shard_count, uint32_t shard_index) {
    if (!r || is_group(r) || shard_count == 0 || shard_index >= shard_count) return FS_ERROR_UNSUPPORTED;
    r->shard_count = shard_count;
    r->shard_index = shard_index;
    return 0;
}

uint32_t fs_last_render_ms(fs_renderer *r, float *ms) {
    if (is_group(r)) { // the frame is done when the slowest member is
        float worst = 0.0f;
        for (fs_renderer *m : r->members) {
            float v = 0.0f;
            const uint32_t rc = fs_last_render_ms(m, &v);
            if (rc) return rc;
            worst = v > worst ? v : worst;
        }
        *ms = worst;
        return 0;
    }
    if (!r || !r->timed) return cudaErrorNotReady;
    DeviceGuard g(r->device);
    cudaError_t err = cudaEventSynchronize(r->ev_stop);
    if (err != cudaSuccess) return err;
    return cudaEventElapsedTime(ms, r->ev_start, r->ev_stop);
}

uint32_t fs_enable_step_counter(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_enable_step_counter(m, enable); });
    if (!r || !r->compute) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    r->count_steps = enable != 0;
    return cudaMemsetAsync(r->step_counter, 0, 4 * sizeof(unsigned long long), r->compute);
}

uint32_t fs_read_step_counter(fs_renderer *r, uint64_t *steps) {
    if (is_group(r)) {
        uint64_t total = 0;
        for (fs_renderer *m : r->members) {
            uint64_t v = 0;
            const uint32_t rc = fs_read_step_counter(m, &v);
            if (rc) return rc;
            total += v;
        }
        *steps = total;
        return 0;
    }
    if (!r || !r->compute) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    unsigned long long v = 0;
    cudaError_t err = cudaMemcpyAsync(&v, r->step_counter, sizeof(v), cudaMemcpyDeviceToHost, r->compute);
    if (err != cudaSuccess) return err;
    err = cudaStreamSynchronize(r->compute);
    *steps = v;
    return err;
}

uint32_t fs_read_step_counters(fs_renderer *r, uint64_t *counters3) {
    if (is_group(r) && counters3) {
        uint64_t total[3] = {0, 0, 0};
        for (fs_renderer *m : r->members) {
            uint64_t v[3];
            const uint32_t rc = fs_read_step_counters(m, v);
            if (rc) return rc;
            for (int k = 0; k < 3; k++) total[k] += v[k];
        }
        for (int k = 0; k < 3; k++) counters3[k] = total[k];
        return 0;
    }
    if (!r || !r->compute || !counters3) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    unsigned long long v[3] = {0, 0, 0};
    cudaError_t err = cudaMemcpyAsync(v, r->step_counter, sizeof(v), cudaMemcpyDeviceToHost, r->compute);
    if (err != cudaSuccess) return err;
    err = cudaStreamSynchronize(r->compute);
    counters3[0] = v[0]; counters3[1] = v[1]; counters3[2] = v[2];
    return err;
}

uint32_t fs_measure_fp32_issue_peak(int32_t device, double *ffma_per_second) {
    DeviceGuard g(device);
    int sms = 0;
    cudaError_t err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (err != cudaSuccess) return err;
    float *sink = nullptr;
    err = cudaMalloc(&sink, sizeof(float));
    if (err != cudaSuccess) return err;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int blocks = sms * 8, threads = 256, iters = 1 << 14;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0);
        ffma_peak_kernel<<<blocks, threads>>>(sink, iters, 1.0f + rep);
        cudaEventRecord(e1);
        err = cudaEventSynchronize(e1);
        if (err != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double n = (double)blocks * threads * (double)iters * 16.0;
        if (rep > 0 && n / (ms * 1e-3) > best) best = n / (ms * 1e-3);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *ffma_per_second = best;
    return err;
}

uint32_t fs_measure_fp64_issue_peak(int32_t device, double *dfma_per_second) {
    DeviceGuard g(device);
    int sms = 0;
    cudaError_t err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (err != cudaSuccess) return err;
    double *sink = nullptr;
    err = cudaMalloc(&sink, sizeof(double));
    if (err != cudaSuccess) return err;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int blocks = sms * 8, threads = 256, iters = 1 << 11;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0);
        dfma_peak_kernel<<<blocks, threads>>>(sink, iters, 1.0 + rep);
        cudaEventRecord(e1);
        err = cudaEventSynchronize(e1);
        if (err != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double n = (double)blocks * threads * (double)iters * 16.0;
        if (rep > 0 && n / (ms * 1e-3) > best) best = n / (ms * 1e-3);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *dfma_per_second = best;
    return err;
}

// Streams the iteration buffer to the host while the render runs.  `host_iter_buffer` has the layout fs_render_current
// fills; if it is not page-locked yet it is registered here (and unregistered when the sink is dropped).
uint32_t fs_set_result_sink(fs_renderer *r, void *host_iter_buffer, uint64_t bytes) {
    if (is_group(r)) {
        // member 0 registers the frame (portable, mapped) and the others map the same registration on their devices.  It
        // lets go of it last, after every member has stopped writing.
        sync_members(r);
        for (size_t i = r->members.size(); i-- > 0;) fs_set_result_sink(r->members[i], nullptr, 0);
        if (!host_iter_buffer) return memory_initialized(r->members[0]) ? 0 : FS_ERROR_UNSUPPORTED;
        for (size_t i = 0; i < r->members.size(); i++) {
            const uint32_t rc = fs_set_result_sink(r->members[i], host_iter_buffer, bytes);
            if (rc) {
                for (size_t k = i; k-- > 0;) fs_set_result_sink(r->members[k], nullptr, 0);
                return rc;
            }
        }
        return 0;
    }
    if (!r || !memory_initialized(r)) return FS_ERROR_UNSUPPORTED;
    DeviceGuard g(r->device);
    cudaStreamSynchronize(r->compute);
    drop_sink(r);
    if (!host_iter_buffer) return 0;
    if (bytes < r->n_cu * r->iter_bytes) return cudaErrorInvalidValue;
    void *dev = nullptr;
    cudaError_t err = cudaHostGetDevicePointer(&dev, host_iter_buffer, 0);
    if (err != cudaSuccess) {
        cudaGetLastError();
        err = cudaHostRegister(host_iter_buffer, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable);
        if (err != cudaSuccess) return err;
        r->sink_registered = true;
        r->sink_host = host_iter_buffer;
        err = cudaHostGetDevicePointer(&dev, host_iter_buffer, 0);
        if (err != cudaSuccess) {
            drop_sink(r);
            return err;
        }
    }
    r->sink_host = host_iter_buffer;
    r->sink_dev = dev;
    return 0;
}

uint32_t fs_set_split_at(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_set_split_at(m, enable); });
    if (!r) return FS_ERROR_UNSUPPORTED;
    r->split_at = enable != 0;
    return 0;
}

#ifdef FS_TILE_TIMING
// development build only: give the LAv2 kernels a buffer of 2 x n_tiles 64-bit words for per-tile {start ns, cycles}
uint32_t fs_debug_tile_times(void *dev_buffer) {
    unsigned long long *p = static_cast<unsigned long long *>(dev_buffer);
    return cudaMemcpyToSymbol(fs::fs_tile_times, &p, sizeof(p));
}
uint32_t fs_debug_at_passes(void *dev_buffer) {
    unsigned int *p = static_cast<unsigned int *>(dev_buffer);
    unsigned int zero = 0;
    cudaMemcpyToSymbol(fs::fs_at_passes_n, &zero, sizeof(zero));
    return cudaMemcpyToSymbol(fs::fs_at_passes, &p, sizeof(p));
}
#endif
#ifdef FS_POOL_DEBUG
// development build only: read and clear the session counters of fs_lav2_pool.cuh
uint32_t fs_debug_pool_counters(uint64_t *out16) {
    unsigned long long v[16];
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(v, pool::fs_pool_dbg, sizeof(v));
    for (int i = 0; i < 16; i++) out16[i] = v[i];
    memset(v, 0, sizeof(v));
    cudaMemcpyToSymbol(pool::fs_pool_dbg, v, sizeof(v));
    return 0;
}
#endif

uint32_t fs_set_at_cycle_detection(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_set_at_cycle_detection(m, enable); });
    if (!r) return FS_ERROR_UNSUPPORTED;
    r->at_cycle = enable != 0;
    return 0;
}

uint32_t fs_set_la_step2(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_set_la_step2(m, enable); });
    if (!r) return FS_ERROR_UNSUPPORTED;
    r->use_la2 = enable != 0;
    return 0;
}

uint32_t fs_selftest_numeric_op(int32_t device, uint32_t op, const void *a, const void *b, void *out, uint64_t n) {
    const uint32_t eb = numeric_op_elem_bytes(op);
    if (eb == 0 || !a || !b || !out) return FS_ERROR_UNSUPPORTED;
    if (n == 0) return 0;
    DeviceGuard g(device);
    void *da = nullptr, *db = nullptr, *dout = nullptr;
    cudaError_t e = cudaMalloc(&da, n * eb);
    if (e == cudaSuccess) e = cudaMalloc(&db, n * eb);
    if (e == cudaSuccess) e = cudaMalloc(&dout, n * eb);
    if (e == cudaSuccess) e = cudaMemcpy(da, a, n * eb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, n * eb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        numeric_op_kernel<<<(unsigned int)((n + 255) / 256), 256>>>(op, da, db, dout, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * eb, cudaMemcpyDeviceToHost);
    cudaFree(da);
    cudaFree(db);
    cudaFree(dout);
    return e;
}

uint32_t fs_set_pool_kernel(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_set_pool_kernel(m, enable); });
    if (!r) return FS_ERROR_UNSUPPORTED;
    r->use_pool = enable != 0;
    return 0;
}

uint32_t fs_set_scaled_steps(fs_renderer *r, int32_t enable) {
    if (is_group(r)) return each_member(r, [&](fs_renderer *m) { return fs_set_scaled_steps(m, enable); });
    if (!r) return FS_ERROR_UNSUPPORTED;
    r->use_scaled = enable != 0;
    return 0;
}

void *fs_device_iter_buffer(fs_renderer *r) {
    return is_group(r) ? selected_iter_buf(r->members[0]) : r && r->iter_buf ? selected_iter_buf(r) : nullptr;
}
uint64_t fs_kernel_launch_count(const fs_renderer *r) {
    if (is_group(r)) {
        uint64_t total = 0;
        for (const fs_renderer *m : r->members) total += m->launches;
        return total;
    }
    return r ? r->launches : 0;
}

} // extern "C"
