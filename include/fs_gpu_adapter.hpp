// fs_gpu_adapter.hpp -- the reference's `GPURenderer` class (FractalSharkLib/GPU_Render.h:20-227) re-created, header-only,
// on top of the C-ABI of fs_gpu.h (libfsgpu.so).
//
// How a FractalShark maintainer uses it: compile FractalSharkLib with this header in place of GPU_Render.h's class body
// (`#include "fs_gpu_adapter.hpp"` from GPU_Render.h after its own includes of BLA.h / BLAS.h / LAstep.h / GPU_Types.h, with
// LAReference.h visible) and link `fsgpu` instead of FractalSharkGpuLib.  Fractal.cpp, RenderThreadPool.cpp and
// FractalSharkCli stay as they are: every public member of the reference class is here with the same template
// parameters, argument order and return convention (uint32_t: 0, a cudaError_t, or a FractalSharkError).
//
// The header needs the reference's own types in scope (RenderAlgorithm, Color16, ReductionResults, GPUPerturbResults,
// LAReference, BLAS, HDRFloat, CudaDblflt, MattDblflt ...); it adds none of its own.  All tables cross the boundary as the
// bytes the reference already holds (layouts asserted in fractalshark_b200/csrc/fs_capi.cu).
// tests/test_adapter.py compiles it against the reference headers (every member template instantiated) and runs
// oracle/_ref/adapter_driver -- a C++ program that renders through this class from the reference's own
// PerturbationResults / LAReference objects -- against the committed reference-kernel fixtures.
#ifndef FS_GPU_ADAPTER_HPP
#define FS_GPU_ADAPTER_HPP

#include "fs_gpu.h"

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <mutex>
#include <vector>

#ifndef FS_GPU_ADAPTER_CLASS
#define FS_GPU_ADAPTER_CLASS GPURenderer // the name Fractal.cpp and RenderThreadPool.cpp use
#endif

namespace fs_gpu_adapter {

// template argument T of the reference entry points -> fs_numeric tag (INTEGRATION.md "Tag mapping")
template <class T> struct NumericTag;
template <> struct NumericTag<float> { static constexpr int32_t v = FS_NUM_F32; };
template <> struct NumericTag<double> { static constexpr int32_t v = FS_NUM_F64; };
template <> struct NumericTag<CudaDblflt<MattDblflt>> { static constexpr int32_t v = FS_NUM_2X32; };
template <> struct NumericTag<HDRFloat<float>> { static constexpr int32_t v = FS_NUM_HDR32; };
template <> struct NumericTag<HDRFloat<double>> { static constexpr int32_t v = FS_NUM_HDR64; };
template <> struct NumericTag<HDRFloat<CudaDblflt<MattDblflt>>> { static constexpr int32_t v = FS_NUM_HDR2X32; };
template <> struct NumericTag<MattDblflt> { static constexpr int32_t v = FS_NUM_2X32; };  // Gpu2x32   GPU_Render.cu:733-771
template <> struct NumericTag<MattDbldbl> { static constexpr int32_t v = FS_NUM_2X64; };  // Gpu2x64
template <> struct NumericTag<MattQFltflt> { static constexpr int32_t v = FS_NUM_4X32; }; // Gpu4x32
template <> struct NumericTag<MattQDbldbl> { static constexpr int32_t v = FS_NUM_4X64; }; // Gpu4x64

// GPUPerturbResults<IterType, T, PExtras> (GPU_Types.h:83-175) -> fs_orbit; xl / yl outlive the call
template <class P, class T> fs_orbit orbit_of(const P *p, T &xl, T &yl) {
    xl = p->GetOrbitXLow();
    yl = p->GetOrbitYLow();
    return fs_orbit{p->GetFullOrbit(), (uint64_t)p->GetCompressedSize(), (uint64_t)p->GetUncompressedSize(),
                    (uint64_t)p->GetPeriodMaybeZero(), &xl, &yl};
}

} // namespace fs_gpu_adapter

class FS_GPU_ADAPTER_CLASS {
public:
    // the reference drives device 0 (GPU_Render.cu:113); FS_GPU_DEVICES=0,1,... renders every frame on the listed GPUs
    FS_GPU_ADAPTER_CLASS() : m_Impl(fs_create_default()) {}
    ~FS_GPU_ADAPTER_CLASS() { fs_destroy(m_Impl); }
    FS_GPU_ADAPTER_CLASS(const FS_GPU_ADAPTER_CLASS &) = delete;
    FS_GPU_ADAPTER_CLASS &operator=(const FS_GPU_ADAPTER_CLASS &) = delete;

    static uint32_t TestCudaIsWorking() { return fs_test_cuda_is_working(); } // GPU_Render.h:25

    template <typename IterType, class T> // GPU_Render.h:27-35
    uint32_t Render(RenderAlgorithm algorithm, T cx, T cy, T dx, T dy, IterType n_iterations, int iteration_precision) {
        return fs_render(m_Impl, (uint32_t)algorithm.Algorithm, fs_gpu_adapter::NumericTag<T>::v, &cx, &cy, &dx, &dy,
                         (uint64_t)n_iterations, iteration_precision);
    }

    template <typename IterType, class T> // GPU_Render.h:37-49
    uint32_t RenderPerturbBLAScaled(RenderAlgorithm algorithm,
                                    const GPUPerturbResults<IterType, T, PerturbExtras::Bad> *double_perturb,
                                    const GPUPerturbResults<IterType, float, PerturbExtras::Bad> *float_perturb, T cx, T cy, T dx,
                                    T dy, T centerX, T centerY, IterType n_iterations, int iteration_precision) {
        T xl, yl;
        float fxl, fyl;
        fs_orbit od = fs_gpu_adapter::orbit_of(double_perturb, xl, yl), of = fs_gpu_adapter::orbit_of(float_perturb, fxl, fyl);
        return fs_render_perturb_bla_scaled(m_Impl, (uint32_t)algorithm.Algorithm, fs_gpu_adapter::NumericTag<T>::v, &od, &of, &cx,
                                            &cy, &dx, &dy, &centerX, &centerY, (uint64_t)n_iterations, iteration_precision);
    }

    template <typename IterType, class T> // GPU_Render.h:65-77 (the MattDblflt overload at :51-63 is never instantiated)
    uint32_t RenderPerturbBLA(RenderAlgorithm algorithm, const GPUPerturbResults<IterType, T, PerturbExtras::Disable> *results,
                              BLAS<IterType, T> *blas, T cx, T cy, T dx, T dy, T centerX, T centerY, IterType n_iterations,
                              int iteration_precision) {
        std::vector<const void *> levels;
        std::vector<uint64_t> counts;
        for (auto &level : blas->m_B) { // BLAS.h:20-22: m_B[level] -> BLA<T>[], levels below m_FirstLevel are empty
            levels.push_back(level.empty() ? nullptr : static_cast<const void *>(level.data()));
            counts.push_back((uint64_t)level.size());
        }
        T xl, yl;
        fs_orbit o = fs_gpu_adapter::orbit_of(results, xl, yl);
        fs_blas b{levels.data(), counts.data(), (uint32_t)levels.size(), (uint32_t)BLAS<IterType, T>::m_FirstLevel, (int32_t)blas->m_LM2};
        return fs_render_perturb_bla(m_Impl, (uint32_t)algorithm.Algorithm, fs_gpu_adapter::NumericTag<T>::v, &o, &b, &cx, &cy, &dx,
                                     &dy, &centerX, &centerY, (uint64_t)n_iterations, iteration_precision);
    }

    template <typename IterType, class T, class SubType, LAv2Mode Mode, PerturbExtras PExtras> // GPU_Render.h:79-88
    uint32_t RenderPerturbLAv2(RenderAlgorithm algorithm, T cx, T cy, T dx, T dy, T centerX, T centerY, IterType n_iterations) {
        return fs_render_perturb_lav2(m_Impl, (uint32_t)algorithm.Algorithm, fs_gpu_adapter::NumericTag<T>::v, (int32_t)Mode,
                                      (int32_t)PExtras, &cx, &cy, &dx, &dy, &centerX, &centerY, (uint64_t)n_iterations);
    }

    template <typename IterType> // GPU_Render.h:91-100
    uint32_t InitializeMemory(uint32_t w, uint32_t h, uint32_t antialiasing, const Color16 *palInterleaved, uint32_t palIters,
                              uint32_t paletteAuxDepth, uint64_t paletteGeneration, bool expectedReuse) {
        static_assert(sizeof(Color16) == sizeof(fs_color16), "Color16 layout (GPU_Types.h:14-16)");
        return fs_initialize_memory(m_Impl, (uint32_t)sizeof(IterType), w, h, antialiasing,
                                    reinterpret_cast<const fs_color16 *>(palInterleaved), palIters, paletteAuxDepth,
                                    paletteGeneration, expectedReuse ? 1 : 0);
    }

    template <typename IterType, class T1, class SubType, PerturbExtras PExtras, class T2> // GPU_Render.h:102-108
    uint32_t InitializePerturb(size_t GenerationNumber1, const GPUPerturbResults<IterType, T1, PExtras> *Perturb1,
                               size_t GenerationNumber2, const GPUPerturbResults<IterType, T2, PExtras> *Perturb2,
                               const LAReference<IterType, T1, SubType, PExtras> *LaReferenceHost) {
        T1 x1, y1;
        T2 x2, y2;
        fs_orbit o1{}, o2{};
        if (Perturb1) o1 = fs_gpu_adapter::orbit_of(Perturb1, x1, y1);
        if (Perturb2) o2 = fs_gpu_adapter::orbit_of(Perturb2, x2, y2);
        fs_la_reference la{};
        if (LaReferenceHost) {
            const auto &las = LaReferenceHost->GetLAs();       // LAReference.h:238-248
            const auto &stages = LaReferenceHost->GetLAStages(); // LAReference.h:250-260
            la = fs_la_reference{las.GetData(),
                                 (uint64_t)las.GetSize(),
                                 stages.GetData(),
                                 (uint64_t)stages.GetSize(),
                                 &LaReferenceHost->GetAT(),
                                 (uint64_t)LaReferenceHost->GetLAStageCount(),
                                 LaReferenceHost->UseAT() ? 1 : 0,
                                 LaReferenceHost->IsValid() ? 1 : 0};
        }
        return fs_initialize_perturb(m_Impl, (uint32_t)sizeof(IterType), fs_gpu_adapter::NumericTag<T1>::v, (int32_t)PExtras,
                                     (uint64_t)GenerationNumber1, Perturb1 ? &o1 : nullptr, fs_gpu_adapter::NumericTag<T2>::v,
                                     (uint64_t)GenerationNumber2, Perturb2 ? &o2 : nullptr, LaReferenceHost ? &la : nullptr);
    }

    template <typename IterType> void ClearMemory() { fs_clear_memory(m_Impl); } // GPU_Render.h:110-111

    static const char *ConvertErrorToString(uint32_t err) { return fs_convert_error_to_string(err); } // GPU_Render.h:113

    // Match in Fractal.cpp (GPU_Render.h:116-120): the padding of the iteration and colour buffers
    static const int32_t NB_THREADS_W = 16;
    static const int32_t NB_THREADS_H = 8;
    static const int32_t NB_THREADS_W_AA = 16;
    static const int32_t NB_THREADS_H_AA = 8;

    template <typename IterType> // GPU_Render.h:123-129
    uint32_t RenderCurrent(IterType n_iterations, IterType *iter_buffer, Color16 *color_buffer, ReductionResults *reduction_results,
                           bool progressive = false) {
        static_assert(sizeof(ReductionResults) == sizeof(fs_reduction), "ReductionResults layout (GPU_Types.h:40-50)");
        return fs_render_current(m_Impl, (uint64_t)n_iterations, iter_buffer, reinterpret_cast<fs_color16 *>(color_buffer),
                                 reinterpret_cast<fs_reduction *>(reduction_results), progressive ? 1 : 0);
    }

    uint32_t SyncComputeStream() { return fs_sync_compute_stream(m_Impl); }   // GPU_Render.h:131
    uint32_t SyncDisplayStream() { return fs_sync_display_stream(m_Impl); }   // GPU_Render.h:132
    uint32_t QueryComputeStream() { return fs_query_compute_stream(m_Impl); } // GPU_Render.h:133
    uint32_t EnqueueComputeDoneCallback() {                                   // GPU_Render.h:134, GPU_Render.cu:603-615
        return fs_enqueue_compute_done_callback(
            m_Impl, [](void *self) { static_cast<FS_GPU_ADAPTER_CLASS *>(self)->SignalComputeDone(); }, this);
    }

    // GPU_Render.h:136-155: host-side completion flag, unchanged
    void ResetComputeDoneFlag() { m_ComputeDoneFlag.store(false, std::memory_order_release); }
    bool IsComputeDone() const { return m_ComputeDoneFlag.load(std::memory_order_acquire); }
    void SignalComputeDone() {
        m_ComputeDoneFlag.store(true, std::memory_order_release);
        if (m_ComputeDoneMutex && m_ComputeDoneCV) {
            std::lock_guard<std::mutex> lk(*m_ComputeDoneMutex);
            m_ComputeDoneCV->notify_all();
        }
    }
    void SetComputeDoneNotification(std::mutex *mutex, std::condition_variable *cv) {
        m_ComputeDoneMutex = mutex;
        m_ComputeDoneCV = cv;
    }

    uint32_t GetWidth() const { return fs_get_width(m_Impl); }   // GPU_Render.h:157
    uint32_t GetHeight() const { return fs_get_height(m_Impl); } // GPU_Render.h:158

    // ---- beyond the reference's interface (optional) ----------------------------------------------------------------
    // one process per GPU, same inputs to each: renderer i of n renders the 4-row bands b % n == i (a device group, see the
    // constructor, needs none of this)
    uint32_t SetShard(uint32_t shard_count, uint32_t shard_index) { return fs_set_shard(m_Impl, shard_count, shard_index); }
    // the LAv2 kernels stream finished pixels into a page-locked host frame (e.g. the ItersMemoryContainer buffer)
    uint32_t SetResultSink(void *host_iter_buffer, uint64_t bytes) { return fs_set_result_sink(m_Impl, host_iter_buffer, bytes); }
    fs_renderer *Handle() { return m_Impl; }

private:
    fs_renderer *m_Impl;
    std::atomic<bool> m_ComputeDoneFlag{false};
    std::mutex *m_ComputeDoneMutex{nullptr};
    std::condition_variable *m_ComputeDoneCV{nullptr};
};

#endif // FS_GPU_ADAPTER_HPP
