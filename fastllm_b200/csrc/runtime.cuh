// Host-side runtime pieces shared by the translation units: launch wrapper (PDL + opt-in shared memory + per-kernel event
// profile + launch counter), device buffer RAII, thread-local error slot, host bf16 rounding.
#pragma once
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace fl {

extern thread_local std::string g_last_error;
extern std::atomic<uint64_t> g_launches;

struct ProfEntry {
    std::string tag;
    uint64_t bytes;
    cudaEvent_t e0, e1;
};
struct Profiler {
    bool on = false;
    std::vector<ProfEntry> entries;
};
extern Profiler g_prof;

inline bool env_flag(const char* name) {
    const char* v = std::getenv(name);
    return v != nullptr && v[0] != '\0' && v[0] != '0';
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// f32 -> bf16 bits, round to nearest even
inline uint16_t host_f32_to_bf16(float f) {
    uint32_t b;
    std::memcpy(&b, &f, 4);
    if ((b & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((b >> 16) | 0x40u);   // NaN stays NaN (quiet), as half::bf16::from_f32 does
    return (uint16_t)((b + 0x7FFFu + ((b >> 16) & 1u)) >> 16);
}

struct LaunchCtx {
    cudaStream_t stream = nullptr;
    bool pdl = !env_flag("FL_NO_PDL");   // programmatic dependent launch on every kernel of the step
    bool capturing = false;   // inside cudaStreamBeginCapture: no events, no profile
    uint64_t captured = 0;    // kernels recorded into the graph being captured
    bool cooperative = false; // cooperative launch: every CTA of the grid co-resident (the persistent decode kernel)
};

// One launch (kernel or NCCL call) enqueued on lc: counted into the graph being captured, or into fl_launch_count.
inline void count_launch(LaunchCtx& lc) {
    if (lc.capturing)
        lc.captured++;
    else
        g_launches.fetch_add(1, std::memory_order_relaxed);
}

// Raises `kern`'s opt-in dynamic shared-memory limit to at least `bytes`.  Idempotent and safe from several threads: the largest
// size set so far is remembered per kernel (attributes are per device; a process drives one, see fl_init).
inline void ensure_smem_optin(const void* kern, size_t bytes) {
    static std::mutex mu;
    static std::map<const void*, size_t> raised;
    std::lock_guard<std::mutex> lk(mu);
    size_t& cur = raised[kern];
    if (bytes <= cur) return;
    FL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
}

// Launches `kern` with optional PDL.  `tag`/`bytes` feed the per-kernel profile (algorithmic bytes of that launch).  Inside a
// profile window kernels run without PDL, so that each one's events bracket it alone.
template <typename... KArgs, typename... Args>
inline void launch(LaunchCtx& lc, const char* tag, uint64_t bytes, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                   Args&&... args) {
    if (smem > 48 * 1024) ensure_smem_optin((const void*)kern, smem);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = lc.stream;
    cudaLaunchAttribute attr[2];
    cfg.attrs = attr;
    const bool prof = g_prof.on && !lc.capturing;
    if (lc.pdl && !prof) {
        attr[cfg.numAttrs].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[cfg.numAttrs++].val.programmaticStreamSerializationAllowed = 1;
    }
    if (lc.cooperative) {
        attr[cfg.numAttrs].id = cudaLaunchAttributeCooperative;
        attr[cfg.numAttrs++].val.cooperative = 1;
    }
    ProfEntry pe;
    if (prof) {
        pe.tag = tag;
        pe.bytes = bytes;
        FL_CUDA(cudaEventCreate(&pe.e0));
        FL_CUDA(cudaEventCreate(&pe.e1));
        FL_CUDA(cudaEventRecord(pe.e0, lc.stream));
    }
    FL_CUDA(cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...));
    if (prof) {
        FL_CUDA(cudaEventRecord(pe.e1, lc.stream));
        g_prof.entries.push_back(pe);
    }
    count_launch(lc);
}

// a start / stop event pair that cannot leak when something between create and destroy throws
struct EventPair {
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    EventPair() {
        FL_CUDA(cudaEventCreate(&e0));
        if (cudaEventCreate(&e1) != cudaSuccess) {
            cudaEventDestroy(e0);
            throw Error(-2, "cudaEventCreate failed");
        }
    }
    EventPair(const EventPair&) = delete;
    EventPair& operator=(const EventPair&) = delete;
    ~EventPair() {
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    }
};

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void alloc(size_t count, bool zero = false) {
        release();
        n = count;
        if (count == 0) return;
        FL_CUDA(cudaMalloc(&p, count * sizeof(T)));
        if (zero) FL_CUDA(cudaMemset(p, 0, count * sizeof(T)));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

template <typename T>
struct PinnedBuf {
    T* p = nullptr;
    size_t n = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf() {
        if (p) cudaFreeHost(p);
    }
    void alloc(size_t count) {
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = count;
        if (count) FL_CUDA(cudaMallocHost(&p, count * sizeof(T)));
    }
};

}  // namespace fl
