// common.h — host plumbing shared by the engine's translation units: error reporting across the
// C ABI (never throw, never abort: include/lzkp_b200.h "Conventions"), launch counting, device
// buffers.  Definitions live in engine.cu.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/lzkp_b200.h"

namespace lzkp {
namespace eng {

int fail(int code, const std::string &msg);      // records the thread-local message, returns code
extern std::atomic<uint64_t> g_launches;         // kernels launched by this process (bench.py gpu_launches)
int ensure_device();                             // LZKP_E_NO_DEVICE when no GPU: there is no CPU fallback
int current_device();                            // the device ensure_device() binds the calling thread to (-1: none yet)
// Binds the calling thread to one device of the engine's device list for the scope's lifetime (replica worker
// threads of a multi-device proving key); ensure_device() inside the scope selects that device.
struct DeviceScope {
    int prev;
    explicit DeviceScope(int dev);
    ~DeviceScope();
    DeviceScope(const DeviceScope &) = delete;
    DeviceScope &operator=(const DeviceScope &) = delete;
};

struct DBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int alloc(size_t n);
    int ensure(size_t n) { return n <= bytes ? LZKP_OK : alloc(n); }
    void release();
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    ~DBuf() { release(); }
    DBuf() = default;
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
};

}  // namespace eng
}  // namespace lzkp

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return ::lzkp::eng::fail(LZKP_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));   \
    } while (0)
#define TRY(expr)                       \
    do {                                \
        int rc_ = (expr);               \
        if (rc_ != LZKP_OK) return rc_; \
    } while (0)
#define LAUNCH(kernel, grid, block, smem, stream, ...)                          \
    do {                                                                        \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);             \
        ::lzkp::eng::g_launches.fetch_add(1, std::memory_order_relaxed);        \
    } while (0)

namespace lzkp {
namespace eng {
// Buffers shared by calls on several streams: every user makes its stream wait on the buffers' last use (the event is
// created by the first user) and records it after its own last enqueue.
inline int event_acquire(cudaEvent_t &last_use, cudaStream_t st) {
    if (!last_use) CUDA_TRY(cudaEventCreateWithFlags(&last_use, cudaEventDisableTiming));
    else CUDA_TRY(cudaStreamWaitEvent(st, last_use, 0));
    return LZKP_OK;
}
inline int event_release(cudaEvent_t last_use, cudaStream_t st) {
    CUDA_TRY(cudaEventRecord(last_use, st));
    return LZKP_OK;
}
template <class T>
inline int upload(DBuf &b, const std::vector<T> &v) {
    TRY(b.alloc(v.size() * sizeof(T)));
    if (!v.empty()) CUDA_TRY(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return LZKP_OK;
}
}  // namespace eng
}  // namespace lzkp
