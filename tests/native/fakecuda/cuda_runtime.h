// TEST INFRASTRUCTURE.  A stand-in for <cuda_runtime.h> that lets the HOST side of the library (classeq2_b200/csrc/
// capi.cpp and its neighbours: planning, packing, chunked pipeline, scatter, multi-device fan-out) compile with g++ and run
// without a GPU, under AddressSanitizer / ThreadSanitizer.  "Device" memory is malloc'ed host memory (so a copy that
// runs past a device buffer is an ASan report), events carry the host clock.  Two modes:
//   * synchronous (default): every "asynchronous" call completes before it returns - the host logic, its buffer sizes
//     and its threads are what is checked;
//   * FAKE_CUDA_ASYNC=1: every stream is a worker thread that runs what was enqueued on it in order - copies, memsets,
//     the fake kernels, event records, waits for events of other streams - while the host thread goes on.  A missing
//     dependency between streams, or between a stream and the host (a buffer reused while a copy may still read it, a
//     result read before its copy has completed), is then a DATA RACE between threads, which ThreadSanitizer reports,
//     or a wrong result.  cudaFree / cudaFreeHost wait for every stream first, as the real ones synchronise the device.
// The kernels' launch functions are supplied by tests/native/fake_kernels.cpp.  Nothing of this is ever linked into the
// product.
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <thread>

typedef int cudaError_t;
enum : int { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2, cudaErrorInvalidConfiguration = 9,
             cudaErrorInvalidDevice = 101, cudaErrorUnknown = 999 };
namespace fakecuda {
inline bool async() { static const bool a = [] { const char *e = getenv("FAKE_CUDA_ASYNC"); return e && atoi(e) != 0; }(); return a; }
inline double now_ms() { using namespace std::chrono; return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count(); }
// One cudaEventRecord: done once the stream reaches it.
struct Ticket {
    std::mutex m;
    std::condition_variable cv;
    bool done = false;
    double t_ms = 0.0;
    void signal() { { std::lock_guard<std::mutex> lk(m); done = true; t_ms = now_ms(); } cv.notify_all(); }
    void wait() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return done; }); }
};
}  // namespace fakecuda
struct FakeCudaStream {
    int device = 0;
    std::mutex m;
    std::condition_variable cv_work, cv_idle;
    std::deque<std::function<void()>> q;
    bool busy = false, stop = false;
    std::thread worker;
    void loop() {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv_work.wait(lk, [&] { return stop || !q.empty(); });
            if (q.empty()) return;                 // stop, and nothing left
            std::function<void()> f = std::move(q.front());
            q.pop_front();
            busy = true;
            lk.unlock();
            f();
            lk.lock();
            busy = false;
            if (q.empty()) cv_idle.notify_all();
        }
    }
    void push(std::function<void()> f) { { std::lock_guard<std::mutex> lk(m); q.push_back(std::move(f)); } cv_work.notify_one(); }
    void drain() { std::unique_lock<std::mutex> lk(m); cv_idle.wait(lk, [&] { return q.empty() && !busy; }); }
};
struct FakeCudaEvent { std::shared_ptr<fakecuda::Ticket> cur; double t_ms = 0.0; };
typedef FakeCudaStream *cudaStream_t;
typedef FakeCudaEvent *cudaEvent_t;
namespace fakecuda {
inline std::mutex &streams_mu() { static std::mutex m; return m; }
inline std::set<FakeCudaStream *> &streams() { static std::set<FakeCudaStream *> s; return s; }
// Runs `f` in stream order: on the stream's worker (async mode, a real stream) or right here.
inline void enqueue(cudaStream_t s, std::function<void()> f) { if (async() && s) s->push(std::move(f)); else f(); }
inline void sync_all_streams() {
    if (!async()) return;
    std::set<FakeCudaStream *> all;
    { std::lock_guard<std::mutex> lk(streams_mu()); all = streams(); }
    for (FakeCudaStream *s : all) s->drain();
}
}  // namespace fakecuda
enum cudaMemcpyKind { cudaMemcpyHostToHost = 0, cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3 };
enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2 };
enum cudaLimit { cudaLimitMaxL2FetchGranularity = 5 };
constexpr unsigned cudaStreamNonBlocking = 1, cudaHostAllocDefault = 0, cudaEventDisableTiming = 2, cudaIpcMemLazyEnablePeerAccess = 1;
struct cudaDeviceProp { int major, minor, multiProcessorCount; };
struct cudaPointerAttributes { cudaMemoryType type; };
struct cudaIpcMemHandle_t { char reserved[64]; };
struct uint2 { unsigned x, y; };
struct uint4 { unsigned x, y, z, w; };

namespace fakecuda {
inline std::mutex &mu() { static std::mutex m; return m; }
inline std::map<const char *, size_t> &pinned() { static std::map<const char *, size_t> m; return m; }   // cudaHostAlloc'ed ranges
inline int device_count() { const char *e = getenv("FAKE_CUDA_DEVICES"); const int n = e ? atoi(e) : 4; return n > 0 ? n : 4; }
inline int &current() { static thread_local int d = 0; return d; }
inline long &live_allocs() { static long n = 0; return n; }    // device + pinned allocations not yet freed (leak check of the tests)
// Fault injection: the N-th allocation from now on (device or pinned) fails, once (0: off).
inline std::atomic<long> &fail_alloc_in() { static std::atomic<long> n{0}; return n; }
inline bool alloc_fails() { long n = fail_alloc_in().load(); while (n > 0 && !fail_alloc_in().compare_exchange_weak(n, n - 1)) {} return n == 1; }
// ... and the N-th call of any of the functions below that can report an error (0: off).  A synchronising call that "fails"
// has still synchronised: what is injected is the error code, not a broken runtime.
inline std::atomic<long> &fail_call_in() { static std::atomic<long> n{0}; return n; }
inline bool call_fails() { long n = fail_call_in().load(); while (n > 0 && !fail_call_in().compare_exchange_weak(n, n - 1)) {} return n == 1; }
inline bool &skip_copies() { static bool b = false; return b; }   // host-overhead timing (tools/micro/host_floor.cpp): a DMA costs the host nothing
}  // namespace fakecuda

inline const char *cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : e == cudaErrorInvalidConfiguration ? "invalid configuration" : "fake CUDA error"; }
inline cudaError_t cudaGetLastError() { return cudaSuccess; }
inline cudaError_t cudaGetDeviceCount(int *n) { *n = fakecuda::device_count(); return cudaSuccess; }
inline cudaError_t cudaSetDevice(int d) { if (fakecuda::call_fails()) return cudaErrorUnknown; if (d < 0 || d >= fakecuda::device_count()) return cudaErrorInvalidDevice; fakecuda::current() = d; return cudaSuccess; }
inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp *p, int d) {
    if (d < 0 || d >= fakecuda::device_count()) return cudaErrorInvalidDevice;
    p->major = 10; p->minor = 0; p->multiProcessorCount = 148;
    return cudaSuccess;
}
inline cudaError_t cudaDeviceSetLimit(cudaLimit, size_t) { return cudaSuccess; }
inline cudaError_t cudaDeviceSynchronize() { fakecuda::sync_all_streams(); return cudaSuccess; }
inline cudaError_t cudaMalloc(void **p, size_t n) {
    if (fakecuda::call_fails() || fakecuda::alloc_fails()) { *p = nullptr; return cudaErrorMemoryAllocation; }
    *p = malloc(n ? n : 1);
    if (!*p) return cudaErrorMemoryAllocation;
    std::lock_guard<std::mutex> lk(fakecuda::mu());
    ++fakecuda::live_allocs();
    return cudaSuccess;
}
inline cudaError_t cudaFree(void *p) {
    fakecuda::sync_all_streams();
    if (p) { std::lock_guard<std::mutex> lk(fakecuda::mu()); --fakecuda::live_allocs(); }
    free(p);
    return cudaSuccess;
}
inline cudaError_t cudaHostAlloc(void **p, size_t n, unsigned) {
    if (fakecuda::call_fails() || fakecuda::alloc_fails()) { *p = nullptr; return cudaErrorMemoryAllocation; }
    *p = malloc(n ? n : 1);
    if (!*p) return cudaErrorMemoryAllocation;
    std::lock_guard<std::mutex> lk(fakecuda::mu());
    fakecuda::pinned()[static_cast<const char *>(*p)] = n ? n : 1;
    ++fakecuda::live_allocs();
    return cudaSuccess;
}
inline cudaError_t cudaFreeHost(void *p) {
    fakecuda::sync_all_streams();
    if (p) { std::lock_guard<std::mutex> lk(fakecuda::mu()); fakecuda::pinned().erase(static_cast<const char *>(p)); --fakecuda::live_allocs(); }
    free(p);
    return cudaSuccess;
}
inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes *a, const void *p) {
    std::lock_guard<std::mutex> lk(fakecuda::mu());
    a->type = cudaMemoryTypeUnregistered;
    auto it = fakecuda::pinned().upper_bound(static_cast<const char *>(p));
    if (it != fakecuda::pinned().begin()) {
        --it;
        if (static_cast<const char *>(p) < it->first + it->second) a->type = cudaMemoryTypeHost;
    }
    return cudaSuccess;
}
inline cudaError_t cudaMemcpy(void *d, const void *s, size_t n, cudaMemcpyKind) { if (fakecuda::call_fails()) return cudaErrorUnknown; if (n) memcpy(d, s, n); return cudaSuccess; }
// (the blocking calls and the NULL stream run on the calling thread: the library's pipelines use their own non-blocking streams)
inline cudaError_t cudaMemcpyAsync(void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t st) {
    if (fakecuda::call_fails()) return cudaErrorUnknown;
    if (n && !fakecuda::skip_copies()) fakecuda::enqueue(st, [d, s, n] { memcpy(d, s, n); });
    return cudaSuccess;
}
inline cudaError_t cudaMemset(void *d, int v, size_t n) { if (n) memset(d, v, n); return cudaSuccess; }
inline cudaError_t cudaMemsetAsync(void *d, int v, size_t n, cudaStream_t st) { if (fakecuda::call_fails()) return cudaErrorUnknown; if (n) fakecuda::enqueue(st, [d, v, n] { memset(d, v, n); }); return cudaSuccess; }
inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned) {
    if (fakecuda::call_fails()) { *s = nullptr; return cudaErrorUnknown; }
    FakeCudaStream *st = new FakeCudaStream;
    st->device = fakecuda::current();
    if (fakecuda::async()) {
        st->worker = std::thread([st] { st->loop(); });
        std::lock_guard<std::mutex> lk(fakecuda::streams_mu());
        fakecuda::streams().insert(st);
    }
    *s = st;
    return cudaSuccess;
}
inline cudaError_t cudaStreamSynchronize(cudaStream_t s) { if (fakecuda::async() && s) s->drain(); return fakecuda::call_fails() ? cudaErrorUnknown : cudaSuccess; }
inline cudaError_t cudaStreamDestroy(cudaStream_t s) {
    if (!s) return cudaSuccess;
    if (fakecuda::async()) {
        s->drain();
        { std::lock_guard<std::mutex> lk(s->m); s->stop = true; }
        s->cv_work.notify_all();
        s->worker.join();
        std::lock_guard<std::mutex> lk(fakecuda::streams_mu());
        fakecuda::streams().erase(s);
    }
    delete s;
    return cudaSuccess;
}
inline cudaError_t cudaEventCreate(cudaEvent_t *e) { if (fakecuda::call_fails()) { *e = nullptr; return cudaErrorUnknown; } *e = new FakeCudaEvent; return cudaSuccess; }
inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned) { return cudaEventCreate(e); }
inline cudaError_t cudaEventDestroy(cudaEvent_t e) { delete e; return cudaSuccess; }
// The event's fields belong to the host thread that uses it (as in the library: one workspace, one caller at a time);
// what crosses to the stream threads is the ticket of one record.
inline cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t s) {
    if (fakecuda::call_fails()) return cudaErrorUnknown;
    auto t = std::make_shared<fakecuda::Ticket>();
    e->cur = t;
    fakecuda::enqueue(s, [t] { t->signal(); });
    return cudaSuccess;
}
inline cudaError_t cudaEventSynchronize(cudaEvent_t e) { if (e->cur) e->cur->wait(); return fakecuda::call_fails() ? cudaErrorUnknown : cudaSuccess; }
inline cudaError_t cudaStreamWaitEvent(cudaStream_t s, cudaEvent_t e, unsigned) {
    if (fakecuda::call_fails()) return cudaErrorUnknown;
    if (std::shared_ptr<fakecuda::Ticket> t = e->cur) fakecuda::enqueue(s, [t] { t->wait(); });   // the record seen at the time of the call
    return cudaSuccess;
}
inline cudaError_t cudaEventElapsedTime(float *ms, cudaEvent_t a, cudaEvent_t b) {
    if (!a->cur || !b->cur) return cudaErrorInvalidValue;
    a->cur->wait(); b->cur->wait();
    *ms = (float)(b->cur->t_ms - a->cur->t_ms);
    return cudaSuccess;
}
inline cudaError_t cudaIpcGetMemHandle(cudaIpcMemHandle_t *h, void *p) { memset(h, 0, sizeof *h); memcpy(h->reserved, &p, sizeof p); return cudaSuccess; }
inline cudaError_t cudaIpcOpenMemHandle(void **p, cudaIpcMemHandle_t h, unsigned) { memcpy(p, h.reserved, sizeof *p); return cudaSuccess; }
inline cudaError_t cudaIpcCloseMemHandle(void *) { return cudaSuccess; }
