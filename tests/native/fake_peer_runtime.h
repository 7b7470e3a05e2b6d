// TEST INFRASTRUCTURE.  The peer-access calls of the CUDA runtime on top of the fake runtime (tests/native/fakecuda/):
// every pair of distinct fake devices can reach each other (FAKE_CUDA_NO_PEER=1: none can); enabling a pair twice
// reports cudaErrorPeerAccessAlreadyEnabled, as the real runtime does.  Force-included (-include) into
// classeq2_b200/csrc/capi_sharded.cu by tests/test_sharded_handle.py.
#pragma once
#include <cuda_runtime.h>

#include <set>
#include <utility>

constexpr cudaError_t cudaErrorPeerAccessAlreadyEnabled = 704;

inline cudaError_t cudaDeviceCanAccessPeer(int *can, int d, int peer) {
    if (fakecuda::call_fails()) return cudaErrorUnknown;
    if (d < 0 || d >= fakecuda::device_count() || peer < 0 || peer >= fakecuda::device_count()) return cudaErrorInvalidDevice;
    const char *e = getenv("FAKE_CUDA_NO_PEER");
    *can = d != peer && !(e && atoi(e) != 0);
    return cudaSuccess;
}
inline cudaError_t cudaDeviceEnablePeerAccess(int peer, unsigned) {
    if (fakecuda::call_fails()) return cudaErrorUnknown;
    if (peer < 0 || peer >= fakecuda::device_count() || peer == fakecuda::current()) return cudaErrorInvalidDevice;
    static std::set<std::pair<int, int>> enabled;
    std::lock_guard<std::mutex> lk(fakecuda::mu());
    return enabled.insert({fakecuda::current(), peer}).second ? cudaSuccess : cudaErrorPeerAccessAlreadyEnabled;
}
