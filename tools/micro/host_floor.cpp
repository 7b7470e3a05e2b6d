// Host-side cost of one cls_place_batch call with the GPU taken out: the C ABI's host side against the fake CUDA runtime of the tests
// (tests/native/fakecuda/), copies and kernels costing nothing - what remains is planning, 2-bit packing or staging,
// descriptors, and the scatter of the result records into the caller's arrays, on this machine's cores.  On a GPU box
// this work runs next to the kernels: it is exposed only where it exceeds them (several GPUs sharing few cores).
//   g++ -O2 -std=c++17 -pthread -Itests/native/fakecuda classeq2_b200/csrc/{capi,place_batch,resident,routed}.cpp tools/micro/host_floor.cpp \
//       tests/native/fake_kernels.cpp classeq2_b200/csrc/{index_build,host_api,host_pack,host_pool}.cpp oracle/classeq_oracle.cpp -o host_floor
//   CLS_HOST_THREADS=4 ./host_floor 10000000
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/classeq_b200.h"

namespace fakek { extern std::atomic<bool> null_placement; }

int main(int argc, char **argv) {
    const uint64_t n = argc > 1 ? strtoull(argv[1], nullptr, 10) : 2000000;
    const uint32_t len = 150;
    // a one-node model: the index is never looked at
    const uint64_t node_id[1] = {0}, child_off[2] = {0, 0}, child_idx[1] = {0}, zero[2] = {0, 0};
    const uint8_t kind[1] = {CLS_KIND_ROOT};
    cls_model_view mv{};
    mv.k_size = 35; mv.m_size = 4; mv.n_nodes = 1; mv.node_id = node_id; mv.node_kind = kind; mv.child_off = child_off; mv.child_idx = child_idx;
    mv.set_off = zero; mv.set_node_ids = zero; mv.entry_bucket = zero; mv.entry_hash = zero; mv.entry_set = zero;
    cls_index *ix = nullptr;
    if (cls_index_create(&mv, 0, &ix) != CLS_OK) { printf("index: %s\n", cls_last_error()); return 1; }
    void *pinned = nullptr;
    cudaHostAlloc(&pinned, n * len, cudaHostAllocDefault);
    std::vector<uint8_t> pageable(n * len);
    uint64_t x = 88172645463325252ull;
    for (uint64_t i = 0; i < n * len; ++i) { x ^= x << 13; x ^= x >> 7; x ^= x << 17; pageable[i] = (uint8_t)"ACGT"[x & 3]; }
    memcpy(pinned, pageable.data(), n * len);
    std::vector<uint64_t> offsets(n + 1);
    for (uint64_t i = 0; i <= n; ++i) offsets[i] = i * len;
    std::vector<uint8_t> status(n); std::vector<uint64_t> node(n); std::vector<int32_t> one(n), rest(n); std::vector<uint32_t> nq(n), nm(n), nr(n), it(n);
    cls_result res{status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data()};
    cls_params params;
    cls_params_default(&params);
    fakek::null_placement = true;
    fakecuda::skip_copies() = true;
    const char *names[] = {"", "host packing", "device packing", "mixed"};
    for (int mode = 1; mode <= 3; ++mode)
        for (int pin = 0; pin < 2; ++pin) {
            cls_set_pack_mode(mode);
            const cls_batch b{n, pin ? static_cast<const uint8_t *>(pinned) : pageable.data(), offsets.data()};
            double best = 1e30;
            cls_timing tm{};
            for (int rep = 0; rep < 4; ++rep) {
                const auto t0 = std::chrono::steady_clock::now();
                if (cls_place_batch(ix, &b, &params, &res) != CLS_OK) { printf("place: %s\n", cls_last_error()); return 1; }
                const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
                if (ms < best) { best = ms; cls_get_timing(ix, &tm); }
            }
            printf("%-15s %-8s  %8.2f ms per %llu reads  (pack/plan %.2f ms)\n", names[mode], pin ? "pinned" : "pageable", best, (unsigned long long)n, tm.pack_ms);
        }
    cls_index_destroy(ix);
    cudaFreeHost(pinned);
    return 0;
}
