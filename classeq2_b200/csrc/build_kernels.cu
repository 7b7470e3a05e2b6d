// cls_model_build_device: the k-mer -> node-set map of the reference's `build-db`
// (map_kmers_to_tree, core/src/use_cases/build_database/mod.rs:26-181) built on the GPU - SURVEY.md
// section 8f, row 4.  Same result as the host builder cls_model_build (host_api.cpp): entries in
// (hash, bucket key) order, node sets numbered in order of their first entry, every tip paired with its own
// sequence.  The steps and their index arithmetic are described in build_steps.hpp; this file holds the
// kernels, the CUB sorts / scans between them and the C ABI entry point.  There is no CPU fallback: without
// a device the call fails with CLS_ERR_CUDA.
//
// Bounds: HBM for the sorts (two 64-bit radix sorts over all occurrences), instruction issue for the
// hashing kernel (byte-wise murmur3 of every window, any k).  No tensor cores: integer hashing and sorting.
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cstdint>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/classeq_b200.h"
#include "build_prep.hpp"
#include "build_steps.hpp"
#include "built_model.hpp"
#include "last_error.hpp"
#include "murmur3_device.cuh"

namespace {

using namespace cls::build;

// ---- kernels ---------------------------------------------------------------------------------------

// One CTA per (tip, tile of windows): the tile's bytes and their reverse complement are staged in shared
// memory once (coalesced), then every thread hashes windows of both strands from there
// (kmers_map.rs:375-398 build_kmer_from_string; :157-159 hash_kmer; :10-13 / :131-137 bucket key).
__global__ void __launch_bounds__(256) build_hash_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ seq_off,
                                                         const uint32_t *__restrict__ seq_len, const uint64_t *__restrict__ occ_off,
                                                         const HashItem *__restrict__ items, uint32_t k, uint32_t m,
                                                         uint32_t strand_bytes, uint64_t *__restrict__ out_hash,
                                                         uint64_t *__restrict__ out_bucket, uint32_t *__restrict__ out_rank) {
    extern __shared__ __align__(16) uint8_t tile[];
    uint8_t *f = tile, *r = tile + strand_bytes;
    const HashItem it = items[blockIdx.x];
    const uint64_t W = (uint64_t)seq_len[it.rank] - k + 1;
    const uint64_t w0 = (uint64_t)it.tile * kTileWindows;
    const uint32_t nw = (uint32_t)(W - w0 < kTileWindows ? W - w0 : kTileWindows);
    const uint32_t nb = nw + k - 1;
    const uint8_t *src = bases + seq_off[it.rank] + w0;
    for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) {
        const uint8_t c = src[i] & 0xDFu;   // upper-case, both strands (kmers_map.rs:410); letters were checked on the host
        f[i] = c;
        r[nb - 1 - i] = comp_byte(c);
    }
    __syncthreads();
    const uint64_t base = occ_off[it.rank];
    const uint32_t mm = m < k ? m : k;
    for (uint32_t x = threadIdx.x; x < 2 * nw; x += blockDim.x) {
        const TileItem ti = tile_item(x, nw, W, w0);
        const uint8_t *s = ti.strand ? r : f;
        const uint64_t o = base + ti.occ;
        out_hash[o] = cls::murmur_window_generic(s, ti.pos, k);
        out_bucket[o] = m == 0 ? 0ull : cls::murmur_window_generic(s, ti.pos, mm);
        out_rank[o] = it.rank;
    }
}

__global__ void iota_kernel(uint32_t *v, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) v[i] = (uint32_t)i;
}

template <typename T>
__global__ void gather_kernel(const T *__restrict__ src, const uint32_t *__restrict__ idx, T *__restrict__ dst, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[idx[i]];
}

__global__ void flags_kernel(const uint64_t *__restrict__ hash, const uint64_t *__restrict__ bucket, const uint32_t *__restrict__ rank,
                             uint64_t *__restrict__ flags, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        flags[i] = occ_flags(hash, bucket, rank, i);
}

// scan[i] = exclusive sum of the flags: low half = entry index, high half = tip-list position
__global__ void scatter_entries_kernel(const uint64_t *__restrict__ hash, const uint64_t *__restrict__ bucket,
                                       const uint32_t *__restrict__ rank, const uint64_t *__restrict__ flags,
                                       const uint64_t *__restrict__ scan, uint64_t n, uint64_t *__restrict__ entry_hash,
                                       uint64_t *__restrict__ entry_bucket, uint32_t *__restrict__ list_off, uint32_t *__restrict__ tips) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t fl = flags[i], sc = scan[i];
        const uint32_t e = (uint32_t)sc, t = (uint32_t)(sc >> 32);
        if (fl & 1ull) { entry_hash[e] = hash[i]; entry_bucket[e] = bucket[i]; list_off[e] = t; }
        if (fl >> 32) tips[t] = rank[i];
    }
}

__global__ void fingerprint_kernel(const uint32_t *__restrict__ list_off, const uint32_t *__restrict__ tips, uint64_t *__restrict__ fp,
                                   uint32_t *__restrict__ eid, uint32_t n_entries) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n_entries; e += gridDim.x * blockDim.x) {
        fp[e] = list_fingerprint(tips + list_off[e], list_off[e + 1] - list_off[e]);
        eid[e] = e;
    }
}

// In fingerprint order: position p starts a new node set unless its tip list equals its predecessor's.
// seg_head[p] = p for such positions, 0 otherwise (a running maximum then gives every position its head).
__global__ void seg_head_kernel(const uint64_t *__restrict__ fp_sorted, const uint32_t *__restrict__ eid_sorted,
                                const uint32_t *__restrict__ list_off, const uint32_t *__restrict__ tips,
                                uint32_t *__restrict__ seg_head, uint32_t n_entries) {
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_entries; p += gridDim.x * blockDim.x) {
        bool same = false;
        if (p > 0 && fp_sorted[p] == fp_sorted[p - 1]) {
            const uint32_t a = eid_sorted[p], b = eid_sorted[p - 1];
            same = lists_equal(tips + list_off[a], list_off[a + 1] - list_off[a], tips + list_off[b], list_off[b + 1] - list_off[b]);
        }
        seg_head[p] = same ? 0u : p;
    }
}

struct MaxOp {
    __host__ __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// rep[e] = the first entry (smallest index: the sort is stable) with the same tip list; is_rep[e] = (rep[e] == e)
__global__ void rep_kernel(const uint32_t *__restrict__ eid_sorted, const uint32_t *__restrict__ head_pos, uint32_t *__restrict__ rep,
                           uint32_t *__restrict__ is_rep, uint32_t n_entries) {
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_entries; p += gridDim.x * blockDim.x) {
        const uint32_t e = eid_sorted[p], r = eid_sorted[head_pos[p]];
        rep[e] = r;
        is_rep[e] = e == r ? 1u : 0u;
    }
}

// set_idx = exclusive sum of is_rep in entry order: sets are numbered in order of their first entry
__global__ void entry_set_kernel(const uint32_t *__restrict__ rep, const uint32_t *__restrict__ is_rep, const uint32_t *__restrict__ set_idx,
                                 uint64_t *__restrict__ entry_set, uint32_t *__restrict__ set_rep, uint32_t n_entries) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n_entries; e += gridDim.x * blockDim.x) {
        entry_set[e] = set_idx[rep[e]];
        if (is_rep[e]) set_rep[set_idx[e]] = e;
    }
}

// Node sets (clade.rs:127-156 get_leaves_with_paths: the ids on the root -> tip path, both ends included;
// kmers_map.rs:119-155: the set of an entry is the union over the tips that contain the k-mer).
__global__ void set_size_kernel(const int32_t *__restrict__ parent, const uint32_t *__restrict__ depth, const uint32_t *__restrict__ rank_node,
                                const uint32_t *__restrict__ set_rep, const uint32_t *__restrict__ list_off, const uint32_t *__restrict__ tips,
                                uint64_t *__restrict__ sizes, uint32_t n_sets) {
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n_sets; s += gridDim.x * blockDim.x) {
        const uint32_t e = set_rep[s];
        sizes[s] = set_size(parent, depth, rank_node, tips + list_off[e], list_off[e + 1] - list_off[e]);
    }
}
__global__ void set_fill_kernel(const int32_t *__restrict__ parent, const uint32_t *__restrict__ depth, const uint32_t *__restrict__ rank_node,
                                const uint64_t *__restrict__ node_id, const uint32_t *__restrict__ set_rep, const uint32_t *__restrict__ list_off,
                                const uint32_t *__restrict__ tips, const uint64_t *__restrict__ set_off, uint64_t *__restrict__ set_nodes,
                                uint32_t n_sets) {
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n_sets; s += gridDim.x * blockDim.x) {
        const uint32_t e = set_rep[s];
        set_fill(parent, depth, rank_node, node_id, tips + list_off[e], list_off[e + 1] - list_off[e], set_nodes + set_off[s]);
    }
}

// ---- host side ---------------------------------------------------------------------------------------

// Device allocations of one call, released together.
struct Arena {
    std::vector<void *> ptrs;
    ~Arena() { for (void *p : ptrs) cudaFree(p); }
    template <typename T>
    cudaError_t alloc(T **out, uint64_t n) {
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, (n ? n : 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = static_cast<T *>(p);
        return e;
    }
    void free_one(void *p) {
        for (auto &q : ptrs)
            if (q == p) { cudaFree(p); q = ptrs.back(); ptrs.pop_back(); return; }
    }
};

struct StreamGuard {
    cudaStream_t s = nullptr;
    ~StreamGuard() { if (s) cudaStreamDestroy(s); }
};

inline uint32_t grid_for(uint64_t n, int sm_count) {
    const uint64_t need = (n + 255) / 256, cap = (uint64_t)sm_count * 8;  // grid-stride loops: a few CTAs per SM
    return (uint32_t)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace

#define BK_TRY(expr)                                                                                            \
    do {                                                                                                        \
        cudaError_t _e = (expr);                                                                                \
        if (_e != cudaSuccess)                                                                                  \
            return cls::set_last_error(_e == cudaErrorMemoryAllocation ? CLS_ERR_OUT_OF_MEMORY : CLS_ERR_CUDA,  \
                                       std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
    } while (0)

static int build_device(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node, const uint8_t *bases,
                        const uint64_t *offsets, int device, cls_built_model **out) {
    using cls::set_last_error;
    if (!tree || !out || (n_tips && (!tip_node || !offsets || !bases))) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    Prep pr;
    {
        std::string err;
        const int rc = prepare(tree, n_tips, tip_node, offsets, pr, err, bases);
        if (rc != CLS_OK) return set_last_error(rc, err);
    }
    const uint32_t k = tree->k_size, m = tree->m_size;
    const uint64_t n_nodes = tree->n_nodes;
    const uint64_t N = pr.occ_off[n_tips];
    if (N > 0x7FFFFFFFull) return set_last_error(CLS_ERR_UNSUPPORTED, "more than 2^31 - 1 k-mer occurrences");
    const uint32_t strand_bytes = (kTileWindows + k - 1 + 15u) & ~15u;
    const size_t tile_smem = (size_t)2 * strand_bytes;
    if ((uint64_t)k > 100 * 1024 || tile_smem > 200 * 1024) return set_last_error(CLS_ERR_UNSUPPORTED, "k_size beyond the tile of the hashing kernel");

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) {
        cudaGetLastError();
        return set_last_error(CLS_ERR_CUDA, "no usable CUDA device (cls_model_build_device has no CPU fallback)");
    }
    if (device < 0 || device >= n_dev) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "device out of range");
    BK_TRY(cudaSetDevice(device));
    int sm_count = 0;
    BK_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));

    auto bm = new cls_built_model();
    std::unique_ptr<cls_built_model> guard(bm);
    bm->k_size = k; bm->m_size = m;
    bm->set_off.push_back(0);
    if (N == 0) { *out = guard.release(); return CLS_OK; }

    StreamGuard sg;  // every call below is ordered on this stream
    BK_TRY(cudaStreamCreateWithFlags(&sg.s, cudaStreamNonBlocking));
    cudaStream_t st = sg.s;
    Arena ar;
    // ---- 1. occurrences ------------------------------------------------------------------------------
    const uint64_t base_lo = offsets[0], base_hi = offsets[n_tips];
    uint8_t *d_bases; uint64_t *d_seq_off, *d_occ_off; uint32_t *d_seq_len; HashItem *d_items;
    BK_TRY(ar.alloc(&d_bases, base_hi - base_lo));
    BK_TRY(ar.alloc(&d_seq_off, n_tips));
    BK_TRY(ar.alloc(&d_seq_len, n_tips));
    BK_TRY(ar.alloc(&d_occ_off, n_tips + 1));
    BK_TRY(ar.alloc(&d_items, pr.items.size()));
    for (auto &o : pr.seq_off) o -= base_lo;
    BK_TRY(cudaMemcpyAsync(d_bases, bases + base_lo, base_hi - base_lo, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_seq_off, pr.seq_off.data(), n_tips * 8, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_seq_len, pr.seq_len.data(), n_tips * 4, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_occ_off, pr.occ_off.data(), (n_tips + 1) * 8, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_items, pr.items.data(), pr.items.size() * sizeof(HashItem), cudaMemcpyHostToDevice, st));
    uint64_t *A, *B, *K, *H1; uint32_t *R, *I0, *I1;
    BK_TRY(ar.alloc(&A, N)); BK_TRY(ar.alloc(&B, N)); BK_TRY(ar.alloc(&K, N)); BK_TRY(ar.alloc(&H1, N));
    BK_TRY(ar.alloc(&R, N)); BK_TRY(ar.alloc(&I0, N)); BK_TRY(ar.alloc(&I1, N));
    BK_TRY(cudaFuncSetAttribute(build_hash_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem));
    build_hash_kernel<<<(uint32_t)pr.items.size(), 256, tile_smem, st>>>(d_bases, d_seq_off, d_seq_len, d_occ_off, d_items, k, m,
                                                                        strand_bytes, A, B, R);
    BK_TRY(cudaGetLastError());
    // ---- 2. order (hash, bucket key, rank): stable sorts by bucket key, then by hash ----------------------
    const uint32_t gN = grid_for(N, sm_count);
    iota_kernel<<<gN, 256, 0, st>>>(I0, N);
    BK_TRY(cudaGetLastError());
    size_t tmp_bytes = 0, need = 0;
    BK_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, B, K, I0, I1, (int64_t)N, 0, 64, st));
    tmp_bytes = need;
    BK_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, A, B, (int64_t)N, st));
    if (need > tmp_bytes) tmp_bytes = need;
    uint8_t *d_tmp;
    BK_TRY(ar.alloc(&d_tmp, tmp_bytes));
    need = tmp_bytes;
    BK_TRY(cub::DeviceRadixSort::SortPairs(d_tmp, need, B, K, I0, I1, (int64_t)N, 0, 64, st));
    gather_kernel<uint64_t><<<gN, 256, 0, st>>>(A, I1, H1, N);
    BK_TRY(cudaGetLastError());
    need = tmp_bytes;
    BK_TRY(cub::DeviceRadixSort::SortPairs(d_tmp, need, H1, K, I1, I0, (int64_t)N, 0, 64, st));
    // K = hashes in final order, I0 = final permutation; H1 <- bucket keys, I1 <- ranks in final order
    gather_kernel<uint64_t><<<gN, 256, 0, st>>>(B, I0, H1, N);
    BK_TRY(cudaGetLastError());
    gather_kernel<uint32_t><<<gN, 256, 0, st>>>(R, I0, I1, N);
    BK_TRY(cudaGetLastError());
    // ---- 3. entries and their tip lists ------------------------------------------------------------------
    flags_kernel<<<gN, 256, 0, st>>>(K, H1, I1, A, N);
    BK_TRY(cudaGetLastError());
    need = tmp_bytes;
    BK_TRY(cub::DeviceScan::ExclusiveSum(d_tmp, need, A, B, (int64_t)N, st));
    uint64_t last_flag = 0, last_scan = 0;
    BK_TRY(cudaMemcpyAsync(&last_flag, A + (N - 1), 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(&last_scan, B + (N - 1), 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaStreamSynchronize(st));
    const uint64_t tot = last_flag + last_scan;
    const uint32_t E = (uint32_t)tot, T = (uint32_t)(tot >> 32);
    uint64_t *d_entry_hash, *d_entry_bucket; uint32_t *d_list_off, *d_tips;
    BK_TRY(ar.alloc(&d_entry_hash, E)); BK_TRY(ar.alloc(&d_entry_bucket, E));
    BK_TRY(ar.alloc(&d_list_off, (uint64_t)E + 1)); BK_TRY(ar.alloc(&d_tips, T));
    scatter_entries_kernel<<<gN, 256, 0, st>>>(K, H1, I1, A, B, N, d_entry_hash, d_entry_bucket, d_list_off, d_tips);
    BK_TRY(cudaGetLastError());
    BK_TRY(cudaMemcpyAsync(d_list_off + E, &T, 4, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaStreamSynchronize(st));  // T is a stack variable
    // the occurrence arrays are no longer needed
    ar.free_one(A); ar.free_one(B); ar.free_one(K); ar.free_one(H1); ar.free_one(R); ar.free_one(I0); ar.free_one(I1);
    ar.free_one(d_bases); ar.free_one(d_tmp);
    // ---- 4. equal tip lists share one node set --------------------------------------------------------------
    const uint32_t gE = grid_for(E, sm_count);
    uint64_t *d_fp, *d_fp_sorted; uint32_t *d_eid, *d_eid_sorted, *d_seg, *d_head, *d_rep, *d_is_rep, *d_set_idx;
    BK_TRY(ar.alloc(&d_fp, E)); BK_TRY(ar.alloc(&d_fp_sorted, E)); BK_TRY(ar.alloc(&d_eid, E)); BK_TRY(ar.alloc(&d_eid_sorted, E));
    BK_TRY(ar.alloc(&d_seg, E)); BK_TRY(ar.alloc(&d_head, E)); BK_TRY(ar.alloc(&d_rep, E)); BK_TRY(ar.alloc(&d_is_rep, E));
    BK_TRY(ar.alloc(&d_set_idx, E));
    size_t tmp2 = 0;
    BK_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, d_fp, d_fp_sorted, d_eid, d_eid_sorted, (int64_t)E, 0, 64, st));
    tmp2 = need;
    BK_TRY(cub::DeviceScan::InclusiveScan(nullptr, need, d_seg, d_head, MaxOp(), (int64_t)E, st));
    if (need > tmp2) tmp2 = need;
    BK_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_is_rep, d_set_idx, (int64_t)E, st));
    if (need > tmp2) tmp2 = need;
    uint64_t *d_sizes_probe = nullptr;
    BK_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_sizes_probe, d_sizes_probe, (int64_t)E, st));
    if (need > tmp2) tmp2 = need;
    uint8_t *d_tmp2;
    BK_TRY(ar.alloc(&d_tmp2, tmp2));
    fingerprint_kernel<<<gE, 256, 0, st>>>(d_list_off, d_tips, d_fp, d_eid, E);
    BK_TRY(cudaGetLastError());
    need = tmp2;
    BK_TRY(cub::DeviceRadixSort::SortPairs(d_tmp2, need, d_fp, d_fp_sorted, d_eid, d_eid_sorted, (int64_t)E, 0, 64, st));
    seg_head_kernel<<<gE, 256, 0, st>>>(d_fp_sorted, d_eid_sorted, d_list_off, d_tips, d_seg, E);
    BK_TRY(cudaGetLastError());
    need = tmp2;
    BK_TRY(cub::DeviceScan::InclusiveScan(d_tmp2, need, d_seg, d_head, MaxOp(), (int64_t)E, st));
    rep_kernel<<<gE, 256, 0, st>>>(d_eid_sorted, d_head, d_rep, d_is_rep, E);
    BK_TRY(cudaGetLastError());
    need = tmp2;
    BK_TRY(cub::DeviceScan::ExclusiveSum(d_tmp2, need, d_is_rep, d_set_idx, (int64_t)E, st));
    uint32_t last_rep = 0, last_idx = 0;
    BK_TRY(cudaMemcpyAsync(&last_rep, d_is_rep + (E - 1), 4, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(&last_idx, d_set_idx + (E - 1), 4, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaStreamSynchronize(st));
    const uint32_t S = last_rep + last_idx;
    uint64_t *d_entry_set; uint32_t *d_set_rep;
    BK_TRY(ar.alloc(&d_entry_set, E)); BK_TRY(ar.alloc(&d_set_rep, S));
    entry_set_kernel<<<gE, 256, 0, st>>>(d_rep, d_is_rep, d_set_idx, d_entry_set, d_set_rep, E);
    BK_TRY(cudaGetLastError());
    // ---- 5. node sets ----------------------------------------------------------------------------------------
    int32_t *d_parent; uint32_t *d_depth, *d_rank_node; uint64_t *d_node_id, *d_sizes, *d_set_off;
    BK_TRY(ar.alloc(&d_parent, n_nodes)); BK_TRY(ar.alloc(&d_depth, n_nodes)); BK_TRY(ar.alloc(&d_node_id, n_nodes));
    BK_TRY(ar.alloc(&d_rank_node, n_tips)); BK_TRY(ar.alloc(&d_sizes, S)); BK_TRY(ar.alloc(&d_set_off, (uint64_t)S + 1));
    BK_TRY(cudaMemcpyAsync(d_parent, pr.parent.data(), n_nodes * 4, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_depth, pr.depth.data(), n_nodes * 4, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_node_id, tree->node_id, n_nodes * 8, cudaMemcpyHostToDevice, st));
    BK_TRY(cudaMemcpyAsync(d_rank_node, pr.rank_node.data(), n_tips * 4, cudaMemcpyHostToDevice, st));
    const uint32_t gS = grid_for(S, sm_count);
    set_size_kernel<<<gS, 256, 0, st>>>(d_parent, d_depth, d_rank_node, d_set_rep, d_list_off, d_tips, d_sizes, S);
    BK_TRY(cudaGetLastError());
    need = tmp2;  // sized above for E >= S items of this type
    BK_TRY(cub::DeviceScan::ExclusiveSum(d_tmp2, need, d_sizes, d_set_off, (int64_t)S, st));
    uint64_t last_size = 0, last_off = 0;
    BK_TRY(cudaMemcpyAsync(&last_size, d_sizes + (S - 1), 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(&last_off, d_set_off + (S - 1), 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaStreamSynchronize(st));
    const uint64_t total_nodes = last_size + last_off;
    uint64_t *d_set_nodes;
    BK_TRY(ar.alloc(&d_set_nodes, total_nodes));
    set_fill_kernel<<<gS, 256, 0, st>>>(d_parent, d_depth, d_rank_node, d_node_id, d_set_rep, d_list_off, d_tips, d_set_off, d_set_nodes, S);
    BK_TRY(cudaGetLastError());
    // ---- results ------------------------------------------------------------------------------------------------
    bm->entry_hash.resize(E); bm->entry_bucket.resize(E); bm->entry_set.resize(E);
    bm->set_off.resize((size_t)S + 1); bm->set_node_ids.resize(total_nodes);
    BK_TRY(cudaMemcpyAsync(bm->entry_hash.data(), d_entry_hash, (size_t)E * 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(bm->entry_bucket.data(), d_entry_bucket, (size_t)E * 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(bm->entry_set.data(), d_entry_set, (size_t)E * 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaMemcpyAsync(bm->set_off.data(), d_set_off, (size_t)S * 8, cudaMemcpyDeviceToHost, st));
    if (total_nodes) BK_TRY(cudaMemcpyAsync(bm->set_node_ids.data(), d_set_nodes, total_nodes * 8, cudaMemcpyDeviceToHost, st));
    BK_TRY(cudaStreamSynchronize(st));
    bm->set_off[S] = total_nodes;
    *out = guard.release();
    return CLS_OK;
}

// Nothing is thrown across the ABI: host allocation failures become CLS_ERR_OUT_OF_MEMORY.
extern "C" int cls_model_build_device(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node, const uint8_t *bases,
                                      const uint64_t *offsets, int device, cls_built_model **out) {
    try {
        return build_device(tree, n_tips, tip_node, bases, offsets, device, out);
    } catch (const std::bad_alloc &) {
        if (out) *out = nullptr;
        return cls::set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while building the model");
    } catch (const std::exception &e) {
        if (out) *out = nullptr;
        return cls::set_last_error(CLS_ERR_INVALID_ARGUMENT, std::string("cls_model_build_device: ") + e.what());
    }
}
