// host.hpp -- host-side objects behind the opaque C handles (internal).
#pragma once

#include <cuda_runtime.h>

#include <mutex>
#include <new>
#include <vector>

#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "kernels.cuh"

struct tl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    size_t total_mem = 0;
    // library-owned stream-ordered pool: freed blocks stay cached for the next call (release
    // threshold raised) without touching the device's default pool, which other users of
    // cudaMallocAsync in the process share
    cudaMemPool_t pool = nullptr;
    uint64_t launches = 0;
    // One distance-matrix block kept across sessions (the largest seen): a matrix session needs n^2 * 4
    // bytes (400 MB at 10k), and whether the stream-ordered pool can hand back the block the previous
    // session returned depends on what has been carved out of it since -- when it cannot, the pool
    // grows by another n^2 block, 40-80 ms on the call's critical path (seen as end-to-end calls of
    // 75-130 ms instead of 65 once sessions of different kinds had run in the process).  Freed with
    // the context.  Sessions of one context run on one stream, so handing the block over is ordered.
    void *mat_block = nullptr;
    size_t mat_bytes = 0;
    // NCCL (resolved at run time with dlopen, see nccl_shim.cu)
    void *nccl_comm = nullptr;
    int rank = 0, world = 1;
    // peer mailboxes for the in-kernel exchange of a sharded scan (shard_exchange.cuh): this rank's
    // own mailbox (cudaMalloc, exported with cudaIpcGetMemHandle) and every peer's, mapped here
    unsigned long long *mailbox = nullptr;
    unsigned long long *peer_mailbox[tl::kMaxPeers] = {};
    bool p2p_ready = false;   // every rank mapped every mailbox (agreed collectively at attach time)
    uint32_t shard_epoch = 0; // bumped by every tl_session_set_shard(count > 1)
    // pinned host slots (512 B each) for asynchronous state snapshots: cudaMallocHost / cudaFreeHost
    // cost milliseconds and synchronise the device, so sessions borrow a slot instead of owning one
    std::mutex pin_mu;
    std::vector<void *> pin_free;   // slots ready to be borrowed
    std::vector<void *> pin_chunks; // cudaMallocHost allocations, freed with the context
    void *borrow_pinned()
    {
        std::lock_guard<std::mutex> lk(pin_mu);
        if (pin_free.empty()) {
            void *chunk = nullptr;
            if (cudaMallocHost(&chunk, 16 * 512) != cudaSuccess) return nullptr;
            pin_chunks.push_back(chunk);
            for (int k = 0; k < 16; ++k) pin_free.push_back(static_cast<char *>(chunk) + 512 * k);
        }
        void *p = pin_free.back();
        pin_free.pop_back();
        return p;
    }
    void return_pinned(void *p)
    {
        std::lock_guard<std::mutex> lk(pin_mu);
        pin_free.push_back(p);
    }
};

enum ProblemKind { PK_EUC_F32 = 0, PK_EUC_NINT = 1, PK_EXPLICIT = 2 };

struct tl_problem {
    tl_ctx *ctx = nullptr;
    uint32_t n = 0;
    ProblemKind kind = PK_EUC_F32;
    tl::Metric metric = tl::Metric::F32_SAFE; // distance code of every kernel (api.cu); EXPLICIT problems keep F32_SAFE
    // upper bound on any city-to-city distance (bounding-box diagonal, rounded up), set only when the
    // coordinates are in the fast-sqrt domain (api.cu: coords_allow_fast_sqrt), else 0
    float dmax = 0.0f;
    float2 *d_xy = nullptr; // city-ordered coordinates (coordinate problems)
    float *d_tri = nullptr; // packed triangle (EXPLICIT problems)
    uint32_t *d_cand = nullptr; // n x cand_k candidate lists for Mode N (tl_problem_set_candidates)
    uint32_t cand_k = 0;
};

namespace tl {

// Stream that device allocations made by the calling host thread are ordered on: the stream of
// the context whose entry point is executing (set by DeviceGuard).  All device memory comes from
// the context's own stream-ordered pool (cudaMallocFromPoolAsync / cudaFreeAsync; release threshold
// raised in tl_ctx_create so freed blocks are reused instead of returned to the driver): a local-search
// call makes ~10 allocations, and cudaMalloc/cudaFree would cost more than the search itself.
inline thread_local cudaStream_t g_alloc_stream = nullptr;
inline thread_local cudaMemPool_t g_alloc_pool = nullptr;

inline cudaError_t dev_alloc(void **p, size_t bytes)
{
    return g_alloc_pool ? cudaMallocFromPoolAsync(p, bytes, g_alloc_pool, g_alloc_stream)
                        : cudaMallocAsync(p, bytes, g_alloc_stream);
}
inline void dev_free(void *p, cudaStream_t st) { cudaFreeAsync(p, st); }

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    cudaStream_t prev_stream = nullptr;
    cudaMemPool_t prev_pool = nullptr;
    explicit DeviceGuard(int dev) { enter(dev); prev_stream = g_alloc_stream; prev_pool = g_alloc_pool; }
    explicit DeviceGuard(const tl_ctx *c)
    {
        enter(c->device);
        prev_stream = g_alloc_stream;
        prev_pool = g_alloc_pool;
        g_alloc_stream = c->stream;
        g_alloc_pool = c->pool;
    }
    ~DeviceGuard()
    {
        g_alloc_stream = prev_stream;
        g_alloc_pool = prev_pool;
        if (prev >= 0) cudaSetDevice(prev);
    }

  private:
    void enter(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
};

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t count = 0;
    cudaStream_t st = nullptr; // stream the block was allocated on (and is freed on)
    cudaError_t alloc(size_t c)
    {
        release();
        count = c;
        if (c == 0) return cudaSuccess;
        st = g_alloc_stream;
        return dev_alloc(reinterpret_cast<void **>(&p), c * sizeof(T));
    }
    void release()
    {
        if (p) dev_free(p, st);
        p = nullptr;
        count = 0;
    }
    // hand the block to / take it from a cache (the context's matrix block): no allocator call
    T *detach()
    {
        T *q = p;
        p = nullptr;
        count = 0;
        return q;
    }
    void adopt(T *q, size_t c)
    {
        release();
        p = q;
        count = c;
        st = g_alloc_stream;
    }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
};

// Margin of the screened scans (common.cuh: kScreenMarginScale), < 0 disables screening.  Screening
// needs the fast-sqrt domain (dmax is 0 outside it) and a finite distance bound; TL_NO_SCREEN turns it off.
inline float screen_margin(const tl_problem *p)
{
    const float m = p->dmax * kScreenMarginScale;
    return (std::isfinite(m) && p->dmax >= kScreenMinDmax && !getenv("TL_NO_SCREEN")) ? m : -1.0f;
}

bool tour_is_permutation(const uint32_t *tour, uint32_t n);
// K2-pop work decomposition (k2_two_opt_pop.cu): item count of one scan; fills band_first
int two_opt_pop_geometry(uint32_t n, int cyclic, int *chunk_out, std::vector<int32_t> &band_first);

// Nothing is thrown across the C ABI: every extern "C" body that can allocate on the host runs
// inside this guard (std::bad_alloc -> TL_ERR_NOMEM, anything else -> TL_ERR_INVALID).
template <class F>
tl_status guarded(F &&body) noexcept
{
    try {
        return body();
    } catch (const std::bad_alloc &) {
        set_error("out of host memory");
        return TL_ERR_NOMEM;
    } catch (...) {
        set_error("unexpected C++ exception inside libteeline_cuda");
        return TL_ERR_INVALID;
    }
}

// NCCL shim (nccl_shim.cu)
tl_status nccl_get_unique_id(uint8_t *id128);
tl_status nccl_comm_init(void **comm, const uint8_t *id128, int rank, int world);
tl_status nccl_all_gather_bytes(void *comm, const void *send, void *recv, size_t bytes_per_rank,
                                cudaStream_t st);
void nccl_comm_destroy(void *comm);
tl_status nccl_barrier(tl_ctx *ctx); // all ranks' streams have reached this point (host-synchronous)
// maps every rank's mailbox into this process (collective; called by tl_ctx_attach_nccl)
tl_status setup_peer_mailboxes(tl_ctx *ctx);
void release_peer_mailboxes(tl_ctx *ctx);

} // namespace tl
