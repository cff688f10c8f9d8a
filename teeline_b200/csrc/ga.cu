// ga.cu -- host side of tl_ga (the epoch loop around the K8 kernels and K4).
#include "host.hpp"

#include <algorithm>
#include <cmath>

using namespace tl;

extern "C" tl_status tl_ga(tl_problem *p, const tl_ga_options *o, const uint32_t *init_tour, uint32_t *best_tour_out,
                           float *best_cost_out, tl_stats *stats)
{
    return guarded([&]() -> tl_status {
    if (!p || !o || !best_tour_out) { set_error("tl_ga: null argument"); return TL_ERR_INVALID; }
    // GAOptions::validate (src/tsp/mod.rs:832-845), same message
    if (!std::isfinite(o->mutation_probability) || o->mutation_probability < 0.0f || o->mutation_probability > 1.0f) {
        set_error("mutation_probability must be in [0, 1] (got %g)", o->mutation_probability);
        return TL_ERR_INVALID;
    }
    if (p->kind == PK_EUC_NINT) { set_error("tl_ga: needs an F32_EXACT or EXPLICIT problem"); return TL_ERR_UNSUPPORTED; }
    const uint32_t n = p->n, P = p->n; // population_size = cities.len() (genetic_algorithm.rs:26)
    if (init_tour && !tour_is_permutation(init_tour, n)) {
        set_error("tl_ga: init_tour is not a permutation of 0..%u", n - 1);
        return TL_ERR_INVALID;
    }
    tl_ctx *c = p->ctx;
    DeviceGuard g(c);
    cudaStream_t st = c->stream;
    const uint64_t launches0 = c->launches;
    if (stats) memset(stats, 0, sizeof *stats);
    constexpr size_t kSmemLimit = 226 * 1024; // 227 KB per CTA on sm_100a, less the kernel's static part
    if (ga_breed_smem_bytes(n, n) > kSmemLimit) {
        set_error("tl_ga: n = %u needs %zu bytes of shared memory per CTA (limit %zu)", n, ga_breed_smem_bytes(n, n),
                  kSmemLimit);
        return TL_ERR_UNSUPPORTED;
    }
    if ((size_t)P * n > ((size_t)1 << 31)) { set_error("tl_ga: population of %u x %u does not fit", P, n); return TL_ERR_NOMEM; }

    DevBuf<uint32_t> d_pop[2], d_init, d_best;
    DevBuf<float> d_fit[2], d_sfit, d_cost;
    DevBuf<int> d_order;
    DevBuf<unsigned long long> d_mut;
    if (d_pop[0].alloc((size_t)P * n) != cudaSuccess || d_pop[1].alloc((size_t)P * n) != cudaSuccess ||
        d_fit[0].alloc(P) != cudaSuccess || d_fit[1].alloc(P) != cudaSuccess || d_sfit.alloc(P) != cudaSuccess ||
        d_order.alloc(P) != cudaSuccess || d_best.alloc(n) != cudaSuccess || d_cost.alloc(1) != cudaSuccess ||
        d_mut.alloc(1) != cudaSuccess || (init_tour && d_init.alloc(n) != cudaSuccess)) {
        cudaGetLastError();
        set_error("tl_ga: device allocation failed (two populations of %u x %u)", P, n);
        return TL_ERR_NOMEM;
    }
    cudaEvent_t e0, e1;
    TL_CUDA_TRY(cudaEventCreate(&e0));
    TL_CUDA_TRY(cudaEventCreate(&e1));
    auto cleanup = [&] { cudaEventDestroy(e0); cudaEventDestroy(e1); };
    cudaError_t e = cudaMemsetAsync(d_mut.p, 0, 8, st);
    if (e == cudaSuccess && init_tour)
        e = cudaMemcpyAsync(d_init.p, init_tour, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    const uint32_t n_seeded = init_tour ? std::max(P / 5, 1u) : 0u; // from_cities_seeded (:207)
    if (e == cudaSuccess)
        e = launch_ga_init(p->d_xy, p->d_tri, n, p->metric == Metric::F32_FAST, d_init.p, n_seeded, o->seed, d_pop[0].p, d_fit[0].p, st);
    c->launches++;
    // The Vec of individuals has L entries: n at first, and after every epoch elites + 2 * (n/2 - n_elite):
    // the reference's population SHRINKS by n_elite (+1 for odd n) in the first epoch and keeps that size
    // (:61-86, the loop bounds use the ORIGINAL size).
    uint32_t L = P;
    const uint32_t pairs = P / 2 > o->n_elite ? P / 2 - o->n_elite : 0u;
    int cur = 0;
    uint32_t epochs_run = 0;
    for (uint32_t epoch = 0; epoch < o->epochs && e == cudaSuccess && n >= 2; ++epoch) {
        const uint32_t ne = std::min(o->n_elite, L);
        e = launch_ga_rank(d_fit[cur].p, L, d_order.p, d_sfit.p, st);
        if (e == cudaSuccess)
            e = launch_ga_breed(p->d_xy, p->d_tri, n, p->metric == Metric::F32_FAST, L, ne, pairs, epoch, o->seed, o->mutation_probability,
                                d_pop[cur].p, d_order.p, d_sfit.p, d_pop[cur ^ 1].p, d_fit[cur ^ 1].p, d_mut.p, st);
        c->launches += 2;
        cur ^= 1;
        L = ne + 2 * pairs;
        ++epochs_run;
        if (L == 0) break; // n_elite = 0 and nothing bred: the reference would panic in best()
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    float best_cost = 0.0f;
    unsigned long long mutations = 0;
    if (e == cudaSuccess && L > 0) {
        launch_ga_best(d_pop[cur].p, d_fit[cur].p, n, L, d_best.p, st);
        launch_tour_lengths_f32(p->d_xy, p->d_tri, n, d_best.p, 1, p->metric == Metric::F32_FAST, false, d_cost.p, c->sm_count, st);
        c->launches += 2;
        e = cudaEventRecord(e1, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(best_tour_out, d_best.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&best_cost, d_cost.p, 4, cudaMemcpyDeviceToHost, st);
    } else if (e == cudaSuccess) {
        e = cudaEventRecord(e1, st);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&mutations, d_mut.p, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    cleanup();
    if (e != cudaSuccess) { set_error("tl_ga: %s", cudaGetErrorString(e)); return TL_ERR_CUDA; }
    if (L == 0) { set_error("tl_ga: the population died out (n_elite = 0 and n < 2)"); return TL_ERR_INVALID; }
    if (best_cost_out) *best_cost_out = best_cost;
    if (stats) {
        stats->passes = epochs_run;
        stats->moves = mutations;
        stats->evals = (uint64_t)epochs_run * 2 * pairs; // children evaluated (one tour length each)
        stats->launches = c->launches - launches0;
        stats->device_ms = ms;
        stats->converged = 1;
        stats->path_used = p->kind == PK_EXPLICIT ? TL_PATH_MATRIX : TL_PATH_RECOMPUTE;
    }
    return TL_OK;
    });
}
