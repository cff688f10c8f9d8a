// aco.cu -- host side of tl_aco (the epoch loop around the K7 kernels and K4).
#include "host.hpp"

#include <cmath>
#include <vector>

using namespace tl;

extern "C" tl_status tl_aco(tl_problem *p, const tl_aco_options *o, const uint32_t *init_tour,
                            uint32_t *best_tour_out, float *best_cost_out, tl_stats *stats)
{
    return guarded([&]() -> tl_status {
    if (!p || !o || !best_tour_out) { set_error("tl_aco: null argument"); return TL_ERR_INVALID; }
    // AcoOptions::validate (src/tsp/mod.rs:1114-1153), same messages
    if (!std::isfinite(o->alpha) || o->alpha < 0.0f) { set_error("alpha must be >= 0 (got %g)", o->alpha); return TL_ERR_INVALID; }
    if (!(o->beta >= 0.0f && o->beta <= 6.0f)) { set_error("beta must be in [0, 6] (got %g)", o->beta); return TL_ERR_INVALID; }
    if (!std::isfinite(o->evaporation_rate) || o->evaporation_rate <= 0.0f || o->evaporation_rate >= 1.0f) {
        set_error("evaporation_rate must be in (0, 1) (got %g)", o->evaporation_rate);
        return TL_ERR_INVALID;
    }
    if (o->num_ants == 0) { set_error("num_ants must be >= 1"); return TL_ERR_INVALID; }
    if (p->kind == PK_EUC_NINT) { set_error("tl_aco: needs an F32_EXACT or EXPLICIT problem"); return TL_ERR_UNSUPPORTED; }
    const uint32_t n = p->n;
    if (init_tour && !tour_is_permutation(init_tour, n)) {
        set_error("tl_aco: init_tour is not a permutation of 0..%u", n - 1);
        return TL_ERR_INVALID;
    }
    tl_ctx *c = p->ctx;
    DeviceGuard g(c);
    cudaStream_t st = c->stream;
    const uint64_t launches0 = c->launches;
    if (stats) memset(stats, 0, sizeof *stats);

    std::vector<uint32_t> best(n);
    if (init_tour) {
        memcpy(best.data(), init_tour, sizeof(uint32_t) * n);
    } else {
        for (uint32_t k = 0; k < n; ++k) best[k] = k;
        if (n > 2) { // positions.shuffle(&mut rng) (ant_colony.rs:132-136), Philox-driven Fisher-Yates
            for (uint32_t i = n - 1; i > 0; --i) {
                uint32_t out[4];
                aco_philox_host(i, 0u, 0u, (uint32_t)aco_stream_shuffle(), (uint32_t)o->seed, (uint32_t)(o->seed >> 32), out);
                const uint32_t j = (uint32_t)(((uint64_t)out[0] * (uint64_t)(i + 1)) >> 32);
                std::swap(best[i], best[j]);
            }
        }
    }
    if (n <= 2) { // ant_colony.rs:107-113: identity order
        for (uint32_t k = 0; k < n; ++k) best[k] = k;
    }
    DevBuf<uint32_t> d_best, d_tours;
    DevBuf<float> d_cost1, d_costs, d_ph, d_eta, d_w;
    DevBuf<unsigned long long> d_impr;
    const size_t nn = (size_t)n * n;
    if (d_best.alloc(n) != cudaSuccess || d_cost1.alloc(1) != cudaSuccess || d_impr.alloc(1) != cudaSuccess) {
        set_error("tl_aco: device allocation failed");
        return TL_ERR_NOMEM;
    }
    cudaEvent_t e0, e1;
    TL_CUDA_TRY(cudaEventCreate(&e0));
    TL_CUDA_TRY(cudaEventCreate(&e1));
    auto cleanup = [&] { cudaEventDestroy(e0); cudaEventDestroy(e1); };
    cudaError_t e = cudaMemcpyAsync(d_best.p, best.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_impr.p, 0, 8, st);
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    // cost of the seed tour: the exact-order sum (distances.tour_length_by_pos)
    launch_tour_lengths_f32(p->d_xy, p->d_tri, n, d_best.p, 1, p->metric == Metric::F32_FAST, false, d_cost1.p, c->sm_count, st);
    c->launches++;
    float best_cost = 0.0f;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&best_cost, d_cost1.p, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cleanup(); set_error("tl_aco: %s", cudaGetErrorString(e)); return TL_ERR_CUDA; }

    unsigned long long improvements = 0;
    if (n > 2 && o->epochs > 0) {
        if (d_tours.alloc((size_t)o->num_ants * n) != cudaSuccess || d_costs.alloc(o->num_ants) != cudaSuccess ||
            d_ph.alloc(nn) != cudaSuccess || d_eta.alloc(nn) != cudaSuccess || d_w.alloc(nn) != cudaSuccess) {
            cudaGetLastError();
            cleanup();
            set_error("tl_aco: three %u x %u f32 matrices (%.1f MB) do not fit device memory", n, n, 3.0 * nn * 4 / 1e6);
            return TL_ERR_NOMEM;
        }
        const float tau0 = (init_tour && best_cost > 0.0f) ? (float)o->num_ants / best_cost : 1.0f;
        const float tau_min = tau0 * 1e-4f; // TAU_MIN_RATIO
        const float keep = 1.0f - o->evaporation_rate;
        launch_aco_fill(d_ph.p, nn, tau0, c->sm_count, st);
        launch_aco_eta(p->d_xy, p->d_tri, n, p->metric == Metric::F32_FAST, o->beta, d_eta.p, c->sm_count, st);
        c->launches += 2;
        if (init_tour) { // deposit_tour(best_pos_seed, best_cost), ant_colony.rs:176-178
            launch_aco_update(d_ph.p, n, nullptr, nullptr, 0, d_best.p, d_cost1.p, d_impr.p, st);
            c->launches++;
        }
        for (uint32_t epoch = 0; epoch < o->epochs && e == cudaSuccess; ++epoch) {
            launch_aco_weights(d_ph.p, d_eta.p, nn, o->alpha, d_w.p, c->sm_count, st);
            e = launch_aco_construct(d_w.p, d_eta.p, n, o->num_ants, epoch, o->seed, d_tours.p, st);
            launch_tour_lengths_f32(p->d_xy, p->d_tri, n, d_tours.p, o->num_ants, p->metric == Metric::F32_FAST, false, d_costs.p,
                                    c->sm_count, st);
            launch_aco_evaporate(d_ph.p, nn, keep, tau_min, c->sm_count, st);
            launch_aco_update(d_ph.p, n, d_tours.p, d_costs.p, o->num_ants, d_best.p, d_cost1.p, d_impr.p, st);
            c->launches += 5;
        }
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(best_tour_out, d_best.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&best_cost, d_cost1.p, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&improvements, d_impr.p, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    cleanup();
    if (e != cudaSuccess) { set_error("tl_aco: %s", cudaGetErrorString(e)); return TL_ERR_CUDA; }
    if (best_cost_out) *best_cost_out = best_cost;
    if (stats) {
        stats->passes = (n > 2) ? o->epochs : 0;
        stats->moves = improvements; // epochs that improved the incumbent
        // roulette weights evaluated: sum over steps s = 1..n-1 of (n - s) unvisited cities, per ant and epoch
        stats->evals = (n > 2) ? (uint64_t)o->epochs * o->num_ants * ((uint64_t)n * (n - 1) / 2) : 0;
        stats->launches = c->launches - launches0;
        stats->device_ms = ms;
        stats->converged = 1;
        stats->path_used = p->kind == PK_EXPLICIT ? TL_PATH_MATRIX : TL_PATH_RECOMPUTE;
    }
    return TL_OK;
    });
}
