// avd_episode.cu -- the per-run episode loop of BatchedTrainer.run on the device: the episode controller (what the host loop does
// between two steps, workers/trainer.py:251-273 per run) and the conditional CUDA graph that repeats the step while runs have
// episodes left (avd_loop_graph).
#include <vector>

#include "avd_common.cuh"

namespace {

constexpr int kThreads = 1024;      // one CTA: a warp per run (grid-stride over runs), so the run-level flags reduce in shared memory

__device__ __forceinline__ bool weighted_on(const avd_episode_io& io, int ep) { return io.weighted && ep >= io.weighted_window; }

// is_valid_step_for_federated_training_with_gradients once is_valid_update_step holds (trainer.py:654-664)
__device__ __forceinline__ bool gradients_round(const avd_episode_io& io, int ep) {
    return io.fed_gradients && ep % io.fed_update_count == 0 && ep <= io.fed_cutoff_episode;
}

__global__ void __launch_bounds__(kThreads) episode_control_kernel(const __grid_constant__ avd_episode_io io) {
    __shared__ int s_active, s_full, s_round, s_local;
    avd_episode_state* st = io.state;
    const int S = io.runs, Pr = io.platoons_per_run, Gr = io.groups_per_run, M = io.M;
    const int64_t P = (int64_t)S * Pr, G = (int64_t)S * Gr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool step = io.mode == AVD_EPISODE_STEP;
    const int flags0 = st->flags;
    const bool round_taken = step && io.learn && (flags0 & AVD_EPISODE_ROUND);
    const bool have_w = flags0 & AVD_EPISODE_HAVE_WEIGHTS;
    const bool have_sums = (flags0 & AVD_EPISODE_HAVE_SUMS) || round_taken;
    const int n_sys_run = io.fed == 1 ? M : Gr, X = io.fed == 1 ? Gr : M;   // systems of one run, members of a system
    const int64_t n_systems = (int64_t)n_sys_run * S;
    if (threadIdx.x == 0) s_active = s_full = s_round = s_local = 0;
    __syncthreads();
    for (int k = warp; k < S; k += kThreads / 32) {
        int left = io.left[k], ep = io.ep[k], i = io.i[k], nrec = io.nrec[k];
        bool end = false;
        if (step && left > 0) {
            bool term = false;
            if (io.global_break)
                for (int p = lane; p < Pr; p += 32) term |= (io.done[(int64_t)k * Pr + p] & 1) != 0;
            term = __any_sync(0xffffffffu, term);
            ++i;
            end = term || i >= io.steps_per_episode;
        }
        if (end) {      // the host loop's update_reward_list(episodic_rewards(k), frl_weight_lists(k)) and run_episode_steps
            const int64_t slot = nrec;
            for (int64_t j = lane; j < (int64_t)M * Pr; j += 32) {
                const int64_t m = j / Pr, col = (int64_t)k * Pr + (j - m * Pr);
                io.log_reward[slot * io.log_pitch + m * P + col] = io.ep_reward[m * P + col];
            }
            const bool wrec = io.fed && io.log_w && weighted_on(io, ep) && have_w && have_sums;
            if (wrec) {
                for (int64_t j = lane; j < (int64_t)n_sys_run * X; j += 32) {
                    const int64_t t = j / X, x = j - t * X, sys = io.fed == 1 ? t * S + k : (int64_t)k * Gr + t;
                    io.log_w[(slot * n_systems + sys) * X + x] = io.fed_w[sys * X + x];
                }
                for (int t = lane; t < n_sys_run; t += 32) {
                    const int64_t sys = io.fed == 1 ? (int64_t)t * S + k : (int64_t)k * Gr + t;
                    io.log_wsum[slot * n_systems + sys] = io.wsum[sys];
                }
            }
            if (lane == 0) {
                io.log_len[slot * S + k] = i;
                io.log_weighted[slot * S + k] = wrec;
            }
            ++nrec;
            ++ep;
            i = 0;
            --left;
        }
        if (step && lane == 0) {
            io.left[k] = left;
            io.ep[k] = ep;
            io.i[k] = i;
            io.nrec[k] = nrec;
        }
        const bool restart = end && left > 0;
        for (int p = lane; p < Pr; p += 32) io.reset_mask[(int64_t)k * Pr + p] = restart;
        // the next step's masks (_step_runs): FRL predicates of (ep, i) before that step's increment
        const bool active = left > 0;
        const bool fed_step = active && io.fed && i % io.fed_update_delay_steps == 0;
        const bool grads = fed_step && gradients_round(io, ep);
        const bool local = active && !fed_step;
        for (int j = lane; j < M * Gr; j += 32) {
            const int m = j / Gr;
            const int64_t a = m * G + (int64_t)k * Gr + (j - m * Gr);
            io.learn_mask[a] = local;
            if (io.round_mask) io.round_mask[a] = grads && (!io.fed_apply_mask || io.fed_apply_mask[a]);
        }
        if (lane == 0) {
            if (active) atomicOr(&s_active, 1);
            if (active && nrec >= io.log_slots) atomicOr(&s_full, 1);
            if (grads) atomicOr(&s_round, 1);
            if (local) atomicOr(&s_local, 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (step) {
            st->buffer_counter += 1;
            st->steps += 1;
            if (round_taken) st->rounds += 1;
        }
        const bool cont = s_active && !s_full && st->buffer_counter < st->learn_from;
        st->flags = (have_w ? AVD_EPISODE_HAVE_WEIGHTS : 0) | (have_sums ? AVD_EPISODE_HAVE_SUMS : 0) | (cont ? AVD_EPISODE_CONTINUE : 0) |
                    (s_round ? AVD_EPISODE_ROUND : 0) | (s_local ? AVD_EPISODE_LOCAL : 0);
        s_active = cont;
    }
    __syncthreads();
    // one handle per thread, after everything else: the call keeps little state alive
    const int h = threadIdx.x;
    if (h < io.n_cont_handles) cudaGraphSetConditional(io.cont_handle[h], s_active ? 1u : 0u);
    else if (h == 2 && io.has_round_handle) cudaGraphSetConditional(io.round_handle, s_active && s_round ? 1u : 0u);
    else if (h == 3 && io.has_local_handle) cudaGraphSetConditional(io.local_handle, s_active && s_local ? 1u : 0u);
}

// _frl_weights_runs (trainer.py): FedAvg weights of the runs past their window, 1 for the others; a round in which no run is past its
// window is a plain mean and leaves the recorded weights (fed_w) as they were.
__global__ void __launch_bounds__(kThreads) episode_weights_kernel(const __grid_constant__ avd_episode_io io) {
    const int S = io.runs, Gr = io.groups_per_run, M = io.M;
    bool any = false;
    for (int k = threadIdx.x; k < S; k += kThreads) any |= weighted_on(io, io.ep[k]);
    any = __syncthreads_or(any);
    const int X = io.fed == 1 ? Gr : M;
    const int64_t n = (int64_t)S * Gr * M;
    for (int64_t j = threadIdx.x; j < n; j += kThreads) {
        const int64_t sys = j / X;
        const int k = (int)(io.fed == 1 ? sys % S : sys / Gr);
        float w = io.round_w[j];
        if (!weighted_on(io, io.ep[k])) io.round_w[j] = w = 1.0f;
        if (any) io.fed_w[j] = w;
    }
    if (threadIdx.x == 0 && any) io.state->flags |= AVD_EPISODE_HAVE_WEIGHTS;
}

}  // namespace

extern "C" int avd_episode_control(const avd_episode_io* io, void* stream) {
    AVD_REQUIRE(io && io->state && io->left && io->ep && io->i && io->nrec, "null episode io or counters");
    AVD_REQUIRE(io->runs >= 1 && io->platoons_per_run >= 1 && io->groups_per_run >= 1 && io->M >= 1 && io->M <= AVD_MAX_FOLLOWERS &&
                    io->platoons_per_run % io->groups_per_run == 0,
                "bad batch: %d runs x %d platoons (%d groups) x %d followers", io->runs, io->platoons_per_run, io->groups_per_run, io->M);
    AVD_REQUIRE(io->mode >= AVD_EPISODE_ARM && io->mode <= AVD_EPISODE_WEIGHTS, "mode %d", io->mode);
    AVD_REQUIRE(io->fed >= 0 && io->fed <= 2, "fed %d", io->fed);
    AVD_REQUIRE(!io->fed || (io->fed_update_delay_steps >= 1 && io->fed_update_count >= 1), "FRL schedule needs delay and count >= 1");
    AVD_REQUIRE(io->n_cont_handles >= 0 && io->n_cont_handles <= 2, "n_cont_handles %d", io->n_cont_handles);
    cudaStream_t st = (cudaStream_t)stream;
    if (io->mode == AVD_EPISODE_WEIGHTS) {
        AVD_REQUIRE(io->fed && io->round_w && io->fed_w, "WEIGHTS needs FRL, round_w and fed_w");
        episode_weights_kernel<<<1, kThreads, 0, st>>>(*io);
        AVD_LAUNCH_OK();
        return AVD_OK;
    }
    AVD_REQUIRE(io->steps_per_episode >= 1 && io->log_slots >= 1, "steps_per_episode %d, log_slots %d", io->steps_per_episode, io->log_slots);
    AVD_REQUIRE(io->done && io->ep_reward && io->reset_mask && io->learn_mask && io->log_reward && io->log_len && io->log_weighted,
                "null done / ep_reward / masks / log");
    AVD_REQUIRE(!io->fed || (io->round_mask && io->wsum), "FRL needs round_mask and wsum");
    AVD_REQUIRE(!io->log_w || (io->log_wsum && io->fed_w), "a weights log needs log_wsum and fed_w");
    AVD_REQUIRE(io->log_pitch >= (int64_t)io->M * io->runs * io->platoons_per_run, "log_pitch %lld below M*P", (long long)io->log_pitch);
    episode_control_kernel<<<1, kThreads, 0, st>>>(*io);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

// ---- conditional graph -----------------------------------------------------------------------------------------------------
struct avd_loop_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<cudaStream_t> capturing;      // streams whose capture has begun and not ended
};

namespace {
constexpr cudaStreamCaptureMode kMode = cudaStreamCaptureModeThreadLocal;

void forget(avd_loop_graph* g, cudaStream_t s) {
    for (size_t j = 0; j < g->capturing.size(); ++j)
        if (g->capturing[j] == s) {
            g->capturing.erase(g->capturing.begin() + j);
            return;
        }
}
}  // namespace

extern "C" int avd_loop_graph_create(avd_loop_graph** out, int32_t n_handles, uint64_t* handles_out) {
    AVD_REQUIRE(out && n_handles >= 0 && (n_handles == 0 || handles_out), "bad arguments");
    *out = nullptr;
    avd_loop_graph* g = new avd_loop_graph();
    cudaError_t e = cudaGraphCreate(&g->graph, 0);
    for (int h = 0; e == cudaSuccess && h < n_handles; ++h) {
        cudaGraphConditionalHandle c = 0;
        e = cudaGraphConditionalHandleCreate(&c, g->graph, 0, 0);
        handles_out[h] = (uint64_t)c;
    }
    if (e != cudaSuccess) {
        if (g->graph) cudaGraphDestroy(g->graph);
        delete g;
        avd::set_error("conditional graph set-up failed: %s", cudaGetErrorString(e));
        return AVD_ERR_CUDA;
    }
    *out = g;
    return AVD_OK;
}

extern "C" int avd_loop_graph_capture_begin(avd_loop_graph* g, void* stream) {
    AVD_REQUIRE(g && g->graph && !g->exec, "graph already built");
    cudaStream_t s = (cudaStream_t)stream;
    AVD_CUDA_OK(cudaStreamBeginCaptureToGraph(s, g->graph, nullptr, nullptr, 0, kMode));
    g->capturing.push_back(s);
    return AVD_OK;
}

extern "C" int avd_loop_graph_cond_begin(avd_loop_graph* g, uint64_t handle, int32_t type, void* parent, void* child) {
    AVD_REQUIRE(g && (type == 0 || type == 1) && parent != child, "bad arguments");
    cudaStream_t ps = (cudaStream_t)parent, cs = (cudaStream_t)child;
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    cudaGraph_t where = nullptr;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    AVD_CUDA_OK(cudaStreamGetCaptureInfo(ps, &status, nullptr, &where, &deps, &n_deps));
    AVD_REQUIRE(status == cudaStreamCaptureStatusActive, "parent stream is not capturing");
    cudaGraphNodeParams prm = {};
    prm.type = cudaGraphNodeTypeConditional;
    prm.conditional.handle = (cudaGraphConditionalHandle)handle;
    prm.conditional.type = type == 1 ? cudaGraphCondTypeWhile : cudaGraphCondTypeIf;
    prm.conditional.size = 1;
    cudaGraphNode_t node = nullptr;
    AVD_CUDA_OK(cudaGraphAddNode(&node, where, deps, n_deps, &prm));
    AVD_CUDA_OK(cudaStreamUpdateCaptureDependencies(ps, &node, 1, cudaStreamSetCaptureDependencies));
    AVD_CUDA_OK(cudaStreamBeginCaptureToGraph(cs, prm.conditional.phGraph_out[0], nullptr, nullptr, 0, kMode));
    g->capturing.push_back(cs);
    return AVD_OK;
}

extern "C" int avd_loop_graph_cond_end(avd_loop_graph* g, void* child) {
    AVD_REQUIRE(g, "null graph");
    cudaStream_t cs = (cudaStream_t)child;
    cudaGraph_t body = nullptr;
    forget(g, cs);
    AVD_CUDA_OK(cudaStreamEndCapture(cs, &body));
    return AVD_OK;
}

extern "C" int avd_loop_graph_capture_end(avd_loop_graph* g, void* stream) {
    AVD_REQUIRE(g && g->graph, "null graph");
    cudaStream_t s = (cudaStream_t)stream;
    cudaGraph_t top = nullptr;
    forget(g, s);
    AVD_CUDA_OK(cudaStreamEndCapture(s, &top));
    AVD_REQUIRE(top == g->graph, "capture ended into another graph");
    AVD_CUDA_OK(cudaGraphInstantiate(&g->exec, g->graph, 0));
    return AVD_OK;
}

extern "C" int avd_loop_graph_launch(avd_loop_graph* g, void* stream) {
    AVD_REQUIRE(g && g->exec, "graph not built");
    AVD_CUDA_OK(cudaGraphLaunch(g->exec, (cudaStream_t)stream));
    avd::count_launch();
    return AVD_OK;
}

extern "C" int avd_loop_graph_destroy(avd_loop_graph* g) {
    if (!g) return AVD_OK;
    const bool failed = !g->capturing.empty();
    while (!g->capturing.empty()) {      // innermost first: a build that failed half way
        cudaGraph_t dummy = nullptr;
        cudaStreamEndCapture(g->capturing.back(), &dummy);
        g->capturing.pop_back();
    }
    cudaGetLastError();
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph && !failed) cudaGraphDestroy(g->graph);    // an invalidated capture may already have released it: leak, never double-free
    delete g;
    return AVD_OK;
}
