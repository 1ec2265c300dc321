// ag_host.cu -- host-only helpers of the C ABI and the pipelined host-buffer executor.
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <new>

#include "ag_rollout.cuh"

extern "C" {

int32_t ag_abi_version(void) { return AG_ABI_VERSION; }

const char *ag_status_string(ag_status s) {
    switch (s) {
        case AG_OK: return "ok";
        case AG_ERR_NULL: return "a required pointer is NULL";
        case AG_ERR_SHAPE: return "bad size / shape / stride";
        case AG_ERR_MODE: return "unknown engine or unsupported combination";
        case AG_ERR_ALIGN: return "pointer not aligned as documented";
        case AG_ERR_NOT_SQUARE: return "The matrix is not square.";   // environment/occupancy_grid.py:81
        default: return s > 0 ? cudaGetErrorString((cudaError_t)s) : "unknown status";
    }
}

void ag_default_params(ag_params *p) {
    if (!p) return;
    p->link_1 = 0.4; p->link_2 = 0.3;                 // robot/two_joint_robot.py:12-13
    p->target_x = -0.2; p->target_y = -0.3;           // scenario/scene_0.py:17
    p->target_j1 = 1.1; p->target_j2 = -0.2;          // scenario/scene_0.py:30
    p->reach_eps = 2e-3;                              // scenario/scene_0.py:122
    p->section_eps = 1e-10;                           // utils/collision_checker.py:81
    p->reward_collision = -1e3;                       // scenario/scene_0.py:96
    p->reward_reach = 1e4;                            // scenario/scene_0.py:99
    p->action_scale = 0.1;                            // scenario/scene_0.py:78
    p->choose_j_tar = 0;                              // scenario/scene_0.py:31
    p->max_reset_tries = 64;
}

int32_t ag_grid_words_per_row(int32_t S) { return (S + 31) / 32; }

int64_t ag_grid_stride_words(int32_t S) {
    const int64_t w = (int64_t)S * ((S + 31) / 32);
    return (w + 3) & ~(int64_t)3;
}

int64_t ag_grid_hier_bytes(int32_t S) {
    const int64_t T = (S + 7) / 8, cw = (T + 31) / 32;
    return ((T * T + 1) & ~(int64_t)1) * 8 + 2 * ((T * cw + 3) & ~(int64_t)3) * 4;     // tiles, summary rows, summary columns
}

ag_status ag_grid_pack_host(const uint8_t *occ, int32_t rows, int32_t cols, uint32_t *bits_out) {
    if (!occ || !bits_out) return AG_ERR_NULL;
    if (rows != cols) return AG_ERR_NOT_SQUARE;        // environment/occupancy_grid.py:80-82
    if (rows < 2) return AG_ERR_SHAPE;
    const int32_t S = rows, wpr = (S + 31) / 32;
    std::memset(bits_out, 0, (size_t)ag_grid_stride_words(S) * sizeof(uint32_t));
    for (int32_t r = 0; r < S; ++r)
        for (int32_t c = 0; c < S; ++c)
            if (occ[(int64_t)r * S + c]) bits_out[(int64_t)r * wpr + (c >> 5)] |= 1u << (c & 31);
    return AG_OK;
}

// environment/occupancy_grid.py:28,59-67.  Host float64, one rounding per operation (x86-64 SSE2;
// the translation unit is compiled without FMA contraction on the host side).
ag_status ag_grid_tables_host(int32_t S, double env_size, double *min_x, double *min_y, double *side) {
    if (!min_x || !min_y || !side) return AG_ERR_NULL;
    if (S < 2) return AG_ERR_SHAPE;
    volatile double den = (double)(S - 1);
    volatile double half = env_size / 2.0;
    *side = env_size / den;                            // :28
    for (int32_t i = 0; i < S; ++i) {
        volatile double scaled = (double)i * env_size; // :59  coord * E
        volatile double q = scaled / den;              //      / (S-1)
        volatile double v = q - half;                  // :60  - E/2.0
        min_x[i] = v;
        min_y[i] = v * -1.0;                           // :64  *= [1,-1]
    }
    return AG_OK;
}

// ------------------------------------------------------------------------------ pipeline
struct ag_pipeline {
    static constexpr int NSTAGE = 3;
    int device;
    int64_t n, chunk;
    int K, record;
    int chunk_steps;       // > 0: slice the rollout over STEPS (contiguous copies), else over envs
    cudaStream_t st[NSTAGE];
    cudaEvent_t ev[NSTAGE];
    float *d_act[NSTAGE];
    float *d_j1[NSTAGE], *d_j2[NSTAGE], *d_rw[NSTAGE];
    uint8_t *d_fl[NSTAGE];
    int64_t *d_stats;      // [NSTAGE][AG_ST_COUNT]
    int64_t *h_stats;      // pinned
    int64_t event_cap;     // event sink of one call (all slices append to it)
    uint32_t *d_events;
    int64_t *d_evcount;
    int64_t *h_evcount;    // pinned
};

namespace {

// the caller's current device, restored on scope exit (single-process multi-GPU callers)
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

void pipeline_sync(ag_pipeline *pl) {
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s)
        if (pl->st[s]) cudaStreamSynchronize(pl->st[s]);
}

}  // namespace

#define AG_CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return (ag_status)e_; } while (0)

static ag_status pipeline_alloc(ag_pipeline *pl, int64_t n, int32_t K, int32_t record, int64_t event_capacity) {
    const size_t ck = pl->chunk_steps > 0 ? (size_t)n * pl->chunk_steps : (size_t)pl->chunk * K;
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s) {
        AG_CU(cudaStreamCreateWithFlags(&pl->st[s], cudaStreamNonBlocking));
        AG_CU(cudaEventCreateWithFlags(&pl->ev[s], cudaEventDisableTiming));
        AG_CU(cudaMalloc(&pl->d_act[s], ck * 2 * sizeof(float)));
        if (record) {
            AG_CU(cudaMalloc(&pl->d_j1[s], ck * sizeof(float)));
            AG_CU(cudaMalloc(&pl->d_j2[s], ck * sizeof(float)));
            AG_CU(cudaMalloc(&pl->d_rw[s], ck * sizeof(float)));
            AG_CU(cudaMalloc(&pl->d_fl[s], ck));
        }
    }
    AG_CU(cudaMalloc(&pl->d_stats, sizeof(int64_t) * AG_ST_COUNT * ag_pipeline::NSTAGE));
    AG_CU(cudaMallocHost(&pl->h_stats, sizeof(int64_t) * AG_ST_COUNT * ag_pipeline::NSTAGE));
    if (event_capacity > 0) {
        AG_CU(cudaMalloc(&pl->d_events, (size_t)event_capacity * 3 * sizeof(uint32_t)));
        AG_CU(cudaMalloc(&pl->d_evcount, sizeof(int64_t)));
        AG_CU(cudaMallocHost(&pl->h_evcount, sizeof(int64_t)));
    }
    return AG_OK;
}

ag_status ag_pipeline_create(ag_pipeline **out, int32_t device, int64_t n, int32_t K, int64_t chunk_envs,
                             int32_t chunk_steps, int32_t record, int64_t event_capacity) {
    if (!out) return AG_ERR_NULL;
    *out = nullptr;
    if (n < 1 || K < 1 || (chunk_steps <= 0 && chunk_envs < 1) || event_capacity < 0) return AG_ERR_SHAPE;
    DeviceGuard guard(device);
    if (guard.err != cudaSuccess) return (ag_status)guard.err;
    ag_pipeline *pl = new (std::nothrow) ag_pipeline();
    if (!pl) return (ag_status)cudaErrorMemoryAllocation;
    std::memset(pl, 0, sizeof(*pl));
    pl->device = device; pl->n = n; pl->K = K; pl->record = record;
    pl->chunk_steps = chunk_steps > 0 ? (chunk_steps < K ? chunk_steps : K) : 0;
    pl->chunk = chunk_envs < n ? chunk_envs : n;
    pl->chunk = (pl->chunk + 255) & ~(int64_t)255;     // block-aligned chunks keep env->grid maps uniform
    pl->event_cap = event_capacity;
    const ag_status st = pipeline_alloc(pl, n, K, record, event_capacity);
    if (st != AG_OK) {                                 // free whatever was created before the failure
        ag_pipeline_destroy(pl);
        return st;
    }
    *out = pl;
    return AG_OK;
}

void ag_pipeline_destroy(ag_pipeline *pl) {
    if (!pl) return;
    DeviceGuard guard(pl->device);
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s) {
        if (pl->st[s]) { cudaStreamSynchronize(pl->st[s]); cudaStreamDestroy(pl->st[s]); }
        if (pl->ev[s]) cudaEventDestroy(pl->ev[s]);
        cudaFree(pl->d_act[s]); cudaFree(pl->d_j1[s]); cudaFree(pl->d_j2[s]); cudaFree(pl->d_rw[s]); cudaFree(pl->d_fl[s]);
    }
    cudaFree(pl->d_stats);
    cudaFreeHost(pl->h_stats);
    cudaFree(pl->d_events); cudaFree(pl->d_evcount);
    cudaFreeHost(pl->h_evcount);
    delete pl;
}

// chunk i: [stream i%3]  H2D actions -> K4 -> D2H records.  Copies of chunk i+1 overlap the kernel of chunk i and the
// read-back of chunk i-1.
static ag_status rollout_host_impl(ag_pipeline *pl, const ag_params *p, const ag_grid *g, const ag_rollout_args *a) {
    const bool rec = a->rec_j1 != nullptr;
    const bool want_events = a->events != nullptr;
    const int64_t n = a->n, K = a->K;
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s)
        AG_CU(cudaMemsetAsync(pl->d_stats + s * AG_ST_COUNT, 0, sizeof(int64_t) * AG_ST_COUNT, pl->st[s]));
    if (want_events) {
        AG_CU(cudaMemsetAsync(pl->d_evcount, 0, sizeof(int64_t), pl->st[0]));
        AG_CU(cudaEventRecord(pl->ev[0], pl->st[0]));
        for (int s = 1; s < ag_pipeline::NSTAGE; ++s) AG_CU(cudaStreamWaitEvent(pl->st[s], pl->ev[0], 0));
    }
    auto stage_args = [&](ag_rollout_args &b, int s) {
        b.stats = pl->d_stats + s * AG_ST_COUNT;
        if (rec) {
            b.rec_j1 = pl->d_j1[s]; b.rec_j2 = pl->d_j2[s];
            b.rec_reward = a->rec_reward ? pl->d_rw[s] : nullptr;      // planes the caller does not want are not written
            b.rec_flags = a->rec_flags ? pl->d_fl[s] : nullptr;
            if (b.rec_flags && !b.rec_reward) b.rec_reward = pl->d_rw[s];   // compact records: the reward plane stays on the device
        }
        b.events = want_events ? pl->d_events : nullptr;
        b.event_count = want_events ? pl->d_evcount : nullptr;
        b.event_capacity = pl->event_cap;
    };
    if (pl->chunk_steps > 0) {
        // Slices of consecutive STEPS over all envs: every copy is one contiguous block (rows t0..t0+k of
        // the [K][n] arrays), which PCIe moves ~7 % faster than the pitched 2-D copies of env slices.  The
        // kernels of consecutive slices depend on each other through the env state (kernel i+1 waits for
        // kernel i's event); copies of neighbouring slices overlap them on the other two streams.
        int i = 0;
        for (int64_t t0 = 0; t0 < K; t0 += pl->chunk_steps, ++i) {
            const int s = i % ag_pipeline::NSTAGE;
            const int64_t k = (K - t0 < pl->chunk_steps) ? K - t0 : pl->chunk_steps;
            cudaStream_t cs = pl->st[s];
            ag_rollout_args b = *a;
            b.K = (int32_t)k;
            b.event_step0 = a->event_step0 + (int32_t)t0;
            stage_args(b, s);
            if (a->actions) {
                AG_CU(cudaMemcpyAsync(pl->d_act[s], a->actions + t0 * n * 2, (size_t)k * n * 8, cudaMemcpyHostToDevice, cs));
                b.actions = pl->d_act[s];
            }
            if (i > 0) AG_CU(cudaStreamWaitEvent(cs, pl->ev[(i - 1) % ag_pipeline::NSTAGE], 0));
            ag_status st = ag_rollout_impl(p, g, &b, n, cs);
            if (st) return st;
            AG_CU(cudaEventRecord(pl->ev[s], cs));
            if (rec) {
                AG_CU(cudaMemcpyAsync(a->rec_j1 + t0 * n, pl->d_j1[s], (size_t)k * n * 4, cudaMemcpyDeviceToHost, cs));
                AG_CU(cudaMemcpyAsync(a->rec_j2 + t0 * n, pl->d_j2[s], (size_t)k * n * 4, cudaMemcpyDeviceToHost, cs));
                if (a->rec_reward)
                    AG_CU(cudaMemcpyAsync(a->rec_reward + t0 * n, pl->d_rw[s], (size_t)k * n * 4, cudaMemcpyDeviceToHost, cs));
                if (a->rec_flags)
                    AG_CU(cudaMemcpyAsync(a->rec_flags + t0 * n, pl->d_fl[s], (size_t)k * n, cudaMemcpyDeviceToHost, cs));
            }
        }
    }
    int i = 0;
    for (int64_t c0 = 0; pl->chunk_steps <= 0 && c0 < n; c0 += pl->chunk, ++i) {
        const int s = i % ag_pipeline::NSTAGE;
        const int64_t cn = (n - c0 < pl->chunk) ? n - c0 : pl->chunk;
        cudaStream_t cs = pl->st[s];
        ag_rollout_args b = *a;
        b.n = cn; b.env_id0 = a->env_id0 + c0;
        b.j1 = a->j1 + c0; b.j2 = a->j2 + c0; b.reward = a->reward + c0; b.flags = a->flags + c0;
        b.step_ctr = a->step_ctr + c0; b.reset_ctr = a->reset_ctr + c0; b.ep_len = a->ep_len + c0;
        b.reset_u = a->reset_u ? a->reset_u + c0 * a->R * 2 : nullptr;
        b.targets = a->targets ? a->targets + c0 * 2 : nullptr;
        if (want_events) return AG_ERR_MODE;           // the event sink numbers envs per launch: step slices only
        stage_args(b, s);
        if (a->actions) {
            AG_CU(cudaMemcpy2DAsync(pl->d_act[s], (size_t)pl->chunk * 8, a->actions + c0 * 2, (size_t)n * 8,
                                    (size_t)cn * 8, (size_t)K, cudaMemcpyHostToDevice, cs));
            b.actions = pl->d_act[s];
        }
        ag_status st = ag_rollout_impl(p, g, &b, pl->chunk, cs);
        if (st) return st;
        if (rec) {
            AG_CU(cudaMemcpy2DAsync(a->rec_j1 + c0, (size_t)n * 4, pl->d_j1[s], (size_t)pl->chunk * 4, (size_t)cn * 4,
                                    (size_t)K, cudaMemcpyDeviceToHost, cs));
            AG_CU(cudaMemcpy2DAsync(a->rec_j2 + c0, (size_t)n * 4, pl->d_j2[s], (size_t)pl->chunk * 4, (size_t)cn * 4,
                                    (size_t)K, cudaMemcpyDeviceToHost, cs));
            if (a->rec_reward)   // optional on the host side: reward is a function of flags (DESIGN.md "compact records")
                AG_CU(cudaMemcpy2DAsync(a->rec_reward + c0, (size_t)n * 4, pl->d_rw[s], (size_t)pl->chunk * 4,
                                        (size_t)cn * 4, (size_t)K, cudaMemcpyDeviceToHost, cs));
            if (a->rec_flags)
                AG_CU(cudaMemcpy2DAsync(a->rec_flags + c0, (size_t)n, pl->d_fl[s], (size_t)pl->chunk, (size_t)cn,
                                        (size_t)K, cudaMemcpyDeviceToHost, cs));
        }
    }
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s)
        AG_CU(cudaMemcpyAsync(pl->h_stats + s * AG_ST_COUNT, pl->d_stats + s * AG_ST_COUNT,
                              sizeof(int64_t) * AG_ST_COUNT, cudaMemcpyDeviceToHost, pl->st[s]));
    for (int s = 0; s < ag_pipeline::NSTAGE; ++s) AG_CU(cudaStreamSynchronize(pl->st[s]));
    if (want_events) {                                 // every kernel is done: the count, then exactly that many events
        AG_CU(cudaMemcpyAsync(pl->h_evcount, pl->d_evcount, sizeof(int64_t), cudaMemcpyDeviceToHost, pl->st[0]));
        AG_CU(cudaStreamSynchronize(pl->st[0]));
        const int64_t cnt = *pl->h_evcount, stored = cnt < pl->event_cap ? cnt : pl->event_cap;
        if (stored > 0)
            AG_CU(cudaMemcpyAsync(a->events, pl->d_events, (size_t)stored * 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, pl->st[0]));
        AG_CU(cudaStreamSynchronize(pl->st[0]));
        *a->event_count = cnt;
    }
    return AG_OK;
}

ag_status ag_rollout_host(ag_pipeline *pl, const ag_params *p, const ag_grid *g, const ag_rollout_args *a,
                          int64_t *stats_host) {
    if (!pl || !p || !g || !a) return AG_ERR_NULL;
    if (a->n != pl->n || a->K != pl->K) return AG_ERR_SHAPE;
    const int njoint = (a->rec_j1 != nullptr) + (a->rec_j2 != nullptr);
    if (njoint == 1 || (njoint == 0 && (a->rec_reward || a->rec_flags))) return AG_ERR_NULL;   // joints: both or none
    if (a->rec_reward && !a->rec_flags) return AG_ERR_NULL;
    if (njoint == 2 && !pl->record) return AG_ERR_MODE;
    if (a->events && (!a->event_count || pl->event_cap <= 0)) return AG_ERR_MODE;
    DeviceGuard guard(pl->device);
    if (guard.err != cudaSuccess) return (ag_status)guard.err;
    const ag_status st = rollout_host_impl(pl, p, g, a);
    if (st != AG_OK) {                                 // nothing may still be writing the caller's buffers
        pipeline_sync(pl);
        return st;
    }
    if (stats_host)
        for (int k = 0; k < AG_ST_COUNT; ++k)
            for (int s = 0; s < ag_pipeline::NSTAGE; ++s) stats_host[k] += pl->h_stats[s * AG_ST_COUNT + k];
    return AG_OK;
}

}  // extern "C"
