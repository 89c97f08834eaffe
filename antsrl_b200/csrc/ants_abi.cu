// ants_abi.cu -- host side of libantsrl_b200.so: the C ABI declared in include/antsrl_b200.h.
// Owns all device state of one batch of environments, orders the kernel launches of observation / step / update
// exactly as the reference orders its object updates (SURVEY.md section 3), and moves state between dense host
// arrays and the pitched HBM layout.
#include "../../include/antsrl_b200.h"
#include "ants_kernels.cuh"
#include "ants_reset.cuh"
#include "ants_pack.cuh"
#include "ants_host_unpack.h"

#include <math.h>
#include <cmath>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using ants::Params;

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (call);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return fail(ANTS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

enum Fam { F_MOVE = 0, F_FOOD, F_PERCEIVE, F_COLLIDE, F_ROCKS, F_EVAP, F_DEPOSIT, F_ABSORB, F_MISC, F_ENV_MOVE, F_ENV_UPDATE,
           F_ENV_FUSED, F_PACK, F_RESET, F_COUNT };
const char *kFamName[F_COUNT] = {"move", "food_commit", "perceive", "collide", "rocks", "evaporate",
                                 "deposit", "absorb", "misc", "env_move", "env_update", "env_update_move", "pack",
                                 "reset"};

struct TimedLaunch {
    cudaEvent_t a, b;
    int fam;
};

// Worker threads of the host-buffer path (process-wide, created on first use): they expand packed observation chunks
// into the caller's dense array while the next chunk is still crossing PCIe.
class HostPool {
public:
    static HostPool &get() {
        static HostPool pool;
        return pool;
    }
    int size() const { return (int)threads_.size(); }
    void submit(std::function<void()> fn) {
        {
            std::lock_guard<std::mutex> lk(m_);
            q_.push_back(std::move(fn));
            ++pending_;
        }
        cv_.notify_one();
    }
    // blocks until every submitted task has run; returns when the last one finished (seconds on the steady clock)
    double wait_idle() {
        std::unique_lock<std::mutex> lk(m_);
        idle_.wait(lk, [&] { return pending_ == 0; });
        return last_idle_;
    }
    static double now() {
        return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    }

private:
    HostPool() {
        int n = 0;
        if (const char *x = getenv("ANTS_HOST_THREADS")) n = atoi(x);
        if (n <= 0) {
            n = (int)std::thread::hardware_concurrency();
            int ranks = 1;                                   // one process per GPU on a node shares the host cores
            if (const char *x = getenv("LOCAL_WORLD_SIZE")) ranks = atoi(x) > 0 ? atoi(x) : 1;
            n = n / ranks;
        }
        n = n < 1 ? 1 : (n > 64 ? 64 : n);
        for (int t = 0; t < n; ++t) threads_.emplace_back([this] { run(); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : threads_) t.join();
    }
    void run() {
        for (;;) {
            std::function<void()> fn;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (q_.empty()) return;
                fn = std::move(q_.front());
                q_.erase(q_.begin());
            }
            fn();
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0) { last_idle_ = now(); idle_.notify_all(); }
            }
        }
    }
    std::mutex m_;
    std::condition_variable cv_, idle_;
    std::vector<std::function<void()>> q_;
    std::vector<std::thread> threads_;
    int pending_ = 0;
    double last_idle_ = 0.0;
    bool stop_ = false;
};

// the packed form of a configuration's observation (ants_pack.cuh): which samples, which channel goes where
void packed_layout_of(const AntsConfig *cfg, AntsPackedLayout *L) {
    memset(L, 0, sizeof *L);
    const int S = 2 * cfg->radius + 1, S2 = S * S, C = cfg->n_channels;
    L->n_samples = S2; L->n_channels = C; L->sample_bytes = ants::kPackSampleBytes;
    for (int k = 0; k < 8; ++k) L->flag_channel[k] = -1;
    L->value_channel[0] = L->value_channel[1] = -1; L->food_channel = -1;
    int nf = 0, nv = 0, nfood = 0;
    bool ok = C >= 1 && C <= 8 && S2 <= 225;
    for (int c = 0; ok && c < C; ++c) {
        const int k = cfg->channel_kind[c];
        if (k == ANTS_CH_PHERO) { if (nv < 2) L->value_channel[nv] = c; ++nv; }
        else if (k == ANTS_CH_FOOD) { if (nfood < 1) L->food_channel = c; ++nfood; }
        else { if (nf < 8) L->flag_channel[nf] = c; ++nf; }
    }
    ok = ok && nv <= 2 && nfood <= 1 && nf <= 8;
    int V = 0;
    for (int k = 0; k < S2 && k < 228; ++k)
        if (!cfg->has_mask || cfg->mask[k]) L->visible_index[V++] = (uint8_t)k;
    L->n_visible = V;
    L->bytes_per_ant = (int64_t)V * ants::kPackSampleBytes;
    L->supported = (ok && V > 0) ? 1 : 0;
}
void unpack_plan_of(const AntsPackedLayout *L, AntsUnpackPlan *u) {
    memset(u, 0, sizeof *u);
    u->V = L->n_visible; u->S2 = L->n_samples; u->C = L->n_channels;
    for (int v = 0; v < L->n_visible; ++v) u->vis[v] = L->visible_index[v];
    for (int k = 0; k < 8; ++k) u->flag_ch[k] = L->flag_channel[k];
    u->val_ch[0] = L->value_channel[0]; u->val_ch[1] = L->value_channel[1]; u->food_ch = L->food_channel;
    ants_unpack_plan_finish(u);
}

}  // namespace

struct AntsBatch {
    AntsConfig cfg;
    Params p;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    std::vector<void *> allocs;
    int64_t device_bytes = 0;
    // generation counters (16 bit on the device)
    uint32_t obs_gen = 0, occ_gen = 0, owner_phase = 0;
    int64_t timestep = 1;
    int rw_alias = 1, act_bool = 1, prev_synced = 1, needs_sweep = 1;
    int wall_flags_valid = 0;       // wall_hit[] was written by the step that precedes this update
    int absorb_par = 0;             // which absorb counter the steps append under
    int steps_queued = 0;           // flat kernels: steps since the last update (each may queue up to E * N absorbs; the
                                    // list holds E * N, so a second one makes the update sweep every disc instead)
    int commit_par = 0;             // which commit counter this step appends under
    int use_pdl = 0;                // programmatic dependent launch of the step kernels (large batches)
    CUtensorMap plane_map;          // diffusion mode: {H, W, 2 * E * P} f64 over both pheromone planes, box 68 x 66 x 1
    int plane_src = 0;              // which half of the plane allocation is current
    uint32_t lazy_now = 0;          // updates since the last fold of plain values (lazy evaporation), small counter
    uint32_t lazy_abs = 0;          // updates since creation / the last unboxing fold (22 bits)
    AntsStats stats;
    // profiling
    int profiling = 0;
    std::vector<TimedLaunch> timed;
    std::vector<cudaEvent_t> event_pool;
    double fam_ms[F_COUNT];
    int64_t fam_launches[F_COUNT];
    // device staging for the host-buffer entry points
    int8_t *st_rot = nullptr, *st_ph = nullptr;
    float *st_obs = nullptr, *st_as = nullptr, *st_state = nullptr;
    double *st_reward = nullptr, *st_noise = nullptr;
    uint32_t *h_counts = nullptr;   // pinned: commit_count, absorb_count readback
    uint32_t *tile_list = nullptr;
    int perceive_smem = 0, perceive_layout = 0, perceive_group = 4, perceive_threads = 128, perceive_slow_wrap = 0;
    int perceive_rows = 0, rows_smem = 0;   // 1 = k_perceive_rows serves this configuration (default channel list, 7x7 window)
    // block-per-environment kernels (ants_env_fused.cuh): move / update / update+move in one launch each
    int fused = 0, env_group = 1, env_cap = 256, env_smem = 0;   // env_cap: ants per block (256, 512 or 1024)
    int move_done = 0;              // ants_rollout: the move of the coming step already ran inside the last update launch
    // packed observation transport of the host-buffer path (ants_pack.cuh)
    AntsPackedLayout pack_layout;
    AntsUnpackPlan *unpack_plan = nullptr;
    ants::PackArgs pack_args;
    uint8_t *st_packed = nullptr;   // device [EN][bytes_per_ant]
    uint8_t *h_packed = nullptr;    // pinned staging of the same size
    uint32_t *d_pack_fail = nullptr;
    std::vector<cudaEvent_t> chunk_ev;
    int pack_disabled = 0;          // a value without a packed form was seen (non-integer food): dense copies until the next import
    // ants_step_host fills the dense host array from two sides: the DMA engine copies the last `dense_frac` of the ants
    // dense while the host threads expand the packed rest; the split follows whichever side finished later
    double dense_frac = 0.2;
    int dense_frac_fixed = 0;
    // ants_rollout: the batch as groups of environments on streams of their own -- the perception kernel of one group
    // (issue bound, all registers of an SM) overlaps the block-per-environment kernel of another (latency bound)
    struct Group { cudaStream_t s = nullptr; cudaEvent_t done = nullptr; int env0 = 0, env1 = 0; };
    std::vector<Group> groups;
    cudaEvent_t ev_fork = nullptr;
    int grouped = 0;                // inside a grouped rollout: the step kernels launch once per group, whole-batch
                                    // passes join the groups first
    // ants_generate_env_maps: device copy of the window's discs (grows to the largest window seen, freed by ants_destroy)
    int4 *reset_discs = nullptr;
    int64_t reset_cap = 0;
    // ants_generate_env_maps_ex: device copy of the Perlin layers' offsets (the same lifetime)
    int2 *reset_offsets = nullptr;
    int64_t reset_offsets_cap = 0;
};

namespace {

template <typename T>
int dev_alloc(AntsBatch *b, T **ptr, int64_t count, bool zero = true) {
    *ptr = nullptr;
    if (count <= 0) count = 1;
    size_t bytes = (size_t)count * sizeof(T);
    void *d = nullptr;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess)
        return fail(ANTS_E_ALLOC, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    if (zero) {
        e = cudaMemsetAsync(d, 0, bytes, b->stream);
        if (e != cudaSuccess) return fail(ANTS_E_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    }
    b->allocs.push_back(d);
    b->device_bytes += (int64_t)bytes;
    *ptr = (T *)d;
    return ANTS_OK;
}

#define TRY(expr)                   \
    do {                            \
        int _r = (expr);            \
        if (_r != ANTS_OK) return _r; \
    } while (0)

cudaEvent_t get_event(AntsBatch *b) {
    if (!b->event_pool.empty()) {
        cudaEvent_t e = b->event_pool.back();
        b->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct LaunchScope {   // counts the launch and, when profiling, brackets it with events on the handle's stream
    AntsBatch *b;
    int fam;
    cudaEvent_t a = nullptr, e = nullptr;
    LaunchScope(AntsBatch *b_, int fam_) : b(b_), fam(fam_) {
        b->stats.kernel_launches++;
        b->fam_launches[fam]++;
        if (b->profiling) {
            a = get_event(b);
            e = get_event(b);
            cudaEventRecord(a, b->stream);
        }
    }
    ~LaunchScope() {
        if (b->profiling) {
            cudaEventRecord(e, b->stream);
            b->timed.push_back({a, e, fam});
        }
    }
};

int collect_timings(AntsBatch *b) {
    if (b->timed.empty()) return ANTS_OK;
    CK(cudaStreamSynchronize(b->stream));
    for (auto &t : b->timed) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t.a, t.b);
        b->fam_ms[t.fam] += ms;
        b->event_pool.push_back(t.a);
        b->event_pool.push_back(t.b);
    }
    b->timed.clear();
    return ANTS_OK;
}

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

struct Scratch {                   // device scratch of import / export, freed on every return path
    void *ptr = nullptr;
    ~Scratch() { if (ptr) cudaFree(ptr); }
};

// Launch of a step-loop kernel with programmatic stream serialisation: the kernel may be scheduled while the last
// blocks of its predecessor still run; every such kernel starts with pdl_begin() (griddepcontrol.wait) before it
// touches memory.  Off while profiling (events between the launches), with ANTS_NO_PDL set, and for small batches
// (measured: +1.5 % at 524 288 ants per launch, but the attribute's host cost loses 18 % at 51 200).
template <typename... KArgs, typename... Args>
void launch_step(AntsBatch *b, cudaStream_t stream, void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem,
                 Args... args) {
    static const bool env_off = getenv("ANTS_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (b->profiling || env_off || !b->use_pdl) ? 0 : 1;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ANTS_E_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    return ANTS_OK;
}

// grouped rollout: the groups' streams branch off the handle's stream and join it again; a whole-batch pass in between
// (generation fold, lazy-field fold, anthill sweep) joins them first
void fork_groups(AntsBatch *b) {
    cudaEventRecord(b->ev_fork, b->stream);
    for (auto &g : b->groups) cudaStreamWaitEvent(g.s, b->ev_fork, 0);
}
void join_groups(AntsBatch *b) {
    for (auto &g : b->groups) {
        cudaEventRecord(g.done, g.s);
        cudaStreamWaitEvent(b->stream, g.done, 0);
    }
}
struct WholeBatchPass {
    AntsBatch *b;
    explicit WholeBatchPass(AntsBatch *b_) : b(b_) { if (b->grouped) join_groups(b); }
    ~WholeBatchPass() { if (b->grouped) fork_groups(b); }
};

// 16-bit (f64 records) or 7/8-bit (compact records) generation counters: before either wraps, ONE pass folds
// every live exploration stamp into "explored long ago" and clears the occupancy stamps.  Called at the start of
// observe / step, before any stamp of the new generation is written.
void maybe_fold_generations(AntsBatch *b) {
    const uint32_t obs_lim = b->p.explored_old - 2u, occ_lim = (b->p.rec16 || b->p.rec8) ? 0x7Eu : 0xFFFEu;
    if (b->obs_gen + 1u >= obs_lim || b->occ_gen + 1u >= occ_lim) {
        WholeBatchPass wb(b);
        LaunchScope ls(b, F_MISC);
        ants::k_meta_renormalize<<<148 * 16, 256, 0, b->stream>>>(b->p, 1, 1);
        b->obs_gen = 0;
        b->occ_gen = 0;
    }
}
uint32_t next_obs_gen(AntsBatch *b) {
    if (b->obs_gen >= b->p.explored_old - 2u) {   // fold live stamps into "explored long ago" before the counter wraps
        WholeBatchPass wb(b);
        LaunchScope ls(b, F_MISC);
        ants::k_meta_renormalize<<<148 * 8, 256, 0, b->stream>>>(b->p, 1, 0);
        b->obs_gen = 0;
    }
    return ++b->obs_gen;
}
uint32_t next_occ_gen(AntsBatch *b) {
    if (b->occ_gen >= ((b->p.rec16 || b->p.rec8) ? 0x7Eu : 0xFFFEu)) {
        WholeBatchPass wb(b);
        LaunchScope ls(b, F_MISC);
        ants::k_meta_renormalize<<<148 * 8, 256, 0, b->stream>>>(b->p, 0, 1);
        b->occ_gen = 0;
    }
    return ++b->occ_gen;
}
uint32_t next_owner_phase(AntsBatch *b) {
    if (b->owner_phase >= 0xFFFEu) {
        cudaMemsetAsync(b->p.owner, 0, (size_t)b->p.E * b->p.plane * sizeof(uint32_t), b->stream);
        b->owner_phase = 0;
    }
    return ++b->owner_phase;
}

// The perception kernel.  In a grouped rollout the row kernel launches once per group of environments on the group's
// stream; otherwise (and always for the generic kernel, which has no env range) once over the whole batch.
int launch_perceive(AntsBatch *b, float *d_obs, float *d_as, float *d_state, double *d_reward, int is_step) {
    const Params &p = b->p;
    const uint32_t og = next_obs_gen(b);
    // (the straight-line layouts of k_perceive decode pheromones from the record words; in diffusion mode the field
    //  lives in the f64 planes, which only its generic channel code reads)
    const int layout = (p.diffuse && !b->perceive_rows) ? 0 : b->perceive_layout;
    if (b->perceive_rows) {
        const AntsBatch::Group whole = {b->stream, nullptr, 0, p.E};
        const AntsBatch::Group *gs = b->grouped ? b->groups.data() : &whole;
        const int n = b->grouped ? (int)b->groups.size() : 1;
        for (int k = 0; k < n; ++k) {
            const int64_t ant0 = (int64_t)gs[k].env0 * p.N, ant1 = (int64_t)gs[k].env1 * p.N;
            const int rblocks = (int)cdiv(ant1 - ant0, ants::kRowsThreads);
            {
                LaunchScope ls(b, F_PERCEIVE);
#define ANTS_ROWS(L, R16, SS)                                                                                     \
    launch_step(b, gs[k].s, ants::k_perceive_rows<L, R16, SS>, (unsigned)rblocks, (unsigned)ants::kRowsThreads,   \
                (size_t)b->rows_smem, p, d_obs, d_as, d_state, d_reward, og, b->occ_gen, is_step,                \
                b->rw_alias, b->lazy_now, b->lazy_abs, ant0, ant1)
#define ANTS_ROWS_S(SS)                                                                          \
    do {                                                                                         \
        if (p.rec8) { if (layout == 2) ANTS_ROWS(2, 2, SS); else ANTS_ROWS(1, 2, SS); }         \
        else if (p.rec16) { if (layout == 2) ANTS_ROWS(2, 1, SS); else ANTS_ROWS(1, 1, SS); }   \
        else { if (layout == 2) ANTS_ROWS(2, 0, SS); else ANTS_ROWS(1, 0, SS); }                \
    } while (0)
                if (p.S == 7) ANTS_ROWS_S(7); else ANTS_ROWS_S(5);
#undef ANTS_ROWS_S
#undef ANTS_ROWS
            }
            TRY(check_launch("k_perceive"));
        }
    } else {
        const uint32_t magic = (1u << 20) / (uint32_t)p.S2 + 1u;   // f / S2 == (f * magic) >> 20 for f < 2048
        const int threads = b->perceive_threads;
        const int blocks = (int)cdiv(p.EN, threads);
        {
            LaunchScope ls(b, F_PERCEIVE);
#define ANTS_PERCEIVE(L, R16)                                                                                          \
    launch_step(b, b->stream, ants::k_perceive<L, R16>, (unsigned)blocks, (unsigned)threads, (size_t)b->perceive_smem, \
                p, d_obs, d_as, d_state, d_reward, og, b->occ_gen, is_step, b->rw_alias, b->perceive_group,             \
                magic, b->perceive_slow_wrap, b->lazy_now, b->lazy_abs)
            if (p.rec8) {                  // served through the generic channel code (accessor-based decode)
                ANTS_PERCEIVE(0, false);
            } else if (p.rec16) {
                if (layout == 1) ANTS_PERCEIVE(1, true);
                else if (layout == 2) ANTS_PERCEIVE(2, true);
                else ANTS_PERCEIVE(0, true);
            } else {
                if (layout == 1) ANTS_PERCEIVE(1, false);
                else if (layout == 2) ANTS_PERCEIVE(2, false);
                else ANTS_PERCEIVE(0, false);
            }
#undef ANTS_PERCEIVE
        }
        TRY(check_launch("k_perceive"));
    }
    b->rw_alias = 0;
    return ANTS_OK;
}


// ------------------------------------------------------------------------------------------------ block-per-env path
// The block-per-environment kernel, once per group of environments on the group's stream in a grouped rollout, else
// once over the whole batch.  Block shape from the ants per block: one ant per thread up to 512, 512 threads x 2 ants
// for 1024 (ants_env_fused.cuh).
template <bool UPDATE, bool MOVE>
int launch_env(AntsBatch *b, ants::EnvArgs a) {
    constexpr int fam = UPDATE ? (MOVE ? F_ENV_FUSED : F_ENV_UPDATE) : F_ENV_MOVE;
    const char *what = UPDATE ? (MOVE ? "k_env<update, move>" : "k_env<update>") : "k_env<move>";
    const Params &p = b->p;
    const AntsBatch::Group whole = {b->stream, nullptr, 0, p.E};
    const AntsBatch::Group *gs = b->grouped ? b->groups.data() : &whole;
    const int n = b->grouped ? (int)b->groups.size() : 1;
    const size_t smem = (size_t)b->env_smem;
    a.group = b->env_group; a.cap = b->env_cap;
    for (int k = 0; k < n; ++k) {
        a.env_base = gs[k].env0; a.env_end = gs[k].env1;
        const unsigned grid = (unsigned)cdiv(a.env_end - a.env_base, b->env_group);
        {
            LaunchScope ls(b, fam);
            if (b->env_cap == 1024) launch_step(b, gs[k].s, ants::k_env<UPDATE, MOVE, 2, 512>, grid, 512u, smem, p, a);
            else if (b->env_cap == 512) launch_step(b, gs[k].s, ants::k_env<UPDATE, MOVE, 1, 512>, grid, 512u, smem, p, a);
            else launch_step(b, gs[k].s, ants::k_env<UPDATE, MOVE, 1, 256>, grid, 256u, smem, p, a);
        }
        TRY(check_launch(what));
    }
    return ANTS_OK;
}

// Lazy evaporation: no pass over the field, values are evaluated at read time from their write timestamps.  An update
// advances the two counters the deposits are stamped with; before either wraps, one pass folds the plain values (8-byte
// records keep 15 bits of the deposit step: expired deposits are cleared every 16384 updates, before an age of
// tab_len <= 16384 could alias; the step counter itself keeps running).
int advance_lazy_counters(AntsBatch *b) {
    const Params &p = b->p;
    const bool unbox = p.rec8 ? ((b->lazy_abs & 0x3FFFu) == 0x3FFFu) : (b->lazy_abs >= ants::kBoxMask - 2u);
    if (b->lazy_now >= p.ts_mask - 1u || unbox) {
        WholeBatchPass wb(b);
        LaunchScope ls(b, F_EVAP);
        ants::k_lazy_fold<<<148 * 16, 256, 0, b->stream>>>(p, b->lazy_now, b->lazy_abs, unbox ? 1 : 0);
        b->lazy_now = 0;
        if (unbox && !p.rec8) b->lazy_abs = 0;
        TRY(check_launch("k_lazy_fold"));
    }
    b->lazy_now += 1;
    b->lazy_abs += 1;
    return ANTS_OK;
}

// host bookkeeping at the start of a step: generation folds, the step's occupancy generation, the move's arguments
void env_args_move(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph, ants::EnvArgs *a) {
    maybe_fold_generations(b);
    a->rot = d_rot; a->ph = d_ph;
    a->occ_gen = next_occ_gen(b);
    a->all_stamp = b->prev_synced ? 0 : 1;
    a->act_on = b->act_bool ? 1.0 : 256.0;
}
// ... of an update: timestep, the lazy field's counters
int env_args_update(AntsBatch *b, const double *d_noise, ants::EnvArgs *a) {
    a->step_id = (uint32_t)b->timestep;
    b->timestep += 1;                                               // environment.py:45
    if (b->p.P > 0 && b->p.lazy) TRY(advance_lazy_counters(b));
    a->noise = d_noise;
    a->use_flag = b->wall_flags_valid;
    a->now = b->lazy_now; a->now_abs = b->lazy_abs;
    return ANTS_OK;
}

int finish_update(AntsBatch *b) {
    const Params &p = b->p;
    b->wall_flags_valid = 0;
    b->stats.active_tiles = 0;
    if (b->needs_sweep) {          // Anthill (order 1000) after an import: whatever the generator put into the disc (Q10)
        WholeBatchPass wb(b);
        LaunchScope ls(b, F_ABSORB);
        ants::k_absorb_sweep<<<p.E, 256, 0, b->stream>>>(p);
        b->needs_sweep = 0;
        TRY(check_launch("absorb"));
    }
    b->prev_synced = 1;
    b->stats.updates++;
    return ANTS_OK;
}

int do_step_fused(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph, float *d_obs, float *d_as, double *d_reward,
                  int32_t *done) {
    if (!b->move_done) {
        ants::EnvArgs a = {};
        env_args_move(b, d_rot, d_ph, &a);
        TRY((launch_env<false, true>(b, a)));
    }
    b->move_done = 0;
    b->prev_synced = 0;
    b->wall_flags_valid = 1;
    TRY(launch_perceive(b, d_obs, d_as, nullptr, d_reward, 1));
    if (done) *done = (b->cfg.max_time == b->timestep) ? 1 : 0;   // RL_api.py:200 (Q15)
    b->stats.steps++;
    return ANTS_OK;
}

int do_update_fused(AntsBatch *b, const double *d_noise) {
    ants::EnvArgs a = {};
    TRY(env_args_update(b, d_noise, &a));
    TRY((launch_env<true, false>(b, a)));
    return finish_update(b);
}

// update_k ; move of step_{k+1} in ONE launch (ants_rollout): legal because nothing between an update and the next
// step's move reads what either writes (quirk Q2 only forbids fusing a step with ITS OWN update)
int do_update_move_fused(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph) {
    if (b->needs_sweep) return fail(ANTS_E_STATE, "internal: fused update+move with a pending anthill sweep");
    ants::EnvArgs a = {};
    TRY(env_args_update(b, nullptr, &a));
    b->prev_synced = 1;
    env_args_move(b, d_rot, d_ph, &a);
    TRY((launch_env<true, true>(b, a)));
    b->wall_flags_valid = 0;
    b->stats.active_tiles = 0;
    b->stats.updates++;
    b->move_done = 1;
    return ANTS_OK;
}

// ------------------------------------------------------------------------------------------------ grouped rollout
int ensure_groups(AntsBatch *b, int want) {
    if (!b->groups.empty()) return ANTS_OK;
    const Params &p = b->p;
    if (cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming) != cudaSuccess) return fail(ANTS_E_CUDA, "cudaEventCreate failed");
    const int blocks = (int)cdiv(p.E, b->env_group);                 // block-per-env kernel: env_group envs per block
    const int G = want < blocks ? want : blocks;
    for (int g = 0; g < G; ++g) {
        AntsBatch::Group gr;
        gr.env0 = (int)((int64_t)blocks * g / G) * b->env_group;
        gr.env1 = g + 1 == G ? p.E : (int)((int64_t)blocks * (g + 1) / G) * b->env_group;
        if (cudaStreamCreateWithFlags(&gr.s, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&gr.done, cudaEventDisableTiming) != cudaSuccess)
            return fail(ANTS_E_CUDA, "stream / event creation for the rollout groups failed");
        b->groups.push_back(gr);
    }
    return ANTS_OK;
}

int do_observe(AntsBatch *b, float *d_obs, float *d_as, float *d_state, double *d_reward) {
    if (!d_obs || !d_as) return fail(ANTS_E_ARG, "ants_observe: obs and agent_state buffers are required");
    const Params &p = b->p;
    maybe_fold_generations(b);
    uint32_t occ = next_occ_gen(b);
    {
        LaunchScope ls(b, F_MOVE);
        ants::k_occ_stamp<<<(int)cdiv(p.EN, 256), 256, 0, b->stream>>>(p, occ);
    }
    TRY(check_launch("k_occ_stamp"));
    TRY(launch_perceive(b, d_obs, d_as, d_state, d_reward, 0));
    b->stats.observations++;
    return ANTS_OK;
}

int do_step(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph, float *d_obs, float *d_as, double *d_reward,
            int32_t *done) {
    if (!d_obs || !d_as) return fail(ANTS_E_ARG, "ants_step: obs and agent_state buffers are required");
    const Params &p = b->p;
    if (d_ph && p.P != 2)
        return fail(ANTS_E_ARG, "pheromone actions need exactly two pheromones (ants.py:92-96), have %d", p.P);
    if (b->fused) return do_step_fused(b, d_rot, d_ph, d_obs, d_as, d_reward, done);
    maybe_fold_generations(b);
    uint32_t phase = next_owner_phase(b);
    uint32_t occ = next_occ_gen(b);
    int blocks = (int)cdiv(p.EN, 256);
    {
        LaunchScope ls(b, F_MOVE);
        launch_step(b, b->stream, ants::k_step_move, (unsigned)blocks, 256u, (size_t)0, p, d_rot, d_ph, phase << 16, occ,
                    b->prev_synced ? 0 : 1, b->act_bool ? 1.0 : 256.0, b->commit_par);
    }
    TRY(check_launch("k_step_move"));
    {
        LaunchScope ls(b, F_FOOD);
        launch_step(b, b->stream, ants::k_food_commit, 64u, 128u, (size_t)0, p, phase << 16, b->absorb_par, b->commit_par);
        b->commit_par ^= 1;
    }
    TRY(check_launch("k_food_commit"));
    if (++b->steps_queued > 1) b->needs_sweep = 1;   // the absorb list may have overflowed (k_food_commit)
    b->prev_synced = 0;
    b->wall_flags_valid = 1;
    TRY(launch_perceive(b, d_obs, d_as, nullptr, d_reward, 1));
    if (done) *done = (b->cfg.max_time == b->timestep) ? 1 : 0;   // RL_api.py:200 (Q15)
    b->stats.steps++;
    return ANTS_OK;
}

int do_update(AntsBatch *b, const double *d_noise) {
    if (b->fused) return do_update_fused(b, d_noise);
    Params &p = b->p;
    int blocks = (int)cdiv(p.EN, 256);
    uint32_t step_id = (uint32_t)b->timestep;
    b->timestep += 1;                                               // environment.py:45
    uint32_t phase = next_owner_phase(b);
    // 1. Walls (order -1) on ants; without rocks also the ant part of Ants.update (order 999), which touches
    //    nothing the objects in between read.
    {
        LaunchScope ls(b, F_COLLIDE);
        launch_step(b, b->stream, ants::k_collide, (unsigned)blocks, 256u, (size_t)0, p, d_noise, step_id, phase << 16,
                    p.R > 0 ? 0 : 1, b->wall_flags_valid, b->absorb_par);
        b->absorb_par ^= 1;
        b->wall_flags_valid = 0;
    }
    TRY(check_launch("k_collide"));
    // 3. CircleObstacles (order 0)
    if (p.R > 0) {
        {
            LaunchScope ls(b, F_ROCKS);
            launch_step(b, b->stream, ants::k_rocks_pushed, (unsigned)cdiv((int64_t)p.E * p.R, 8), 256u, (size_t)0, p);
        }
        TRY(check_launch("k_rocks_pushed"));
        {
            LaunchScope ls(b, F_ROCKS);
            launch_step(b, b->stream, ants::k_rocks_push_ants, (unsigned)blocks, 256u, (size_t)0, p, phase << 16);
        }
        TRY(check_launch("k_rocks_push_ants"));
    }
    // 1b + 4. wall zeroing of the field (walls.py:30) and Pheromone.update (order 0)
    if (p.P > 0) {
        if (p.lazy) {
            TRY(advance_lazy_counters(b));
            b->stats.active_tiles = 0;
        } else if (b->cfg.diffuse_factor != 0.0) {
            int nbx = (int)cdiv(p.W, ants::kStX), nby = (int)cdiv(p.H, ants::kStY);
            {
                LaunchScope ls(b, F_EVAP);
                ants::k_diffuse_tma<<<(unsigned)((int64_t)nbx * nby * p.E * p.P), 256, 0, b->stream>>>(
                    p, b->plane_map, b->plane_src * p.E * p.P, nbx, nby);
            }
            TRY(check_launch("k_diffuse_tma"));
            std::swap(p.phero_pl, p.phero_alt);            // the stencil's output is the field from now on
            b->plane_src ^= 1;
            b->stats.active_tiles = b->stats.total_tiles;
        } else if (b->cfg.evap_mode == ANTS_EVAP_ACTIVE_TILES) {
            CK(cudaMemsetAsync(p.tile_counter, 0, sizeof(unsigned long long), b->stream));
            {
                LaunchScope ls(b, F_EVAP);
                ants::k_tiles_compact<<<148 * 4, 256, 0, b->stream>>>(p, b->tile_list);
            }
            TRY(check_launch("k_tiles_compact"));
            LaunchScope ls(b, F_EVAP);
            ants::k_evaporate_tiles<<<148 * 16, 256, 0, b->stream>>>(p, b->tile_list);
        } else {
            LaunchScope ls(b, F_EVAP);
            ants::k_evaporate_dense<<<148 * 16, 256, 0, b->stream>>>(p);
        }
        TRY(check_launch("evaporate"));
        // 6. Ants.update (order 999): deposit
        {
            LaunchScope ls(b, F_DEPOSIT);
            launch_step(b, b->stream, ants::k_deposit_commit, (unsigned)blocks, 256u, (size_t)0, p, phase << 16,
                        b->lazy_now, b->lazy_abs);
        }
        TRY(check_launch("k_deposit_commit"));
    }
    // 7. Anthill (order 1000): the queued cells were absorbed by the first blocks of k_collide; after an import one
    //    sweep over the disc takes whatever the generator put there (Q10), after several steps without an update
    //    whatever did not fit the list
    if (b->needs_sweep) {
        LaunchScope ls(b, F_ABSORB);
        ants::k_absorb_sweep<<<p.E, 256, 0, b->stream>>>(p);
        b->needs_sweep = 0;
        TRY(check_launch("absorb"));
    }
    b->steps_queued = 0;
    b->prev_synced = 1;
    b->stats.updates++;
    return ANTS_OK;
}

int ensure_staging(AntsBatch *b) {
    if (b->st_obs) return ANTS_OK;
    const Params &p = b->p;
    TRY(dev_alloc(b, &b->st_rot, p.EN, false));
    TRY(dev_alloc(b, &b->st_ph, p.EN, false));
    TRY(dev_alloc(b, &b->st_obs, p.EN * p.S2 * p.C, false));
    TRY(dev_alloc(b, &b->st_as, p.EN * 2, false));
    TRY(dev_alloc(b, &b->st_state, p.EN * (2 + p.P), false));
    TRY(dev_alloc(b, &b->st_reward, p.EN, false));
    TRY(dev_alloc(b, &b->st_noise, p.EN, false));
    return ANTS_OK;
}

int ensure_packed(AntsBatch *b) {
    if (b->st_packed) return ANTS_OK;
    const int64_t bytes = b->p.EN * b->pack_layout.bytes_per_ant;
    TRY(dev_alloc(b, &b->st_packed, bytes + 64, false));
    TRY(dev_alloc(b, &b->d_pack_fail, 1));
    if (cudaHostAlloc((void **)&b->h_packed, (size_t)bytes + 64, cudaHostAllocDefault) != cudaSuccess)
        return fail(ANTS_E_ALLOC, "cudaHostAlloc of %lld bytes (packed observation staging) failed", (long long)bytes);
    int max_chunks = 16;
    if (const char *x = getenv("ANTS_E2E_CHUNKS")) max_chunks = atoi(x) < 1 ? 1 : (atoi(x) > 256 ? 256 : atoi(x));
    b->chunk_ev.resize(max_chunks);
    for (auto &e : b->chunk_ev)
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess)
            return fail(ANTS_E_CUDA, "cudaEventCreate failed");
    return ANTS_OK;
}

// The observation of the last step (dense in st_obs) -> packed on the device -> host, in chunks; with h_obs the chunks
// are expanded into the dense host array by the worker threads while the following ones are still on the bus.
// Returns 1 if some value of this step has no packed form (the caller copies dense).
int packed_transfer(AntsBatch *b, uint8_t *h_dst, float *h_obs, float *h_agent_state, double *h_reward) {
    const Params &p = b->p;
    const AntsPackedLayout &L = b->pack_layout;
    const int64_t EN = p.EN, bpa = L.bytes_per_ant, dense = (int64_t)p.S2 * p.C;
    const double t_start = HostPool::now();
    // ants [0, n_packed) cross PCIe packed (and are expanded by the host threads when a dense array is wanted); ants
    // [n_packed, EN) are copied dense by the DMA engine
    int64_t n_dense = 0;
    if (h_obs) {
        n_dense = (int64_t)(b->dense_frac * (double)EN) / 64 * 64;
        n_dense = n_dense < 0 ? 0 : (n_dense > EN ? EN : n_dense);
    }
    const int64_t n_packed = EN - n_dense;
    CK(cudaMemsetAsync(b->d_pack_fail, 0, sizeof(uint32_t), b->stream));
    int n_chunks = (int)(n_packed / (b->chunk_ev.size() > 16 ? 2048 : 16384));
    n_chunks = n_chunks < 1 ? 1 : (n_chunks > (int)b->chunk_ev.size() ? (int)b->chunk_ev.size() : n_chunks);
    const int64_t per = (cdiv(n_packed > 0 ? n_packed : 1, n_chunks) + 63) / 64 * 64;
    int used = 0;
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t a0 = c * per, n = n_packed - a0 < per ? n_packed - a0 : per;
        if (n <= 0) break;
        {
            LaunchScope ls(b, F_PACK);
            ants::k_pack_obs<<<(unsigned)cdiv(n * L.n_visible, 256), 256, 0, b->stream>>>(b->pack_args, b->st_obs, b->st_packed, a0, n,
                                                                                       b->d_pack_fail);
        }
        TRY(check_launch("k_pack_obs"));
        CK(cudaMemcpyAsync(h_dst + a0 * bpa, b->st_packed + a0 * bpa, (size_t)(n * bpa), cudaMemcpyDeviceToHost, b->stream));
        CK(cudaEventRecord(b->chunk_ev[c], b->stream));
        used = c + 1;
    }
    if (n_dense > 0)
        CK(cudaMemcpyAsync(h_obs + n_packed * dense, b->st_obs + n_packed * dense, (size_t)(n_dense * dense) * sizeof(float),
                           cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(h_agent_state, b->st_as, (size_t)EN * 8, cudaMemcpyDeviceToHost, b->stream));
    if (h_reward) CK(cudaMemcpyAsync(h_reward, b->st_reward, (size_t)EN * 8, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(b->h_counts + 8, b->d_pack_fail, sizeof(uint32_t), cudaMemcpyDeviceToHost, b->stream));
    if (h_obs) {
        HostPool &pool = HostPool::get();
        const AntsUnpackPlan *plan = b->unpack_plan;
        const int T = pool.size();
        for (int c = 0; c < used; ++c) {
            const int64_t a0 = c * per, n = n_packed - a0 < per ? n_packed - a0 : per;
            CK(cudaEventSynchronize(b->chunk_ev[c]));
            const int64_t piece = cdiv(n, T);
            for (int64_t s0 = 0; s0 < n; s0 += piece) {
                const int64_t cnt = n - s0 < piece ? n - s0 : piece, first = a0 + s0;
                pool.submit([=] { ants_unpack_range(plan, h_dst + first * bpa, cnt, h_obs + first * dense); });
            }
        }
    }
    CK(cudaStreamSynchronize(b->stream));
    if (h_obs) {
        const double t_dma = HostPool::now();
        const double t_cpu = used > 0 ? HostPool::get().wait_idle() : t_dma;
        if (!b->dense_frac_fixed && !b->h_counts[8]) {
            // move the split towards the side that finished first (half of the imbalance per step)
            const double total = HostPool::now() - t_start;
            if (total > 0.0) b->dense_frac += 0.5 * (t_cpu - t_dma) / total * (b->dense_frac > 0.05 ? b->dense_frac + 0.3 : 0.35);
            b->dense_frac = b->dense_frac < 0.0 ? 0.0 : (b->dense_frac > 0.9 ? 0.9 : b->dense_frac);
        }
    }
    return b->h_counts[8] ? 1 : ANTS_OK;
}

bool packed_path_wanted(const AntsBatch *b) {
    if (!b->pack_layout.supported || b->pack_disabled || getenv("ANTS_E2E_DENSE")) return false;
    if (getenv("ANTS_E2E_PACKED")) return true;                        // (tests: also for small batches)
    return b->p.EN * b->p.S2 * b->p.C * 4 >= (int64_t)(4 << 20);       // small batches: one dense copy is cheaper
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

int ants_abi_version(void) { return ANTS_ABI_VERSION; }
const char *ants_last_error(void) { return g_err.c_str(); }

int ants_create(const AntsConfig *cfg, AntsBatch **out) {
    if (!cfg || !out) return fail(ANTS_E_ARG, "ants_create: null argument");
    *out = nullptr;
    if (cfg->abi_version != ANTS_ABI_VERSION)
        return fail(ANTS_E_ARG, "abi_version %d != %d", cfg->abi_version, ANTS_ABI_VERSION);
    if (cfg->n_envs < 1 || cfg->n_ants < 1 || cfg->w < 1 || cfg->h < 1)
        return fail(ANTS_E_ARG, "n_envs, n_ants, w, h must be >= 1");
    if (cfg->n_ants > ANTS_MAX_ANTS) return fail(ANTS_E_ARG, "n_ants %d > %d", cfg->n_ants, ANTS_MAX_ANTS);
    if ((int64_t)cfg->n_envs * cfg->n_ants >= (1ll << 31)) return fail(ANTS_E_ARG, "n_envs * n_ants must be < 2^31");
    if (cfg->n_phero < 0 || cfg->n_phero > ANTS_MAX_PHERO) return fail(ANTS_E_ARG, "n_phero out of range");
    if (cfg->n_rocks < 0 || cfg->n_rocks > ANTS_MAX_ROCKS) return fail(ANTS_E_ARG, "n_rocks out of range");
    if (cfg->radius < 0 || cfg->radius > ANTS_MAX_RADIUS) return fail(ANTS_E_ARG, "radius out of range");
    if (cfg->n_channels < 1 || cfg->n_channels > ANTS_MAX_CHANNELS) return fail(ANTS_E_ARG, "n_channels out of range");
    if (cfg->reward_kind < 0 || cfg->reward_kind > 2) return fail(ANTS_E_ARG, "reward_kind out of range");
    for (int c = 0; c < cfg->n_channels; ++c) {
        int k = cfg->channel_kind[c];
        if (k < 0 || k > ANTS_CH_ROCKS) return fail(ANTS_E_ARG, "channel %d: unknown kind %d", c, k);
        if (k == ANTS_CH_PHERO) {
            if (cfg->channel_arg[c] < 0 || cfg->channel_arg[c] >= cfg->n_phero)
                return fail(ANTS_E_ARG, "channel %d: pheromone index out of range", c);
            if (!cfg->has_max_val)
                return fail(ANTS_E_ARG, "a perceived pheromone needs max_val (RL_api.py:125 divides by it)");
        }
        if (k == ANTS_CH_ROCKS && cfg->n_rocks == 0) return fail(ANTS_E_ARG, "rocks channel without rocks");
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(ANTS_E_CUDA, "no CUDA device (%s); libantsrl_b200 has no CPU path",
                    ce == cudaSuccess ? "device count 0" : cudaGetErrorString(ce));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(ANTS_E_ARG, "device %d of %d", cfg->device, ndev);
    CK(cudaSetDevice(cfg->device));

    AntsBatch *b = new AntsBatch();
    b->cfg = *cfg;
    memset(&b->stats, 0, sizeof b->stats);
    memset(b->fam_ms, 0, sizeof b->fam_ms);
    memset(b->fam_launches, 0, sizeof b->fam_launches);
    if (cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete b;
        return fail(ANTS_E_CUDA, "cudaStreamCreate failed");
    }
    b->stream = b->own_stream;
    Params &p = b->p;
    memset(&p, 0, sizeof p);
    p.E = cfg->n_envs; p.N = cfg->n_ants; p.W = cfg->w; p.H = cfg->h; p.P = cfg->n_phero; p.R = cfg->n_rocks;
    p.Hp = (int)(cdiv(cfg->h, 16) * 16);
    p.Wp = (int)(cdiv(cfg->w, 16) * 16);
    p.nby = p.Hp / 8;
    p.EN = (int64_t)p.E * p.N;
    b->use_pdl = (p.EN >= 131072 || getenv("ANTS_FORCE_PDL")) ? 1 : 0;   // (ANTS_FORCE_PDL: the parity tests under PDL)
    if (getenv("ANTS_NO_PDL")) b->use_pdl = 0;
    p.plane = (int64_t)p.Wp * p.Hp;
    p.radius = cfg->radius; p.S = 2 * cfg->radius + 1; p.S2 = p.S * p.S; p.C = cfg->n_channels;
    p.has_mask = cfg->has_mask;
    p.rule_n = 0;
    for (int c = 0; c < p.C; ++c) {
        p.ch_kind[c] = cfg->channel_kind[c];
        p.ch_arg[c] = cfg->channel_arg[c];
        if (cfg->channel_kind[c] == ANTS_CH_FOOD) p.rule_op[p.rule_n++] = 0;
        if (cfg->channel_kind[c] == ANTS_CH_ANTHILL) p.rule_op[p.rule_n++] = 1;
    }
    p.reward_kind = cfg->reward_kind;
    p.explore_on = (cfg->reward_kind == ANTS_REWARD_EXPLORE) ||
                   (cfg->reward_kind == ANTS_REWARD_ALL &&
                    (cfg->reward_factors[0] != 0.0 || cfg->reward_factors[3] != 0.0));
    p.has_max_val = cfg->has_max_val;
    p.tiles_x = (int)cdiv(p.W, ants::kTile);
    p.tiles_y = p.Hp / ants::kTile;
    // cell record: { f64 phero[P]; f64 food; u32 meta; u8 wall; pad } in 32 B (P <= 2) or 64 B
    p.food_off = 8 * p.P; p.meta_off = 8 * p.P + 8; p.wall_off = 8 * p.P + 12;
    p.rec_shift = (8 * p.P + 16 <= 32) ? 5 : 6;
    p.rec16 = 0; p.ts_mask = 0xFFFu; p.explored_old = 0xFFFFu;
    if (cfg->record_format == ANTS_REC_COMPACT) {
        if (!(cfg->evap_mode == ANTS_EVAP_LAZY && cfg->diffuse_factor == 0.0 && p.P >= 1 && p.P <= 2)) {
            ants_destroy(b);
            return fail(ANTS_E_ARG, "compact records need evap_mode LAZY, no diffusion and 1 or 2 pheromones");
        }
        p.rec16 = 1; p.rec_shift = 4; p.ts_mask = 0xFFu; p.explored_old = 0x7Fu;
    } else if (cfg->record_format == ANTS_REC_COMPACT8) {
        if (!(cfg->evap_mode == ANTS_EVAP_LAZY && cfg->diffuse_factor == 0.0 && p.P >= 1 && p.P <= 2)) {
            ants_destroy(b);
            return fail(ANTS_E_ARG, "compact records need evap_mode LAZY, no diffusion and 1 or 2 pheromones");
        }
        p.rec8 = 1; p.rec_shift = 3; p.ts_mask = 0xFFu; p.explored_old = 0x7Fu;
    } else if (cfg->record_format != ANTS_REC_F64) {
        int bad = cfg->record_format;
        ants_destroy(b);
        return fail(ANTS_E_ARG, "unknown record_format %d", bad);
    }
    p.ts_off = 8 * p.P + 16;
    p.grid_w = (int)cdiv(p.W, 1 << ants::kGridShift);
    p.grid_h = (int)cdiv(p.H, 1 << ants::kGridShift);
    p.delta = cfg->delta; p.fwd_delta = cfg->fwd_delta; p.reward_threshold = cfg->reward_threshold;
    p.max_speed = cfg->max_speed; p.max_rot_speed = cfg->max_rot_speed;
    p.csr = cfg->carry_speed_reduction; p.bsr = cfg->backward_speed_reduction;
    p.f_explore = cfg->reward_factors[0]; p.f_food = cfg->reward_factors[1]; p.f_anthill = cfg->reward_factors[2];
    p.f_explore_hold = cfg->reward_factors[3]; p.f_heading = cfg->reward_factors[4];
    // pheromone.py:7-9: ring = DF, centre = 1 - 8 DF, all times (1 - EVAP)
    {
        volatile double ring = 1.0 * cfg->diffuse_factor;
        volatile double centre = 1.0 - 8.0 * cfg->diffuse_factor;
        volatile double keep = 1.0 - cfg->evap_factor;
        p.filt_ring = ring * keep;
        p.filt_center = centre * keep;
    }
    p.phero_max_val = cfg->phero_max_val; p.max_hold = cfg->max_hold;
    p.lazy = (cfg->evap_mode == ANTS_EVAP_LAZY && cfg->diffuse_factor == 0.0 && p.P > 0) ? 1 : 0;
    p.log2_keep = p.filt_center > 0.0 ? log2(p.filt_center) : -1e300;
    p.rng_seed = cfg->rng_seed; p.env_id_base = cfg->env_id_base;

    {   // block-per-environment kernels: lazy field (no pass between the rocks and the deposit), <= 1024 ants per env,
        // (env-in-block, cell) keys in 32 bits
        const int cap = p.N <= 256 ? 256 : (p.N <= 512 ? 512 : 1024);
        int g = cap / (p.N > 0 ? p.N : 1);
        g = g < 1 ? 1 : (g > ants::kEnvMaxGroup ? ants::kEnvMaxGroup : g);
        while (g > 1 && (int64_t)g * p.plane >= 0xFFFFFFF0ll) --g;
        b->fused = ((p.lazy || p.P == 0) && cfg->diffuse_factor == 0.0 && p.N <= 1024 && p.plane < 0xFFFFFFF0ll &&
                    !getenv("ANTS_NO_FUSED")) ? 1 : 0;
        b->env_group = g;
        b->env_cap = cap;
        // The block-per-environment kernel is heavy (256 threads x 64 registers, 33 KB of shared memory): launched as a
        // programmatic dependent it sits on the SMs waiting for the perception kernel and takes registers and shared
        // memory from it (measured: rollouts 0.37-0.61 ms per step against 0.36 for separate launches), so the pair
        // runs in plain stream order
        if (b->fused && !getenv("ANTS_FORCE_PDL")) b->use_pdl = 0;
        b->env_smem = cap * 32 + g * p.R * 4;
    }
    int rc = ANTS_OK;
    auto A = [&](int r) { if (rc == ANTS_OK) rc = r; };
    const int64_t EN = p.EN, cells = (int64_t)p.E * p.plane;
    A(dev_alloc(b, &p.x, EN)); A(dev_alloc(b, &p.y, EN)); A(dev_alloc(b, &p.theta, EN));
    A(dev_alloc(b, &p.prev_x, EN)); A(dev_alloc(b, &p.prev_y, EN)); A(dev_alloc(b, &p.prev_theta, EN));
    A(dev_alloc(b, &p.holding, EN)); A(dev_alloc(b, &p.seed, EN));
    A(dev_alloc(b, &p.act, EN * (p.P > 0 ? p.P : 1)));
    A(dev_alloc(b, &p.mandibles, EN)); A(dev_alloc(b, &p.reward_state, EN));
    A(dev_alloc(b, &p.rw_holding_prev, EN)); A(dev_alloc(b, &p.rw_prev_dist, EN)); A(dev_alloc(b, &p.rewards, EN));
    A(dev_alloc(b, &p.cells, cells << p.rec_shift));
    if (p.rec8) { A(dev_alloc(b, &p.side_val, cells * 3)); A(dev_alloc(b, &p.side_ts, cells * 2)); }
    p.diffuse = (cfg->diffuse_factor != 0.0 && p.P > 0) ? 1 : 0;
    if (p.diffuse) {
        A(dev_alloc(b, &p.phero_pl, 2 * cells * p.P));
        p.phero_alt = p.phero_pl ? p.phero_pl + cells * p.P : nullptr;
    }
    if (!b->fused) A(dev_alloc(b, &p.owner, cells));       // (the block-per-env kernels find owners in shared memory)
    if (cfg->evap_mode == ANTS_EVAP_ACTIVE_TILES && cfg->diffuse_factor == 0.0)
    {
        A(dev_alloc(b, &p.tile_active, (int64_t)p.E * p.tiles_x * p.tiles_y));
        A(dev_alloc(b, &b->tile_list, (int64_t)p.E * p.tiles_x * p.tiles_y, false));
    }
    A(dev_alloc(b, &p.hill, (int64_t)p.E * 4));
    A(dev_alloc(b, &p.hill_food, (int64_t)p.E));
    A(dev_alloc(b, &p.rock_c, (int64_t)p.E * p.R * 2)); A(dev_alloc(b, &p.rock_rad, (int64_t)p.E * p.R));
    A(dev_alloc(b, &p.rock_w, (int64_t)p.E * p.R));
    A(dev_alloc(b, &p.rock_grid, (int64_t)p.E * p.grid_w * p.grid_h));
    A(dev_alloc(b, &p.rock_touch, (int64_t)p.E * p.R));
    A(dev_alloc(b, &p.food_delta, EN, false));
    A(dev_alloc(b, &p.commit_list, EN, false)); A(dev_alloc(b, &p.commit_count, 2));
    A(dev_alloc(b, &p.absorb_list, EN * 2, false)); A(dev_alloc(b, &p.absorb_count, b->fused ? (p.E > 2 ? p.E : 2) : 2));
    A(dev_alloc(b, &p.wall_hit, EN));
    A(dev_alloc(b, &p.tile_counter, 1));
    A(dev_alloc(b, &p.plain_flag, 1));

    b->stats.total_tiles = (int64_t)p.E * p.tiles_x * p.tiles_y;
    // perception tables, RL_api.py:92-93: coords[i][j] = ((j - r) * DELTA, (i - r) * DELTA)
    double *d_off = nullptr;
    uint8_t *d_mask = nullptr;
    A(dev_alloc(b, &d_off, p.S)); A(dev_alloc(b, &d_mask, p.S2));
    if (rc != ANTS_OK) { ants_destroy(b); return rc; }
    if (p.diffuse) {
        // tensor map over both planes: extents are the TRUE map size, so the TMA unit zero-fills the convolution's
        // border (pheromone.py:44 boundary='fill'); the pitch is the padded row
        typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                     const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
            ants_destroy(b);
            return fail(ANTS_E_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
        }
        const cuuint64_t dims[3] = {(cuuint64_t)p.H, (cuuint64_t)p.W, (cuuint64_t)(2 * (int64_t)p.E * p.P)};
        const cuuint64_t strides[2] = {(cuuint64_t)p.Hp * 8, (cuuint64_t)p.plane * 8};
        const cuuint32_t box[3] = {(cuuint32_t)(ants::kStY + 2 + ants::kStPadY), (cuuint32_t)(ants::kStX + 2), 1u};
        const cuuint32_t estr[3] = {1u, 1u, 1u};
        CUresult cr = ((EncodeFn)fn)(&b->plane_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void *)p.phero_pl, dims, strides,
                                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) {
            ants_destroy(b);
            return fail(ANTS_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)cr);
        }
    }
    {
        std::vector<double> off(p.S);
        std::vector<uint8_t> mk(p.S2, 1);
        for (int k = 0; k < p.S; ++k) {
            volatile double fk = (double)(k - p.radius);
            off[k] = fk * cfg->delta;
        }
        if (cfg->has_mask)
            for (int k = 0; k < p.S2; ++k) mk[k] = cfg->mask[k] ? 1 : 0;
        for (int k = 0; k < 16; ++k) {
            p.off_c[k] = k < p.S ? off[k] : 0.0;
            uint32_t bits = 0;
            for (int j = 0; k < p.S && j < p.S; ++j) bits |= (uint32_t)(mk[k * p.S + j] ? 1u : 0u) << j;
            p.mask_rows[k] = bits;
        }
        cudaMemcpy(d_off, off.data(), p.S * sizeof(double), cudaMemcpyHostToDevice);
        cudaMemcpy(d_mask, mk.data(), p.S2, cudaMemcpyHostToDevice);
        p.samp_off = d_off; p.mask = d_mask;
        // pheromone.py:44-45 applied k times to max_val, with the reference's rounding at every step, until 0
        const int kTabCap = 16384;
        std::vector<double> tab;
        std::vector<float> tobs;
        volatile double v = cfg->has_max_val ? cfg->phero_max_val : 0.0;
        volatile double inv = cfg->has_max_val && cfg->phero_max_val != 0.0 ? 1.0 / cfg->phero_max_val : 0.0;
        for (int k = 0; k < kTabCap; ++k) {
            const double vv = v;
            tab.push_back(vv);
            volatile double ob = vv * inv;
            tobs.push_back((float)ob);
            if (v == 0.0) break;
            volatile double nv = v * p.filt_center;
            v = nv < 0.01 ? 0.0 : nv;
        }
        p.tab_len = (int)tab.size();
        if (p.lazy && cfg->has_max_val && tab.back() != 0.0) {
            // a saturated deposit must decay to 0 within the table (boxed deposits read 0 beyond it, and the 15-bit
            // deposit step of the 8-byte records is recycled every 16384 updates)
            ants_destroy(b);
            return fail(ANTS_E_ARG, "evap_factor %g: a max_val deposit needs more than %d updates to fall below 0.01; "
                        "use evap_mode DENSE or ACTIVE_TILES", cfg->evap_factor, kTabCap);
        }
        double *d_table = nullptr;
        float *d_tobs = nullptr;
        if (dev_alloc(b, &d_table, p.tab_len) != ANTS_OK || dev_alloc(b, &d_tobs, p.tab_len) != ANTS_OK) {
            ants_destroy(b);
            return ANTS_E_ALLOC;
        }
        cudaMemcpy(d_table, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice);
        cudaMemcpy(d_tobs, tobs.data(), tobs.size() * sizeof(float), cudaMemcpyHostToDevice);
        p.decay_obs = d_tobs;
        p.decay_table = d_table;
    }
    {   // ants per staged chunk: as many as fit ~12 KB per warp, keeping the chunk a multiple of 16 B and the
        // flat sample index below 2048 (magic division); threads per block: as many warps as fit ~100 KB
        int sc_bytes = p.S2 * p.C * 4;
        int g = ants::kMaxGroup;
        while (g > 1 && (g * sc_bytes > 8 * 1024 || g * p.S2 >= 2048)) g >>= 1;
        b->perceive_group = g;
        int threads = ants::kPerceiveThreads;
        auto smem_for = [&](int t) {
            return (int)((((t / 32) * g * p.S2 * p.C + 3) & ~3) * 4 + t * sizeof(ants::AntPrep) +
                         p.S2 * sizeof(ants::SampleTab) + t * 4 + p.S2 + 64);
        };
        while (threads > 32 && smem_for(threads) > 100 * 1024) threads >>= 1;
        b->perceive_threads = threads;
        b->perceive_smem = smem_for(threads);
        // sample offsets reach at most radius*DELTA*sqrt(2) + |fwd_delta| + 1 cells from the ant: one conditional
        // add/subtract wraps them unless the map is smaller than that
        double reach = p.radius * cfg->delta * 1.5 + fabs(cfg->fwd_delta) + 2.0;
        b->perceive_slow_wrap = (p.W <= reach || p.H <= reach) ? 1 : 0;
    }
    {   // straight-line perception code for the generator's default channel list (with / without rocks)
        const int std6[6] = {ANTS_CH_ANTS, ANTS_CH_PHERO, ANTS_CH_PHERO, ANTS_CH_ANTHILL, ANTS_CH_WALLS, ANTS_CH_FOOD};
        bool ok = p.P == 2 && (p.C == 6 || p.C == 7) && cfg->has_max_val;
        for (int c = 0; ok && c < 6; ++c) ok = p.ch_kind[c] == std6[c];
        ok = ok && p.ch_arg[1] == 0 && p.ch_arg[2] == 1;
        if (ok && p.C == 7) ok = p.ch_kind[6] == ANTS_CH_ROCKS;
        b->perceive_layout = ok ? (p.C == 7 ? 2 : 1) : 0;
    }
    {   // the row-per-lane kernel serves the default channel lists with a 7x7 (default) or 5x5 window
        const int C = p.C;
        b->perceive_rows = (b->perceive_layout != 0 && (p.S == 7 || p.S == 5) && !b->perceive_slow_wrap &&
                            !getenv("ANTS_PERCEIVE_GENERIC")) ? 1 : 0;
        b->rows_smem = (ants::kRowsThreads / 32) * ants::kRowsTiles * ants::kRowsGroup * p.S2 * C * 4 +
                       ants::kRowsThreads * (int)sizeof(ants::RowPrep) + ants::kRowsThreads * p.S;
    }
    if (b->perceive_rows) {
        const void *fns[12] = {(const void *)ants::k_perceive_rows<1, 0, 7>, (const void *)ants::k_perceive_rows<2, 0, 7>,
                               (const void *)ants::k_perceive_rows<1, 1, 7>, (const void *)ants::k_perceive_rows<2, 1, 7>,
                               (const void *)ants::k_perceive_rows<1, 2, 7>, (const void *)ants::k_perceive_rows<2, 2, 7>,
                               (const void *)ants::k_perceive_rows<1, 0, 5>, (const void *)ants::k_perceive_rows<2, 0, 5>,
                               (const void *)ants::k_perceive_rows<1, 1, 5>, (const void *)ants::k_perceive_rows<2, 1, 5>,
                               (const void *)ants::k_perceive_rows<1, 2, 5>, (const void *)ants::k_perceive_rows<2, 2, 5>};
        for (int k = 0; k < 12 && b->rows_smem > 48 * 1024; ++k)
            if (cudaFuncSetAttribute(fns[k], cudaFuncAttributeMaxDynamicSharedMemorySize, b->rows_smem) != cudaSuccess) {
                ants_destroy(b);
                return fail(ANTS_E_CUDA, "k_perceive_rows needs %d B of shared memory", b->rows_smem);
            }
        // Shared memory / L1 split of the SM for the row kernel, in percent of shared memory: 72 % = 164 KB shared (16 - 18
        // one-warp blocks) + 92 KB L1.  The record gathers live on L1 hits; left to itself the driver sizes the split for the
        // occupancy the register count allows and leaves 28 - 60 KB of L1 (25 % slower, ants_perceive_rows.cuh).
        const char *cv = getenv("ANTS_ROWS_CARVEOUT");
        const int carve = cv ? atoi(cv) : 72;
        if (carve >= 0)
            for (int k = 0; k < 12; ++k) cudaFuncSetAttribute(fns[k], cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    }
    if (b->perceive_smem > 48 * 1024) {
        cudaError_t e = cudaSuccess;
        const void *fns[6] = {(const void *)ants::k_perceive<0, false>, (const void *)ants::k_perceive<1, false>,
                              (const void *)ants::k_perceive<2, false>, (const void *)ants::k_perceive<0, true>,
                              (const void *)ants::k_perceive<1, true>, (const void *)ants::k_perceive<2, true>};
        for (int k = 0; k < 6 && e == cudaSuccess; ++k)
            e = cudaFuncSetAttribute(fns[k], cudaFuncAttributeMaxDynamicSharedMemorySize, b->perceive_smem);
        if (e != cudaSuccess) {
            ants_destroy(b);
            return fail(ANTS_E_CUDA, "perception window needs %d B of shared memory: %s", b->perceive_smem,
                        cudaGetErrorString(e));
        }
    }
    {   // packed observation transport
        if (const char *x = getenv("ANTS_E2E_DENSE_FRACTION")) { b->dense_frac = atof(x); b->dense_frac_fixed = 1; }
        packed_layout_of(cfg, &b->pack_layout);
        b->unpack_plan = new AntsUnpackPlan();
        unpack_plan_of(&b->pack_layout, b->unpack_plan);
        ants::PackArgs &pa = b->pack_args;
        memset(&pa, 0, sizeof pa);
        pa.V = b->pack_layout.n_visible; pa.S2 = p.S2; pa.C = p.C;
        for (int k = 0; k < 8; ++k) pa.flag_ch[k] = b->pack_layout.flag_channel[k];
        pa.val_ch[0] = b->pack_layout.value_channel[0]; pa.val_ch[1] = b->pack_layout.value_channel[1];
        pa.food_ch = b->pack_layout.food_channel;
        for (int v = 0; v < pa.V; ++v) pa.vis[v] = b->pack_layout.visible_index[v];
    }
    if (cudaHostAlloc((void **)&b->h_counts, 64, cudaHostAllocDefault) != cudaSuccess) {
        ants_destroy(b);
        return fail(ANTS_E_ALLOC, "cudaHostAlloc failed");
    }
    cudaError_t se = cudaStreamSynchronize(b->stream);
    if (se != cudaSuccess) {
        ants_destroy(b);
        return fail(ANTS_E_CUDA, "initialisation failed: %s", cudaGetErrorString(se));
    }
    b->stats.device_bytes = b->device_bytes;
    *out = b;
    return ANTS_OK;
}

int ants_destroy(AntsBatch *b) {
    if (!b) return ANTS_OK;
    cudaSetDevice(b->cfg.device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    for (auto &t : b->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (auto e : b->event_pool) cudaEventDestroy(e);
    for (void *d : b->allocs) cudaFree(d);
    if (b->h_counts) cudaFreeHost(b->h_counts);
    for (auto &g : b->groups) { if (g.s) { cudaStreamSynchronize(g.s); cudaStreamDestroy(g.s); } if (g.done) cudaEventDestroy(g.done); }
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->h_packed) cudaFreeHost(b->h_packed);
    if (b->reset_discs) cudaFree(b->reset_discs);
    if (b->reset_offsets) cudaFree(b->reset_offsets);
    for (auto e : b->chunk_ev) cudaEventDestroy(e);
    delete b->unpack_plan;
    if (b->own_stream) cudaStreamDestroy(b->own_stream);
    delete b;
    return ANTS_OK;
}

int ants_set_stream(AntsBatch *b, void *cuda_stream) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaStreamSynchronize(b->stream));
    b->stream = (cudaStream_t)cuda_stream;   // 0 = the legacy default stream (what torch uses by default)
    return ANTS_OK;
}

int ants_synchronize(AntsBatch *b) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    CK(cudaStreamSynchronize(b->stream));
    return ANTS_OK;
}

int ants_import_env_state(AntsBatch *b, int32_t env0, int32_t n_envs, const AntsHostState *s) {
    if (!b || !s) return fail(ANTS_E_ARG, "null argument");
    Params &p = b->p;
    if (env0 < 0 || n_envs < 1 || (int64_t)env0 + n_envs > p.E)
        return fail(ANTS_E_ARG, "env window [%d, %d) outside the batch of %d envs", env0, env0 + n_envs, p.E);
    // the per-ant and rock arrays (kilobytes per env) are checked here, before anything is uploaded: the handle stays as
    // it was.  A NaN or infinite value has no counterpart the kernels could follow (NaN positions index no cell, and a
    // NaN activation would deposit a saturated trail where the reference's convolution spreads NaN).
    const size_t an_all = (size_t)n_envs * p.N;
    const struct { const char *name; const double *v; size_t n, per_env; } finite[] = {
        {"x", s->x, an_all, (size_t)p.N}, {"y", s->y, an_all, (size_t)p.N}, {"theta", s->theta, an_all, (size_t)p.N},
        {"prev_x", s->prev_x, an_all, (size_t)p.N}, {"prev_y", s->prev_y, an_all, (size_t)p.N},
        {"prev_theta", s->prev_theta, an_all, (size_t)p.N}, {"holding", s->holding, an_all, (size_t)p.N},
        {"activation", s->activation, an_all * p.P, (size_t)p.N * p.P},
        {"rock_centers", s->rock_centers, (size_t)n_envs * p.R * 2, (size_t)p.R * 2},
        {"rock_radii", s->rock_radii, (size_t)n_envs * p.R, (size_t)p.R},
        {"rock_weights", s->rock_weights, (size_t)n_envs * p.R, (size_t)p.R}};
    for (const auto &f : finite)
        if (f.v)
            for (size_t i = 0; i < f.n; ++i)
                if (!std::isfinite(f.v[i]))
                    return fail(ANTS_E_ARG, "env %d: %s[%zu] is %g; imported values must be finite", env0 + (int)(i / f.per_env),
                                f.name, i % f.per_env, f.v[i]);
    if (p.diffuse && s->activation) {                  // a plane value's sign bit is the wall flag: no negative deposits
        const size_t n = (size_t)n_envs * p.N * p.P;
        for (size_t i = 0; i < n; ++i)
            if (!(s->activation[i] >= 0.0))
                return fail(ANTS_E_ARG, "env %d, ant %d: activation %g; with diffusion an activation must be >= 0",
                            env0 + (int)(i / ((size_t)p.N * p.P)), (int)(i / p.P % p.N), s->activation[i]);
    }
    CK(cudaSetDevice(b->cfg.device));
    cudaStream_t st = b->stream;
    const bool whole = n_envs == p.E;
    const size_t a0 = (size_t)env0 * p.N, an = (size_t)n_envs * p.N;      // the window's ants
    const size_t AN8 = an * sizeof(double);
    auto up = [&](double *dst, const double *src) -> cudaError_t {
        return src ? cudaMemcpyAsync(dst + a0, src, AN8, cudaMemcpyHostToDevice, st) : cudaSuccess;
    };
    CK(up(p.x, s->x)); CK(up(p.y, s->y)); CK(up(p.theta, s->theta));
    CK(up(p.prev_x, s->prev_x ? s->prev_x : s->x)); CK(up(p.prev_y, s->prev_y ? s->prev_y : s->y));
    CK(up(p.prev_theta, s->prev_theta ? s->prev_theta : s->theta));
    CK(up(p.holding, s->holding)); CK(up(p.seed, s->seed));
    CK(up(p.rw_holding_prev, s->rw_holding_prev)); CK(up(p.rw_prev_dist, s->rw_prev_dist));
    CK(up(p.rewards, s->rewards));
    if (s->mandibles) CK(cudaMemcpyAsync(p.mandibles + a0, s->mandibles, an, cudaMemcpyHostToDevice, st));
    if (s->reward_state) CK(cudaMemcpyAsync(p.reward_state + a0, s->reward_state, an, cudaMemcpyHostToDevice, st));
    std::vector<double> act_t;
    if (s->activation && p.P > 0) {                                        // device layout [P][E*N]
        act_t.resize(an * p.P);
        for (size_t i = 0; i < an; ++i)
            for (int k = 0; k < p.P; ++k) act_t[(size_t)k * an + i] = s->activation[i * p.P + k];
        for (int k = 0; k < p.P; ++k)
            CK(cudaMemcpyAsync(p.act + (size_t)k * p.EN + a0, act_t.data() + (size_t)k * an, AN8, cudaMemcpyHostToDevice, st));
    }
    if (s->x && s->prev_x && s->prev_y && s->y) {
        const bool same = memcmp(s->x, s->prev_x, AN8) == 0 && memcmp(s->y, s->prev_y, AN8) == 0;
        b->prev_synced = same ? (whole ? 1 : b->prev_synced) : 0;          // (one flag for the batch: unsynced wins)
    } else if (s->x && whole) {
        b->prev_synced = 1;
    }
    // map fields: dense host array -> device scratch -> pack kernel into the cell records
    const size_t ncell = (size_t)n_envs * p.W * p.H;
    Scratch scratch;
    uint32_t *d_bad = nullptr;                                             // one word after the data: the kBad* flags
    if (s->phero || s->food || s->walls || s->explored) {
        size_t need = ncell * 8 * ((s->phero && p.P > 1) ? p.P : 1);
        const size_t flag_off = need;
        need += sizeof(uint32_t);
        cudaError_t me = cudaMalloc(&scratch.ptr, need);
        if (me != cudaSuccess) return fail(ANTS_E_ALLOC, "import scratch of %zu bytes: %s", need, cudaGetErrorString(me));
        d_bad = (uint32_t *)((char *)scratch.ptr + flag_off);
        CK(cudaMemsetAsync(d_bad, 0, sizeof(uint32_t), st));
    }
    void *const d_tmp = scratch.ptr;
    if (s->phero && p.P > 0) {
        CK(cudaMemcpyAsync(d_tmp, s->phero, ncell * 8 * p.P, cudaMemcpyHostToDevice, st));
        for (int k = 0; k < p.P; ++k)
            ants::k_pack_f64<<<148 * 8, 256, 0, st>>>(p, (const double *)d_tmp, p.P, k, 8 * k, k, b->lazy_now, b->lazy_abs,
                                                      env0, n_envs, d_bad);
        TRY(check_launch("k_pack_f64"));
        if (p.tile_active) {
            ants::k_tiles_from_phero<<<148 * 4, 256, 0, st>>>(p, env0, n_envs);
            TRY(check_launch("k_tiles_from_phero"));
        }
    }
    if (s->food) {
        CK(cudaMemcpyAsync(d_tmp, s->food, ncell * 8, cudaMemcpyHostToDevice, st));
        ants::k_pack_f64<<<148 * 8, 256, 0, st>>>(p, (const double *)d_tmp, 1, 0, p.food_off, -1, 0u, 0u, env0, n_envs,
                                                  d_bad);
        TRY(check_launch("k_pack_f64"));
        b->needs_sweep = 1;
    }
    if (s->walls) {
        CK(cudaMemcpyAsync(d_tmp, s->walls, ncell, cudaMemcpyHostToDevice, st));
        ants::k_pack_u8<<<148 * 8, 256, 0, st>>>(p, (const uint8_t *)d_tmp, 0, env0, n_envs);      // Walls.__init__: astype(bool)
        TRY(check_launch("k_pack_u8"));
    }
    if (p.diffuse && (s->walls || s->phero)) {         // the planes carry the wall bit in their sign
        ants::k_plane_walls<<<148 * 8, 256, 0, st>>>(p, env0, n_envs, s->phero ? d_bad : nullptr);
        TRY(check_launch("k_plane_walls"));
    }
    uint32_t bad = 0;
    if (d_bad) CK(cudaMemcpyAsync(&bad, d_bad, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (s->explored) {
        CK(cudaMemcpyAsync(d_tmp, s->explored, ncell, cudaMemcpyHostToDevice, st));
        ants::k_pack_u8<<<148 * 8, 256, 0, st>>>(p, (const uint8_t *)d_tmp, 1, env0, n_envs);
        TRY(check_launch("k_pack_u8"));
        // explored cells are stored as "explored long ago" / 0 and occupancy as 0: valid under any generation, so the
        // counters only restart when the whole batch was replaced
        if (whole) { b->obs_gen = 0; b->occ_gen = 0; }
    }
    std::vector<int32_t> hill4;
    if (s->anthill_xyr) {
        hill4.resize((size_t)n_envs * 4);
        for (int e = 0; e < n_envs; ++e) {
            int32_t r = s->anthill_xyr[3 * e + 2];
            hill4[4 * e] = s->anthill_xyr[3 * e]; hill4[4 * e + 1] = s->anthill_xyr[3 * e + 1];
            hill4[4 * e + 2] = r; hill4[4 * e + 3] = r < 0 ? -1 : r * r;
        }
        CK(cudaMemcpyAsync(p.hill + (size_t)env0 * 4, hill4.data(), hill4.size() * 4, cudaMemcpyHostToDevice, st));
        ants::k_hill_mark<<<148 * 8, 256, 0, st>>>(p, env0, n_envs);
        TRY(check_launch("k_hill_mark"));
        b->needs_sweep = 1;
    }
    if (s->anthill_food) CK(cudaMemcpyAsync(p.hill_food + env0, s->anthill_food, (size_t)n_envs * 8, cudaMemcpyHostToDevice, st));
    if (p.R > 0) {
        const size_t r0 = (size_t)env0 * p.R, rn = (size_t)n_envs * p.R;
        if (s->rock_centers) CK(cudaMemcpyAsync(p.rock_c + r0 * 2, s->rock_centers, rn * 16, cudaMemcpyHostToDevice, st));
        if (s->rock_radii) CK(cudaMemcpyAsync(p.rock_rad + r0, s->rock_radii, rn * 8, cudaMemcpyHostToDevice, st));
        if (s->rock_weights) CK(cudaMemcpyAsync(p.rock_w + r0, s->rock_weights, rn * 8, cudaMemcpyHostToDevice, st));
        ants::k_rock_grid_build<<<n_envs, 128, 0, st>>>(p, env0);
        TRY(check_launch("k_rock_grid_build"));
    }
    if (p.owner) CK(cudaMemsetAsync(p.owner, 0, (size_t)p.E * p.plane * sizeof(uint32_t), st));
    b->move_done = 0;
    if (s->food) b->pack_disabled = 0;
    // queued anthill absorbs refer to the old food field / disc: dropped when one of them is replaced (the sweep of the
    // next update takes whatever lies in the disc, Q10).  The flat kernels keep one batch-wide queue, so a partial import
    // drops all of it: an entry of a replaced env may name a cell outside its new disc, and the entries of the other envs
    // lie in discs that the same sweep covers.
    if (s->food || s->anthill_xyr) {
        if (b->fused) CK(cudaMemsetAsync(p.absorb_count + env0, 0, (size_t)n_envs * sizeof(uint32_t), st));
        else CK(cudaMemsetAsync(p.absorb_count, 0, 2 * sizeof(uint32_t), st));
    }
    if (s->x || s->y) b->wall_flags_valid = 0;
    b->owner_phase = 0;
    // batch-wide scalars: only when the caller provides them (0 / negative = leave as they are)
    if (s->timestep > 0) b->timestep = s->timestep;
    if (s->rw_alias >= 0) b->rw_alias = s->rw_alias ? 1 : 0;
    if (s->act_bool >= 0) b->act_bool = s->act_bool ? 1 : 0;
    CK(cudaStreamSynchronize(st));   // host temporaries above must outlive the copies
    if (bad & ants::kBadNonFinite)
        return fail(ANTS_E_ARG, "an imported pheromone or food value is NaN or infinite (import the window again)");
    if (bad & ants::kBadAboveMax)
        return fail(ANTS_E_ARG, "an imported pheromone value is above max_val %g; lazy fields hold values <= max_val "
                    "(import the window again)", p.phero_max_val);
    if (bad & ants::kBadNegative)
        return fail(ANTS_E_ARG, "an imported pheromone value is negative or NaN; with diffusion values must be >= 0 "
                    "(import the window again)");
    return ANTS_OK;
}

int ants_import_state(AntsBatch *b, const AntsHostState *s) {
    if (!b) return fail(ANTS_E_ARG, "null argument");
    return ants_import_env_state(b, 0, b->p.E, s);
}

// Checks a Perlin layer of n envs on a W x H map (the ANTS_E_ARG cases of the header) and fills its device form, all
// but the offsets pointer.  The checks keep every integer part of the noise inside int32, computed in float as pnoise2
// computes: each octave's period 1024 * freq, and the scaled coordinates x' * freq of the map's edge cells, which bound
// those of every cell because rounding is monotone (numpy silently casts NaN or out-of-range values to garbage).
static int perlin_layer_check(const AntsPerlinLayer *L, int n, int W, int H, const char *what, ants::PerlinArgs *out) {
    if (!L->offsets) return fail(ANTS_E_ARG, "%s: NULL offsets", what);
    if (L->octaves < 1 || L->octaves > ants::kPerlinMaxOctaves)
        return fail(ANTS_E_ARG, "%s: octaves %d outside 1 ... %d", what, L->octaves, ants::kPerlinMaxOctaves);
    if (!std::isfinite(L->scale) || L->scale == 0.0) return fail(ANTS_E_ARG, "%s: scale %g", what, L->scale);
    const float pers = (float)L->persistence, lac = (float)L->lacunarity;
    if (!std::isfinite(pers) || !std::isfinite(lac))
        return fail(ANTS_E_ARG, "%s: persistence %g or lacunarity %g is not a finite float", what, L->persistence,
                    L->lacunarity);
    const float lim = 2147483648.f;                          // 2^31
    float freq[ants::kPerlinMaxOctaves];
    freq[0] = 1.f;
    for (int o = 0; o < L->octaves; ++o) {
        if (o > 0) freq[o] = freq[o - 1] * lac;
        const float rep = 1024.f * freq[o];
        if (!(std::fabs(rep) < lim) || rep == 0.f)
            return fail(ANTS_E_ARG, "%s: octave %d has the period %g (1024 * freq must be finite, non-zero, below 2^31)",
                        what, o + 1, (double)rep);
    }
    for (int e = 0; e < n; ++e)
        for (int c = 0; c < 4; ++c) {
            const int64_t cell = (c & 1) ? (c < 2 ? W : H) - 1 : 0;
            const float x = (float)((double)(cell + L->offsets[2 * e + (c >> 1)]) / L->scale);
            for (int o = 0; o < L->octaves; ++o) {
                const float xf = x * freq[o];
                if (!(std::fabs(xf) < lim))
                    return fail(ANTS_E_ARG, "%s: env %d, octave %d: the coordinate %g of a map edge is not finite or not "
                                "below 2^31", what, e, o + 1, (double)xf);
            }
        }
    out->offsets = nullptr;
    out->scale = L->scale;
    out->density = L->density;
    out->octaves = L->octaves;
    out->persistence = pers;
    out->lacunarity = lac;
    return ANTS_OK;
}

// ants_generate_env_maps and ants_generate_env_maps_ex (NULL Perlin layers: the former)
static int generate_env_maps(AntsBatch *b, int32_t env0, int32_t n_envs, const int32_t *anthill_xyr,
                             int32_t n_wall_discs, const int32_t *wall_discs, const AntsPerlinLayer *wall_perlin,
                             int32_t n_food_discs, const int32_t *food_discs, const AntsPerlinLayer *food_perlin) {
    if (!b || !anthill_xyr) return fail(ANTS_E_ARG, "null argument");
    Params &p = b->p;
    if (env0 < 0 || n_envs < 1 || (int64_t)env0 + n_envs > p.E)
        return fail(ANTS_E_ARG, "env window [%d, %d) outside the batch of %d envs", env0, env0 + n_envs, p.E);
    if (n_wall_discs < 0 || n_food_discs < 0) return fail(ANTS_E_ARG, "negative disc count");
    if ((n_wall_discs > 0 && !wall_discs) || (n_food_discs > 0 && !food_discs)) return fail(ANTS_E_ARG, "null disc array");
    if ((wall_perlin && n_wall_discs != 0) || (food_perlin && n_food_discs != 0))
        return fail(ANTS_E_ARG, "a layer given both discs and Perlin noise");
    for (int e = 0; e < n_envs; ++e)
        if (anthill_xyr[3 * e + 2] < 0) return fail(ANTS_E_ARG, "env %d: negative anthill radius", env0 + e);
    ants::ResetPerlin pl = {};
    if (wall_perlin) TRY(perlin_layer_check(wall_perlin, n_envs, p.W, p.H, "wall layer", &pl.wall));
    if (food_perlin) TRY(perlin_layer_check(food_perlin, n_envs, p.W, p.H, "food layer", &pl.food));
    // the discs of env e as (xc, yc, r, 0): its wall discs, then its food discs; each must lie inside the map
    const int K = n_wall_discs + n_food_discs;
    std::vector<int4> discs((size_t)n_envs * K);
    for (int e = 0; e < n_envs; ++e)
        for (int k = 0; k < K; ++k) {
            const int32_t *d = k < n_wall_discs ? wall_discs + ((size_t)e * n_wall_discs + k) * 3
                                                : food_discs + ((size_t)e * n_food_discs + (k - n_wall_discs)) * 3;
            if (d[2] < 0 || d[0] - d[2] < 0 || d[0] + d[2] >= p.W || d[1] - d[2] < 0 || d[1] + d[2] >= p.H)
                return fail(ANTS_E_ARG, "env %d: %s disc %d (%d, %d, r %d) does not lie inside the %d x %d map", env0 + e,
                            k < n_wall_discs ? "wall" : "food", k < n_wall_discs ? k : k - n_wall_discs, d[0], d[1], d[2],
                            p.W, p.H);
            discs[(size_t)e * K + k] = make_int4(d[0], d[1], d[2], 0);
        }
    // the offsets of the Perlin layers: the wall layer's n_envs pairs, then the food layer's
    std::vector<int2> offs;
    for (const AntsPerlinLayer *L : {wall_perlin, food_perlin})
        if (L)
            for (int e = 0; e < n_envs; ++e) offs.push_back(make_int2(L->offsets[2 * e], L->offsets[2 * e + 1]));
    CK(cudaSetDevice(b->cfg.device));
    cudaStream_t st = b->stream;
    const bool whole = n_envs == p.E;
    if ((int64_t)discs.size() > b->reset_cap) {
        CK(cudaStreamSynchronize(st));                      // (the old buffer may still be read by an earlier launch)
        if (b->reset_discs) { cudaFree(b->reset_discs); b->reset_discs = nullptr; b->reset_cap = 0; }
        cudaError_t me = cudaMalloc(&b->reset_discs, discs.size() * sizeof(int4));
        if (me != cudaSuccess) { b->reset_discs = nullptr; return fail(ANTS_E_ALLOC, "disc buffer: %s", cudaGetErrorString(me)); }
        b->reset_cap = (int64_t)discs.size();
    }
    if (!discs.empty())
        CK(cudaMemcpyAsync(b->reset_discs, discs.data(), discs.size() * sizeof(int4), cudaMemcpyHostToDevice, st));
    if ((int64_t)offs.size() > b->reset_offsets_cap) {
        CK(cudaStreamSynchronize(st));
        if (b->reset_offsets) { cudaFree(b->reset_offsets); b->reset_offsets = nullptr; b->reset_offsets_cap = 0; }
        cudaError_t me = cudaMalloc(&b->reset_offsets, offs.size() * sizeof(int2));
        if (me != cudaSuccess) { b->reset_offsets = nullptr; return fail(ANTS_E_ALLOC, "offset buffer: %s", cudaGetErrorString(me)); }
        b->reset_offsets_cap = (int64_t)offs.size();
    }
    if (!offs.empty()) {
        CK(cudaMemcpyAsync(b->reset_offsets, offs.data(), offs.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
        if (wall_perlin) pl.wall.offsets = b->reset_offsets;
        if (food_perlin) pl.food.offsets = b->reset_offsets + (wall_perlin ? n_envs : 0);
    }
    std::vector<int32_t> hill4((size_t)n_envs * 4);
    for (int e = 0; e < n_envs; ++e) {
        const int32_t r = anthill_xyr[3 * e + 2];
        hill4[4 * e] = anthill_xyr[3 * e]; hill4[4 * e + 1] = anthill_xyr[3 * e + 1];
        hill4[4 * e + 2] = r; hill4[4 * e + 3] = r * r;
    }
    CK(cudaMemcpyAsync(p.hill + (size_t)env0 * 4, hill4.data(), hill4.size() * 4, cudaMemcpyHostToDevice, st));
    ants::ResetArgs a;
    a.discs = b->reset_discs; a.kw = n_wall_discs; a.kf = n_food_discs; a.env0 = env0;
    a.tiles_x = (int)cdiv(p.Wp, ants::kResetTile); a.tiles_y = (int)cdiv(p.Hp, ants::kResetTile);
    const unsigned grid = (unsigned)((int64_t)n_envs * a.tiles_x * a.tiles_y);
    {
        LaunchScope ls(b, F_RESET);
        if (wall_perlin || food_perlin) {
            switch (p.rec_shift) {
                case 3: ants::k_reset_maps<8, true><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                case 4: ants::k_reset_maps<16, true><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                case 5: ants::k_reset_maps<32, true><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                default: ants::k_reset_maps<64, true><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
            }
        } else {
            switch (p.rec_shift) {
                case 3: ants::k_reset_maps<8><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                case 4: ants::k_reset_maps<16><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                case 5: ants::k_reset_maps<32><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
                default: ants::k_reset_maps<64><<<grid, ants::kResetThreads, 0, st>>>(p, a, pl); break;
            }
        }
    }
    TRY(check_launch("k_reset_maps"));
    if (p.tile_active)
        CK(cudaMemsetAsync(p.tile_active + (size_t)env0 * p.tiles_x * p.tiles_y, 0, (size_t)n_envs * p.tiles_x * p.tiles_y, st));
    // the same bookkeeping as an import of food, walls, explored, pheromones and the anthill (ants_import_env_state)
    if (p.owner) CK(cudaMemsetAsync(p.owner, 0, (size_t)p.E * p.plane * sizeof(uint32_t), st));
    if (b->fused) CK(cudaMemsetAsync(p.absorb_count + env0, 0, (size_t)n_envs * sizeof(uint32_t), st));
    else CK(cudaMemsetAsync(p.absorb_count, 0, 2 * sizeof(uint32_t), st));   // (the whole batch-wide queue, as above)
    b->needs_sweep = 1;                                     // food may lie inside the new anthill disc (Q10)
    b->move_done = 0;
    b->pack_disabled = 0;
    b->wall_flags_valid = 0;
    b->owner_phase = 0;
    if (whole) { b->obs_gen = 0; b->occ_gen = 0; }
    CK(cudaStreamSynchronize(st));   // host temporaries above must outlive the copies
    return ANTS_OK;
}

int ants_generate_env_maps(AntsBatch *b, int32_t env0, int32_t n_envs, const int32_t *anthill_xyr, int32_t n_wall_discs,
                           const int32_t *wall_discs, int32_t n_food_discs, const int32_t *food_discs) {
    return generate_env_maps(b, env0, n_envs, anthill_xyr, n_wall_discs, wall_discs, nullptr, n_food_discs, food_discs,
                             nullptr);
}

int ants_generate_env_maps_ex(AntsBatch *b, int32_t env0, int32_t n_envs, const int32_t *anthill_xyr,
                              int32_t n_wall_discs, const int32_t *wall_discs, const AntsPerlinLayer *wall_perlin,
                              int32_t n_food_discs, const int32_t *food_discs, const AntsPerlinLayer *food_perlin) {
    return generate_env_maps(b, env0, n_envs, anthill_xyr, n_wall_discs, wall_discs, wall_perlin, n_food_discs,
                             food_discs, food_perlin);
}

int ants_perlin_noise(int32_t device, const AntsPerlinLayer *layer, int32_t n, int32_t w, int32_t h, float *d_out,
                      void *stream) {
    if (!layer || !d_out) return fail(ANTS_E_ARG, "null argument");
    if (n < 1 || w < 1 || h < 1) return fail(ANTS_E_ARG, "empty field: n %d, w %d, h %d", n, w, h);
    ants::PerlinArgs L;
    TRY(perlin_layer_check(layer, n, w, h, "layer", &L));
    const int tiles_x = (int)cdiv(w, ants::kPerlinTile), tiles_y = (int)cdiv(h, ants::kPerlinTile);
    if ((int64_t)n * tiles_x * tiles_y > 0x7fffffff) return fail(ANTS_E_ARG, "field of %d x %d x %d too large", n, w, h);
    CK(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    Scratch off;
    CK(cudaMalloc(&off.ptr, (size_t)n * sizeof(int2)));
    CK(cudaMemcpyAsync(off.ptr, layer->offsets, (size_t)n * sizeof(int2), cudaMemcpyHostToDevice, st));
    L.offsets = (const int2 *)off.ptr;
    ants::k_perlin_field<<<(unsigned)((int64_t)n * tiles_x * tiles_y), ants::kPerlinThreads, 0, st>>>(
        L, w, h, tiles_y, tiles_x * tiles_y, d_out);
    TRY(check_launch("k_perlin_field"));
    CK(cudaStreamSynchronize(st));   // the offsets buffer is freed on return
    return ANTS_OK;
}

int ants_export_env_state(AntsBatch *b, int32_t env0, int32_t n_envs, AntsHostState *s) {
    if (!b || !s) return fail(ANTS_E_ARG, "null argument");
    Params &p = b->p;
    if (env0 < 0 || n_envs < 1 || (int64_t)env0 + n_envs > p.E)
        return fail(ANTS_E_ARG, "env window [%d, %d) outside the batch of %d envs", env0, env0 + n_envs, p.E);
    CK(cudaSetDevice(b->cfg.device));
    cudaStream_t st = b->stream;
    const size_t a0 = (size_t)env0 * p.N, an = (size_t)n_envs * p.N;      // the window's ants
    auto down = [&](double *dst, const double *src) -> cudaError_t {
        return dst ? cudaMemcpyAsync(dst, src + a0, an * sizeof(double), cudaMemcpyDeviceToHost, st) : cudaSuccess;
    };
    CK(down(s->x, p.x)); CK(down(s->y, p.y)); CK(down(s->theta, p.theta));
    CK(down(s->prev_x, p.prev_x)); CK(down(s->prev_y, p.prev_y)); CK(down(s->prev_theta, p.prev_theta));
    CK(down(s->holding, p.holding)); CK(down(s->seed, p.seed));
    CK(down(s->rw_holding_prev, p.rw_holding_prev)); CK(down(s->rw_prev_dist, p.rw_prev_dist));
    CK(down(s->rewards, p.rewards));
    if (s->mandibles) CK(cudaMemcpyAsync(s->mandibles, p.mandibles + a0, an, cudaMemcpyDeviceToHost, st));
    if (s->reward_state) CK(cudaMemcpyAsync(s->reward_state, p.reward_state + a0, an, cudaMemcpyDeviceToHost, st));
    std::vector<double> act_t;                                             // device layout [P][E*N]
    if (s->activation && p.P > 0) {
        act_t.resize(an * p.P);
        for (int k = 0; k < p.P; ++k)
            CK(cudaMemcpyAsync(act_t.data() + (size_t)k * an, p.act + (size_t)k * p.EN + a0, an * sizeof(double),
                               cudaMemcpyDeviceToHost, st));
    }
    // map fields: unpack kernel from the cell records -> device scratch -> dense host array
    const size_t ncell = (size_t)n_envs * p.W * p.H;
    Scratch scratch;
    if ((s->phero && p.P > 0) || s->food || s->walls || s->explored) {
        size_t need = ncell * 8 * ((s->phero && p.P > 1) ? p.P : 1);
        cudaError_t me = cudaMalloc(&scratch.ptr, need);
        if (me != cudaSuccess) return fail(ANTS_E_ALLOC, "export scratch of %zu bytes: %s", need, cudaGetErrorString(me));
    }
    void *const d_tmp = scratch.ptr;
    if (s->phero && p.P > 0) {
        for (int k = 0; k < p.P; ++k)
            ants::k_unpack_f64<<<148 * 8, 256, 0, st>>>(p, (double *)d_tmp, p.P, k, 8 * k, k, b->lazy_now, b->lazy_abs, env0, n_envs);
        TRY(check_launch("k_unpack_f64"));
        CK(cudaMemcpyAsync(s->phero, d_tmp, ncell * 8 * p.P, cudaMemcpyDeviceToHost, st));
    }
    if (s->food) {
        ants::k_unpack_f64<<<148 * 8, 256, 0, st>>>(p, (double *)d_tmp, 1, 0, p.food_off, -1, 0u, 0u, env0, n_envs);
        TRY(check_launch("k_unpack_f64"));
        CK(cudaMemcpyAsync(s->food, d_tmp, ncell * 8, cudaMemcpyDeviceToHost, st));
    }
    if (s->walls) {
        ants::k_unpack_u8<<<148 * 8, 256, 0, st>>>(p, (uint8_t *)d_tmp, 0, env0, n_envs);
        TRY(check_launch("k_unpack_u8"));
        CK(cudaMemcpyAsync(s->walls, d_tmp, ncell, cudaMemcpyDeviceToHost, st));
    }
    if (s->explored) {
        ants::k_unpack_u8<<<148 * 8, 256, 0, st>>>(p, (uint8_t *)d_tmp, 1, env0, n_envs);
        TRY(check_launch("k_unpack_u8"));
        CK(cudaMemcpyAsync(s->explored, d_tmp, ncell, cudaMemcpyDeviceToHost, st));
    }
    std::vector<int32_t> hill4;
    if (s->anthill_xyr) {
        hill4.resize((size_t)n_envs * 4);
        CK(cudaMemcpyAsync(hill4.data(), p.hill + (size_t)env0 * 4, hill4.size() * 4, cudaMemcpyDeviceToHost, st));
    }
    if (s->anthill_food) CK(cudaMemcpyAsync(s->anthill_food, p.hill_food + env0, (size_t)n_envs * 8, cudaMemcpyDeviceToHost, st));
    if (p.R > 0) {
        const size_t r0 = (size_t)env0 * p.R, rn = (size_t)n_envs * p.R;
        if (s->rock_centers) CK(cudaMemcpyAsync(s->rock_centers, p.rock_c + r0 * 2, rn * 16, cudaMemcpyDeviceToHost, st));
        if (s->rock_radii) CK(cudaMemcpyAsync(s->rock_radii, p.rock_rad + r0, rn * 8, cudaMemcpyDeviceToHost, st));
        if (s->rock_weights) CK(cudaMemcpyAsync(s->rock_weights, p.rock_w + r0, rn * 8, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    if (s->activation && p.P > 0)
        for (size_t i = 0; i < an; ++i)
            for (int k = 0; k < p.P; ++k) s->activation[i * p.P + k] = act_t[(size_t)k * an + i];
    if (s->anthill_xyr)
        for (int e = 0; e < n_envs; ++e) {
            s->anthill_xyr[3 * e] = hill4[4 * e]; s->anthill_xyr[3 * e + 1] = hill4[4 * e + 1];
            s->anthill_xyr[3 * e + 2] = hill4[4 * e + 2];
        }
    s->timestep = b->timestep;
    s->rw_alias = b->rw_alias;
    s->act_bool = b->act_bool;
    return ANTS_OK;
}

int ants_export_state(AntsBatch *b, AntsHostState *s) {
    if (!b) return fail(ANTS_E_ARG, "null argument");
    return ants_export_env_state(b, 0, b->p.E, s);
}

int ants_activate_all_pheromones(AntsBatch *b, const double *act, int32_t is_bool) {
    if (!b || !act) return fail(ANTS_E_ARG, "null argument");
    CK(cudaSetDevice(b->cfg.device));
    Params &p = b->p;
    if (p.P == 0) return ANTS_OK;
    std::vector<double> act_t((size_t)p.EN * p.P);
    for (int64_t i = 0; i < p.EN; ++i)
        for (int k = 0; k < p.P; ++k) {
            double v = act[i * p.P + k];
            if (!is_bool && !std::isfinite(v))         // (bool activations map NaN to 1, as numpy's astype(bool))
                return fail(ANTS_E_ARG, "env %d, ant %d: activation %g; activations must be finite", (int)(i / p.N),
                            (int)(i % p.N), v);
            if (p.diffuse && !is_bool && !(v >= 0.0))  // a plane value's sign bit is the wall flag: no negative deposits
                return fail(ANTS_E_ARG, "env %d, ant %d: activation %g; with diffusion an activation must be >= 0",
                            (int)(i / p.N), (int)(i % p.N), v);
            act_t[(size_t)k * p.EN + i] = is_bool ? (v != 0.0 ? 1.0 : 0.0) : v;
        }
    CK(cudaMemcpyAsync(p.act, act_t.data(), act_t.size() * sizeof(double), cudaMemcpyHostToDevice, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    b->act_bool = is_bool ? 1 : 0;
    return ANTS_OK;
}

int ants_observe(AntsBatch *b, float *d_obs, float *d_agent_state, float *d_state, double *d_reward) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    return do_observe(b, d_obs, d_agent_state, d_state, d_reward);
}

int ants_step(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph, float *d_obs, float *d_agent_state,
              double *d_reward, int32_t *done) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    return do_step(b, d_rot, d_ph, d_obs, d_agent_state, d_reward, done);
}

int ants_update(AntsBatch *b, const double *d_noise) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    return do_update(b, d_noise);
}

int ants_rollout(AntsBatch *b, const int8_t *d_rot_tape, const int8_t *d_ph_tape, int32_t n_steps, float *d_obs,
                 float *d_agent_state, double *d_reward) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    const int64_t EN = b->p.EN;
    if (n_steps <= 0) return ANTS_OK;
    if (!d_obs || !d_agent_state) return fail(ANTS_E_ARG, "ants_rollout: obs and agent_state buffers are required");
    if (d_ph_tape && b->p.P != 2)
        return fail(ANTS_E_ARG, "pheromone actions need exactly two pheromones (ants.py:92-96), have %d", b->p.P);
    // Groups of environments on streams of their own for large batches on the block-per-env kernels
    // (ANTS_ROLLOUT_GROUPS overrides: 1 = off).  The step kernels launch once per group; host bookkeeping (generation
    // counters, lazy-field counters, timestep) advances once per step for the whole batch, and the rare whole-batch
    // passes (folds, the anthill sweep after an import) join the groups first.  Groups share no state: the results are
    // those of the plain loop.
    int want = (b->fused && b->perceive_rows && EN >= 131072) ? 4 : 1;
    if (const char *x = getenv("ANTS_ROLLOUT_GROUPS")) want = atoi(x);
    if (want > 1 && b->fused && b->perceive_rows && !b->profiling) {
        TRY(ensure_groups(b, want));
        b->grouped = b->groups.size() > 1 ? 1 : 0;
        if (b->grouped) fork_groups(b);
    }
    int rc = ANTS_OK;
    for (int t = 0; t < n_steps && rc == ANTS_OK; ++t) {
        const int8_t *r = d_rot_tape ? d_rot_tape + (int64_t)t * EN : nullptr;
        const int8_t *h = d_ph_tape ? d_ph_tape + (int64_t)t * EN : nullptr;
        rc = do_step(b, r, h, d_obs, d_agent_state, d_reward, nullptr);
        if (rc != ANTS_OK) break;
        // update_t and the move of step_{t+1} in one launch; do_step(t + 1) then only perceives
        if (b->fused && t + 1 < n_steps && !b->needs_sweep)
            rc = do_update_move_fused(b, d_rot_tape ? r + EN : nullptr, d_ph_tape ? h + EN : nullptr);
        else
            rc = do_update(b, nullptr);
    }
    if (b->grouped) join_groups(b);
    b->grouped = 0;
    return rc;
}

int ants_sample_actions(AntsBatch *b, uint64_t seed, int32_t n_rotations, int32_t n_pheromones, int8_t *d_rot,
                        int8_t *d_ph) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    if (n_rotations < 1 || n_rotations > 127 || n_pheromones < 1 || n_pheromones > 127)
        return fail(ANTS_E_ARG, "ants_sample_actions: action counts must be in 1..127");
    CK(cudaSetDevice(b->cfg.device));
    const Params &p = b->p;
    ants::k_sample_actions<<<(unsigned)cdiv(p.EN, 256), 256, 0, b->stream>>>(p, seed, (uint32_t)b->timestep, n_rotations,
                                                                             n_pheromones, d_rot, d_ph);
    b->stats.kernel_launches++;
    return check_launch("k_sample_actions");
}

void *ants_host_alloc(uint64_t bytes) {
    void *ptr = nullptr;
    if (cudaHostAlloc(&ptr, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        fail(ANTS_E_ALLOC, "cudaHostAlloc of %llu bytes failed", (unsigned long long)bytes);
        cudaGetLastError();
        return nullptr;
    }
    return ptr;
}

int ants_host_free(void *ptr) {
    if (ptr) CK(cudaFreeHost(ptr));
    return ANTS_OK;
}

int ants_observe_host(AntsBatch *b, float *h_obs, float *h_agent_state, float *h_state, double *h_reward) {
    if (!b || !h_obs || !h_agent_state) return fail(ANTS_E_ARG, "null argument");
    CK(cudaSetDevice(b->cfg.device));
    TRY(ensure_staging(b));
    const Params &p = b->p;
    TRY(do_observe(b, b->st_obs, b->st_as, h_state ? b->st_state : nullptr, b->st_reward));
    CK(cudaMemcpyAsync(h_obs, b->st_obs, (size_t)p.EN * p.S2 * p.C * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(h_agent_state, b->st_as, (size_t)p.EN * 8, cudaMemcpyDeviceToHost, b->stream));
    if (h_state) CK(cudaMemcpyAsync(h_state, b->st_state, (size_t)p.EN * (2 + p.P) * 4, cudaMemcpyDeviceToHost, b->stream));
    if (h_reward) CK(cudaMemcpyAsync(h_reward, b->st_reward, (size_t)p.EN * 8, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return ANTS_OK;
}

int ants_step_host(AntsBatch *b, const int8_t *h_rot, const int8_t *h_ph, float *h_obs, float *h_agent_state,
                   double *h_reward, int32_t *done) {
    if (!b || !h_obs || !h_agent_state) return fail(ANTS_E_ARG, "null argument");
    CK(cudaSetDevice(b->cfg.device));
    TRY(ensure_staging(b));
    const Params &p = b->p;
    if (h_rot) CK(cudaMemcpyAsync(b->st_rot, h_rot, (size_t)p.EN, cudaMemcpyHostToDevice, b->stream));
    if (h_ph) CK(cudaMemcpyAsync(b->st_ph, h_ph, (size_t)p.EN, cudaMemcpyHostToDevice, b->stream));
    TRY(do_step(b, h_rot ? b->st_rot : nullptr, h_ph ? b->st_ph : nullptr, b->st_obs, b->st_as, b->st_reward, done));
    if (packed_path_wanted(b)) {
        // the observation crosses PCIe packed (visible samples, 12 bytes each) and is expanded by the host threads
        TRY(ensure_packed(b));
        const int rc = packed_transfer(b, b->h_packed, h_obs, h_agent_state, h_reward);
        if (rc == ANTS_OK) return ANTS_OK;
        if (rc != 1) return rc;
        b->pack_disabled = 1;              // e.g. a non-integer amount of food: this and the following steps go dense
    }
    CK(cudaMemcpyAsync(h_obs, b->st_obs, (size_t)p.EN * p.S2 * p.C * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(h_agent_state, b->st_as, (size_t)p.EN * 8, cudaMemcpyDeviceToHost, b->stream));
    if (h_reward) CK(cudaMemcpyAsync(h_reward, b->st_reward, (size_t)p.EN * 8, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return ANTS_OK;
}

int ants_packed_layout(const AntsConfig *cfg, AntsPackedLayout *out) {
    if (!cfg || !out) return fail(ANTS_E_ARG, "null argument");
    if (cfg->radius < 0 || cfg->radius > ANTS_MAX_RADIUS || cfg->n_channels < 1 || cfg->n_channels > ANTS_MAX_CHANNELS)
        return fail(ANTS_E_ARG, "radius / n_channels out of range");
    packed_layout_of(cfg, out);
    return ANTS_OK;
}

int ants_step_host_packed(AntsBatch *b, const int8_t *h_rot, const int8_t *h_ph, void *h_packed, float *h_agent_state,
                          double *h_reward, int32_t *done) {
    if (!b || !h_packed || !h_agent_state) return fail(ANTS_E_ARG, "null argument");
    if (!b->pack_layout.supported) return fail(ANTS_E_ARG, "this configuration has no packed observation form");
    CK(cudaSetDevice(b->cfg.device));
    TRY(ensure_staging(b));
    TRY(ensure_packed(b));
    const Params &p = b->p;
    if (h_rot) CK(cudaMemcpyAsync(b->st_rot, h_rot, (size_t)p.EN, cudaMemcpyHostToDevice, b->stream));
    if (h_ph) CK(cudaMemcpyAsync(b->st_ph, h_ph, (size_t)p.EN, cudaMemcpyHostToDevice, b->stream));
    TRY(do_step(b, h_rot ? b->st_rot : nullptr, h_ph ? b->st_ph : nullptr, b->st_obs, b->st_as, b->st_reward, done));
    const int rc = packed_transfer(b, (uint8_t *)h_packed, nullptr, h_agent_state, h_reward);
    if (rc == 1)
        return fail(ANTS_E_STATE, "an observation value of this step has no packed form (non-integer food): the step was "
                                  "taken; read it with ants_observe-style dense copies (ants_step_host)");
    return rc;
}

int ants_unpack_obs(const AntsPackedLayout *layout, const void *h_packed, int64_t n_ants, float *h_obs, int32_t n_threads) {
    if (!layout || !h_packed || !h_obs || n_ants < 0) return fail(ANTS_E_ARG, "null argument");
    if (!layout->supported) return fail(ANTS_E_ARG, "unsupported packed layout");
    AntsUnpackPlan *plan = new AntsUnpackPlan();
    unpack_plan_of(layout, plan);
    const int64_t bpa = layout->bytes_per_ant, dense = (int64_t)layout->n_samples * layout->n_channels;
    const uint8_t *src = (const uint8_t *)h_packed;
    if (n_threads == 1 || n_ants < 1024) {
        ants_unpack_range(plan, src, n_ants, h_obs);
    } else {
        HostPool &pool = HostPool::get();
        int T = n_threads <= 0 ? pool.size() : (n_threads < pool.size() ? n_threads : pool.size());
        const int64_t piece = cdiv(n_ants, (int64_t)T * 4);
        for (int64_t s0 = 0; s0 < n_ants; s0 += piece) {
            const int64_t cnt = n_ants - s0 < piece ? n_ants - s0 : piece;
            pool.submit([=] { ants_unpack_range(plan, src + s0 * bpa, cnt, h_obs + s0 * dense); });
        }
        pool.wait_idle();
    }
    delete plan;
    return ANTS_OK;
}

int ants_update_host(AntsBatch *b, const double *h_noise) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    CK(cudaSetDevice(b->cfg.device));
    if (h_noise) {
        TRY(ensure_staging(b));
        CK(cudaMemcpyAsync(b->st_noise, h_noise, (size_t)b->p.EN * 8, cudaMemcpyHostToDevice, b->stream));
        TRY(do_update(b, b->st_noise));
        CK(cudaStreamSynchronize(b->stream));   // the caller may reuse h_noise
        return ANTS_OK;
    }
    return do_update(b, nullptr);
}

int ants_get_stats(AntsBatch *b, AntsStats *out) {
    if (!b || !out) return fail(ANTS_E_ARG, "null argument");
    CK(cudaSetDevice(b->cfg.device));
    CK(cudaMemcpyAsync(b->h_counts, b->p.commit_count + (b->commit_par ^ 1), 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(b->h_counts + 1, b->p.absorb_count + b->absorb_par, 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(b->h_counts + 2, b->p.tile_counter, 8, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    b->stats.food_commits = b->fused ? 0 : b->h_counts[0];     // (counted by the flat kernels only)
    b->stats.absorb_events = b->fused ? 0 : b->h_counts[1];
    if (b->p.tile_active) {
        unsigned long long t;
        memcpy(&t, b->h_counts + 2, 8);
        b->stats.active_tiles = (int64_t)t;
    } else {
        b->stats.active_tiles = b->stats.total_tiles;
    }
    b->stats.device_bytes = b->device_bytes;
    b->stats.e2e_dense_permille = (int64_t)(b->dense_frac * 1000.0 + 0.5);
    *out = b->stats;
    return ANTS_OK;
}

int ants_set_profiling(AntsBatch *b, int32_t on) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    TRY(collect_timings(b));
    b->profiling = on ? 1 : 0;
    return ANTS_OK;
}

int ants_get_kernel_ms(AntsBatch *b, const char *name, double *ms, int64_t *launches) {
    if (!b || !name) return fail(ANTS_E_ARG, "null argument");
    TRY(collect_timings(b));
    for (int f = 0; f < F_COUNT; ++f)
        if (strcmp(name, kFamName[f]) == 0) {
            if (ms) *ms = b->fam_ms[f];
            if (launches) *launches = b->fam_launches[f];
            return ANTS_OK;
        }
    return fail(ANTS_E_ARG, "unknown kernel family '%s'", name);
}

int ants_reset_kernel_ms(AntsBatch *b) {
    if (!b) return fail(ANTS_E_ARG, "null handle");
    TRY(collect_timings(b));
    memset(b->fam_ms, 0, sizeof b->fam_ms);
    memset(b->fam_launches, 0, sizeof b->fam_launches);
    return ANTS_OK;
}

}  // extern "C"
