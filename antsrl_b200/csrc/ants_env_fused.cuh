// ants_env_fused.cuh -- the per-ant kernels of the step loop fused into ONE kernel whose blocks own whole environments.
//
// The flat kernels (k_step_move, k_food_commit, k_collide, k_rocks_pushed, k_rocks_push_ants, k_deposit_commit in
// ants_kernels.cuh) split the iteration wherever "all ants of an environment have finished phase k" is needed -- the
// last-writer scatters of the reference (quirk Q1: ants.py:116, pheromone.py:39), the ordered sum of the ants' pushes
// on a rock (circle_obstacles.py:38-40) -- and resolve the scatters through a global `owner` array (atomicMax per ant,
// re-read by a follow-up kernel: two random DRAM sectors per ant and scatter).  Here a block owns G consecutive
// environments (G * N <= CAP ants, CAP in {256, 512, 1024}: 256 or 512 threads with one ant each, or 512 threads with
// two for the 1024-ant block), so those phase boundaries are block barriers, the owner of a cell is found in a
// shared-memory hash table (cell -> highest ant index, atomicCAS / atomicMax on shared memory) and the rock pushes are
// summed from positions staged in shared memory.  Per iteration of `update(); step()` the ants' state is read and
// written once, and the record of the cell an ant stands on is loaded once for the pheromone deposit (update) AND the
// mandible rule of the next step (RL_api.py:178-185: after an update prev_ants == ants, so it is the same cell and the
// same winner).
//
//   k_env<UPDATE, MOVE, APT, TPB>:
//     UPDATE: Environment.update() (environment.py:42-47) for lazy-evaporation handles: Anthill absorb of the cells
//             queued by the previous move (anthill.py:41-46), Walls.update on ants (walls.py:24-28),
//             CircleObstacles.update (circle_obstacles.py:32-58), the ant part of Ants.update (ants.py:123-130) and
//             the pheromone deposit with its clamp (pheromone.py:36-41)
//     MOVE:   RLApi.step lines 178-196 (mandible rule, food pickup / drop with its last-writer scatter, pheromone
//             activation, rotate, forward on the torus) + occupancy stamp + wall flag of the new cell
//   <1,0> = ants_update, <0,1> = first half of ants_step, <1,1> = update_k ; step_{k+1} inside ants_rollout.
// Used when the field is lazy (or there are no pheromones), N <= 1024 and the keys fit 32 bits; everything else keeps
// the flat kernels (ANTS_NO_FUSED forces them, for A/B tests).
//
// Measured on the cfg4 shard (512 envs x 1024 ants, 8-byte records, one B200) and left out of the code again:
//   * the 1024-ant block as 256 threads x 4 ants or 1024 x 1: 0.111 and 0.098 ms against 0.090 for 512 x 2;
//   * update+move: the move ahead of the mandible rule, again where the holding changes: 0.111 against 0.098 ms;
//   * the move's occupancy stamp as a store without a load, the wall bit read by the update: 0.117 against 0.101 ms;
//   * the per-ant helpers (wrap, sincos, food load, deposit) called instead of inlined: 0.103 against 0.098 ms.
#pragma once

namespace ants {

constexpr int kEnvThreads = 256;
constexpr int kEnvMaxGroup = 32;             // environments per block (rock-touch words in shared memory: G * R)

struct EnvArgs {
    const int8_t *rot, *ph;                  // MOVE: actions [E][N] or NULL (RL_api.py:187,190)
    const double *noise;                     // UPDATE: collision noise tape [E][N] or NULL (Philox)
    uint32_t step_id;                        // UPDATE: Environment.timestep before the increment (Philox counter)
    uint32_t occ_gen;                        // MOVE: occupancy generation of this step
    int32_t all_stamp;                       // MOVE alone: prev_ants may differ from ants (two steps without an update)
    int32_t use_flag;                        // UPDATE: wall_hit[] was written by the preceding move
    double act_on;                           // MOVE: 256 (float activations) or 1 (bool dtype, ants.py:83)
    uint32_t now, now_abs;                   // UPDATE: lazy-field counters of this update (deposit timestamps)
    int32_t group, cap;                      // envs per block, ants per block
    int32_t env_base, env_end;               // the envs [env_base, env_end) of the batch (ants_rollout: groups on own streams)
};

__device__ __forceinline__ uint32_t env_hash_slot(uint32_t key, uint32_t mask) { return (key * 2654435761u >> 11) & mask; }
// cell -> highest (ant index + 1) among the inserting ants
__device__ __forceinline__ void env_hash_max(uint32_t *keys, uint32_t *vals, uint32_t mask, uint32_t key, uint32_t val) {
    uint32_t h = env_hash_slot(key, mask);
    while (true) {
        const uint32_t k = atomicCAS(&keys[h], 0u, key);
        if (k == 0u || k == key) { atomicMax(&vals[h], val); return; }
        h = (h + 1u) & mask;
    }
}
__device__ __forceinline__ uint32_t env_hash_get(const uint32_t *keys, const uint32_t *vals, uint32_t mask, uint32_t key) {
    uint32_t h = env_hash_slot(key, mask);
    while (true) {
        const uint32_t k = keys[h];
        if (k == key) return vals[h];
        if (k == 0u) return 0u;
        h = (h + 1u) & mask;
    }
}

// Anthill.update for one cell: qte -= qte * area, food += gain (anthill.py:44-46).  Atomic: a cell can sit in the queue
// twice when several steps ran without an update.
__device__ __forceinline__ void env_absorb_cell(const Params &p, int e, int cell) {
    uint8_t *fr = rec_at(p, e, cell);
    double v;
    if (p.rec8) {              // the food code is the low half of the record's second word
        const uint32_t c = atomicAnd(reinterpret_cast<unsigned int *>(fr + 4), 0xFFFF0000u) & 0xFFFFu;
        v = c != kFoodEsc ? (double)c : (double)p.side_val[rec8_index(p, fr) * 3 + 2];
    } else if (p.rec16) v = (double)__uint_as_float(atomicExch(reinterpret_cast<unsigned int *>(fr + 8), 0u));
    else v = __longlong_as_double((long long)atomicExch(reinterpret_cast<unsigned long long *>(fr + p.food_off), 0ull));
    if (v != 0.0) atomicAdd(p.hill_food + e, v);
}

__device__ __forceinline__ void prefetch_l2(const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }

// Heavy or rare pieces of the per-ant work are kept out of line: the kernel body is unrolled over the ants of a thread,
// and inlining them four times made it 12 000 instructions (ncu: 2.5 stall cycles per instruction waiting for the
// instruction cache).
__device__ __noinline__ double env_noise(const Params &p, int e, uint32_t step_id, int ant) {
    return philox_uniform(p.rng_seed, (uint32_t)(p.env_id_base + e), step_id, (uint32_t)ant);
}
// the owner of a cell adds its activations and clamps (ants.py:98-100, pheromone.py:36-41)
__device__ __forceinline__ void env_deposit(const Params &p, uint8_t *rec, int64_t i, uint32_t now, uint32_t now_abs, double av0, double av1) {
    for (int q = 0; q < p.P; ++q) {
        const double av = q == 0 ? av0 : (q == 1 ? av1 : p.act[(int64_t)q * p.EN + i]);   // (the first two were loaded with the ant state)
        if (av == 0.0) continue;
        double v = phero_value(p, rec, q, now, now_abs) + av;                           // (evaporated up to this update)
        if (p.has_max_val) v = fmin(v, p.phero_max_val);
        phero_store(p, rec, q, v, now, now_abs);
    }
}
// the owner writes the food of its cell (ants.py:116); returns what is stored (f32 in compact records)
__device__ __noinline__ double env_food_commit(const Params &p, uint8_t *fr, double v) {
    st_food(p, fr, v);
    return ld_food(p, fr);
}

// the rock-grid entries follow a rock that moved (clear the old box, set the new one); a whole warp calls this
__device__ __noinline__ void env_move_rock_grid(const Params &p, int e, int r, double cx, double cy, double nx, double ny, double rad, int lane) {
    rock_grid_mark_warp(p, e, r, cx, cy, rad, false, lane);
    __syncwarp();                                      // orders the clears before the sets (the boxes overlap)
    rock_grid_mark_warp(p, e, r, nx, ny, rad, true, lane);
}
// rock-grid word of an ant position (positions of the step loop lie in [0, W] x [0, H]: ants.py:69-71; W itself is
// quirk Q14 and maps to cell 0 like everywhere else)
__device__ __forceinline__ const unsigned long long *env_grid_word(const Params &p, int e, double x, double y) {
    int gx = cell_of(x, p.W) >> kGridShift, gy = cell_of(y, p.H) >> kGridShift;
    gx = min(max(gx, 0), p.grid_w - 1); gy = min(max(gy, 0), p.grid_h - 1);
    return p.rock_grid + ((int64_t)e * p.grid_w + gx) * p.grid_h + gy;
}

// which of the candidate rocks does an ant standing at (x, y) push (circle_obstacles.py:35-37)?  Out of line: one copy of
// the f64 square roots instead of one per unrolled ant.
__device__ __noinline__ void env_touch_rocks(const Params &p, int e, double x, double y, unsigned long long rm, uint32_t *touch_row,
                                             uint32_t chunk_bit) {
    const double *rc = p.rock_c + (int64_t)e * p.R * 2;
    const double *rr = p.rock_rad + (int64_t)e * p.R;
    while (rm) {
        const int r = __ffsll((long long)rm) - 1;
        rm &= rm - 1;
        const double vx = rc[2 * r] - x, vy = rc[2 * r + 1] - y;
        if (!(sqrt(vx * vx + vy * vy) > rr[r])) atomicOr(&touch_row[r], chunk_bit);
    }
}
// rocks push the ant (circle_obstacles.py:53-58): candidates in rock order like np.sum(axis=1); the centres were just
// rewritten by this block, so they are read past the L1
__device__ __noinline__ void env_push_by_rocks(const Params &p, int e, unsigned long long rm, double *x, double *y) {
    const double *rc = p.rock_c + (int64_t)e * p.R * 2;
    const double *rr = p.rock_rad + (int64_t)e * p.R;
    double sx = 0.0, sy = 0.0;
    while (rm) {
        const int r = __ffsll((long long)rm) - 1;
        rm &= rm - 1;
        const double vx = __ldcg(rc + 2 * r) - *x, vy = __ldcg(rc + 2 * r + 1) - *y;
        const double d = sqrt(vx * vx + vy * vy);
        const double rad = rr[r];
        if (!(d > rad)) {
            const double fac = 1.0 - rad / (d + 0.001);
            sx += vx * fac; sy += vy * fac;
        }
    }
    *x = pymod_near(*x + sx, (double)p.W);                             // translate_ants -> warp_xy
    *y = pymod_near(*y + sy, (double)p.H);
}

constexpr int kEnvMinBlocks = 4;   // resident 256-thread blocks per SM at 64 registers
template <bool UPDATE, bool MOVE, int APT, int TPB>
__global__ void __launch_bounds__(TPB, (kEnvMinBlocks * kEnvThreads) / TPB)
k_env(const __grid_constant__ Params p, const EnvArgs a) {
    pdl_begin();
    constexpr int CAP = APT * TPB;
    extern __shared__ __align__(16) unsigned char env_smem[];
    double *xs = reinterpret_cast<double *>(env_smem);                 // [CAP] positions between the phases
    double *ys = xs + CAP;
    uint32_t *hkeys = reinterpret_cast<uint32_t *>(ys + CAP);          // [2 CAP]
    uint32_t *hvals = hkeys + 2 * CAP;                                 // [2 CAP]
    uint32_t *touch = hvals + 2 * CAP;                                 // [group * R] ant-chunks touching a rock
    constexpr uint32_t HMASK = 2u * CAP - 1u;

    const int tid = threadIdx.x;
    const int env0 = a.env_base + blockIdx.x * a.group;
    const int n_env = min(a.group, a.env_end - env0);
    const int n_loc = n_env * p.N;                                     // ants of this block
    const int64_t i0 = (int64_t)env0 * p.N;
    const int W = p.W, H = p.H;
    const double Wd = (double)W, Hd = (double)H;

    // The mandible rule (RL_api.py:180-184, quirk Q5) walks perceived_objects: food ORs (food > 0) into the mandibles,
    // the anthill ANDs (not in hill).  Both are idempotent, so only the last rule and whether the other kind precedes it
    // matter: 0 none, 1 OR, 2 AND, 3 (m | f) & !h, 4 (m & !h) | f.
    int rule_mode = 0;
    if (MOVE) {
        bool seen_or = false, seen_and = false;
        for (int q = 0; q < p.rule_n; ++q) {
            if (p.rule_op[q] == 0) { seen_or = true; rule_mode = seen_and ? 4 : 1; }
            else { seen_and = true; rule_mode = seen_or ? 3 : 2; }
        }
    }
    for (int k = tid; k < 2 * CAP; k += TPB) { hkeys[k] = 0u; hvals[k] = 0u; }
    if (UPDATE && p.R > 0)
        for (int k = tid; k < n_env * p.R; k += TPB) touch[k] = 0u;

    // Per-ant values that live across the barriers (unrolled: registers).  Loads of the APT ants of a thread are issued
    // together, with the index of an idle slot clamped to the block's last ant: the kernel lives on memory-level
    // parallelism (two random DRAM sectors per ant: the cell it deposits on and the cell it moves to).
    double th[APT];
    int newcell[APT];              // MOVE: the cell the ant moves to
    int cell[APT];                 // UPDATE: the cell the ant ends the update in; MOVE alone: its prev cell
    int el[APT];                   // environment within the block
    int lac[APT];                  // the ant's slot in the block (clamped)
    bool valid[APT];
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        const int la = tid + k * TPB;
        valid[k] = la < n_loc;
        lac[k] = valid[k] ? la : (n_loc - 1);
        el[k] = a.group == 1 ? 0 : lac[k] / p.N;
        th[k] = 0.0; cell[k] = 0; newcell[k] = 0;
    }
    // record of cell c of the block's env g: (g * plane + c) fits 32 bits (the hash keys rely on the same bound)
    uint8_t *const cells0 = p.cells + (((int64_t)env0 * p.plane) << p.rec_shift);
    const uint32_t plane32 = (uint32_t)p.plane;
    const int rshift = p.rec_shift;
    auto rec_of = [&](int g, int c) -> uint8_t * { return cells0 + ((size_t)((uint32_t)g * plane32 + (uint32_t)c) << rshift); };

    if (UPDATE) {
        // the ants' positions and wall flags are requested before the absorb pass (which does not touch them): its queue
        // counter is a round trip of its own, and nothing behind its barrier and stores would be moved up by the compiler
        double x[APT], y[APT];
        bool in_wall[APT];
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            const int64_t i = i0 + lac[k];
            x[k] = p.x[i]; y[k] = p.y[i]; th[k] = p.theta[i];
            in_wall[k] = a.use_flag ? p.wall_hit[i] != 0 : false;
            // what the later phases read, requested now (no registers held): the activations of the depositing owners,
            // the ant state of the move
            if (p.P > 0) { prefetch_l2(p.act + i); if (p.P > 1) prefetch_l2(p.act + p.EN + i); }
            prefetch_l2(p.reward_state + i);
            if (MOVE) { prefetch_l2(p.holding + i); prefetch_l2(p.mandibles + i); if (a.rot != nullptr) prefetch_l2(a.rot + i); }
        }
        // ---- Anthill.update (anthill.py:41-46) for the cells queued by the previous move: nothing else in the update
        //      reads the food field
        for (int g = 0; g < n_env; ++g) {
            const int e = env0 + g;
            const uint32_t cnt = p.absorb_count[e];
            if (cnt == 0u) continue;
            if (cnt <= (uint32_t)p.N) {
                for (uint32_t k = tid; k < cnt; k += TPB) env_absorb_cell(p, e, (int)p.absorb_list[(int64_t)e * p.N + k]);
            } else {
                // more cells were queued than the env's segment holds (several steps without an update): sweep the disc
                const int32_t *hl = p.hill + 4 * e;
                const int r = hl[2];
                const int x0 = max(hl[0] - r, 0), x1 = min(hl[0] + r, W - 1), y0 = max(hl[1] - r, 0), y1 = min(hl[1] + r, H - 1);
                const int bw = x1 - x0 + 1, bh = y1 - y0 + 1;
                if (bw > 0 && bh > 0)
                    for (int t = tid; t < bw * bh; t += TPB) {
                        const int cx = x0 + t / bh, cy = y0 + t % bh;
                        if (in_hill(hl, cx, cy)) env_absorb_cell(p, e, cidx(p, cx, cy));
                    }
            }
        }
        __syncthreads();
        if (tid < n_env) p.absorb_count[env0 + tid] = 0u;
        // ---- Walls.update on ants (walls.py:24-28) + which rocks does an ant push (circle_obstacles.py:35-37)
        const int Gc = ((p.N + 31) / 32 + 31) / 32 * 32;               // ants per touch chunk (<= 32 chunks)
        // Walls.update (walls.py:24-25): the wall bit of the cell the ant stands on, left in wall_hit[] by the move of
        // the previous step; without such a move (an update after an import or another update) read from the record
        if (!a.use_flag) {
#pragma unroll
            for (int k = 0; k < APT; ++k)
                in_wall[k] = ld_wall(p, rec_of(el[k], cidx(p, cell_of(x[k], W), cell_of(y[k], H))));
        }
        unsigned long long rm[APT];
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            const int64_t i = i0 + lac[k];
            const int e = env0 + el[k], ant = lac[k] - el[k] * p.N;
            if (in_wall[k]) {
                x[k] = p.prev_x[i]; y[k] = p.prev_y[i];
                const double u = a.noise ? a.noise[i] : env_noise(p, e, a.step_id, ant);
                th[k] += u - 0.5;                                      // not re-wrapped (Q3)
            }
            rm[k] = p.R > 0 ? *env_grid_word(p, e, x[k], y[k]) : 0ull;
        }
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            if (!valid[k]) continue;
            xs[lac[k]] = x[k]; ys[lac[k]] = y[k];
            if (rm[k]) {
                const int ant = lac[k] - el[k] * p.N;
                env_touch_rocks(p, env0 + el[k], x[k], y[k], rm[k], touch + el[k] * p.R, 1u << (ant / Gc));
            }
        }
        if (p.R > 0) {
            __syncthreads();
            // ---- ants push rocks (circle_obstacles.py:38-40): a warp per touched (env, rock) sums the pushes of the
            //      touched ant-chunks in ant order (= np.sum(axis=0); untouched ants add exact 0), moves the rock and
            //      its rock-grid entries
            const int warp = tid >> 5, lane = tid & 31;
            for (int pr = warp; pr < n_env * p.R; pr += TPB / 32) {
                uint32_t tm = touch[pr];
                if (tm == 0u) continue;
                const int g = pr / p.R, r = pr - g * p.R, e = env0 + g;
                double *rc = p.rock_c + (int64_t)e * p.R * 2;
                const double cx = rc[2 * r], cy = rc[2 * r + 1], rad = p.rock_rad[(int64_t)e * p.R + r], wt = p.rock_w[(int64_t)e * p.R + r];
                const double *xe = xs + g * p.N, *ye = ys + g * p.N;
                double sx = 0.0, sy = 0.0;
                while (tm) {
                    const int c = __ffs(tm) - 1;
                    tm &= tm - 1;
                    const int a_end = min((c + 1) * Gc, p.N);
                    for (int a0 = c * Gc; a0 < a_end; a0 += 32) {
                        const int aa = a0 + lane;
                        double px = 0.0, py = 0.0;
                        bool hit = false;
                        if (aa < a_end) {
                            const double vx = cx - xe[aa], vy = cy - ye[aa];
                            const double d = sqrt(vx * vx + vy * vy);
                            if (!(d > rad)) {
                                const double fac = 1.0 - rad / (d + 0.001);
                                px = vx * fac; py = vy * fac; hit = true;
                            }
                        }
                        unsigned m = __ballot_sync(0xffffffffu, hit);
                        while (m) {
                            const int l = __ffs(m) - 1;
                            m &= m - 1;
                            sx += __shfl_sync(0xffffffffu, px, l);
                            sy += __shfl_sync(0xffffffffu, py, l);
                        }
                    }
                }
                const double nx = cx - sx / wt, ny = cy - sy / wt;
                if (lane == 0) { rc[2 * r] = nx; rc[2 * r + 1] = ny; }
                if (nx != cx || ny != cy) env_move_rock_grid(p, e, r, cx, cy, nx, ny, rad, lane);
            }
            __threadfence_block();
            __syncthreads();
            // ---- rocks push ants (circle_obstacles.py:53-58).  The grid and the centres were just rewritten by this
            //      block: read them past the L1.
#pragma unroll
            for (int k = 0; k < APT; ++k) rm[k] = __ldcg(env_grid_word(p, env0 + el[k], x[k], y[k]));
#pragma unroll
            for (int k = 0; k < APT; ++k)
                if (rm[k]) env_push_by_rocks(p, env0 + el[k], rm[k], &x[k], &y[k]);
        }
        // ---- prev snapshot and reward_state decay (ants.py:124,130), ownership of the deposit cell (pheromone.py:39, Q1)
        uint8_t rs[APT];
#pragma unroll
        for (int k = 0; k < APT; ++k) rs[k] = p.reward_state[i0 + lac[k]];
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            if (!valid[k]) continue;
            const int64_t i = i0 + lac[k];
            const int ant = lac[k] - el[k] * p.N;
            if (p.R > 0) { xs[lac[k]] = x[k]; ys[lac[k]] = y[k]; }
            p.prev_x[i] = x[k]; p.prev_y[i] = y[k]; p.prev_theta[i] = th[k];
            if (!MOVE) { p.x[i] = x[k]; p.y[i] = y[k]; p.theta[i] = th[k]; }
            p.reward_state[i] = (uint8_t)((double)rs[k] * 0.9);        // ants.py:130
            cell[k] = cidx(p, cell_of(x[k], W), cell_of(y[k], H));
            if (p.P > 0 || MOVE) {
                prefetch_l2(rec_of(el[k], cell[k]));                   // consumed after the barrier
                env_hash_max(hkeys, hvals, HMASK, (uint32_t)(el[k] * p.plane + cell[k]) + 1u, (uint32_t)ant + 1u);
            }
        }
        __syncthreads();
    }

    // ---- MOVE alone: the mandible rule reads the food of the PREV cell (RL_api.py:178); its winner is found here
    double fd[APT];
    int flags[APT];                // bit 0: this ant owns its cell; bit 1: delta != 0; bit 2: the prev cell lies in the hill
#pragma unroll
    for (int k = 0; k < APT; ++k) { fd[k] = 0.0; flags[k] = 0; }
    if (MOVE && !UPDATE) {
        double px[APT], py[APT];
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            const int64_t i = i0 + lac[k];
            xs[lac[k]] = p.x[i]; ys[lac[k]] = p.y[i]; th[k] = p.theta[i];      // (idle slots rewrite the last ant's values)
            px[k] = p.prev_x[i]; py[k] = p.prev_y[i];
        }
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            cell[k] = cidx(p, cell_of(px[k], W), cell_of(py[k], H));
            fd[k] = ld_food(p, rec_of(el[k], cell[k]));
        }
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            if (!valid[k]) continue;
            const int e = env0 + el[k], ant = lac[k] - el[k] * p.N;
            const bool hill = in_hill(p.hill + 4 * e, cell_of(xs[lac[k]], W), cell_of(ys[lac[k]], H));   // RL_api.py:184: CURRENT cell
            if (a.all_stamp || fd[k] > 0.0 || hill)
                env_hash_max(hkeys, hvals, HMASK, (uint32_t)(el[k] * p.plane + cell[k]) + 1u, (uint32_t)ant + 1u);
        }
        __syncthreads();
    }

    // ---- UPDATE: the owner of each cell deposits (ants.py:98-100, pheromone.py:36-41).  MOVE: mandible rule and the
    //      bookkeeping of pickup / drop (ants.py:102-117), rotation and forward move (ants.py:62-80); the food field
    //      itself and the stamps of the new cell are written after the next barrier
    double hold[APT];
    uint8_t mand[APT];
    int8_t rot[APT], phv[APT];     // (every load of the tapes here: past the first store of the loop below a load waits its turn)
    if (MOVE) {
#pragma unroll
        for (int k = 0; k < APT; ++k) {
            const int64_t i = i0 + lac[k];
            hold[k] = p.holding[i]; mand[k] = p.mandibles[i];
            rot[k] = a.rot != nullptr ? a.rot[i] : (int8_t)0;
            phv[k] = a.ph != nullptr ? a.ph[i] : (int8_t)0;
        }
    }
    double av0[APT], av1[APT];     // the activations an owner deposits (ants.py:98-100)
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        const int64_t i = i0 + lac[k];
        av0[k] = (UPDATE && p.P > 0) ? p.act[i] : 0.0;
        av1[k] = (UPDATE && p.P > 1) ? p.act[p.EN + i] : 0.0;
    }
    if (UPDATE && MOVE) {
#pragma unroll
        for (int k = 0; k < APT; ++k) fd[k] = ld_food(p, rec_of(el[k], cell[k]));   // prev cell == this cell after an update
    }
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        if (!valid[k]) continue;
        const int64_t i = i0 + lac[k];
        const int e = env0 + el[k], ant = lac[k] - el[k] * p.N;
        uint8_t *rec = rec_of(el[k], cell[k]);
        const bool own = env_hash_get(hkeys, hvals, HMASK, (uint32_t)(el[k] * p.plane + cell[k]) + 1u) == (uint32_t)ant + 1u;
        if (UPDATE && own && p.P > 0) env_deposit(p, rec, i, a.now, a.now_abs, av0[k], av1[k]);
        if (MOVE) {
            const double x0 = xs[lac[k]], y0 = ys[lac[k]];
            const bool hill = in_hill(p.hill + 4 * e, cell_of(x0, W), cell_of(y0, H));  // RL_api.py:184
            double h = hold[k];
            const int m_old = mand[k] != 0;
            const int fpos = fd[k] > 0.0 ? 1 : 0, out = hill ? 0 : 1;                   // RL_api.py:180-184 (Q5)
            const int m = rule_mode == 0 ? m_old : rule_mode == 1 ? (m_old | fpos) : rule_mode == 2 ? (m_old & out)
                          : rule_mode == 3 ? ((m_old | fpos) & out) : ((m_old & out) | fpos);
            const bool closing = m && !m_old, opening = !m && m_old;                    // ants.py:103-104
            const double taken = closing ? fmin(p.max_hold, fmax(0.0, fd[k])) : 0.0;    // ants.py:111
            const double dropped = opening ? h : 0.0;                                   // ants.py:114
            const double delta = dropped - taken;
            h = h + (taken - dropped);                                                  // ants.py:117
            p.mandibles[i] = (uint8_t)m;
            p.holding[i] = h;
            // (after an update the prev cell IS the current cell: its hill bit decides whether dropped food is queued)
            flags[k] = (own ? 1 : 0) | (delta != 0.0 ? 2 : 0) | ((UPDATE && hill) ? 4 : 0);
            fd[k] = fd[k] + delta;                                                      // what the owner will write (ants.py:116)
            double t = th[k];
            if (a.rot != nullptr) t = pymod_near(t + (double)rot[k] * p.max_rot_speed, 6.283185307179586);   // ants.py:62-67
            double fwd = (1.0 * p.max_speed) * (1.0 - h * p.csr);                       // RL_api.py:194
            if (fwd < 0.0) fwd *= p.bsr;                                                // RL_api.py:195
            double sn, cs;
            sincos(t, &sn, &cs);
            const double x = pymod_near(x0 + cs * fwd, Wd);                             // ants.py:69-80
            const double y = pymod_near(y0 + sn * fwd, Hd);
            p.x[i] = x; p.y[i] = y; p.theta[i] = t;
            newcell[k] = cidx(p, cell_of(x, W), cell_of(y, H));
            prefetch_l2(rec_of(el[k], newcell[k]));
        }
    }
    if (!MOVE) return;
    __syncthreads();               // every ant has read its cell's food before any owner rewrites it

    // ---- MOVE: the owners write the food (ants.py:116, Q1); activation (ants.py:89-96); wall flag and occupancy stamp
    //      of the new cell
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        if (!valid[k]) continue;
        const int64_t i = i0 + lac[k];
        const int e = env0 + el[k];
        if ((flags[k] & 3) == 3) {
            uint8_t *fr = rec_of(el[k], cell[k]);
            const double nv = env_food_commit(p, fr, fd[k]);
            bool queue = nv != 0.0;
            if (queue) {
                if (UPDATE) queue = (flags[k] & 4) != 0;
                else {                                                 // prev cell != current cell: test the prev cell itself
                    const int cx = cell_of(p.prev_x[i], W), cy = cell_of(p.prev_y[i], H);
                    queue = in_hill(p.hill + 4 * e, cx, cy);
                }
            }
            if (queue) {
                const uint32_t s = atomicAdd(p.absorb_count + e, 1u);
                if (s < (uint32_t)p.N) p.absorb_list[(int64_t)e * p.N + s] = (uint32_t)cell[k];
            }
        }
        if (a.ph != nullptr) {                                                          // ants.py:89-96
            const int v = phv[k];
            p.act[i] = (v == 1) ? a.act_on : 0.0;
            p.act[p.EN + i] = (v != 0 && v != 1) ? a.act_on : 0.0;
        }
    }
    // Occupancy stamp of the new cell (RL_api.py:136-142) and its wall bit for the coming update
    // (the loads of all the thread's ants first, then the stores: a load behind a store is not moved up by the compiler)
    uint32_t meta[APT];            // compact records: the 16 bits [hill | occ stamp][wall | explored stamp]; else the wall bit
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        const uint8_t *orec = rec_of(el[k], newcell[k]);
        meta[k] = (p.rec8 || p.rec16) ? (uint32_t)*reinterpret_cast<const uint16_t *>(orec + (p.rec8 ? 6 : 12))
                                      : (ld_wall(p, orec) ? 0x8000u : 0u);
    }
#pragma unroll
    for (int k = 0; k < APT; ++k) {
        if (!valid[k]) continue;
        uint8_t *orec = rec_of(el[k], newcell[k]);
        p.wall_hit[i0 + lac[k]] = (uint8_t)(meta[k] >> 15);            // for Walls.update of the coming update
        if (p.rec8 || p.rec16) orec[p.rec8 ? 6 : 12] = (uint8_t)((meta[k] & 0x80u) | (a.occ_gen & 0x7Fu));
        else st_occ(p, orec, a.occ_gen);
    }
}

}  // namespace ants
