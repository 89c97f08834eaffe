// ants_perceive_rows.cuh -- the perception + reward kernel for the generator's default channel list
// (RL_api.py:96-165, reward_custom.py:79-106, ants.py:119-121), "row per lane" mapping.
//
// The generic kernel (k_perceive in ants_kernels.cuh) spreads a chunk's samples over the lanes by a flat sample
// index: every sample re-derives its ant and its window position and re-reads the ant's frame from shared memory,
// and the exploration counts need a ballot split at the ant boundaries -- ncu showed ~490 warp instructions per ant
// with the issue slots as the limiter.  Here a warp still owns 32 consecutive ants and walks them in chunks of 4
// (the bulk-store granule: 4 * S*S * C * 4 bytes is always a multiple of 16), but lane l of the chunk is
//     ant  a = l / S        row  i = l % S        (4 * S <= 32 lanes active; 28 of 32 for the default 7x7 window)
// and loops over the S columns j of its row.  Everything that depends on (ant, row) -- cos/sin of the frame, the
// shifted position, st*Y and ct*Y of RL_api.py:110-111, the anthill, the record base, the row's mask bits -- lives in
// registers for the whole row; the column offset X = off[j] is a kernel-parameter constant after unrolling, so a
// sample costs two f64 multiplies, four adds and two conversions for its cell (bit-identical to the reference's
// ct*X - st*Y, st*X + ct*Y: every product is rounded separately, -fmad=false), one 128-bit record load (compact
// records; two for f64 records), a branch-free decode and C shared-memory stores.  All record loads of a row are in
// flight before the first is decoded.  Exploration counts are per-lane adds, summed over the S rows in the epilogue.
// The staged (4 x S*S x C) f32 tile leaves with one TMA bulk store, as before.
//
// Round 2 (0.240 -> 0.177 ms on the cfg4 shard, 224 -> 195 warp instructions per ant): the kernel's pointers may alias
// as far as the compiler knows, so in phase A (thread per ant) every load that followed a store waited for the
// previous round trip -- all loads of the ant's state are now issued before the first store (-18 %); the rock channel
// of the few ants a rock can reach is evaluated by the whole warp instead of the ant's S row lanes (-6 %); blocks of
// one warp (the block index is warp-uniform to the compiler); the reward terms of phase C wait in shared memory, not in
// registers of the chunk loop; ages go to float through the 2^23 exponent trick; half of the column products follow
// from the symmetry of the window offsets.
#pragma once

namespace ants {

constexpr int kRowsThreads = 32;
constexpr int kRowsOcc = 20;         // resident one-warp blocks per SM: 20 warps at 96 registers
constexpr int kRowsGroup = 4;
constexpr int kRowsTiles = 1;        // staging tiles per warp

struct RowPrep {                 // 96 bytes per ant, shared memory (phase A -> phase B, C)
    double ct, st;               // cos / sin(theta + pi/2)
    double xf, yf;               // position shifted forward by perception_fwd_delta
    unsigned long long rocks;    // further candidate rocks (beyond the first) whose disc can reach the window
    int e, flags;                // environment; 2 = a rock may reach the window, 4 = more than one
    double rcx, rcy, rrad;       // the first candidate rock
    double r_other, r_mult;      // phase A -> phase C: the reward terms that do not need the exploration count ...
    int rs_prev, pad;            // ... and the ant's reward_state (kept out of the registers of the chunk loop)
};

// one conditional add or subtract wraps a sample coordinate onto the torus (np.mod on ints, RL_api.py:118-119) when
// the window reaches less than one map size past the border: of v, v + n, v - n the one in [0, n) is the smallest as
// an unsigned number
__device__ __forceinline__ int wrap1(int v, int n) {
    return (int)min(min((unsigned)v, (unsigned)(v + n)), (unsigned)(v - n));
}
// np.round(v).astype(int) (half to even, RL_api.py:117) for |v| < 2^31 without the quarter-rate F2I.F64: adding
// 1.5 * 2^52 leaves the rounded integer (two's complement) in the low word of the sum -- the add itself rounds to
// nearest-even, exactly like rint()
__device__ __forceinline__ int round_half_even(double v) { return __double2loint(v + 6755399441055744.0); }
__device__ __forceinline__ float ex2_approx(float x) {   // MUFU.EX2 (2^-22 relative); arguments here are in [-15, 0]
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 16-byte record load.  (Measured alternatives, all slower on the cfg4 shard: ld.global.L2::128B / L2::64B prefetch
// sizes and the non-coherent path, 0.35 ms against 0.29 ms.)
__device__ __forceinline__ uint4 ld_record16(const uint8_t *rp) { return *reinterpret_cast<const uint4 *>(rp); }
// 8-byte record load.  (Cache policies measured on the cfg4 shard, 0.177 ms with the default: .cg (L2 only) 0.232,
// L1::no_allocate 0.270, L1::evict_first 0.204, L1::evict_last 0.177 -- half of the gathers hit in L1.)
__device__ __forceinline__ uint2 ld_record8(const uint8_t *rp) { return *reinterpret_cast<const uint2 *>(rp); }

// value of a pheromone field that is neither zero nor a live boxed deposit outside walls (rare): kept out of line
__device__ __noinline__ float phero_obs_slow(const Params &p, const uint8_t *rp, int k, uint32_t now, uint32_t now_abs) {
    const double inv_max = 1.0 / p.phero_max_val;
    return (float)(phero_value(p, rp, k, now, now_abs) * inv_max);
}

// exact rock test of one sample cell against the candidate rocks (RL_api.py:132-135, strict <)
__device__ __noinline__ float rock_channel(const Params &p, int e, unsigned long long rm, int ix, int iy) {
    const double *rc = p.rock_c + (int64_t)e * p.R * 2;
    const double *rr = p.rock_rad + (int64_t)e * p.R;
    while (rm) {
        const int r = __ffsll((long long)rm) - 1;
        rm &= rm - 1;
        const double ddx = (double)ix - rc[2 * r], ddy = (double)iy - rc[2 * r + 1];
        if (sqrt(ddx * ddx + ddy * ddy) < rr[r]) return 1.f;
    }
    return 0.f;
}

// Measured on the cfg4 shard (512 envs x 1024 ants, 8-byte records, one B200) and left out of the code again:
//   * all 32 * S rows of a warp handed to the lanes without idle lanes (two staging tiles): 0.279 ms against 0.241;
//   * the record loads of chunk g + 1 issued before chunk g is decoded (two register sets): 0.278 - 0.338 ms;
//   * L2 prefetch of the next chunk's records: 0.254 (4 samples per row) and 0.269 ms (all 7) against 0.240;
//   * a second copy of the chunk loop for warps with all 32 ants (no ragged-end bookkeeping): 0.2248 against 0.2223;
//   * 80 registers for 24 warps per SM (8 bytes of spills): 0.226 ms against 0.177;
//   * shared memory / L1 split (ANTS_ROWS_CARVEOUT, profiles/r2_bench/perceive_carveout.txt): 164 KB shared + 92 KB L1
//     with 16 resident warps 0.177 ms; 196 / 228 KB shared (20 warps, <= 60 KB L1) 0.221 ms; 132 KB (13 warps, 124 KB
//     L1) 0.1815; 100 KB (10 warps) 0.204 -- the gathers need ~90 KB of L1, more warps than 16 do not pay for taking it
//     away.  ants_create asks for the 164 KB split (the driver's own choice follows the register count: it gave the
//     80-register C = 6 kernel of cfg3 the 228 KB split, 0.205 ms against 0.154);
//   * prep record cut to 64 bytes (the first rock's disc re-read from global memory in the rock path): 0.186 against
//     0.177 at every split (perceive_carveout_prep64.txt);
//   * 2 or 3 ants per thread in phases A / C (a warp serving 64 or 96 ants, the round trips of phase A paid once for all
//     of them; prep record cut to 64 bytes with the first rock's disc re-read from global memory): 0.247 and 0.282 ms
//     against 0.189 for the same code with one ant per thread (profiles/r2_bench/perceive_variants_apt.txt).
template <int LAYOUT, int REC, int S>      // REC: 0 = f64 records, 1 = compact 16-byte, 2 = compact 8-byte
__global__ void __launch_bounds__(kRowsThreads, kRowsOcc)
k_perceive_rows(const __grid_constant__ Params p, float *__restrict__ obs, float *__restrict__ agent_state, float *__restrict__ state_out,
                double *__restrict__ reward_out, uint32_t obs_gen, uint32_t occ_gen, int is_step, int rw_alias,
                uint32_t now, uint32_t now_abs, int64_t ant0, int64_t ant_end) {
    // (ants [ant0, ant_end) of the batch: ants_rollout runs groups of environments on streams of their own)
    pdl_begin();
    static_assert(LAYOUT == 1 || LAYOUT == 2, "default channel lists only");
    constexpr bool REC16 = (REC == 1), REC8 = (REC == 2);
    constexpr int SH = REC8 ? 3 : (REC16 ? 4 : 5);                    // log2(record bytes)
    static_assert(kRowsGroup * S <= 32, "a chunk's rows must fit one warp");
    constexpr int S2 = S * S, C = (LAYOUT == 2) ? 7 : 6, SC = S2 * C;
    constexpr int G = kRowsGroup, ROWS = G * S, TILE = G * SC;       // TILE * 4 bytes is a multiple of 16
    constexpr int NW = kRowsThreads / 32;
    constexpr int UNR = (REC != 0) ? S : (S + 1) / 2;                 // record loads in flight per lane
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *s_obs = reinterpret_cast<float *>(smem_raw);               // [NW][TILE]
    RowPrep *prep = reinterpret_cast<RowPrep *>(s_obs + NW * kRowsTiles * TILE);   // [threads]
    uint8_t *s_rowcnt = reinterpret_cast<uint8_t *>(prep + kRowsThreads);   // [threads][S]

    const int tid = threadIdx.x;
    const int64_t base = ant0 + (int64_t)blockIdx.x * kRowsThreads;
    const bool explore_on = p.explore_on != 0;

    // ---- phase A (thread per ant): frame, reward terms that do not need the exploration count, small outputs.
    // The kernel's pointers may alias as far as the compiler knows, so a load after a store waits for it: every load
    // of the ant's state is issued first, the stores come last, and the dependent chain is state -> rock grid word ->
    // rock discs (ncu, round 2: phase A / C were 12 % of the instructions and 29 % of the warps' stall samples).
    int my_rock_flags = 0;
    {
        double r_other = 0.0, r_mult = 1.0;
        int rs_prev = 0;                                                       // reward_state, used by phase C
        const int64_t i = base + tid;
        if (i < ant_end) {
            const int e = (int)(i / p.N);
            const double x = p.x[i], y = p.y[i], th = p.theta[i], hold = p.holding[i];
            const double hprev = rw_alias ? hold : p.rw_holding_prev[i];       // Q18
            const double pdist = (p.reward_kind == 0) ? p.rw_prev_dist[i] : 0.0;
            const int32_t *hl = p.hill + 4 * e;
            const int32_t hx = hl[0], hy = hl[1];
            const float seed_f = (float)p.seed[i];
            const uint8_t mand = p.mandibles[i];
            const bool want_state = state_out != nullptr;
            const double act0 = (want_state && p.P > 0) ? p.act[i] : 0.0;
            const double act1 = (want_state && p.P > 1) ? p.act[(int64_t)p.EN + i] : 0.0;
            if (is_step) rs_prev = p.reward_state[i];
            double s0, c0, st, ct;
            sincos(th, &s0, &c0);
            RowPrep q;
            q.xf = x; q.yf = y;
            if (p.fwd_delta != 0.0) { q.xf = x + c0 * p.fwd_delta; q.yf = y + s0 * p.fwd_delta; }   // RL_api.py:103-104
            q.e = e;
            // grid candidates (the word is on its way while the frame and the reward terms are computed)
            unsigned long long rm = (LAYOUT == 2) ? rock_candidates(p, e, q.xf, q.yf) : 0ull;
            sincos(th + 3.141592653589793 * 0.5, &st, &ct);                    // RL_api.py:101,107-108
            q.ct = ct; q.st = st;
            const double d = hold - hprev;
            double nd = 0.0;
            if (p.reward_kind == 0) {                                          // All_Rewards, reward_custom.py:79-106
                const double r_food = d < 0.0 ? 0.0 : d;
                const double r_hill = d < 0.0 ? 1.0 : 0.0;
                const double ddx = x - (double)hx, ddy = y - (double)hy;
                nd = sqrt(ddx * ddx + ddy * ddy);
                const double heading = (pdist > nd && hold > 0.0) ? 0.1 : 0.0;
                r_other = r_food * p.f_food + r_hill * p.f_anthill + heading * p.f_heading;
                r_mult = (hold == 0.0) ? p.f_explore : p.f_explore_hold;
            } else if (p.reward_kind == 2) {                                   // Food_Reward, :37-40
                r_other = d < 0.0 ? 10.0 : d;
            }
            q.flags = 0;
            q.rcx = q.rcy = 0.0; q.rrad = -1.0;
            q.rocks = 0ull;
            if (LAYOUT == 2 && rm) {
                // narrowed to the rocks whose disc can reach the window: a sample lies within
                // radius*DELTA*sqrt(2) + 0.5 (rounding) of (xf, yf) on the torus.  The discs of the first two
                // candidates are loaded together (more than two are rare)
                const double *rc = p.rock_c + (int64_t)e * p.R * 2;
                const double *rr = p.rock_rad + (int64_t)e * p.R;
                const double reach = (double)p.radius * p.delta * 1.4142135623730951 + 1.0;
                auto near = [&](double cx, double cy, double rad) -> bool {
                    double dx = fabs(q.xf - cx), dy = fabs(q.yf - cy);
                    dx = fmin(dx, fabs((double)p.W - dx));
                    dy = fmin(dy, fabs((double)p.H - dy));
                    const double L = rad + reach;
                    return dx < L && dy < L && dx * dx + dy * dy < L * L;
                };
                const int ra = __ffsll((long long)rm) - 1;
                unsigned long long it = rm & (rm - 1);
                const int rb = it ? __ffsll((long long)it) - 1 : ra;
                it &= it - 1;
                const double ax = rc[2 * ra], ay = rc[2 * ra + 1], arad = rr[ra];
                const double bx = rc[2 * rb], by = rc[2 * rb + 1], brad = rr[rb];
                const bool ka = near(ax, ay, arad), kb = (rb != ra) && near(bx, by, brad);
                unsigned long long keep = (ka ? 1ull << ra : 0ull) | (kb ? 1ull << rb : 0ull);
                while (it) {
                    const int r = __ffsll((long long)it) - 1;
                    it &= it - 1;
                    if (near(rc[2 * r], rc[2 * r + 1], rr[r])) keep |= 1ull << r;
                }
                if (keep) {
                    const int r = __ffsll((long long)keep) - 1;            // the first candidate rides in the prep record
                    keep &= keep - 1;
                    if (r == ra) { q.rcx = ax; q.rcy = ay; q.rrad = arad; }
                    else if (r == rb) { q.rcx = bx; q.rcy = by; q.rrad = brad; }
                    else { q.rcx = rc[2 * r]; q.rcy = rc[2 * r + 1]; q.rrad = rr[r]; }
                    q.flags = keep ? 6 : 2;
                    q.rocks = keep;
                }
                my_rock_flags = q.flags;
            }
            q.r_other = r_other; q.r_mult = r_mult; q.rs_prev = rs_prev; q.pad = 0;
            prep[tid] = q;
            // the stores
            if (p.reward_kind == 0) { p.rw_prev_dist[i] = nd; p.rw_holding_prev[i] = hold; }
            else if (p.reward_kind == 2) p.rw_holding_prev[i] = hold;
            agent_state[2 * i] = (float)hold;                                  // RL_api.py:160-162
            agent_state[2 * i + 1] = seed_f;
            if (want_state) {                                                  // RL_api.py:155-158
                float *so = state_out + i * (2 + p.P);
                so[0] = (float)mand;
                so[1] = (float)hold;
                if (p.P > 0) so[2] = act0 > 0.0 ? 1.f : 0.f;
                if (p.P > 1) so[3] = act1 > 0.0 ? 1.f : 0.f;
                for (int k = 2; k < p.P; ++k) so[2 + k] = p.act[(int64_t)k * p.EN + i] > 0.0 ? 1.f : 0.f;
            }
        }
    }
    __syncwarp();        // a warp only reads the prep records of its own 32 ants
    const uint32_t rock_ants = (LAYOUT == 2) ? __ballot_sync(0xffffffffu, my_rock_flags != 0) : 0u;   // bit a: ant a of the warp

    // ---- phase B: a lane processes one window row of one ant (its S columns); two ways of handing out the rows
    const int warp = tid >> 5, lane = tid & 31;
    const int W = p.W, H = p.H;
    const int nby64m = (p.nby << 6) - 64;
    // ages that still show a value: the table's last entry is the 0 the reference's < 0.01 cut produced
    const uint32_t tab_len = p.tab_len > 0 ? (uint32_t)p.tab_len - 1u : 0u;
    const float decay_c = (float)p.log2_keep;                       // obs = 2^(age * log2(keep)), see below
    const float decay_c2 = -8388608.f * decay_c;
    // 2^23 + table length as a float (8-byte records: live ages are < 2^15, everything else reads >= 2^15)
    const float tab_len_f = __uint_as_float(0x4B000000u | (tab_len < 0x8000u ? tab_len : 0x8000u));
    const bool eager = (REC == 0) && !p.lazy;                       // f64 fields hold plain current values (no decay on read)
    const bool eager_planes = eager && p.diffuse != 0;              // ... in the diffusion planes (sign bit = wall)
    const double inv_max = 1.0 / p.phero_max_val;
    const bool any_plain = !eager && *p.plain_flag != 0u;           // lazy field: plain (non-boxed) values may exist
    // boxed deposit b = box | t: (box | now) - b = now - t = age; zero and plain values give an "age" >= 2^22
    const uint32_t nowb = REC16 ? box32(now_abs) : (REC8 ? now_abs : (now_abs & kBoxMask));
    // 8-byte records: both 15-bit deposit steps of a cell are aged in one subtraction (bit 15 of each half set in the
    // minuend: no borrow crosses the halves)
    const uint32_t nowb2 = ((now_abs & kBox8Mask) | kBox8) * 0x00010001u;
    const uint32_t ogs = obs_gen << 8;
    float *wobs0 = s_obs + warp * kRowsTiles * TILE;
    constexpr bool kLateWait = (UNR >= S);
    constexpr bool ROCKS = LAYOUT == 2;
    // one row: sample cells, record loads, decode, staging-tile stores; returns the row's count of unexplored samples
    // phase 2 = the whole row; phase 0 = only issue the record loads into (lo, hi, cell); phase 1 = only consume them
    // exact rock test of one sample cell against the ant's candidate rocks (RL_api.py:132-135): strict sqrt(d2) < r,
    // decided on the squares unless d2 is within 1e-12 of r^2
    auto rock_hit = [&](const RowPrep &q, const int ix, const int iy) -> bool {
        const double ddx = (double)ix - q.rcx, ddy = (double)iy - q.rcy, rad = q.rrad;
        const double d2 = ddx * ddx + ddy * ddy, r2 = rad * rad;
        bool hit = d2 < r2 * 0.999999999999;
        if (!hit && d2 <= r2 * 1.000000000001) hit = sqrt(d2) < rad;
        if (!hit && (q.flags & 4)) hit = rock_channel(p, q.e, q.rocks, ix, iy) != 0.f;
        return hit;
    };
    auto row_body = [&](const RowPrep &q, const double offY, const uint32_t mrow, const uint32_t orow_s,
                        const uint32_t amask, uint4 (&lo)[UNR], uint4 (&hi)[UNR], uint32_t (&cell)[UNR],
                        const int phase, const uint32_t rbits) -> int {
        const double ct = q.ct, st = q.st, xf = q.xf, yf = q.yf;
        const int e = q.e;
        const uint8_t *cells = p.cells + (((int64_t)e * p.plane) << SH);
        asm volatile("" : "+l"(cells));                            // one opaque 64-bit base: one IMAD.WIDE per sample address
        const double *plane0 = eager_planes ? p.phero_pl + (int64_t)e * 2 * p.plane : nullptr;   // [e][k = 0, 1]
        const double stY = st * offY, ctY = ct * offY;             // RL_api.py:110-111
        int cnt = 0;                                               // (rbits, bit j: a rock covers the sample at column j)
        constexpr int RH = S / 2;
        // The window offsets are (j - radius) * DELTA (RL_api.py:92-93): ct * X and st * X are computed for the columns
        // right of the centre only -- a product's sign flips exactly with its factor's
        double ctX[RH > 0 ? RH : 1], stX[RH > 0 ? RH : 1];
        if (phase != 1) {
#pragma unroll
            for (int k = 0; k < RH; ++k) { ctX[k] = ct * p.off_c[RH + 1 + k]; stX[k] = st * p.off_c[RH + 1 + k]; }
        }
#pragma unroll
        for (int j0 = 0; j0 < S; j0 += UNR) {
            if (phase != 1) {
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int j = j0 + u;
                if (j < S) {
                    // sample cell, RL_api.py:110-119: round_half_even(rot(theta + pi/2) * offset + xy_f) mod (W, H)
                    double cX, sX;                         // ct * X, st * X with X = off_c[j] = -off_c[S - 1 - j]
                    if (j == RH) { cX = 0.0; sX = 0.0; }           // (the sign of a zero is lost in the sums below)
                    else if (j > RH) { cX = ctX[j - RH - 1]; sX = stX[j - RH - 1]; }
                    else { cX = -ctX[RH - 1 - j]; sX = -stX[RH - 1 - j]; }
                    const double rx = cX - stY;
                    const double ry = sX + ctY;
                    int ix = round_half_even(rx + xf), iy = round_half_even(ry + yf);
                    ix = wrap1(ix, W); iy = wrap1(iy, H);
                    // cidx(): 8 x 8 blocks of 64 records; (x & 7) * 8 = 8 x - 64 (x >> 3), (y >> 3) * 64 + (y & 7) = y + 56 (y >> 3)
                    cell[u] = (uint32_t)((ix >> 3) * nby64m + ix * 8 + (iy >> 3) * 56 + iy);
                    const uint8_t *rp = cells + ((size_t)cell[u] << SH);
                    if (REC8) {                    // the whole cell in one 64-bit load, four cells per sector
                        const uint2 v8 = ld_record8(rp);
                        lo[u] = make_uint4(v8.x, v8.y, 0u, 0u);
                    } else if (REC == 0 && eager_planes) {  // diffusion: the two pheromone values come from the row-major planes
                        const double *pv = plane0 + (int64_t)ix * p.Hp + iy;
                        const double d0 = pv[0], d1 = pv[p.plane];
                        lo[u] = make_uint4((uint32_t)__double2loint(d0), (uint32_t)__double2hiint(d0) & 0x7FFFFFFFu,
                                           (uint32_t)__double2loint(d1), (uint32_t)__double2hiint(d1) & 0x7FFFFFFFu);
                    } else {
                        lo[u] = ld_record16(rp);
                    }
                    if (REC == 0) hi[u] = *reinterpret_cast<const uint4 *>(rp + 16);
                    asm volatile("" : "+r"(cell[u]));      // the decode keeps the 32-bit cell index, not the 64-bit address
                }
            }
            }
            if (phase == 0) return 0;
            if (kLateWait) {
                if (lane == 0) bulk_store_wait_read<kRowsTiles - 1>();
                __syncwarp(amask);
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int j = j0 + u;
                if (j < S) {
                    uint8_t *rp = const_cast<uint8_t *>(cells) + ((size_t)cell[u] << SH);
                    bool wl, occupied, fresh, seen_now, hill;
                    uint32_t age0, age1;
                    float m0 = 0.f, m1 = 0.f;      // 2^23 + age as floats (8-byte records)
                    float v5;                      // food as the f32 observation shows it
                    if (REC8) {
                        const uint32_t pk = lo[u].y >> 16;                 // [hill|occ][wall|explored]
                        occupied = (pk & 0x7Fu) == occ_gen;
                        hill = (pk & 0x80u) != 0;
                        wl = (pk & 0x8000u) != 0;
                        fresh = (pk & 0x7F00u) == 0u;
                        seen_now = (pk & 0x7F00u) == ogs;
                        v5 = (float)(lo[u].y & 0xFFFFu);                   // (an escaped amount is patched in below)
                        // per half: age = (now - step) mod 2^15 for a boxed deposit (bit 15 set), >= 2^15 (= expired) else
                        const uint32_t d2 = nowb2 - (lo[u].x & 0x7FFF7FFFu);
                        const uint32_t a2 = (d2 & 0x7FFF7FFFu) | (~lo[u].x & 0x80008000u);
                        age0 = a2 & 0xFFFFu; age1 = a2 >> 16;
                        // bytes [age lo, age hi, 00, 4B] = the float 2^23 + age: one PRMT instead of mask + I2F
                        m0 = __uint_as_float(__byte_perm(a2, 0x4B000000u, 0x7610u));
                        m1 = __uint_as_float(__byte_perm(a2, 0x4B000000u, 0x7632u));
                        if (explore_on && fresh) rp[7] = (uint8_t)(((pk >> 8) & 0x80u) | obs_gen);
                    } else if (REC16) {
                        const uint32_t pk = lo[u].w;
                        occupied = (pk & 0x7Fu) == occ_gen;
                        hill = (pk & 0x80u) != 0;
                        wl = (pk & 0x8000u) != 0;
                        fresh = (pk & 0x7F00u) == 0u;
                        seen_now = (pk & 0x7F00u) == ogs;
                        v5 = __uint_as_float(lo[u].z);
                        age0 = nowb - lo[u].x; age1 = nowb - lo[u].y;
                        if (explore_on && fresh) rp[13] = (uint8_t)(((pk >> 8) & 0x80u) | obs_gen);
                    } else {
                        occupied = (hi[u].z >> 16) == occ_gen;
                        wl = (hi[u].w & 1u) != 0;
                        hill = (hi[u].w & 2u) != 0;
                        fresh = (hi[u].z & 0xFFFFu) == 0u;
                        seen_now = (hi[u].z & 0xFFFFu) == obs_gen;
                        v5 = (float)__hiloint2double((int)hi[u].y, (int)hi[u].x);
                        // f64 fields: boxed <=> the high word carries the NaN box; the deposit step is the low word
                        const bool bx0 = p.lazy && (lo[u].y & 0xFFF80000u) == 0x7FF80000u;
                        const bool bx1 = p.lazy && (lo[u].w & 0xFFF80000u) == 0x7FF80000u;
                        age0 = bx0 ? ((nowb - lo[u].x) & kBoxMask) : 0xFFFFFFFFu;
                        age1 = bx1 ? ((nowb - lo[u].z) & kBoxMask) : 0xFFFFFFFFu;
                        if (explore_on && fresh) *reinterpret_cast<uint16_t *>(rp + 24) = (uint16_t)obs_gen;
                    }
                    if (explore_on) cnt += (fresh || seen_now) ? 1 : 0;    // gather-before-scatter, Q7
                    // pheromone channels, RL_api.py:124-125.  A saturated deposit of age k shows
                    // (float)(max_val * keep^k / max_val) = keep^k (the reference's per-step rounding moves it by
                    // ~1e-16 k): evaluated as 2^(k log2 keep) in f32, < 1.2e-6 relative (bar 1e-5); the < 0.01
                    // cut is the exact table length; inside a wall only a deposit of this very update shows.
                    float v1, v2;
                    if (REC8) {
                        // (2^23 + age) c - 2^23 c in one fused rounding = the rounded product age * c (2^23 c is exact);
                        // the floats 2^23 + n order like the integers n
                        const float limf = wl ? 8388609.f : tab_len_f;
                        v1 = m0 < limf ? ex2_approx(__fmaf_rn(m0, decay_c, decay_c2)) : 0.f;
                        v2 = m1 < limf ? ex2_approx(__fmaf_rn(m1, decay_c, decay_c2)) : 0.f;
                    } else {
                        const uint32_t lim = wl ? 1u : tab_len;
                        v1 = age0 < lim ? ex2_approx((float)age0 * decay_c) : 0.f;
                        v2 = age1 < lim ? ex2_approx((float)age1 * decay_c) : 0.f;
                    }
                    if (REC == 0 && eager) {       // eager f64 fields (dense / tiles / diffusion): phero / max_val
                        v1 = (float)(__hiloint2double((int)lo[u].y, (int)lo[u].x) * inv_max);
                        v2 = (float)(__hiloint2double((int)lo[u].w, (int)lo[u].z) * inv_max);
                    }
                    const float v0 = occupied ? 1.f : 0.f;                                   // :136-142
                    const float v3 = hill ? 1.f : 0.f;                                       // :130-131 (disc bit of the record)
                    const float v4 = wl ? 1.f : 0.f;                                         // :128-129
                    const float v6 = ((rbits >> j) & 1u) ? 1.f : 0.f;                        // :132-135
                    const uint32_t vis = (mrow >> j) & 1u;     // masked slots keep the -1 written once above
                    const uint32_t oaddr = orow_s + (uint32_t)(j * C * 4);
                    if (LAYOUT == 2)
                        asm volatile("{\n .reg .pred pv;\n setp.ne.u32 pv, %0, 0;\n"
                                     " @pv st.shared.f32 [%1], %2;\n @pv st.shared.f32 [%1+4], %3;\n"
                                     " @pv st.shared.f32 [%1+8], %4;\n @pv st.shared.f32 [%1+12], %5;\n"
                                     " @pv st.shared.f32 [%1+16], %6;\n @pv st.shared.f32 [%1+20], %7;\n"
                                     " @pv st.shared.f32 [%1+24], %8;\n}"
                                     ::"r"(vis), "r"(oaddr), "f"(v0), "f"(v1), "f"(v2), "f"(v3), "f"(v4), "f"(v5), "f"(v6) : "memory");
                    else
                        asm volatile("{\n .reg .pred pv;\n setp.ne.u32 pv, %0, 0;\n"
                                     " @pv st.shared.f32 [%1], %2;\n @pv st.shared.f32 [%1+4], %3;\n"
                                     " @pv st.shared.f32 [%1+8], %4;\n @pv st.shared.f32 [%1+12], %5;\n"
                                     " @pv st.shared.f32 [%1+16], %6;\n @pv st.shared.f32 [%1+20], %7;\n}"
                                     ::"r"(vis), "r"(oaddr), "f"(v0), "f"(v1), "f"(v2), "f"(v3), "f"(v4), "f"(v5) : "memory");
                }
            }
            if (any_plain) {   // plain pheromone values (bool activations, imports, eager modes) may exist: patch them in
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int j = j0 + u;
                    if (j >= S || !((mrow >> j) & 1u)) continue;
                    const uint8_t *rp = cells + ((size_t)cell[u] << SH);
                    bool pl0, pl1;
                    if (REC8) {
                        const uint2 r2 = *reinterpret_cast<const uint2 *>(rp);
                        pl0 = (r2.x & 0xFFFFu) == 1u; pl1 = (r2.x >> 16) == 1u;
                        if ((r2.y & 0xFFFFu) == kFoodEsc)                  // a non-integer amount of food
                            asm volatile("st.shared.f32 [%0+20], %1;" ::"r"(orow_s + (uint32_t)(j * C * 4)), "f"((float)ld_food(p, rp)) : "memory");
                    } else {
                        const uint4 r4 = *reinterpret_cast<const uint4 *>(rp);
                        pl0 = REC16 ? (r4.x != 0u && !is_boxed32(r4.x))
                                    : ((r4.x | r4.y) != 0u && !(p.lazy && (r4.y & 0xFFF80000u) == 0x7FF80000u));
                        pl1 = REC16 ? (r4.y != 0u && !is_boxed32(r4.y))
                                    : ((r4.z | r4.w) != 0u && !(p.lazy && (r4.w & 0xFFF80000u) == 0x7FF80000u));
                    }
                    const uint32_t oaddr = orow_s + (uint32_t)(j * C * 4);
                    if (pl0) asm volatile("st.shared.f32 [%0+4], %1;" ::"r"(oaddr), "f"(phero_obs_slow(p, rp, 0, now, now_abs)) : "memory");
                    if (pl1) asm volatile("st.shared.f32 [%0+8], %1;" ::"r"(oaddr), "f"(phero_obs_slow(p, rp, 1, now, now_abs)) : "memory");
                }
            }
        }
        return cnt;
    };
    // flush n_in ants' staged (S2 x C) f32 observations: one TMA bulk store when 16 B granular, else plain stores
    auto flush = [&](const float *wobs, int64_t i0, int n_in) {
        float *dst = obs + i0 * SC;
        const uint32_t bytes = (uint32_t)(n_in * SC * 4);
        if ((bytes & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) bulk_store_s2g(dst, wobs, bytes);
        } else {
            __syncwarp();
            for (int t = lane; t < n_in * SC; t += 32) dst[t] = wobs[t];
            __syncwarp();
        }
    };
    const int64_t wbase = base + warp * 32;
    const int la = lane / S, li = lane - la * S;
    const bool lane_on = lane < ROWS;
    const double offY = p.off_c[lane_on ? li : 0];
    uint32_t mrow = p.mask_rows[lane_on ? li : 0];
    // this lane's row of the staging tile (fixed for the whole kernel), as a shared-space address
    uint32_t orow_s = (uint32_t)__cvta_generic_to_shared(wobs0 + ((lane_on ? la : 0) * S2 + (lane_on ? li : 0) * S) * C);
    asm volatile("" : "+r"(orow_s), "+r"(mrow));                   // keep them in registers (no rematerialisation)
    // masked samples read -1 in every channel (RL_api.py:147-148) and their tile slots are never written again
    if (lane_on) {
#pragma unroll
        for (int j = 0; j < S; ++j)
            if (!((mrow >> j) & 1u))
#pragma unroll
                for (int c = 0; c < C; ++c)
                    asm volatile("st.shared.f32 [%0], %1;" ::"r"(orow_s + (uint32_t)((j * C + c) * 4)), "f"(-1.f) : "memory");
    }
    // The rock channel of the chunk's ants a rock may reach (bits of fa), by the whole warp: the S*S samples of such an
    // ant go over the lanes (the same arithmetic as in row_body, so the same cells), the hits come back to the ant's
    // row lanes as ballots.  Returns this lane's row bits.  (Warp-converged call; the ant's S row lanes alone would
    // leave the other rows of the chunk idle for S iterations: ncu showed 15 % of the kernel's instructions there.)
    auto rock_rows = [&](const int g, uint32_t fa) -> uint32_t {
        uint32_t rb = 0u;
        while (fa) {
            const int a = __ffs((int)fa) - 1;
            fa &= fa - 1u;
            const RowPrep &q = prep[warp * 32 + g + a];
            const double ct = q.ct, st = q.st, xf = q.xf, yf = q.yf;
#pragma unroll 1
            for (int s0 = 0; s0 < S2; s0 += 32) {
                const int s = s0 + lane;
                bool hit = false;
                if (s < S2) {
                    const int i = s / S, j = s - i * S;
                    const double X = p.off_c[j], Y = p.off_c[i];
                    const double stY = st * Y, ctY = ct * Y;
                    const double rx = ct * X - stY;
                    const double ry = st * X + ctY;
                    int ix = round_half_even(rx + xf), iy = round_half_even(ry + yf);
                    ix = wrap1(ix, W); iy = wrap1(iy, H);
                    hit = rock_hit(q, ix, iy);
                }
                const uint32_t b = __ballot_sync(0xffffffffu, hit);
                const int sh = li * S - s0;                        // this lane's row starts at sample li * S of the window
                if (lane_on && la == a && sh > -S && sh < 32)
                    rb |= (sh >= 0 ? (b >> sh) : (b << -sh)) & ((1u << S) - 1u);
            }
        }
        return rb;
    };
    uint4 lo[UNR], hi[UNR];
    uint32_t cell[UNR];
#pragma unroll 1
    for (int g = 0; g < 32; g += G) {                              // one chunk of G ants: loads, decode, flush
        const int64_t i0 = wbase + g;
        if (i0 >= ant_end) break;
        const int n_in = (ant_end - i0 < G) ? (int)(ant_end - i0) : G;
        const uint32_t amask = (n_in * S >= 32) ? 0xffffffffu : ((1u << (n_in * S)) - 1u);   // the lanes with a row
        if (!kLateWait) {
            if (lane == 0) bulk_store_wait_read<kRowsTiles - 1>();
            __syncwarp();
        }
        const bool row_on = lane_on && la < n_in;
        const RowPrep &q = prep[warp * 32 + g + (row_on ? la : 0)];
        const uint32_t fa = ROCKS ? ((rock_ants >> g) & ((1u << G) - 1u)) : 0u;             // warp-uniform
        uint32_t rb = 0u;
        int cnt;
        if (UNR >= S) {
            // the record loads first, the (rare) rock evaluation while they are in flight, then the decode
            if (row_on) row_body(q, offY, mrow, orow_s, amask, lo, hi, cell, 0, 0u);
            if (fa) rb = rock_rows(g, fa);
            cnt = row_on ? row_body(q, offY, mrow, orow_s, amask, lo, hi, cell, 1, rb) : 0;
        } else {
            if (fa) rb = rock_rows(g, fa);
            cnt = row_on ? row_body(q, offY, mrow, orow_s, amask, lo, hi, cell, 2, rb) : 0;
        }
        if (row_on) s_rowcnt[(warp * 32 + g + la) * S + li] = (uint8_t)cnt;
        flush(wobs0, i0, n_in);
    }
    __syncwarp();

    // ---- phase C: reward epilogue, thread per ant (this warp's own ants)
    {
        const int64_t i = base + tid;
        if (i < ant_end) {
            int count = 0;
            if (explore_on) {
#pragma unroll
                for (int k = 0; k < S; ++k) count += s_rowcnt[tid * S + k];
            }
            const double r_other = prep[tid].r_other, r_mult = prep[tid].r_mult;
            const int rs_prev = prep[tid].rs_prev;
            double reward;
            if (p.reward_kind == 1) {
                reward = (double)count / 10.0;                                 // reward_custom.py:19
            } else if (p.reward_kind == 0) {
                reward = 0.0;
                if (explore_on) reward += ((double)count / 10.0) * r_mult;     // :89-94
                reward += r_other;                                             // :106
            } else {
                reward = r_other;
            }
            p.rewards[i] = reward;
            if (reward_out != nullptr) reward_out[i] = reward;
            if (is_step) {                                                     // ants.py:119-121 (Q16)
                int rs = rs_prev;                                              // (loaded in phase A)
                rs += ((reward - p.reward_threshold) > 0.0) ? 255 : 0;
                p.reward_state[i] = (uint8_t)(rs > 255 ? 255 : rs);
            }
        }
    }
    if (lane == 0) bulk_store_wait_read();   // smem must stay valid until the last bulk store has read it
}

}  // namespace ants
