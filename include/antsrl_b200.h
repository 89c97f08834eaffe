/*
 * antsrl_b200.h -- C ABI of libantsrl_b200.so: the AntsRL environment step loop as sm_100a CUDA kernels over a
 * batch of E independent environments held in structure-of-arrays layout in HBM.
 *
 * The reference (SelennLamson/AntsRL) has no FFI; its boundary for this path is the Python object surface
 *   RLApi.observation()            environment/RL_api.py:96-165
 *   RLApi.step(rotation, phero)    environment/RL_api.py:168-204
 *   Environment.update()           environment/environment.py:42-47  (dispatching Walls/CircleObstacles/
 *                                  Pheromone/Ants/Anthill.update: walls.py:22-30, circle_obstacles.py:32-58,
 *                                  pheromone.py:43-45, ants.py:123-130, anthill.py:41-46)
 *   Ants.activate_all_pheromones() environment/ants.py:86-87
 *   reward.observation()/step()    environment/rewards/reward_custom.py:17-22,37-40,79-106; reward.py:29-38
 * Each entry point below names the reference method it replaces.  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.  All functions return 0 on success and a negative ANTS_E_* code on
 * failure; ants_last_error() returns the message of the last failure on the calling thread.  A handle is bound
 * to one CUDA device and one stream and is not thread-safe.  There is no CPU fallback: without a CUDA device
 * ants_create fails with ANTS_E_CUDA.
 *
 * Index conventions: ants arrays are [E][N]; planes are [E][W][H] with the reference's [x][y] order (y
 * contiguous); pheromone planes [E][P][W][H]; activation [E][N][P]; rocks [E][R](x,y).  Host arrays are
 * dense (no pitch); the library pads rows in HBM internally.
 */
#ifndef ANTSRL_B200_H
#define ANTSRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ANTS_ABI_VERSION 1
#define ANTS_MAX_PHERO 4
#define ANTS_MAX_CHANNELS 16
#define ANTS_MAX_RADIUS 7            /* perception window (2r+1)^2 <= 225 samples */
#define ANTS_MAX_SAMPLES 225
#define ANTS_MAX_ROCKS 64
#define ANTS_MAX_ANTS 65535          /* ant index is packed in 16 bits of the ownership stamp */

enum { ANTS_OK = 0, ANTS_E_ARG = -1, ANTS_E_CUDA = -2, ANTS_E_STATE = -3, ANTS_E_ALLOC = -4 };

/* perceived_objects entries, RL_api.py:123-142 */
enum { ANTS_CH_ANTS = 0, ANTS_CH_PHERO = 1, ANTS_CH_ANTHILL = 2, ANTS_CH_WALLS = 3, ANTS_CH_FOOD = 4,
       ANTS_CH_ROCKS = 5 };
/* reward_custom.py: All_Rewards (:43), ExplorationReward (:8), Food_Reward (:28) */
enum { ANTS_REWARD_ALL = 0, ANTS_REWARD_EXPLORE = 1, ANTS_REWARD_FOOD = 2 };
/* pheromone field maintenance (DIFFUSE_FACTOR == 0; a non-zero factor always runs the dense stencil):
 *   DENSE        a pass over every cell each update, exactly pheromone.py:43-45
 *   ACTIVE_TILES the same arithmetic, only over 16x16 tiles that hold pheromone (bit-identical to DENSE)
 *   LAZY         no pass at all: each value carries the update index at which it was written and is decayed when
 *                read (saturated max_val deposits through a table with the reference's exact rounding, other
 *                values as v * (1-EVAP)^k, ~1e-13 relative from the repeated product) */
enum { ANTS_EVAP_DENSE = 0, ANTS_EVAP_ACTIVE_TILES = 1, ANTS_EVAP_LAZY = 2 };

/* map cell record in HBM:
 *   F64      { f64 phero[P]; f64 food; u32 meta; u8 wall; timestamps }  32 B (P <= 2) / 64 B: every evap mode
 *   COMPACT  { f32 phero0; f32 phero1; f32 food; 4 x u8 stamps }        16 B: two cells per DRAM sector.  Needs
 *            ANTS_EVAP_LAZY, P <= 2 and no diffusion.  Saturated (max_val) deposits stay bit-exact through the
 *            decay table; other pheromone values and non-integer food are rounded to f32 (6e-8 relative). */
/*   COMPACT8 { u16 phero0; u16 phero1; u16 food; 2 x u8 stamps }             8 B: four cells per DRAM sector.  Same
 *            requirements as COMPACT.  A pheromone code is a boxed saturated deposit (15-bit update index, decoded
 *            through the decay table: bit-exact) or an escape to a side array holding the plain f32 value; food is an
 *            integer count 0..65534 (what the reference's maps hold) or an escape to the side array. */
enum { ANTS_REC_F64 = 0, ANTS_REC_COMPACT = 1, ANTS_REC_COMPACT8 = 2 };

typedef struct AntsConfig {
    int32_t abi_version;             /* must be ANTS_ABI_VERSION */
    int32_t device;                  /* CUDA device ordinal */
    int32_t n_envs, n_ants, w, h;    /* E, N, W, H */
    int32_t n_phero, n_rocks;        /* P <= ANTS_MAX_PHERO, R <= ANTS_MAX_ROCKS */
    int32_t max_time;                /* Environment.max_time, environment.py:26 */
    /* perception, RLApi.setup_perception RL_api.py:80-93 */
    int32_t radius;
    int32_t has_mask;
    uint8_t mask[ANTS_MAX_SAMPLES];  /* row-major (2r+1)x(2r+1), 1 = visible */
    int32_t n_channels;
    int32_t channel_kind[ANTS_MAX_CHANNELS];
    int32_t channel_arg[ANTS_MAX_CHANNELS];   /* pheromone index for ANTS_CH_PHERO */
    double delta;                    /* DELTA = 1.1, RL_api.py:15 */
    double fwd_delta;                /* perception_fwd_delta */
    /* RLApi.__init__, RL_api.py:23 */
    double reward_threshold, max_speed, max_rot_speed, carry_speed_reduction, backward_speed_reduction;
    /* reward, reward_custom.py:44-50 */
    int32_t reward_kind;
    double reward_factors[5];        /* fct_explore, fct_food, fct_anthill, fct_explore_holding, fct_headinganthill */
    /* pheromone.py:5-10, environment_generator.py:93,97 */
    double diffuse_factor, evap_factor;
    int32_t has_max_val;
    double phero_max_val;
    double max_hold;
    /* collision noise when no tape is passed to ants_update: Philox4x32-10 keyed by
     * (rng_seed, env_id_base + e, timestep, ant) -- results do not depend on how envs are sharded */
    uint64_t rng_seed;
    int64_t env_id_base;
    int32_t evap_mode;               /* ANTS_EVAP_* */
    int32_t record_format;           /* ANTS_REC_* */
    int32_t reserved[6];
} AntsConfig;

/* Host-side SoA view of the whole batch for import/export.  NULL members are skipped. */
typedef struct AntsHostState {
    double *x, *y, *theta;                    /* Ants.ants, ants.py:27          [E][N] */
    double *prev_x, *prev_y, *prev_theta;     /* Ants.prev_ants, ants.py:30     [E][N] */
    double *holding, *seed;                   /* ants.py:37,41                  [E][N] */
    double *activation;                       /* Ants.phero_activation          [E][N][P] */
    uint8_t *mandibles, *reward_state;        /* ants.py:36,38                  [E][N] */
    double *rw_holding_prev, *rw_prev_dist, *rewards;   /* reward_custom.py:52-60   [E][N] */
    uint8_t *explored;                        /* explored_map, reward_custom.py:68   [E][W][H] */
    uint8_t *walls;                           /* Walls.map, walls.py:16         [E][W][H] */
    double *phero;                            /* Pheromone.phero, pheromone.py:28    [E][P][W][H] */
    double *food;                             /* Food.qte, food.py:15           [E][W][H] */
    int32_t *anthill_xyr;                     /* Anthill.x,y,radius anthill.py:22-24 [E][3] */
    double *anthill_food;                     /* Anthill.food, anthill.py:27    [E] */
    double *rock_centers, *rock_radii, *rock_weights;   /* circle_obstacles.py:22-24 [E][R][2],[E][R],[E][R] */
    /* batch-wide scalars.  On import: timestep <= 0, rw_alias < 0, act_bool < 0 leave the handle's value untouched */
    int64_t timestep;                         /* Environment.timestep, environment.py:27 (all envs in lockstep) */
    int32_t rw_alias;                         /* reward still aliases Ants.holding, reward_custom.py:66-67 */
    int32_t act_bool;                         /* phero_activation still has bool dtype, ants.py:83 */
} AntsHostState;

typedef struct AntsStats {
    int64_t steps, updates, observations;
    int64_t kernel_launches;                  /* kernels launched by this handle so far */
    int64_t active_tiles;                     /* pheromone tiles processed by the last update (tile mode) */
    int64_t total_tiles;
    int64_t food_commits, absorb_events;      /* of the last step / update */
    int64_t device_bytes;                     /* HBM held by the handle */
    int64_t e2e_dense_permille;               /* ants_step_host: share of the ants (in 1/1000) the DMA engine copies dense while
                                                 the host threads expand the packed rest (follows the slower side) */
} AntsStats;

typedef struct AntsBatch AntsBatch;

int ants_abi_version(void);
const char *ants_last_error(void);

/* Environment.__init__ + EnvironmentGenerator.generate's object construction, for E envs at once. */
int ants_create(const AntsConfig *cfg, AntsBatch **out);
int ants_destroy(AntsBatch *b);
/* run on an existing cudaStream_t (e.g. torch's current stream; NULL = the legacy default stream).  A new
 * handle runs on its own non-blocking stream until this is called. */
int ants_set_stream(AntsBatch *b, void *cuda_stream);
int ants_synchronize(AntsBatch *b);

/* state in / out (host pointers, dense layout).  Also how reference-generated maps reach the GPU. */
int ants_import_state(AntsBatch *b, const AntsHostState *s);
int ants_export_state(AntsBatch *b, AntsHostState *s);
/* the same for the envs [env0, env0 + n_envs) only: the host arrays hold n_envs environments.  This is what
 * Environment.save_state() (environment.py:36-40: a visualize_copy of every object, pickled by main.py:139-147 for
 * the viewer) needs for ONE environment of a large batch without moving the other E - 1. */
int ants_export_env_state(AntsBatch *b, int32_t env0, int32_t n_envs, AntsHostState *s);
/* ... and the import of such a window: a new map / new ants for the envs [env0, env0 + n_envs) only (main.py:66-79
 * generates a new environment per episode), or a large batch uploaded in slices.  The scalars stay batch-wide. */
int ants_import_env_state(AntsBatch *b, int32_t env0, int32_t n_envs, const AntsHostState *s);
/* With DIFFUSE_FACTOR != 0 the sign bit of a pheromone plane value is the wall flag of its cell, so negative and NaN
 * pheromone values cannot be represented there (the reference allows them): ants_import_env_state returns ANTS_E_ARG
 * for such an activation before it uploads anything, and for such a pheromone value after the window's import has
 * run -- the window must then be imported again. */
/* A new episode's map for the envs [env0, env0 + n_envs), written on the device from the generator's random draws
 * instead of dense planes (EnvironmentGenerator.generate, environment_generator.py:60-72, with CirclesGenerator walls
 * and food).  Host arrays: anthill_xyr [n_envs][3], wall_discs [n_envs][n_wall_discs][3], food_discs
 * [n_envs][n_food_discs][3] of (xc, yc, r).  A cell is a wall iff some wall disc has (x-xc)^2 + (y-yc)^2 <= r^2 and the
 * cell lies outside the anthill disc; its food is 1.0 iff some food disc covers it and it is not a wall; pheromones,
 * explored and occupancy are 0.  Afterwards the envs are in the state an import of food, walls, explored, pheromones
 * and anthill leaves (the first update sweeps the anthill disc); the ants, rocks, anthill store and batch scalars are
 * not touched: ants_import_env_state uploads those (kilobytes per env).  ANTS_E_ARG, with the handle unchanged, for a
 * window outside the batch, a negative count or radius, or a disc that does not lie inside the map. */
int ants_generate_env_maps(AntsBatch *b, int32_t env0, int32_t n_envs, const int32_t *anthill_xyr, int32_t n_wall_discs,
                           const int32_t *wall_discs, int32_t n_food_discs, const int32_t *food_discs);

/* A map layer of PerlinGenerator (map_generators.py:9-25, the reference's default walls): env e's layer is set at cell
 * (x, y) iff (double)pnoise2(x', y', octaves, persistence, lacunarity, repeat 1024) > density, with
 * x' = (float)((double)(x + offset_x) / scale) and y' likewise (utils.perlin_noise_generator; the float32 algorithm of
 * antsrl_b200/perlin.py, bit for bit).  The generator's parameters are shared by the envs; the offsets are the two
 * random.randint(-10000, 10000) draws of each env. */
typedef struct AntsPerlinLayer {
    const int32_t *offsets;      /* host [n_envs][2]: (offset_x, offset_y) of each env */
    double scale;                /* x = (float)((double)(cell_x + offset_x) / scale), y likewise */
    double density;              /* a cell is set iff (double)pnoise2(x, y) > density */
    int32_t octaves;             /* 1 ... 32 */
    int32_t reserved;
    double persistence, lacunarity;   /* rounded to float, as pnoise2 does */
} AntsPerlinLayer;
/* ants_generate_env_maps with layers that may be Perlin noise: a layer whose *_perlin pointer is non-NULL is that noise
 * (its disc count must be 0), otherwise it is the discs, exactly as ants_generate_env_maps.  Walls and food follow the
 * same rules (a wall outside the anthill disc; food 1.0 where the food layer is set and the cell is not a wall).
 * ANTS_E_ARG, with the handle unchanged, for what ants_generate_env_maps rejects and for: octaves outside 1 ... 32; a
 * scale that is 0 or not finite; a persistence or lacunarity that is not finite; a layer given both discs and Perlin
 * noise; NULL offsets; an octave whose period 1024 * freq (in float) is 0, not finite or at least 2^31 in magnitude; a
 * map edge whose coordinate x' * freq (in float) is not finite or at least 2^31 in magnitude (the integer parts of the
 * noise stay in int32). */
int ants_generate_env_maps_ex(AntsBatch *b, int32_t env0, int32_t n_envs, const int32_t *anthill_xyr,
                              int32_t n_wall_discs, const int32_t *wall_discs, const AntsPerlinLayer *wall_perlin,
                              int32_t n_food_discs, const int32_t *food_discs, const AntsPerlinLayer *food_perlin);
/* utils.perlin_noise_generator on the device, without a handle: the float32 field pnoise2 (the value before the density
 * threshold, which is ignored) of the n offset pairs of `layer` on a w x h map, written to the DEVICE buffer
 * d_out [n][w][h] on `stream` (a cudaStream_t, NULL = the legacy default stream) of CUDA device `device`; returns when
 * the field is written.  The same device code as the Perlin layers of ants_generate_env_maps_ex, and the same
 * ANTS_E_ARG cases. */
int ants_perlin_noise(int32_t device, const AntsPerlinLayer *layer, int32_t n, int32_t w, int32_t h, float *d_out,
                      void *stream);

/* Ants.activate_all_pheromones, ants.py:86-87.  act: host [E][N][P].  With DIFFUSE_FACTOR != 0, ANTS_E_ARG with the
 * handle unchanged for a negative or NaN activation (the plane's sign bit is the wall flag). */
int ants_activate_all_pheromones(AntsBatch *b, const double *act, int32_t is_bool);

/* RLApi.observation(), RL_api.py:96-165 (side effect on reward state, as the reference).
 * DEVICE pointers: obs f32 [E][N][S][S][C]; agent_state f32 [E][N][2]; state f32 [E][N][2+P] (may be NULL);
 * reward f64 [E][N] (may be NULL). */
int ants_observe(AntsBatch *b, float *d_obs, float *d_agent_state, float *d_state, double *d_reward);

/* RLApi.step(rotation, on_off_pheromones), RL_api.py:168-204.  DEVICE pointers; d_rot / d_ph int8 [E][N] or
 * NULL (= the reference's None: leave heading / activation unchanged).  *done (host) = max_time == timestep. */
int ants_step(AntsBatch *b, const int8_t *d_rot, const int8_t *d_ph, float *d_obs, float *d_agent_state,
              double *d_reward, int32_t *done);

/* Environment.update(), environment.py:42-47.  d_noise: DEVICE f64 [E][N] uniforms in [0,1) replacing the
 * np.random.random draw of walls.py:28 (ant a consumes d_noise[e][a] iff it collides), or NULL for Philox. */
int ants_update(AntsBatch *b, const double *d_noise);

/* T x [step(actions_t); update()] with device-resident action tapes [T][E][N] and Philox noise; the outputs
 * of the last step stay in the buffers.  Used by the throughput benchmark (no host round trip per step). */
int ants_rollout(AntsBatch *b, const int8_t *d_rot_tape, const int8_t *d_ph_tape, int32_t n_steps,
                 float *d_obs, float *d_agent_state, double *d_reward);

/* The exploration branch of the reference's agents (agents/collect_agent.py:172-177: rotation = randint(0,
 * n_rotations) - n_rotations // 2, pheromone = randint(0, n_pheromones) per ant) drawn on the device into DEVICE
 * int8 [E][N] buffers (either may be NULL), so a random-agent episode needs no host round trip.  Philox4x32-10
 * keyed by (seed, env_id_base + e, timestep, ant): the draws do not depend on how envs are sharded. */
int ants_sample_actions(AntsBatch *b, uint64_t seed, int32_t n_rotations, int32_t n_pheromones, int8_t *d_rot,
                        int8_t *d_ph);

/* Host-buffer variants (the reference-facing path: numpy in, numpy out).  Buffers obtained from
 * ants_host_alloc are pinned and are copied to/from directly; other host memory is staged. */
void *ants_host_alloc(uint64_t bytes);
int ants_host_free(void *p);
int ants_observe_host(AntsBatch *b, float *h_obs, float *h_agent_state, float *h_state, double *h_reward);
int ants_step_host(AntsBatch *b, const int8_t *h_rot, const int8_t *h_ph, float *h_obs, float *h_agent_state,
                   double *h_reward, int32_t *done);
int ants_update_host(AntsBatch *b, const double *h_noise);

/* ---- packed observations: what crosses PCIe on the host-buffer path.
 * The dense observation is 4 C bytes per sample (1372 B per ant for the generator's 7x7x7 window); only the visible
 * samples carry information (environment_generator.py:35-41 masks 12 of 49 to the constant -1, RL_api.py:147-148), the
 * ants / anthill / walls / rocks channels are 0/1 (RL_api.py:128-142) and the food channel holds integer counts.  Packed
 * form, per ant: n_visible samples of 12 bytes { f32 value_channel[0]; f32 value_channel[1]; u16 food; u8 flags; u8 0 }
 * (flags bit k = flag_channel[k]); ants_unpack_obs rebuilds the dense (N, S, S, C) f32 array bit for bit on host
 * threads.  ants_step_host uses this transport internally (same signature, same result, ~3x fewer PCIe bytes);
 * ants_step_host_packed hands the packed buffer to the caller, who expands all of it, part of it or none. */
typedef struct AntsPackedLayout {
    int32_t supported;               /* 0: this configuration has no packed form (more than two pheromone channels, ...) */
    int32_t n_samples, n_channels;   /* S*S, C of the dense observation */
    int32_t n_visible;               /* samples per ant in the packed form */
    int32_t sample_bytes;            /* 12 */
    int64_t bytes_per_ant;           /* n_visible * sample_bytes */
    int32_t flag_channel[8];         /* dense channel behind bit k of the flags byte, -1 = unused */
    int32_t value_channel[2];        /* dense channels stored as f32 (pheromones), -1 = unused */
    int32_t food_channel;            /* dense channel stored as u16 count, -1 = none */
    uint8_t visible_index[228];      /* row-major sample index of packed sample v */
} AntsPackedLayout;
/* pure function of the configuration (needs no device) */
int ants_packed_layout(const AntsConfig *cfg, AntsPackedLayout *out);
/* RLApi.step with host buffers; the observation arrives packed: h_packed holds E*N*bytes_per_ant (+16) bytes.  Returns
 * ANTS_E_STATE if a value of this step has no packed form (a non-integer amount of food): use ants_step_host then. */
int ants_step_host_packed(AntsBatch *b, const int8_t *h_rot, const int8_t *h_ph, void *h_packed, float *h_agent_state,
                          double *h_reward, int32_t *done);
/* packed -> dense for n_ants consecutive ants, on n_threads host threads (0 = all cores).  Host code only. */
int ants_unpack_obs(const AntsPackedLayout *layout, const void *h_packed, int64_t n_ants, float *h_obs, int32_t n_threads);

int ants_get_stats(AntsBatch *b, AntsStats *out);
/* time (ms) spent by the named kernel family since the last reset, measured with CUDA events on the handle's
 * stream when profiling is enabled with ants_set_profiling(b, 1): "perceive", "env_move", "env_update",
 * "env_update_move" (block-per-environment kernels), "evaporate", "absorb", "misc", "pack", "reset"
 * (ants_generate_env_maps); and for handles on the
 * flat kernels (non-lazy field, > 1024 ants per env) "move", "food_commit", "collide", "rocks", "deposit" */
int ants_set_profiling(AntsBatch *b, int32_t on);
int ants_get_kernel_ms(AntsBatch *b, const char *name, double *ms, int64_t *launches);
int ants_reset_kernel_ms(AntsBatch *b);

#ifdef __cplusplus
}
#endif
#endif /* ANTSRL_B200_H */
