/* mfmarl_batched.h -- batched, device-resident C ABI of the B200 battle engine (new; the reference has
 * no batched interface -- SURVEY.md section 8b "Batched extension").
 *
 * One engine steps E independent environments in lockstep.  State lives in HBM for the life of the
 * engine.  Observation / action / result buffers are caller-owned DEVICE memory (e.g.
 * torch.Tensor.data_ptr()), passed as plain pointers with the shapes stated below; `stream` is a
 * cudaStream_t passed as void* (NULL = default stream).  For E = 1 and rng_mode = MFB_RNG_MINSTD the
 * results are bit-identical to the single-env ABI of mfmarl_magent.h and hence to the reference engine
 * (GridWorld.cc:303-426,430-496,498-694,696-728,760-770).
 *
 * Every function returns 0 on success, -1 on error (message from mfb_last_error()); nothing aborts.
 */
#ifndef MFMARL_BATCHED_H
#define MFMARL_BATCHED_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mfb_engine mfb_engine;

enum { MFB_RNG_MINSTD = 0, MFB_RNG_PHILOX = 1, MFB_RNG_INJECT = 2 };

typedef struct mfb_config {
    int n_envs;            /* E: environments owned by this engine (this GPU's shard)               */
    int map_width, map_height;
    int capacity;          /* agent slots per group (rounded up to a multiple of 4)                 */
    int embedding_size;    /* 10 for battle                                                          */
    int rng_mode;          /* attack-order shuffle: MINSTD = reference parity, PHILOX = production   */
    unsigned seed;
    int env_base;          /* global id of env 0 (keys Philox, so results do not depend on sharding) */
    int max_steps;         /* with auto_reset: episode horizon (0 = none)                            */
    int auto_reset;        /* re-place the armies when an episode ends (done or horizon)             */
    int device;            /* CUDA device ordinal, -1 = current                                      */
    int step_threads;      /* 0 = auto                                                               */
    int obs_tile_agents;   /* agents per observation CTA, 0 = auto: clamp(capacity, 64, 256)         */
    int obs_record;        /* per-env observation record kept by k_step for k_obs: -1 = auto (on for
                              capacity >= 256), 0 = off, 1 = on; same observations either way          */
    int concurrent_step_envs; /* pipelined use: envs of a sibling engine whose mfb_step runs on another stream while
                              this engine's mfb_observe streams; the observation kernel then leaves SM slots free
                              where a step CTA does not fit beside it (0 = not pipelined)                     */
    int random_sides;      /* with auto_reset: every env draws per episode (Philox keyed by seed, env, episode)
                              whether the two armies swap their starting blocks AND ids -- generate_map picks
                              the left army with random.randint(0, 1) each round (senario_battle.py:14) and
                              the block added first gets the low ids                                       */
    /* agent type (python/magent/builtin/config/battle.py:16-29) and the attack reward rules (:41-42) */
    float hp, speed, view_radius, attack_radius, damage, step_recover, kill_supply;
    float step_reward, kill_reward, dead_penalty, attack_penalty, attack_bonus[2];
} mfb_config;

int mfb_default_config(mfb_config *cfg);                 /* battle defaults, E = 1, 40x40, cap 64    */
int mfb_create(const mfb_config *cfg, mfb_engine **out);
int mfb_destroy(mfb_engine *eng);

/* episode set-up: the same placement goes to every env (GridWorld::reset / add_agents "custom") */
int mfb_reset(mfb_engine *eng);
int mfb_add_walls(mfb_engine *eng, int n, const int *xs, const int *ys);             /* host arrays */
int mfb_add_agents(mfb_engine *eng, int group, int n, const int *xs, const int *ys,  /* host arrays */
                   int *n_added);
/* A placement of its own for every env: xs / ys are host arrays [n_envs][n].  As in the reference, a position that
 * is occupied, a wall or out of range is skipped -- per env (GridWorld.cc:180-187) -- and ids are handed out per env
 * in add order, so the envs may hold different numbers of agents.  n_added (may be NULL) receives [n_envs] counts.
 * Once used, mfb_add_agents / mfb_add_walls apply to every env's own template; auto_reset re-places each env from
 * ITS template. */
int mfb_add_agents_per_env(mfb_engine *eng, int group, int n, const int *xs, const int *ys, int *n_added);
int mfb_set_seed(mfb_engine *eng, unsigned long seed);

/* sizes: key in {"capacity","n_envs","n_action","view_size","n_channel","feature_size","attack_base"} */
int mfb_query(mfb_engine *eng, const char *key, int *out);

/* K1.  d_view float[E][2][cap][13][13][7], d_feature float[E][2][cap][feature_size]; rows >= num are
 * not written.  group_mask: 1 = group 0 only, 2 = group 1 only, 3 = both.                           */
int mfb_observe(mfb_engine *eng, float *d_view, float *d_feature, int group_mask, void *stream);

/* K1 with one output block PER GROUP, each [E][cap][...] and contiguous -- the layout a per-group policy network
 * consumes without a gather (senario_battle.py:100-111 feeds models[g] its own group's rows).  A NULL view pointer
 * skips that group. */
int mfb_observe_groups(mfb_engine *eng, float *d_view0, float *d_feature0, float *d_view1, float *d_feature1,
                       void *stream);

/* K1 with bf16 rows in the layout a bf16 channels-last policy network consumes directly:
 *   d_viewG  __nv_bfloat16[E][cap][13][13][8]: the 7 channels of mfb_observe_groups rounded to nearest-even bf16,
 *            channel 7 = 0 (a cell is one 16-byte vector); d_featureG stays float[E][cap][feature_size].
 * Same values as casting the fp32 observation (tests compare bit for bit); 2840 instead of 4868 bytes per agent. */
int mfb_observe_groups_bf16(mfb_engine *eng, void *d_view0, float *d_feature0, void *d_view1, float *d_feature1,
                            void *stream);

/* K2, fused set_action(g0), set_action(g1), step, get_reward, get_alive, mean action, clear_dead.
 *   d_actions      int32[E][2][cap]       in
 *   d_attack_perm  int32[E][2*cap]        in, only for MFB_RNG_INJECT (else NULL)
 *   d_reward       float[E][2][cap]       out, indexed like the observation rows of this step
 *   d_alive        uint8[E][2][cap]       out
 *   d_mean_action  float[E][2][n_action]  out (senario_battle.py:141), may be NULL
 *   d_done         int32[E]               out
 * clear_dead: 1 = compact survivors in the same launch (the play loop's order), 0 = leave the dead
 * in the lists (then call mfb_clear_dead).                                                          */
int mfb_step(mfb_engine *eng, const int32_t *d_actions, const int32_t *d_attack_perm, float *d_reward,
             uint8_t *d_alive, float *d_mean_action, int32_t *d_done, int clear_dead, void *stream);
int mfb_clear_dead(mfb_engine *eng, void *stream);

/* K5 standalone: out[r][b] = #{i < num[r] : actions[r][i] == b} / num[r]   (senario_battle.py:141,255) */
int mfb_mean_action(const int32_t *d_actions /* [rows][cap] */, const int32_t *d_num /* [rows] */,
                    float *d_out /* [rows][n_action] */, int rows, int cap, int n_action, void *stream);

/* K7: neighbourhood mean action per agent, the local form of the mean action of mean-field MARL:
 * a_bar_i = 1/N_i sum_{j in N(i)} onehot(a_j).  For every listed slot i < num[e][g] (a dead agent still listed
 * before clear_dead included), N(i) = the agents j != i of the SAME group, j < num[e][g], that are alive, have acted
 * (last_action < n_action; it is n_action after a placement or an auto-reset) and stand at an offset
 * pos_j - pos_i inside the disc CircleRange(radius, 0, 1) of Range.h:171-215 (radius cast to float, distances in
 * double, no wrap-around).  out[b] = (float)count_b / (float)|N(i)| rounded to nearest; a row with |N(i)| = 0 is all
 * zeros (the zero initial mean action of senario_battle.py:93), and so are rows >= num.  Called after
 * mfb_step(..., clear_dead = 1) its rows line up with the next observation's rows.
 *   radius    0 < radius <= view_radius (6 for battle); anything else, NaN included, is an error and launches nothing
 *   d_outG    float[E][cap][n_action] per group, 16-byte aligned -- the row layout of mfb_observe_groups; NULL skips
 *             that group
 * Reads the engine state only (no RNG, no state change); a pending placement is committed first. */
int mfb_local_mean_action(mfb_engine *eng, double radius, float *d_out0, float *d_out1, void *stream);

/* state read-back into HOST buffers (synchronises `stream`): key in
 *   "num" int32[E][2], "dead_ct" int32[E][2], "pos" int32[E][2][cap][2], "hp" float[E][2][cap],
 *   "id" int32[E][2][cap], "alive" uint8[E][2][cap], "last_action" int32[E][2][cap],
 *   "step_ct" int32[E], "rng" uint32[E], "agent_steps" uint64[E] (agents stepped since creation),
 *   "side" int32[E] (1 = armies swapped this episode, random_sides), "episode" int32[E]              */
int mfb_get(mfb_engine *eng, const char *key, void *host_buf, void *stream);
/* device pointer to the live int32[E][2] agent counts (for masking on the device) */
int mfb_num_device_ptr(mfb_engine *eng, const int32_t **out);

/* device pointers to live engine state, valid until mfb_destroy (read-only for the caller; they change with every
 * launch on the engine's stream; a placement made by mfb_add_agents reaches the device with the next launch or
 * mfb_get): "num" int32[E][2], "id" int32[E][2][cap], "pos" int32[E][2][cap] (x | y << 16),
 * "hp" float[E][2][cap], "step_ct" int32[E] */
int mfb_state_device_ptr(mfb_engine *eng, const char *key, const void **out);

/* Host-buffer convenience used for the end-to-end measurement: pinned-host actions in, results out.
 * Copies h_actions -> device, runs mfb_step (clear_dead = 1), copies the results back, synchronises. */
int mfb_step_host(mfb_engine *eng, const int32_t *h_actions, float *h_reward, uint8_t *h_alive,
                  float *h_mean_action, int32_t *h_done, void *stream);

/* Pipelined variant: returns as soon as the work is enqueued.  The action upload runs on an internal copy
 * stream (so it overlaps kernels already queued on `stream`, e.g. mfb_observe), k_step runs on `stream`, and
 * the results are copied to the pinned host buffers on a second copy stream (overlapping the next
 * mfb_observe).  Two internal staging sets alternate: *ticket (0/1) names the one used; the host buffers
 * of a call are valid after mfb_host_wait(eng, ticket) and must not be reused before it. */
int mfb_step_host_async(mfb_engine *eng, const int32_t *h_actions, float *h_reward, uint8_t *h_alive,
                        float *h_mean_action, int32_t *h_done, void *stream, int *ticket);
int mfb_host_wait(mfb_engine *eng, int ticket);

/* Device memory for large, mostly-zero output blocks such as the observation rows.  Where the GPU supports generic
 * compression (CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED) the block is a cuMemCreate allocation with
 * CU_MEM_ALLOCATION_COMP_GENERIC: the L2 compresses its lines on the way to DRAM, losslessly and invisibly to loads and
 * stores, so sparse rows cost fewer HBM bytes to write.  Elsewhere, or when the driver grants no compression, it is a
 * plain cudaMalloc, and so is a block the driver has no compressible memory left for.  *compressed tells which
 * (1 / 0).  The block is zeroed, and the call synchronises the device.  mfb_free_device synchronises the whole device
 * before it releases a block, so it must not run while a stream is capturing a CUDA graph; it accepts NULL and nothing
 * else that mfb_alloc_device did not return. */
int mfb_alloc_device(unsigned long bytes, int device, void **ptr, int *compressed);
int mfb_free_device(void *ptr);

const char *mfb_last_error(void);

/* ---- K6: Ising tabular mean-field Q-learning, one fused sweep over a batch of lattices -----------------
 * Replaces the loop body of main_MFQ_Ising.py:105-134 (Boltzmann action per site from Q[i, s, :] with
 * s = up-neighbour count on the old lattice, spin <- action, reward on the new lattice
 * (examples/ising_model/Ising.py:101-111), Q[i,s,a] += lr (r - Q[i,s,a])) for `n_lattices` independent
 * side x side tori.  All pointers are DEVICE memory.
 *   dtype          0 = fp32 (production), 1 = fp64 (the reference's precision; used for trajectory parity)
 *   d_spins        int8 [n_lattices][side][side]      in/out, values {0, 1}
 *   d_q            T    [n_lattices][5][side*side][2]  in/out, entry (s, a) of site i at ((s*N + i)*2 + a)
 *   d_uniforms     T    [n_lattices][side*side] or NULL: injected uniforms (test hook; a = [u >= p0]);
 *                  NULL = Philox4x32-10, key (seed, lattice_base + lattice), counter (column, row / 4, step, 0);
 *                  output word row % 4 is the site's draw, u = that word (rounded toward zero to 24 bits) / 2^32
 *   d_update_mask  uint8[n_lattices][side*side] or NULL: the act group (act_rate < 1); NULL = all sites
 *   d_n_up         int32[n_lattices]  out: up spins after the sweep (order parameter = |2 up - N| / N)
 *   d_reward_sum,
 *   d_mse          T    [n_lattices]  out (may be NULL): sum of rewards; mse vs reward_target / N
 * Returns 0, or -1 with the message in mfb_last_error(). */
int mfi_step(int dtype, int n_lattices, int side, int8_t *d_spins, void *d_q, double temperature, double lr,
             const void *d_uniforms, const uint8_t *d_update_mask, unsigned seed, unsigned lattice_base,
             unsigned step, int32_t *d_n_up, void *d_reward_sum, void *d_mse, void *stream);

/* K6r / K6p / K6s: `n_sweeps` sweeps in ONE launch with the Q table resident in shared memory.  A lattice is split into
 * strips of rows, one CTA each.  For the fp32 sides 64, 128, 256 (strips of 16 rows) and 512 (strips of 8 rows) the
 * strips are ordinary CTAs of a persistent, cooperatively launched grid that fills the GPU (144 of 148 SMs at side 256)
 * and exchange their halo rows through L2 (K6s; MFMARL_ISING_PERSIST=1 selects its predecessor K6p at 128 / 256); other
 * shapes, and MFMARL_ISING_PERSIST=0, use a thread-block cluster of mfi_resident_cluster_size() CTAs per lattice (K6r:
 * 1 for side <= 64, 4 for 128, 16 for 256 in fp32; mfi_resident_cluster_size(fp32, 512) = 64 is K6s's strip count).  Either way: same semantics and the same Philox keys as
 * n_sweeps calls of mfi_step with step = step0 .. step0+n_sweeps-1 (bit-identical results); the Q table is read and
 * written once per launch.
 *   d_temperatures  T    [n_sweeps]                          in (the schedule of main_MFQ_Ising.py:108-112)
 *   d_uniforms      T    [n_sweeps][n_lattices][side*side]   or NULL (test hook)
 *   d_update_mask   uint8[n_sweeps][n_lattices][side*side]   or NULL: the act group of every sweep (act_rate < 1)
 *   d_n_up          int32[n_sweeps][n_lattices]              out, MUST be zeroed by the caller
 *   d_reward_sum    T    [n_sweeps][n_lattices]              out or NULL, MUST be zeroed by the caller
 * mfi_resident_cluster_size returns 0 when the shape is not supported (then loop over mfi_step). */
int mfi_resident_cluster_size(int dtype, int side);
int mfi_run(int dtype, int n_lattices, int side, int n_sweeps, int8_t *d_spins, void *d_q,
            const void *d_temperatures, double lr, const void *d_uniforms, const uint8_t *d_update_mask, unsigned seed,
            unsigned lattice_base, unsigned step0, int32_t *d_n_up, void *d_reward_sum, void *stream);

/* The Ising ENVIRONMENT interface (examples/ising_model/multiagent/environment.py:49-92 `_step` / `_reset`,
 * multiagent/core.py:99-125 `IsingWorld.step`, Ising.py:101-118 reward / observation) for callers that bring their
 * own policy, e.g. the unmodified main_MFQ_Ising.py over python/examples/ising_model (same package layout as the
 * reference).  All pointers are DEVICE memory; N = side * side.
 *   d_spins    int8 [n_lattices][N]      in/out
 *   d_actions  int32[n_lattices][N] or NULL: spin_i <- (action_i <= 0 ? 0 : 1) first (environment.py:112-114);
 *              NULL = observe the lattice as it is (`_reset`)
 *   d_obs      uint8[n_lattices][N][4] or NULL: the 4 torus neighbours' spins, ascending flat index of the
 *              neighbour -- the order of global_state.flatten()[np.where(spin_mask == 1)] (Ising.py:113-118)
 *   d_reward   float[n_lattices][N] or NULL: 0.5 * sigma_i * sum_nbr sigma_j on the new lattice (Ising.py:101-111)
 *   d_n_up     int32[n_lattices] or NULL: up spins (order parameter |2 up - N| / N, core.py:106-110) */
int mfi_env_step(int n_lattices, int side, int8_t *d_spins, const int32_t *d_actions, uint8_t *d_obs,
                 float *d_reward, int32_t *d_n_up, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MFMARL_BATCHED_H */
