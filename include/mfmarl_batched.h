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
    int step_threads;      /* threads per k_step CTA: <= 0 = auto; 33..1024, rounded up to a multiple of 32;
                              1..32 and > 1024 make mfb_create fail with a message naming the value           */
    int obs_tile_agents;   /* agents per observation CTA, 0 = auto: clamp(capacity, 64, 256)         */
    int obs_record;        /* per-env observation record kept by k_step for k_obs: -1 = auto (on for
                              capacity >= 256, and wherever the kernels run from HBM), 0 = off (refused
                              where they run from HBM), 1 = on; same observations either way             */
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
/* Random placement: n agents of `group` go to cells drawn at random inside the rectangle [x0, x0+w) x [y0, y0+h)
 * (w = h = 0: the whole map, i.e. the reference's get_random_blank).  Every env draws its own cells, at the commit
 * that follows this call and again at every auto-reset, so each episode of each env starts from fresh draws.
 *   - The op is appended to the engine's placement program; its n agents take the next n ids in call order, whatever
 *     the draws.  An episode start places the fixed template first, then runs the random ops in call order.  After
 *     mfb_add_agents_per_env they draw around each env's own template.  mfb_add_agents, mfb_add_agents_per_env and
 *     mfb_add_walls after a random op are refused until mfb_reset (a random agent could take a fixed agent's cell).
 *   - A candidate cell is blank when x + 1 < W, y + 1 < H (the reference's is_blank_area bound for a 1x1 body) and it
 *     holds no wall, no fixed agent and no earlier random agent of this episode; candidates are drawn until one is.
 *     MFB_RNG_MINSTD (and INJECT): candidate t is the next two draws r1, r2 of the env's own minstd stream ("rng"),
 *     x = x0 + r1 % w, y = y0 + r2 % h (whole map: r1 % (W - 1), r2 % (H - 1)), and the stream continues from there
 *     into the attack shuffles: at E = 1 with whole-map ops this is add_agents(method="random") of the single-env ABI,
 *     cell for cell and draw for draw.  MFB_RNG_PHILOX: candidate t of op k (k counts the ops since mfb_reset) is
 *     Philox4x32-10 with key (seed, env_base + e) and counter (t, k, episode, generation | 0x80000000), x = x0 +
 *     mulhi(word0, w), y = y0 + mulhi(word1, h); generation counts the mfb_reset calls since mfb_create (a commit sets
 *     episode to 0).  The top bit of word 3 keeps these draws apart from the attack shuffle's counter (i, step, 0, 0)
 *     and random_sides' (episode, 0x51DE, 0, 0) under the same key.
 *   - random_sides: an env that swaps sides swaps the groups of its random ops too, and their ids go with them.
 *   - An agent gives up after W*H + 1 failed candidates (the reference's limit); it and the rest of its op are not
 *     placed, and mfb_get "placement_short" counts them per env (the env's last placement).
 *   - Returns -1 and changes nothing for a group other than 0 or 1, n < 0, a rectangle that leaves the map or has no
 *     interior cell, and an op that cannot fit in some env: fewer blank cells in its rectangle (walls and fixed agents
 *     excluded) than n plus the n of the earlier ops whose rectangles overlap it.  The capacity grows as for
 *     mfb_add_agents. */
int mfb_add_agents_random(mfb_engine *eng, int group, int n, int x0, int y0, int w, int h);
int mfb_set_seed(mfb_engine *eng, unsigned long seed);

/* sizes: key in {"capacity","n_envs","n_action","view_size","n_channel","feature_size","attack_base"}.
 * "state_bytes": R, the size of one env's state record (mfb_save_envs; depends on the capacity only).
 * "hbm_kernels": the kernels that run from HBM at the engine's geometry (map, capacity after the pending placement)
 * because their shared-memory layout exceeds a CTA's: bit 0 k_step, 1 k_obs, 2 k_obs_record, 3 k_local_mean_action.
 * Launch shape: "step_threads" the CTA width k_step launches with (after the auto rules); "obs_record" 1 if the engine
 * keeps the observation record, else 0; "obs_tile" and "obs_grid" the agents per work item and the CTAs of the engine's
 * last observation launch (0 before the first one). */
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
 *   "side" int32[E] (1 = armies swapped this episode, random_sides), "episode" int32[E],
 *   "placement_short" int32[E] (random agents the env's last placement could not place, mfb_add_agents_random),
 *   "walls" uint8[H][W] (1 = obstacle: the border ring and add_walls; the engine's, not per env)     */
int mfb_get(mfb_engine *eng, const char *key, void *host_buf, void *stream);
/* device pointer to the live int32[E][2] agent counts (for masking on the device) */
int mfb_num_device_ptr(mfb_engine *eng, const int32_t **out);

/* device pointers to live engine state, valid until mfb_destroy (read-only for the caller; they change with every
 * launch on the engine's stream; a placement made by mfb_add_agents reaches the device with the next launch or
 * mfb_get): "num" int32[E][2], "id" int32[E][2][cap], "pos" int32[E][2][cap] (x | y << 16),
 * "hp" float[E][2][cap], "step_ct" int32[E] */
int mfb_state_device_ptr(mfb_engine *eng, const char *key, const void **out);

/* ---- Save, restore and fork environments ------------------------------------------------------------------
 * Each env is saved as one record of R bytes (mfb_query "state_bytes"; R = 96 + 64 * cap, a multiple of 16), all
 * 32-bit words little-endian:
 *   bytes  0..31   magic 0x5342464D ("MFBS"), format version 1, W, H, cap, n_action, embedding_size, 0
 *   bytes 32..39   uint64 FNV-1a hash of the engine's H*W wall bytes ("walls"), taken when the placement is committed
 *   bytes 40..95   num[2], dead_ct[2], rng (minstd state), step_ct, id_counter, side, episode, init_num[2], 0, 0, 0
 *   bytes 96..     eight [2][cap] slices, raw (rows at or past num included, so a record round-trips byte for byte):
 *                  pos (x | y << 16), hp (f32), id, state (dead | last_op << 8 | last_action << 16), next_rew (f32),
 *                  last_rew (f32), then the env's placement template: pos, id (the shared template where the engine
 *                  has one) -- what auto-reset re-places the env from
 * Not in a record: agent_steps (an engine statistic), the observation record and k_step's HBM workspace (derived from
 * the state, rebuilt on load), the walls (the engine's; identified by the hash) and the engine config (agent type,
 * rewards, seed, rng_mode, env_base, max_steps, random_sides).  An exact continuation needs an engine created with the
 * same config.
 *   envs   HOST int32[n] env indices, or NULL = all n_envs in order (then n must equal n_envs)
 *   d_out / d_in   DEVICE [n][R], 16-byte aligned
 * mfb_save_envs commits a pending placement first (as mfb_get does), then is asynchronous on `stream`; repeated indices
 * are allowed.  A save or load with an index list copies it to an engine-owned device buffer; that copy is ordered on
 * `stream` after the previous call that used the buffer, on whatever stream (the host does not wait).
 * mfb_load_envs validates before it writes anything.  On the host: n in [1, n_envs], indices in range and not repeated,
 * buffers not NULL.  On the device, k_state_check checks every record: magic and version; W, H, cap, n_action equal
 * to the engine's (a record of another capacity needs an engine created with that capacity); the wall hash; num,
 * dead_ct and init_num in [0, cap]; every listed agent position (slots < num) and template position (< init_num) on
 * the map; last_action <= n_action.  Reading its verdicts back is the one synchronisation of a load (of `stream`).  A
 * bad record returns -1 with "mfb_load_envs: record k: <reason>" and leaves the engine unchanged; otherwise
 * k_load_envs writes the envs.  After a load:
 *   - an engine with one shared template whose template differs from a loaded one's moves to one template per env
 *     (as mfb_add_agents_per_env does), so auto-reset re-places every loaded env from its record's template;
 *   - the engine counts as stepped: mfb_add_agents follows the after-step rules, mfb_reset discards everything;
 *   - the observation record is rebuilt where the engine keeps one.
 * RNG: the random_sides draw at auto-reset is Philox keyed by the global env id env_base + e in EVERY rng_mode.
 *   - MFB_RNG_MINSTD: the attack shuffle's stream state travels in the record.  Without random_sides a loaded env
 *     continues exactly as its source would have, at any index.  With random_sides it does so at any index only up to
 *     its next auto-reset; from there on, at another global id, it draws its own side.
 *   - MFB_RNG_PHILOX: the attack shuffle is keyed by env_base + e too, so at another global id a loaded env draws its
 *     own attack orders from the first step.
 * At the source's global id a loaded env reproduces its source exactly in both modes (create the engine with a
 * matching env_base to replay any env).
 * Random placement ops (mfb_add_agents_random) are engine configuration like max_steps: they are not in a record, and
 * its template slices hold the fixed part only.  A record loaded into an engine with the same placement program (the
 * same ops after as many mfb_reset calls) continues exactly through its next auto-resets too: MINSTD draws from the
 * rng in the record, Philox from its episode and global id. */
int mfb_save_envs(mfb_engine *eng, int n, const int32_t *envs, void *d_out /* device [n][R] */, void *stream);
int mfb_load_envs(mfb_engine *eng, int n, const int32_t *envs, const void *d_in /* device [n][R] */, void *stream);

/* Observation rows rendered from state records (kernel k_render_obs), e.g. for a replay that stores one record per
 * (env, step) instead of every agent's row.  Row k of the output is bit for bit what mfb_observe_groups writes for slot
 * `slot` of group `group` when an env of this engine holds record `record`, with the engine's walls: the view disc,
 * both minimaps (count / num over every listed agent, dead or not; 0 / 0 = 0) with the "+1" self marker, id bits, the
 * one-hot last action, last_rew, x / W, y / H -- rows of dead but still listed agents included.
 *   d_records   DEVICE [n_records][R] state records (mfb_save_envs), 16-byte aligned
 *   d_rows      DEVICE int32[n_rows][3]: (record index, group, slot), 16-byte aligned
 *   d_view      DEVICE float[n_rows][13][13][7], d_feature float[n_rows][feature_size], 16-byte aligned; exactly these
 *               rows are written, nothing past row n_rows - 1
 *   d_bad_rows  DEVICE int32 or NULL: set to the number of rows zeroed by the rules below (no synchronisation)
 * Input from outside never makes the kernel read or write outside these buffers.  A row comes out all zeros (view and
 * features) when its record index is not in [0, n_records), its group is not 0 or 1, its slot is not in [0, cap), its
 * slot is at or past the record's num[group], its own position is off the map, or its record's header does not match
 * this engine (magic, version, W, H, cap, n_action, wall hash).  Inside a record num is clamped to [0, cap], and listed
 * agents whose position is off the map are neither drawn nor counted in the minimaps.
 * A pending placement is committed first (as mfb_save_envs does); then the call is asynchronous on `stream` and changes
 * no engine state.  Returns -1 ("mfb_render_observations: ...") for n_rows < 0, n_records < 1 with n_rows > 0, a NULL
 * buffer or one that is not 16-byte aligned, before anything is launched. */
int mfb_render_observations(mfb_engine *eng, int n_records, const void *d_records, int n_rows, const int32_t *d_rows,
                            float *d_view, float *d_feature, int32_t *d_bad_rows /* may be NULL */, void *stream);

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
 *                  fp32: output word row % 4 is the site's draw, u = that word (rounded toward zero to 24 bits) / 2^32;
 *                  fp64: two calls, counter word 3 = 0 for rows 4j, 4j+1 and 1 for rows 4j+2, 4j+3, each call serving
 *                  two rows: (hi, lo) = output words (0, 1) for the even row and (2, 3) for the odd one, and
 *                  u = ((hi >> 5) * 2^26 + (lo >> 6)) / 2^53 (53 bits, in [0, 1))
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

/* Per-lattice temperature schedules: mfi_step / mfi_run with one schedule per lattice, e.g. one batch holding every
 * (temperature, replica) point of an order-parameter-against-temperature curve.  Lattice b draws sweep k at
 * d_temperatures[k][b]; everything else (Philox keys, act groups, outputs, fp32 / fp64, the bits) is as above, so
 * lattice b of a batch equals that lattice run alone with lattice_base + b and its own schedule.
 *   mfi_step_lattices  d_temperatures  T [n_lattices]            device (K6)
 *   mfi_run_lattices   d_temperatures  T [n_sweeps][n_lattices]  device (K6s at the fp32 sides 64 / 128 / 256 / 512,
 *                                                                the generic K6r elsewhere and in fp64)
 * The fp32 overrides that select a kernel without per-lattice tables -- MFMARL_ISING_PERSIST=1 (K6p), an
 * MFMARL_ISING_RPT other than 0 or 8, and MFMARL_ISING_PERSIST=0 at sides 64 / 128 / 256 (the specialised K6r) unless
 * MFMARL_ISING_RPT=0 -- make mfi_run_lattices return -1 with a message naming the variable, and nothing is launched
 * (MFMARL_ISING_RPT=0 selects the generic K6r, which has the tables). */
int mfi_step_lattices(int dtype, int n_lattices, int side, int8_t *d_spins, void *d_q, const void *d_temperatures,
                      double lr, const void *d_uniforms, const uint8_t *d_update_mask, unsigned seed,
                      unsigned lattice_base, unsigned step, int32_t *d_n_up, void *d_reward_sum, void *d_mse,
                      void *stream);
int mfi_run_lattices(int dtype, int n_lattices, int side, int n_sweeps, int8_t *d_spins, void *d_q,
                     const void *d_temperatures, double lr, const void *d_uniforms, const uint8_t *d_update_mask,
                     unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up, void *d_reward_sum,
                     void *stream);

/* ---- K8: checkerboard single-spin-flip Metropolis on the same lattice model (the MCMC reference of the Ising curve)
 * H = -1/2 sum_bonds sigma_i sigma_j = -1/2 sum_i r_i (sigma = 2 spin - 1, r_i = the environment's reward; coupling 1/2,
 * Tc = 1 / ln(1 + sqrt 2) ~ 1.1346, MF-Q's temperature axis; flipping site i changes H by h below).  One sweep: every site with (x + y) even, then every site with (x + y) odd.  Site
 * i flips when h = sigma_i sum_nbr sigma_j <= 0, and for h in {2, 4} when its Philox word r satisfies r < thr_h with
 *   thr_h = min(floor(exp(-h / T) * 2^32), 2^32 - 1)   computed on the HOST in double with the C library's exp
 * (Python's math.exp is the same function), so a CPU restatement reproduces every decision.
 * Philox4x32-10: key (seed, lattice_base + lattice); site (x, y) of colour c = (x + y) & 1 in sweep step0 + k uses
 * output word ((x & 31) >> 1) & 3 of counter ((y * ceil(side / 32) + x / 32) * 4 + (x & 31) / 8, step0 + k, c, 2)
 * (the 2 keeps the stream apart from MF-Q's, which has 0 or 1 there).
 *   side            even, 2 <= side <= 512
 *   d_spins         int8 [n_lattices][side][side]   in/out, values {0, 1}
 *   h_temperatures  double [n_sweeps][n_lattices]   HOST memory: every T finite and > 0 (the thresholds are computed
 *                   from it on the host and uploaded with the launch)
 *   d_n_up          int32[n_sweeps][n_lattices]     out or NULL: up spins after each sweep
 *   d_bond_sum      int32[n_sweeps][n_lattices]     out or NULL: sum over the 2N bonds of sigma_i sigma_j after each sweep
 *                   (= sum_i r_i, MF-Q's reward_sum; energy per site = -bond_sum / N)
 * Bad input (odd side or out of range, T <= 0, inf or NaN) returns -1 before anything is launched. */
int mfi_metropolis(int n_lattices, int side, int n_sweeps, int8_t *d_spins, const double *h_temperatures,
                   unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up, int32_t *d_bond_sum,
                   void *stream);

/* ---- K9: Swendsen-Wang cluster updates on the same lattice model (the MCMC reference near Tc and at odd sides)
 * H = -1/2 sum_bonds sigma_i sigma_j as for K8.  Site i = y * side + x owns its right bond to ((x + 1) mod side, y) and
 * its down bond to (x, (y + 1) mod side): 2N bonds (at side 2 the two bonds between a pair of sites are distinct).
 * One sweep:
 *   1. a bond is active iff its two spins are aligned and its Philox word r satisfies r < thr with
 *        thr = min(floor((1 - exp(-1 / T)) * 2^32), 2^32 - 1)   computed on the HOST in double with the C library's exp
 *      (T = 1e-3 clamps to 2^32 - 1; T = 1e20 gives 0, no bonds);
 *   2. clusters are the connected components of the active bonds; a cluster's canonical label is its SMALLEST flat site
 *      index (the kernel's result depends on this label only, never on the order in which its threads merge);
 *   3. the cluster with root r flips as a whole iff r's flip word has its top bit set (word >= 2^31);
 *   4. d_n_up / d_bond_sum as for K8, of the final spins of the sweep.
 * Philox4x32-10: key (seed, lattice_base + lattice); in sweep step0 + k
 *   bond words of site i: counter (i >> 1, step0 + k, 0, 3), output word 2 (i & 1) = its right bond,
 *                         2 (i & 1) + 1 = its down bond
 *   flip word of root r:  output word r & 3 of counter (r >> 2, step0 + k, 1, 3)
 * (the 3 keeps the stream apart from MF-Q's 0 / 1 and K8's 2).
 *   side            2 <= side <= 256, odd or even (the uint16 cluster labels of a lattice live in shared memory)
 *   other arguments as for mfi_metropolis
 * Bad input (side out of range, T <= 0, inf or NaN, null spins or temperatures, fewer than one lattice or one sweep)
 * returns -1 with a message prefixed "mfi_swendsen_wang: " before anything is launched or written. */
int mfi_swendsen_wang(int n_lattices, int side, int n_sweeps, int8_t *d_spins, const double *h_temperatures,
                      unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up, int32_t *d_bond_sum,
                      void *stream);

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
