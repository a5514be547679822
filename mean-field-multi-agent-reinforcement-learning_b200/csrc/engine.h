// Host side of the battle engine: owns the HBM-resident state of E lock-stepped environments and
// launches the kernels of battle_kernels.cuh.  Used by both C ABIs:
//   runtime_api.cu   the reference's 19 runtime_api.h symbols (one env, caller-owned HOST buffers)
//   batched_api.cu   mfb_* (E envs, caller-owned DEVICE buffers, explicit stream)
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "battle_types.h"

namespace mfmarl {

struct Fatal : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define MF_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t err__ = (expr);                                                                \
        if (err__ != cudaSuccess)                                                                  \
            throw ::mfmarl::Fatal(std::string(#expr) + " failed: " + cudaGetErrorString(err__) +   \
                                  " (" __FILE__ ":" + std::to_string(__LINE__) + ")");             \
    } while (0)

// Circular range tables (reference Range.h:171-215), computed once on the host.
struct CircleRange {
    int width = 0, count = 0, center = 0;
    std::vector<unsigned char> in;   // [width*width]
    std::vector<int> dx, dy;         // [count], row-major over the mask
    CircleRange() = default;
    CircleRange(float radius, float inner_radius, int parity);
};

struct AgentTypeParams {   // the attributes of AgentType.h:21-45 that reach the battle path
    float hp = 10, speed = 2, view_radius = 6, attack_radius = 1.5f;
    float damage = 2, step_recover = 0.1f, kill_supply = 0;
    float step_reward = -0.005f, kill_reward = 5, dead_penalty = -0.1f, attack_penalty = -0.1f;
};

struct EngineConfig {
    int n_envs = 1, width = 40, height = 40, capacity = 64, embedding_size = 10;
    int rng_mode = RNG_MINSTD, max_steps = 0, env_base = 0, device = -1 /* current */;
    int step_threads = 0 /* <= 0 auto; else 33..1024, rounded up to a multiple of 32 */, obs_tile_agents = 0 /* auto: clamp(cap, 64, 256); 64 with the observation record */;
    int concurrent_step_envs = 0 /* envs of a sibling engine whose k_step runs (on another stream) while this engine's
                                    k_obs streams: k_obs then leaves SM slots free for it where the two do not fit together */;
    int random_sides = 0 /* auto-reset draws per env and episode whether the armies swap their starting blocks */;
    int obs_cached = -1 /* observation record: -1 auto (capacity >= 256, or MFMARL_OBS_CACHED), 0 off, 1 on; always on
                           where the kernels run from HBM (0 is refused there) */;
    unsigned seed = 0;
    AgentTypeParams type;
    float attack_bonus[kGroups] = {0.2f, 0.2f};
};

class Engine {
public:
    explicit Engine(const EngineConfig &cfg);
    ~Engine();
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;

    // ---- episode set-up (host side; takes effect at the next kernel) ----
    void reset();                                              // GridWorld::reset
    int add_walls(int n, const int *xs, const int *ys);        // add_agents(group = -1, "custom")
    int add_agents(int group, int n, const int *xs, const int *ys);   // add_agents(group, "custom"), the same in every env
    // a placement of its own for every env: xs / ys are [E][n]; occupied or out-of-range cells are skipped PER ENV
    // (GridWorld.cc:180-187), so the envs may end up with different counts; n_added (may be null) receives [E] counts
    void add_agents_per_env(int group, int n, const int *xs, const int *ys, int *n_added);
    // mfb_add_agents_random: appends a random op to the placement program (w = h = 0: the whole map); refuses, changing
    // nothing, a bad group or n, a rectangle off the map or without an interior cell, and an op that cannot fit in some env
    void add_agents_random(int group, int n, int x0, int y0, int w, int h);
    void set_seed(unsigned long seed);                         // set_config("seed")

    // ---- kernels ----
    void observe(float *d_view, float *d_feature, int group_mask, cudaStream_t st);
    // per-group output blocks [E][cap][...] (env_stride = cap) or any layout with `env_stride` rows between envs
    // bf16 = true: d_view[g] are __nv_bfloat16 [E][cap][13][13][8] blocks (channel 7 = 0), the rows a bf16 channels-last
    // policy reads without a cast or a padding pass; features stay fp32
    void observe_groups(float *const d_view[kGroups], float *const d_feature[kGroups], int env_stride, int group_mask,
                        cudaStream_t st, bool bf16 = false);
    void step(const StepIO &io, cudaStream_t st);
    static void mean_action(const int32_t *d_actions, const int32_t *d_num, float *d_out, int rows,
                            int cap, int n_action, cudaStream_t st);
    // K7: neighbourhood mean action of every listed agent (mfmarl_batched.h mfb_local_mean_action); out[g] is a
    // 16-byte aligned float [E][cap][n_action] block or null (group skipped).  0 < radius <= view_radius.
    void local_mean_action(double radius, float *const out[kGroups], cudaStream_t st);

    // E == 1: overwrite the agent records with a host copy (mapped pinned memory; runtime_api.cu rolls back a speculative
    // clear_dead with it).  Asynchronous on `st`.
    void restore_state(const int32_t *pos, const int32_t *id, const uint32_t *state, const float *hp, const float *next_rew,
                       const float *last_rew, const int32_t *num, const int32_t *dead_ct, cudaStream_t st);

    // ---- per-env state records (mfmarl_batched.h mfb_save_envs / mfb_load_envs; engine_state.cu) ----
    size_t state_bytes() const;                  // R: bytes of one env's record at the current capacity
    // envs: host int32[n] env indices, or null = every env in order (n = E); d_out / d_in: device [n][R], 16-byte aligned
    void save_envs(int n, const int32_t *envs, void *d_out, cudaStream_t st);   // asynchronous; repeated indices allowed
    void load_envs(int n, const int32_t *envs, const void *d_in, cudaStream_t st);   // validates every record first (syncs)
    // observation rows of listed (record, group, slot) triples, as k_obs would write them for an env holding the record
    // (mfb_render_observations); asynchronous, changes no engine state.  d_bad_rows (may be null) receives the rows zeroed
    void render_observations(int n_records, const void *d_records, int n_rows, const int32_t *d_rows, float *d_view,
                             float *d_feature, int32_t *d_bad_rows, cudaStream_t st);

    // ---- state access ----
    void commit(cudaStream_t st);                // upload a pending placement
    void download_num(cudaStream_t st);          // refresh h_num from the device (syncs)
    const BattleParams &params() const { return P_; }
    void set_rng_mode(int mode) { P_.rng_mode = mode; }
    // a caller that replays captured step launches (CUDA graph) tells the engine that the device state has moved on:
    // what Engine::step notes itself when it launches (late add_agents then reads the device state back first)
    void mark_stepped() { stepped_ = true; }
    const std::vector<unsigned char> &host_walls() const { return h_walls_; }
    // E == 1 helpers for add_agents(method="random"): the engine RNG lives on the device
    uint32_t pull_rng0();
    void push_rng0(uint32_t s);
    bool cell_blank_for_placement(int x, int y);   // Map::is_blank_area for a 1x1 body, host view
    const BattleState &state() const { return S_; }
    const int32_t *placement_short() const { return RP_.place_short; }   // [E] (mfb_get "placement_short")
    int cap() const { return P_.cap; }
    int n_envs() const { return P_.E; }
    int n_action() const { return P_.n_move + P_.n_attack; }
    int host_num(int env, int group) const { return h_num_[env * 2 + group]; }
    // the caller already knows the counts after clear_dead (it holds the alive flags): no device round trip
    void set_host_num(int env, int group, int n) { h_num_[env * 2 + group] = n; }
    bool placement_pending() const { return placement_dirty_; }
    size_t slots() const { return (size_t)P_.E * 2 * P_.cap; }
    const CircleRange &view_range() const { return view_; }
    const CircleRange &attack_range() const { return attack_; }
    const CircleRange &move_range() const { return move_; }
    // kernels whose shared-memory layout for the current geometry (map, capacity) exceeds a CTA's shared memory, so
    // they run from HBM instead: a mask of HBM_* (mfb_query "hbm_kernels")
    enum { HBM_STEP = 1, HBM_OBS = 2, HBM_RECORD = 4, HBM_LOCAL_MEAN = 8 };
    int hbm_kernels() const;
    // launch shape: k_step's CTA width after the auto rules; k_obs's tile and grid of the last observe (0 before one)
    int step_threads() const;
    int last_obs_tile() const { return last_obs_tile_; }
    int last_obs_grid() const { return last_obs_grid_; }

private:
    void alloc_state(int cap);
    size_t grid_template_bytes() const;
    void free_state();
    void grow(int need_cap);
    void late_add_sync_down();   // E == 1 only: device state -> host records
    void late_add_sync_up();
    void rebuild_obs_records(cudaStream_t st);   // observation records of every env from the state arrays (obs_cached)
    void require_obs_record(int cap);            // geometries that run from HBM: record on, or refuse a forced "off"
    const int32_t *upload_targets(int n, const int32_t *envs, const void *buf, bool load, cudaStream_t st);

    struct LateRecords;                    // scratch of one late add_agents call (E == 1)
    std::unique_ptr<LateRecords> late_;

    EngineConfig cfg_;
    BattleParams P_{};
    BattleState S_{};
    CircleRange view_, attack_, move_;
    int device_ = 0;
    int n_sm_ = 148;
    int obs_attr_[2] = {-1, -1};           // shared-memory size the occupancy below was queried for (fp32 rows, bf16 rows)
    unsigned obs_launches_ = 0;            // k_obs launches so far (picks the ticket pair)
    int obs_ctas_per_sm_[2] = {2, 2};      // resident k_obs CTAs per SM at that size (occupancy query)
    int obs_grid_limit_ = 0;               // MFMARL_OBS_GRID: cap on k_obs CTAs (leaves SM slots to a concurrent k_step)
    int last_obs_tile_ = 0, last_obs_grid_ = 0;   // tile_agents and grid of the last k_obs launch
    int obs_debug_ = 0;                    // MFMARL_OBS_DEBUG at construction (profiling experiments only)
    std::map<float, LocalMeanIO> local_discs_;   // K7 disc tables by radius (n_offsets, delta filled)
    bool obs_cached_off_ = false;          // the record was switched off explicitly (config or MFMARL_OBS_CACHED=0)

    // host-side placement template (what add_agents has built since the last reset)
    std::vector<unsigned char> h_walls_;          // [H*W]
    std::vector<int> h_occ_;                      // [H*W] 0 free, 1 taken (walls + placed agents)
    std::vector<int> h_tpos_[kGroups], h_tid_[kGroups];
    int h_id_counter_ = 0;
    // per-env placement (after the first add_agents_per_env): the template above replicated, then diverging
    struct EnvTemplate { std::vector<unsigned char> occ; std::vector<int> pos[kGroups], id[kGroups]; int id_counter = 0; };
    std::vector<EnvTemplate> h_env_;              // empty = shared template
    void split_template();                        // shared -> per-env
    void refuse_after_random(const char *what) const;   // fixed placements and walls must come before the random ops
    std::vector<RandomOp> h_random_;              // the random ops since the last reset, in call order
    RandomPlacement RP_{};                        // what k_place / k_step see of them (ops uploaded at commit)
    size_t d_random_cap_ = 0;                     // RandomOp slots allocated at RP_.ops
    bool placement_dirty_ = true;
    bool stepped_ = false;                        // a step has run since the last placement upload
    std::vector<int> h_num_;                      // [E][2] mirror, refreshed by download_num
    unsigned long long wall_hash_ = 0;            // FNV-1a 64 of h_walls_ as last committed (identifies the walls of a record)
    int32_t *d_state_io_ = nullptr;               // save / load scratch: env indices, then the check kernel's verdicts
    size_t state_io_words_ = 0;
    cudaEvent_t state_io_done_ = nullptr;         // the last save / load launch that reads the scratch
};

// error reporting shared by the two C ABIs
void set_last_error(const std::string &msg);
const char *last_error();
int report_fatal(const char *where, const std::exception &ex);   // prints; aborts unless MAGENT_ERRORS=return

}  // namespace mfmarl
