// Shared host/device parameter blocks for the battle kernels.
//
// Data layout in HBM (one engine = E lock-stepped environments, G = 2 groups, `cap` agent slots per
// group, SoA so that a warp reading consecutive agents of one env reads consecutive words):
//
//   pos        int32 [E][2][cap]   x | y << 16                     (Agent::pos, GridWorld.h:240)
//   hp         f32   [E][2][cap]                                     (Agent::hp,  GridWorld.h:242)
//   id         int32 [E][2][cap]                                     (Agent::id,  GridWorld.h:236)
//   state      u32   [E][2][cap]   dead | last_op << 8 | last_action << 16
//   next_rew   f32   [E][2][cap]                                     (Agent::next_reward)
//   last_rew   f32   [E][2][cap]                                     (Agent::last_reward)
//   num        int32 [E][2]        agents in the list, dead ones included until clear_dead
//   dead_ct    int32 [E][2]
//   rng        u32   [E]           minstd_rand0 state (parity mode)
//   step_ct    int32 [E]
//   walls      u8    [E or 1][H*W] 1 = obstacle (border ring + add_walls)
//
// The occupancy grid (Map::slots / channel_ids, Map.h:72-74) is NOT stored: every kernel rebuilds it
// in shared memory from walls + the alive agents, so there is a single source of truth and
// clear_dead never has to patch a map.  (Geometries whose working set exceeds a CTA's shared memory
// rebuild it in a per-env HBM workspace instead: Engine::hbm_kernels.)
#pragma once
#include <stdint.h>

namespace mfmarl {

constexpr int kGroups = 2;
constexpr int kMaxMoves = 32;    // |move range| (13 for speed 2)
constexpr int kMaxAttacks = 32;  // |attack range| (8 for radius 1.5)
constexpr int kMaxActions = 64;
constexpr int kObsTicketRing = 8;   // k_obs launches of one engine that may be in flight at once
constexpr int kObsDiscSlots = 128;   // 4 passes x 32 lanes cover the <= 113 in-disc cells of the 13x13 window
// battle observation geometry (view disc radius 6 -> 13x13 window, 1 wall + 2 x (has, hp, minimap) channels)
constexpr int kView = 13, kViewCells = 169, kChan = 7, kViewRow = kViewCells * kChan;   // 1183 floats

// EventOp values the battle path can produce (reference grid_def.h:18-24)
enum : uint32_t { OP_KILL = 3, OP_COLLIDE = 6, OP_ATTACK = 7, OP_NULL = 11 };

enum RngMode : int {
    RNG_MINSTD = 0,  // libstdc++ minstd_rand0, one stream per env: bit-parity with the reference
    RNG_PHILOX = 1,  // Philox4x32-10 keyed by (seed, global env id, step): production mode
    RNG_INJECT = 2,  // attack order supplied by the caller (test hook)
};

enum StepPhase : int {
    PH_SETACT = 1,     // GridWorld::set_action  (GridWorld.cc:430-496)
    PH_STEP = 2,       // GridWorld::step        (GridWorld.cc:498-694)
    PH_EXPORT = 4,     // get_reward + get_info("alive") (GridWorld.cc:760-770,801-806) + mean action
    PH_CLEAR = 8,      // GridWorld::clear_dead  (GridWorld.cc:696-728)
    PH_AUTORESET = 16, // batched extension: re-place the armies when an episode ends
};

struct BattleParams {
    int E, W, H, cap;
    int env_base;           // global id of env 0 of this engine (multi-GPU sharding; keys Philox)
    int embedding_size;     // 10
    int n_move, n_attack;   // 13, 8 -> action space 21
    int view;               // 13 (kernels are specialised for 13)
    int feature_size;       // embedding + n_action + 1 + 2 = 34
    int scale_w, scale_h;   // minimap scale: ceil(W / view)
    int wall_stride;        // H*W, or 0 when every env shares one wall map
    int rng_mode;
    int max_steps;          // auto-reset horizon (0 = none)
    int tmpl_stride;        // 0: one placement template for every env; 4*cap: a template per env (add_agents_per_env)
    int random_sides;       // auto-reset: each env draws (Philox, keyed by env and episode) whether the two armies swap
                            // their starting blocks, as generate_map does per round (senario_battle.py:14)
    int obs_cached;         // k_obs starts an item from the per-env observation record (large groups, and every geometry
                            // whose kernels run from HBM) instead of the agent arrays
    int move_bands;         // 0, or the reference's NUM_SEP_BUFFER when W*H > 99*99 ("large map mode", GridWorld.cc:79-88):
    int band_width;         //   moves run x-band by x-band, then the band-boundary buffer (GridWorld.cc:443-463,662-672)
    uint32_t seed;
    float hp, damage, step_recover, kill_supply;
    float step_reward, kill_reward, dead_penalty, attack_penalty;
    float attack_bonus[kGroups];   // the two `attack` reward rules (config/battle.py:41-42)
    int8_t move_dx[kMaxMoves], move_dy[kMaxMoves];
    int8_t att_dx[kMaxAttacks], att_dy[kMaxAttacks];
    uint32_t disc[8];       // view disc mask, bit c of word c/32 for view cell c = vy*view + vx
    uint8_t obs_cell[kObsDiscSlots];   // k_obs lane schedule: slot p*32 + lane -> in-disc view cell (255 = idle), chosen
                                       // so that the cells of one pass fall into distinct shared-memory banks when possible
};

struct BattleState {   // device pointers
    int32_t *pos; float *hp; int32_t *id; uint32_t *state; float *next_rew; float *last_rew;
    int32_t *num; int32_t *dead_ct; uint32_t *rng; int32_t *step_ct; int32_t *id_counter;
    uint8_t *walls;
    uint16_t *grid_template;           // [(H+12)*(W+12)] padded occupancy grid holding only the walls (kind << 14)
    uint8_t *mini_lut;                 // [W] x / scale_w, then [H] (y / scale_h) * view: minimap cell of a position
    unsigned char *obs_record;         // [E][obs_record_layout().total] when obs_cached (battle_kernels.cuh), followed by
                                       // k_step's workspace [E][step_smem_layout().total] when k_step runs from HBM
    unsigned long long *agent_steps;   // [E] running count of agents taken through a step (statistic)
    int32_t *obs_ticket;               // [2] of this launch (ring of kObsTicketRing pairs): next item, CTAs finished (rewound by the last CTA)
    // episode template for auto-reset
    int32_t *init_pos; int32_t *init_num;   // [T][2][2][cap] (pos, then id), [T][2]; T = 1 or E (BattleParams::tmpl_stride)
    int32_t *side;                     // [E] 1 = the armies started this episode on swapped sides (random_sides)
    int32_t *episode;                  // [E] episodes started since the placement (keys the side draw)
};

// Host mirror of ONE environment's agent records (single-env ABI): mapped pinned memory k_step writes at its end,
// so the getters of runtime_api.cu answer without a copy on the critical path.
struct StepMirror {
    int32_t *pos; int32_t *id; uint32_t *state; float *hp; float *next_rew; float *last_rew;   // [2][cap] each
    int32_t *head;   // [8]: num[2], dead_ct[2], done, step_ct, 0, 0
};

struct StepIO {
    const int32_t *actions;     // [E][2][cap] (PH_SETACT)
    const int32_t *attack_perm; // [E][2*cap]  (RNG_INJECT) new order -> pre-shuffle index
    float *reward;              // [E][2][cap] (PH_EXPORT)
    uint8_t *alive;             // [E][2][cap]
    float *mean_action;         // [E][2][n_action]
    int32_t *done;              // [E]
    int32_t *attack_events;     // optional [E][1 + 3*2*cap]: count, then per attack of the shuffled order (attacker id or
                                // -1 when it was dead at its turn, target x, target y) -- the render trace's events
    StepMirror mirror;          // optional (E == 1, pos != nullptr): the records as this launch leaves them
    int phases;
    int setact_mask;            // groups whose actions are applied by PH_SETACT
    int group_seq[kGroups];     // order in which groups called set_action (-1 = did not act)
};

struct ObsIO {
    float *view[kGroups];     // per group: rows of env e start at e * env_stride agent rows ([13][13][7] each)
    float *feature[kGroups];  // per group, same indexing ([feature_size] each)
    int env_stride;  // agent rows between consecutive envs: 2*cap for the [E][2][cap] block, cap for per-group blocks
    int group_mask;  // which groups to produce
    int tile_agents; // agents per CTA tile
    int tiles_per_group;
    int debug;       // only read by -DMF_PROFILE_BUILD binaries (profiling experiments): 1 = skip row composition
};

// K7 (k_local_mean_action): neighbourhood mean action.  Passed by value as a __grid_constant__ parameter; the disc
// part (n_offsets, delta) is built on the host once per radius (Engine::local_mean_action).
constexpr int kLocalMaxTile = 128;   // observers per CTA (= threads)
struct LocalMeanIO {
    float *out[kGroups];       // per group [E][cap][n_action]
    int group[kGroups];        // blockIdx.z -> group (only the groups asked for are launched)
    int W, H, cap, n_action;
    int tile;                  // observers per CTA = blockDim.x, a multiple of 32
    int n_offsets;             // cells of the disc other than the centre
    int16_t delta[kViewCells]; // their offsets in the padded u8 grid (row pitch W + 2 * kPad)
};

}  // namespace mfmarl
