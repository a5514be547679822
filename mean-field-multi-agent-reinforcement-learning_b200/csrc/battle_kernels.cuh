// Hand-written sm_100a kernels for the MAgent battle hot path.
//
//   k_obs   (K1)  GridWorld::get_observation + Map::extract_view   (GridWorld.cc:303-426, Map.cc:130-218)
//   k_step  (K2)  set_action + step + get_reward/alive + mean action + clear_dead, one CTA per env
//                 (GridWorld.cc:430-496, 498-694, 696-728, 744-770; Map.cc:220-369;
//                  RewardEngine.cc:216-240,373-443; senario_battle.py:141)
//   k_mean_action (K5) standalone group mean action (senario_battle.py:141,255)
//   k_local_mean_action (K7) per-agent neighbourhood mean action over a view-range disc (read-only)
//   k_place       episode (re)initialisation from a placement template (GridWorld.cc:76-124,256-269)
//
// All arithmetic that reaches an output is ordered IEEE fp32 (compiled with -fmad=false, explicit
// _rn intrinsics where the reference divides), so results are bit-identical to the C++ engine.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "battle_types.h"
#include "rng.cuh"

namespace mfmarl {

// ----------------------------------------------------------------------------------------------
// small helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ int pos_x(int p) { return p & 0xFFFF; }
__device__ __forceinline__ int pos_y(int p) { return (p >> 16) & 0xFFFF; }
__device__ __forceinline__ int pack_pos(int x, int y) { return (x & 0xFFFF) | (y << 16); }
__device__ __forceinline__ uint32_t st_dead(uint32_t s) { return s & 1u; }
__device__ __forceinline__ uint32_t st_op(uint32_t s) { return (s >> 8) & 0xFFu; }
__device__ __forceinline__ uint32_t st_act(uint32_t s) { return (s >> 16) & 0xFFu; }
__device__ __forceinline__ uint32_t st_with_op(uint32_t s, uint32_t op) { return (s & ~0xFF00u) | (op << 8); }
__device__ __forceinline__ uint32_t make_state(uint32_t dead, uint32_t op, uint32_t act) {
    return dead | (op << 8) | (act << 16);
}

// Block-wide exclusive scan of TWO predicates at once (ballot + popc inside each warp, per-warp totals through
// shared memory, both counts packed into one int: low half a, high half b -- counts stay below 65536).  Must be
// reached by every thread of the block.  s_warp needs 32 ints.  Returns the packed exclusive prefix.
__device__ __forceinline__ int block_scan_flags2(bool fa, bool fb, int *s_warp, int &total) {
    const unsigned ba = __ballot_sync(0xFFFFFFFFu, fa), bb = __ballot_sync(0xFFFFFFFFu, fb);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) s_warp[w] = __popc(ba) | (__popc(bb) << 16);
    __syncthreads();
    const int nw = (blockDim.x + 31) >> 5;
    int before = 0, tot = 0;
    if (nw <= 4) {                     // narrow CTAs (64 v 64): a 2-4 term loop is shorter than a shuffle scan
        for (int k = 0; k < nw; k++) {
            const int c = s_warp[k];
            before += (k < w) ? c : 0;
            tot += c;
        }
    } else {                           // wide CTAs: lane k reads warp k's count, one shuffle scan serves every lane
        const int c = lane < nw ? s_warp[lane] : 0;
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += v;
        }
        tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
        before = __shfl_sync(0xFFFFFFFFu, incl - c, w);
    }
    __syncthreads();
    total = tot;
    const unsigned lt = (1u << lane) - 1u;
    return before + (__popc(ba & lt) | (__popc(bb & lt) << 16));
}
__device__ __forceinline__ int block_scan_flag(bool flag, int *s_warp, int &total) {
    return block_scan_flags2(flag, false, s_warp, total);
}

// ----------------------------------------------------------------------------------------------
// Observation record (large groups only, BattleParams::obs_cached): what k_obs needs to know about an environment,
// laid out exactly as k_obs wants it in shared memory, so that an observation work item starts with ONE bulk copy
// instead of re-deriving it from the agent arrays (at 512 v 512 that set-up was 18 % of k_obs, ncu round 1, and it
// forced 128-agent tiles -- 512 items for 296 CTAs).  Written by whoever changes the state: k_step at its end,
// k_obs_record after a placement.
//   grid   u16 [(H+12)*(W+12)]  padded occupancy: kind << 14 | slot, kind 1 = wall, 2 = group 0, 3 = group 1 (alive only)
//   hp10   f32 [2*cap]          hp / max_hp per slot (Map.cc:208)
//   mini   f32 [2][169]         minimap of each group: count / num over everything still listed (GridWorld.cc:341-380)
// ----------------------------------------------------------------------------------------------
constexpr int kPad = kView / 2;   // the padded grid carries a 6-cell empty margin: view windows never need a bounds test
struct ObsRecord { int grid, hp10, mini, total; };
__host__ __device__ inline ObsRecord obs_record_layout(int W, int H, int cap) {
    ObsRecord R;
    R.grid = 0;
    R.hp10 = ((W + 2 * kPad) * (H + 2 * kPad) * 2 + 15) & ~15;
    R.mini = R.hp10 + 4 * 2 * cap;                 // cap is a multiple of 4: stays 16-byte aligned
    R.total = (R.mini + 4 * 2 * kViewCells + 15) & ~15;
    return R;
}

// Builds env e's record from the state arrays in HBM (as the calling CTA left them: call after a __syncthreads that
// follows the write-back).  s_pg: shared scratch of R.hp10 bytes (16-byte aligned), s_cnt: 2*169 ints.
__device__ __forceinline__ void build_obs_record(const BattleParams &P, const BattleState &S, int e, uint16_t *s_pg, int *s_cnt) {
    const int tid = threadIdx.x, nt = blockDim.x, W = P.W, cap = P.cap, PW = W + 2 * kPad;
    const ObsRecord R = obs_record_layout(P.W, P.H, cap);
    unsigned char *rec = S.obs_record + (size_t)e * R.total;
    const size_t ebase = (size_t)e * 2 * cap;
    for (int c = tid; c < R.hp10 / 16; c += nt) ((uint4 *)s_pg)[c] = ((const uint4 *)S.grid_template)[c];
    for (int c = tid; c < 2 * kViewCells; c += nt) s_cnt[c] = 0;
    const int n0 = S.num[e * 2], n1 = S.num[e * 2 + 1];
    __syncthreads();
    const uint8_t *lut = S.mini_lut;
    float *hp10 = (float *)(rec + R.hp10);
    for (int s = tid; s < 2 * cap; s += nt) {
        const int gg = s >= cap, i = s - gg * cap;
        if (i >= (gg ? n1 : n0)) continue;
        const int p = S.pos[ebase + s], x = pos_x(p), y = pos_y(p);
        atomicAdd(&s_cnt[gg * kViewCells + lut[W + y] + lut[x]], 1);       // dead or not (GridWorld.cc:359-370)
        if (!st_dead(S.state[ebase + s])) {
            s_pg[(y + kPad) * PW + x + kPad] = (uint16_t)(((2 + gg) << 14) | s);
            hp10[s] = __fdiv_rn(S.hp[ebase + s], P.hp);
        }
    }
    __syncthreads();
    for (int c = tid; c < R.hp10 / 16; c += nt) ((uint4 *)rec)[c] = ((const uint4 *)s_pg)[c];
    float *mini = (float *)(rec + R.mini);
    for (int c = tid; c < 2 * kViewCells; c += nt) {
        const int tot = c >= kViewCells ? n1 : n0;
        mini[c] = tot > 0 ? __fdiv_rn((float)s_cnt[c], (float)tot) : 0.0f;   // GridWorld.cc:372-377; 0/0 defined as 0
    }
}

// The same record for maps whose padded grid does not fit in shared memory: the grid is built in place in the env's
// record in HBM (walls from the template, then the alive agents).  Only the minimap counts stay in shared memory
// (s_cnt: 2*169 ints).
__device__ __forceinline__ void build_obs_record_hbm(const BattleParams &P, const BattleState &S, int e, int *s_cnt) {
    const int tid = threadIdx.x, nt = blockDim.x, W = P.W, cap = P.cap, PW = W + 2 * kPad;
    const ObsRecord R = obs_record_layout(P.W, P.H, cap);
    unsigned char *rec = S.obs_record + (size_t)e * R.total;
    uint16_t *grid = (uint16_t *)rec;
    const size_t ebase = (size_t)e * 2 * cap;
    for (int c = tid; c < R.hp10 / 16; c += nt) ((uint4 *)rec)[c] = ((const uint4 *)S.grid_template)[c];
    for (int c = tid; c < 2 * kViewCells; c += nt) s_cnt[c] = 0;
    const int n0 = S.num[e * 2], n1 = S.num[e * 2 + 1];
    __syncthreads();
    const uint8_t *lut = S.mini_lut;
    float *hp10 = (float *)(rec + R.hp10);
    for (int s = tid; s < 2 * cap; s += nt) {
        const int gg = s >= cap, i = s - gg * cap;
        if (i >= (gg ? n1 : n0)) continue;
        const int p = S.pos[ebase + s], x = pos_x(p), y = pos_y(p);
        atomicAdd(&s_cnt[gg * kViewCells + lut[W + y] + lut[x]], 1);
        if (!st_dead(S.state[ebase + s])) {
            grid[(y + kPad) * PW + x + kPad] = (uint16_t)(((2 + gg) << 14) | s);
            hp10[s] = __fdiv_rn(S.hp[ebase + s], P.hp);
        }
    }
    __syncthreads();
    float *mini = (float *)(rec + R.mini);
    for (int c = tid; c < 2 * kViewCells; c += nt) {
        const int tot = c >= kViewCells ? n1 : n0;
        mini[c] = tot > 0 ? __fdiv_rn((float)s_cnt[c], (float)tot) : 0.0f;
    }
}

// Episode start from the placement template of env e (k_place at commit, k_step's auto-reset).  `side` = 1 swaps the
// armies: group g takes the other block's positions AND ids -- generate_map adds the left block first, so the ids
// follow the side, not the group (senario_battle.py:14-37).
__device__ __forceinline__ void place_from_template(const BattleParams &P, const BattleState &S, int e, int side) {
    const int cap = P.cap, n_action = P.n_move + P.n_attack;
    const size_t ebase = (size_t)e * 2 * cap;
    const int32_t *tpos = S.init_pos + (size_t)e * P.tmpl_stride;          // [2][cap] pos, then [2][cap] id
    const int32_t *tnum = S.init_num + (P.tmpl_stride ? 2 * e : 0);
    for (int s = threadIdx.x; s < 2 * cap; s += blockDim.x) {
        const int g = s >= cap, i = s - g * cap, src = (side ? 1 - g : g) * cap + i;
        const bool live = i < tnum[side ? 1 - g : g];
        S.pos[ebase + s] = live ? tpos[src] : 0;
        S.hp[ebase + s] = P.hp;
        S.id[ebase + s] = live ? tpos[2 * cap + src] : 0;
        S.state[ebase + s] = make_state(0, OP_NULL, (uint32_t)n_action);   // GridWorld.h:145
        S.next_rew[ebase + s] = P.step_reward;                             // Agent::init_reward
        S.last_rew[ebase + s] = 0.0f;
    }
    if (threadIdx.x < 2) { S.num[e * 2 + threadIdx.x] = tnum[side ? 1 - threadIdx.x : threadIdx.x]; S.dead_ct[e * 2 + threadIdx.x] = 0; }
    if (threadIdx.x == 0) { S.step_ct[e] = 0; S.id_counter[e] = tnum[0] + tnum[1]; S.side[e] = side; }
}

// minstd_rand0 after n steps from state s: s * 16807^n mod (2^31 - 1), square and multiply over a table of
// 16807^(2^b) -- the reference's sequential chain (GridWorld.cc:510-515 draws one number per attack) without the chain.
// 14 bits: n <= 2 * 8191, one draw per attack of a step (tests/test_minstd_jump_table.py checks the table).
__device__ __forceinline__ uint32_t minstd_jump(uint32_t s, uint32_t n) {
    const uint32_t pw[14] = {16807u, 282475249u, 984943658u, 1457850878u, 1137522503u, 1636807826u,
                             685118024u, 515204530u, 897054849u, 2038299453u, 1836275591u, 349037107u,
                             149796865u, 1186652285u};
    uint64_t acc = s;
#pragma unroll
    for (int b = 0; b < 14; b++)
        if ((n >> b) & 1u) acc = (acc * pw[b]) % 2147483647ull;
    return (uint32_t)acc;
}

// Random placement (mfb_add_agents_random), the second stage of an episode start: call after place_from_template and a
// __syncthreads, from every thread of the CTA.  occ: scratch bitmap of W*H bits (shared or global memory).
//
// The reference's sequential loop (GridWorld.cc:236-255, Map::get_random_blank Map.cc:49-63; runtime_api.cu's host
// loop): per agent, draw candidates until one is blank -- inside x + 1 < W, y + 1 < H, not a wall, not an agent -- and
// give up after W*H + 1 failures (then the rest of the op is not placed either).  One warp runs it 32 candidates at a
// time: lane l evaluates candidate t + l against the bitmap; a candidate is accepted if it is blank and the first blank
// one of the batch on its cell (__match_any_sync), and a lane-uniform scan of the accepted mask replays the sequential
// bookkeeping (agents placed, failures of the current agent) to find how many candidates the loop consumed.  MINSTD:
// candidate t is draws 2t+1 and 2t+2 of the env's stream (x = x0 + r1 % w, y = y0 + r2 % h), and the stream is left
// right after the last candidate consumed.  Philox: candidate t of op k is counter (t, k, episode, generation | 2^31)
// under the key (seed, env_base + e), x = x0 + mulhi(word0, w), y = y0 + mulhi(word1, h); the top bit of word 3 keeps
// it apart from the attack shuffle's (i, step, 0, 0) and random_sides' (episode, 0x51DE, 0, 0) counters.
__device__ __forceinline__ void place_random(const BattleParams &P, const BattleState &S, const RandomPlacement &RP, int e,
                                             int side, int episode, uint32_t *occ) {
    const int tid = threadIdx.x, nt = blockDim.x, W = P.W, H = P.H, cap = P.cap, cells = W * H;
    const int words = (cells + 31) >> 5;
    const size_t ebase = (size_t)e * 2 * cap;
    const uint8_t *walls = S.walls + (size_t)e * P.wall_stride;
    for (int w = tid; w < words; w += nt) {
        uint32_t bits = 0;
        for (int b = 0; b < 32 && 32 * w + b < cells; b++) bits |= (uint32_t)(walls[32 * w + b] != 0) << b;
        occ[w] = bits;
    }
    __syncthreads();
    const int n0 = S.num[e * 2], n1 = S.num[e * 2 + 1];   // the fixed template, as place_from_template left it
    for (int s = tid; s < 2 * cap; s += nt) {
        const int g = s >= cap, i = s - g * cap;
        if (i < (g ? n1 : n0)) {
            const int p = S.pos[ebase + s], c = pos_y(p) * W + pos_x(p);
            atomicOr(&occ[c >> 5], 1u << (c & 31));
        }
    }
    __syncthreads();
    if (tid >= 32) return;
    const volatile uint32_t *vocc = occ;   // this warp's own atomics must be seen by its later loads (global: not L1)
    const int lane = tid;
    const unsigned full = 0xFFFFFFFFu, below = (1u << lane) - 1u;
    const bool minstd = P.rng_mode != RNG_PHILOX;
    const uint32_t max_fails = (uint32_t)cells + 1u;
    uint32_t rs = minstd ? S.rng[e] : 0u;
    int num0 = n0, num1 = n1, id_end = S.id_counter[e], short_ct = 0;
    for (int k = 0; k < RP.n_ops; k++) {
        const RandomOp op = RP.ops[k];
        const int g = op.group ^ side, id0 = id_end + op.id0, base = g ? num1 : num0;
        int placed = 0;
        uint32_t fails = 0, t = 0;
        bool gave_up = false;
        while (placed < op.n && !gave_up) {
            uint32_t x, y, rs_after = 0;
            if (minstd) {
                const uint32_t r1 = minstd_jump(rs, 2u * lane + 1u), r2 = minstd_next(r1);
                x = (uint32_t)op.x0 + r1 % (uint32_t)op.w; y = (uint32_t)op.y0 + r2 % (uint32_t)op.h;
                rs_after = r2;
            } else {
                const uint4 r = philox4x32_10(make_uint4(t + lane, (uint32_t)k, (uint32_t)episode, RP.generation | 0x80000000u),
                                              make_uint2(P.seed, (uint32_t)(P.env_base + e)));
                x = (uint32_t)op.x0 + __umulhi(r.x, (uint32_t)op.w); y = (uint32_t)op.y0 + __umulhi(r.y, (uint32_t)op.h);
            }
            const int c = (int)(y * W + x);
            const bool blank = x + 1 < (uint32_t)W && y + 1 < (uint32_t)H && !((vocc[c >> 5] >> (c & 31)) & 1u);
            const unsigned peers = __match_any_sync(full, blank ? c : -1 - lane);
            unsigned ok = __ballot_sync(full, blank && lane == __ffs(peers) - 1);
            // the sequential loop over this batch: accepted candidates in lane order, failures in between
            unsigned acc = 0;
            int consumed = 32, pos = 0;
            for (;;) {
                const int next = ok ? __ffs(ok) - 1 : 32;
                const uint32_t gap = (uint32_t)(next - pos);
                if (fails + gap >= max_fails) { consumed = pos + (int)(max_fails - fails); gave_up = true; break; }
                if (next == 32) { fails += gap; break; }
                acc |= 1u << next; ok &= ok - 1u; fails = 0; pos = next + 1;
                if (placed + __popc(acc) == op.n) { consumed = pos; break; }
            }
            if ((acc >> lane) & 1u) {
                const int idx = placed + __popc(acc & below), s = g * cap + base + idx;
                S.pos[ebase + s] = pack_pos((int)x, (int)y);
                S.id[ebase + s] = id0 + idx;
                atomicOr(&occ[c >> 5], 1u << (c & 31));
            }
            placed += __popc(acc);
            if (minstd) rs = __shfl_sync(full, rs_after, consumed - 1);
            t += (uint32_t)consumed;
            __syncwarp();
        }
        if (g) num1 += placed; else num0 += placed;
        short_ct += op.n - placed;
    }
    if (lane == 0) {
        S.num[e * 2] = num0; S.num[e * 2 + 1] = num1;
        if (RP.n_ops > 0) {
            const RandomOp last = RP.ops[RP.n_ops - 1];
            S.id_counter[e] = id_end + last.id0 + last.n;
        }
        if (minstd) S.rng[e] = rs;
        RP.place_short[e] = short_ct;
    }
}

// ----------------------------------------------------------------------------------------------
// K2: fused step
// ----------------------------------------------------------------------------------------------
struct StepSmem {  // byte offsets into dynamic shared memory
    int pos, hp, nr, state, att, aux, mv, mvt, tag_a, tag_v, mvidx, scr0, scr1, grid, misc, total;
};
__host__ __device__ inline StepSmem step_smem_layout(int W, int H, int cap, int obs_cached) {
    StepSmem L;
    const int n = 2 * cap;
    int o = 0;
    L.pos = o;   o += 4 * n;
    L.hp = o;    o += 4 * n;
    L.nr = o;    o += 4 * n;
    L.state = o; o += 4 * n;
    L.att = o;   o += 4 * n;   // attack list: slot | attack index << 16 (| 1 << 31 once it acted)
    L.aux = o;   o += 4 * n;   // shuffle draws, then victim slot per attack (-1 = miss)
    L.mv = o;    o += 4 * n;   // move list: slot | move index << 16
    L.mvt = o;   o += 4 * n;   // target cell per move, or -1 = no attempt (outside the board, dead mover)
    L.scr0 = o;  o += 4 * n;   // shuffle: list heads | attacks: hits per slot, attacker flag | moves: result per mover
    L.scr1 = o;  o += 4 * n;   // shuffle: list links | attacks: the entangled attacks, in order | moves: dependency
    L.tag_a = o; o += 2 * n;   // batch tag: slot attacks in the current 32-attack batch
    L.tag_v = o; o += 2 * n;   // batch tag: slot is attacked in the current batch
    L.mvidx = o; o += 2 * n;   // 1 + index in the move list of a mover that tries to leave its cell (0 = it stays)
    L.misc = o;  o += 4 * 128; // warp totals [32], counters, action histogram [2][32]
    L.grid = o;                    // per cell: occupant code (low half: 0 empty, 1 wall, 2 + slot) | claim << 16, the first
    {                              // mover entitled to the cell (min over move-list indices, 0xFFFF = nobody);
        int bytes = 4 * W * H;     // afterwards the scratch of build_obs_record (padded u16 grid + minimap counts)
        const int need = obs_record_layout(W, H, cap).hp10 + 4 * 2 * kViewCells;
        if (obs_cached && need > bytes) bytes = need;
        o += (bytes + 15) & ~15;
    }
    L.total = (o + 15) & ~15;
    return L;
}

enum { MISC_WARP = 0, MISC_N = 32, MISC_DEAD = 34, MISC_FLAG = 40, MISC_HIST = 64 };   // ints in s_misc

// mover results while the move phase runs
enum : int { MV_FAIL = 0, MV_OK = 1, MV_WAIT = 2 };

// Dynamic shared memory of k_step<true>: s_misc, then the minimap counts of build_obs_record_hbm.
constexpr int kStepHbmSmem = 4 * 128 + 4 * 2 * kViewCells;
// k_step<true>'s workspace: [E][step_smem_layout().total], right after the E observation records
__host__ __device__ inline unsigned char *step_workspace(const BattleParams &P, const BattleState &S) {
    return S.obs_record + (size_t)P.E * obs_record_layout(P.W, P.H, P.cap).total;
}

// HBM = false: the working set lives in dynamic shared memory (step_smem_layout(...).total bytes).  HBM = true, for
// geometries whose layout exceeds a CTA's shared memory: the same layout in HBM, in the env's slice of the workspace
// that follows the observation records (always kept at such geometries) in their allocation -- the shared atomics
// become global atomics on the env's own lines, served by L2.  Only s_misc and the minimap counts stay in shared
// memory (kStepHbmSmem bytes), and the observation record is built in place.
// RANDOM = true (engines with random placement ops): the auto-reset runs place_random after the template.  A separate
// instantiation, so that an engine without random ops runs k_step with the registers and code it always had.
template <bool HBM, bool RANDOM = false>
__global__ void k_step(const __grid_constant__ BattleParams P, const BattleState S, const StepIO io, const RandomPlacement RP) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const StepSmem L = step_smem_layout(P.W, P.H, P.cap, P.obs_cached);
    unsigned char *const ws = HBM ? step_workspace(P, S) + (size_t)blockIdx.x * L.total : nullptr;
#define STEP_AT(off) (HBM ? ws + (off) : smem_raw + (off))
    int *s_pos = (int *)STEP_AT(L.pos);
    float *s_hp = (float *)STEP_AT(L.hp);
    float *s_nr = (float *)STEP_AT(L.nr);
    uint32_t *s_state = (uint32_t *)STEP_AT(L.state);
    uint32_t *s_att = (uint32_t *)STEP_AT(L.att);
    int *s_aux = (int *)STEP_AT(L.aux);
    uint32_t *s_mv = (uint32_t *)STEP_AT(L.mv);
    int *s_mvt = (int *)STEP_AT(L.mvt);
    int *s_scr0 = (int *)STEP_AT(L.scr0);
    int *s_scr1 = (int *)STEP_AT(L.scr1);
    uint16_t *s_tag_a = (uint16_t *)STEP_AT(L.tag_a);
    uint16_t *s_tag_v = (uint16_t *)STEP_AT(L.tag_v);
    uint16_t *s_mvidx = (uint16_t *)STEP_AT(L.mvidx);
    int *s_misc = (int *)(smem_raw + L.misc);
    if constexpr (HBM) s_misc = (int *)smem_raw;
    uint32_t *s_grid = (uint32_t *)STEP_AT(L.grid);
#undef STEP_AT
    constexpr uint32_t kNoClaim = 0xFFFF0000u;

    const int e = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int cap = P.cap, W = P.W, H = P.H, cells = W * H;
    const int n_action = P.n_move + P.n_attack;
    const size_t ebase = (size_t)e * 2 * cap;
    const int phases = io.phases;
    const int step_before = S.step_ct[e];   // read by all threads long before thread 0 rewrites it

    // ---- load: agent records -> smem, occupancy grid from walls + alive agents ----
    if (tid < 2) { s_misc[MISC_N + tid] = S.num[e * 2 + tid]; s_misc[MISC_DEAD + tid] = S.dead_ct[e * 2 + tid]; }
    const uint8_t *walls = S.walls + (size_t)e * P.wall_stride;
    if ((cells & 3) == 0) {   // 4 wall bytes -> 4 grid words per thread
        for (int c = tid; c < (cells >> 2); c += nt) {
            const uint32_t w4 = ((const uint32_t *)walls)[c];
            ((uint4 *)s_grid)[c] = make_uint4(kNoClaim | (w4 & 0xFFu), kNoClaim | ((w4 >> 8) & 0xFFu),
                                              kNoClaim | ((w4 >> 16) & 0xFFu), kNoClaim | (w4 >> 24));
        }
    } else {
        for (int c = tid; c < cells; c += nt) s_grid[c] = kNoClaim | walls[c];
    }
    __syncthreads();
    const int n0 = s_misc[MISC_N], n1 = s_misc[MISC_N + 1];
    for (int s = tid; s < 2 * cap; s += nt) {
        const int g = s >= cap, i = s - g * cap;
        if (i < (g ? n1 : n0)) {
            const int p = S.pos[ebase + s];
            uint32_t st = S.state[ebase + s];
            if ((phases & PH_SETACT) && ((io.setact_mask >> g) & 1)) {
                int a = io.actions[ebase + s];                    // Agent::set_action, GridWorld.cc:485
                a = (a < 0 || a >= n_action) ? n_action : a;      // out-of-range: recorded, never executed
                st = (st & 0xFF00FFFFu) | ((uint32_t)a << 16);
            }
            s_pos[s] = p; s_hp[s] = S.hp[ebase + s]; s_nr[s] = S.next_rew[ebase + s];
            s_state[s] = st;
            if (!st_dead(st)) s_grid[pos_y(p) * W + pos_x(p)] = kNoClaim | (uint32_t)(2 + s);
        }
        s_tag_a[s] = 0; s_tag_v[s] = 0; s_mvidx[s] = 0; s_scr0[s] = 0;
    }
    __syncthreads();

    int done = 0;
    if (phases & PH_STEP) {
        // ---- attack / move lists in set_action call order (GridWorld.cc:481-495).  On a large map (W*H > 99*99,
        //      GridWorld.cc:79-88) the reference files the moves into x-band buffers at set_action (:443-463) and runs
        //      buffer 0 .. NUM_SEP-1, then the boundary buffer (:662-672): the move list is built pass by pass in
        //      that order, each pass in call order ----
        int nA = 0, nM = 0;
        const int n_pass = P.move_bands > 0 ? P.move_bands + 1 : 1;
        for (int pass = 0; pass < n_pass; pass++) {
            for (int gi = 0; gi < kGroups; gi++) {
                const int g = io.group_seq[gi];
                if (g < 0) continue;
                const int ng = g ? n1 : n0;
                for (int base = 0; base < ng; base += nt) {
                    const int i = base + tid, s = g * cap + i;
                    const bool valid = i < ng;
                    const int a = valid ? (int)st_act(s_state[s]) : n_action;
                    bool is_mv = valid && a < P.n_move;
                    const bool is_at = pass == 0 && valid && a >= P.n_move && a < n_action;
                    if (is_mv && n_pass > 1) {
                        const int x = pos_x(s_pos[s]), xr = x % P.band_width;
                        const int band = (xr < 4 || xr > P.band_width - 4) ? P.move_bands : x / P.band_width;
                        is_mv = band == pass;
                    }
                    int tot;
                    const int p = block_scan_flags2(is_at, is_mv, s_misc + MISC_WARP, tot);
                    if (is_at) s_att[nA + (p & 0xFFFF)] = (uint32_t)s | ((uint32_t)(a - P.n_move) << 16);
                    if (is_mv) s_mv[nM + (p >> 16)] = (uint32_t)s | ((uint32_t)a << 16);
                    nA += tot & 0xFFFF; nM += tot >> 16;
                }
            }
        }
        __syncthreads();

        // ---- shuffle attacks (GridWorld.cc:510-515): inside-out Fisher-Yates, draw i picks j_i in [0, i] and swaps
        //      positions i and j_i ----
        if (P.rng_mode == RNG_INJECT) {
            const int32_t *perm = io.attack_perm + (size_t)e * 2 * cap;
            for (int i = tid; i < nA; i += nt) s_aux[i] = (int)s_att[perm[i]];
            __syncthreads();
            for (int i = tid; i < nA; i += nt) s_att[i] = (uint32_t)s_aux[i];
        } else if (nA > 0) {
            // the draws, all at once: Philox is counter based; the reference's minstd_rand0 chain is jumped ahead
            // (state after i+1 steps = state * 16807^(i+1))
            const uint32_t rs0 = P.rng_mode == RNG_MINSTD ? S.rng[e] : 0u;
            uint32_t rs_end = 0;                       // the engine's state after the last draw (held by the thread that made it)
            bool made_last_draw = false;
            for (int i = tid; i < nA; i += nt) {
                if (P.rng_mode == RNG_PHILOX) {
                    const uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)step_before, 0u, 0u),
                                                  make_uint2(P.seed, (uint32_t)(P.env_base + e)));
                    s_aux[i] = (int)(r.x % (uint32_t)(i + 1));
                } else {
                    const uint32_t rs = minstd_jump(rs0, (uint32_t)(i + 1));
                    s_aux[i] = (int)rs % (i + 1);
                    if (i == nA - 1) { rs_end = rs; made_last_draw = true; }
                }
                s_scr0[i] = -1;
            }
            __syncthreads();
            if (made_last_draw) S.rng[e] = rs_end;     // (after the barrier: every thread has read the old state by now)
            // No swap is executed.  Position i still holds element i when step i runs, so the content of position q
            // after all steps < t is: element i* if i* is the LAST step in (q, t) that swapped into q (j_i* = q);
            // otherwise what position j_q held after the steps < q (step q itself moved it in).  Every final position
            // follows that trace on its own -- O(log n) hops expected -- through per-position lists of the steps
            // that swap into it.  (tests/test_parallel_resolve_model.py checks this against the swap loop.)
            for (int i = tid; i < nA; i += nt) s_scr1[i] = atomicExch(&s_scr0[s_aux[i]], i);
            __syncthreads();
            for (int p = tid; p < nA; p += nt) {
                int q = p, t = nA, src;
                for (;;) {
                    int best = -1;
                    for (int i = s_scr0[q]; i >= 0; i = s_scr1[i])
                        if (i > q && i < t && i > best) best = i;
                    if (best >= 0) { src = best; break; }
                    const int jq = s_aux[q];
                    if (jq == q) { src = q; break; }
                    t = q; q = jq;
                }
                s_mvt[p] = (int)s_att[src];                     // (s_mvt is free until the move phase)
            }
            __syncthreads();
            for (int p = tid; p < nA; p += nt) s_att[p] = (uint32_t)s_mvt[p];
            for (int s = tid; s < 2 * cap; s += nt) s_scr0[s] = 0;
        }
        __syncthreads();

        // ---- victims (Map::get_attack_obj, Map.cc:220-263): positions are frozen during the attack
        //      phase, so the only thing that can change before an attack's turn is the victim dying.
        //      s_scr0[slot] counts the attacks aimed at the slot (low half) and flags the slot as an attacker ----
        for (int i = tid; i < nA; i += nt) {
            const uint32_t ent = s_att[i];
            const int k = ent & 0xFFFF, a = ent >> 16, p = s_pos[k];
            const int tx = pos_x(p) + P.att_dx[a], ty = pos_y(p) + P.att_dy[a];
            int v = -1;
            if (tx >= 0 && tx < W && ty >= 0 && ty < H) {
                const int code = (int)(s_grid[ty * W + tx] & 0xFFFFu);
                if (code >= 2 && ((code - 2) >= cap) != (k >= cap)) v = code - 2;
            }
            s_aux[i] = v;
            atomicAdd(&s_scr0[k], 0x10000);
            if (v >= 0) atomicAdd(&s_scr0[v], 1);
        }
        __syncthreads();

        // ---- ordered attack resolve (GridWorld.cc:524-557 run single-threaded, Map::do_attack Map.cc:266-321) ----
        auto one_attack = [&](int k, int v, int i) {
            if (st_dead(s_state[k])) return;                               // attacker died earlier this step
            s_att[i] |= 0x80000000u;                                       // it acted: a render attack event (GridWorld.cc:533)
            if (v < 0 || st_dead(s_state[v])) {                            // blank / wall / team-mate / already dead
                s_nr[k] = s_nr[k] + P.attack_penalty;
                return;
            }
            const float hp = s_hp[v] - P.damage;                           // Agent::be_attack, GridWorld.h:208-214
            s_hp[v] = hp;
            float reward = 0.0f;
            if (hp < 0.0f) {
                s_state[v] |= 1u;
                s_nr[v] = P.dead_penalty;
                const int pv = s_pos[v];
                s_grid[pos_y(pv) * W + pos_x(pv)] = kNoClaim;              // Map::remove_agent
                atomicAdd(&s_misc[MISC_DEAD + (v >= cap)], 1);
                s_state[k] = st_with_op(s_state[k], OP_KILL);
                s_hp[k] = fminf(P.hp, s_hp[k] + P.kill_supply);            // Agent::add_hp
                reward = P.kill_reward;
            } else {
                s_state[k] = st_with_op(s_state[k], OP_ATTACK);
            }
            s_nr[k] = s_nr[k] + (reward + P.attack_penalty);               // GridWorld.cc:556
        };
        // (1) ISOLATED attacks, all at once.  (k -> v) is isolated when nobody attacks k this step -- so k is alive at
        // its turn whenever that is -- and either it hits nothing, or it is the only attack on v and cannot change what
        // v itself does (v does not attack, or survives the hit).  Such an attack reads and writes nothing any other
        // attack of the step reads or writes, so its place in the shuffled order does not matter.  kill_supply > 0
        // would let a kill change the killer's hp, which a later hit on the killer reads: then nothing is isolated.
        // (2) The entangled rest keeps its order: compacted in order, resolved below.
        int nE = 0;
        for (int base = 0; base < nA; base += nt) {
            const int i = base + tid;
            bool entangled = false;
            if (i < nA) {
                const int k = (int)(s_att[i] & 0xFFFF), v = s_aux[i];
                bool iso = P.kill_supply == 0.0f && (s_scr0[k] & 0xFFFF) == 0;
                if (iso && v >= 0) {
                    const int cv = s_scr0[v];
                    iso = (cv & 0xFFFF) == 1 && ((cv >> 16) == 0 || !(s_hp[v] - P.damage < 0.0f));
                }
                if (iso) one_attack(k, v, i);
                entangled = !iso;
            }
            int tot;
            const int p = block_scan_flag(entangled, s_misc + MISC_WARP, tot);
            if (entangled) s_scr1[nE + p] = i;
            nE += tot;
        }
        __syncthreads();
        // Sequential semantics for the entangled attacks, executed by warp 0 in batches of 32 consecutive entries.
        // An attack (k -> v) whose attacker is attacked by nobody else in the batch and whose victim
        // neither is attacked by another lane nor attacks in this batch touches state no other lane of the
        // batch reads or writes: those lanes run in parallel.  The rest ("complex") run one lane at a time
        // in lane order, i.e. in the shuffled order; since the simple lanes commute with them the result is
        // bit-identical to the one-by-one loop.
        if (tid < 32) {
            const int lane = tid;
            for (int i0 = 0, bid = 1; i0 < nE; i0 += 32, bid++) {
                const bool valid = i0 + lane < nE;
                const int i = valid ? s_scr1[i0 + lane] : 0;
                const int k = valid ? (int)(s_att[i] & 0xFFFF) : 0;
                const int v = valid ? s_aux[i] : -1;
                if (valid) s_tag_a[k] = (uint16_t)bid;
                if (v >= 0) s_tag_v[v] = (uint16_t)bid;
                __syncwarp();
                const unsigned same_v = __match_any_sync(0xFFFFFFFFu, v >= 0 ? v : -1 - lane);
                const bool complex = valid && (s_tag_v[k] == bid ||
                                               (v >= 0 && (__popc(same_v) > 1 || s_tag_a[v] == bid)));
                if (valid && !complex) one_attack(k, v, i);
                __syncwarp();
                unsigned todo = __ballot_sync(0xFFFFFFFFu, complex);
                while (todo) {
                    const int l = __ffs(todo) - 1;
                    todo &= todo - 1;
                    if (lane == l) one_attack(k, v, i);
                    __syncwarp();
                }
            }
        }
        __syncthreads();

        if (io.attack_events) {   // RenderAttackEvent{id, obj_x, obj_y} in processing order (GridWorld.cc:518-560)
            int32_t *ev = io.attack_events + (size_t)e * (1 + 6 * cap);
            if (tid == 0) ev[0] = nA;
            for (int i = tid; i < nA; i += nt) {
                const uint32_t ent = s_att[i];
                const int k = ent & 0xFFFF, a = (ent >> 16) & 0x7FFF, p = s_pos[k];
                ev[1 + 3 * i] = (ent >> 31) ? S.id[ebase + k] : -1;
                ev[2 + 3 * i] = pos_x(p) + P.att_dx[a];
                ev[3 + 3 * i] = pos_y(p) + P.att_dy[a];
            }
        }
        // ---- starve / recover (GridWorld.cc:574-595, Agent::starve GridWorld.h:199-206) ----
        for (int s = tid; s < 2 * cap; s += nt) {
            const int g = s >= cap, i = s - g * cap;
            if (i >= (g ? n1 : n0) || st_dead(s_state[s])) continue;
            if (P.step_recover > 0.0f) {
                s_hp[s] = fminf(P.hp, s_hp[s] + P.step_recover);
            } else {
                const float hp = s_hp[s] - (-P.step_recover);
                s_hp[s] = hp;
                if (hp < 0.0f) {
                    s_state[s] |= 1u; s_nr[s] = P.dead_penalty;
                    s_grid[pos_y(s_pos[s]) * W + pos_x(s_pos[s])] = kNoClaim;
                    atomicAdd(&s_misc[MISC_DEAD + g], 1);
                }
            }
        }
        __syncthreads();

        // ---- ordered moves, first come first served (GridWorld.cc:631-672, Map::do_move Map.cc:324-369), resolved
        //      without walking the list.  What mover m finds in its target cell at its turn depends only on
        //        * what stands there before the move phase: nothing, a wall, or an agent o, and
        //        * o's own turn j_o if o tries to leave (a mover staying put -- move (0, 0) -- never frees its cell):
        //      movers with m < j_o find o still there; of those with m > j_o (or all, if the cell was empty) only the
        //      FIRST can get the cell -- an atomicMin over list indices per cell -- and it does iff the cell was empty
        //      or o really left, i.e. iff o won ITS target: a chain, followed by pointer jumping until every mover
        //      knows.  Everybody else collides with whoever holds the cell at their turn (or, at a wall, does nothing).
        //      Then all winners vacate, then enter.  (Model + exactness test: tests/test_parallel_resolve_model.py.)
        for (int m = tid; m < nM; m += nt) {
            const uint32_t ent = s_mv[m];
            const int k = ent & 0xFFFF, a = ent >> 16, p = s_pos[k];
            const int nx = pos_x(p) + P.move_dx[a], ny = pos_y(p) + P.move_dy[a];
            const bool cand = !(nx < 0 || ny < 0 || nx + 1 >= W || ny + 1 >= H) && !st_dead(s_state[k]);   // Map.cc:466-468
            s_mvt[m] = cand ? ny * W + nx : -1;
            if (cand && pack_pos(nx, ny) != p) s_mvidx[k] = (uint16_t)(m + 1);
        }
        __syncthreads();
        for (int m = tid; m < nM; m += nt) {
            const int tc = s_mvt[m], k = (int)(s_mv[m] & 0xFFFF);
            int res = MV_FAIL, dep = -1;
            if (tc >= 0) {
                const int occ = (int)(s_grid[tc] & 0xFFFFu);
                if (occ == 0) res = MV_WAIT;                                   // contender for an empty cell
                else if (occ >= 2 && occ != 2 + k) {
                    const int j = (int)s_mvidx[occ - 2] - 1;
                    if (j >= 0 && j < m) { res = MV_WAIT; dep = j; }           // the occupant had its turn before m
                    else s_state[k] = st_with_op(s_state[k], OP_COLLIDE);      // it is still there (no reward effect in battle)
                }                                                              // own cell: stays; wall: nothing (Map.cc:498-513)
                if (res == MV_WAIT) atomicMin(&s_grid[tc], ((uint32_t)m << 16) | (uint32_t)occ);   // every contender sees the same occupant
            }
            s_scr0[m] = res; s_scr1[m] = dep;
        }
        __syncthreads();
        for (int m = tid; m < nM; m += nt) {
            if (s_scr0[m] != MV_WAIT) continue;
            if ((s_grid[s_mvt[m]] >> 16) != (uint32_t)m) {                            // an earlier contender is entitled to the cell
                s_scr0[m] = MV_FAIL;
                const int k = (int)(s_mv[m] & 0xFFFF);
                s_state[k] = st_with_op(s_state[k], OP_COLLIDE);
            } else if (s_scr1[m] < 0) s_scr0[m] = MV_OK;
        }
        for (;;) {
            __syncthreads();
            if (tid == 0) s_misc[MISC_FLAG] = 0;
            __syncthreads();
            bool waiting = false;
            for (int m = tid; m < nM; m += nt) {
                if (s_scr0[m] != MV_WAIT) continue;
                const int d = s_scr1[m], r = s_scr0[d];        // a racing writer can only turn WAIT into the final value
                if (r == MV_WAIT) { s_scr1[m] = s_scr1[d]; waiting = true; }   // same fate as the occupant's occupant
                else {
                    s_scr0[m] = r;
                    if (r == MV_FAIL) { const int k = (int)(s_mv[m] & 0xFFFF); s_state[k] = st_with_op(s_state[k], OP_COLLIDE); }
                }
            }
            if (waiting) s_misc[MISC_FLAG] = 1;
            __syncthreads();
            if (!s_misc[MISC_FLAG]) break;
        }
        for (int m = tid; m < nM; m += nt)
            if (s_scr0[m] == MV_OK) { const int p = s_pos[s_mv[m] & 0xFFFF]; s_grid[pos_y(p) * W + pos_x(p)] = kNoClaim; }
        __syncthreads();
        for (int m = tid; m < nM; m += nt)
            if (s_scr0[m] == MV_OK) {
                const int k = (int)(s_mv[m] & 0xFFFF), tc = s_mvt[m];
                s_grid[tc] = kNoClaim | (uint32_t)(2 + k);
                const int ty = tc / W;
                s_pos[k] = pack_pos(tc - ty * W, ty);
            }
        __syncthreads();

        // ---- reward rules (calc_reward GridWorld.cc:744-758): for the battle rule set an agent whose
        //      last_op is OP_ATTACK necessarily hit the other group; dead agents included ----
        for (int s = tid; s < 2 * cap; s += nt) {
            const int g = s >= cap, i = s - g * cap;
            if (i < (g ? n1 : n0) && st_op(s_state[s]) == OP_ATTACK) s_nr[s] = s_nr[s] + P.attack_bonus[g];
        }
        // ---- done (GridWorld.cc:680-686) ----
        done = (n0 - s_misc[MISC_DEAD] <= 0) || (n1 - s_misc[MISC_DEAD + 1] <= 0);
        __syncthreads();
        if (tid == 0) {
            if (io.done) io.done[e] = done;
            S.step_ct[e] = step_before + 1;
            S.agent_steps[e] += (unsigned long long)(n0 + n1);
        }
    }

    // ---- export: get_reward (+ group reward, always 0), alive, mean action of this step ----
    if (phases & PH_EXPORT) {
        for (int s = tid; s < 2 * cap; s += nt) {
            const int g = s >= cap, i = s - g * cap;
            if (i < (g ? n1 : n0)) {
                if (io.reward) io.reward[ebase + s] = s_nr[s] + 0.0f;
                if (io.alive) io.alive[ebase + s] = (uint8_t)!st_dead(s_state[s]);
            }
        }
        if (io.mean_action) {
            // one-hot mean = action histogram / n: lanes of a warp holding the same (group, action) elect one of them
            // to add their count to the shared histogram
            if (tid < 64) s_misc[MISC_HIST + tid] = 0;
            __syncthreads();
            for (int base = 0; base < 2 * cap; base += nt) {
                const int s = base + tid, g = s >= cap, i = s - g * cap;
                const bool valid = s < 2 * cap && i < (g ? n1 : n0);
                const int a = valid ? (int)st_act(s_state[s]) : n_action;
                const int key = (valid && a < n_action) ? g * 32 + a : -1 - (int)(tid & 31);
                const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
                if (key >= 0 && (int)(tid & 31) == __ffs(peers) - 1) atomicAdd(&s_misc[MISC_HIST + key], __popc(peers));
            }
            __syncthreads();
            if (tid < 64) {
                const int g = tid >> 5, b = tid & 31, ng = g ? n1 : n0;
                if (b < n_action)
                    io.mean_action[((size_t)e * 2 + g) * n_action + b] =
                        ng > 0 ? __fdiv_rn((float)s_misc[MISC_HIST + tid], (float)ng) : 0.0f;
            }
        }
    }

    // ---- write back; clear_dead = stable compaction of the survivors (GridWorld.cc:696-728) ----
    const bool horizon = (phases & PH_STEP) && P.max_steps > 0 && step_before + 1 >= P.max_steps;
    if ((phases & PH_AUTORESET) && (done || horizon)) {
        __syncthreads();
        int side = 0;
        const int episode = S.episode[e] + 1;
        __syncthreads();                                  // everybody has read the counter before thread 0 advances it
        if (P.random_sides) {
            const uint4 r = philox4x32_10(make_uint4((uint32_t)episode, 0x51DEu, 0u, 0u), make_uint2(P.seed, (uint32_t)(P.env_base + e)));
            side = (int)(r.x & 1u);
        }
        place_from_template(P, S, e, side);
        if constexpr (RANDOM) {   // the step's grid is dead by now: its shared memory holds the placer's bitmap
            __syncthreads();
            place_random(P, S, RP, e, side, episode,
                         HBM ? RP.occ + (size_t)e * ((cells + 31) >> 5) : (uint32_t *)(smem_raw + L.grid));
        }
        if (tid == 0) S.episode[e] = episode;
    } else if (phases & PH_CLEAR) {
        for (int g = 0; g < kGroups; g++) {
            const int ng = g ? n1 : n0;
            int kept = 0;
            for (int base = 0; base < ng; base += nt) {
                const int i = base + tid, s = g * cap + i;
                const bool keep = i < ng && !st_dead(s_state[s]);
                // ids are read at the old index before the scan's barriers; survivors only move to lower or
                // equal indices of rounds already consumed, so the in-place rewrite cannot clobber a pending read
                const int my_id = keep ? S.id[ebase + s] : 0;
                int tot;
                const int p = block_scan_flag(keep, s_misc + MISC_WARP, tot);
                if (keep) {
                    const size_t d = ebase + (size_t)g * cap + kept + p;
                    S.pos[d] = s_pos[s]; S.hp[d] = s_hp[s]; S.id[d] = my_id;
                    S.state[d] = make_state(0, OP_NULL, st_act(s_state[s]));   // Agent::init_reward
                    S.last_rew[d] = s_nr[s];
                    S.next_rew[d] = P.step_reward;
                }
                kept += tot;
            }
            if (tid == 0) { S.num[e * 2 + g] = kept; S.dead_ct[e * 2 + g] = 0; }
        }
    } else if (phases & (PH_STEP | PH_SETACT)) {
        for (int s = tid; s < 2 * cap; s += nt) {
            const int g = s >= cap, i = s - g * cap;
            if (i < (g ? n1 : n0)) {
                S.pos[ebase + s] = s_pos[s]; S.hp[ebase + s] = s_hp[s];
                S.state[ebase + s] = s_state[s]; S.next_rew[ebase + s] = s_nr[s];
            }
        }
        if (tid < 2) S.dead_ct[e * 2 + tid] = s_misc[MISC_DEAD + tid];
    }
    if (io.mirror.pos != nullptr) {                               // single-env ABI: the host's copy of the records
        __syncthreads();                                          // the write-back above is visible to the whole CTA
        for (int s = tid; s < 2 * cap; s += nt) {
            io.mirror.pos[s] = S.pos[ebase + s]; io.mirror.id[s] = S.id[ebase + s]; io.mirror.state[s] = S.state[ebase + s];
            io.mirror.hp[s] = S.hp[ebase + s]; io.mirror.next_rew[s] = S.next_rew[ebase + s];
            io.mirror.last_rew[s] = S.last_rew[ebase + s];
        }
        if (tid < 2) { io.mirror.head[tid] = S.num[e * 2 + tid]; io.mirror.head[2 + tid] = S.dead_ct[e * 2 + tid]; }
        if (tid == 0) { io.mirror.head[4] = done; io.mirror.head[5] = S.step_ct[e]; }
    }
    if (P.obs_cached && (phases & (PH_STEP | PH_CLEAR))) {        // positions / alive flags / slot indices changed
        __syncthreads();                                          // the write-back above is visible to the whole CTA
        if constexpr (HBM)
            build_obs_record_hbm(P, S, e, (int *)(smem_raw + 4 * 128));
        else
            build_obs_record(P, S, e, (uint16_t *)(smem_raw + L.grid),
                             (int *)(smem_raw + L.grid + obs_record_layout(P.W, P.H, P.cap).hp10));
    }
}

// the observation record of every env after a placement (commit / late add); one CTA per env.  HBM = true: the padded
// grid is built in place in the record (shared memory: the 2*169 minimap counts only)
template <bool HBM>
__global__ void k_obs_record(const __grid_constant__ BattleParams P, const BattleState S) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    if constexpr (HBM)
        build_obs_record_hbm(P, S, blockIdx.x, (int *)smem_raw);
    else
        build_obs_record(P, S, blockIdx.x, (uint16_t *)smem_raw, (int *)(smem_raw + obs_record_layout(P.W, P.H, P.cap).hp10));
}

// ----------------------------------------------------------------------------------------------
// K1: observations.  Persistent CTAs take (env, group, tile of agents) work items from a ticket counter.
//
// The per-agent view is 13*13*7 fp32 = 4732 B, >90 % zeros, and it is the whole of the HBM traffic
// of the path.  Rows are composed in shared memory and streamed out by the TMA engine: 8 agents'
// rows sit back to back in a staging buffer (37 856 B, a multiple of 16) and one elected thread
// hands the chunk to a single cp.async.bulk shared->global store; two staging buffers keep a store
// in flight while the next chunk is composed.
//
// Composition is incremental.  The staging rows are zeroed once per CTA; cells outside the view disc never
// change again.  For the first two chunks of an item every row also receives the part all agents of the group
// share (the two minimap channels).  For each agent its warp then only
//   - looks the 113 in-disc view cells up in the shared-memory occupancy grid (4 passes of 32 lanes on a
//     host-built schedule, BattleParams::obs_cell; the grid carries a 6-cell empty margin, so a window never
//     needs a bounds test: one add + one 16-bit load),
//   - rewrites the five occupancy channels (wall, own has/hp, other has/hp) of those cells,
//   - moves the "+1" self marker of the two minimap channels.
// Shared-memory stores are stride-7-word (coprime with the 32 banks) and the schedule keeps a pass's cells in
// distinct residues mod 32 where it can: (nearly) conflict-free.
// The map is never re-read from HBM: occupancy/hp grid and both minimaps are rebuilt per item from the
// SoA agent arrays, whose loads are all issued up front (one memory round trip per item).
// ----------------------------------------------------------------------------------------------
#ifndef MF_OBS_CHUNK
#define MF_OBS_CHUNK 8
#endif
constexpr int kObsChunk = MF_OBS_CHUNK;                        // agents per bulk store (multiple of 4) = warps per CTA
constexpr int kObsThreads = 32 * kObsChunk, kObsWarps = kObsThreads / 32;
constexpr int kObsCtasPerSm = 16 / kObsChunk;                  // resident CTAs per SM the kernel is tuned for
constexpr int kObsStageBytes = kObsChunk * kViewRow * 4;       // 37 856, a multiple of 16
// bf16 rows (mfb_observe_groups_bf16): [169 cells][8 channels] bf16 -- channel 7 is padding, so a cell is one 16-byte
// vector and a row (2704 B) is what a bf16 channels-last convolution reads without a cast or a padding pass
constexpr int kViewRowBf16Bytes = kViewCells * 16;
constexpr int kObsPasses = (kViewCells + 31) / 32;             // 6
static_assert(kObsChunk == kObsWarps, "one warp composes one row of a chunk");

struct ObsSmem { int stage0, stage1, rec, hp10, mini, cnt, code, fxy, tmpl, record, total; };
constexpr int kObsMaxTile = kObsThreads;   // agents per CTA tile, upper bound (one record per thread)
// The pristine wall template is kept in shared memory when two CTAs per SM still fit with it (40x40: +5.4 KB);
// larger maps copy it from global memory (L2) per item instead.
__host__ __device__ inline bool obs_template_in_smem(int W, int H) { return (W + 2 * kPad) * (H + 2 * kPad) * 2 <= 8 * 1024; }
__host__ __device__ inline ObsSmem obs_smem_layout(int W, int H, int cap, int cached, int bf16 = 0) {
    ObsSmem L; int o = 0;
    const int stage_bytes = bf16 ? kObsChunk * kViewRowBf16Bytes : kObsStageBytes;
    L.stage0 = o; o += stage_bytes;
    L.stage1 = o; o += stage_bytes;
    L.rec = o;    o += 16 * kObsMaxTile;                              // (pos, id, state, last_rew) of the tile's agents
    L.record = L.cnt = L.tmpl = 0;
    if (cached == 2) {                                                // the record is read where it is, in HBM / L2
        L.code = L.hp10 = L.mini = 0;
        L.fxy = o;    o += 4 * (W + H);
        o = (o + 15) & ~15;
    } else if (cached) {                                              // the env's observation record, as one bulk copy lands it
        const ObsRecord R = obs_record_layout(W, H, cap);
        L.record = o; L.code = o + R.grid; L.hp10 = o + R.hp10; L.mini = o + R.mini; o += R.total;   // (16-byte pieces)
        L.fxy = o;    o += 4 * (W + H);
        o = (o + 15) & ~15;
    } else {
        L.hp10 = o;   o += 4 * 2 * cap;                                   // hp / max_hp per agent slot
        L.mini = o;   o += 4 * 2 * kViewCells;
        L.cnt = o;    o += 4 * 2 * kViewCells;
        L.code = o;   o += (2 * (W + 2 * kPad) * (H + 2 * kPad) + 3) & ~3;  // u16 per padded cell: kind << 14 | slot
        L.fxy = o;    o += 4 * (W + H);                                    // x / W and y / H as tables (features 32, 33)
        o = (o + 15) & ~15;
        L.tmpl = o;   if (obs_template_in_smem(W, H)) o += (2 * (W + 2 * kPad) * (H + 2 * kPad) + 15) & ~15;
    }
    L.total = (o + 127) & ~127;
    return L;
}

__device__ __forceinline__ void bulk_store_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
    const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(saddr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" :: "n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// cell kinds in the CTA-local grid.  Rebuilt per item (CACHED = false) they are relative to the observing group; in the
// observation record (CACHED = true) they name the group: 2 + group
enum : uint32_t { KIND_EMPTY = 0, KIND_WALL = 1, KIND_OWN = 2, KIND_OTHER = 3 };

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {     // round to nearest even, like torch's .to(bfloat16)
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// REC_HBM (CACHED only, for records too large for shared memory): the view look-ups, hp / 10 and the minimaps are read
// from the env's record in HBM / L2 instead of a shared-memory copy; everything after the look-ups is unchanged.
template <bool CACHED, bool BF16, bool REC_HBM = false>
__global__ void __launch_bounds__(kObsThreads, BF16 ? kObsCtasPerSm + 1 : kObsCtasPerSm)   // bf16 rows: smaller staging, 3 CTAs fit
k_obs(const __grid_constant__ BattleParams P, const BattleState S, const ObsIO io) {
    static_assert(CACHED || !REC_HBM, "the HBM record mode reads the observation record");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const ObsSmem L = obs_smem_layout(P.W, P.H, P.cap, REC_HBM ? 2 : (int)CACHED, BF16);
    constexpr int kRowBytes = BF16 ? kViewRowBf16Bytes : kViewRow * 4;
    constexpr int kStageBytes = kObsChunk * kRowBytes;
    float *const s_stage0 = (float *)(smem_raw + L.stage0), *const s_stage1 = (float *)(smem_raw + L.stage1);
    int4 *s_rec = (int4 *)(smem_raw + L.rec);
    float *s_hp10 = (float *)(smem_raw + L.hp10);
    float *s_mini = (float *)(smem_raw + L.mini);
    int *s_cnt = (int *)(smem_raw + L.cnt);
    uint16_t *s_code = (uint16_t *)(smem_raw + L.code);
    float *s_fxy = (float *)(smem_raw + L.fxy);
    const bool tmpl_smem = !CACHED && obs_template_in_smem(P.W, P.H);
    const uint4 *s_tmpl = tmpl_smem ? (const uint4 *)(smem_raw + L.tmpl) : (const uint4 *)S.grid_template;
    const uint32_t rec_bytes = (uint32_t)obs_record_layout(P.W, P.H, P.cap).total;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = P.W, H = P.H, cap = P.cap;
    const int PW = W + 2 * kPad, pcells = PW * (H + 2 * kPad);
    const int FS = P.feature_size, emb = P.embedding_size, n_action = P.n_move + P.n_attack;
    const uint8_t *lut = S.mini_lut;   // [W] x / scale_w, then [H] (y / scale_h) * 13

    // ---- per-lane view geometry: cell c = pass * 32 + lane -> offset in the padded grid relative to the
    //      window's top-left corner; cells outside the view disc keep offset 0 with the disc bit cleared ----
    constexpr int kDiscPasses = kObsDiscSlots / 32;
    int off[kDiscPasses], cell7[kDiscPasses];     // grid offset and staging-row offset (cell * 7) of this lane's cells; -1 = idle
#pragma unroll
    for (int it = 0; it < kDiscPasses; it++) {
        const int c = P.obs_cell[it * 32 + lane];
        const int vy = c / kView, vx = c - vy * kView;
        off[it] = c < kViewCells ? vy * PW + vx : 0;
        cell7[it] = c < kViewCells ? c * kChan : -1;
    }
    // cells outside the view disc never carry occupancy: their five occupancy channels are zeroed once here and
    // never written again (the minimap channels of all 169 cells are refreshed per item below)
    for (int i = tid; i < 2 * kStageBytes / 16; i += kObsThreads) ((uint4 *)s_stage0)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tmpl_smem)
        for (int c = tid; c < (pcells * 2 + 15) / 16; c += kObsThreads)   // padded grid with the walls, built at commit
            ((uint4 *)(smem_raw + L.tmpl))[c] = ((const uint4 *)S.grid_template)[c];
    for (int i = tid; i < W + H; i += kObsThreads)       // GridWorld.cc:419-420, the same IEEE divisions done once
        s_fxy[i] = i < W ? __fdiv_rn((float)i, (float)W) : __fdiv_rn((float)(i - W), (float)H);

    // Persistent CTAs: each loops over work items (env, group, tile).  The bulk stores are asynchronous, so
    // the grid rebuild of the next item overlaps the drain of this item's last chunks, and the staging-buffer
    // parity simply carries on across items.
    int buf = 0;
    const int groups_per_env = io.group_mask == 3 ? 2 : 1;
    const int n_items = P.E * groups_per_env * io.tiles_per_group;
    // Work distribution is DYNAMIC: a CTA takes its next item from a global ticket counter.  With a static split the
    // kernel ends when the slowest SM ends, and SMs do not drain stores at the same rate (GPCs of 16-20 SMs share
    // their path to L2): measured with the bare store loop (profiles/tma_store_probe.cu), 2.55 GB of 37 856-byte
    // bulk stores take 0.402 ms split statically over the CTAs and 0.346 ms handed out 8 chunks per ticket.
    // The ticket of the NEXT item is requested at the start of the current one, so its latency is never waited for;
    // the last CTA to finish rewinds the counters for the next launch.
    __shared__ int s_next;
    if (tid == 0) s_next = atomicAdd(&S.obs_ticket[0], 1);
    for (;;) {
        __syncthreads();                                  // s_next is set; every warp is done with the previous item
        const int item = s_next;
        __syncthreads();                                  // ... and has read it before thread 0 replaces it
        if (item >= n_items) break;
        int next_ticket = 0;
        if (tid == 0) next_ticket = atomicAdd(&S.obs_ticket[0], 1);
        int t = item;
        const int tile = t % io.tiles_per_group; t /= io.tiles_per_group;
        int g, e;
        if (io.group_mask == 3) { g = t & 1; e = t >> 1; } else { g = io.group_mask >> 1; e = t; }
        const size_t ebase = (size_t)e * 2 * cap;
        const size_t gbase = ebase + (size_t)g * cap;
        const int a_begin = tile * io.tile_agents;
        int n0, n1, ng, a_end;
        if constexpr (CACHED) {
            // The env's observation record (occupancy grid, hp / 10 per slot, both minimaps -- written by k_step) is copied
            // into shared memory as it is; every warp has finished with the previous item's record (barriers above).
            // cp.async (LDGSTS), 16 bytes per thread and instruction, NOT a bulk copy: a bulk load is queued in the SM's
            // TMA unit behind this CTA's (and its neighbour's) 38 KB bulk stores still draining -- ncu showed 24 % of
            // the samples waiting on that load's mbarrier with 32-agent tiles; the LSU path only pays the L2 latency.
            if constexpr (REC_HBM) {
                unsigned char *rec = S.obs_record + (size_t)e * rec_bytes;
                const ObsRecord R = obs_record_layout(P.W, P.H, P.cap);
                s_code = (uint16_t *)rec; s_hp10 = (float *)(rec + R.hp10); s_mini = (float *)(rec + R.mini);
            } else {
                const unsigned char *src = S.obs_record + (size_t)e * rec_bytes;
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_raw + L.record);
                for (uint32_t c = (uint32_t)tid * 16u; c < rec_bytes; c += kObsThreads * 16u)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst + c), "l"(src + c) : "memory");
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
            n0 = S.num[e * 2]; n1 = S.num[e * 2 + 1];
            int4 my_rec = make_int4(0, 0, 0, 0);                                   // agent a_begin + tid of the tile
            if (tid < io.tile_agents && a_begin + tid < cap) {
                const size_t s = gbase + a_begin + tid;
                my_rec = make_int4(S.pos[s], S.id[s], (int)S.state[s], __float_as_int(S.last_rew[s]));
            }
            ng = g ? n1 : n0;
            a_end = min(ng, a_begin + io.tile_agents);
            if (tid < a_end - a_begin) s_rec[tid] = my_rec;
            if constexpr (!REC_HBM) asm volatile("cp.async.wait_all;" ::: "memory");   // this thread's pieces have landed; the barrier at the top of
            if (a_begin >= ng) {                               // the first chunk (or of the next item) publishes everybody's
                if (tid == 0) s_next = next_ticket;
                continue;
            }
        } else {
        // Every global read of the item is issued here, up front and independent of the others (none waits for
        // `num`): slot state for the occupancy grid and the minimaps, and the tile's agent records.  One memory
        // round trip per item instead of four dependent ones.
        n0 = S.num[e * 2]; n1 = S.num[e * 2 + 1];
        constexpr int kPre = 4;                       // slots tid + j*256, j < 4, in registers (covers cap <= 512)
        int slot_pos[kPre]; uint32_t slot_state[kPre]; float slot_hp[kPre];
#pragma unroll
        for (int j = 0; j < kPre; j++) {
            const int s = tid + j * kObsThreads;
            slot_pos[j] = 0; slot_state[j] = 1u; slot_hp[j] = 0.0f;
            if (s < 2 * cap) { slot_pos[j] = S.pos[ebase + s]; slot_state[j] = S.state[ebase + s]; slot_hp[j] = S.hp[ebase + s]; }
        }
        int4 my_rec = make_int4(0, 0, 0, 0);                                       // agent a_begin + tid of the tile
        if (tid < io.tile_agents && a_begin + tid < cap) {
            const size_t s = gbase + a_begin + tid;
            my_rec = make_int4(S.pos[s], S.id[s], (int)S.state[s], __float_as_int(S.last_rew[s]));
        }
        ng = g ? n1 : n0;
        if (a_begin >= ng) {                              // nothing to do (uniform across the CTA)
            if (tid == 0) s_next = next_ticket;
            continue;
        }
        a_end = min(ng, a_begin + io.tile_agents);

        // ---- padded occupancy grid (kind << 14 | slot per cell), hp/10 per slot, minimap counts ----
        for (int c = tid; c < (pcells * 2 + 15) / 16; c += kObsThreads) ((uint4 *)s_code)[c] = s_tmpl[c];
        for (int c = tid; c < 2 * kViewCells; c += kObsThreads) s_cnt[c] = 0;
        if (tid < a_end - a_begin) s_rec[tid] = my_rec;
        __syncthreads();
        auto place = [&](int s, int p, uint32_t st, float hp) {
            const int gg = s >= cap, i = s - gg * cap;
            if (i < (gg ? n1 : n0)) {
                const int x = pos_x(p), y = pos_y(p);
                // minimap counts every agent still in the list, dead or not (GridWorld.cc:359-370)
                atomicAdd(&s_cnt[gg * kViewCells + lut[W + y] + lut[x]], 1);
                if (!st_dead(st)) {
                    s_code[(y + kPad) * PW + x + kPad] = (uint16_t)(((gg == g ? KIND_OWN : KIND_OTHER) << 14) | s);
                    s_hp10[s] = __fdiv_rn(hp, P.hp);       // Map.cc:208
                }
            }
        };
#pragma unroll
        for (int j = 0; j < kPre; j++) {
            const int s = tid + j * kObsThreads;
            if (s < 2 * cap) place(s, slot_pos[j], slot_state[j], slot_hp[j]);
        }
        for (int s = tid + kPre * kObsThreads; s < 2 * cap; s += kObsThreads)      // cap > 512: the rest from global
            place(s, S.pos[ebase + s], S.state[ebase + s], S.hp[ebase + s]);
        __syncthreads();
        for (int c = tid; c < 2 * kViewCells; c += kObsThreads) {
            const int gg = c >= kViewCells;
            // GridWorld.cc:372-377.  An empty group is unreachable in the reference's loop (done ends the episode
            // first, and :357 would dereference agents[0]); the batched driver keeps stepping finished envs, so the
            // 0/0 is defined as 0 here instead of NaN.
            const int tot = gg ? n1 : n0;
            s_mini[c] = tot > 0 ? __fdiv_rn((float)s_cnt[c], (float)tot) : 0.0f;
        }
        }
        const uint32_t kind_own = CACHED ? 2u + (uint32_t)g : (uint32_t)KIND_OWN;
        const uint32_t kind_oth = CACHED ? 3u - (uint32_t)g : (uint32_t)KIND_OTHER;
        // (the barrier at the top of the first chunk orders s_mini before its readers)
        const float *mini_own = s_mini + g * kViewCells, *mini_oth = s_mini + (1 - g) * kViewCells;

        // ---- stream the tile: compose, bulk-store ----
        // (selects, not io.view[g]: a dynamic index into a kernel parameter would spill the struct to local memory)
        float *vout = (float *)((unsigned char *)(g ? io.view[1] : io.view[0]) + (size_t)e * io.env_stride * kRowBytes);
        float *fout = (g ? io.feature[1] : io.feature[0]) + (size_t)e * io.env_stride * FS;
        int self_prev1 = -1, self_prev2 = -1;   // self-marker cell of the row in the other / this buffer
        int stale = 2;                          // staging buffers whose minimap channels belong to another item
        for (int c0 = a_begin; c0 < a_end; c0 += kObsChunk, buf ^= 1) {
            const int cn = min(kObsChunk, a_end - c0);
            // the store issued two chunks ago read this buffer: wait until its smem reads are done
            if (tid == 0) bulk_wait_read<1>();
            __syncthreads();
            int self_new = -1;
            #ifdef MF_PROFILE_BUILD
            if (warp < cn && !(io.debug & 1)) {
#else
            if (warp < cn) {
#endif
                const int4 rec = s_rec[c0 - a_begin + warp];
                const int p = rec.x, ax = pos_x(p), ay = pos_y(p);
                const int id = rec.y;
                const uint32_t st = (uint32_t)rec.z;
                const float last_rew = __int_as_float(rec.w);
                unsigned char *const row_b = (unsigned char *)(buf ? s_stage1 : s_stage0) + warp * kRowBytes;
                float *const row = (float *)row_b;
                // window top-left corner (ax - 6, ay - 6) in padded coordinates is simply (ax, ay)
                const uint16_t *win = s_code + ay * PW + ax;
                // staged (all grid look-ups, then all hp look-ups, then the stores): a store of one pass would otherwise
                // order the next pass's loads behind it and the four load -> load -> store chains would run back to back
                uint32_t code[kDiscPasses]; float hpv[kDiscPasses];
#pragma unroll
                for (int it = 0; it < kDiscPasses; it++) code[it] = (uint32_t)win[off[it]];      // idle lanes read offset 0
#pragma unroll
                for (int it = 0; it < kDiscPasses; it++) hpv[it] = s_hp10[code[it] & 0x3FFFu];
                self_new = lut[W + ay] + lut[ax];
                if constexpr (BF16) {
                    // one 16-byte vector per cell: {wall, own, own hp, own minimap | other, other hp, other minimap, 0} in bf16
                    if (stale > 0) {                    // new item: cells outside the disc only ever hold the two minimaps
#pragma unroll
                        for (int it = 0; it < kObsPasses; it++) {
                            const int c = it * 32 + lane;
                            if (c < kViewCells)
                                *(uint4 *)(row_b + c * 16) = make_uint4(0u, pack_bf16x2(0.0f, mini_own[c]), 0u, pack_bf16x2(mini_oth[c], 0.0f));
                        }
                    } else if (lane == 0 && self_prev2 >= 0) {      // the row's previous self marker (it may sit outside the disc)
                        *(uint4 *)(row_b + self_prev2 * 16) = make_uint4(0u, pack_bf16x2(0.0f, mini_own[self_prev2]), 0u,
                                                                          pack_bf16x2(mini_oth[self_prev2], 0.0f));
                    }
                    __syncwarp();
#pragma unroll
                    for (int it = 0; it < kDiscPasses; it++) {
                        if (cell7[it] >= 0) {
                            const uint32_t k = code[it] >> 14;
                            const int c = cell7[it] / kChan;
                            const float own = k == kind_own ? 1.0f : 0.0f, oth = k == kind_oth ? 1.0f : 0.0f;
                            *(uint4 *)(row_b + c * 16) = make_uint4(
                                pack_bf16x2(k == KIND_WALL ? 1.0f : 0.0f, own), pack_bf16x2(k == kind_own ? hpv[it] : 0.0f, mini_own[c]),
                                pack_bf16x2(oth, k == kind_oth ? hpv[it] : 0.0f), pack_bf16x2(mini_oth[c], 0.0f));
                        }
                    }
                    __syncwarp();
                    if (lane == 0) {                    // self marker in BOTH minimap channels (GridWorld.cc:396-408)
                        ((uint16_t *)(row_b + self_new * 16))[3] = (uint16_t)(pack_bf16x2(mini_own[self_new] + 1.0f, 0.0f) & 0xFFFFu);
                        ((uint16_t *)(row_b + self_new * 16))[6] = (uint16_t)(pack_bf16x2(mini_oth[self_new] + 1.0f, 0.0f) & 0xFFFFu);
                    }
                } else {
#pragma unroll
                for (int it = 0; it < kDiscPasses; it++) {
                    if (cell7[it] >= 0) {               // only the last pass has idle lanes
                        const uint32_t k = code[it] >> 14;
                        float *o = row + cell7[it];
                        o[0] = k == KIND_WALL ? 1.0f : 0.0f;
                        o[1] = k == kind_own ? 1.0f : 0.0f;
                        o[2] = k == kind_own ? hpv[it] : 0.0f;
                        o[4] = k == kind_oth ? 1.0f : 0.0f;
                        o[5] = k == kind_oth ? hpv[it] : 0.0f;
                    }
                }
                if (stale > 0) {                        // new item: refresh the part all its agents share
#pragma unroll
                    for (int it = 0; it < kObsPasses; it++) {
                        const int c = it * 32 + lane;
                        if (c < kViewCells) { row[c * kChan + 3] = mini_own[c]; row[c * kChan + 6] = mini_oth[c]; }
                    }
                }
                // self marker in BOTH minimap channels (GridWorld.cc:396-408): move it
                __syncwarp();
                if (lane == 0) {
                    if (stale <= 0 && self_prev2 >= 0) {
                        row[self_prev2 * kChan + 3] = mini_own[self_prev2];
                        row[self_prev2 * kChan + 6] = mini_oth[self_prev2];
                    }
                    row[self_new * kChan + 3] = mini_own[self_new] + 1.0f;
                    row[self_new * kChan + 6] = mini_oth[self_new] + 1.0f;
                }
                }
                // features (GridWorld.cc:411-421): id bits LSB first, one-hot last action, last reward, x/W, y/H
                const float fx = s_fxy[ax], fy = s_fxy[W + ay];
                const int act = (int)st_act(st);
                float *f = fout + (size_t)(c0 + warp) * FS;
                for (int k = lane; k < FS; k += 32) {
                    float v = (k < emb) ? (float)((id >> k) & 1) : ((k - emb == act) ? 1.0f : 0.0f);   // GridWorld.h:162-171
                    v = k == emb + n_action ? last_rew : v;
                    v = k == emb + n_action + 1 ? fx : v;
                    v = k == emb + n_action + 2 ? fy : v;
                    f[k] = v;
                }
            }
            self_prev2 = self_prev1; self_prev1 = self_new;
            stale--;
            fence_proxy_async_smem();   // make the generic-proxy smem writes visible to the async proxy
            __syncthreads();
            if (tid == 0) {
                // rows are 4732 B (= 12 mod 16): a ragged tail is rounded up to 16 B; the <= 12 spill bytes land
                // in the next, unused row of the same [cap] block (cap is a multiple of 4, see engine.cu)
                const uint32_t bytes = ((uint32_t)cn * kRowBytes + 15u) & ~15u;     // (bf16 rows are 16-byte multiples)
                bulk_store_s2g((unsigned char *)vout + (size_t)c0 * kRowBytes, buf ? s_stage1 : s_stage0, bytes);
                bulk_commit();
            }
        }
        if (tid == 0) s_next = next_ticket;
    }
    if (tid == 0) {
        bulk_wait<0>();
        if (atomicAdd(&S.obs_ticket[1], 1) == (int)gridDim.x - 1) { S.obs_ticket[0] = 0; S.obs_ticket[1] = 0; }
    }
}

// ----------------------------------------------------------------------------------------------
// K5: group mean action, standalone (senario_battle.py:141,255): out[e][g][b] = #{i : act_i = b} / n
// One warp per (env, group); 21 ballots per 32 agents, lane b owns bin b.
// ----------------------------------------------------------------------------------------------
__global__ void k_mean_action(const int32_t *__restrict__ actions, const int32_t *__restrict__ num,
                              float *__restrict__ out, int n_rows, int cap, int n_action) {
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (row >= n_rows) return;
    const int n = num[row];
    const int32_t *a = actions + (size_t)row * cap;
    int cnt = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const int v = i < n ? a[i] : -1;
        for (int b = 0; b < n_action; b++) {
            const int c = __popc(__ballot_sync(0xFFFFFFFFu, v == b));
            if (lane == b) cnt += c;
        }
    }
    if (lane < n_action) out[(size_t)row * n_action + lane] = n > 0 ? __fdiv_rn((float)cnt, (float)n) : 0.0f;
}

// ----------------------------------------------------------------------------------------------
// K7: neighbourhood mean action.  Observer i of (env e, group g) gets
//   out[b] = #{j != i same group : alive_j, last_action_j = b < n_action, pos_j - pos_i in the disc} / (that count)
// (0 when nobody counts), the disc being CircleRange(radius, 0, 1) (Range.h:171-215) with radius <= view_radius, so it
// fits the kPad margin.  Rows >= num are zero.  Reads the engine state only.
//
// One CTA per (env, tile of observers, group).  The CTA builds a padded u8 grid of its group in shared memory (a cell
// holds last_action + 1 of the alive agent that stands there and has acted, else 0); each thread then walks the disc
// of one observer (no bounds tests), 8 probes in flight at a time, and counts the hits into its own column of a
// [bin][thread] histogram (lanes never share a bank) with shared atomics whose result nobody waits for.  The centre is
// skipped: a live observer stands there itself, while a listed dead one may have been stepped on, and then the agent
// on its cell counts.  The histogram region is then reused for the rows, staged [thread][bin], and stored as one
// contiguous block: cap and the tile are multiples of 4, so every tile is a whole number of 16-byte vectors.
// ----------------------------------------------------------------------------------------------
constexpr int kLocalBins = 32;   // n_action <= 32 (Engine checks move + attack <= 32)
struct LocalMeanSmem { int grid, hist, total; };
__host__ __device__ inline LocalMeanSmem local_mean_smem_layout(int W, int H, int tile, int n_action, bool grid = true) {
    LocalMeanSmem L; int o = 0;
    L.grid = o;  if (grid) o += ((W + 2 * kPad) * (H + 2 * kPad) + 15) & ~15;
    L.hist = o;  o += 4 * n_action * tile;   // u32 [bin][thread], then f32 [thread][bin] rows
    L.total = o;
    return L;
}

//
// REC_HBM (maps whose u8 grid does not fit beside the histogram): no grid is built.  The observation record's padded
// grid already holds every alive listed agent as kind << 14 | slot (kind 2 + group); a probe counts a cell when the
// kind is the observer's group and the agent there has acted, its last action read from the state arrays.
template <bool REC_HBM>
__global__ void __launch_bounds__(kLocalMaxTile) k_local_mean_action(const __grid_constant__ LocalMeanIO io, const BattleState S) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const LocalMeanSmem L = local_mean_smem_layout(io.W, io.H, io.tile, io.n_action, !REC_HBM);
    uint8_t *s_grid = smem_raw + L.grid;
    uint32_t *s_hist = (uint32_t *)(smem_raw + L.hist);
    float *s_stage = (float *)(smem_raw + L.hist);
    const int tid = threadIdx.x, nt = blockDim.x;
    const int e = blockIdx.x, first = blockIdx.y * nt, g = io.group[blockIdx.z];
    const int cap = io.cap, n_action = io.n_action, PW = io.W + 2 * kPad;
    const size_t base = ((size_t)e * kGroups + g) * cap;
    const int n = S.num[e * kGroups + g];

    if constexpr (!REC_HBM)
        for (int c = tid; c < (L.hist - L.grid) / 16; c += nt) ((uint4 *)s_grid)[c] = make_uint4(0u, 0u, 0u, 0u);
    for (int b = 0; b < n_action; b++) s_hist[b * nt + tid] = 0u;
    if constexpr (!REC_HBM) {
        __syncthreads();
        for (int s = tid; s < n; s += nt) {
            const uint32_t st = S.state[base + s], a = st_act(st);
            if (!st_dead(st) && a < (uint32_t)n_action) {
                const int p = S.pos[base + s];
                s_grid[(pos_y(p) + kPad) * PW + pos_x(p) + kPad] = (uint8_t)(a + 1);
            }
        }
    }
    __syncthreads();

    const int i = first + tid;
    uint32_t *h = s_hist + tid;                           // h[b * nt] = bin b of this thread
    if (i < n) {
        const int p = S.pos[base + i];
        if constexpr (REC_HBM) {
            const ObsRecord R = obs_record_layout(io.W, io.H, cap);
            const uint16_t *c = (const uint16_t *)(S.obs_record + (size_t)e * R.total) + (pos_y(p) + kPad) * PW + pos_x(p) + kPad;
            const uint32_t kind = 2u + (uint32_t)g;
            const uint32_t *st_env = S.state + (size_t)e * kGroups * cap;   // record slots index [2][cap]
            auto bin = [&](uint32_t code) -> uint32_t {   // last action + 1 of a same-group agent that acted, else 0
                if ((code >> 14) != kind) return 0u;
                const uint32_t a = st_act(st_env[code & 0x3FFFu]);
                return a < (uint32_t)n_action ? a + 1 : 0u;
            };
            for (int k = 0; k < io.n_offsets; k += 8) {
                uint32_t v[8];
#pragma unroll
                for (int u = 0; u < 8; u++) v[u] = k + u < io.n_offsets ? __ldg(c + io.delta[k + u]) : 0u;
#pragma unroll
                for (int u = 0; u < 8; u++) v[u] = bin(v[u]);
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (v[u]) atomicAdd(h + (v[u] - 1) * nt, 1u);
            }
            if (st_dead(S.state[base + i])) {
                const uint32_t v = bin(__ldg(c));
                if (v) atomicAdd(h + (v - 1) * nt, 1u);
            }
        } else {
        const uint8_t *c = s_grid + (pos_y(p) + kPad) * PW + pos_x(p) + kPad;
        for (int k = 0; k < io.n_offsets; k += 8) {
            uint32_t v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = k + u < io.n_offsets ? c[io.delta[k + u]] : 0u;
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (v[u]) atomicAdd(h + (v[u] - 1) * nt, 1u);
        }
        if (st_dead(S.state[base + i])) {
            const uint32_t v = c[0];
            if (v) atomicAdd(h + (v - 1) * nt, 1u);
        }
        }
    }
    uint32_t cnt[kLocalBins], total = 0;
#pragma unroll
    for (int b = 0; b < kLocalBins; b++) {
        cnt[b] = b < n_action ? h[b * nt] : 0u;
        total += cnt[b];
    }
    __syncthreads();                                      // every column is read: the region now takes the rows
    float *row = s_stage + tid * n_action;                // (rows of threads past num are zeros: their counts are)
#pragma unroll
    for (int b = 0; b < kLocalBins; b++)
        if (b < n_action) row[b] = cnt[b] ? __fdiv_rn((float)cnt[b], (float)total) : 0.0f;
    __syncthreads();
    const int rows = min(nt, cap - first);
    float4 *dst = (float4 *)(io.out[g] + ((size_t)e * cap + first) * n_action);
    for (int v = tid; v < rows * n_action / 4; v += nt) dst[v] = ((const float4 *)s_stage)[v];
}

// ----------------------------------------------------------------------------------------------
// episode (re)initialisation: every env gets the placement template, then the random ops
// ----------------------------------------------------------------------------------------------
__global__ void k_place(const __grid_constant__ BattleParams P, const BattleState S, const RandomPlacement RP) {
    const int e = blockIdx.x;
    place_from_template(P, S, e, 0);
    if (threadIdx.x == 0) S.episode[e] = 0;
    if (RP.n_ops) {
        __syncthreads();
        place_random(P, S, RP, e, 0, 0, RP.occ + (size_t)e * ((P.W * P.H + 31) >> 5));
    } else if (threadIdx.x == 0) {
        RP.place_short[e] = 0;
    }
}

}  // namespace mfmarl
