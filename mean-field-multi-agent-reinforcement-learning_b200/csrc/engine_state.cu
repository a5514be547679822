// Save, restore and fork environments: the per-env state record of mfmarl_batched.h (mfb_save_envs / mfb_load_envs).
//
//   k_state_check  validates records before anything is written (one CTA per record)
//   k_save_envs    gathers listed envs into records                (one CTA per record)
//   k_load_envs    scatters validated records into listed envs     (one CTA per record)
//   k_render_obs   observation rows of (record, group, slot) triples (one warp per row; mfb_render_observations)
//
// Record of R = 96 + 64 * cap bytes (the layout is documented in include/mfmarl_batched.h):
//   words 0..23   header and per-env scalars (StateWord below)
//   byte  96      8 slices of [2][cap] 32-bit words: pos, hp, id, state, next_rew, last_rew, template pos, template id
// cap is a multiple of 4, so every slice starts 16-byte aligned and is copied with 16-byte vectors.
#include <climits>
#include <string>
#include <vector>

#include "engine.h"

namespace mfmarl {

namespace {
constexpr uint32_t kStateMagic = 0x5342464Du;   // "MFBS"
constexpr uint32_t kStateVersion = 1;
constexpr int kStateHead = 96;
constexpr int kStateSlices = 8;
constexpr int kStateThreads = 256;
enum StateWord {
    W_MAGIC, W_VERSION, W_W, W_H, W_CAP, W_NACT, W_EMB, W_RSVD, W_HASH_LO, W_HASH_HI,
    W_NUM, W_DEAD = W_NUM + 2, W_RNG = W_DEAD + 2, W_STEP, W_IDC, W_SIDE, W_EPISODE, W_INIT_NUM,
    W_WORDS = kStateHead / 4
};
// k_state_check's verdict per record: int32[8]
enum { V_CODE, V_A, V_B, V_TMPL_DIFFERS, V_NUM0, V_NUM1, V_WORDS = 8 };
enum CheckCode {
    C_OK, C_MAGIC, C_MAP, C_CAP, C_NACT, C_WALLS, C_NUM, C_DEAD, C_INIT_NUM, C_POS, C_ACTION, C_TPOS
};

__host__ __device__ inline size_t state_record_bytes(int cap) { return kStateHead + (size_t)kStateSlices * 2 * cap * 4; }

// the [2][cap] slice j of env e in the engine: 0..5 agent records, 6..7 the env's placement template
__device__ __forceinline__ int32_t *engine_slice(const BattleParams &P, const BattleState &S, int e, int j) {
    const size_t ebase = (size_t)e * 2 * P.cap;
    switch (j) {
        case 0: return S.pos + ebase;
        case 1: return (int32_t *)S.hp + ebase;
        case 2: return S.id + ebase;
        case 3: return (int32_t *)S.state + ebase;
        case 4: return (int32_t *)S.next_rew + ebase;
        case 5: return (int32_t *)S.last_rew + ebase;
        default: return S.init_pos + (size_t)e * P.tmpl_stride + (size_t)(j - 6) * 2 * P.cap;
    }
}

__device__ __forceinline__ bool on_map(const BattleParams &P, uint32_t p) {
    return (p & 0xFFFFu) < (uint32_t)P.W && (p >> 16) < (uint32_t)P.H;
}
}  // namespace

__global__ void __launch_bounds__(kStateThreads)
k_state_check(const __grid_constant__ BattleParams P, const BattleState S, const unsigned char *__restrict__ in,
              unsigned long long wall_hash, int n_action, int32_t *__restrict__ verdict) {
    __shared__ uint32_t s_h[W_WORDS];
    __shared__ int s_code, s_a, s_b, s_bad, s_differs;
    const int k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, cap = P.cap;
    const unsigned char *rec = in + (size_t)k * state_record_bytes(cap);
    if (tid < W_WORDS) s_h[tid] = ((const uint32_t *)rec)[tid];
    __syncthreads();
    if (tid == 0) {
        int code = C_OK, a = 0, b = 0;
        const int32_t *h = (const int32_t *)s_h;
        const unsigned long long hash = (unsigned long long)s_h[W_HASH_HI] << 32 | s_h[W_HASH_LO];
        auto in_cap = [&](int off, int c) {
            for (int g = 0; g < kGroups && code == C_OK; g++)
                if (h[off + g] < 0 || h[off + g] > cap) { code = c; a = g; b = h[off + g]; }
        };
        if (s_h[W_MAGIC] != kStateMagic || s_h[W_VERSION] != kStateVersion) { code = C_MAGIC; a = (int)s_h[W_MAGIC]; b = (int)s_h[W_VERSION]; }
        else if (h[W_W] != P.W || h[W_H] != P.H) { code = C_MAP; a = h[W_W]; b = h[W_H]; }
        else if (h[W_CAP] != cap) { code = C_CAP; a = h[W_CAP]; }
        else if (h[W_NACT] != n_action) { code = C_NACT; a = h[W_NACT]; }
        else if (hash != wall_hash) code = C_WALLS;
        else {
            in_cap(W_NUM, C_NUM);
            in_cap(W_DEAD, C_DEAD);
            in_cap(W_INIT_NUM, C_INIT_NUM);
        }
        s_code = code; s_a = a; s_b = b; s_bad = INT_MAX;
        // the engine's shared template against the record's (raw words, so that save -> load -> save is exact)
        s_differs = P.tmpl_stride == 0 && (h[W_INIT_NUM] != S.init_num[0] || h[W_INIT_NUM + 1] != S.init_num[1]);
    }
    __syncthreads();
    if (s_code == C_OK) {
        const int32_t *h = (const int32_t *)s_h;
        const int per = cap / 2;                                   // 16-byte vectors per [2][cap] slice
        const uint4 *slices = (const uint4 *)(rec + kStateHead);
        for (int v = tid; v < per; v += nt) {
            const int s = 4 * v, g = s >= cap, i = s - g * cap;   // (a vector never straddles the groups: cap % 4 == 0)
            const uint4 pos = slices[v], st = slices[3 * per + v], tpos = slices[6 * per + v];
            const uint32_t p[4] = {pos.x, pos.y, pos.z, pos.w}, a[4] = {st.x, st.y, st.z, st.w},
                           t[4] = {tpos.x, tpos.y, tpos.z, tpos.w};
            int bad = INT_MAX;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                if (i + q < h[W_NUM + g] && !on_map(P, p[q])) bad = min(bad, C_POS << 16 | (s + q));
                if (i + q < h[W_NUM + g] && ((a[q] >> 16) & 0xFFu) > (uint32_t)n_action) bad = min(bad, C_ACTION << 16 | (s + q));
                if (i + q < h[W_INIT_NUM + g] && !on_map(P, t[q])) bad = min(bad, C_TPOS << 16 | (s + q));
            }
            if (bad != INT_MAX) atomicMin(&s_bad, bad);
        }
        if (P.tmpl_stride == 0) {
            const uint4 *mine = (const uint4 *)S.init_pos;
            bool differs = false;
            for (int v = tid; v < 2 * per; v += nt) {
                const uint4 x = slices[6 * per + v], y = mine[v];
                differs |= x.x != y.x || x.y != y.y || x.z != y.z || x.w != y.w;
            }
            if (differs) s_differs = 1;
        }
        __syncthreads();
        if (tid == 0 && s_bad != INT_MAX) {
            const int slot = s_bad & 0xFFFF;
            s_code = s_bad >> 16; s_a = slot >= cap; s_b = slot - s_a * cap;
        }
    }
    if (tid == 0) {
        int32_t *out = verdict + (size_t)k * V_WORDS;
        out[V_CODE] = s_code; out[V_A] = s_a; out[V_B] = s_b; out[V_TMPL_DIFFERS] = s_differs;
        out[V_NUM0] = (int32_t)s_h[W_NUM]; out[V_NUM1] = (int32_t)s_h[W_NUM + 1];
    }
}

__global__ void __launch_bounds__(kStateThreads)
k_save_envs(const __grid_constant__ BattleParams P, const BattleState S, const int32_t *__restrict__ envs,
            unsigned char *__restrict__ out, unsigned long long wall_hash, int n_action) {
    const int k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, cap = P.cap;
    const int e = envs ? envs[k] : k;
    unsigned char *rec = out + (size_t)k * state_record_bytes(cap);
    if (tid < W_WORDS) {
        const int32_t *tnum = S.init_num + (P.tmpl_stride ? 2 * e : 0);
        uint32_t w = 0;
        switch (tid) {
            case W_MAGIC: w = kStateMagic; break;
            case W_VERSION: w = kStateVersion; break;
            case W_W: w = P.W; break;
            case W_H: w = P.H; break;
            case W_CAP: w = cap; break;
            case W_NACT: w = n_action; break;
            case W_EMB: w = P.embedding_size; break;
            case W_HASH_LO: w = (uint32_t)wall_hash; break;
            case W_HASH_HI: w = (uint32_t)(wall_hash >> 32); break;
            case W_NUM: case W_NUM + 1: w = S.num[2 * e + tid - W_NUM]; break;
            case W_DEAD: case W_DEAD + 1: w = S.dead_ct[2 * e + tid - W_DEAD]; break;
            case W_RNG: w = S.rng[e]; break;
            case W_STEP: w = S.step_ct[e]; break;
            case W_IDC: w = S.id_counter[e]; break;
            case W_SIDE: w = S.side[e]; break;
            case W_EPISODE: w = S.episode[e]; break;
            case W_INIT_NUM: case W_INIT_NUM + 1: w = tnum[tid - W_INIT_NUM]; break;
            default: break;
        }
        ((uint32_t *)rec)[tid] = w;
    }
    const int per = cap / 2;
    uint4 *dst = (uint4 *)(rec + kStateHead);
#pragma unroll
    for (int j = 0; j < kStateSlices; j++) {
        const uint4 *src = (const uint4 *)engine_slice(P, S, e, j);
        for (int v = tid; v < per; v += nt) dst[j * per + v] = src[v];
    }
}

// records validated by k_state_check; the templates are written only where the engine keeps one per env
__global__ void __launch_bounds__(kStateThreads)
k_load_envs(const __grid_constant__ BattleParams P, const BattleState S, const int32_t *__restrict__ envs,
            const unsigned char *__restrict__ in) {
    const int k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, cap = P.cap;
    const int e = envs ? envs[k] : k;
    const unsigned char *rec = in + (size_t)k * state_record_bytes(cap);
    const int32_t *h = (const int32_t *)rec;
    if (tid < 2) {
        S.num[2 * e + tid] = h[W_NUM + tid];
        S.dead_ct[2 * e + tid] = h[W_DEAD + tid];
        if (P.tmpl_stride) S.init_num[2 * e + tid] = h[W_INIT_NUM + tid];
    }
    if (tid == 0) {
        S.rng[e] = (uint32_t)h[W_RNG]; S.step_ct[e] = h[W_STEP]; S.id_counter[e] = h[W_IDC];
        S.side[e] = h[W_SIDE]; S.episode[e] = h[W_EPISODE];
    }
    const int per = cap / 2;
    const uint4 *src = (const uint4 *)(rec + kStateHead);
    const int slices = P.tmpl_stride ? kStateSlices : kStateSlices - 2;
    for (int j = 0; j < slices; j++) {
        uint4 *dst = (uint4 *)engine_slice(P, S, e, j);
        for (int v = tid; v < per; v += nt) dst[v] = src[j * per + v];
    }
}

// ---- k_render_obs: observation rows rendered again from state records (mfb_render_observations) ----
// One warp per output row.  A sampled batch almost never has two rows of one record, so nothing is built per record:
// the warp scans its record's <= 2 * cap listed agents once, counting the minimaps and drawing the alive ones that fall
// in its 13 x 13 window into per-warp shared memory, composes the row there one cell per lane, and drains it with
// 16-byte stores (rows are 4732 B, so row k starts 12 k mod 16 bytes past a 16-byte boundary: a 0-3 float head and
// tail go out as scalars -- nothing is written past row k, since a gather output has no padding behind its last row).
// The formulas are k_obs's (battle_kernels.cuh): walls from the engine's padded grid_template, hp / max_hp with
// __fdiv_rn, count / num with 0 / 0 = 0, the "+1" self marker in both minimap channels, the features of
// GridWorld.cc:411-421.
constexpr int kRenderWarps = 4, kRenderThreads = 32 * kRenderWarps;
constexpr int kRenderStage = kViewRow + 5;   // floats of a warp's staged row: up to 3 of alignment shift, 16-byte multiple
constexpr int kRenderPad = kView / 2;   // the 6-cell empty margin of grid_template

__global__ void __launch_bounds__(kRenderThreads)
k_render_obs(const __grid_constant__ BattleParams P, const uint16_t *__restrict__ grid_template,
             const uint8_t *__restrict__ mini_lut, const unsigned char *__restrict__ records, int n_records,
             const int32_t *__restrict__ rows, int n_rows, float *__restrict__ view, float *__restrict__ feature,
             int32_t *__restrict__ bad_rows, unsigned long long wall_hash) {
    __shared__ __align__(16) float s_row[kRenderWarps][kRenderStage];   // the row, shifted to row k's 16-byte phase
    __shared__ int s_cnt[kRenderWarps][2 * kViewCells];     // minimap counts, then (in place) count / num as floats
    __shared__ uint8_t s_kind[kRenderWarps][kViewCells + 7];   // window cell: 0 empty, 1 wall, 2 + group of an alive agent
    __shared__ float s_hp[kRenderWarps][kViewCells];         // hp / max_hp of that agent
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const size_t k = (size_t)blockIdx.x * kRenderWarps + w;
    if (k >= (size_t)n_rows) return;                         // (warp-uniform)
    const int cap = P.cap, W = P.W, H = P.H, FS = P.feature_size, emb = P.embedding_size;
    const int n_action = P.n_move + P.n_attack;
    float *const vrow = view + k * kViewRow;
    float *const frow = feature + k * FS;
    const int r = rows[3 * k], g = rows[3 * k + 1], slot = rows[3 * k + 2];

    bool ok = (unsigned)r < (unsigned)n_records && (unsigned)g < (unsigned)kGroups && (unsigned)slot < (unsigned)cap;
    const unsigned char *rec = records + (ok ? (size_t)r * state_record_bytes(cap) : 0);
    int n0 = 0, n1 = 0;                                      // (scalars: a dynamically indexed array would go to local memory)
    if (ok) {
        const uint32_t *h = (const uint32_t *)rec;
        const unsigned long long hash = (unsigned long long)h[W_HASH_HI] << 32 | h[W_HASH_LO];
        ok = h[W_MAGIC] == kStateMagic && h[W_VERSION] == kStateVersion && (int)h[W_W] == W && (int)h[W_H] == H &&
             (int)h[W_CAP] == cap && (int)h[W_NACT] == n_action && hash == wall_hash;
        n0 = min(max((int)h[W_NUM], 0), cap);
        n1 = min(max((int)h[W_NUM + 1], 0), cap);
    }
    const int32_t *pos = (const int32_t *)(rec + kStateHead);   // slices [2][cap]: 0 pos, 1 hp, 2 id, 3 state, 5 last_rew
    const float *hp = (const float *)(pos + 2 * cap);
    const int32_t *id = pos + 4 * cap;
    const uint32_t *state = (const uint32_t *)(pos + 6 * cap);
    const float *last_rew = (const float *)(pos + 10 * cap);
    const int s_self = g * cap + slot;
    ok = ok && slot < (g ? n1 : n0);
    const uint32_t p_self = ok ? (uint32_t)pos[s_self] : 0u;
    ok = ok && on_map(P, p_self);
    if (!ok) {
        for (int i = lane; i < kViewRow; i += 32) vrow[i] = 0.0f;
        for (int i = lane; i < FS; i += 32) frow[i] = 0.0f;
        if (lane == 0 && bad_rows) atomicAdd(bad_rows, 1);
        return;
    }
    const int ax = (int)(p_self & 0xFFFFu), ay = (int)(p_self >> 16), PW = W + 2 * kRenderPad;
    int *const cnt = s_cnt[w];
    uint8_t *const kind = s_kind[w];
    float *const hpc = s_hp[w];
    for (int c = lane; c < kViewCells; c += 32) {
        const int vy = c / kView, vx = c - vy * kView;
        kind[c] = (uint8_t)(grid_template[(size_t)(ay + vy) * PW + ax + vx] >> 14);   // window corner (ax - 6, ay - 6)
    }
    for (int c = lane; c < 2 * kViewCells; c += 32) cnt[c] = 0;
    __syncwarp();
    for (int gg = 0; gg < kGroups; gg++) {
        for (int i = lane; i < (gg ? n1 : n0); i += 32) {
            const int s = gg * cap + i;
            const uint32_t q = (uint32_t)pos[s];
            if (!on_map(P, q)) continue;                          // (only a record from outside: neither drawn nor counted)
            const int x = (int)(q & 0xFFFFu), y = (int)(q >> 16);
            atomicAdd(&cnt[gg * kViewCells + mini_lut[W + y] + mini_lut[x]], 1);   // dead or not (GridWorld.cc:359-370)
            const int dx = x - ax + kRenderPad, dy = y - ay + kRenderPad;
            if ((unsigned)dx < (unsigned)kView && (unsigned)dy < (unsigned)kView && !(state[s] & 1u)) {
                kind[dy * kView + dx] = (uint8_t)(2 + gg);
                hpc[dy * kView + dx] = __fdiv_rn(hp[s], P.hp);   // Map.cc:208
            }
        }
    }
    __syncwarp();
    float *const mini = (float *)cnt;
    for (int c = lane; c < 2 * kViewCells; c += 32) {
        const int tot = c >= kViewCells ? n1 : n0;
        mini[c] = tot > 0 ? __fdiv_rn((float)cnt[c], (float)tot) : 0.0f;   // GridWorld.cc:372-377; 0/0 defined as 0
    }
    __syncwarp();
    const float *mini_own = mini + g * kViewCells, *mini_oth = mini + (1 - g) * kViewCells;
    const uint32_t kind_own = 2u + (uint32_t)g, kind_oth = 3u - (uint32_t)g;
    const int self_c = mini_lut[W + ay] + mini_lut[ax];
    // row float j sits at s_row[w][shift + j]: shift + j is a multiple of 4 exactly where vrow + j is 16-byte aligned
    const int head = (int)((4 - (k * 3) % 4) % 4);            // floats before row k's first 16-byte boundary
    const int shift = (4 - head) % 4;
    float *const row = s_row[w] + shift;
    for (int c = lane; c < kViewCells; c += 32) {              // one cell per lane: stride-7 words, no bank conflicts
        const uint32_t kd = (P.disc[c >> 5] >> (c & 31)) & 1u ? kind[c] : 0u;   // occupancy only inside the view disc
        const float h = hpc[c], self = c == self_c ? 1.0f : 0.0f;
        float *o = row + c * kChan;
        o[0] = kd == 1u ? 1.0f : 0.0f;
        o[1] = kd == kind_own ? 1.0f : 0.0f;
        o[2] = kd == kind_own ? h : 0.0f;
        o[3] = self != 0.0f ? mini_own[c] + self : mini_own[c];   // self marker in both minimaps (GridWorld.cc:396-408)
        o[4] = kd == kind_oth ? 1.0f : 0.0f;
        o[5] = kd == kind_oth ? h : 0.0f;
        o[6] = self != 0.0f ? mini_oth[c] + self : mini_oth[c];
    }
    __syncwarp();
    if (lane < head) vrow[lane] = row[lane];
    const int n4 = (kViewRow - head) >> 2;
    const float4 *src4 = (const float4 *)(row + head);
    float4 *dst4 = (float4 *)(vrow + head);
    for (int q = lane; q < n4; q += 32) dst4[q] = src4[q];
    const int tail = head + 4 * n4;
    if (lane < kViewRow - tail) vrow[tail + lane] = row[tail + lane];
    // features (GridWorld.cc:411-421): id bits LSB first, one-hot last action, last reward, x / W, y / H
    const int my_id = id[s_self], act = (int)((state[s_self] >> 16) & 0xFFu);
    const float rew = last_rew[s_self];
    for (int j = lane; j < FS; j += 32) {
        float v = (j < emb) ? (float)((my_id >> j) & 1) : ((j - emb == act) ? 1.0f : 0.0f);
        v = j == emb + n_action ? rew : v;
        v = j == emb + n_action + 1 ? __fdiv_rn((float)ax, (float)W) : v;
        v = j == emb + n_action + 2 ? __fdiv_rn((float)ay, (float)H) : v;
        frow[j] = v;
    }
}

namespace {
const char *check_reason(int code) {
    switch (code) {
        case C_MAGIC: return "not a battle state record of this format version";
        case C_MAP: return "map size differs from the engine's";
        case C_CAP: return "capacity differs from the engine's";
        case C_NACT: return "action count differs from the engine's";
        case C_WALLS: return "wall map differs from the engine's (FNV-1a hash)";
        case C_NUM: return "num outside [0, cap]";
        case C_DEAD: return "dead_ct outside [0, cap]";
        case C_INIT_NUM: return "template num outside [0, cap]";
        case C_POS: return "agent position off the map";
        case C_ACTION: return "last action above n_action";
        case C_TPOS: return "template position off the map";
        default: return "invalid record";
    }
}
}  // namespace

size_t Engine::state_bytes() const { return state_record_bytes(P_.cap); }

// Host-side checks of a save / load request, then the index list goes to the device (null for "all envs in order").
// The scratch holds [n] indices, then [n][V_WORDS] verdicts.  A save of every env does not use it.  Where it is used,
// its writes are ordered on `st` after the last launch that read it (on whatever stream): the host does not wait.
const int32_t *Engine::upload_targets(int n, const int32_t *envs, const void *buf, bool load, cudaStream_t st) {
    if (!buf) throw Fatal(std::string("null ") + (load ? "input" : "output") + " buffer");
    if ((uintptr_t)buf & 15) throw Fatal("record buffer must be 16-byte aligned");
    if (n < 1 || (load && n > P_.E))
        throw Fatal("n = " + std::to_string(n) + (load ? " outside [1, n_envs = " + std::to_string(P_.E) + "]" : std::string(" < 1")));
    if (!envs && n != P_.E) throw Fatal(std::string("envs = NULL means every env: n must be n_envs = ") + std::to_string(P_.E));
    if (envs) {
        std::vector<char> seen(load ? (size_t)P_.E : 0, 0);
        for (int k = 0; k < n; k++) {
            if (envs[k] < 0 || envs[k] >= P_.E)
                throw Fatal("env index " + std::to_string(envs[k]) + " at " + std::to_string(k) + " out of range [0, " + std::to_string(P_.E) + ")");
            if (load && seen[(size_t)envs[k]]++) throw Fatal("env " + std::to_string(envs[k]) + " is a load target twice");
        }
    }
    if (!envs && !load) return nullptr;
    const size_t need = (size_t)n * (1 + V_WORDS);
    if (!state_io_done_) MF_CUDA(cudaEventCreateWithFlags(&state_io_done_, cudaEventDisableTiming));
    if (need > state_io_words_) {
        MF_CUDA(cudaFree(d_state_io_));   // (cudaFree waits for the device: no launch still reads the old scratch)
        d_state_io_ = nullptr;
        MF_CUDA(cudaMalloc(&d_state_io_, need * 4));
        state_io_words_ = need;
    }
    MF_CUDA(cudaStreamWaitEvent(st, state_io_done_, 0));
    if (!envs) return nullptr;
    MF_CUDA(cudaMemcpyAsync(d_state_io_, envs, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    return d_state_io_;
}

void Engine::save_envs(int n, const int32_t *envs, void *d_out, cudaStream_t st) {
    commit(st);
    const int32_t *d_envs = upload_targets(n, envs, d_out, false, st);
    k_save_envs<<<n, kStateThreads, 0, st>>>(P_, S_, d_envs, (unsigned char *)d_out, wall_hash_, n_action());
    MF_CUDA(cudaGetLastError());
    if (d_envs) MF_CUDA(cudaEventRecord(state_io_done_, st));
}

void Engine::render_observations(int n_records, const void *d_records, int n_rows, const int32_t *d_rows, float *d_view,
                                 float *d_feature, int32_t *d_bad_rows, cudaStream_t st) {
    if (n_rows < 0) throw Fatal("n_rows = " + std::to_string(n_rows) + " < 0");
    if (n_rows > 0 && n_records < 1) throw Fatal("n_records = " + std::to_string(n_records) + " < 1 with rows to render");
    const std::pair<const void *, const char *> bufs[] = {{d_records, "records"}, {d_rows, "rows"}, {d_view, "view"},
                                                          {d_feature, "feature"}};
    for (const auto &b : bufs) {
        if (!b.first) throw Fatal(std::string("null ") + b.second + " buffer");
        if ((uintptr_t)b.first & 15) throw Fatal(std::string(b.second) + " buffer must be 16-byte aligned");
    }
    if ((uintptr_t)d_bad_rows & 3) throw Fatal("bad_rows counter must be 4-byte aligned");
    commit(st);
    if (d_bad_rows) MF_CUDA(cudaMemsetAsync(d_bad_rows, 0, 4, st));
    if (n_rows == 0) return;
    const unsigned blocks = (unsigned)(((size_t)n_rows + kRenderWarps - 1) / kRenderWarps);
    k_render_obs<<<blocks, kRenderThreads, 0, st>>>(P_, S_.grid_template, S_.mini_lut, (const unsigned char *)d_records,
                                                     n_records, d_rows, n_rows, d_view, d_feature, d_bad_rows, wall_hash_);
    MF_CUDA(cudaGetLastError());
}

void Engine::load_envs(int n, const int32_t *envs, const void *d_in, cudaStream_t st) {
    commit(st);
    const int32_t *d_envs = upload_targets(n, envs, d_in, true, st);
    int32_t *d_verdict = d_state_io_ + n;
    k_state_check<<<n, kStateThreads, 0, st>>>(P_, S_, (const unsigned char *)d_in, wall_hash_, n_action(), d_verdict);
    MF_CUDA(cudaGetLastError());
    std::vector<int32_t> verdict((size_t)n * V_WORDS);
    MF_CUDA(cudaMemcpyAsync(verdict.data(), d_verdict, verdict.size() * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(cudaStreamSynchronize(st));   // the one synchronisation of a load
    bool differs = false;
    for (int k = 0; k < n; k++) {
        const int32_t *v = &verdict[(size_t)k * V_WORDS];
        if (v[V_CODE] == C_OK) { differs |= v[V_TMPL_DIFFERS] != 0; continue; }
        std::string msg = "record " + std::to_string(k) + ": " + check_reason(v[V_CODE]);
        switch (v[V_CODE]) {
            case C_MAP: msg += " (record " + std::to_string(v[V_A]) + "x" + std::to_string(v[V_B]) + ", engine " + std::to_string(P_.W) + "x" + std::to_string(P_.H) + ")"; break;
            case C_CAP: msg += " (record " + std::to_string(v[V_A]) + ", engine " + std::to_string(P_.cap) + "): create the engine with the record's capacity"; break;
            case C_NACT: msg += " (record " + std::to_string(v[V_A]) + ", engine " + std::to_string(n_action()) + ")"; break;
            case C_NUM: case C_DEAD: case C_INIT_NUM: msg += " (group " + std::to_string(v[V_A]) + ": " + std::to_string(v[V_B]) + ", cap " + std::to_string(P_.cap) + ")"; break;
            case C_POS: case C_ACTION: case C_TPOS: msg += " (group " + std::to_string(v[V_A]) + ", slot " + std::to_string(v[V_B]) + ")"; break;
            default: break;
        }
        throw Fatal(msg);
    }
    if (differs) {   // auto-reset must re-place each loaded env from its own template: one template per env from now on
        const size_t T = (size_t)4 * P_.cap, E = (size_t)P_.E;
        for (size_t have = 1; have < E; have *= 2) {   // replicate the shared template into every env's slot
            const size_t c = std::min(have, E - have);
            MF_CUDA(cudaMemcpyAsync(S_.init_pos + have * T, S_.init_pos, c * T * 4, cudaMemcpyDeviceToDevice, st));
            MF_CUDA(cudaMemcpyAsync(S_.init_num + have * 2, S_.init_num, c * 2 * 4, cudaMemcpyDeviceToDevice, st));
        }
        P_.tmpl_stride = (int)T;
    }
    k_load_envs<<<n, kStateThreads, 0, st>>>(P_, S_, d_envs, (const unsigned char *)d_in);
    MF_CUDA(cudaGetLastError());
    for (int k = 0; k < n; k++) {
        const int e = envs ? envs[k] : k;
        h_num_[(size_t)e * 2] = verdict[(size_t)k * V_WORDS + V_NUM0];
        h_num_[(size_t)e * 2 + 1] = verdict[(size_t)k * V_WORDS + V_NUM1];
    }
    stepped_ = true;
    rebuild_obs_records(st);
    MF_CUDA(cudaEventRecord(state_io_done_, st));
}

}  // namespace mfmarl
