// Save, restore and fork environments: the per-env state record of mfmarl_batched.h (mfb_save_envs / mfb_load_envs).
//
//   k_state_check  validates records before anything is written (one CTA per record)
//   k_save_envs    gathers listed envs into records                (one CTA per record)
//   k_load_envs    scatters validated records into listed envs     (one CTA per record)
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
