// Host engine: HBM state, placement, kernel launches.  See engine.h.
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>

#include "battle_kernels.cuh"

namespace mfmarl {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_last_error(const std::string &msg) { g_last_error = msg; }
const char *last_error() { return g_last_error.c_str(); }

int report_fatal(const char *where, const std::exception &ex) {
    set_last_error(std::string(where) + ": " + ex.what());
    fprintf(stderr, "[magent/b200] fatal in %s: %s\n", where, ex.what());
    const char *mode = getenv("MAGENT_ERRORS");
    if (mode && strcmp(mode, "return") == 0) return -1;
    // the reference throws std::runtime_error through the C boundary (utility.h:77-81), which
    // terminates a ctypes caller; do the same, loudly
    abort();
}

// ---------------------------------------------------------------------------------------------
// range tables: a disc of the given radius on a square of odd/even width (reference Range.h:171-215)
// ---------------------------------------------------------------------------------------------
CircleRange::CircleRange(float radius, float inner_radius, int parity) {
    const double eps = 1e-8;
    width = 2 * (int)(radius + eps) + parity;
    center = (int)radius;
    if (width % 2 != parity) width++;
    in.assign((size_t)width * width, 0);
    const double delta = parity == 0 ? 0.5 : 0.0;
    for (int i = 0; i < width; i++)
        for (int j = 0; j < width; j++) {
            const double ax = std::fabs(j - center + delta), ay = std::fabs(i - center + delta);
            const double dis = std::sqrt(ax * ax + ay * ay);
            if (dis < radius + eps && dis > inner_radius - eps) {
                in[(size_t)i * width + j] = 1;
                dx.push_back(j - center);
                dy.push_back(i - center);
                count++;
            }
        }
}

void Engine::split_template() {
    if (!h_env_.empty()) return;
    h_env_.resize((size_t)P_.E);
    for (EnvTemplate &t : h_env_) {
        t.occ.assign(h_occ_.begin(), h_occ_.end());
        for (int g = 0; g < kGroups; g++) { t.pos[g] = h_tpos_[g]; t.id[g] = h_tid_[g]; }
        t.id_counter = h_id_counter_;
    }
}

void Engine::refuse_after_random(const char *what) const {
    // a random agent could take a fixed agent's (or wall's) cell, and that agent would be skipped in some episodes only
    if (!h_random_.empty())
        throw Fatal(std::string(what) + " after add_agents_random is not supported (call reset first): the fixed "
                    "placement and the walls come before the random ops");
}

void Engine::add_agents_random(int group, int n, int x0, int y0, int w, int h) {
    const int W = P_.W, H = P_.H;
    if (group < 0 || group >= kGroups) throw Fatal("group = " + std::to_string(group) + " is not 0 or 1");
    if (n < 0) throw Fatal("n = " + std::to_string(n) + " is negative");
    if (stepped_) throw Fatal("add_agents_random after stepping is not supported (call reset first)");
    const std::string rect = "rectangle x0 = " + std::to_string(x0) + ", y0 = " + std::to_string(y0) +
                             ", w = " + std::to_string(w) + ", h = " + std::to_string(h);
    if (w == 0 && h == 0) { x0 = 0; y0 = 0; w = W - 1; h = H - 1; }   // the whole map: Map::get_random_blank's draw
    if (w <= 0 || h <= 0) throw Fatal(rect + ": w and h must both be positive, or both 0 for the whole map");
    if (x0 < 0 || y0 < 0 || x0 > W - w || y0 > H - h)
        throw Fatal(rect + " leaves the " + std::to_string(W) + "x" + std::to_string(H) + " map");
    // cells that can be blank: inside the border ring (walls) and the is_blank_area bound x + 1 < W, y + 1 < H
    const int ix0 = std::max(x0, 1), ix1 = std::min(x0 + w - 1, W - 2), iy0 = std::max(y0, 1), iy1 = std::min(y0 + h - 1, H - 2);
    if (ix0 > ix1 || iy0 > iy1) throw Fatal(rect + " has no interior cell");
    // the earlier ops whose rectangles overlap this one may take up to their n of its cells
    long long taken = 0;
    for (const RandomOp &o : h_random_)
        if (o.x0 < x0 + w && x0 < o.x0 + o.w && o.y0 < y0 + h && y0 < o.y0 + o.h) taken += o.n;
    const size_t T = h_env_.empty() ? 1 : h_env_.size();
    for (size_t e = 0; e < T; e++) {
        long long blank = 0;
        for (int y = iy0; y <= iy1; y++)
            for (int x = ix0; x <= ix1; x++) {
                const size_t c = (size_t)y * W + x;
                blank += (h_env_.empty() ? h_occ_[c] : h_env_[e].occ[c]) == 0;
            }
        if (blank < taken + n)
            throw Fatal("n = " + std::to_string(n) + " does not fit" + (h_env_.empty() ? std::string() : " in env " + std::to_string(e)) +
                        ": the " + rect + " has " + std::to_string(blank) + " blank cells, and earlier random ops whose "
                        "rectangles overlap it place up to " + std::to_string(taken) + " agents");
    }
    RandomOp op{group, n, x0, y0, w, h, 0, 0};
    if (!h_random_.empty()) op.id0 = h_random_.back().id0 + h_random_.back().n;
    h_random_.push_back(op);
    placement_dirty_ = true;
}

void Engine::add_agents_per_env(int group, int n, const int *xs, const int *ys, int *n_added) {
    if (group < 0 || group >= kGroups) throw Fatal("invalid group handle in add_agents_per_env");
    if (stepped_) throw Fatal("add_agents_per_env after stepping is not supported (call reset first)");
    refuse_after_random("add_agents_per_env");
    split_template();
    for (int e = 0; e < P_.E; e++) {   // per env: GridWorld.cc:256-269; Map::add_agent Map.cc:75-97; add_or_error :180-187
        EnvTemplate &t = h_env_[(size_t)e];
        int added = 0;
        for (int i = 0; i < n; i++) {
            const int x = xs[(size_t)e * n + i], y = ys[(size_t)e * n + i];
            if (x < 0 || y < 0 || x + 1 >= P_.W || y + 1 >= P_.H) continue;
            const size_t c = (size_t)y * P_.W + x;
            if (t.occ[c] != 0) continue;
            t.occ[c] = 2;
            t.pos[group].push_back(x | (y << 16));
            t.id[group].push_back(t.id_counter++);
            added++;
        }
        if (n_added) n_added[e] = added;
    }
    placement_dirty_ = true;
}

// E == 1, device state is newer than the template: pull the full records, patch, push back.
struct Engine::LateRecords {
    std::vector<int32_t> pos, id; std::vector<float> hp, nr, lr; std::vector<uint32_t> state;
    int num[2], dead[2];
};


// ---------------------------------------------------------------------------------------------
// construction
// ---------------------------------------------------------------------------------------------
static int round_up(int v, int m) { return (v + m - 1) / m * m; }

// dynamic shared memory a CTA may use; a kernel whose layout for the engine's geometry needs more runs from HBM
constexpr int kSmemLimit = 227 * 1024;
static int local_mean_tile(int cap) { return std::min(kLocalMaxTile, round_up(cap, 32)); }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-function, per-device setting shared by every engine of the
// process: it is only ever RAISED, so that an engine of a small geometry cannot pull it below what a larger engine
// (created earlier, launching later) still needs.
static void raise_dynamic_smem(const void *func, int bytes, int device) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, int> granted;
    std::lock_guard<std::mutex> lock(mu);
    int &cur = granted[std::make_pair(func, device)];
    if (bytes <= cur) return;
    if (bytes > kSmemLimit)
        throw Fatal("geometry needs " + std::to_string(bytes) + " B of shared memory per CTA (limit 232448): map or capacity too large");
    MF_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    // the same L1 / shared-memory split for k_obs and k_step: the two kernels alternate every step (and overlap on two
    // streams), and an SM has to drain before it can change its carve-out
    MF_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    cur = bytes;
}

Engine::Engine(const EngineConfig &cfg) : cfg_(cfg) {
    int ndev = 0;
    cudaError_t err = cudaGetDeviceCount(&ndev);
    if (err != cudaSuccess || ndev == 0)
        throw Fatal(std::string("no CUDA device: the battle engine has no CPU fallback (") +
                    cudaGetErrorString(err) + ")");
    if (cfg.device >= 0) MF_CUDA(cudaSetDevice(cfg.device));
    MF_CUDA(cudaGetDevice(&device_));
    MF_CUDA(cudaDeviceGetAttribute(&n_sm_, cudaDevAttrMultiProcessorCount, device_));

    if (cfg.n_envs < 1 || cfg.width < 3 || cfg.height < 3 || cfg.width > 4096 || cfg.height > 4096)
        throw Fatal("invalid engine config (n_envs / map size)");
    // k_step's mean-action export zeroes and writes its [2][32] histogram with threads 0..63: a one-warp CTA would
    // leave group 1's bins unset; 1024 is the CUDA limit on threads per block
    if (cfg.step_threads > 1024 || (cfg.step_threads > 0 && cfg.step_threads <= 32))
        throw Fatal("step_threads = " + std::to_string(cfg.step_threads) +
                    " unsupported: k_step runs 33 to 1024 threads per CTA (rounded up to a multiple of 32), or <= 0 for auto");

    view_ = CircleRange(cfg.type.view_radius, 0.0f, 1);
    attack_ = CircleRange(cfg.type.attack_radius, 0.5f, 1);   // inner radius = width / 2.0f (AgentType.cc:107)
    move_ = CircleRange(cfg.type.speed, 0.0f, 1);
    if (view_.width != kView)
        throw Fatal("view range " + std::to_string(view_.width) + "x" + std::to_string(view_.width) +
                    " unsupported: the observation kernel is specialised for the 13x13 battle view");
    if (move_.count > kMaxMoves || attack_.count > kMaxAttacks || move_.count + attack_.count > 32)
        throw Fatal("move/attack range too large (at most 32 actions)");

    P_.E = cfg.n_envs; P_.W = cfg.width; P_.H = cfg.height;
    P_.env_base = cfg.env_base;
    P_.embedding_size = cfg.embedding_size;
    P_.n_move = move_.count; P_.n_attack = attack_.count;
    P_.view = kView;
    P_.feature_size = cfg.embedding_size + P_.n_move + P_.n_attack + 1 + 2;   // GridWorld.cc:1010-1018
    P_.scale_w = (cfg.width + kView - 1) / kView;                             // GridWorld.cc:341-342
    P_.scale_h = (cfg.height + kView - 1) / kView;
    P_.wall_stride = 0;
    P_.rng_mode = cfg.rng_mode; P_.max_steps = cfg.max_steps; P_.seed = cfg.seed;
    {   // observation record (battle_kernels.cuh): worth it when groups are large -- the per-item rebuild of the occupancy
        // grid from the agent arrays then dominates k_obs's set-up and forces coarse tiles
        const char *env = getenv("MFMARL_OBS_CACHED");
        const int want = cfg.obs_cached >= 0 ? cfg.obs_cached : (env ? atoi(env) : -1);
        P_.obs_cached = want >= 0 ? (want != 0) : (round_up(cfg.capacity, 4) >= 256);
        obs_cached_off_ = want == 0;
    }
    P_.move_bands = 0; P_.band_width = cfg.width;
    if (cfg.width * cfg.height > 99 * 99) {                       // GridWorld.cc:79-88 "large_map_mode"
        P_.move_bands = cfg.width * cfg.height > 1000 * 1000 ? 16 : 8;
        P_.band_width = (cfg.width + P_.move_bands - 1) / P_.move_bands;   // GridWorld.cc:439
    }
    P_.hp = cfg.type.hp; P_.damage = cfg.type.damage; P_.step_recover = cfg.type.step_recover;
    P_.kill_supply = cfg.type.kill_supply; P_.step_reward = cfg.type.step_reward;
    P_.kill_reward = cfg.type.kill_reward; P_.dead_penalty = cfg.type.dead_penalty;
    P_.attack_penalty = cfg.type.attack_penalty;
    for (int g = 0; g < kGroups; g++) P_.attack_bonus[g] = cfg.attack_bonus[g];
    for (int i = 0; i < move_.count; i++) { P_.move_dx[i] = (int8_t)move_.dx[i]; P_.move_dy[i] = (int8_t)move_.dy[i]; }
    for (int i = 0; i < attack_.count; i++) { P_.att_dx[i] = (int8_t)attack_.dx[i]; P_.att_dy[i] = (int8_t)attack_.dy[i]; }
    memset(P_.disc, 0, sizeof(P_.disc));
    for (int c = 0; c < kViewCells; c++)
        if (view_.in[c]) P_.disc[c >> 5] |= 1u << (c & 31);
    {   // lane schedule of k_obs: only in-disc cells are ever rewritten (the others stay 0 in the staging rows).  A cell's
        // channel-j store goes to bank (7 c + j) mod 32, so two cells of one pass collide iff they agree mod 32:
        // give every cell the first pass in which its residue is still free (falling back to any free slot).
        memset(P_.obs_cell, 255, sizeof(P_.obs_cell));
        const int passes = kObsDiscSlots / 32;
        std::vector<int> left;
        for (int c = 0; c < kViewCells; c++) {
            if (!view_.in[c]) continue;
            bool placed = false;
            for (int p = 0; p < passes && !placed; p++)
                if (P_.obs_cell[p * 32 + (c & 31)] == 255) { P_.obs_cell[p * 32 + (c & 31)] = (uint8_t)c; placed = true; }
            if (!placed) left.push_back(c);
        }
        for (int c : left) {
            int slot = -1;
            for (int s = 0; s < kObsDiscSlots && slot < 0; s++) if (P_.obs_cell[s] == 255) slot = s;
            if (slot < 0) throw Fatal("view disc has more than 128 cells: k_obs lane schedule too small");
            P_.obs_cell[slot] = (uint8_t)c;
        }
    }

    require_obs_record(std::max(4, round_up(cfg.capacity, 4)));   // (refuses before anything is allocated)

    // cap-independent per-env arrays
    const size_t E = (size_t)P_.E;
    MF_CUDA(cudaMalloc(&S_.num, E * 2 * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.dead_ct, E * 2 * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.rng, E * sizeof(uint32_t)));
    MF_CUDA(cudaMalloc(&S_.step_ct, E * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.id_counter, E * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.walls, (size_t)P_.W * P_.H));
    MF_CUDA(cudaMalloc(&S_.init_num, E * 2 * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.side, E * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&S_.episode, E * sizeof(int32_t)));
    MF_CUDA(cudaMalloc(&RP_.place_short, E * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.side, 0, E * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.episode, 0, E * sizeof(int32_t)));
    MF_CUDA(cudaMemset(RP_.place_short, 0, E * sizeof(int32_t)));
    P_.tmpl_stride = 0; P_.random_sides = cfg.random_sides != 0;
    MF_CUDA(cudaMalloc(&S_.grid_template, grid_template_bytes()));
    {   // minimap cell of a position, as a table: the kernels never divide by the runtime scale
        if ((P_.H - 1) / P_.scale_h * kView + (P_.W - 1) / P_.scale_w > 255) throw Fatal("minimap table overflow");
        std::vector<uint8_t> lut((size_t)P_.W + P_.H);
        for (int x = 0; x < P_.W; x++) lut[x] = (uint8_t)(x / P_.scale_w);
        for (int y = 0; y < P_.H; y++) lut[(size_t)P_.W + y] = (uint8_t)((y / P_.scale_h) * kView);
        MF_CUDA(cudaMalloc(&S_.mini_lut, lut.size()));
        MF_CUDA(cudaMemcpy(S_.mini_lut, lut.data(), lut.size(), cudaMemcpyHostToDevice));
    }
    MF_CUDA(cudaMalloc(&S_.agent_steps, E * sizeof(unsigned long long)));
    MF_CUDA(cudaMemset(S_.agent_steps, 0, E * sizeof(unsigned long long)));
    MF_CUDA(cudaMalloc(&S_.obs_ticket, 2 * kObsTicketRing * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.obs_ticket, 0, 2 * kObsTicketRing * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.num, 0, E * 2 * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.dead_ct, 0, E * 2 * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.step_ct, 0, E * sizeof(int32_t)));
    MF_CUDA(cudaMemset(S_.id_counter, 0, E * sizeof(int32_t)));
    h_num_.assign(E * 2, 0);
#ifdef MF_PROFILE_BUILD
    { const char *dbg = getenv("MFMARL_OBS_DEBUG"); obs_debug_ = dbg ? atoi(dbg) : 0; }
#endif
    { const char *lim = getenv("MFMARL_OBS_GRID"); obs_grid_limit_ = lim ? atoi(lim) : 0; }
    set_seed(cfg.seed);   // seed 0 -> minstd state 1, as GridWorld.cc:31 random_engine.seed(0)
    alloc_state(std::max(4, round_up(cfg.capacity, 4)));
    reset();
    RP_.generation = 0;
}

Engine::~Engine() {
    free_state();
    cudaFree(S_.num); cudaFree(S_.dead_ct); cudaFree(S_.rng); cudaFree(S_.step_ct);
    cudaFree(S_.id_counter); cudaFree(S_.walls); cudaFree(S_.init_num); cudaFree(S_.agent_steps); cudaFree(S_.obs_ticket); cudaFree(S_.mini_lut); cudaFree(S_.grid_template);
    cudaFree(S_.side); cudaFree(S_.episode);
    cudaFree(RP_.place_short); cudaFree(RP_.occ); cudaFree((void *)RP_.ops);
    cudaFree(d_state_io_);
    if (state_io_done_) cudaEventDestroy(state_io_done_);
}

size_t Engine::grid_template_bytes() const {
    const size_t cells = (size_t)(P_.W + 2 * (kView / 2)) * (P_.H + 2 * (kView / 2));
    return (cells * 2 + 15) / 16 * 16;
}

// A geometry at which k_step or k_obs cannot keep its grid in shared memory runs them from HBM, and those variants read
// (k_obs) or build (k_step) the observation record: switch it on, or refuse an explicit "off".
void Engine::require_obs_record(int cap) {
    if (P_.obs_cached) return;
    const int W = P_.W, H = P_.H;
    const bool big = step_smem_layout(W, H, cap, 0).total > kSmemLimit || obs_smem_layout(W, H, cap, 0).total > kSmemLimit ||
                     local_mean_smem_layout(W, H, local_mean_tile(cap), n_action()).total > kSmemLimit;
    if (!big) return;
    if (obs_cached_off_)
        throw Fatal("observation record switched off (obs_record = 0 or MFMARL_OBS_CACHED=0), but a " + std::to_string(W) +
                    "x" + std::to_string(H) + " map with capacity " + std::to_string(cap) +
                    " does not fit in shared memory: its kernels run from HBM and read the observation record there; "
                    "leave obs_record at -1 (auto) or 1");
    P_.obs_cached = 1;
}

int Engine::hbm_kernels() const {
    const int W = P_.W, H = P_.H, cap = P_.cap;
    int m = 0;
    if (step_smem_layout(W, H, cap, P_.obs_cached).total > kSmemLimit) m |= HBM_STEP;
    // (one choice for fp32 and bf16 rows: the fp32 layout is the larger)
    if (P_.obs_cached && obs_smem_layout(W, H, cap, 1).total > kSmemLimit) m |= HBM_OBS;
    if (P_.obs_cached && obs_record_layout(W, H, cap).hp10 + 4 * 2 * kViewCells > kSmemLimit) m |= HBM_RECORD;
    if (local_mean_smem_layout(W, H, local_mean_tile(cap), n_action()).total > kSmemLimit) m |= HBM_LOCAL_MEAN;
    return m;
}

void Engine::alloc_state(int cap) {
    if (2 * cap > 0x3FFF) throw Fatal("capacity too large for the 14-bit slot field of the occupancy grid");
    require_obs_record(cap);
    P_.cap = cap;
    const size_t n = slots();
    MF_CUDA(cudaMalloc(&S_.pos, n * 4)); MF_CUDA(cudaMalloc(&S_.hp, n * 4));
    MF_CUDA(cudaMalloc(&S_.id, n * 4)); MF_CUDA(cudaMalloc(&S_.state, n * 4));
    MF_CUDA(cudaMalloc(&S_.next_rew, n * 4)); MF_CUDA(cudaMalloc(&S_.last_rew, n * 4));
    MF_CUDA(cudaMalloc(&S_.init_pos, (size_t)P_.E * 4 * cap * 4));     // room for a template per env
    S_.obs_record = nullptr;
    if (P_.obs_cached) {   // (hbm_kernels() & HBM_STEP implies obs_cached: require_obs_record)
        const size_t bytes = (size_t)P_.E * obs_record_layout(P_.W, P_.H, cap).total;
        const size_t ws = (hbm_kernels() & HBM_STEP) ? (size_t)P_.E * step_smem_layout(P_.W, P_.H, cap, 1).total : 0;
        MF_CUDA(cudaMalloc(&S_.obs_record, bytes + ws));
        MF_CUDA(cudaMemset(S_.obs_record, 0, bytes));
    }
    MF_CUDA(cudaMemset(S_.pos, 0, n * 4)); MF_CUDA(cudaMemset(S_.hp, 0, n * 4));
    MF_CUDA(cudaMemset(S_.id, 0, n * 4)); MF_CUDA(cudaMemset(S_.state, 0, n * 4));
    MF_CUDA(cudaMemset(S_.next_rew, 0, n * 4)); MF_CUDA(cudaMemset(S_.last_rew, 0, n * 4));
}

void Engine::free_state() {
    cudaFree(S_.pos); cudaFree(S_.hp); cudaFree(S_.id); cudaFree(S_.state);
    cudaFree(S_.next_rew); cudaFree(S_.last_rew); cudaFree(S_.init_pos); cudaFree(S_.obs_record);
    S_.obs_record = nullptr;
    S_.pos = nullptr; S_.hp = nullptr; S_.id = nullptr; S_.state = nullptr;
    S_.next_rew = S_.last_rew = nullptr; S_.init_pos = nullptr;
}

void Engine::set_seed(unsigned long seed) {
    // libstdc++ linear_congruential_engine<.., 16807, 0, 2147483647>::seed: s mod m, 0 -> 1
    unsigned long s = seed % 2147483647ul;
    std::vector<uint32_t> h((size_t)P_.E, (uint32_t)(s == 0 ? 1 : s));
    MF_CUDA(cudaMemcpy(S_.rng, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    P_.seed = (uint32_t)seed;
}

// ---------------------------------------------------------------------------------------------
// placement (host)
// ---------------------------------------------------------------------------------------------
void Engine::reset() {   // GridWorld::reset (GridWorld.cc:76-124) + Map::reset (Map.cc:23-47); RNG untouched
    const int W = P_.W, H = P_.H;
    h_walls_.assign((size_t)W * H, 0);
    for (int i = 0; i < W; i++) { h_walls_[i] = 1; h_walls_[(size_t)(H - 1) * W + i] = 1; }
    for (int i = 0; i < H; i++) { h_walls_[(size_t)i * W] = 1; h_walls_[(size_t)i * W + W - 1] = 1; }
    h_occ_.assign(h_walls_.begin(), h_walls_.end());
    for (int g = 0; g < kGroups; g++) { h_tpos_[g].clear(); h_tid_[g].clear(); }
    h_id_counter_ = 0;
    h_env_.clear();
    h_random_.clear();
    RP_.generation++;   // (the constructor's own reset leaves it at 0)
    placement_dirty_ = true;
    stepped_ = false;
    std::fill(h_num_.begin(), h_num_.end(), 0);
}

int Engine::add_walls(int n, const int *xs, const int *ys) {   // GridWorld.cc:203-211, Map::add_wall Map.cc:108-115
    if (stepped_) throw Fatal("add_walls after stepping is not supported (call reset first)");
    refuse_after_random("add_walls");
    int added = 0;
    for (int i = 0; i < n; i++) {
        const int x = xs[i], y = ys[i];
        if (x < 0 || y < 0 || x >= P_.W || y >= P_.H) continue;
        const size_t c = (size_t)y * P_.W + x;
        if (h_occ_[c] == 2) continue;   // an agent stands there: ignored
        bool taken = false;
        for (const EnvTemplate &t : h_env_) taken = taken || t.occ[c] == 2;
        if (taken) continue;            // (per-env placements: an agent of some env stands there)
        h_walls_[c] = 1; h_occ_[c] = 1; added++;
        for (EnvTemplate &t : h_env_) t.occ[c] = 1;
    }
    placement_dirty_ = true;
    return added;
}

int Engine::add_agents(int group, int n, const int *xs, const int *ys) {
    if (group < 0 || group >= kGroups) throw Fatal("invalid group handle in add_agents");
    refuse_after_random("add_agents");
    if (stepped_) {
        if (P_.E != 1) throw Fatal("add_agents after stepping is only supported for a single env");
        late_add_sync_down();
    }
    if (!h_env_.empty()) {          // per-env templates: the same request goes to every env
        if (stepped_) throw Fatal("add_agents after stepping is not supported with per-env placements");
        std::vector<int> rx((size_t)P_.E * n), ry((size_t)P_.E * n), cnt((size_t)P_.E);
        for (int e = 0; e < P_.E; e++) { std::copy(xs, xs + n, rx.begin() + (size_t)e * n); std::copy(ys, ys + n, ry.begin() + (size_t)e * n); }
        add_agents_per_env(group, n, rx.data(), ry.data(), cnt.data());
        return cnt[0];
    }
    int added = 0;
    for (int i = 0; i < n; i++) {   // GridWorld.cc:256-269; Map::add_agent Map.cc:75-97; add_or_error :180-187
        const int x = xs[i], y = ys[i];
        if (x < 0 || y < 0 || x + 1 >= P_.W || y + 1 >= P_.H) continue;   // is_blank_area bounds
        const size_t c = (size_t)y * P_.W + x;
        if (h_occ_[c] != 0) continue;                                      // occupied: ignored
        h_occ_[c] = 2;
        h_tpos_[group].push_back(x | (y << 16));
        h_tid_[group].push_back(h_id_counter_++);
        added++;
    }
    if (stepped_) late_add_sync_up(); else placement_dirty_ = true;
    return added;
}

void Engine::late_add_sync_down() {
    MF_CUDA(cudaDeviceSynchronize());
    const size_t n = slots();
    if (!late_) late_.reset(new LateRecords());
    LateRecords &R = *late_;
    R.pos.resize(n); R.id.resize(n); R.hp.resize(n); R.nr.resize(n); R.lr.resize(n); R.state.resize(n);
    MF_CUDA(cudaMemcpy(R.pos.data(), S_.pos, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.id.data(), S_.id, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.hp.data(), S_.hp, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.nr.data(), S_.next_rew, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.lr.data(), S_.last_rew, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.state.data(), S_.state, n * 4, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.num, S_.num, 8, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(R.dead, S_.dead_ct, 8, cudaMemcpyDeviceToHost));
    MF_CUDA(cudaMemcpy(&h_id_counter_, S_.id_counter, 4, cudaMemcpyDeviceToHost));
    h_occ_.assign(h_walls_.begin(), h_walls_.end());
    for (int g = 0; g < kGroups; g++) {
        h_tpos_[g].clear(); h_tid_[g].clear();
        for (int i = 0; i < R.num[g]; i++) {
            const size_t s = (size_t)g * P_.cap + i;
            if (!(R.state[s] & 1u)) h_occ_[(size_t)((R.pos[s] >> 16) & 0xFFFF) * P_.W + (R.pos[s] & 0xFFFF)] = 2;
        }
    }
}

void Engine::late_add_sync_up() {
    LateRecords &R = *late_;
    const int old_cap = P_.cap;
    int need = 0;
    for (int g = 0; g < kGroups; g++) need = std::max(need, R.num[g] + (int)h_tpos_[g].size());
    const int new_cap = need > old_cap ? round_up(need, 64) : old_cap;
    const size_t n = (size_t)2 * new_cap;
    std::vector<int32_t> pos(n, 0), id(n, 0); std::vector<float> hp(n, 0), nr(n, 0), lr(n, 0);
    std::vector<uint32_t> st(n, 0);
    int num[2];
    for (int g = 0; g < kGroups; g++) {
        for (int i = 0; i < R.num[g]; i++) {
            const size_t s = (size_t)g * old_cap + i, d = (size_t)g * new_cap + i;
            pos[d] = R.pos[s]; id[d] = R.id[s]; hp[d] = R.hp[s]; nr[d] = R.nr[s]; lr[d] = R.lr[s]; st[d] = R.state[s];
        }
        num[g] = R.num[g];
        for (size_t k = 0; k < h_tpos_[g].size(); k++) {
            const size_t d = (size_t)g * new_cap + num[g]++;
            pos[d] = h_tpos_[g][k]; id[d] = h_tid_[g][k]; hp[d] = P_.hp; nr[d] = P_.step_reward; lr[d] = 0.0f;
            st[d] = 0u | (OP_NULL << 8) | ((uint32_t)n_action() << 16);
        }
    }
    if (new_cap != old_cap) { free_state(); alloc_state(new_cap); }
    MF_CUDA(cudaMemcpy(S_.pos, pos.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.id, id.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.hp, hp.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.next_rew, nr.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.last_rew, lr.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.state, st.data(), n * 4, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.num, num, 8, cudaMemcpyHostToDevice));
    MF_CUDA(cudaMemcpy(S_.id_counter, &h_id_counter_, 4, cudaMemcpyHostToDevice));
    h_num_[0] = num[0]; h_num_[1] = num[1];
    rebuild_obs_records(nullptr);
    MF_CUDA(cudaStreamSynchronize(nullptr));
}

void Engine::restore_state(const int32_t *pos, const int32_t *id, const uint32_t *state, const float *hp,
                           const float *next_rew, const float *last_rew, const int32_t *num, const int32_t *dead_ct,
                           cudaStream_t st) {
    if (P_.E != 1) throw Fatal("restore_state needs a single env");
    const size_t bytes = slots() * 4;
    MF_CUDA(cudaMemcpyAsync(S_.pos, pos, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.id, id, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.state, state, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.hp, hp, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.next_rew, next_rew, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.last_rew, last_rew, bytes, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.num, num, 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.dead_ct, dead_ct, 8, cudaMemcpyHostToDevice, st));
    h_num_[0] = num[0]; h_num_[1] = num[1];
    rebuild_obs_records(st);
}

void Engine::rebuild_obs_records(cudaStream_t st) {
    if (!P_.obs_cached) return;
    if (hbm_kernels() & HBM_RECORD) {
        k_obs_record<true><<<P_.E, 256, 4 * 2 * kViewCells, st>>>(P_, S_);
    } else {
        const int smem = obs_record_layout(P_.W, P_.H, P_.cap).hp10 + 4 * 2 * kViewCells;
        raise_dynamic_smem((const void *)k_obs_record<false>, smem, device_);
        k_obs_record<false><<<P_.E, 256, smem, st>>>(P_, S_);
    }
    MF_CUDA(cudaGetLastError());
}

uint32_t Engine::pull_rng0() {
    uint32_t s = 1;
    MF_CUDA(cudaDeviceSynchronize());
    MF_CUDA(cudaMemcpy(&s, S_.rng, 4, cudaMemcpyDeviceToHost));
    return s;
}
void Engine::push_rng0(uint32_t s) { MF_CUDA(cudaMemcpy(S_.rng, &s, 4, cudaMemcpyHostToDevice)); }

bool Engine::cell_blank_for_placement(int x, int y) {
    if (stepped_) {
        if (P_.E != 1) throw Fatal("placement queries after stepping need a single env");
        late_add_sync_down();   // refreshes h_occ_ from the device; nothing is modified
        h_tpos_[0].clear(); h_tpos_[1].clear(); h_tid_[0].clear(); h_tid_[1].clear();
    }
    if (x < 0 || y < 0 || x + 1 >= P_.W || y + 1 >= P_.H) return false;
    return h_occ_[(size_t)y * P_.W + x] == 0;
}

void Engine::grow(int need_cap) {
    if (need_cap <= P_.cap) return;
    free_state();
    alloc_state(round_up(need_cap, 64));
}

void Engine::commit(cudaStream_t st) {
    if (!placement_dirty_) return;
    const bool per_env = !h_env_.empty();
    size_t rnd[kGroups] = {0, 0};   // a group's random agents sit behind its fixed ones (random_sides swaps both)
    for (const RandomOp &o : h_random_) rnd[o.group] += (size_t)o.n;
    size_t need = std::max(h_tpos_[0].size() + rnd[0], h_tpos_[1].size() + rnd[1]);
    for (const EnvTemplate &t : h_env_) need = std::max(need, std::max(t.pos[0].size() + rnd[0], t.pos[1].size() + rnd[1]));
    grow((int)need);
    RP_.n_ops = (int)h_random_.size();
    if (!h_random_.empty()) {
        if (h_random_.size() > d_random_cap_) {
            cudaFree((void *)RP_.ops); RP_.ops = nullptr;
            RandomOp *ops = nullptr;
            MF_CUDA(cudaMalloc(&ops, h_random_.size() * sizeof(RandomOp)));
            RP_.ops = ops; d_random_cap_ = h_random_.size();
        }
        MF_CUDA(cudaMemcpyAsync((void *)RP_.ops, h_random_.data(), h_random_.size() * sizeof(RandomOp), cudaMemcpyHostToDevice, st));
        if (!RP_.occ) MF_CUDA(cudaMalloc(&RP_.occ, (size_t)P_.E * ((P_.W * P_.H + 31) / 32) * 4));
    }
    const int cap = P_.cap;
    const size_t T = per_env ? (size_t)P_.E : 1;
    std::vector<int32_t> tmpl(T * 4 * cap, 0), num(T * 2, 0);
    for (size_t e = 0; e < T; e++)
        for (int g = 0; g < kGroups; g++) {
            const std::vector<int> &pos = per_env ? h_env_[e].pos[g] : h_tpos_[g], &id = per_env ? h_env_[e].id[g] : h_tid_[g];
            num[e * 2 + g] = (int32_t)pos.size();
            for (size_t i = 0; i < pos.size(); i++) {
                tmpl[e * 4 * cap + (size_t)g * cap + i] = pos[i];
                tmpl[e * 4 * cap + (size_t)2 * cap + (size_t)g * cap + i] = id[i];
            }
        }
    P_.tmpl_stride = per_env ? 4 * cap : 0;
    // pageable sources: these copies are synchronous with respect to the host
    MF_CUDA(cudaMemcpyAsync(S_.init_pos, tmpl.data(), tmpl.size() * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.init_num, num.data(), num.size() * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaMemcpyAsync(S_.walls, h_walls_.data(), h_walls_.size(), cudaMemcpyHostToDevice, st));
    wall_hash_ = 14695981039346656037ull;   // FNV-1a 64
    for (unsigned char b : h_walls_) wall_hash_ = (wall_hash_ ^ b) * 1099511628211ull;
    // the observation kernel's shared-memory grid starts from this image: walls only, 6-cell empty margin
    std::vector<uint16_t> gtmpl(grid_template_bytes() / 2, 0);
    const int PW = P_.W + 2 * (kView / 2);
    for (int y = 0; y < P_.H; y++)
        for (int x = 0; x < P_.W; x++)
            if (h_walls_[(size_t)y * P_.W + x]) gtmpl[(size_t)(y + kView / 2) * PW + x + kView / 2] = (uint16_t)(1u << 14);
    MF_CUDA(cudaMemcpyAsync(S_.grid_template, gtmpl.data(), gtmpl.size() * 2, cudaMemcpyHostToDevice, st));
    MF_CUDA(cudaStreamSynchronize(st));
    k_place<<<P_.E, 128, 0, st>>>(P_, S_, RP_);
    MF_CUDA(cudaGetLastError());
    rebuild_obs_records(st);
    // a placement is a per-episode event: wait for it, so that whatever stream the next launch uses (the legacy
    // stream of mfb_query, a non-blocking side stream of the caller) it is ordered after the new state
    MF_CUDA(cudaStreamSynchronize(st));
    for (int e = 0; e < P_.E; e++) { const size_t t = per_env ? (size_t)e : 0; h_num_[e * 2] = num[t * 2]; h_num_[e * 2 + 1] = num[t * 2 + 1]; }
    if (!h_random_.empty()) download_num(st);   // the draws decide how many agents each env holds
    placement_dirty_ = false;
    stepped_ = false;
}

void Engine::download_num(cudaStream_t st) {
    MF_CUDA(cudaMemcpyAsync(h_num_.data(), S_.num, h_num_.size() * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(cudaStreamSynchronize(st));
}

// ---------------------------------------------------------------------------------------------
// launches
// ---------------------------------------------------------------------------------------------
void Engine::observe(float *d_view, float *d_feature, int group_mask, cudaStream_t st) {
    // one [E][2][cap] block: group g's rows of env e start at (e*2 + g) * cap
    float *v[kGroups] = {d_view, d_view + (size_t)P_.cap * kViewRow};
    float *f[kGroups] = {d_feature, d_feature + (size_t)P_.cap * P_.feature_size};
    observe_groups(v, f, 2 * P_.cap, group_mask, st);
}

void Engine::observe_groups(float *const d_view[kGroups], float *const d_feature[kGroups], int env_stride,
                            int group_mask, cudaStream_t st, bool bf16) {
    commit(st);
    if (group_mask < 1 || group_mask > 3) throw Fatal("observe: bad group mask");
    ObsIO io;
    for (int g = 0; g < kGroups; g++) {
        io.view[g] = d_view[g]; io.feature[g] = d_feature[g];
        if (((group_mask >> g) & 1) && (!d_view[g] || !d_feature[g])) throw Fatal("observe: null output buffer");
        if (((group_mask >> g) & 1) && ((uintptr_t)d_view[g] & 15)) throw Fatal("observe: view buffer must be 16-byte aligned");
    }
    io.env_stride = env_stride; io.group_mask = group_mask;
    io.debug = obs_debug_;
    const int hbm = hbm_kernels();
    const bool rec_hbm = hbm & HBM_OBS;
    const ObsSmem L = obs_smem_layout(P_.W, P_.H, P_.cap, rec_hbm ? 2 : P_.obs_cached, bf16);
    void (*kern)(const BattleParams, const BattleState, const ObsIO) =
        rec_hbm ? (bf16 ? k_obs<true, true, true> : k_obs<true, false, true>) :
        P_.obs_cached ? (bf16 ? k_obs<true, true> : k_obs<true, false>) : (bf16 ? k_obs<false, true> : k_obs<false, false>);
    raise_dynamic_smem((const void *)kern, L.total, device_);
    int &ctas_per_sm = obs_ctas_per_sm_[bf16 ? 1 : 0];
    if (obs_attr_[bf16 ? 1 : 0] != L.total) {
        MF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, kObsThreads, L.total));
        obs_attr_[bf16 ? 1 : 0] = L.total;
    }
    // persistent CTAs (as many per SM as the shared memory allows) take (env, group, tile) work items from a ticket counter
    size_t ctas = (size_t)std::max(1, ctas_per_sm) * n_sm_;
    // Pipelined use (two engines on two streams): the sibling's k_step runs while this k_obs streams.  Where a k_step CTA
    // does not fit beside a full complement of k_obs CTAs (512 v 512: 73 KB next to 2 x 103 KB), it would wait for a
    // k_obs CTA to EXIT -- and persistent CTAs all exit at the end.  Leaving one k_obs slot free per expected k_step CTA
    // lets the two kernels really overlap: C4 on two streams 1.07e9 -> 1.16e9 agent-steps/s (profiles/r02).
    if (cfg_.concurrent_step_envs > 0) {
        const int step_smem = ((hbm & HBM_STEP) ? kStepHbmSmem : step_smem_layout(P_.W, P_.H, P_.cap, P_.obs_cached).total) + 1024;
        const int sm_smem = 227 * 1024, obs_smem = L.total + 1024;
        const int fit_beside_full = (sm_smem - ctas_per_sm * obs_smem) / step_smem;
        if (fit_beside_full < 1 && ctas_per_sm > 1) {
            const int per_freed_slot = std::max(1, (sm_smem - (ctas_per_sm - 1) * obs_smem) / step_smem);
            const size_t reserve = ((size_t)cfg_.concurrent_step_envs + per_freed_slot - 1) / per_freed_slot;
            ctas = ctas > reserve + (size_t)n_sm_ ? ctas - reserve : (size_t)n_sm_;
        }
    }
    // tile: a larger tile amortises the per-item grid rebuild over more agents (it matters when groups are large),
    // but the items must stay numerous enough to balance over the CTAs: measured at cap 512 x 128 envs, 128-agent
    // tiles (1024 items) beat 256 (512 items for 296 CTAs) and 64
    int want_tile = cfg_.obs_tile_agents;
    if (want_tile <= 0 && P_.obs_cached) {
        // an item starts with one copy of the env's record, so tiles can be small: many items per CTA, and the
        // last wave is short.  Measured at C4 on two streams (with the slot reservation above): 64 > 48 ~ 96 > 128 > 32
        want_tile = 64;
    } else if (want_tile <= 0) {
        want_tile = std::min(256, std::max(64, P_.cap));
        const size_t groups = (size_t)P_.E * (group_mask == 3 ? 2 : 1);
        while (want_tile > 128 && groups * ((P_.cap + want_tile - 1) / want_tile) < 3 * ctas) want_tile /= 2;
        // a handful of environments (the single-env ABI): latency, not throughput -- one chunk per CTA
        while (want_tile > kObsChunk && groups * ((P_.cap + want_tile - 1) / want_tile) < ctas / 8) want_tile /= 2;
    }
    io.tile_agents = std::min(kObsMaxTile, std::max(kObsChunk, round_up(want_tile, kObsChunk)));
    io.tiles_per_group = (P_.cap + io.tile_agents - 1) / io.tile_agents;
    const size_t items = (size_t)P_.E * (group_mask == 3 ? 2 : 1) * io.tiles_per_group;
    unsigned grid = (unsigned)std::min<size_t>(items, ctas);
    if (obs_grid_limit_ > 0) grid = std::min(grid, (unsigned)obs_grid_limit_);   // experiment knob (MFMARL_OBS_GRID)
    // every launch takes its own ticket pair from a small ring, so observe launches of one engine may overlap on
    // different streams (the last CTA of a launch rewinds its pair)
    BattleState S = S_;
    S.obs_ticket += 2 * (obs_launches_++ % kObsTicketRing);
    kern<<<grid, kObsThreads, L.total, st>>>(P_, S, io);
    MF_CUDA(cudaGetLastError());
    last_obs_tile_ = io.tile_agents;
    last_obs_grid_ = (int)grid;
}

int Engine::step_threads() const {
    int threads = cfg_.step_threads > 0 ? cfg_.step_threads : std::min(1024, std::max(64, P_.cap));
    // a few environments cannot fill the GPU anyway: wider CTAs shorten the parallel phases (grid load, lists, scans)
    if (cfg_.step_threads <= 0 && P_.E <= n_sm_ / 2) threads = std::max(threads, 256);
    return round_up(threads, 32);
}

void Engine::step(const StepIO &io, cudaStream_t st) {
    commit(st);
    const bool hbm = hbm_kernels() & HBM_STEP;
    const StepSmem L = step_smem_layout(P_.W, P_.H, P_.cap, P_.obs_cached);
    // the random placer only ever runs in the auto-reset branch
    const bool rnd = RP_.n_ops > 0 && (io.phases & PH_AUTORESET);
    void (*kern)(const BattleParams, const BattleState, const StepIO, const RandomPlacement) =
        hbm ? (rnd ? k_step<true, true> : k_step<true>) : (rnd ? k_step<false, true> : k_step<false>);
    if (!hbm) raise_dynamic_smem((const void *)kern, L.total, device_);
    const int threads = step_threads();
    kern<<<P_.E, threads, hbm ? kStepHbmSmem : L.total, st>>>(P_, S_, io, RP_);
    MF_CUDA(cudaGetLastError());
    if (io.phases & (PH_STEP | PH_CLEAR | PH_SETACT)) stepped_ = true;
}

void Engine::mean_action(const int32_t *d_actions, const int32_t *d_num, float *d_out, int rows, int cap,
                         int n_action, cudaStream_t st) {
    if (n_action > 32) throw Fatal("mean_action: at most 32 actions");
    const int warps_per_block = 8;
    const int blocks = (rows + warps_per_block - 1) / warps_per_block;
    k_mean_action<<<blocks, warps_per_block * 32, 0, st>>>(d_actions, d_num, d_out, rows, cap, n_action);
    MF_CUDA(cudaGetLastError());
}

void Engine::local_mean_action(double radius, float *const out[kGroups], cudaStream_t st) {
    const double view_radius = cfg_.type.view_radius;
    if (!(radius > 0.0 && radius <= view_radius)) {   // also NaN
        char msg[160];
        snprintf(msg, sizeof(msg), "local_mean_action: radius %g outside (0, view_radius = %g]", radius, view_radius);
        throw Fatal(msg);
    }
    int group_mask = 0;
    for (int g = 0; g < kGroups; g++) {
        if (!out[g]) continue;
        if ((uintptr_t)out[g] & 15) throw Fatal("local_mean_action: output buffer must be 16-byte aligned");
        group_mask |= 1 << g;
    }
    commit(st);
    if (!group_mask) return;
    const float r = (float)radius;                     // the engine's ranges are built from float radii
    auto it = local_discs_.find(r);
    if (it == local_discs_.end()) {
        const CircleRange disc(r, 0.0f, 1);
        if (disc.center > kPad) throw Fatal("local_mean_action: disc wider than the grid margin");
        LocalMeanIO t{};
        const int PW = P_.W + 2 * kPad;
        for (int k = 0; k < disc.count; k++)
            if (disc.dx[k] != 0 || disc.dy[k] != 0) t.delta[t.n_offsets++] = (int16_t)(disc.dy[k] * PW + disc.dx[k]);
        it = local_discs_.emplace(r, t).first;
    }
    LocalMeanIO io = it->second;
    io.W = P_.W; io.H = P_.H; io.cap = P_.cap; io.n_action = n_action();
    io.tile = local_mean_tile(P_.cap);
    int ng = 0;
    for (int g = 0; g < kGroups; g++) {
        io.out[g] = out[g];
        if ((group_mask >> g) & 1) io.group[ng++] = g;
    }
    const dim3 grid((unsigned)P_.E, (unsigned)((P_.cap + io.tile - 1) / io.tile), (unsigned)ng);
    if (hbm_kernels() & HBM_LOCAL_MEAN) {   // probes the observation record's grid (always kept at such geometries)
        if (!P_.obs_cached) throw Fatal("local_mean_action: a map this large needs the observation record");
        k_local_mean_action<true><<<grid, io.tile, local_mean_smem_layout(P_.W, P_.H, io.tile, io.n_action, false).total, st>>>(io, S_);
    } else {
        const LocalMeanSmem L = local_mean_smem_layout(P_.W, P_.H, io.tile, io.n_action);
        raise_dynamic_smem((const void *)k_local_mean_action<false>, L.total, device_);
        k_local_mean_action<false><<<grid, io.tile, L.total, st>>>(io, S_);
    }
    MF_CUDA(cudaGetLastError());
}

}  // namespace mfmarl
