// mfb_*: batched, device-resident C ABI (include/mfmarl_batched.h).
#include <cudaTypedefs.h>

#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "../../include/mfmarl_batched.h"
#include "engine.h"

using namespace mfmarl;

struct mfb_engine {
    std::unique_ptr<Engine> eng;
    bool auto_reset = false;
    // staging for mfb_step_host
    int32_t *d_actions = nullptr, *d_done = nullptr;
    float *d_reward = nullptr, *d_mean = nullptr;
    uint8_t *d_alive = nullptr;
    size_t staged_slots = 0;
    // pipelined host path (mfb_step_host_async): two staging sets, copy streams, events
    struct Slot {
        int32_t *d_actions = nullptr, *d_done = nullptr; float *d_reward = nullptr, *d_mean = nullptr;
        uint8_t *d_alive = nullptr;
        cudaEvent_t in_done = nullptr, step_done = nullptr, out_done = nullptr;
        bool used = false;
    } slot[2];
    cudaStream_t cs_in = nullptr, cs_out = nullptr;
    size_t async_slots = 0;
    unsigned long long async_calls = 0;
    ~mfb_engine() {
        cudaFree(d_actions); cudaFree(d_done); cudaFree(d_reward); cudaFree(d_mean); cudaFree(d_alive);
        for (Slot &s : slot) {
            cudaFree(s.d_actions); cudaFree(s.d_done); cudaFree(s.d_reward); cudaFree(s.d_mean); cudaFree(s.d_alive);
            if (s.in_done) cudaEventDestroy(s.in_done);
            if (s.step_done) cudaEventDestroy(s.step_done);
            if (s.out_done) cudaEventDestroy(s.out_done);
        }
        if (cs_in) cudaStreamDestroy(cs_in);
        if (cs_out) cudaStreamDestroy(cs_out);
    }
};

namespace {
int fail(const char *where, const std::exception &ex) {
    set_last_error(std::string(where) + ": " + ex.what());
    return -1;
}
Engine &E(mfb_engine *h) {
    if (!h || !h->eng) throw Fatal("null engine handle");
    return *h->eng;
}

// Compressible device memory (mfb_alloc_device).  The driver's virtual-memory calls are looked up through the runtime,
// so libmagent.so needs no libcuda at link or load time (the CPU-only tests load it on machines without a driver).
struct DriverVmm {
    PFN_cuDeviceGet get_device = nullptr;
    PFN_cuDeviceGetAttribute get_attribute = nullptr;
    PFN_cuMemGetAllocationGranularity granularity = nullptr;
    PFN_cuMemAddressReserve reserve = nullptr;
    PFN_cuMemAddressFree address_free = nullptr;
    PFN_cuMemCreate create = nullptr;
    PFN_cuMemGetAllocationPropertiesFromHandle properties = nullptr;
    PFN_cuMemRelease release = nullptr;
    PFN_cuMemMap map = nullptr;
    PFN_cuMemUnmap unmap = nullptr;
    PFN_cuMemSetAccess set_access = nullptr;
};

const DriverVmm &driver_vmm() {
    static const DriverVmm d = [] {
        DriverVmm v;
        auto get = [](const char *sym, void **fn) {
            cudaDriverEntryPointQueryResult q;
            MF_CUDA(cudaGetDriverEntryPointByVersion(sym, fn, 12000, cudaEnableDefault, &q));
            if (q != cudaDriverEntryPointSuccess || !*fn) throw Fatal(std::string("driver entry point missing: ") + sym);
        };
        get("cuDeviceGet", (void **)&v.get_device);
        get("cuDeviceGetAttribute", (void **)&v.get_attribute);
        get("cuMemGetAllocationGranularity", (void **)&v.granularity);
        get("cuMemAddressReserve", (void **)&v.reserve);
        get("cuMemAddressFree", (void **)&v.address_free);
        get("cuMemCreate", (void **)&v.create);
        get("cuMemGetAllocationPropertiesFromHandle", (void **)&v.properties);
        get("cuMemRelease", (void **)&v.release);
        get("cuMemMap", (void **)&v.map);
        get("cuMemUnmap", (void **)&v.unmap);
        get("cuMemSetAccess", (void **)&v.set_access);
        return v;
    }();
    return d;
}

void cu_check(CUresult r, const char *what) {
    if (r != CUDA_SUCCESS) throw Fatal(std::string(what) + " failed: CUresult " + std::to_string((int)r));
}

struct DeviceBlock { size_t size; CUmemGenericAllocationHandle handle; };   // size 0: a cudaMalloc fallback
std::mutex g_blocks_mu;
std::map<void *, DeviceBlock> g_blocks;

// The caller's current device is restored when the allocator returns.
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { MF_CUDA(cudaGetDevice(&prev)); MF_CUDA(cudaSetDevice(dev)); }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Reserve + create + map + access, all or nothing.  Returns nullptr (and keeps nothing) when the driver hands back an
// allocation without generic compression, or has no compressible memory left for it (the caller then falls back to
// cudaMalloc, which reports a real out-of-memory itself).
void *map_compressible(const DriverVmm &d, size_t bytes, int device, size_t *mapped, CUmemGenericAllocationHandle *h) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    cu_check(d.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM), "cuMemGetAllocationGranularity");
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUdeviceptr va = 0;
    cu_check(d.reserve(&va, size, gran, 0, 0), "cuMemAddressReserve");
    CUresult r = d.create(h, size, &prop, 0);
    if (r != CUDA_SUCCESS) {
        d.address_free(va, size);
        if (r == CUDA_ERROR_OUT_OF_MEMORY) return nullptr;
        cu_check(r, "cuMemCreate");
    }
    CUmemAllocationProp got = {};
    r = d.properties(&got, *h);
    if (r == CUDA_SUCCESS && got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) {
        d.release(*h); d.address_free(va, size);
        return nullptr;
    }
    if (r == CUDA_SUCCESS) r = d.map(va, size, 0, *h, 0);
    if (r == CUDA_SUCCESS) {
        CUmemAccessDesc acc = {};
        acc.location = prop.location;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        r = d.set_access(va, size, &acc, 1);
        if (r != CUDA_SUCCESS) d.unmap(va, size);
    }
    if (r != CUDA_SUCCESS) { d.release(*h); d.address_free(va, size); cu_check(r, "mapping compressible memory"); }
    *mapped = size;
    return (void *)va;
}
}  // namespace

#define MFB_BEGIN try {
#define MFB_END(name) } catch (const std::exception &ex) { return fail(name, ex); } return 0;

extern "C" {

int mfb_default_config(mfb_config *c) {
    MFB_BEGIN
    memset(c, 0, sizeof(*c));
    c->n_envs = 1; c->map_width = c->map_height = 40; c->capacity = 64; c->embedding_size = 10;
    c->rng_mode = MFB_RNG_MINSTD; c->device = -1; c->obs_tile_agents = 0; c->obs_record = -1;
    AgentTypeParams t;
    c->hp = t.hp; c->speed = t.speed; c->view_radius = t.view_radius; c->attack_radius = t.attack_radius;
    c->damage = t.damage; c->step_recover = t.step_recover; c->kill_supply = t.kill_supply;
    c->step_reward = t.step_reward; c->kill_reward = t.kill_reward; c->dead_penalty = t.dead_penalty;
    c->attack_penalty = t.attack_penalty; c->attack_bonus[0] = c->attack_bonus[1] = 0.2f;
    MFB_END("mfb_default_config")
}

int mfb_create(const mfb_config *c, mfb_engine **out) {
    MFB_BEGIN
    EngineConfig ec;
    ec.n_envs = c->n_envs; ec.width = c->map_width; ec.height = c->map_height; ec.capacity = c->capacity;
    ec.embedding_size = c->embedding_size; ec.rng_mode = c->rng_mode; ec.seed = c->seed;
    ec.env_base = c->env_base; ec.max_steps = c->max_steps; ec.device = c->device;
    ec.step_threads = c->step_threads; ec.obs_tile_agents = c->obs_tile_agents; ec.obs_cached = c->obs_record; ec.random_sides = c->random_sides;
    ec.concurrent_step_envs = c->concurrent_step_envs;
    ec.type.hp = c->hp; ec.type.speed = c->speed; ec.type.view_radius = c->view_radius;
    ec.type.attack_radius = c->attack_radius; ec.type.damage = c->damage; ec.type.step_recover = c->step_recover;
    ec.type.kill_supply = c->kill_supply; ec.type.step_reward = c->step_reward; ec.type.kill_reward = c->kill_reward;
    ec.type.dead_penalty = c->dead_penalty; ec.type.attack_penalty = c->attack_penalty;
    ec.attack_bonus[0] = c->attack_bonus[0]; ec.attack_bonus[1] = c->attack_bonus[1];
    std::unique_ptr<mfb_engine> h(new mfb_engine());
    h->eng.reset(new Engine(ec));
    h->auto_reset = c->auto_reset != 0;
    *out = h.release();
    MFB_END("mfb_create")
}

int mfb_destroy(mfb_engine *h) {
    MFB_BEGIN
    if (h) { cudaDeviceSynchronize(); delete h; }
    MFB_END("mfb_destroy")
}

int mfb_reset(mfb_engine *h) { MFB_BEGIN E(h).reset(); MFB_END("mfb_reset") }
int mfb_add_walls(mfb_engine *h, int n, const int *xs, const int *ys) { MFB_BEGIN E(h).add_walls(n, xs, ys); MFB_END("mfb_add_walls") }
int mfb_add_agents(mfb_engine *h, int group, int n, const int *xs, const int *ys, int *n_added) {
    MFB_BEGIN
    const int added = E(h).add_agents(group, n, xs, ys);
    if (n_added) *n_added = added;
    MFB_END("mfb_add_agents")
}
int mfb_add_agents_per_env(mfb_engine *h, int group, int n, const int *xs, const int *ys, int *n_added) {
    MFB_BEGIN
    E(h).add_agents_per_env(group, n, xs, ys, n_added);
    MFB_END("mfb_add_agents_per_env")
}
int mfb_add_agents_random(mfb_engine *h, int group, int n, int x0, int y0, int w, int hgt) {
    MFB_BEGIN
    E(h).add_agents_random(group, n, x0, y0, w, hgt);
    MFB_END("mfb_add_agents_random")
}
int mfb_set_seed(mfb_engine *h, unsigned long seed) { MFB_BEGIN E(h).set_seed(seed); MFB_END("mfb_set_seed") }

int mfb_query(mfb_engine *h, const char *key, int *out) {
    MFB_BEGIN
    Engine &e = E(h);
    e.commit(nullptr);
    const std::string k(key);
    if (k == "capacity") *out = e.cap();
    else if (k == "n_envs") *out = e.n_envs();
    else if (k == "n_action") *out = e.n_action();
    else if (k == "view_size") *out = e.params().view;
    else if (k == "n_channel") *out = 7;
    else if (k == "feature_size") *out = e.params().feature_size;
    else if (k == "attack_base") *out = e.params().n_move;
    else if (k == "hbm_kernels") *out = e.hbm_kernels();   // 1 k_step, 2 k_obs, 4 k_obs_record, 8 k_local_mean_action
    else if (k == "step_threads") *out = e.step_threads();   // k_step's CTA width
    else if (k == "obs_record") *out = e.params().obs_cached;
    else if (k == "obs_tile") *out = e.last_obs_tile();       // k_obs's tile_agents and grid at the last observe
    else if (k == "obs_grid") *out = e.last_obs_grid();
    else if (k == "state_bytes") *out = (int)e.state_bytes();
    else throw Fatal("mfb_query: unknown key " + k);
    MFB_END("mfb_query")
}

int mfb_observe(mfb_engine *h, float *d_view, float *d_feature, int group_mask, void *stream) {
    MFB_BEGIN
    E(h).observe(d_view, d_feature, group_mask, (cudaStream_t)stream);
    MFB_END("mfb_observe")
}

int mfb_observe_groups(mfb_engine *h, float *d_view0, float *d_feature0, float *d_view1, float *d_feature1,
                       void *stream) {
    MFB_BEGIN
    float *v[kGroups] = {d_view0, d_view1}, *f[kGroups] = {d_feature0, d_feature1};
    const int mask = (d_view0 ? 1 : 0) | (d_view1 ? 2 : 0);
    E(h).observe_groups(v, f, E(h).params().cap, mask, (cudaStream_t)stream);
    MFB_END("mfb_observe_groups")
}

int mfb_observe_groups_bf16(mfb_engine *h, void *d_view0, float *d_feature0, void *d_view1, float *d_feature1,
                            void *stream) {
    MFB_BEGIN
    float *v[kGroups] = {(float *)d_view0, (float *)d_view1}, *f[kGroups] = {d_feature0, d_feature1};
    const int mask = (d_view0 ? 1 : 0) | (d_view1 ? 2 : 0);
    E(h).observe_groups(v, f, E(h).params().cap, mask, (cudaStream_t)stream, true);
    MFB_END("mfb_observe_groups_bf16")
}

int mfb_step(mfb_engine *h, const int32_t *d_actions, const int32_t *d_attack_perm, float *d_reward,
             uint8_t *d_alive, float *d_mean_action, int32_t *d_done, int clear_dead, void *stream) {
    MFB_BEGIN
    Engine &e = E(h);
    if (e.params().rng_mode == RNG_INJECT && !d_attack_perm) throw Fatal("rng_mode INJECT needs d_attack_perm");
    StepIO io{};
    io.actions = d_actions; io.attack_perm = d_attack_perm; io.reward = d_reward; io.alive = d_alive;
    io.mean_action = d_mean_action; io.done = d_done;
    io.phases = PH_SETACT | PH_STEP | PH_EXPORT | (clear_dead ? PH_CLEAR : 0) | (h->auto_reset ? PH_AUTORESET : 0);
    io.setact_mask = 3; io.group_seq[0] = 0; io.group_seq[1] = 1;
    e.step(io, (cudaStream_t)stream);
    MFB_END("mfb_step")
}

int mfb_clear_dead(mfb_engine *h, void *stream) {
    MFB_BEGIN
    StepIO io{};
    io.phases = PH_CLEAR; io.group_seq[0] = io.group_seq[1] = -1;
    E(h).step(io, (cudaStream_t)stream);
    MFB_END("mfb_clear_dead")
}

int mfb_mean_action(const int32_t *d_actions, const int32_t *d_num, float *d_out, int rows, int cap,
                    int n_action, void *stream) {
    MFB_BEGIN
    Engine::mean_action(d_actions, d_num, d_out, rows, cap, n_action, (cudaStream_t)stream);
    MFB_END("mfb_mean_action")
}

int mfb_local_mean_action(mfb_engine *h, double radius, float *d_out0, float *d_out1, void *stream) {
    MFB_BEGIN
    float *out[kGroups] = {d_out0, d_out1};
    E(h).local_mean_action(radius, out, (cudaStream_t)stream);
    MFB_END("mfb_local_mean_action")
}

int mfb_get(mfb_engine *h, const char *key, void *host_buf, void *stream) {
    MFB_BEGIN
    Engine &e = E(h);
    cudaStream_t st = (cudaStream_t)stream;
    e.commit(st);
    const BattleState &S = e.state();
    const size_t n = e.slots(), ne = (size_t)e.n_envs();
    const std::string k(key);
    auto copy = [&](const void *d, size_t bytes) {
        MF_CUDA(cudaMemcpyAsync(host_buf, d, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaStreamSynchronize(st));
    };
    if (k == "num") copy(S.num, ne * 2 * 4);
    else if (k == "dead_ct") copy(S.dead_ct, ne * 2 * 4);
    else if (k == "hp") copy(S.hp, n * 4);
    else if (k == "id") copy(S.id, n * 4);
    else if (k == "step_ct") copy(S.step_ct, ne * 4);
    else if (k == "side") copy(S.side, ne * 4);
    else if (k == "episode") copy(S.episode, ne * 4);
    else if (k == "placement_short") copy(e.placement_short(), ne * 4);
    else if (k == "rng") copy(S.rng, ne * 4);
    else if (k == "agent_steps") copy(S.agent_steps, ne * 8);
    else if (k == "walls") memcpy(host_buf, e.host_walls().data(), e.host_walls().size());
    else if (k == "pos" || k == "alive" || k == "last_action") {
        std::vector<int32_t> tmp(n);
        MF_CUDA(cudaMemcpyAsync(tmp.data(), k == "pos" ? (const void *)S.pos : (const void *)S.state, n * 4,
                                cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaStreamSynchronize(st));
        if (k == "pos") {
            int32_t *o = (int32_t *)host_buf;
            for (size_t i = 0; i < n; i++) { o[2 * i] = tmp[i] & 0xFFFF; o[2 * i + 1] = (tmp[i] >> 16) & 0xFFFF; }
        } else if (k == "alive") {
            uint8_t *o = (uint8_t *)host_buf;
            for (size_t i = 0; i < n; i++) o[i] = !(tmp[i] & 1);
        } else {
            int32_t *o = (int32_t *)host_buf;
            for (size_t i = 0; i < n; i++) o[i] = (tmp[i] >> 16) & 0xFF;
        }
    } else throw Fatal("mfb_get: unknown key " + k);
    MFB_END("mfb_get")
}

int mfb_save_envs(mfb_engine *h, int n, const int32_t *envs, void *d_out, void *stream) {
    MFB_BEGIN
    E(h).save_envs(n, envs, d_out, (cudaStream_t)stream);
    MFB_END("mfb_save_envs")
}

int mfb_render_observations(mfb_engine *h, int n_records, const void *d_records, int n_rows, const int32_t *d_rows,
                            float *d_view, float *d_feature, int32_t *d_bad_rows, void *stream) {
    MFB_BEGIN
    E(h).render_observations(n_records, d_records, n_rows, d_rows, d_view, d_feature, d_bad_rows, (cudaStream_t)stream);
    MFB_END("mfb_render_observations")
}

int mfb_load_envs(mfb_engine *h, int n, const int32_t *envs, const void *d_in, void *stream) {
    MFB_BEGIN
    E(h).load_envs(n, envs, d_in, (cudaStream_t)stream);
    MFB_END("mfb_load_envs")
}

int mfb_num_device_ptr(mfb_engine *h, const int32_t **out) {
    MFB_BEGIN
    *out = E(h).state().num;
    MFB_END("mfb_num_device_ptr")
}

int mfb_state_device_ptr(mfb_engine *h, const char *key, const void **out) {
    MFB_BEGIN
    Engine &e = E(h);
    const BattleState &S = e.state();
    const std::string k(key);
    if (k == "num") *out = S.num;
    else if (k == "id") *out = S.id;
    else if (k == "pos") *out = S.pos;
    else if (k == "hp") *out = S.hp;
    else if (k == "step_ct") *out = S.step_ct;
    else throw Fatal("mfb_state_device_ptr: unknown key " + k);
    MFB_END("mfb_state_device_ptr")
}

int mfb_step_host(mfb_engine *h, const int32_t *h_actions, float *h_reward, uint8_t *h_alive,
                  float *h_mean_action, int32_t *h_done, void *stream) {
    MFB_BEGIN
    Engine &e = E(h);
    cudaStream_t st = (cudaStream_t)stream;
    e.commit(st);
    const size_t n = e.slots(), ne = (size_t)e.n_envs(), na = (size_t)e.n_action();
    if (h->staged_slots != n) {
        cudaFree(h->d_actions); cudaFree(h->d_done); cudaFree(h->d_reward); cudaFree(h->d_mean); cudaFree(h->d_alive);
        MF_CUDA(cudaMalloc(&h->d_actions, n * 4)); MF_CUDA(cudaMalloc(&h->d_reward, n * 4));
        MF_CUDA(cudaMalloc(&h->d_alive, n)); MF_CUDA(cudaMalloc(&h->d_mean, ne * 2 * na * 4));
        MF_CUDA(cudaMalloc(&h->d_done, ne * 4));
        h->staged_slots = n;
    }
    MF_CUDA(cudaMemcpyAsync(h->d_actions, h_actions, n * 4, cudaMemcpyHostToDevice, st));
    StepIO io{};
    io.actions = h->d_actions; io.reward = h->d_reward; io.alive = h->d_alive; io.mean_action = h->d_mean; io.done = h->d_done;
    io.phases = PH_SETACT | PH_STEP | PH_EXPORT | PH_CLEAR | (h->auto_reset ? PH_AUTORESET : 0);
    io.setact_mask = 3; io.group_seq[0] = 0; io.group_seq[1] = 1;
    e.step(io, st);
    if (h_reward) MF_CUDA(cudaMemcpyAsync(h_reward, h->d_reward, n * 4, cudaMemcpyDeviceToHost, st));
    if (h_alive) MF_CUDA(cudaMemcpyAsync(h_alive, h->d_alive, n, cudaMemcpyDeviceToHost, st));
    if (h_mean_action) MF_CUDA(cudaMemcpyAsync(h_mean_action, h->d_mean, ne * 2 * na * 4, cudaMemcpyDeviceToHost, st));
    if (h_done) MF_CUDA(cudaMemcpyAsync(h_done, h->d_done, ne * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(cudaStreamSynchronize(st));
    MFB_END("mfb_step_host")
}

int mfb_step_host_async(mfb_engine *h, const int32_t *h_actions, float *h_reward, uint8_t *h_alive,
                        float *h_mean_action, int32_t *h_done, void *stream, int *ticket) {
    MFB_BEGIN
    Engine &e = E(h);
    cudaStream_t st = (cudaStream_t)stream;
    e.commit(st);
    const size_t n = e.slots(), ne = (size_t)e.n_envs(), na = (size_t)e.n_action();
    if (!h->cs_in) {
        MF_CUDA(cudaStreamCreateWithFlags(&h->cs_in, cudaStreamNonBlocking));
        MF_CUDA(cudaStreamCreateWithFlags(&h->cs_out, cudaStreamNonBlocking));
        for (mfb_engine::Slot &s : h->slot) {
            MF_CUDA(cudaEventCreateWithFlags(&s.in_done, cudaEventDisableTiming));
            MF_CUDA(cudaEventCreateWithFlags(&s.step_done, cudaEventDisableTiming));
            MF_CUDA(cudaEventCreateWithFlags(&s.out_done, cudaEventDisableTiming));
        }
    }
    if (h->async_slots != n) {
        MF_CUDA(cudaDeviceSynchronize());
        for (mfb_engine::Slot &s : h->slot) {
            cudaFree(s.d_actions); cudaFree(s.d_done); cudaFree(s.d_reward); cudaFree(s.d_mean); cudaFree(s.d_alive);
            MF_CUDA(cudaMalloc(&s.d_actions, n * 4)); MF_CUDA(cudaMalloc(&s.d_reward, n * 4));
            MF_CUDA(cudaMalloc(&s.d_alive, n)); MF_CUDA(cudaMalloc(&s.d_mean, ne * 2 * na * 4));
            MF_CUDA(cudaMalloc(&s.d_done, ne * 4));
            s.used = false;
        }
        h->async_slots = n;
    }
    const int which = (int)(h->async_calls++ & 1);
    mfb_engine::Slot &s = h->slot[which];
    // inputs: this slot's action buffer is free once the k_step that read it two calls ago has finished
    if (s.used) MF_CUDA(cudaStreamWaitEvent(h->cs_in, s.step_done, 0));
    MF_CUDA(cudaMemcpyAsync(s.d_actions, h_actions, n * 4, cudaMemcpyHostToDevice, h->cs_in));
    MF_CUDA(cudaEventRecord(s.in_done, h->cs_in));
    // step: after the actions landed, and after this slot's previous results were copied out
    MF_CUDA(cudaStreamWaitEvent(st, s.in_done, 0));
    if (s.used) MF_CUDA(cudaStreamWaitEvent(st, s.out_done, 0));
    StepIO io{};
    io.actions = s.d_actions; io.reward = s.d_reward; io.alive = s.d_alive; io.mean_action = s.d_mean; io.done = s.d_done;
    io.phases = PH_SETACT | PH_STEP | PH_EXPORT | PH_CLEAR | (h->auto_reset ? PH_AUTORESET : 0);
    io.setact_mask = 3; io.group_seq[0] = 0; io.group_seq[1] = 1;
    e.step(io, st);
    MF_CUDA(cudaEventRecord(s.step_done, st));
    // outputs: on the second copy stream, overlapping whatever the caller launches next on `stream`
    MF_CUDA(cudaStreamWaitEvent(h->cs_out, s.step_done, 0));
    if (h_reward) MF_CUDA(cudaMemcpyAsync(h_reward, s.d_reward, n * 4, cudaMemcpyDeviceToHost, h->cs_out));
    if (h_alive) MF_CUDA(cudaMemcpyAsync(h_alive, s.d_alive, n, cudaMemcpyDeviceToHost, h->cs_out));
    if (h_mean_action) MF_CUDA(cudaMemcpyAsync(h_mean_action, s.d_mean, ne * 2 * na * 4, cudaMemcpyDeviceToHost, h->cs_out));
    if (h_done) MF_CUDA(cudaMemcpyAsync(h_done, s.d_done, ne * 4, cudaMemcpyDeviceToHost, h->cs_out));
    MF_CUDA(cudaEventRecord(s.out_done, h->cs_out));
    s.used = true;
    if (ticket) *ticket = which;
    MFB_END("mfb_step_host_async")
}

int mfb_host_wait(mfb_engine *h, int ticket) {
    MFB_BEGIN
    E(h);
    if (ticket < 0 || ticket > 1) throw Fatal("mfb_host_wait: bad ticket");
    if (h->slot[ticket].used) MF_CUDA(cudaEventSynchronize(h->slot[ticket].out_done));
    MFB_END("mfb_host_wait")
}

int mfb_alloc_device(unsigned long bytes, int device, void **ptr, int *compressed) {
    MFB_BEGIN
    if (!ptr || !compressed) throw Fatal("mfb_alloc_device: null output pointer");
    if (bytes == 0) throw Fatal("mfb_alloc_device: zero bytes");
    *ptr = nullptr; *compressed = 0;
    DeviceGuard guard(device);
    MF_CUDA(cudaFree(nullptr));                           // the device's primary context is current for the driver calls
    const DriverVmm &d = driver_vmm();
    CUdevice cu_dev;
    int supported = 0;
    cu_check(d.get_device(&cu_dev, device), "cuDeviceGet");
    cu_check(d.get_attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, cu_dev), "cuDeviceGetAttribute");
    DeviceBlock blk{0, 0};
    void *p = supported ? map_compressible(d, bytes, device, &blk.size, &blk.handle) : nullptr;
    if (!p) { MF_CUDA(cudaMalloc(&p, bytes)); blk.size = 0; }
    // zeroed, as torch.zeros hands out a fresh buffer; synchronised because the caller's streams may not order
    // themselves after the legacy default stream
    cudaError_t err = cudaMemset(p, 0, bytes);
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) {
        if (blk.size) { d.unmap((CUdeviceptr)p, blk.size); d.release(blk.handle); d.address_free((CUdeviceptr)p, blk.size); }
        else cudaFree(p);
        MF_CUDA(err);
    }
    {
        std::lock_guard<std::mutex> lock(g_blocks_mu);
        g_blocks[p] = blk;
    }
    *ptr = p;
    *compressed = blk.size != 0;
    MFB_END("mfb_alloc_device")
}

int mfb_free_device(void *ptr) {
    MFB_BEGIN
    if (!ptr) return 0;
    DeviceBlock blk;
    {
        std::lock_guard<std::mutex> lock(g_blocks_mu);
        auto it = g_blocks.find(ptr);
        if (it == g_blocks.end()) throw Fatal("mfb_free_device: pointer not from mfb_alloc_device");
        blk = it->second;
        g_blocks.erase(it);
    }
    MF_CUDA(cudaDeviceSynchronize());                     // no queued kernel may still write the block
    if (blk.size == 0) {
        MF_CUDA(cudaFree(ptr));
    } else {
        const DriverVmm &d = driver_vmm();
        cu_check(d.unmap((CUdeviceptr)ptr, blk.size), "cuMemUnmap");
        cu_check(d.release(blk.handle), "cuMemRelease");
        cu_check(d.address_free((CUdeviceptr)ptr, blk.size), "cuMemAddressFree");
    }
    MFB_END("mfb_free_device")
}

const char *mfb_last_error(void) { return last_error(); }

}  // extern "C"
