// The drop-in boundary: the reference's runtime_api.h C symbols (examples/battle_model/src/runtime_api.h:20-55,
// implemented there in runtime_api.cc:15-169) over the CUDA engine.  One game = one environment;
// every data buffer is a caller-owned HOST array sized from get_info("num") exactly as the reference's
// Python binding does (python/magent/gridworld.py:282-342,377-389), so each call ends with a
// device->host copy.  Declared in include/mfmarl_magent.h.
//
// Scope: the battle path (SURVEY.md section 8).  Configurations the kernels are not built for
// (turn_mode, food_mode, bodies larger than 1x1, sector ranges, reward rules other than
// `any(a) attack any(b) -> a`) fail loudly at reset instead of running something different.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <memory>
#include <string>
#include <vector>

#include "../../include/mfmarl_magent.h"
#include "engine.h"

using namespace mfmarl;

namespace {

struct TypeDef {   // AgentType.cc:30-84
    int width = 1, length = 1;
    float view_angle = 360, attack_angle = 0;
    bool attack_in_group = false, can_absorb = false;
    AgentTypeParams p;
    TypeDef() { p.hp = 1.0f; p.speed = 1.0f; p.view_radius = 1; p.attack_radius = 0; p.damage = 0;
                p.step_recover = 0; p.kill_supply = 0; p.step_reward = 0; p.kill_reward = 0;
                p.dead_penalty = 0; p.attack_penalty = 0; }
};

struct Symbol { int group = 0, index = -1; };
struct Node { int op = -1; std::vector<int> inputs; };
struct Rule { int on; std::vector<int> receivers; std::vector<float> values; bool terminal, auto_value; };

struct Game {
    // config (GridWorld::set_config, GridWorld.cc:126-155)
    int width = 0, height = 0, embedding_size = 0;
    bool food_mode = false, turn_mode = false, minimap_mode = false, goal_mode = false;
    bool seed_set = false; unsigned long seed = 0;
    std::map<std::string, TypeDef> types;
    std::vector<std::string> groups;
    std::vector<Symbol> symbols;
    std::vector<Node> nodes;
    std::vector<Rule> rules;

    std::unique_ptr<Engine> eng;
    cudaStream_t st = nullptr;

    // device staging for the host-buffer ABI, sized for staged_cap agents per group (d_done: one word)
    float *d_view = nullptr, *d_feat = nullptr;
    int32_t *d_actions = nullptr, *d_perm = nullptr, *d_events = nullptr, *d_done = nullptr;
    int staged_cap = 0;
    std::vector<int> seq;          // groups in set_action call order since the last step
    bool inject_next = false;

    // Host mirror (pinned, mapped).  Every env_* call of the reference ABI is synchronous, so the cost of one environment
    // is what sits between a call and its answer, not kernel time:
    //   * set_action only stages the actions on the host; env_step runs set_action x2 + step in ONE launch that reads
    //     them straight from the pinned buffer (if an observation or a getter is asked for in between, the staged
    //     actions are applied first);
    //   * k_step itself writes the agents' records into the mirror (StepIO::mirror): get_reward, get_alive, get_pos,
    //     get_agent_id, mean_info, global_minimap and render answer from it, no copy;
    //   * SPECULATION: the play loop (senario_battle.py:96-168) always continues step -> get_reward / get_alive ->
    //     clear_dead -> get_observation x2.  env_step therefore also enqueues clear_dead, the observation kernel for both
    //     groups and one device->host copy per observation buffer BEHIND the step, and returns as soon as the step's
    //     own results are on the host; the rest runs while the caller is busy with the rewards.  clear_dead then only
    //     commits what already ran, get_observation waits for an event that has normally fired.  Any other call
    //     order (an observation before clear_dead, a second step, add_agents ...) ROLLS BACK: the records k_step left
    //     in the mirror are written back to the device, and the call proceeds as if nothing had been enqueued.
    char *pin = nullptr; int pin_cap = 0;
    struct Mirror { int32_t *pos, *id; uint32_t *state; float *hp, *rew, *lrew; int32_t *head; } mir[2] = {};
    int cur = 0;                   // mir[cur] is the one the getters read (view())
    int32_t *m_actions = nullptr;
    float *m_view = nullptr, *m_feat = nullptr;
    unsigned pending_mask = 0;     // groups whose staged actions have not reached the device yet
    cudaEvent_t ev_step = nullptr, ev_spec = nullptr;

    // What the host holds of the agent records (state) and of both groups' observation rows (obs).  Fresh: they are in
    // mir[cur] / m_view, m_feat.  OnEvent: they will be in mir[cur ^ 1] / m_view, m_feat once ev_spec fires.
    // spec_enqueued: clear_dead + the observations are enqueued behind the last step and not committed yet.
    // Invariant: spec_enqueued implies state == Fresh && obs == Stale.
    enum Held { Stale, Fresh, OnEvent };
    Held state = Stale, obs = Stale;
    bool spec_enqueued = false;

    // The steady play-loop step (set_action x2 + step, then the speculative clear_dead + observe x2 + two copies) is
    // six enqueues, and at one 64 v 64 env the HOST side of those enqueues is what env_step costs.  Once the same
    // sequence has run twice it is captured into a CUDA graph and replayed with one launch; the two events become
    // external event-record nodes.  The key holds every value baked into a graph, so a graph is only replayed while
    // all of them are unchanged, and anything else captures a new one.
    struct GraphKey {
        int into, seq0, seq1, setact_mask;
        const void *pin, *d_view, *d_feat, *d_done, *d_perm;
        BattleParams P; BattleState S;
    };
    struct StepGraph { GraphKey key; cudaGraphExec_t exec; };
    std::vector<StepGraph> graphs;
    int plain_steps = 0;           // eligible steps enqueued call by call so far (the first two warm every attribute up)
    int graph_replays = 0;         // env_step calls served by a graph launch (mfmarl_step_graph_replays)

    // render trace (RenderGenerator.cc): config.json once, then frames appended to video_<file_ct>.txt
    std::string render_dir;
    bool first_render = true;
    int file_ct = 0, frame_ct = 0, frame_per_file = 10000;
    std::vector<int32_t> events;   // (id, x, y) of the last step's attacks, processing order

    ~Game() {
        cudaFree(d_view); cudaFree(d_feat); cudaFree(d_actions); cudaFree(d_perm); cudaFree(d_done); cudaFree(d_events);
        cudaFreeHost(pin);
        if (ev_step) cudaEventDestroy(ev_step);
        if (ev_spec) cudaEventDestroy(ev_spec);
        drop_graphs();
    }

    void drop_graphs() {
        for (StepGraph &sg : graphs) if (sg.exec) cudaGraphExecDestroy(sg.exec);
        graphs.clear();
    }

    const Mirror &view() const { return mir[cur]; }
    StepMirror mirror_io(int which) const {
        const Mirror &m = mir[which];
        return StepMirror{m.pos, m.id, m.state, m.hp, m.rew, m.lrew, m.head};
    }

    // the host's copies no longer describe the device.  Only env_reset gets here with a speculative step still enqueued
    // (every other path rolled it back first), and its placement overwrites what ran.
    void invalidate() { state = Stale; obs = Stale; spec_enqueued = false; }

    // env_step: the step left its records in mir[into]; `enqueued` = clear_dead + observe were enqueued behind it
    void after_step(int into, bool enqueued) { cur = into; state = Fresh; obs = Stale; spec_enqueued = enqueued; }

    // clear_dead right after a step: what was enqueued behind the step becomes the state once ev_spec fires
    void commit_spec() { spec_enqueued = false; state = OnEvent; obs = OnEvent; }

    // something other than clear_dead followed a step: undo the speculative clear_dead (see above)
    void rollback() {
        if (!spec_enqueued) return;
        MF_CUDA(cudaEventSynchronize(ev_spec));
        const Mirror &m = view();                          // the records as the step left them
        engine().restore_state(m.pos, m.id, m.state, m.hp, m.rew, m.lrew, m.head, m.head + 2, st);
        MF_CUDA(cudaStreamSynchronize(st));
        spec_enqueued = false; obs = Stale;
    }

    void ensure_mirror() {
        const int cap = engine().cap(), FS = engine().params().feature_size;
        if (pin_cap >= cap) return;
        std::vector<int32_t> keep(m_actions ? m_actions : nullptr, m_actions ? m_actions + 2 * pin_cap : nullptr);
        const int old_cap = pin_cap;
        if (st) MF_CUDA(cudaStreamSynchronize(st));
        cudaFreeHost(pin);
        const size_t n = (size_t)2 * cap;
        MF_CUDA(cudaMallocHost(&pin, 2 * (n * 4 * 6 + 64) + n * 4 + n * (kViewRow + FS) * 4));
        char *p = pin;
        for (Mirror &m : mir) {
            m.pos = (int32_t *)p; p += n * 4; m.id = (int32_t *)p; p += n * 4; m.state = (uint32_t *)p; p += n * 4;
            m.hp = (float *)p; p += n * 4; m.rew = (float *)p; p += n * 4; m.lrew = (float *)p; p += n * 4;
            m.head = (int32_t *)p; p += 64;
        }
        m_actions = (int32_t *)p; p += n * 4;
        m_view = (float *)p; p += n * kViewRow * 4; m_feat = (float *)p;
        memset(m_actions, 0, n * 4);
        for (int grp = 0; grp < 2 && old_cap > 0; grp++)      // staged actions survive a capacity growth
            memcpy(m_actions + (size_t)grp * cap, keep.data() + (size_t)grp * old_cap, (size_t)old_cap * 4);
        pin_cap = cap;
        cur = 0;
        invalidate();
    }

    // staged set_action calls -> device (one SETACT launch); only needed when something looks at the state before step
    void flush_actions() {
        if (!pending_mask) return;
        Engine &E = engine();
        MF_CUDA(cudaMemcpyAsync(d_actions, m_actions, (size_t)2 * E.cap() * 4, cudaMemcpyHostToDevice, st));
        StepIO io{};
        io.actions = d_actions; io.phases = PH_SETACT; io.setact_mask = (int)pending_mask;
        io.group_seq[0] = io.group_seq[1] = -1;
        E.step(io, st);
        pending_mask = 0;
        invalidate();
    }

    void enqueue_state_download() {
        Engine &E = engine();
        const BattleState &S = E.state();
        const Mirror &m = view();
        const size_t bytes = (size_t)2 * E.cap() * 4;
        MF_CUDA(cudaMemcpyAsync(m.pos, S.pos, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaMemcpyAsync(m.id, S.id, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaMemcpyAsync(m.state, S.state, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaMemcpyAsync(m.hp, S.hp, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaMemcpyAsync(m.rew, S.next_rew, bytes, cudaMemcpyDeviceToHost, st));
    }

    void fetch_state() {
        flush_actions();
        if (state == Fresh) return;
        if (state == OnEvent) {                    // the records after clear_dead were written behind the step
            MF_CUDA(cudaEventSynchronize(ev_spec));
            cur ^= 1;
        } else {
            enqueue_state_download();
            MF_CUDA(cudaStreamSynchronize(st));
        }
        state = Fresh;
    }

    const TypeDef &type_of(int group) const {
        if (group < 0 || group >= (int)groups.size()) throw Fatal("invalid group handle " + std::to_string(group));
        return types.at(groups[group]);
    }

    void check_supported() const {
        if (groups.size() != 2) throw Fatal("the CUDA battle engine supports exactly two groups");
        const TypeDef &a = type_of(0), &b = type_of(1);
        if (groups[0] != groups[1] && memcmp(&a.p, &b.p, sizeof(a.p)) != 0)
            throw Fatal("both groups must use the same agent type attributes");
        if (turn_mode || food_mode || goal_mode) throw Fatal("turn_mode / food_mode / goal_mode are out of scope");
        if (!minimap_mode) throw Fatal("minimap_mode must be on (7-channel battle observation)");
        if (a.width != 1 || a.length != 1) throw Fatal("only 1x1 agent bodies are supported");
        if (a.view_angle != 360.0f || a.attack_angle != 360.0f) throw Fatal("only circular view/attack ranges are supported");
        if (a.attack_in_group || a.can_absorb) throw Fatal("attack_in_group / can_absorb are out of scope");
        if (width <= 0 || height <= 0) throw Fatal("map_width / map_height not configured");
    }

    // reduce the reward DSL to the one shape the battle config uses (RewardEngine.cc:216-240,373-443)
    void attack_bonus(float out[2]) const {
        out[0] = out[1] = 0.0f;
        bool seen[2] = {false, false};
        for (const Rule &r : rules) {
            if (r.on < 0 || r.on >= (int)nodes.size()) throw Fatal("reward rule refers to an undefined event node");
            const Node &n = nodes[r.on];
            bool ok = n.op == 7 /* OP_ATTACK */ && n.inputs.size() == 2 && r.receivers.size() == 1 &&
                      r.receivers[0] == n.inputs[0] && !r.terminal;
            // (auto_value is not looked at: the reference's binding calls add_reward_rule with 6 of its 7 arguments,
            //  gridworld.py:719-722, so the flag is whatever the stack held, and the engine only reads it for OP_ALIGN
            //  nodes, RewardEngine.cc:252)
            if (ok) {
                const Symbol &a = symbols.at(n.inputs[0]), &b = symbols.at(n.inputs[1]);
                ok = a.index == -1 && b.index == -1 && a.group != b.group && a.group >= 0 && a.group < 2 && !seen[a.group];
                if (ok) { out[a.group] = r.values[0]; seen[a.group] = true; }
            }
            if (!ok) throw Fatal("unsupported reward rule: only Event(any(a), 'attack', any(b)) -> receiver a, one per group");
        }
    }

    Engine &engine() {
        if (!eng) throw Fatal("env_reset must be called before this function");
        return *eng;
    }

    void ensure_engine() {
        if (eng) return;
        check_supported();
        EngineConfig c;
        c.n_envs = 1; c.width = width; c.height = height; c.capacity = 64;
        c.embedding_size = embedding_size; c.rng_mode = RNG_MINSTD; c.seed = (unsigned)(seed % 2147483647ul);
        c.type = type_of(0).p;
        attack_bonus(c.attack_bonus);
        eng.reset(new Engine(c));
        if (seed_set) eng->set_seed(seed);
        MF_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        MF_CUDA(cudaEventCreateWithFlags(&ev_step, cudaEventDisableTiming));
        MF_CUDA(cudaEventCreateWithFlags(&ev_spec, cudaEventDisableTiming));
    }

    void ensure_staging() {
        Engine &E = engine();
        if (E.placement_pending()) invalidate();
        E.commit(st);
        const int cap = E.cap();
        if (staged_cap < cap) {
            cudaFree(d_view); cudaFree(d_feat); cudaFree(d_actions); cudaFree(d_perm); cudaFree(d_events);
            MF_CUDA(cudaMalloc(&d_view, (size_t)2 * cap * kViewRow * 4 + 64));
            MF_CUDA(cudaMalloc(&d_feat, (size_t)2 * cap * E.params().feature_size * 4));
            MF_CUDA(cudaMalloc(&d_actions, (size_t)2 * cap * 4));
            MF_CUDA(cudaMalloc(&d_perm, (size_t)2 * cap * 4));
            MF_CUDA(cudaMalloc(&d_events, (size_t)(1 + 6 * cap) * 4));
            MF_CUDA(cudaMemset(d_actions, 0, (size_t)2 * cap * 4));
            staged_cap = cap;
        }
        if (!d_done) MF_CUDA(cudaMalloc(&d_done, 4));
        ensure_mirror();
    }
};

Game *G(EnvHandle h) {
    if (!h) throw Fatal("null game handle");
    return reinterpret_cast<Game *>(h);
}

bool streq(const char *a, const char *b) { return strcmp(a, b) == 0; }

template <typename T>
std::vector<T> pull(const T *dptr, size_t n, cudaStream_t st) {
    std::vector<T> h(n);
    if (n) {
        MF_CUDA(cudaMemcpyAsync(h.data(), dptr, n * sizeof(T), cudaMemcpyDeviceToHost, st));
        MF_CUDA(cudaStreamSynchronize(st));
    }
    return h;
}

}  // namespace

#define API_BEGIN try {
#define API_END(name) } catch (const std::exception &ex) { return report_fatal(name, ex); } return 0;

extern "C" {

int env_new_game(EnvHandle *game, const char *name) {
    API_BEGIN
    if (!streq(name, "GridWorld")) throw Fatal(std::string("invalid name of game: ") + name + " (only GridWorld is built)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw Fatal("no CUDA device visible: this engine has no CPU fallback");
    *game = reinterpret_cast<EnvHandle>(new Game());
    API_END("env_new_game")
}

int env_delete_game(EnvHandle game) {
    API_BEGIN
    Game *g = reinterpret_cast<Game *>(game);
    if (g) { if (g->st) { cudaStreamSynchronize(g->st); } g->eng.reset(); if (g->st) cudaStreamDestroy(g->st); delete g; }
    API_END("env_delete_game")
}

int env_config_game(EnvHandle game, const char *name, void *p_value) {
    API_BEGIN
    Game *g = G(game);
    const int ivalue = *(int *)p_value;
    const bool bvalue = *(bool *)p_value;
    if (streq(name, "map_width")) g->width = ivalue;
    else if (streq(name, "map_height")) g->height = ivalue;
    else if (streq(name, "food_mode")) g->food_mode = bvalue;
    else if (streq(name, "turn_mode")) g->turn_mode = bvalue;
    else if (streq(name, "minimap_mode")) g->minimap_mode = bvalue;
    else if (streq(name, "goal_mode")) g->goal_mode = bvalue;
    else if (streq(name, "embedding_size")) g->embedding_size = ivalue;
    else if (streq(name, "render_dir")) g->render_dir = (const char *)p_value;      // GridWorld.cc:148-149
    else if (streq(name, "seed")) {                       // GridWorld.cc:150-151
        g->seed = (unsigned long)ivalue; g->seed_set = true;
        if (g->eng) g->eng->set_seed(g->seed);
    } else throw Fatal(std::string("invalid argument in GridWorld::set_config : ") + name);
    if (g->eng && !streq(name, "seed") && !streq(name, "render_dir"))
        throw Fatal("game configuration cannot change after the first reset");
    API_END("env_config_game")
}

int env_reset(EnvHandle game) {
    API_BEGIN
    Game *g = G(game);
    g->ensure_engine();
    g->eng->reset();
    g->seq.clear();
    g->pending_mask = 0; g->invalidate();         // (whatever was enqueued behind a step is overwritten by the placement)
    g->file_ct++; g->frame_ct = 0;                        // RenderGenerator::next_file (GridWorld.cc:102)
    API_END("env_reset")
}

int env_get_observation(EnvHandle game, GroupHandle group, float **buffer) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->type_of(group);
    g->rollback();                            // an observation BEFORE clear_dead still lists the dead
    g->ensure_staging();
    g->flush_actions();                       // features carry the last action (GridWorld.cc:411-417)
    const int n = E.host_num(0, group), cap = E.cap(), FS = E.params().feature_size;
    if (n == 0) return 0;
    if (g->obs == Game::OnEvent) {            // both groups' rows were computed and copied behind the last step
        MF_CUDA(cudaEventSynchronize(g->ev_spec));
        g->obs = Game::Fresh;
    }
    if (g->obs != Game::Fresh) {              // both groups in one launch, one batch of copies, one synchronisation
        const int n0 = E.host_num(0, 0), n1 = E.host_num(0, 1);
        E.observe(g->d_view, g->d_feat, (n0 > 0 ? 1 : 0) | (n1 > 0 ? 2 : 0), g->st);
        for (int grp = 0; grp < 2; grp++) {
            const int ng = grp ? n1 : n0;
            if (ng == 0) continue;
            MF_CUDA(cudaMemcpyAsync(g->m_view + (size_t)grp * cap * kViewRow, g->d_view + (size_t)grp * cap * kViewRow,
                                    (size_t)ng * kViewRow * 4, cudaMemcpyDeviceToHost, g->st));
            MF_CUDA(cudaMemcpyAsync(g->m_feat + (size_t)grp * cap * FS, g->d_feat + (size_t)grp * cap * FS,
                                    (size_t)ng * FS * 4, cudaMemcpyDeviceToHost, g->st));
        }
        MF_CUDA(cudaStreamSynchronize(g->st));
        g->obs = Game::Fresh;
    }
    memcpy(buffer[0], g->m_view + (size_t)group * cap * kViewRow, (size_t)n * kViewRow * 4);
    memcpy(buffer[1], g->m_feat + (size_t)group * cap * FS, (size_t)n * FS * 4);
    API_END("env_get_observation")
}

int env_set_action(EnvHandle game, GroupHandle group, const int *actions) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->type_of(group);
    g->rollback();
    g->ensure_staging();
    for (int s : g->seq)
        if (s == group) throw Fatal("set_action called twice for one group before step");
    const int n = E.host_num(0, group);
    if (n > 0) memcpy(g->m_actions + (size_t)group * E.cap(), actions, (size_t)n * 4);   // staged; applied by env_step
    g->pending_mask |= 1u << group;
    g->seq.push_back(group);
    g->invalidate();                          // last_action changes (features, mean_info)
    API_END("env_set_action")
}

int env_step(EnvHandle game, int *done) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->rollback();                            // a second step without clear_dead keeps the dead in the lists
    g->ensure_staging();
    const int cap = E.cap();
    const int into = g->cur ^ 1;              // the step's records go to the mirror the getters are not reading
    StepIO io{};
    io.phases = PH_STEP; io.done = g->d_done; io.attack_perm = g->d_perm;
    io.group_seq[0] = g->seq.size() > 0 ? g->seq[0] : -1;
    io.group_seq[1] = g->seq.size() > 1 ? g->seq[1] : -1;
    io.mirror = g->mirror_io(into);
    if (g->pending_mask) {                    // set_action(g0), set_action(g1) and step in one launch; the kernel reads
        io.actions = g->m_actions;            // the staged actions from the mapped pinned buffer itself
        io.phases |= PH_SETACT; io.setact_mask = (int)g->pending_mask;
        g->pending_mask = 0;
    }
    if (g->inject_next) E.set_rng_mode(RNG_INJECT);
    const bool want_events = !g->first_render;            // GridWorld.cc:533,559: recorded once a frame was rendered
    if (want_events) io.attack_events = g->d_events;
    // what the play loop asks for next is enqueued behind the step: clear_dead (its records into the OTHER mirror),
    // both groups' observations, one copy per observation buffer
    auto enqueue = [&](bool with_spec, unsigned event_flags) {
        E.step(io, g->st);
        MF_CUDA(cudaEventRecordWithFlags(g->ev_step, g->st, event_flags));
        if (!with_spec) return;
        StepIO c{};
        c.phases = PH_CLEAR; c.group_seq[0] = c.group_seq[1] = -1; c.mirror = g->mirror_io(g->cur);
        E.step(c, g->st);
        E.observe(g->d_view, g->d_feat, 3, g->st);
        const int FS = E.params().feature_size;
        MF_CUDA(cudaMemcpyAsync(g->m_view, g->d_view, (size_t)2 * cap * kViewRow * 4, cudaMemcpyDeviceToHost, g->st));
        MF_CUDA(cudaMemcpyAsync(g->m_feat, g->d_feat, (size_t)2 * cap * FS * 4, cudaMemcpyDeviceToHost, g->st));
        MF_CUDA(cudaEventRecordWithFlags(g->ev_spec, g->st, event_flags));
    };
    const bool with_spec = !want_events;
    const bool graphable = with_spec && !g->inject_next && io.phases == (PH_STEP | PH_SETACT);
    if (graphable && g->plain_steps >= 2) {
        Game::GraphKey key;
        memset(&key, 0, sizeof(key));         // memcmp compares the padding too
        key.into = into; key.seq0 = io.group_seq[0]; key.seq1 = io.group_seq[1]; key.setact_mask = io.setact_mask;
        key.pin = g->pin; key.d_view = g->d_view; key.d_feat = g->d_feat; key.d_done = g->d_done; key.d_perm = g->d_perm;
        memcpy(&key.P, &E.params(), sizeof(BattleParams)); memcpy(&key.S, &E.state(), sizeof(BattleState));
        const Game::StepGraph *hit = nullptr;
        for (const Game::StepGraph &sg : g->graphs)
            if (memcmp(&sg.key, &key, sizeof(key)) == 0) hit = &sg;
        if (!hit) {
            if (g->graphs.size() >= 8) g->drop_graphs();
            cudaGraph_t graph = nullptr;
            MF_CUDA(cudaStreamBeginCapture(g->st, cudaStreamCaptureModeThreadLocal));
            try { enqueue(true, cudaEventRecordExternal); }
            catch (...) { cudaStreamEndCapture(g->st, &graph); if (graph) cudaGraphDestroy(graph); throw; }
            MF_CUDA(cudaStreamEndCapture(g->st, &graph));
            cudaGraphExec_t exec = nullptr;
            const cudaError_t err = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (err != cudaSuccess) throw Fatal(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(err));
            g->graphs.push_back({key, exec});
            hit = &g->graphs.back();
        }
        MF_CUDA(cudaGraphLaunch(hit->exec, g->st));
        E.mark_stepped();                     // (Engine::step did not run on the host this time)
        g->graph_replays++;
    } else {
        enqueue(with_spec, cudaEventRecordDefault);
        if (graphable) g->plain_steps++;
    }
    if (g->inject_next) { E.set_rng_mode(RNG_MINSTD); g->inject_next = false; }
    if (want_events) {
        const std::vector<int32_t> raw = pull(g->d_events, (size_t)1 + 6 * cap, g->st);
        g->events.clear();
        for (int i = 0; i < raw[0]; i++)
            if (raw[1 + 3 * i] >= 0) g->events.insert(g->events.end(), raw.begin() + 1 + 3 * i, raw.begin() + 4 + 3 * i);
    }
    MF_CUDA(cudaEventSynchronize(g->ev_step));            // rewards, alive flags, positions, done: in the mirror now
    g->after_step(into, with_spec);
    *done = g->view().head[4];
    g->seq.clear();
    API_END("env_step")
}

int env_get_reward(EnvHandle game, GroupHandle group, float *buffer) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->type_of(group);
    g->ensure_staging();
    const int n = E.host_num(0, group);
    g->fetch_state();
    const float *rew = g->view().rew + (size_t)group * E.cap();
    for (int i = 0; i < n; i++) buffer[i] = rew[i] + 0.0f;   // + Group::get_reward(), always 0 (GridWorld.cc:764-768)
    API_END("env_get_reward")
}

int env_get_info(EnvHandle game, GroupHandle group, const char *name, void *void_buffer) {
    API_BEGIN
    Game *g = G(game);
    int *ibuf = (int *)void_buffer;
    float *fbuf = (float *)void_buffer;
    bool *bbuf = (bool *)void_buffer;

    // ---- answers that do not need the engine (callable before reset, like the reference) ----
    if (streq(name, "action_space") || streq(name, "view_space") || streq(name, "feature_space") ||
        streq(name, "attack_base") || streq(name, "view2attack")) {
        const TypeDef &t = g->type_of(group);
        const CircleRange view(t.p.view_radius, 0.0f, t.width % 2), attack(t.p.attack_radius, t.width / 2.0f, t.width % 2),
            move(t.p.speed, 0.0f, 1);
        const int n_action = move.count + attack.count;
        if (streq(name, "action_space")) ibuf[0] = n_action;
        else if (streq(name, "view_space")) {              // GridWorld.cc:929-934
            ibuf[0] = view.width; ibuf[1] = view.width;
            ibuf[2] = 1 + (g->food_mode ? 1 : 0) + (int)g->groups.size() * (g->minimap_mode ? 3 : 2);
        } else if (streq(name, "feature_space"))           // GridWorld.cc:1010-1018
            ibuf[0] = g->embedding_size + n_action + 1 + (g->goal_mode ? 2 : 0) + (g->minimap_mode ? 2 : 0);
        else if (streq(name, "attack_base")) ibuf[0] = move.count;
        else {                                             // view2attack, GridWorld.cc:937-954
            for (int i = 0; i < view.width * view.width; i++) ibuf[i] = -1;
            for (int i = 0; i < attack.count; i++)
                ibuf[(attack.dy[i] + view.center) * view.width + attack.dx[i] + view.center] = i;
        }
        return 0;
    }
    if (streq(name, "groups_info")) {                      // GridWorld.cc:957-972
        static const int colors[4][3] = {{192, 64, 64}, {64, 64, 192}, {64, 192, 64}, {64, 64, 64}};
        for (size_t i = 0; i < g->groups.size(); i++) {
            const TypeDef &t = g->type_of((int)i);
            ibuf[5 * i] = t.width; ibuf[5 * i + 1] = t.length;
            for (int k = 0; k < 3; k++) ibuf[5 * i + 2 + k] = colors[i % 4][k];
        }
        return 0;
    }
    if (streq(name, "both_attack")) { ibuf[0] = 0; return 0; }

    Engine &E = g->engine();
    g->ensure_staging();
    const int cap = E.cap();
    const BattleState &S = E.state();

    if (streq(name, "walls_info")) {                       // GridWorld.cc:871-880
        const std::vector<unsigned char> &w = E.host_walls();
        int ct = 0;
        for (size_t i = 0; i < w.size(); i++)
            if (w[i]) { ct++; ibuf[2 * ct] = (int)(i % E.params().W); ibuf[2 * ct + 1] = (int)(i / E.params().W); }
        ibuf[0] = ct;
        return 0;
    }
    if (streq(name, "global_minimap")) {                   // GridWorld.cc:811-846
        const int vh = (int)lroundf(fbuf[0]), vw = (int)lroundf(fbuf[1]);
        const int ng = 2;
        memset(fbuf, 0, sizeof(float) * vh * vw * ng);
        const int scale_h = (E.params().H + vh - 1) / vh, scale_w = (E.params().W + vw - 1) / vw;
        for (int i = 0; i < ng; i++) {
            const int channel = ((i - group + ng) % ng + ng) % ng;
            const int n = E.host_num(0, i);
            g->fetch_state();
            const int32_t *pos = g->view().pos + (size_t)i * cap;
            for (int j = 0; j < n; j++)
                fbuf[(((pos[j] >> 16) & 0xFFFF) / scale_h * vw + (pos[j] & 0xFFFF) / scale_w) * ng + channel] += 1.0f;
            for (int k = 0; k < vh * vw; k++) fbuf[k * ng + channel] /= (size_t)n;
        }
        return 0;
    }

    g->type_of(group);
    const int n = E.host_num(0, group);
    if (streq(name, "num")) {
        ibuf[0] = n;
    } else if (streq(name, "id")) {
        g->fetch_state();
        memcpy(ibuf, g->view().id + (size_t)group * cap, (size_t)n * 4);
    } else if (streq(name, "pos")) {
        g->fetch_state();
        const int32_t *pos = g->view().pos + (size_t)group * cap;
        for (int i = 0; i < n; i++) { ibuf[2 * i] = pos[i] & 0xFFFF; ibuf[2 * i + 1] = (pos[i] >> 16) & 0xFFFF; }
    } else if (streq(name, "alive")) {
        g->fetch_state();
        const uint32_t *st = g->view().state + (size_t)group * cap;
        for (int i = 0; i < n; i++) bbuf[i] = !(st[i] & 1u);
    } else if (streq(name, "mean_info")) {                 // GridWorld.cc:849-870
        g->fetch_state();
        const int32_t *pos = g->view().pos + (size_t)group * cap;
        const uint32_t *st = g->view().state + (size_t)group * cap;
        const int n_action = E.n_action();
        std::vector<int> counter(n_action + 1, 0);
        float sum_x = 0, sum_y = 0;
        for (int i = 0; i < n; i++) {
            sum_x += (float)(pos[i] & 0xFFFF); sum_y += (float)((pos[i] >> 16) & 0xFFFF);
            counter[std::min<int>((st[i] >> 16) & 0xFF, n_action)]++;
        }
        const size_t an = (size_t)n;
        fbuf[0] = sum_x / an; fbuf[1] = sum_y / an;
        for (int i = 0; i < n_action; i++) fbuf[2 + i] = (float)(1.0 * counter[i] / an);
    } else {
        throw Fatal(std::string("unsupported info name in GridWorld::get_info : ") + name);
    }
    API_END("env_get_info")
}

// The on-disk trace of RenderGenerator.cc:57-185, byte for byte: <dir>/config.json at the first call, then one frame
// per call appended to <dir>/video_<n>.txt -- "W n" + wall cells before the first frame of a file, "F agents attacks 0",
// one "id hp dir x y group" line per agent still in the lists (dead ones included until clear_dead, hp as an integer
// percentage clamped to [0, 100], dir = dir2angle[NORTH] = 270), one "0 id x y" line per attack of the last step.
int env_render(EnvHandle game) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->ensure_staging();
    const TypeDef &t0 = g->type_of(0);
    if (g->first_render) {
        g->first_render = false;
        if (!g->render_dir.empty()) {
            std::ofstream f(g->render_dir + "/config.json");
            const int colors[4][3] = {{192, 64, 64}, {64, 64, 192}, {64, 192, 64}, {64, 64, 64}};
            auto rgba = [](int r, int gr, int b, float alpha) {
                std::stringstream ss;
                ss << "\"rgba(" << r << "," << gr << "," << b << "," << alpha << ")\"";
                return ss.str();
            };
            auto kv = [&f](const char *key, const std::string &value, bool last = false) {
                f << "\"" << key << "\": " << value << (last ? "" : ",") << std::endl;
            };
            auto num = [](float v) { std::stringstream ss; ss << v; return ss.str(); };
            f << "{" << std::endl;
            kv("width", std::to_string(g->width)); kv("height", std::to_string(g->height));
            kv("static-file", "\"static.map\""); kv("obstacle-style", rgba(127, 127, 127, 1));
            kv("dynamic-file-directory", "\".\""); kv("attack-style", rgba(63, 63, 63, 0.8f));
            kv("minimap-width", "300"); kv("minimap-height", "250");
            f << "\"group\" : [" << std::endl;
            for (size_t i = 0; i < g->groups.size(); i++) {
                const TypeDef &t = g->type_of((int)i);
                const int *c = colors[i % 4];
                f << "{" << std::endl;
                kv("height", std::to_string(t.length)); kv("width", std::to_string(t.width));
                kv("style", rgba(c[0], c[1], c[2], 1)); kv("anchor", "[0, 0]");
                kv("max-speed", std::to_string((int)t.p.speed)); kv("speed-style", rgba(c[0], c[1], c[2], 0.01f));
                kv("vision-radius", num(t.p.view_radius)); kv("vision-angle", num(t.view_angle));
                kv("vision-style", rgba(c[0], c[1], c[2], 0.2f));
                kv("attack-radius", num(t.p.attack_radius)); kv("attack-angle", num(t.attack_angle));
                kv("attack-style", rgba(c[0], c[1], c[2], 0.1f)); kv("broadcast-radius", "1", true);
                f << (i + 1 == g->groups.size() ? "}" : "},") << std::endl;
            }
            f << "]" << std::endl << "}" << std::endl;
        }
    }
    if (g->render_dir.empty()) return 0;
    std::ofstream out(g->render_dir + "/video_" + std::to_string(g->file_ct) + ".txt",
                      g->frame_ct == 0 ? std::ios::out : std::ios::app);
    if (g->frame_ct == 0) {
        const std::vector<unsigned char> &w = E.host_walls();
        out << "W " << std::count_if(w.begin(), w.end(), [](unsigned char c) { return c != 0; }) << std::endl;
        for (int i = 0; i < g->width * g->height; i++)
            if (w[i]) out << i % g->width << " " << i / g->width << std::endl;
    }
    const BattleState &S = E.state();
    const int cap = E.cap();
    const int n0 = E.host_num(0, 0), n1 = E.host_num(0, 1);
    out << "F " << n0 + n1 << " " << g->events.size() / 3 << " " << 0 << std::endl;
    for (int grp = 0; grp < 2; grp++) {
        const int n = grp ? n1 : n0;
        g->fetch_state();
        const int32_t *pos = g->view().pos + (size_t)grp * cap, *id = g->view().id + (size_t)grp * cap;
        const float *hp = g->view().hp + (size_t)grp * cap;
        for (int j = 0; j < n; j++) {
            const int pct = std::min(100, std::max(0, (int)(100 * hp[j] / t0.p.hp)));
            out << id[j] << " " << pct << " " << 270 /* NORTH: turn_mode is off, GridWorld.cc:264 */ << " " << (pos[j] & 0xFFFF) << " " << (pos[j] >> 16) << " " << grp << std::endl;
        }
    }
    for (size_t i = 0; i + 2 < g->events.size(); i += 3)
        out << 0 << " " << g->events[i] << " " << g->events[i + 1] << " " << g->events[i + 2] << std::endl;
    if (g->frame_ct++ > g->frame_per_file) { g->frame_ct = 0; g->file_ct++; }
    API_END("env_render")
}

int env_render_next_file(EnvHandle game) {
    API_BEGIN
    Game *g = G(game);
    g->file_ct++; g->frame_ct = 0;
    API_END("env_render_next_file")
}

int gridworld_register_agent_type(EnvHandle game, const char *name, int n, const char **keys, float *values) {
    API_BEGIN
    Game *g = G(game);
    if (g->types.count(name)) throw Fatal(std::string("duplicated name of agent type in GridWorld::register_agent_type : ") + name);
    TypeDef t;
    for (int i = 0; i < n; i++) {
        const char *k = keys[i]; const float v = values[i];
        auto as_int = [&](float x) { return (int)(x + 0.5f); };
        if (streq(k, "width")) t.width = as_int(v);
        else if (streq(k, "length")) t.length = as_int(v);
        else if (streq(k, "speed")) t.p.speed = v;
        else if (streq(k, "hp")) t.p.hp = v;
        else if (streq(k, "view_radius")) t.p.view_radius = v;
        else if (streq(k, "view_angle")) t.view_angle = v;
        else if (streq(k, "attack_radius")) t.p.attack_radius = v;
        else if (streq(k, "attack_angle")) t.attack_angle = v;
        else if (streq(k, "damage")) t.p.damage = v;
        else if (streq(k, "step_recover")) t.p.step_recover = v;
        else if (streq(k, "kill_supply")) t.p.kill_supply = v;
        else if (streq(k, "step_reward")) t.p.step_reward = v;
        else if (streq(k, "kill_reward")) t.p.kill_reward = v;
        else if (streq(k, "dead_penalty")) t.p.dead_penalty = v;
        else if (streq(k, "attack_penalty")) t.p.attack_penalty = v;
        else if (streq(k, "attack_in_group")) t.attack_in_group = as_int(v) != 0;
        else if (streq(k, "can_absorb")) t.can_absorb = as_int(v) != 0;
        else if (streq(k, "hear_radius") || streq(k, "speak_radius") || streq(k, "speak_ability") ||
                 streq(k, "trace") || streq(k, "eat_ability") || streq(k, "food_supply") ||
                 streq(k, "view_x_offset") || streq(k, "view_y_offset") || streq(k, "att_x_offset") ||
                 streq(k, "att_y_offset") || streq(k, "turn_x_offset") || streq(k, "turn_y_offset")) {
            /* accepted, no effect on the battle path (offsets are recomputed, AgentType.cc:115-118) */
        } else throw Fatal(std::string("invalid agent config in AgentType::AgentType : ") + k);
    }
    g->types.emplace(name, t);
    API_END("gridworld_register_agent_type")
}

int gridworld_new_group(EnvHandle game, const char *agent_type_name, GroupHandle *group) {
    API_BEGIN
    Game *g = G(game);
    if (!g->types.count(agent_type_name)) throw Fatal(std::string("invalid name of agent type in new_group : ") + agent_type_name);
    if (g->eng) throw Fatal("groups cannot be added after the first reset");
    *group = (GroupHandle)g->groups.size();
    g->groups.push_back(agent_type_name);
    API_END("gridworld_new_group")
}

int gridworld_add_agents(EnvHandle game, GroupHandle group, int n, const char *method,
                         const int *pos_x, const int *pos_y, const int *dir) {
    API_BEGIN
    (void)dir;   // no turn_mode: every agent faces NORTH (GridWorld.cc:264)
    Game *g = G(game);
    Engine &E = g->engine();
    g->rollback();
    std::vector<int> xs, ys;
    if (streq(method, "custom")) {
        xs.assign(pos_x, pos_x + n); ys.assign(pos_y, pos_y + n);
    } else if (streq(method, "fill")) {                    // GridWorld.cc:212-223,270-296: xs = {x, y, width, height(, dir)}
        for (int x = pos_x[0]; x < pos_x[0] + pos_x[2]; x++)
            for (int y = pos_x[1]; y < pos_x[1] + pos_x[3]; y++) { xs.push_back(x); ys.push_back(y); }
    } else if (streq(method, "random")) {                  // GridWorld.cc:194-202,236-255 + Map::get_random_blank Map.cc:49-63
        uint32_t rs = E.pull_rng0();
        const int W = E.params().W, H = E.params().H;
        for (int i = 0; i < n; i++) {
            int tries = 0;
            while (true) {
                rs = (uint32_t)(((uint64_t)rs * 16807ull) % 2147483647ull); const int x = (int)rs % (W - 1);
                rs = (uint32_t)(((uint64_t)rs * 16807ull) % 2147483647ull); const int y = (int)rs % (H - 1);
                if (E.cell_blank_for_placement(x, y)) {
                    if (group == -1) E.add_walls(1, &x, &y); else E.add_agents(group, 1, &x, &y);
                    break;
                }
                if (tries++ > W * H) throw Fatal("cannot find a blank position in a filled map");
            }
        }
        E.push_rng0(rs);
        if (group != -1) { E.commit(g->st); }
        g->invalidate();                      // the host mirror predates the new agents
        return 0;
    } else throw Fatal(std::string("unsupported method in GridWorld::add_agents : ") + method);

    if (group == -1) E.add_walls((int)xs.size(), xs.data(), ys.data());
    else { g->type_of(group); E.add_agents(group, (int)xs.size(), xs.data(), ys.data()); }
    g->invalidate();                          // rows of the new agents are not in the host mirror yet (also after a late add)
    API_END("gridworld_add_agents")
}

int gridworld_clear_dead(EnvHandle game) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->ensure_staging();
    StepIO io{};
    g->fetch_state();                         // (already on the host after env_step: no synchronisation)
    // the survivors' count follows from the alive flags the host already holds, so the compaction kernel is only
    // enqueued -- it runs back to back with whatever comes next (normally the observation kernel)
    for (int grp = 0; grp < 2; grp++) {
        const int n = E.host_num(0, grp);
        const uint32_t *st = g->view().state + (size_t)grp * E.cap();
        int alive = 0;
        for (int i = 0; i < n; i++) alive += !(st[i] & 1u);
        E.set_host_num(0, grp, alive);
    }
    if (g->spec_enqueued) {                   // it already ran behind the step: commit
        g->commit_spec();
        return 0;
    }
    io.phases = PH_CLEAR; io.group_seq[0] = io.group_seq[1] = -1;
    E.step(io, g->st);
    g->invalidate();
    API_END("gridworld_clear_dead")
}

int gridworld_set_goal(EnvHandle, GroupHandle, const char *, const int *) {
    API_BEGIN
    throw Fatal("gridworld_set_goal is deprecated in the reference and out of scope here");
    API_END("gridworld_set_goal")
}

int gridworld_define_agent_symbol(EnvHandle game, int no, int group, int index) {
    API_BEGIN
    Game *g = G(game);
    if (no < 0) throw Fatal("negative symbol number");
    if (no >= (int)g->symbols.size()) g->symbols.resize(no + 1);
    g->symbols[no].group = group; g->symbols[no].index = index;
    API_END("gridworld_define_agent_symbol")
}

int gridworld_define_event_node(EnvHandle game, int no, int op, int *inputs, int n_inputs) {
    API_BEGIN
    Game *g = G(game);
    if (no < 0) throw Fatal("negative event node number");
    if (no >= (int)g->nodes.size()) g->nodes.resize(no + 1);
    g->nodes[no].op = op;
    g->nodes[no].inputs.assign(inputs, inputs + n_inputs);
    API_END("gridworld_define_event_node")
}

int gridworld_add_reward_rule(EnvHandle game, int on, int *receiver, float *value, int n_receiver,
                              bool is_terminal, bool auto_value) {
    API_BEGIN
    Game *g = G(game);
    Rule r;
    r.on = on; r.receivers.assign(receiver, receiver + n_receiver); r.values.assign(value, value + n_receiver);
    r.terminal = is_terminal; r.auto_value = auto_value;
    g->rules.push_back(r);
    API_END("gridworld_add_reward_rule")
}

// ---- test hook (not in the reference ABI): the next env_step resolves attacks in the given order ----
int mfmarl_inject_attack_order(EnvHandle game, const int *perm, int n) {
    API_BEGIN
    Game *g = G(game);
    Engine &E = g->engine();
    g->ensure_staging();
    if (n > 2 * E.cap()) throw Fatal("attack order longer than the agent capacity");
    if (n > 0) MF_CUDA(cudaMemcpyAsync(g->d_perm, perm, (size_t)n * 4, cudaMemcpyHostToDevice, g->st));
    MF_CUDA(cudaStreamSynchronize(g->st));
    g->inject_next = true;
    API_END("mfmarl_inject_attack_order")
}

int mfmarl_step_graph_replays(EnvHandle game) { return game ? reinterpret_cast<Game *>(game)->graph_replays : -1; }

const char *mfmarl_last_error(void) { return last_error(); }

}  // extern "C"
