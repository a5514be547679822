/* mfmarl_magent.h -- the reference-facing C ABI of the B200 battle engine.
 *
 * Every entry point below replaces, symbol for symbol and argument for argument, the function of the
 * same name that the reference exports from libmagent.so and that its Python binding calls through
 * ctypes (python/magent/c_lib.py:13-30, python/magent/gridworld.py).  Reference declarations:
 * examples/battle_model/src/runtime_api.h:20-55; implementations: runtime_api.cc:15-169.
 *
 * Contract (identical to the reference unless noted):
 *   - one EnvHandle = one game; not re-entrant per handle; single caller thread
 *   - every data buffer is caller-owned HOST memory, sized by the caller from env_get_info("num")
 *   - every function returns 0; fatal conditions print a message and abort() -- the reference throws
 *     std::runtime_error through the C boundary (utility.h:77-81), which also terminates the caller.
 *     With MAGENT_ERRORS=return in the environment they return -1 instead and the message is
 *     available from mfmarl_last_error().
 *   - there is NO CPU fallback: without a CUDA device env_new_game fails.
 * Scope: the battle path.  discrete_snake_* and the *_infer_action boosters of runtime_api.h:57-72 are
 * not on the path and are not exported.
 */
#ifndef MFMARL_MAGENT_H
#define MFMARL_MAGENT_H

#include <stdbool.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *EnvHandle;   /* reference: Environment*  (Environment.h:36) */
typedef int GroupHandle;   /* reference: Environment.h:12 */

/* ---- general environment ------------------------------------------------- reference runtime_api.h */
int env_new_game(EnvHandle *game, const char *name);                               /* :21, .cc:15-32  */
int env_delete_game(EnvHandle game);                                               /* :22, .cc:34-38  */
int env_config_game(EnvHandle game, const char *name, void *p_value);              /* :23, .cc:40-44  */
int env_reset(EnvHandle game);                                                     /* :26, .cc:47-51  */
/* buffer[0] = float[n][13][13][7] views, buffer[1] = float[n][34] features                           */
int env_get_observation(EnvHandle game, GroupHandle group, float **buffer);        /* :27, .cc:53-57  */
int env_set_action(EnvHandle game, GroupHandle group, const int *actions);         /* :28, .cc:59-63  */
int env_step(EnvHandle game, int *done);                                           /* :29, .cc:65-69  */
int env_get_reward(EnvHandle game, GroupHandle group, float *buffer);              /* :30, .cc:71-75  */
/* keys: num id pos alive action_space view_space feature_space mean_info view2attack attack_base
 *       global_minimap walls_info groups_info both_attack          (GridWorld.cc:777-978)            */
int env_get_info(EnvHandle game, GroupHandle group, const char *name, void *buffer); /* :33, .cc:78-82 */
int env_render(EnvHandle game);            /* no-op: rendering is out of scope */  /* :36, .cc:85-89  */
int env_render_next_file(EnvHandle game);  /* no-op */                             /* :37, .cc:91-96  */

/* ---- gridworld special --------------------------------------------------------------------------- */
int gridworld_register_agent_type(EnvHandle game, const char *name, int n,
                                  const char **keys, float *values);               /* :43, .cc:102-107 */
int gridworld_new_group(EnvHandle game, const char *agent_type_name, GroupHandle *group); /* :44, .cc:109-113 */
/* method: "custom" (pos_x/pos_y/dir arrays of n), "fill" (pos_x = {x, y, w, h, dir}), "random" (n);
 * group -1 adds walls                                                                                */
int gridworld_add_agents(EnvHandle game, GroupHandle group, int n, const char *method,
                         const int *pos_x, const int *pos_y, const int *dir);      /* :45, .cc:115-120 */
int gridworld_clear_dead(EnvHandle game);                                          /* :49, .cc:123-127 */
int gridworld_set_goal(EnvHandle game, GroupHandle group, const char *method,
                       const int *linear_buffer);  /* deprecated upstream: fatal */ /* :50, .cc:129-133 */
int gridworld_define_agent_symbol(EnvHandle game, int no, int group, int index);   /* :53, .cc:136-140 */
int gridworld_define_event_node(EnvHandle game, int no, int op, int *inputs, int n_inputs); /* :54, .cc:142-146 */
int gridworld_add_reward_rule(EnvHandle game, int on, int *receiver, float *value, int n_receiver,
                              bool is_terminal, bool auto_value);                  /* :55, .cc:148-153 */

/* ---- additions (not in the reference) ------------------------------------------------------------ */
/* Test hook: the next env_step resolves its attacks in the order perm[0..n) (indices into the attack
 * list in set_action call order) instead of shuffling with the engine RNG (GridWorld.cc:510-515).    */
int mfmarl_inject_attack_order(EnvHandle game, const int *perm, int n);
/* Test hook: how many env_step calls of this game were served by replaying the captured CUDA graph of the steady
 * play-loop step; -1 for a null handle.                                                                           */
int mfmarl_step_graph_replays(EnvHandle game);
const char *mfmarl_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* MFMARL_MAGENT_H */
