/* ql_cuda_nstep.h — n-step returns and double-DQN targets on the device: the companion of ql_cuda.h for the Rainbow-style
 * targets of the device learner. Same ABI rules as ql_cuda.h (status codes, qlc_last_error_string, QLC_VERSION). Stream order:
 * both calls are asynchronous on `stream` and follow ql_cuda.h's rule for its asynchronous calls: queued after the submitted host
 * steps of the env, with the env's time read when they are queued, so after qlc_env_step on the same stream they see that step. */
#ifndef QL_CUDA_NSTEP_H
#define QL_CUDA_NSTEP_H

#include "ql_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- n-step returns and double-DQN targets read straight from the replay ring (DESIGN.md §14). Transition i (logical index)
 * is followed in its env by i + n_envs. The walk from i takes records j = 0, 1, ... and stops at the first j where the record is
 * done (terminal) or truncated, j = n_step - 1, j is the newest time in the replay, or the next record starts an episode (a
 * reset by the caller). With m = j + 1 records: G = sum gamma^j r_j (f32, in order), disc = gamma^m (0 where terminal), and the
 * bootstrap state is state_next of boot = i + (m - 1) n_envs. The target is y = G where terminal, else G + Q_boot * disc, with
 * Q_boot = max_a Q_target(boot), or with double DQN Q_target(boot)[argmax_a Q_online(boot)]. Deterministic. ---- */
#define QLC_NSTEP_MAX 64
/* n-step returns of replay transitions idx_dev [n] (logical indices): return_dev [n] f32 = G, discount_dev [n] f32 = disc
 * (0 where terminal), boot_idx_dev [n] u32 = the logical index whose state_next bootstraps (any output may be NULL).
 * 1 <= n_step <= QLC_NSTEP_MAX, 0 <= gamma <= 1. An index >= len gives 0, 0 and the index itself. Asynchronous on `stream`. */
int32_t qlc_replay_nstep(qlc_env* env, const uint32_t* idx_dev, uint32_t n, uint32_t n_step, float gamma,
                         float* return_dev, float* discount_dev, uint32_t* boot_idx_dev, void* stream);
/* qlc_qnet_train_weighted with n-step / double-DQN targets from target_net (required, same env); y_dev [n_batches][batch]
 * (may be NULL) receives the target each item was trained on. n_step = 1, double_dqn = 0 is qlc_qnet_train_weighted's
 * arithmetic bit for bit. The target network is evaluated once per call; with double_dqn = 1 the online network's greedy
 * action for minibatch j comes from the weights after updates 0 .. j-1, so n_batches = k calls give the bits of k calls. */
int32_t qlc_qnet_train_nstep(qlc_qnet* qnet, const uint32_t* idx_dev, const float* weight_dev, uint32_t batch, uint32_t n_batches,
                             qlc_qnet* target_net, float gamma, uint32_t n_step, int32_t double_dqn,
                             float* loss_dev, float* td_dev, float* y_dev, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* QL_CUDA_NSTEP_H */
