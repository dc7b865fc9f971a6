/*
 * boatenv.h -- C ABI of libboatenv.so: the B200-native (sm_100a) batched
 * implementation of the environment-step hot path of Nilau1998/SAC-Agent.
 *
 * The reference has no FFI layer: its boundary is the duck-typed Python object that
 * main.py, Recorder and BaseAgent touch (SURVEY.md section 8b).  Every entry point
 * below names the reference interface (file:line, relative to the reference root)
 * whose batched generalisation it is.  The reference-side binding (a ctypes stub)
 * is shown in INTEGRATION.md; sac-agent_b200/_lib.py is the binding this repo ships.
 *
 * Conventions
 *   - plain C types only; every tensor argument is a caller-owned DEVICE pointer
 *     (e.g. torch.Tensor.data_ptr()) unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - return value: 0 = OK, negative = argument / configuration error (below),
 *     positive = cudaError_t of the failing CUDA call;
 *   - a handle is bound to one device, is not thread-safe, one handle per GPU;
 *   - there is no CPU fallback: every compute entry point launches sm_100a kernels.
 *   - `precision` is 32 (production: fp32 state/obs, float actions) or 64
 *     (validation: fp64 in the reference's operation order, double actions).
 *     Element type T below means float or double accordingly.  In the 32-bit mode everything a termination
 *     threshold is applied to after accumulation is carried exactly in the same state bytes: the rudder angle
 *     (boat_env.py:72-73, :102-108) as a 44-bit fixed-point number (2^-42 rad), s_x / s_y (:85-93) as int32 fixed
 *     point; get/set_field and env_state_host exchange plain numbers.  Actions are clamped to +-64 before the
 *     rudder update (no outcome changes: |action| >= 21 breaks the rudder from any unbroken state).
 */
#ifndef BOATENV_H
#define BOATENV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define BOATENV_API __attribute__((visibility("default")))
#else
#define BOATENV_API
#endif

#define BOATENV_OK 0
#define BOATENV_EINVAL (-1)        /* NULL / out-of-range argument                          */
#define BOATENV_EEXPERIMENT (-2)   /* unknown experiment: the ValueError of wind.py:65-67   */
#define BOATENV_EFIXEDPOINTS (-3)  /* fixed_points < 4: the ValueError of wind.py:73-75     */
#define BOATENV_EUNSUPPORTED (-4)  /* valid for the reference, not for this build (e.g.
                                      fixed_points > 16, t_max/dt > 2^20 - 64)             */
#define BOATENV_ENODEVICE (-5)     /* no CUDA device / not an sm_100 device                 */
#define BOATENV_ESTATE (-6)        /* step() before reset()                                 */
#define BOATENV_EALIGN (-7)        /* a tensor pointer is not 16-byte aligned               */

#define BOATENV_OBS_DIM 11         /* boat_env.py:308-323 return_state                      */

/* Termination codes written to term_out (boat_env.py:84-105, cascade order). */
#define BOATENV_TERM_NONE 0
#define BOATENV_TERM_REACHED_GOAL 1
#define BOATENV_TERM_OUT_OF_BOUNDS 2
#define BOATENV_TERM_OUT_OF_FUEL 3
#define BOATENV_TERM_TIMEOUT 4
#define BOATENV_TERM_RUDDER_BROKEN 5

/* step flags */
#define BOATENV_AUTO_RESET 1u      /* on done: count it, start the next episode in-kernel;
                                      obs_out then holds the NEW episode's first observation
                                      and final_obs_out (if given) the terminal one          */

/* The keys of configs/original_config.yaml that the hot path reads (SURVEY.md
 * section 5).  Plain doubles/ints; filled by the host binding from the YAML. */
typedef struct boatenv_params {
    int32_t experiment;        /* base_settings.experiment  wind.py:30, boat_env.py:166 */
    int32_t test_mode;         /* base_settings.test_mode   boat_env.py:72              */
    double dt;                 /* base_settings.dt          boat_env.py:153             */
    double t_max;              /* base_settings.t_max       boat_env.py:154, wind.py:14 */
    double track_width;        /* boat_env.track_width      boat_env.py:148,311         */
    double oob_offset;         /* boat_env.boat_out_of_bounds_offset  boat_env.py:200   */
    double goal_line;          /* boat_env.goal_line        boat_env.py:85,310          */
    double fuel;               /* boat.fuel                 boat_env.py:180             */
    double boat_m, boat_m_x, boat_m_y, boat_I, boat_Iz;           /* boat_env.py:214-281 */
    double propeller_diameter, wake_friction, c_r_front, c_r_side, thrust_deduction;
    double rho, boat_area_front, boat_area_side, boat_l, boat_b, rudder_area;
    int32_t fixed_points;      /* wind.fixed_points         wind.py:73,77               */
    int32_t _pad;
    double max_velocity;       /* wind.max_velocity         wind.py:41                  */
    double direction;          /* wind.direction, degrees   wind.py:44                  */
} boatenv_params;

typedef struct boatenv_handle *boatenv_t;

/* ---- life cycle ------------------------------------------------------------------ */

/* BoatEnv(config, experiment)  boat_env.py:10-65, batched over n_envs instances.
 * Episode randomness (the np.random draws of boat_env.py:147 and wind.py:78) comes
 * from Philox4x32-10 keyed by `seed` with counter (env_id_offset + i, episode), so
 * results do not depend on how envs are sharded over GPUs. */
BOATENV_API int boatenv_create(const boatenv_params *params, int64_t n_envs, uint64_t seed,
                   int64_t env_id_offset, int precision, int device, boatenv_t *out);
BOATENV_API int boatenv_destroy(boatenv_t h);

/* ---- gym API --------------------------------------------------------------------- */

/* BoatEnv.reset()  boat_env.py:120-126 for every env: new Boat (:144-201), new Wind
 * (wind.py:12-18).  obs_out: T[n_envs][11] or NULL.  mask: uint8[n_envs] or NULL (all). */
BOATENV_API int boatenv_reset(boatenv_t h, const uint8_t *mask, void *obs_out, void *stream);

/* BoatEnv.step(action)  boat_env.py:67-115 for every env.
 *   actions       T[n_envs]            (action[0] of each env; not clipped, like :73)
 *   obs_out       T[n_envs][11]        normalised state (:308-323)
 *   reward_out    T[n_envs]
 *   done_out      uint8[n_envs], or NULL when term_out is given (done == (term != 0): one byte per
 *                 env-step of HBM writes less)
 *   term_out      uint8[n_envs] or NULL  BOATENV_TERM_* of this step
 *   final_obs_out T[n_envs][11] or NULL  written only where done (terminal observation)
 */
BOATENV_API int boatenv_step(boatenv_t h, const void *actions, void *obs_out, void *reward_out,
                 uint8_t *done_out, uint8_t *term_out, void *final_obs_out, uint32_t flags,
                 void *stream);

/* K fused sub-steps of boat_env.py:67-115 with the env state held in registers:
 *   actions  T[K][n_envs] (action_stride = n_envs) or T[n_envs] repeated K times
 *            (action_stride = 0).
 * An env stops at its first done inside the window.  obs_out is the observation after
 * its last executed sub-step (or the new episode's first one under AUTO_RESET),
 * reward_out the sum over executed sub-steps, steps_out (int32[n_envs] or NULL) their
 * number. */
BOATENV_API int boatenv_step_k(boatenv_t h, const void *actions, int64_t action_stride, int32_t k,
                   void *obs_out, void *reward_out, uint8_t *done_out, uint8_t *term_out,
                   int32_t *steps_out, uint32_t flags, void *stream);

/* The same step through HOST buffers (pinned or pageable): copies actions H2D, steps,
 * copies obs/reward/done D2H, chunked over internal streams so that the copies overlap
 * the kernel.  Starts after the work queued on the legacy default stream and blocks until
 * the results are in host memory.  This is the end-to-end
 * call a CPU-side agent loop (main.py:80-81) makes.  Up to 2048 envs (the reference's single-env
 * loop included) it runs zero-copy instead: the kernel reads and writes mapped pinned memory
 * directly, one launch and one synchronize per call. */
BOATENV_API int boatenv_step_host(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                      uint8_t *done_host, uint32_t flags);
/* The same, also returning the termination codes (BOATENV_TERM_*) of this step in term_host: what the
 * single-env drop-in needs to maintain info['termination'] and its counters (boat_env.py:87-105). */
BOATENV_API int boatenv_step_host_term(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                           uint8_t *done_host, uint8_t *term_host, uint32_t flags);
/* boatenv_step_host / _term order themselves after the work queued on the legacy default stream.  This variant
 * names the caller's stream instead (the one its reset / step / learner kernels for this handle were queued on):
 * the internal copy / compute streams wait for an EVENT recorded there -- never a device-wide synchronise, so a
 * learner running on another stream of the same process keeps running.  term_host may be NULL.
 * main.py:80-81 with a CPU-side agent. */
BOATENV_API int boatenv_step_host_stream(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                             uint8_t *done_host, uint8_t *term_host, uint32_t flags, void *stream);
/* K fused sub-steps (boatenv_step_k) through HOST buffers: actions_host T[K][n_envs] in, ONE observation /
 * summed reward / done / termination code / executed-sub-step count per env out -- a host-side agent that
 * repeats or plans K actions moves K times fewer bytes per env-step over PCIe.  term_host and steps_host
 * (int32[n_envs]) may be NULL.  boat_env.py:67-115 K times per call. */
BOATENV_API int boatenv_step_k_host(boatenv_t h, const void *actions_host, int32_t k, void *obs_host, void *reward_host,
                        uint8_t *done_host, uint8_t *term_host, int32_t *steps_host, uint32_t flags, void *stream);

/* ---- state access (env.boat.* of main.py:94, recorder.py:36,46) -------------------- */

enum boatenv_field {
    BOATENV_F_V_X = 0, BOATENV_F_V_Y = 1, BOATENV_F_V_R = 2, BOATENV_F_RUDDER = 3,
    BOATENV_F_S_X = 4, BOATENV_F_S_Y = 5, BOATENV_F_S_R = 6, BOATENV_F_EPISODE_REWARD = 7,
    BOATENV_F_STEP_INDEX = 8,   /* uint32: Boat.index; t = index*dt, fuel = fuel0 - index */
    BOATENV_F_EPISODE = 9       /* uint32: episodes started by this env, minus one        */
};
/* out / in: T[n_envs] for fields 0..7, uint32[n_envs] for fields 8..9 (device). */
BOATENV_API int boatenv_get_field(boatenv_t h, int field, void *out, void *stream);
BOATENV_API int boatenv_set_field(boatenv_t h, int field, const void *in, void *stream);

/* All ten fields of ONE env (boatenv_field order, as doubles) into HOST memory with one launch:
 * what `env.boat.s_x ... rudder_angle` of main.py:94 and `return_all_data` (boat_env.py:128-140,
 * called by the Recorder every step, recorder.py:24-36) read.  Blocking. */
BOATENV_API int boatenv_env_state_host(boatenv_t h, int64_t env_index, double *out_host /* [10] */);

/* env.boat.wind.wind_velocity / .wind_angle (wind.py:16-17, recorder.py:46-47): the
 * current episode's tables of env `env_index`, double[L] each (device). */
BOATENV_API int boatenv_wind_table(boatenv_t h, int64_t env_index, double *wind_velocity_out,
                       double *wind_angle_out, void *stream);
BOATENV_API int boatenv_wind_length(boatenv_t h); /* int(t_max/dt)  wind.py:14-15 */

/* ---- episode recording (postprocessing/recorder.py:18-56, main.py:79) -------------- */

/* Caller-owned device columns of a recording ring, each [capacity][n_ids] row-major: row t holds
 * the recorded envs in `ids` order.  The eight state / step columns are T; term is
 * BOATENV_TERM_*; episode is BOATENV_F_EPISODE of the env when the row was taken. */
typedef struct boatenv_record_ring {
    void *s_x, *s_y, *v_x, *v_y, *s_r, *rudder_angle, *action, *reward;
    uint8_t *term;
    uint32_t *episode;
    int64_t capacity;
} boatenv_record_ring;

/* One recorder row of recorder.py:24-36 (return_all_data, boat_env.py:128-140) for n_ids envs in one
 * launch: writes row (row % capacity) of `ring` from local env ids int64[n_ids] (device; each in
 * [0, n_envs) -- an id outside is skipped, its entries left as they were).  s_x .. rudder_angle are
 * the values boatenv_get_field returns, bit for bit; action / reward / term are entry ids[j] of the
 * step's actions T[n_envs], reward T[n_envs] and term uint8[n_envs], each of which may be NULL
 * (zeros: the row of a state no step led to, e.g. right after reset).  Queued on `stream` after
 * the step it records; no synchronisation. */
BOATENV_API int boatenv_record_rows(boatenv_t h, const int64_t *ids, int64_t n_ids, const void *actions,
                        const void *reward, const uint8_t *term, const boatenv_record_ring *ring, int64_t row,
                        void *stream);

/* Validation hook: replace the Philox draws by caller-supplied ones for every episode
 * started after this call (fixture replay, differential tests against the reference).
 *   s_y_start int32[n_envs] or NULL; knots double[n_envs][2][fixed_points] or NULL
 * (device; copied).  Passing both NULL restores Philox. */
BOATENV_API int boatenv_set_episode_draws(boatenv_t h, const int32_t *s_y_start, const double *knots,
                              void *stream);

/* HOST function (no GPU work): the draws Philox makes for (seed, global env id,
 * episode): s_y_start as np.random.randint(-0.8*W, 0.8*W) (boat_env.py:147-150) and
 * knots_out[2][fixed_points] as the two np.random.sample(fixed_points) draws
 * (wind.py:78).  Lets a CPU reference be fed the identical episode randomness. */
BOATENV_API int boatenv_episode_draws_host(const boatenv_params *params, uint64_t seed, int64_t global_env_id,
                               uint32_t episode, int32_t *s_y_start_out, double *knots_out);

/* The same for n_ids global env ids and episodes [episode_begin, episode_begin + n_episodes) in one call
 * (the sampled-subset parity tests at benchmark size draw 10^5 episodes):
 *   s_y_start_out int32[n_episodes][n_ids] or NULL; knots_out double[n_episodes][n_ids][2][fixed_points] or NULL. */
BOATENV_API int boatenv_episode_draws_batch_host(const boatenv_params *params, uint64_t seed,
                               const int64_t *global_env_ids, int64_t n_ids, uint32_t episode_begin,
                               int32_t n_episodes, int32_t *s_y_start_out, double *knots_out);

/* ---- checkpoint / resume ----------------------------------------------------------- */

/* The reference checkpoints network weights only (networks/base_network.py:13-17); env state is
 * lost on restart.  Here the complete env state (all per-env scalars, step / episode indices,
 * wind coefficients, the cumulative statistics) is one opaque device blob: together with the
 * counter-based Philox streams it makes resume exact.  boatenv_state_bytes gives its size;
 * export / import copy it to / from a caller-owned device buffer.  A blob is only valid for a
 * handle created with the same params, n_envs and precision. */
BOATENV_API int64_t boatenv_state_bytes(boatenv_t h);
BOATENV_API int boatenv_export_state(boatenv_t h, void *blob_out, void *stream);
BOATENV_API int boatenv_import_state(boatenv_t h, const void *blob_in, void *stream);

/* ---- statistics (info dict of boat_env.py:24-32, cumulative) ----------------------- */

/* out_host[8] = { reached_goal, out_of_bounds, out_of_fuel, timeout, rudder_broken,
 *                 episodes_finished, sum(episode_reward), sum(episode_reward^2) } */
BOATENV_API int boatenv_get_counters(boatenv_t h, double *out_host, void *stream);
/* The same 8 doubles reduced into a device buffer (for an NCCL all-reduce). */
BOATENV_API int boatenv_reduce_counters(boatenv_t h, double *out_device, void *stream);

/* Fill T[n_envs] with the uniform(-1,1) policy "A1" of SURVEY.md 8(d): Philox keyed by
 * (seed, global env id, step_counter).  Benchmark / test input generator. */
BOATENV_API int boatenv_fill_uniform_actions(boatenv_t h, uint64_t step_counter, double scale, void *actions_out,
                                 void *stream);

/* ---- replay buffer (agent/buffer.py:3-35) ------------------------------------------ */

typedef struct boatreplay_handle *boatreplay_t;

/* ReplayBuffer(max_size, input_shape, n_actions)  buffer.py:4-11 (device resident). */
BOATENV_API int boatreplay_create(int64_t max_size, int32_t obs_dim, int32_t n_actions, int precision,
                      int device, boatreplay_t *out);
BOATENV_API int boatreplay_destroy(boatreplay_t r);
/* store_transition (buffer.py:13-22) for a batch of n rows, row i going to slot
 * (mem_cntr + i) % mem_size.  s, s2: T[n][obs_dim]; a: T[n][n_actions]; r: T[n];
 * done: uint8[n]. */
BOATENV_API int boatreplay_store(boatreplay_t r, int64_t n, const void *s, const void *a, const void *rew,
                     const void *s2, const uint8_t *done, void *stream);
/* sample_buffer (buffer.py:24-35): `batch` uniform draws with replacement from
 * [0, min(mem_cntr, mem_size)), Philox keyed by (seed, counter); gathers the five
 * arrays.  idx_out int64[batch] or NULL. */
BOATENV_API int boatreplay_sample(boatreplay_t r, int64_t batch, uint64_t seed, uint64_t counter, void *s_out,
                      void *a_out, void *r_out, void *s2_out, uint8_t *done_out, int64_t *idx_out,
                      void *stream);
/* The gather of buffer.py:29-33 with caller-supplied indices int64[batch] (device). */
BOATENV_API int boatreplay_gather(boatreplay_t r, int64_t batch, const int64_t *idx, void *s_out, void *a_out,
                      void *r_out, void *s2_out, uint8_t *done_out, void *stream);
/* Checkpoint restore: sets the store counter (buffer.py:6 mem_cntr).  The next store goes to slot mem_cntr % mem_size,
 * samples draw from [0, min(mem_cntr, mem_size)). */
/* boatreplay_sample for the rings of a population in ONE launch (member m on blockIdx.y = m): member m's rows equal
 * boatreplay_sample(m.ring, batch, m.seed, m.counter, m.s_out, m.a_out, m.r_out, m.s2_out, m.done_out, NULL) bit for
 * bit.  members_host: HOST array of n_members (1..BOATAGENT_SAC_MAX_MEMBERS) entries; the rings share precision
 * and device.  Errors (checked before anything is launched): BOATENV_EINVAL for a bad count, a NULL table, ring or
 * output, mixed precisions or devices; BOATENV_ESTATE for an empty ring. */
typedef struct boatreplay_sample_member {
    boatreplay_t ring;
    uint64_t seed, counter;
    void *s_out, *a_out, *r_out, *s2_out;
    uint8_t *done_out;
} boatreplay_sample_member;
BOATENV_API int boatreplay_sample_members(const boatreplay_sample_member *members_host, int32_t n_members,
                                          int64_t batch, void *stream);
BOATENV_API int boatreplay_set_mem_cntr(boatreplay_t r, int64_t mem_cntr);
BOATENV_API int64_t boatreplay_mem_cntr(boatreplay_t r); /* buffer.py:6  */
BOATENV_API int64_t boatreplay_mem_size(boatreplay_t r); /* buffer.py:5  */

/* env.step + agent.remember (main.py:81-88) in ONE kernel: steps every env and writes
 * the transition (obs_inout as s, action, reward, new obs as s', done) straight into
 * the ring.  obs_inout T[n_envs][11] holds the current observations on entry and the
 * next ones on return.  done_flag_mode: 0 = store done (any termination), 1 = store
 * (term == reached_goal) like main.py:83-88. */
BOATENV_API int boatenv_step_store(boatenv_t h, boatreplay_t r, const void *actions, void *obs_inout,
                       void *reward_out, uint8_t *done_out, uint8_t *term_out, int done_flag_mode,
                       uint32_t flags, void *stream);

/* ---- the actor's tanh-squashed Gaussian head (networks/networks.py:47-70) ------------ */

/* ActorNetwork.sample_normal after the two linear heads, fused: from mean, raw_std, eps (all
 * float32 [rows][n_actions], device; eps = the standard-normal draw) and max_action float32
 * [n_actions] to action [rows][n_actions] and log_prob [rows] (summed over the actions).
 * backward: gradients w.r.t. mean and raw_std of the REPARAMETERISED draw (rsample, :61), given
 * grad_action [rows][n_actions] and / or grad_log_prob [rows] (either may be NULL = zero). */
BOATENV_API int boatagent_gaussian_head_forward(const float *mean, const float *raw_std, const float *eps,
                                    const float *max_action, int64_t rows, int32_t n_actions,
                                    float *action_out, float *log_prob_out, void *stream);
BOATENV_API int boatagent_gaussian_head_backward(const float *mean, const float *raw_std, const float *eps,
                                     const float *max_action, const float *grad_action,
                                     const float *grad_log_prob, int64_t rows, int32_t n_actions,
                                     float *grad_mean_out, float *grad_raw_std_out, void *stream);

/* One optimiser step for ALL of the agent's networks -- torch.optim.Adam with its defaults
 * (networks.py:31,88,121), a learning rate per slot -- and, for slots with a `target`, the Polyak
 * average target = tau * param + (1 - tau) * target of update_network_parameters
 * (continuous_agent.py:66-80), in one launch.  slots_host: HOST array (copied into the kernel
 * arguments), all pointers float32 device tensors of `numel` elements.  state_dev: int64[2] on the
 * device, zero-initialised by the caller: [0] = steps taken (incremented by the launch), [1] internal. */
#define BOATAGENT_ADAM_MAX_SLOTS 64
typedef struct boatagent_adam_slot {
    float *param;
    const float *grad;
    float *exp_avg, *exp_avg_sq;
    float *target;          /* NULL: no target network for this tensor */
    int64_t numel;
    float lr;
    int32_t _pad;
} boatagent_adam_slot;
BOATENV_API int boatagent_adam_polyak_step(const boatagent_adam_slot *slots_host, int32_t n_slots, float beta1,
                               float beta2, float eps, float tau, int64_t *state_dev, void *stream);

/* choose_action (continuous_agent.py:57-61) for n envs in one tcgen05 kernel: ActorNetwork.forward
 * (networks.py:38-45, three 256-wide dense layers, bf16 inputs / fp32 accumulation) and the
 * non-reparameterised tanh-squashed draw (:47-65).  weight_blob: BOATAGENT_POLICY_BLOB_BYTES device
 * bytes, 16-byte aligned: [fc1 256 x 16 (obs_dim zero padded)][fc2 256 x 256] as bf16 in 8x8
 * core-matrix order -- element (row, k) of an R-row matrix at (k / 8) * (R * 16) + row * 16 +
 * (k % 8) * 2 --, then the heads as fp32 [16][256] row-major (mean rows, then std rows, zero
 * padded), then the fp32 biases [256][256][16].  obs float32 [n][obs_dim] (obs_dim <= 16); eps
 * float32 [n][n_actions] standard-normal draws or NULL (then Philox(seed; env, step) + Box-Muller);
 * n_actions 1, 2, 4 or 8. */
#define BOATAGENT_POLICY_BLOB_BYTES (256 * 16 * 2 + 256 * 256 * 2 + 16 * 256 * 4 + 256 * 4 + 256 * 4 + 16 * 4)
BOATENV_API int boatagent_policy_act(const void *weight_blob, const float *obs, const float *eps,
                         const float *max_action, uint64_t seed, uint64_t step, int64_t n, int32_t obs_dim,
                         int32_t n_actions, float *action_out, void *stream);

/* Closed-loop rollout of the tcgen05 policy on a BoatEnv handle (render_model, main.py:137-172, over every env of
 * the handle): the forward pass of boatagent_policy_act and one K = 1 boatenv_step sub-step without
 * BOATENV_AUTO_RESET, fused in one persistent kernel.  fp32 handles, n_actions = 1, weight_blob and max_action as
 * for boatagent_policy_act.  Sub-step t of env i acts with the action boatagent_policy_act gives row i with
 * step = step0 + t (Philox(seed; i, step) + Box-Muller), or with eps = 0 under BOATAGENT_ROLLOUT_DETERMINISTIC
 * (action = tanh(mean) * max_action).
 * Every env takes min(max_steps, steps until its episode ends) steps.  An env whose episode ends is then frozen:
 * no auto-reset and no further steps; its counters are updated once, as the step kernel does, and its state stays
 * the terminal state.  An env whose episode had already ended before the call is stepped on from its terminal
 * state, as boatenv_step would: reset it first.
 * obs_in float32 [N][11] is each env's last observation (what reset / step wrote); the first action needs it,
 * because the observation holds the last sub-step's accelerations, which the state does not.  Outputs, per env:
 *   obs_out    float32 [N][11]  the last observation (the terminal one if the episode ended); may alias obs_in
 *   return_out float32 [N]      the episode_reward slot (BOATENV_F_EPISODE_REWARD) after the last step
 *   steps_out  int32 [N]        steps taken in this call
 *   term_out   uint8 [N]        BOATENV_TERM_* of the ending step, 0 = still running after max_steps
 * At the end every env's state is written back (dyn slots, step index, wind coefficients; the episode number is
 * untouched), so get_field, export_state, step and another rollout continue exactly where the rollout stopped.
 * Errors: BOATENV_EUNSUPPORTED for an fp64 handle, BOATENV_ESTATE before reset, BOATENV_EINVAL for NULL
 * pointers, max_steps < 1 or unknown flags, BOATENV_EALIGN for a weight_blob that is not 16-byte aligned. */
#define BOATAGENT_ROLLOUT_DETERMINISTIC 1u   /* action = tanh(mean) * max_action */
BOATENV_API int boatagent_rollout(boatenv_t h, const void *weight_blob, const float *max_action, uint64_t seed,
                                  uint64_t step0, int32_t max_steps, uint32_t flags, const float *obs_in,
                                  float *obs_out, float *return_out, int32_t *steps_out, uint8_t *term_out,
                                  void *stream);

/* Experience collection with the tcgen05 policy (the main.py:78-90 loop body -- choose_action, env.step,
 * agent.remember -- over `steps` steps and every env of the handle) in one persistent kernel.  Each step is exactly
 * boatagent_policy_act (step = step0 + t, Philox draws, never deterministic) followed by
 * boatenv_step_store(..., BOATENV_AUTO_RESET): fp32 handles, n_actions = 1, weight_blob and max_action as for
 * boatagent_policy_act.  Row i of step t goes to ring slot (mem_cntr + t * n_envs + i) % mem_size:
 *   state = the observation the env acted on, action, reward, new_state = the observation after the step (the
 *   terminal one if the episode ended, written before the reset), terminal = (term == reached_goal) for
 *   done_flag_mode 1, (term != 0) for done_flag_mode 0.
 * An env whose episode ends is reset in the kernel as BOATENV_AUTO_RESET does (counters updated once, episode
 * number + 1, the new episode's draws) and keeps stepping.  On return the handle, the ring and the outputs are what
 * `steps` rounds of boatagent_policy_act and boatenv_step_store leave behind:
 *   obs_inout  float32 [N][11]  the current observations on entry, the last (post-reset) ones on return
 *   reward_out float32 [N], done_out / term_out uint8 [N] (either may be NULL, not both)  of the last step
 * and mem_cntr has grown by steps * n_envs.
 * Errors (a rejected call changes nothing): BOATENV_EUNSUPPORTED for an fp64 handle or a ring that is not fp32 with
 * obs_dim 11 and one action, BOATENV_ESTATE before reset, BOATENV_EINVAL for NULL pointers, steps < 1, a
 * done_flag_mode other than 0 / 1, ring and handle on different devices, or steps * n_envs > mem_size (rows of one
 * call may not share a slot), BOATENV_EALIGN for a weight_blob that is not 16-byte aligned. */
BOATENV_API int boatagent_collect(boatenv_t h, boatreplay_t r, const void *weight_blob, const float *max_action,
                                  uint64_t seed, uint64_t step0, int32_t steps, int done_flag_mode,
                                  float *obs_inout, float *reward_out, uint8_t *done_out, uint8_t *term_out,
                                  void *stream);

/* boatagent_collect that also records selected envs (the Recorder of main.py:79, postprocessing/recorder.py:18-56)
 * inside the kernel: after step t (and after its auto-reset), the recorder row of every env in `ids` goes to row
 * (row + t) % ring->capacity of `ring` -- exactly what boatenv_record_rows(h, ids, n_ids, actions, reward, term,
 * ring, row + t, ...) writes after the t-th round of boatagent_policy_act + boatenv_step_store: the state as
 * boatenv_get_field returns it (an ended episode's row holds the next episode's first state), the step's action,
 * reward and term code, and the episode number after the reset.  ids int64[n_ids] (device) are local env ids in any
 * order and must be unique; an id outside [0, n_envs) is skipped, its entries left as they were.  The ring is fp32
 * (the handle's precision).  Everything else -- ring rows, write-back, outputs, counters -- is boatagent_collect's.
 * Errors: those of boatagent_collect, and BOATENV_EINVAL for NULL ids, ring or ring column, n_ids <= 0 or
 * > 2^31 - 1, capacity <= 0, row < 0, or steps > capacity (one call would overwrite its own rows).  A rejected call
 * changes nothing. */
BOATENV_API int boatagent_collect_record(boatenv_t h, boatreplay_t r, const void *weight_blob, const float *max_action,
                                         uint64_t seed, uint64_t step0, int32_t steps, int done_flag_mode,
                                         float *obs_inout, float *reward_out, uint8_t *done_out, uint8_t *term_out,
                                         const int64_t *ids, int64_t n_ids, const boatenv_record_ring *ring,
                                         int64_t row, void *stream);

/* One SAC-v1 update (SACLearner.update) of the BoatEnv agent -- obs_dim 11, one action, 256-wide layers -- in two
 * tcgen05 kernels: the five networks' forward and backward passes per 128-row tile of the batch, then the gradient
 * reductions, Adam and the Polyak average of the target value network.  The 256 x 256 products (fc2 forward, its
 * input gradient and its weight gradient) and fc1's forward run with bf16 operands and fp32 accumulation; the heads,
 * the Gaussian head, fc1's gradients, the losses and the optimiser run in fp32.  Reductions run in a fixed order
 * without float atomics: an update is bit-reproducible.
 *   state, new_state float32 [batch][11]; action, reward float32 [batch]; done uint8 [batch]; eps float32 [2][batch]
 *   (the standard-normal draws of the two sample_normal calls); max_action float32 [1] (device);
 *   batch a positive multiple of 128;
 *   slots_host: the 26 slots of boatagent_adam_polyak_step in DeviceAdam's order -- actor fc1 w, b, fc2 w, b, mean w,
 *   b, std w, b; critic 1 and critic 2 fc1 w, b, fc2 w, b, q w, b; value fc1 w, b, fc2 w, b, v w, b with `target`
 *   the target value network's tensors (NULL for every other slot).  `param` is read, `grad` receives the batch
 *   gradient (as the fp32 learner leaves p.grad), then Adam (beta1, beta2, adam_eps, the slot's lr) and the Polyak
 *   average (tau) run as in boatagent_adam_polyak_step, with adam_state int64[2] as there;
 *   losses_out float32 [3] (device): value, actor, critic loss;
 *   workspace: boatagent_sac_update_workspace_bytes(batch) device bytes, 16-byte aligned.
 * Errors: BOATENV_EINVAL for NULL pointers, a batch that is not a positive multiple of 128, n_slots != 26, a slot
 * whose numel is not the agent's shape, a missing or extra target, a workspace that is too small; BOATENV_EALIGN for
 * a workspace or parameter that is not 16-byte aligned. */
BOATENV_API int64_t boatagent_sac_update_workspace_bytes(int64_t batch);   /* BOATENV_EINVAL for a bad batch */
BOATENV_API int boatagent_sac_update(const float *state, const float *action, const float *reward,
                                     const float *new_state, const uint8_t *done, const float *eps,
                                     const float *max_action, int64_t batch, float gamma, float reward_scale,
                                     const boatagent_adam_slot *slots_host, int32_t n_slots, float beta1,
                                     float beta2, float adam_eps, float tau, int64_t *adam_state, float *losses_out,
                                     void *workspace, int64_t workspace_bytes, void *stream);
/* The gradients of boatagent_sac_update without its optimiser step, for data-parallel training: every replica
 * computes the gradients of its own batch, the replicas all-reduce them, and each applies the same Adam step.
 * Arguments and errors as boatagent_sac_update's, without the Adam hyper-parameters and state.  Each slot's `grad`
 * receives grad_scale times the batch gradient and losses_out grad_scale times the three losses; parameters, targets,
 * Adam moments and step counter are only read (the moments not at all).  grad_scale = 1 / world makes a SUM
 * all-reduce the mean, exactly when world is a power of two.
 * With grad_scale = 1, this call followed by boatagent_adam_polyak_step on the same slots (and the same adam_state)
 * equals one boatagent_sac_update bit for bit: gradients, weights, targets, Adam moments, step counter and losses.
 * The split costs one extra launch (the Adam kernel). */
BOATENV_API int boatagent_sac_gradients(const float *state, const float *action, const float *reward,
                                        const float *new_state, const uint8_t *done, const float *eps,
                                        const float *max_action, int64_t batch, float gamma, float reward_scale,
                                        const boatagent_adam_slot *slots_host, int32_t n_slots, float grad_scale,
                                        float *losses_out, void *workspace, int64_t workspace_bytes, void *stream);

/* Population training on one GPU: one SAC update of each of n_members INDEPENDENT agents (the reference's `main.py -p N`
 * members, main.py:215-235, each with its own utils/hyperparameter_tuner.py draw) in the two kernels of
 * boatagent_sac_update, launched once for all of them (member m on blockIdx.y = m).  Member m computes exactly what
 * boatagent_sac_update computes with its entry's arguments, bit for bit.  Each entry of members_host (a HOST array,
 * copied into the kernel arguments) names one agent:
 *   state .. max_action, slots / n_slots, gamma, reward_scale, adam_state, losses: as for boatagent_sac_update (the
 *   slots carry the member's learning rates); tau: the member's Polyak factor.
 * Shared by all members: batch (a positive multiple of 128), beta1, beta2, adam_eps.  Members must not share
 * parameters, gradients, moments, adam_state or losses.
 *   workspace: n_members * boatagent_sac_update_workspace_bytes(batch) device bytes, 16-byte aligned; member m uses
 *   the slice at m times that size.
 * Errors (checked for every member before anything is launched): BOATENV_EINVAL for n_members outside
 * 1..BOATAGENT_SAC_MAX_MEMBERS, a NULL table, workspace or adam_state, a workspace that is too small, and every
 * argument error of boatagent_sac_update; BOATENV_EALIGN as there. */
#define BOATAGENT_SAC_MAX_MEMBERS 16   /* the member tables fill most of the 32,764 bytes of kernel parameters */
typedef struct boatagent_sac_member {
    const float *state, *action, *reward, *new_state;
    const uint8_t *done;
    const float *eps, *max_action;
    const boatagent_adam_slot *slots;   /* HOST array of n_slots (26) slots */
    int32_t n_slots;
    float gamma, reward_scale, tau;
    int64_t *adam_state;
    float *losses;
} boatagent_sac_member;
BOATENV_API int boatagent_sac_update_members(const boatagent_sac_member *members_host, int32_t n_members,
                                             int64_t batch, float beta1, float beta2, float adam_eps, void *workspace,
                                             int64_t workspace_bytes, void *stream);
/* Data-parallel population training: boatagent_sac_update_members split as boatagent_sac_gradients splits
 * boatagent_sac_update, so that each member's gradients can be all-reduced over the ranks that train it.
 *
 * boatagent_sac_gradients_members: boatagent_sac_gradients of every member in one launch pair.  Each slot's `grad`
 * receives grad_scale times the member's batch gradient and `losses` grad_scale times its three losses; parameters,
 * targets, Adam moments and step counters are not written, `tau` and `adam_state` are not read (adam_state may be
 * NULL).  Member m's results equal a boatagent_sac_gradients call with its entry's arguments, bit for bit.  Table,
 * workspace and errors as boatagent_sac_update_members, without the adam_state check.
 *
 * boatagent_adam_polyak_members: boatagent_adam_polyak_step(slots, 26, beta1, beta2, adam_eps, tau, adam_state) of
 * every member in one launch (member m on blockIdx.y = m, the same 2048-element chunks on blockIdx.x): each member
 * reads its slots' `grad`, steps with its slots' learning rates, its `tau` and its adam_state, bit for bit as that
 * call.  The batch, draw and loss pointers are not read.  Members must not share parameters, moments, targets or
 * adam_state.  Errors (checked for every member before anything is launched): BOATENV_EINVAL for a NULL table,
 * n_members outside 1..BOATAGENT_SAC_MAX_MEMBERS, n_slots != 26, a NULL slot pointer, a slot whose numel is not the
 * agent's shape, a missing or extra target, a NULL adam_state.
 *
 * With grad_scale = 1, boatagent_sac_gradients_members followed by boatagent_adam_polyak_members equals
 * boatagent_sac_update_members bit for bit: gradients, weights, targets, Adam moments, step counters and losses. */
BOATENV_API int boatagent_sac_gradients_members(const boatagent_sac_member *members_host, int32_t n_members,
                                                int64_t batch, float grad_scale, void *workspace,
                                                int64_t workspace_bytes, void *stream);
BOATENV_API int boatagent_adam_polyak_members(const boatagent_sac_member *members_host, int32_t n_members, float beta1,
                                              float beta2, float adam_eps, void *stream);

/* ---- toy integrator envs (environment/toy_car.py, toy_parachute.py) ---------------- */

typedef struct boattoy_handle *boattoy_t;
#define BOATTOY_CAR 0
#define BOATTOY_PARACHUTE 1
/* params_host: double[n_params] shared by all envs, jitter: each env's parameters are
 * scaled by 1 + jitter*u, u = Philox uniform(-1,1) keyed (seed, env, param); env 0 is
 * never jittered.  toy_car params: {accel, v_limit, dtheta, dt}; toy_parachute params:
 * {h0, h1, area_free, area_chute, mass, c_w, rho, g, dt_integrator}. */
BOATENV_API int boattoy_create(int kind, int64_t n_envs, const double *params_host, int32_t n_params,
                   double jitter, uint64_t seed, int precision, int device, boattoy_t *out);
BOATENV_API int boattoy_destroy(boattoy_t t);
BOATENV_API int boattoy_reset(boattoy_t t, void *stream);
/* k loop iterations of toy_car.py:22-32 / toy_parachute.py:23-40 per env.
 * out: T[n_envs][4]: car {s_x, s_y, v, angle}; parachute {s, v, a, integrator calls}.
 * done_out uint8[n_envs] or NULL (parachute: s < 0 reached; the env then stays put). */
BOATENV_API int boattoy_step(boattoy_t t, int32_t k, void *out, uint8_t *done_out, void *stream);
/* HOST function (no GPU work): the per-env parameters that envs [env_begin, env_begin + n_envs) of a toy handle
 * created with (params_host, jitter, seed) use -- out double[n_envs][n_params], env 0 = the script constants
 * (toy_car.py:7-8,11,23; toy_parachute.py:8-15).  Lets a CPU reference run the jittered envs. */
BOATENV_API int boattoy_params_host(int kind, const double *params_host, int32_t n_params, double jitter, uint64_t seed,
                        int64_t env_begin, int64_t n_envs, double *out);

/* ---- misc -------------------------------------------------------------------------- */
BOATENV_API const char *boatenv_version(void);
BOATENV_API const char *boatenv_error_string(int code);
/* Number of kernels this library has launched in this process (all handles). */
BOATENV_API int64_t boatenv_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* BOATENV_H */
