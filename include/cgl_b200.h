/*
 * cgl_b200.h -- C ABI of libcgl_b200.so: the B200-native (sm_100a) Game-of-Life env step.
 *
 * This is the drop-in boundary for the hot path of BADBEEF6502/ECEN743-Project-CGoL
 * (class `sim`, /root/reference/CGL/CGL.py).  The reference has no FFI of its own: its device
 * path is a PyCUDA kernel string (`run`, CGL/CGL.py:146-182) plus four memcpys
 * (`__step_state_gpu`, CGL/CGL.py:203-208).  Every entry point below cites the reference
 * lines it replaces.  Plain pointers and sizes only -- no torch / numpy types.  The Python
 * host (ecen743-project-cgol_b200/CGL.py, cgl_b200/) binds it with ctypes; INTEGRATION.md shows
 * the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - "device" pointers are CUDA device pointers on the current device; all device entry points
 *     are asynchronous on `stream` (a cudaStream_t passed as void*, NULL = legacy default).
 *   - world plane, bit-packed: per env `rows` rows of W = ceil(cols/32) uint32 words;
 *     bit j of word w = cell at column 32*w + j; padding bits are zero.  Batch = [n_envs][rows][W].
 *   - stable plane: int8 [n_envs][rows*cols], the reference's own row-major order
 *     (it IS the observation, CGL/CGL.py:281-285).
 *   - return value: 0 on success; >0 = cudaError_t; <0 = CGL_E_* argument error.
 *     cgl_last_error() returns a thread-local message for the last failure.
 */
#ifndef CGL_B200_H
#define CGL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGL_B200_ABI_VERSION 1

#define CGL_E_BADARG   (-1)   /* null pointer / zero size / unsupported shape */
#define CGL_E_BADINDEX (-2)   /* toggle index outside [0, size] (host-buffer entry points only) */
#define CGL_E_NOMEM    (-3)

typedef void *cgl_stream_t;

int cgl_abi_version(void);
const char *cgl_last_error(void);

/* ---- device-side waits never hang and never compute on stale data ---------------------------
 * Several kernels wait on the device for a token written by another CTA, launch or GPU (chained env steps,
 * chained life strips, the halo exchange).  Every such wait is bounded by a wall-clock deadline
 * (cgl_set_wait_timeout_ms, default 2000 ms, per process; applied to the current device at once and to other
 * devices at their next cgl_alarm_words call).  A waiter that gives up writes nothing that depends on the
 * missing data, does not publish its own token, and stores 1 into its ALARM WORD: host-mapped pinned
 * int32[CGL_ALARM_WORDS] owned by the library.  cgl_alarm_words returns the host pointer (and installs the
 * words on the current device); the host may read them at any time without synchronising and clears them by
 * writing 0.  Index: 0 = an action / toggle index outside [0, side*side] was ignored (the reference raises
 * ValueError at toggle time, CGL/CGL.py:327-328), 1 = chained env step token timeout, 2 = life-mode strip
 * token timeout, 3 = halo exchange timeout (a ring neighbour never delivered). */
#define CGL_ALARM_WORDS 4
int cgl_alarm_words(int **host_words_out);
int cgl_set_wait_timeout_ms(uint32_t ms);
/* Test hook: which = 1 makes the next chained cgl_life_run wait for strip tokens that never arrive (exercises the
 * bounded wait + alarm path; tests only). */
int cgl_test_fault(int which);

/* Number of CUDA devices / name + SM count of `device` (replaces the device banner query,
 * CGL/CGL.py:120-140).  name_out may be NULL. */
int cgl_device_count(int *count_out);
int cgl_device_info(int device, char *name_out, int name_cap, int *sm_count_out,
                    int *cc_major_out, int *cc_minor_out, uint64_t *total_mem_out);

/* uint32 words per packed row. */
uint32_t cgl_words_per_row(uint32_t cols);

/* ---- layout conversion at the API boundary ---------------------------------------------
 * pack:   cells uint8 [n_envs][rows*cols] (nonzero = alive) -> packed world.
 * unpack: packed world -> cells uint8 {0,1}.     (reference array format: CGL/CGL.py:94,107) */
int cgl_pack(const uint8_t *cells_dev, uint32_t *world_dev, uint64_t n_envs, uint32_t rows,
             uint32_t cols, cgl_stream_t stream);
int cgl_unpack(const uint32_t *world_dev, uint8_t *cells_dev, uint64_t n_envs, uint32_t rows,
               uint32_t cols, cgl_stream_t stream);

/* stable = alive ? spawn : 0   (constructor, CGL/CGL.py:111-112). */
int cgl_init_stable(const uint32_t *world_dev, int8_t *stable_dev, uint64_t n_envs, uint32_t side,
                    int spawn, cgl_stream_t stream);

/* ---- sim.toggle_state, CGL/CGL.py:322-328 -------------------------------------------------
 * idx_dev: int32 [n_envs][k].  For every env: each DISTINCT valid index in its row is toggled
 * once (numpy gather-then-scatter semantics) and stable[idx] = spawn.  idx == side*side is the
 * "do nothing" action; anything else out of range is skipped and sets *err_flag_dev |= 1
 * (err_flag_dev may be NULL). */
int cgl_toggle(uint32_t *world_dev, int8_t *stable_dev, uint64_t n_envs, uint32_t side,
               const int32_t *idx_dev, uint32_t k, int spawn, int *err_flag_dev,
               cgl_stream_t stream);

/* ---- the env step: toggle (optional) -> generation -> stability -> reward ----------------
 * Replaces kernel `run` (CGL/CGL.py:147-181) + `__step_state_gpu` (:203-208) + reward()
 * (:255-256) + alive() (:259-260) for n_envs independent environments, fused in one launch on
 * the fast path (side % 32 == 0, 32 <= side <= 256) and three launches otherwise.
 *   world_in_dev   packed world at t.  Scratch after the call (the generic path applies the
 *                  toggle in place); world_out_dev receives t+1.  Must not alias.
 *   stable_dev     updated in place.
 *   actions_dev    int32 [n_envs] or NULL: one toggle_state(action) per env before the step
 *                  (CGL/main.py:66-67); action == side*side is the no-op; other out-of-range
 *                  values are ignored and set *err_flag_dev |= 1.
 *   reward_out_dev int32 [n_envs] or NULL;  alive_out_dev uint32 [n_envs] or NULL. */
int cgl_env_step(uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev,
                 uint64_t n_envs, uint32_t side, const int32_t *actions_dev, int spawn,
                 int stable_max, int32_t *reward_out_dev, uint32_t *alive_out_dev,
                 int *err_flag_dev, cgl_stream_t stream);

/* Chained env steps (fused sides only): identical results to cgl_env_step, but consecutive calls on
 * the same stream depend on each other PER ENVIRONMENT instead of per launch.  token_dev: uint32
 * [n_envs].  Env e waits until token[e] == want and stores token[e] = publish when its planes are
 * written; the caller uses one id per world plane (want = id of world_in, publish = id of
 * world_out, all tokens initialised to the id of the current plane), which also makes a captured
 * CUDA graph of an even number of steps replayable.  The next launch's first CTAs then run while this
 * launch's last CTAs finish (programmatic dependent launch without the grid-wide wait).  Anything
 * else that touches the state between two chained steps is ordered by the stream as usual.  A
 * token that does not arrive within the wait bound (cgl_set_wait_timeout_ms) sets bit 1 of *err_flag_dev and the
 * alarm word, and the env is SKIPPED (nothing written, token not published) instead of being stepped from stale
 * planes. */
int cgl_env_step_chained(uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev,
                         uint64_t n_envs, uint32_t side, const int32_t *actions_dev, int spawn,
                         int stable_max, int32_t *reward_out_dev, uint32_t *alive_out_dev,
                         int *err_flag_dev, uint32_t *token_dev, uint32_t want, uint32_t publish,
                         cgl_stream_t stream);

/* ---- the general form: every env-step entry point above and below is a thin wrapper of this one ----
 * One struct describes a step completely, so a caller (or a binding) fills it once per buffer set and passes one
 * pointer per step.  Zero-initialise it; fields not mentioned keep the meaning they have in cgl_env_step.
 *   stable_in_dev / stable_out_dev   read / written stability planes (out == NULL or == in: in place)
 *   dead_rule / empty / empty_min / masked_toggle   the CGL_action+ fork's variants (all 0 = the base env)
 *   chain_mode   how consecutive steps on one stream depend on each other (fused sides only for 1 and 2):
 *     CGL_CHAIN_NONE  per launch (programmatic dependent launch, the whole previous grid);
 *     CGL_CHAIN_IDS   per environment through token_dev[e], `want` / `publish` = ids of the world planes
 *                     (see cgl_env_step_chained): a captured CUDA graph of an even number of steps replays;
 *     CGL_CHAIN_SEQ   per environment through token_dev[e] holding SEQUENCE NUMBERS: env e waits for
 *                     token[e] == want and publishes want + 1.  The fastest form (a CTA releases its dependents
 *                     at entry: 24.9 vs 25.7 us per 4096 x 128^2 step), but consecutive steps must carry
 *                     consecutive numbers, so a captured graph cannot be replayed.  If seq_counter_host is not
 *                     NULL the library reads `want` from it and increments it after the launch (the caller keeps
 *                     one host counter per env batch and initialises all tokens to its value). */
#define CGL_CHAIN_NONE 0u
#define CGL_CHAIN_IDS  1u
#define CGL_CHAIN_SEQ  2u
typedef struct cgl_env_step_args {
    uint32_t *world_in_dev, *world_out_dev;
    const int8_t *stable_in_dev;
    int8_t *stable_out_dev;
    uint64_t n_envs;
    uint32_t side;
    int32_t spawn, stable_max, dead_rule, empty, empty_min, masked_toggle;
    const int32_t *actions_dev;       /* or NULL */
    int32_t *reward_out_dev;          /* or NULL */
    uint32_t *alive_out_dev;          /* or NULL */
    int *err_flag_dev;                /* or NULL */
    uint32_t *token_dev;              /* chain_mode 1, 2 */
    uint32_t want, publish, chain_mode;
    uint32_t *seq_counter_host;       /* chain_mode 2, or NULL */
} cgl_env_step_args_t;
int cgl_env_step_ex(const cgl_env_step_args_t *args, cgl_stream_t stream);

/* A sequence of env steps enqueued by ONE call: step i (i = 0 .. n_steps-1) is cgl_env_step_ex(&steps[(first + i) %
 * n_descs]).  A caller that rotates several env batches and ping-pong planes describes one full cycle and lets it
 * repeat.  The launches are issued back to back from C (the host cost of a step is one kernel launch), on `stream`,
 * asynchronously.  The descriptors must stay valid only for the duration of the call. */
int cgl_env_step_seq(const cgl_env_step_args_t *steps, uint32_t n_descs, uint64_t n_steps, uint64_t first,
                     cgl_stream_t stream);
/* cgl_env_step_seq with two CUDA events (cudaEvent_t, may be NULL) recorded on `stream` immediately before the first
 * and after the last launch -- for timing a region of K steps on the device without the binding's call overhead
 * between the start event and the first launch (bench.py). */
int cgl_env_step_seq_timed(const cgl_env_step_args_t *steps, uint32_t n_descs, uint64_t n_steps, uint64_t first,
                           cgl_stream_t stream, void *start_event, void *stop_event);

/* Out-of-place env step: as cgl_env_step / cgl_env_step_chained (token_dev == NULL: plain stream order;
 * otherwise the chained form), but the stability plane is READ from stable_in_dev and the new plane is
 * WRITTEN to stable_out_dev, a second int8 [n_envs, side*side] buffer (stable_in_dev is left untouched on
 * the fused sides).  This is how the batched DQN loop records transitions: the caller hands the env the
 * next slot of its replay ring, so ExperienceReplay.add (CGL/dqn.py:24-36, two state copies per step)
 * costs no memory traffic.  stable_in_dev == stable_out_dev is the in-place step.  Generic sides copy the
 * plane first and do not take tokens. */
int cgl_env_step_io(uint32_t *world_in_dev, uint32_t *world_out_dev, const int8_t *stable_in_dev,
                    int8_t *stable_out_dev, uint64_t n_envs, uint32_t side, const int32_t *actions_dev,
                    int spawn, int stable_max, int32_t *reward_out_dev, uint32_t *alive_out_dev,
                    int *err_flag_dev, uint32_t *token_dev, uint32_t want, uint32_t publish,
                    cgl_stream_t stream);

/* Many plain env steps (no actions) in ONE launch with each environment resident in shared memory:
 * the step loop of CGL/bench.py:39-40, and -- with stop_when_fixed -- the convergence loop of
 * CGL/CGL_action+/validate.py:133-139 (step until a step leaves the world unchanged, at most max_steps
 * steps; the reference copies the world to the host and compares there after every step).
 *   world_in_dev / world_out_dev  packed world before / after; MAY alias (each env is read completely
 *                                 before it is written).   stable_dev is updated in place.
 *   steps_out_dev  int32 [n_envs] or NULL: steps actually executed per env (== max_steps unless
 *                  stop_when_fixed ended the env early; the step that found the fixed point counts).
 *   reward_out_dev / alive_out_dev as in cgl_env_step (of the final state; valid for max_steps == 0 too).
 * Sides: the fused sides (multiples of 32 up to 256) and any side <= 274. */
int cgl_env_run(const uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev, uint64_t n_envs,
                uint32_t side, uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max,
                int32_t *steps_out_dev, int32_t *reward_out_dev, uint32_t *alive_out_dev, cgl_stream_t stream);

/* cgl_env_run with the CGL_action+ fork's dead-cell rule (dead_rule / empty / empty_min as in
 * cgl_env_step_rule) -- the fork's validate.py convergence loop runs on the fork's env. */
int cgl_env_run_rule(const uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev, uint64_t n_envs,
                     uint32_t side, uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max,
                     int dead_rule, int empty, int empty_min, int32_t *steps_out_dev, int32_t *reward_out_dev,
                     uint32_t *alive_out_dev, cgl_stream_t stream);

/* Value counts of the stability plane, the device form of breakdown_stable (CGL/CGL_action+/CGL.py:
 * 294-297, np.unique(..., return_counts=True)): hist_out_dev uint32 [n_envs][256],
 * hist[e][v + 128] = number of cells of env e whose stability equals v. */
int cgl_breakdown_stable(const int8_t *stable_dev, uint64_t n_envs, uint64_t size, uint32_t *hist_out_dev,
                         cgl_stream_t stream);

/* ---- the CGL_action+ fork of the env (CGL/CGL_action+/CGL.py) --------------------------------
 * Same step with three differences, each an argument here:
 *   dead_rule      what a cell that is dead after the step gets:
 *                    0  0                                            (the base env, CGL/CGL.py:179,242)
 *                    1  (s == empty_min) ? s : int8(s - 1)           (the fork's CUDA kernel, :190-193)
 *                    2  min(int8(s + empty), empty_min)              (the fork's CPU step, :256)
 *                  the fork's two back ends disagree, so the caller chooses which one to reproduce;
 *   masked_toggle  1: a toggled cell gets SPAWN only if it is alive after the toggle, else 0 (:382-384);
 *                  0: SPAWN either way (base env, CGL/CGL.py:326);
 *   empty          initial stability of dead cells (cgl_init_stable_rule; also replaces a 0 SPAWN, :124-126).
 * Everything else (planes, actions, tokens, stable_in/out, outputs) is as in cgl_env_step_io; with
 * dead_rule = 0, masked_toggle = 0 the results equal cgl_env_step's. */
int cgl_env_step_rule(uint32_t *world_in_dev, uint32_t *world_out_dev, const int8_t *stable_in_dev,
                      int8_t *stable_out_dev, uint64_t n_envs, uint32_t side, const int32_t *actions_dev,
                      int spawn, int stable_max, int dead_rule, int empty, int empty_min, int masked_toggle,
                      int32_t *reward_out_dev, uint32_t *alive_out_dev, int *err_flag_dev, uint32_t *token_dev,
                      uint32_t want, uint32_t publish, cgl_stream_t stream);

/* cgl_toggle with the fork's masked stability write (masked = 1), K indices per env
 * (CGL_action+/helper.py:108-132 passes the four cells of a 2x2 block). */
int cgl_toggle_rule(uint32_t *world_dev, int8_t *stable_dev, uint64_t n_envs, uint32_t side,
                    const int32_t *idx_dev, uint32_t k, int spawn, int masked, int *err_flag_dev,
                    cgl_stream_t stream);

/* stable = alive ? spawn : 0, then zeros -> empty (CGL_action+/CGL.py:122-126). */
int cgl_init_stable_rule(const uint32_t *world_dev, int8_t *stable_dev, uint64_t n_envs, uint32_t side,
                         int spawn, int empty, cgl_stream_t stream);

/* ---- one environment, one launch: the body of the reference's training loop -------------------
 * CGL/main.py:64-72 per iteration: toggle_state(action) (CGL/CGL.py:322-328) -> step() (:247-252: two H2D copies,
 * kernel `run` :147-181, two D2H copies :203-208) -> get_stable(shallow) (:281-285) -> reward() (:255-256).
 * cgl_sim_step does all of it for ONE environment of any side <= cgl_sim_step_max_side() in ONE kernel:
 *   action        index in [0, side*side) toggled before the step, or side*side = none; passed BY VALUE, so
 *                 nothing the host may rewrite later is read by the kernel
 *   dead_rule / empty / empty_min / masked_toggle   as in cgl_env_step_rule (0, 0, 0, 0 = the base env)
 *   obs_mirror    NULL, or int8[side*side] the kernel ALSO stores the new stability plane to -- the caller's
 *                 pinned host-mapped observation buffer (no device-to-host copy)
 *   result        NULL, or int32[4] (device or pinned host-mapped): [0] = reward, [1] = live cells, then -- after
 *                 system-scope fences, so mirror and result are complete when it shows -- [2] = seq.  The host
 *                 polls [2] instead of synchronising the stream.
 * world_in / world_out / stable are the resident device planes as in cgl_env_step. */
int cgl_sim_step(const uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev, uint32_t side,
                 int32_t action, int spawn, int stable_max, int dead_rule, int empty, int empty_min,
                 int masked_toggle, int8_t *obs_mirror, int32_t *result, uint32_t seq, cgl_stream_t stream);
uint32_t cgl_sim_step_max_side(void);
/* The same call for bindings: everything that stays the same from step to step lives in a struct the caller fills
 * once.  The current world is in world_a_dev if *flip_planes is even, else in world_b_dev; the library steps into
 * the other plane and increments *flip_planes (a host counter owned by the caller; NULL = always a -> b). */
typedef struct cgl_sim_step_args {
    uint32_t *world_a_dev, *world_b_dev;
    int8_t *stable_dev;
    uint32_t side;
    int32_t spawn, stable_max, dead_rule, empty, empty_min, masked_toggle;
    int8_t *obs_mirror;
    int32_t *result;
    uint32_t *flip_planes;
} cgl_sim_step_args_t;
int cgl_sim_step_ex(const cgl_sim_step_args_t *args, int32_t action, uint32_t seq, cgl_stream_t stream);

/* The resident form of cgl_sim_step for the same loop (CGL/main.py:64-72) when the caller steps ONE environment over
 * and over: cgl_sim_serve launches a single-CTA kernel that keeps the environment in shared memory and serves steps
 * without any further launch, copy or stream synchronisation.
 *   cmd_host      pinned host-mapped uint64 the host writes with one store: (seq << 32) | action, action as in
 *                 cgl_sim_step, or CGL_SIM_QUIT to make the kernel leave.  A command is new when its seq differs
 *                 from the last one served (`last_seq` at launch).
 *   args->result  pinned host-mapped int32[8], 16-byte aligned (so must args->obs_mirror be; cmd_host 8-byte
 *                 aligned): per served step ONE 16-byte store {reward, live cells, seq, 0}
 *                 after the new observation is complete in args->obs_mirror (system-scope fence in between); when
 *                 the kernel has left -- planes written back to world_a/world_b (whichever held the state, see
 *                 flip_planes; not advanced) and stable_dev -- result[4] = launch_id.  result[5] / result[6] are
 *                 diagnostics of the last served step: nanoseconds from "command seen" to "step computed" and to
 *                 "observation mirror fenced" on the device clock.
 *   linger_us     the kernel also leaves by itself after this long without a new command (1..100000), so a device-
 *                 wide synchronisation elsewhere in the process is never held up for longer; the host notices
 *                 result[4] == launch_id and launches again with the next step.
 * `stream` must not be synchronised with by the host while commands are outstanding (use a non-blocking stream of
 * its own).  Sides up to cgl_sim_serve_max_side(). */
#define CGL_SIM_QUIT 0xFFFFFFFEu
int cgl_sim_serve(const cgl_sim_step_args_t *args, const void *cmd_host, uint32_t last_seq, uint32_t launch_id,
                  uint32_t linger_us, cgl_stream_t stream);
uint32_t cgl_sim_serve_max_side(void);

/* Which path cgl_env_step takes for `side`: 1 = fused fast kernel, 0 = generic kernels. */
int cgl_env_step_is_fused(uint32_t side);

/* Number of kernel launches one cgl_env_step call issues (for bench.py's gpu_launches). */
int cgl_env_step_launches(uint32_t side, int has_actions);

/* ---- world-only generations ("life mode": the world half of `run`, CGL/CGL.py:154-170) -----
 * One generation of n_envs independent (rows x cols) grids.  Columns always wrap (torus).
 * wrap_rows = 1: rows wrap (the reference's torus).  wrap_rows = 0: rows outside the array are
 * dead -- used for row bands that carry their own ghost rows (multi-GPU halo exchange).
 * alive_out_dev: uint32 [n_envs] popcount of the result, or NULL. */
int cgl_life_step(const uint32_t *world_in_dev, uint32_t *world_out_dev, uint64_t n_envs,
                  uint32_t rows, uint32_t cols, int wrap_rows, uint32_t *alive_out_dev,
                  cgl_stream_t stream);

/* `gens` generations of ONE (rows x cols) grid, ping-ponging between buf_a (input) and buf_b,
 * `k` generations per HBM pass (temporal blocking in registers; k = 1 streams).  For k = 4, 8, 16 the bulk of the
 * run is ONE cooperative launch in which a warp keeps its strip for all passes and waits only for its neighbour
 * strips (cgl_life_persist.cu); otherwise one launch per pass, chained strip by strip.
 * *result_in_a_out = 1 if the final state is in buf_a else 0.  The blocked kernels need cols % 32 == 0 and
 * cols >= 960; other shapes fall back to cgl_life_step per generation. */
int cgl_life_run(uint32_t *buf_a_dev, uint32_t *buf_b_dev, uint32_t rows, uint32_t cols,
                 int wrap_rows, uint32_t gens, uint32_t k, int *result_in_a_out,
                 cgl_stream_t stream);

/* Optional set-up call: time a few strip lengths of the k-blocked kernel for this (rows, cols, k)
 * on the caller's buffers (buf_b is clobbered, buf_a untouched) and remember the fastest for later
 * cgl_life_run calls.  Synchronises the stream. */
int cgl_life_tune(uint32_t *buf_a_dev, uint32_t *buf_b_dev, uint32_t rows, uint32_t cols, int wrap_rows,
                  uint32_t k, cgl_stream_t stream);

/* ---- reductions ----------------------------------------------------------------------------
 * reward(): np.add.reduce(stable, dtype=int32), CGL/CGL.py:255-256 (wraps mod 2^32).
 * alive():  np.add.reduce(world, dtype=uint32), CGL/CGL.py:259-260. */
int cgl_reward(const int8_t *stable_dev, uint64_t n_envs, uint64_t size, int32_t *reward_out_dev,
               cgl_stream_t stream);
int cgl_alive(const uint32_t *world_dev, uint64_t n_envs, uint64_t words_per_env,
              uint32_t *alive_out_dev, cgl_stream_t stream);
/* match(): (world == other).all(), CGL/CGL.py:269-270, on packed planes.
 * *equal_out_dev (int32) = 1 if all n_words are equal else 0. */
int cgl_match(const uint32_t *a_dev, const uint32_t *b_dev, uint64_t n_words, int *equal_out_dev,
              cgl_stream_t stream);

/* ---- host-buffer entry point: literal replacement of sim.__step_state_gpu -----------------
 * CGL/CGL.py:203-208: H2D world + stable, one generation, D2H world + stable, in place into
 * the caller's numpy buffers (reference array format: uint8 / int8 [side*side]).  Synchronous.
 * Internally packs on the device and runs the same kernels as cgl_env_step. */
int cgl_step_state_gpu(uint8_t *world_host, int8_t *stable_host, uint32_t side, int spawn,
                       int stable_max);

/* Batched host-buffer step (used for the end-to-end bench): actions int32[n_envs] or NULL on the
 * host; resident device state (packed world ping-pong + stable) identified by the pointers;
 * copies actions H2D, steps, copies reward (and the observation if obs_host != NULL) D2H.
 * All host buffers should be pinned for the copies to be asynchronous. Synchronous on return. */
int cgl_env_step_host(uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev,
                      uint64_t n_envs, uint32_t side, const int32_t *actions_host,
                      int32_t *actions_dev_scratch, int spawn, int stable_max,
                      int32_t *reward_dev_scratch, int32_t *reward_host, int8_t *obs_host,
                      cgl_stream_t stream);

/* cgl_env_step_host without the final synchronisation: returns as soon as the copies and the step are
 * enqueued on `stream`.  The caller calls cgl_stream_wait(stream) (or any stream synchronisation) before it
 * reads reward_host / obs_host or overwrites actions_host.  Splitting the environments into two groups on two
 * streams overlaps one group's host round trip (result read, next actions, enqueue) with the other group's
 * step -- the usual double-buffered rollout. */
int cgl_env_step_host_async(uint32_t *world_in_dev, uint32_t *world_out_dev, int8_t *stable_dev,
                            uint64_t n_envs, uint32_t side, const int32_t *actions_host,
                            int32_t *actions_dev_scratch, int spawn, int stable_max,
                            int32_t *reward_dev_scratch, int32_t *reward_host, int8_t *obs_host,
                            cgl_stream_t stream);
int cgl_stream_wait(cgl_stream_t stream);

/* ---- host-driven rollout: the training loop's env side with the host out of the GPU's way -----------
 * CGL/main.py:64-72 per step: the host hands every env an action (toggle_state, CGL/CGL.py:322-328), steps it
 * (:247-252) and reads its reward (:255-256).  A rollout object owns n_groups GROUPS of envs_per_group environments
 * (resident device planes supplied by the caller) that are stepped alternately, each on its own stream: while one
 * group's step runs the host serves the other -- its rewards are read, `policy` fills its next actions, its next
 * step is enqueued.  The data dependence (an env's next action may depend on its last reward) is kept per group:
 * `policy` is called for a group only after that group's previous step has completed.
 *   per group step   ONE cudaGraphLaunch of [H2D copy of the group's pinned int32 action buffer -> fused env step
 *                    (-> D2H copy of the int8 observation plane if obs_host was given)]; the kernel writes the rewards
 *                    straight into the group's pinned, host-mapped reward buffer; completion is an event the host polls.
 *   n_replicas       every group rotates over n_replicas resident env batches (global step s uses replica s %
 *                    n_replicas): lets a benchmark keep the working set above the L2 size.  1 = a plain rollout.
 *   planes           world_a_dev / world_b_dev / stable_dev: [n_groups * n_replicas] device pointers, index
 *                    group * n_replicas + replica; world_a holds the current world at creation.
 *   obs_host         NULL, or [n_groups] pinned int8 buffers of envs_per_group * side^2 bytes.
 *   flags            CGL_ROLLOUT_ZERO_COPY_ACTIONS: no H2D copy node -- the kernel reads each env's action straight
 *                    from the pinned, host-mapped action buffer over PCIe (one load per env, issued first thing by
 *                    the env's CTA).  Takes the copy engine's latency out of every group step.
 * cgl_rollout_buffers: the group's pinned action (host writes) and reward (host reads) buffers, int32[envs_per_group];
 *                    actions start as side*side ("do nothing").
 * cgl_rollout_run:   `steps` steps of every group.  policy(user, group, step, reward_host, actions_host) may be NULL
 *                    (the action buffers are then used as they are).  Returns when every group has finished.
 * cgl_rollout_parity: 0 if (group, replica)'s current world is in its world_a plane, 1 if in world_b. */
typedef struct cgl_rollout cgl_rollout_t;
typedef void (*cgl_policy_fn)(void *user, uint32_t group, uint64_t step, const int32_t *reward_host,
                              int32_t *actions_host);
#define CGL_ROLLOUT_ZERO_COPY_ACTIONS 1u
int cgl_rollout_create(cgl_rollout_t **out, uint32_t n_groups, uint32_t n_replicas, uint32_t *const *world_a_dev,
                       uint32_t *const *world_b_dev, int8_t *const *stable_dev, uint64_t envs_per_group,
                       uint32_t side, int spawn, int stable_max, int8_t *const *obs_host, uint32_t flags);
int cgl_rollout_buffers(cgl_rollout_t *r, uint32_t group, int32_t **actions_host, int32_t **reward_host);
int cgl_rollout_run(cgl_rollout_t *r, uint64_t steps, cgl_policy_fn policy, void *user);
int cgl_rollout_parity(const cgl_rollout_t *r, uint32_t group, uint32_t replica);
int cgl_rollout_destroy(cgl_rollout_t *r);

/* ---- CUDA IPC helpers for the row-band halo exchange over NVLink (multi-GPU life mode) ----
 * One process per GPU; each rank exports its ghost-row buffer and maps its neighbours'. */
int cgl_ipc_get_handle(void *dev_ptr, uint8_t handle_out[64]);
int cgl_ipc_open_handle(const uint8_t handle[64], void **dev_ptr_out);
int cgl_ipc_close_handle(void *dev_ptr);

/* Push `n_words` from a local buffer into a peer-mapped buffer and then publish `seq` to the
 * peer's flag word (release semantics), in one kernel; the peer waits with cgl_halo_wait. */
int cgl_halo_push(const uint32_t *src_dev, uint32_t *peer_dst_dev, uint64_t n_words,
                  uint32_t *peer_flag_dev, uint32_t seq, cgl_stream_t stream);
/* Block the stream until *flag_dev >= seq (written by a peer GPU). */
int cgl_halo_wait(const uint32_t *flag_dev, uint32_t seq, cgl_stream_t stream);
/* The whole exchange of one rank in ONE launch (2 CTAs: one per ring neighbour): push my top rows
 * to the upper neighbour's landing slot and my bottom rows to the lower one's, publish `seq`, wait
 * for their strips of the same block and move them into my ghost rows. */
int cgl_halo_exchange(const uint32_t *top_src_dev, const uint32_t *bot_src_dev, uint32_t *peer_up_landing,
                      uint32_t *peer_dn_landing, uint32_t *peer_up_flag, uint32_t *peer_dn_flag,
                      const uint32_t *my_landing_up, const uint32_t *my_landing_dn, const uint32_t *my_flag_up,
                      const uint32_t *my_flag_dn, uint32_t *ghost_up_dev, uint32_t *ghost_dn_dev,
                      uint64_t n_words, uint32_t seq, cgl_stream_t stream);
/* Same wait, then copy n_words from the landing zone `src_dev` into the ghost rows `dst_dev`. */
int cgl_halo_wait_copy(const uint32_t *flag_dev, uint32_t seq, const uint32_t *src_dev, uint32_t *dst_dev,
                       uint64_t n_words, cgl_stream_t stream);
/* One row-band block with the halo exchange FUSED into the generation kernel (multi-GPU life mode).
 * The band buffer holds `ghost` ghost rows, the owned rows, `ghost` ghost rows.  Runs `gens`
 * (<= ghost; 1,2,3,4,6,8,12 or 16) generations in -> out in one launch; the kernel writes this
 * rank's first/last `ghost` owned rows straight into the ring neighbours' OUTPUT buffers
 * (peer_up_out / peer_dn_out: CUDA-IPC mapped, same layout) and bumps their arrival counters
 * (peer_*_ctr: uint32[2] = {from_above, from_below}); strips that read ghost rows first wait on
 * my_ctr until both neighbours completed block_index - 1.  block_index = 1 for the first block after
 * the ghosts were filled by a plain exchange (counters zeroed), then 2, 3, ...  No extra launch, no
 * host synchronisation, interior strips never wait. */
int cgl_life_band_block(const uint32_t *in_dev, uint32_t *out_dev, uint32_t buf_rows, uint32_t cols,
                        uint32_t ghost, uint32_t gens, uint32_t *peer_up_out, uint32_t *peer_dn_out,
                        uint32_t *peer_up_ctr, uint32_t *peer_dn_ctr, const uint32_t *my_ctr,
                        uint32_t block_index, cgl_stream_t stream);

/* Row-band run with the halo exchange INSIDE the kernel (the default multi-GPU path of life mode): n_sub sub-steps
 * of k generations (k = 4, 8 or 16; ghost a multiple of k) over this rank's band buffers (ghost rows, owned rows,
 * ghost rows; buf_a holds the current state, the result is in buf_a if n_sub is even, else in buf_b) in ONE
 * cooperative launch -- a warp keeps its strip of rows for the whole call and waits only for its neighbour strips.
 * Every ghost / k sub-steps (a "block") and after the last sub-step, the strips that own the first / last `ghost`
 * owned rows store them into the ring neighbours' landing zones (peer_*_landing[slot], CUDA-IPC mapped, ghost x
 * cols/32 words each, slot = block & 1) and bump their arrival counters (peer_*_ctr); at the start of a block the
 * strips that read ghost rows wait on my_ctr_* and copy what they will read from my_landing_*[slot] into the
 * band buffer.  Interior strips never wait for another GPU.
 *   block_index   blocks (= pushes) consumed by earlier calls since the counters were zeroed; the caller adds
 *                 ceil(n_sub / (ghost / k)) after each call.
 *   initial_push  1 on a fresh grid (counters zeroed, block_index 0): the edge rows of buf_a are pushed before the
 *                 first sub-step.  With n_sub = 0 the call only pushes.
 * Bounded waits: a neighbour that never delivers raises alarm word 3, the kernel stores nothing further and ends.
 * cgl_life_band_run_supported: 1 if a band of this shape fits a cooperative launch on the current device. */
int cgl_life_band_run(uint32_t *buf_a_dev, uint32_t *buf_b_dev, uint32_t buf_rows, uint32_t cols, uint32_t ghost,
                      uint32_t k, uint32_t n_sub, uint32_t block_index, int initial_push,
                      uint32_t *const peer_up_landing[2], uint32_t *const peer_dn_landing[2], uint32_t *peer_up_ctr,
                      uint32_t *peer_dn_ctr, const uint32_t *const my_landing_up[2],
                      const uint32_t *const my_landing_dn[2], const uint32_t *my_ctr_up, const uint32_t *my_ctr_dn,
                      cgl_stream_t stream);
int cgl_life_band_run_supported(uint32_t buf_rows, uint32_t cols, uint32_t k);

/* Plain cudaMalloc'ed (zero-filled) device memory: IPC handles need whole allocations, which
 * a caching allocator's sub-blocks are not. */
int cgl_dev_alloc(uint64_t bytes, void **dev_ptr_out);
int cgl_dev_free(void *dev_ptr);
int cgl_dev_memset(void *dev_ptr, int value, uint64_t bytes, cgl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CGL_B200_H */
