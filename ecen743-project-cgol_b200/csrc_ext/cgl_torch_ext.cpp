// cgl_torch_ext.cpp -- the thin PyTorch C++ extension over the C ABI (include/cgl_b200.h).
//
// What the reference does between numpy and its kernel (/root/reference/CGL/CGL.py:203-208: two H2D copies, the
// launch, two D2H copies) is, on the torch side of this build, a function that takes CUDA tensors, checks them,
// picks up torch's current stream and calls libcgl_b200.so.  No arithmetic happens here: every function below is
// argument checking + one C-ABI call, so the C ABI stays the one boundary (INTEGRATION.md) and this file is the
// torch-typed face of it:
//   env_step       toggle + generation + int8 stability + reward for a batch          -> cgl_env_step_ex
//   env_run        k plain steps / run-until-fixed in one launch                       -> cgl_env_run_rule
//   env_run_ex     the same with an action schedule and per-step reward / alive traces -> cgl_env_run_ex
//                  and, with obs_trace, the observation after every step               -> cgl_env_run_obs
//                  or, with max_period, until the world repeats one of its last P     -> cgl_env_run_cycle
//                  or, with until_settled, until the world repeats any earlier world   -> cgl_env_run_settle
//   env_action_rewards  every action's next-step reward and the greedy action per env  -> cgl_env_action_rewards
//   pack / unpack  uint8 cells <-> bit-packed world at the API boundary                -> cgl_pack / cgl_unpack
//   reward / alive the reference's reductions (CGL/CGL.py:255-260)                     -> cgl_reward / cgl_alive
//   life_run       world-only generations (life mode)                                  -> cgl_life_run
//   life_run_pop   the same, recording the population after every generation           -> cgl_life_run_pop
// cgl_b200/batched.py uses env_step for BatchedSim.step when the tensors are plain (the struct-cached ctypes path
// serves the rest), tests/test_gpu_torch_ext.py checks every function against the ctypes binding.
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include "../../include/cgl_b200.h"

namespace {

void check_rc(int rc, const char *what)
{
    TORCH_CHECK(rc == 0, what, " failed (rc=", rc, "): ", cgl_last_error());
}

void check_cuda(const at::Tensor &t, at::ScalarType dtype, const char *name)
{
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (there is no CPU path)");
    TORCH_CHECK(t.scalar_type() == dtype, name, " has the wrong dtype");
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}

cgl_stream_t stream_of(const at::Tensor &t)
{
    return static_cast<cgl_stream_t>(c10::cuda::getCurrentCUDAStream(t.get_device()).stream());
}

template <class T>
T *ptr(const c10::optional<at::Tensor> &t)
{
    return t.has_value() ? static_cast<T *>(t->data_ptr()) : nullptr;
}

// One env step for n_envs environments.  world_in / world_out: int32 [n_envs, side, W] (bit-packed uint32 words);
// stable_in / stable_out: int8 [n_envs, side*side] (may be the same tensor); actions: int32 [n_envs] or None.
// chain_mode 0: stream order; 1: plane-id tokens (want / publish); 2: sequence-number tokens (want = seq).
void env_step(const at::Tensor &world_in, const at::Tensor &world_out, const at::Tensor &stable_in,
              const at::Tensor &stable_out, const c10::optional<at::Tensor> &actions,
              const c10::optional<at::Tensor> &reward_out, const c10::optional<at::Tensor> &alive_out,
              const c10::optional<at::Tensor> &err_flag, const c10::optional<at::Tensor> &tokens, int64_t side,
              int64_t spawn, int64_t stable_max, int64_t dead_rule, int64_t empty, int64_t empty_min, bool masked_toggle,
              int64_t chain_mode, int64_t want, int64_t publish)
{
    check_cuda(world_in, at::kInt, "world_in");
    check_cuda(world_out, at::kInt, "world_out");
    check_cuda(stable_in, at::kChar, "stable_in");
    check_cuda(stable_out, at::kChar, "stable_out");
    const int64_t size = side * side, W = (side + 31) / 32;
    TORCH_CHECK(side >= 1 && stable_in.numel() % size == 0, "stable_in does not hold whole environments of this side");
    const int64_t n = stable_in.numel() / size;
    TORCH_CHECK(world_in.numel() == n * side * W && world_out.numel() == n * side * W && stable_out.numel() == n * size,
                "plane shapes do not match ", n, " environments of side ", side);
    if (actions) { check_cuda(*actions, at::kInt, "actions"); TORCH_CHECK(actions->numel() == n, "one action per env"); }
    if (reward_out) { check_cuda(*reward_out, at::kInt, "reward_out"); TORCH_CHECK(reward_out->numel() == n, "one reward per env"); }
    if (alive_out) { check_cuda(*alive_out, at::kInt, "alive_out"); TORCH_CHECK(alive_out->numel() == n, "one count per env"); }
    if (err_flag) check_cuda(*err_flag, at::kInt, "err_flag");
    if (tokens) { check_cuda(*tokens, at::kInt, "tokens"); TORCH_CHECK(tokens->numel() == n, "one token per env"); }
    TORCH_CHECK(chain_mode == 0 || tokens.has_value(), "chained steps need tokens");
    c10::cuda::CUDAGuard guard(world_in.device());
    cgl_env_step_args_t a = {};
    a.world_in_dev = static_cast<uint32_t *>(world_in.data_ptr());
    a.world_out_dev = static_cast<uint32_t *>(world_out.data_ptr());
    a.stable_in_dev = static_cast<const int8_t *>(stable_in.data_ptr());
    a.stable_out_dev = static_cast<int8_t *>(stable_out.data_ptr());
    a.n_envs = (uint64_t)n;
    a.side = (uint32_t)side;
    a.spawn = (int32_t)spawn; a.stable_max = (int32_t)stable_max; a.dead_rule = (int32_t)dead_rule;
    a.empty = (int32_t)empty; a.empty_min = (int32_t)empty_min; a.masked_toggle = masked_toggle ? 1 : 0;
    a.actions_dev = ptr<const int32_t>(actions);
    a.reward_out_dev = ptr<int32_t>(reward_out);
    a.alive_out_dev = ptr<uint32_t>(alive_out);
    a.err_flag_dev = ptr<int>(err_flag);
    a.token_dev = ptr<uint32_t>(tokens);
    a.chain_mode = (uint32_t)chain_mode; a.want = (uint32_t)want; a.publish = (uint32_t)publish;
    check_rc(cgl_env_step_ex(&a, stream_of(world_in)), "cgl_env_step_ex");
}

// max_steps plain steps (optionally until the world stops changing) in one launch; world updated in place.
// Returns steps executed per env (int32 [n_envs]).
at::Tensor env_run(const at::Tensor &world, const at::Tensor &stable, int64_t side, int64_t max_steps, bool until_fixed,
                   int64_t spawn, int64_t stable_max, int64_t dead_rule, int64_t empty, int64_t empty_min,
                   const c10::optional<at::Tensor> &reward_out, const c10::optional<at::Tensor> &alive_out)
{
    check_cuda(world, at::kInt, "world");
    check_cuda(stable, at::kChar, "stable");
    const int64_t size = side * side;
    TORCH_CHECK(side >= 1 && stable.numel() % size == 0 && max_steps >= 0, "bad shape");
    const int64_t n = stable.numel() / size;
    c10::cuda::CUDAGuard guard(world.device());
    at::Tensor steps = at::empty({n}, world.options().dtype(at::kInt));
    check_rc(cgl_env_run_rule(static_cast<const uint32_t *>(world.data_ptr()), static_cast<uint32_t *>(world.data_ptr()),
                              static_cast<int8_t *>(stable.data_ptr()), (uint64_t)n, (uint32_t)side, (uint32_t)max_steps,
                              until_fixed ? 1 : 0, (int)spawn, (int)stable_max, (int)dead_rule, (int)empty, (int)empty_min,
                              static_cast<int32_t *>(steps.data_ptr()), ptr<int32_t>(reward_out), ptr<uint32_t>(alive_out),
                              stream_of(world)),
             "cgl_env_run_rule");
    return steps;
}

// env_run with an action schedule (int32 [max_steps, n_envs]) and per-step traces (int32 [max_steps, n_envs], row t
// = after step t), each optional; masked_toggle and err_flag (int32 [1]) as in env_step.  obs_trace (int8
// [max_steps, n_envs, side*side]) receives the stability plane after every step; `stable` is then read only.
// max_period (1..CGL_RUN_MAX_PERIOD) stops each env when its world repeats one of its last max_period worlds; period
// (int32 [n_envs], optional) receives the cycle length or 0.  It takes no until_fixed, actions or obs_trace.
// until_settled stops each env at its first repeated world of any period; period receives that period or 0.  It
// takes no max_period, until_fixed, actions or obs_trace.
// Returns steps per env.
at::Tensor env_run_ex(const at::Tensor &world, const at::Tensor &stable, int64_t side, int64_t max_steps,
                      bool until_fixed, int64_t spawn, int64_t stable_max, int64_t dead_rule, int64_t empty,
                      int64_t empty_min, bool masked_toggle, const c10::optional<at::Tensor> &actions,
                      const c10::optional<at::Tensor> &reward_trace, const c10::optional<at::Tensor> &alive_trace,
                      const c10::optional<at::Tensor> &reward_out, const c10::optional<at::Tensor> &alive_out,
                      const c10::optional<at::Tensor> &err_flag, const c10::optional<at::Tensor> &obs_trace,
                      int64_t max_period, const c10::optional<at::Tensor> &period, bool until_settled)
{
    check_cuda(world, at::kInt, "world");
    check_cuda(stable, at::kChar, "stable");
    const int64_t size = side * side;
    TORCH_CHECK(side >= 1 && stable.numel() % size == 0 && max_steps >= 0, "bad shape");
    const int64_t n = stable.numel() / size;
    const std::pair<const c10::optional<at::Tensor> *, const char *> sched[3] = {
        {&actions, "actions"}, {&reward_trace, "reward_trace"}, {&alive_trace, "alive_trace"}};
    for (const auto &p : sched) {
        if (!p.first->has_value()) continue;
        check_cuda(**p.first, at::kInt, p.second);
        TORCH_CHECK((*p.first)->dim() == 2 && (*p.first)->size(0) == max_steps && (*p.first)->size(1) == n, p.second,
                    " must be [max_steps, n_envs]");
    }
    if (reward_out.has_value()) check_cuda(*reward_out, at::kInt, "reward_out");
    if (alive_out.has_value()) check_cuda(*alive_out, at::kInt, "alive_out");
    if (err_flag.has_value()) check_cuda(*err_flag, at::kInt, "err_flag");
    if (obs_trace.has_value()) {
        check_cuda(*obs_trace, at::kChar, "obs_trace");
        TORCH_CHECK(obs_trace->dim() == 3 && obs_trace->size(0) == max_steps && obs_trace->size(1) == n &&
                        obs_trace->size(2) == size,
                    "obs_trace must be [max_steps, n_envs, side*side]");
        TORCH_CHECK(obs_trace->device() == world.device(), "obs_trace must be on the world's device");
    }
    TORCH_CHECK(max_period >= 0 && max_period <= CGL_RUN_MAX_PERIOD, "max_period must be in 0..", CGL_RUN_MAX_PERIOD);
    TORCH_CHECK(max_period == 0 || (!until_fixed && !actions.has_value() && !obs_trace.has_value()),
                "max_period replaces until_fixed and takes no actions or obs_trace");
    TORCH_CHECK(!until_settled || (max_period == 0 && !until_fixed && !actions.has_value() && !obs_trace.has_value()),
                "until_settled takes no max_period, until_fixed, actions or obs_trace");
    if (period.has_value()) {
        TORCH_CHECK(max_period > 0 || until_settled, "period needs max_period or until_settled");
        check_cuda(*period, at::kInt, "period");
        TORCH_CHECK(period->numel() == n, "one period per env");
        TORCH_CHECK(period->device() == world.device(), "period must be on the world's device");
    }
    c10::cuda::CUDAGuard guard(world.device());
    at::Tensor steps = at::empty({n}, world.options().dtype(at::kInt));
    cgl_env_run_obs_args_t o = {};
    cgl_env_run_args_t &a = o.run;
    a.world_in_dev = static_cast<const uint32_t *>(world.data_ptr());
    a.world_out_dev = static_cast<uint32_t *>(world.data_ptr());
    a.stable_dev = static_cast<int8_t *>(stable.data_ptr());
    a.n_envs = (uint64_t)n; a.side = (uint32_t)side; a.max_steps = (uint32_t)max_steps;
    a.stop_when_fixed = until_fixed ? 1 : 0; a.spawn = (int32_t)spawn; a.stable_max = (int32_t)stable_max;
    a.dead_rule = (int32_t)dead_rule; a.empty = (int32_t)empty; a.empty_min = (int32_t)empty_min;
    a.masked_toggle = masked_toggle ? 1 : 0;
    a.actions_dev = ptr<const int32_t>(actions);
    a.reward_trace_dev = ptr<int32_t>(reward_trace);
    a.alive_trace_dev = ptr<uint32_t>(alive_trace);
    a.steps_out_dev = static_cast<int32_t *>(steps.data_ptr());
    a.reward_out_dev = ptr<int32_t>(reward_out);
    a.alive_out_dev = ptr<uint32_t>(alive_out);
    a.err_flag_dev = ptr<int>(err_flag);
    o.obs_trace_dev = ptr<int8_t>(obs_trace);
    if (until_settled)
        check_rc(cgl_env_run_settle(&a, ptr<int32_t>(period), stream_of(world)), "cgl_env_run_settle");
    else if (max_period > 0)
        check_rc(cgl_env_run_cycle(&a, (uint32_t)max_period, ptr<int32_t>(period), stream_of(world)), "cgl_env_run_cycle");
    else if (obs_trace.has_value()) check_rc(cgl_env_run_obs(&o, stream_of(world)), "cgl_env_run_obs");
    else check_rc(cgl_env_run_ex(&a, stream_of(world)), "cgl_env_run_ex");
    return steps;
}

// The reward every action would give (rewards_out int32 [n_envs, side*side + 1]) and / or the greedy action and its
// reward (best_action_out, best_reward_out: int32 [n_envs]); at least one output.  world / stable are only read.
void env_action_rewards(const at::Tensor &world, const at::Tensor &stable, int64_t side, int64_t spawn,
                        int64_t stable_max, int64_t dead_rule, int64_t empty, int64_t empty_min, bool masked_toggle,
                        const c10::optional<at::Tensor> &rewards_out, const c10::optional<at::Tensor> &best_action_out,
                        const c10::optional<at::Tensor> &best_reward_out)
{
    check_cuda(world, at::kInt, "world");
    check_cuda(stable, at::kChar, "stable");
    const int64_t size = side * side, W = (side + 31) / 32;
    TORCH_CHECK(side >= 1 && stable.numel() % size == 0 && stable.numel() > 0, "stable does not hold whole environments");
    const int64_t n = stable.numel() / size;
    TORCH_CHECK(world.numel() == n * side * W, "world does not match ", n, " environments of side ", side);
    TORCH_CHECK(world.device() == stable.device(), "world and stable must be on the same device");
    const std::pair<const c10::optional<at::Tensor> *, const char *> outs[3] = {
        {&rewards_out, "rewards_out"}, {&best_action_out, "best_action_out"}, {&best_reward_out, "best_reward_out"}};
    for (const auto &o : outs) {
        if (!o.first->has_value()) continue;
        check_cuda(**o.first, at::kInt, o.second);
        TORCH_CHECK((*o.first)->device() == world.device(), o.second, " must be on the world's device");
    }
    if (rewards_out) TORCH_CHECK(rewards_out->numel() == n * (size + 1), "rewards_out must be [n_envs, side*side + 1]");
    if (best_action_out) TORCH_CHECK(best_action_out->numel() == n, "one best action per env");
    if (best_reward_out) TORCH_CHECK(best_reward_out->numel() == n, "one best reward per env");
    c10::cuda::CUDAGuard guard(world.device());
    cgl_env_action_rewards_args_t a = {};
    a.world_dev = static_cast<const uint32_t *>(world.data_ptr());
    a.stable_dev = static_cast<const int8_t *>(stable.data_ptr());
    a.n_envs = (uint64_t)n; a.side = (uint32_t)side;
    a.spawn = (int32_t)spawn; a.stable_max = (int32_t)stable_max; a.dead_rule = (int32_t)dead_rule;
    a.empty = (int32_t)empty; a.empty_min = (int32_t)empty_min; a.masked_toggle = masked_toggle ? 1 : 0;
    a.rewards_out_dev = ptr<int32_t>(rewards_out);
    a.best_action_out_dev = ptr<int32_t>(best_action_out);
    a.best_reward_out_dev = ptr<int32_t>(best_reward_out);
    check_rc(cgl_env_action_rewards(&a, stream_of(world)), "cgl_env_action_rewards");
}

// uint8 cells [n_envs, rows*cols] (nonzero = alive) -> int32 [n_envs, rows, W] packed words.
at::Tensor pack(const at::Tensor &cells, int64_t rows, int64_t cols)
{
    check_cuda(cells, at::kByte, "cells");
    TORCH_CHECK(rows >= 1 && cols >= 1 && cells.numel() % (rows * cols) == 0, "cells do not hold whole grids");
    const int64_t n = cells.numel() / (rows * cols), W = (cols + 31) / 32;
    c10::cuda::CUDAGuard guard(cells.device());
    at::Tensor world = at::empty({n, rows, W}, cells.options().dtype(at::kInt));
    check_rc(cgl_pack(static_cast<const uint8_t *>(cells.data_ptr()), static_cast<uint32_t *>(world.data_ptr()), (uint64_t)n,
                      (uint32_t)rows, (uint32_t)cols, stream_of(cells)),
             "cgl_pack");
    return world;
}

at::Tensor unpack(const at::Tensor &world, int64_t rows, int64_t cols)
{
    check_cuda(world, at::kInt, "world");
    const int64_t W = (cols + 31) / 32;
    TORCH_CHECK(rows >= 1 && cols >= 1 && world.numel() % (rows * W) == 0, "world does not hold whole grids");
    const int64_t n = world.numel() / (rows * W);
    c10::cuda::CUDAGuard guard(world.device());
    at::Tensor cells = at::empty({n, rows * cols}, world.options().dtype(at::kByte));
    check_rc(cgl_unpack(static_cast<const uint32_t *>(world.data_ptr()), static_cast<uint8_t *>(cells.data_ptr()),
                        (uint64_t)n, (uint32_t)rows, (uint32_t)cols, stream_of(world)),
             "cgl_unpack");
    return cells;
}

at::Tensor reward(const at::Tensor &stable, int64_t size)
{
    check_cuda(stable, at::kChar, "stable");
    TORCH_CHECK(size >= 1 && stable.numel() % size == 0, "stable does not hold whole environments");
    const int64_t n = stable.numel() / size;
    c10::cuda::CUDAGuard guard(stable.device());
    at::Tensor out = at::empty({n}, stable.options().dtype(at::kInt));
    check_rc(cgl_reward(static_cast<const int8_t *>(stable.data_ptr()), (uint64_t)n, (uint64_t)size,
                        static_cast<int32_t *>(out.data_ptr()), stream_of(stable)),
             "cgl_reward");
    return out;
}

at::Tensor alive(const at::Tensor &world, int64_t words_per_env)
{
    check_cuda(world, at::kInt, "world");
    TORCH_CHECK(words_per_env >= 1 && world.numel() % words_per_env == 0, "world does not hold whole environments");
    const int64_t n = world.numel() / words_per_env;
    c10::cuda::CUDAGuard guard(world.device());
    at::Tensor out = at::empty({n}, world.options().dtype(at::kInt));
    check_rc(cgl_alive(static_cast<const uint32_t *>(world.data_ptr()), (uint64_t)n, (uint64_t)words_per_env,
                       static_cast<uint32_t *>(out.data_ptr()), stream_of(world)),
             "cgl_alive");
    return out;
}

// gens generations of one rows x cols grid, k per HBM pass, ping-ponging a <-> b.  True if the result is in a.
bool life_run(const at::Tensor &a, const at::Tensor &b, int64_t rows, int64_t cols, bool wrap_rows, int64_t gens, int64_t k)
{
    check_cuda(a, at::kInt, "a");
    check_cuda(b, at::kInt, "b");
    const int64_t W = (cols + 31) / 32;
    TORCH_CHECK(a.numel() == rows * W && b.numel() == rows * W, "buffers must hold rows * ceil(cols/32) words");
    c10::cuda::CUDAGuard guard(a.device());
    int in_a = 0;
    check_rc(cgl_life_run(static_cast<uint32_t *>(a.data_ptr()), static_cast<uint32_t *>(b.data_ptr()), (uint32_t)rows,
                          (uint32_t)cols, wrap_rows ? 1 : 0, (uint32_t)gens, (uint32_t)k, &in_a, stream_of(a)),
             "cgl_life_run");
    return in_a != 0;
}

// life_run that also writes pop (int64 [gens]): live cells of rows [count_row0, count_row0 + count_rows) after each
// generation.  True if the result is in a.
bool life_run_pop(const at::Tensor &a, const at::Tensor &b, int64_t rows, int64_t cols, bool wrap_rows, int64_t gens,
                  int64_t k, int64_t count_row0, int64_t count_rows, const at::Tensor &pop)
{
    check_cuda(a, at::kInt, "a");
    check_cuda(b, at::kInt, "b");
    check_cuda(pop, at::kLong, "pop");
    const int64_t W = (cols + 31) / 32;
    TORCH_CHECK(a.numel() == rows * W && b.numel() == rows * W, "buffers must hold rows * ceil(cols/32) words");
    TORCH_CHECK(a.device() == b.device() && pop.device() == a.device(), "a, b and pop must be on the same device");
    TORCH_CHECK(pop.numel() == gens, "pop must hold one count per generation");
    TORCH_CHECK(count_row0 >= 0 && count_rows >= 1 && count_row0 + count_rows <= rows,
                "count window [count_row0, count_row0 + count_rows) must lie inside the rows");
    c10::cuda::CUDAGuard guard(a.device());
    int in_a = 0;
    check_rc(cgl_life_run_pop(static_cast<uint32_t *>(a.data_ptr()), static_cast<uint32_t *>(b.data_ptr()), (uint32_t)rows,
                              (uint32_t)cols, wrap_rows ? 1 : 0, (uint32_t)gens, (uint32_t)k, (uint32_t)count_row0,
                              (uint32_t)count_rows, static_cast<uint64_t *>(pop.data_ptr()), &in_a, stream_of(a)),
             "cgl_life_run_pop");
    return in_a != 0;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m)
{
    m.doc() = "Thin PyTorch C++ extension over libcgl_b200.so (see include/cgl_b200.h)";
    m.def("abi_version", &cgl_abi_version);
    m.def("env_step", &env_step, py::arg("world_in"), py::arg("world_out"), py::arg("stable_in"), py::arg("stable_out"),
          py::arg("actions"), py::arg("reward_out"), py::arg("alive_out"), py::arg("err_flag"), py::arg("tokens"),
          py::arg("side"), py::arg("spawn"), py::arg("stable_max"), py::arg("dead_rule") = 0, py::arg("empty") = 0,
          py::arg("empty_min") = 0, py::arg("masked_toggle") = false, py::arg("chain_mode") = 0, py::arg("want") = 0,
          py::arg("publish") = 0);
    m.def("env_run", &env_run, py::arg("world"), py::arg("stable"), py::arg("side"), py::arg("max_steps"),
          py::arg("until_fixed") = false, py::arg("spawn") = -1, py::arg("stable_max") = 1, py::arg("dead_rule") = 0,
          py::arg("empty") = 0, py::arg("empty_min") = 0, py::arg("reward_out") = py::none(), py::arg("alive_out") = py::none());
    m.def("env_run_ex", &env_run_ex, py::arg("world"), py::arg("stable"), py::arg("side"), py::arg("max_steps"),
          py::arg("until_fixed") = false, py::arg("spawn") = -1, py::arg("stable_max") = 1, py::arg("dead_rule") = 0,
          py::arg("empty") = 0, py::arg("empty_min") = -128, py::arg("masked_toggle") = false,
          py::arg("actions") = py::none(), py::arg("reward_trace") = py::none(), py::arg("alive_trace") = py::none(),
          py::arg("reward_out") = py::none(), py::arg("alive_out") = py::none(), py::arg("err_flag") = py::none(),
          py::arg("obs_trace") = py::none(), py::arg("max_period") = 0, py::arg("period") = py::none(),
          py::arg("until_settled") = false);
    m.def("env_action_rewards", &env_action_rewards, py::arg("world"), py::arg("stable"), py::arg("side"),
          py::arg("spawn") = -1, py::arg("stable_max") = 1, py::arg("dead_rule") = 0, py::arg("empty") = 0,
          py::arg("empty_min") = -128, py::arg("masked_toggle") = false, py::arg("rewards_out") = py::none(),
          py::arg("best_action_out") = py::none(), py::arg("best_reward_out") = py::none());
    m.def("pack", &pack);
    m.def("unpack", &unpack);
    m.def("reward", &reward);
    m.def("alive", &alive);
    m.def("life_run", &life_run);
    m.def("life_run_pop", &life_run_pop, py::arg("a"), py::arg("b"), py::arg("rows"), py::arg("cols"), py::arg("wrap_rows"),
          py::arg("gens"), py::arg("k"), py::arg("count_row0"), py::arg("count_rows"), py::arg("pop"));
}
