"""Batched DQN loop around BatchedSim -- SURVEY.md section 8 row f1 (the caller of the env step).

The reference trains ONE environment per process: every step `DQNAgent.select_action`
(/root/reference/CGL/dqn.py:127-134) moves the observation host -> device and runs the Q network twice,
and `ExperienceReplay.add` (:24-36) copies state and next_state (2 x side^2 bytes) into the buffer
through four `torch.tensor(...)` host round trips.  Once the env step costs microseconds that loop is
>99 % agent and copy time, so the B200-native loop is organised around the data instead:

  * TrajectoryReplay: the replay memory IS the environments' trajectory.  One int8 ring
    obs[slot, env, cell] in HBM; the env kernel reads slot t and writes its next observation straight into
    slot t+1 (`BatchedSim.step(obs_out=...)` -> `cgl_env_step_io`), rewards land in reward[t] the same
    way.  A transition is the index pair (t, env): state = obs[t, env], next_state = obs[t+1, env].
    Recording a step therefore moves no bytes at all (the reference moves 2 x size per env step, as
    much as the step itself reads and writes), and the ring holds each observation once, not twice.
  * select_action for all B environments is one Q forward ([B, size] int8 -> [B, size+1]), argmax and
    the epsilon-greedy draw on the device; nothing returns to the host inside the loop.
  * learn / target_update follow dqn.py:137-172 operation for operation (plain torch: the networks are
    library GEMMs, not part of the hot path).

Same hyper-parameters and update schedule as `DQNAgent` (dqn.py:63-124): `step()` records, learns once
the memory holds more than `batch_size` transitions, and soft-updates the target network inside `learn`
and again every `update_freq` steps.  What "one step" means changes from one transition to B transitions.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F


class QNetwork(nn.Module):
    """state -> Q values, the reference's three-layer MLP (dqn.py:41-59): hidden width 2*action_dim unless
    `hidden` is given.  int8 observations are widened to float32 on entry (dqn.py:56)."""

    def __init__(self, state_dim: int, action_dim: int, hidden: int | None = None, device=None):
        super().__init__()
        hidden = action_dim * 2 if hidden is None else hidden
        self.l1 = nn.Linear(state_dim, hidden, device=device)
        self.l2 = nn.Linear(hidden, hidden, device=device)
        self.l3 = nn.Linear(hidden, action_dim, device=device)

    def forward(self, state: torch.Tensor) -> torch.Tensor:
        q = F.relu(self.l1(state.to(torch.float32)))
        q = F.relu(self.l2(q))
        return self.l3(q)


class TrajectoryReplay:
    """Replay memory laid out as the trajectory of B lock-stepped environments (see the module docstring).

    `env` is a BatchedSim (or anything with n_envs, size, device, stable, bind_observation(buf),
    step(actions, obs_out=, reward_out=) and reset(); run() also needs run(k, actions=, reward_trace=, obs_trace=)).
    `max_size` counts transitions like the reference's
    `max_size` (dqn.py:12); the ring has ceil(max_size / B) + 1 observation slots.
    """

    def __init__(self, env, max_size: int, batch_size: int, seed: int = 0):
        self.env = env
        self.B, self.state_dim = env.n_envs, env.size
        self.device = torch.device(env.device)
        self.batch_size = batch_size
        self.slots = max(2, -(-max_size // self.B) + 1)
        self.max_size = (self.slots - 1) * self.B
        dev = self.device
        self.obs = torch.empty((self.slots, self.B, self.state_dim), dtype=torch.int8, device=dev)
        self.action = torch.zeros((self.slots, self.B), dtype=torch.int32, device=dev)
        self.reward = torch.zeros((self.slots, self.B), dtype=torch.int32, device=dev)
        self._obs_v, self._act_v, self._rew_v = (list(x.unbind(0)) for x in (self.obs, self.action, self.reward))
        # Ring step k (k = 0, 1, ...) reads obs slot k % slots and writes slot (k+1) % slots.  The last
        # slots-1 ring steps are resident; the ones that were episode boundaries (reset) are "holes".
        # Only the host keeps this bookkeeping: recording a step issues no device work besides the env step.
        self.t = 0                                           # ring steps so far (slot of the live obs = t % slots)
        self._holes: list[int] = []                          # resident ring steps that are not transitions
        self._hadj = None                                    # device tensor of holes[i] - i (see sample_indices)
        self._gen = torch.Generator(device=dev)
        self._gen.manual_seed(seed)
        env.bind_observation(self._obs_v[0])

    # -- bookkeeping ------------------------------------------------------------------------------
    def _window_start(self) -> int:
        lo = max(0, self.t - (self.slots - 1))
        if self._holes and self._holes[0] < lo:
            self._holes = [h for h in self._holes if h >= lo]
            self._hadj = None
        return lo

    def valid_steps(self) -> list[int]:
        """Resident ring steps that are transitions (host-side list, for tests and introspection)."""
        lo = self._window_start()
        holes = set(self._holes)
        return [k for k in range(lo, self.t) if k not in holes]

    @property
    def size(self) -> int:
        """Transitions available to sample() (the reference's `size`, dqn.py:35)."""
        return (self.t - self._window_start() - len(self._holes)) * self.B

    @property
    def state(self) -> torch.Tensor:
        """The live observation int8 [B, size] (what `env.get_stable(shallow=True)` is to main.py:60,70)."""
        return self._obs_v[self.t % self.slots]

    # -- recording --------------------------------------------------------------------------------
    def action_slot(self) -> torch.Tensor:
        """int32 [B] row of the ring where the actions of the NEXT step belong; `select_action(out=...)`
        writes there so that recording the action is free as well."""
        return self._act_v[self.t % self.slots]

    def step(self, actions: torch.Tensor | None):
        """toggle_state(action) + step + reward for every env (main.py:66-71), recorded as B transitions.
        Returns (next_state, reward) = views of the ring."""
        s, n = self.t % self.slots, (self.t + 1) % self.slots
        act = self._act_v[s]
        if actions is None:
            act.fill_(self.state_dim)                         # the reference's "do nothing" index
        elif actions.data_ptr() != act.data_ptr():
            act.copy_(actions.reshape(self.B))
        self.env.step(None if actions is None else act, obs_out=self._obs_v[n], reward_out=self._rew_v[s])
        self.t += 1
        return self._obs_v[n], self._rew_v[s]

    def run(self, actions: torch.Tensor):
        """k ring steps in on-chip env runs (`env.run(k, actions=, reward_trace=, obs_trace=)`): leaves the ring, `t`
        and the env exactly as k calls of step(actions[i]) do.  actions: int32 [k, B] with 1 <= k <= slots - 1.
        The observations go straight into their ring slots, in two runs where the slots wrap the ring end; the
        rewards and actions, whose rows wrap one step earlier, through a [k, B] scratch and at most two copies each.
        Returns (next_state, reward) of the last step = views of the ring."""
        if not isinstance(actions, torch.Tensor) or actions.dim() != 2 or actions.shape[1] != self.B:
            raise TypeError("actions must be an int32 tensor [k, n_envs]")
        k = actions.shape[0]
        if not 1 <= k <= self.slots - 1:
            raise ValueError(f"k = {k} ring steps: 1 <= k <= slots - 1 = {self.slots - 1} are resident")
        actions = actions.contiguous()
        rew = torch.empty((k, self.B), dtype=torch.int32, device=self.device)
        o = (self.t + 1) % self.slots                         # obs slot of step 0's next observation
        k1 = min(k, self.slots - o)
        self.env.run(k1, actions=actions[:k1], reward_trace=rew[:k1], obs_trace=self.obs[o:o + k1])
        if k1 < k:
            self.env.run(k - k1, actions=actions[k1:], reward_trace=rew[k1:], obs_trace=self.obs[:k - k1])
        s = self.t % self.slots                               # action / reward slot of step 0
        j = min(k, self.slots - s)
        self.action[s:s + j].copy_(actions[:j])
        self.reward[s:s + j].copy_(rew[:j])
        if j < k:
            self.action[:k - j].copy_(actions[j:])
            self.reward[:k - j].copy_(rew[j:])
        self.t += k
        last = (self.t - 1) % self.slots
        return self._obs_v[self.t % self.slots], self._rew_v[last]

    def reset(self) -> torch.Tensor:
        """env.reset() (main.py:59) into a fresh slot; the jump from the last observation of the old episode
        to the first of the new one is not a transition and is never sampled."""
        if self.t == 0:
            self.env.reset()
            return self.state
        n = (self.t + 1) % self.slots
        self._holes.append(self.t)
        self._hadj = None
        self.env.bind_observation(self._obs_v[n])
        self.env.reset()
        self.t += 1
        return self._obs_v[n]

    # -- sampling ---------------------------------------------------------------------------------
    def sample_indices(self):
        """(slot, env) of `batch_size` transitions, uniform over the resident ones, drawn on the device.
        The j-th valid ring step is lo + j + #{i : holes[i] - i <= lo + j}; the hole table changes only
        when an episode boundary enters or leaves the window."""
        lo = self._window_start()
        n_valid = self.t - lo - len(self._holes)
        if n_valid <= 0:
            raise RuntimeError("the replay memory is empty")
        k = torch.randint(lo, lo + n_valid, (self.batch_size,), device=self.device, generator=self._gen)
        if self._holes:
            if self._hadj is None:
                self._hadj = torch.tensor([h - i for i, h in enumerate(self._holes)], device=self.device)
            k = k + torch.searchsorted(self._hadj, k, right=True)
        env = torch.randint(0, self.B, (self.batch_size,), device=self.device, generator=self._gen)
        return k % self.slots, env

    def gather(self, slot: torch.Tensor, env: torch.Tensor):
        """The reference's sample() tuple (dqn.py:39-41) for the given transitions: states int8 [n, size],
        actions int32 [n, 1], rewards int32 [n, 1], next_states int8 [n, size]."""
        nxt = (slot + 1) % self.slots
        flat = self.obs.view(self.slots * self.B, self.state_dim)
        return (flat[slot * self.B + env], self.action[slot, env].unsqueeze(1),
                self.reward[slot, env].unsqueeze(1), flat[nxt * self.B + env])

    def sample(self):
        return self.gather(*self.sample_indices())


class BatchedDQNAgent:
    """`DQNAgent` (dqn.py:61-177) for B environments stepped together on one device."""

    def __init__(self, env, discount: float = 0.99, tau: float = 1e-3, lr: float = 5e-4, update_freq: int = 4,
                 max_size: int = int(1e5), batch_size: int = 64, seed: int = 0, hidden: int | None = None,
                 act_dtype: torch.dtype | None = None, group=None):
        self.env = env
        # Data parallel over GPUs (SURVEY.md section 8e): every rank owns a shard of the environments
        # (BatchedSim.shard) and of the replay ring; the only exchange is the gradient all-reduce in learn().
        # group: a torch.distributed process group, or True for the default group.  All ranks must pass the
        # same seed (identical initial weights); exploration and sampling streams are offset by the rank.
        self.group = None
        self.world_size, self.rank = 1, 0
        if group is not None and group is not False:
            import torch.distributed as dist
            self.group = dist.group.WORLD if group is True else group
            self.world_size, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        # act_dtype (opt-in, e.g. torch.bfloat16): run the ACTING forward of select_action in that type on the
        # tensor cores (weights are re-cast from the fp32 master copy each call).  The reference acts in fp32
        # (dqn.py:56 and its "can change this to float16" note); near-ties of Q may then pick another action.
        self.act_dtype = act_dtype
        self.device = torch.device(env.device)
        self.state_dim, self.action_dim = env.size, env.size + 1          # get_state_dim / get_action_space_dim
        self.discount, self.tau, self.lr = float(discount), float(tau), float(lr)
        self.update_freq, self.batch_size = update_freq, batch_size
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(seed + 7919 * self.rank)
        # weight init, reproducible per seed, without disturbing the caller's CPU or CUDA generators
        with torch.random.fork_rng(devices=[self.device] if self.device.type == "cuda" else []):
            torch.manual_seed(seed)
            self.Q = QNetwork(self.state_dim, self.action_dim, hidden, self.device)
            self.Q_target = QNetwork(self.state_dim, self.action_dim, hidden, self.device)
        # one multi-tensor launch per update on the GPU (same arithmetic as the reference's optim.Adam)
        self.optimizer = torch.optim.Adam(self.Q.parameters(), lr=self.lr, fused=self.device.type == "cuda")
        self.memory = TrajectoryReplay(env, max_size, batch_size, seed + 7919 * self.rank)
        self.t_train = 0

    # -- acting -------------------------------------------------------------------------------------
    @torch.no_grad()
    def select_action(self, state: torch.Tensor, epsilon: float, out: torch.Tensor | None = None) -> torch.Tensor:
        """Epsilon-greedy for every env (dqn.py:127-134): the greedy action argmax Q(s), and with probability
        epsilon a uniformly random action DIFFERENT from the greedy one (the reference redraws until it
        differs).  state int8 [B, size] -> int32 [B] on the device."""
        if self.act_dtype is None:
            q = self.Q(state)
        else:
            dt = self.act_dtype
            q = state.to(dt)
            for i, layer in enumerate((self.Q.l1, self.Q.l2, self.Q.l3)):
                q = F.linear(q, layer.weight.to(dt), layer.bias.to(dt))
                if i < 2:
                    q = F.relu(q)
        greedy = q.argmax(dim=1)
        B = greedy.shape[0]
        explore = torch.rand(B, device=self.device, generator=self._gen) < epsilon
        other = torch.randint(0, self.action_dim - 1, (B,), device=self.device, generator=self._gen)
        other = other + (other >= greedy).to(other.dtype)
        a = torch.where(explore, other, greedy).to(torch.int32)
        if out is not None:
            out.copy_(a)
            return out
        return a

    def reset(self) -> torch.Tensor:
        return self.memory.reset()

    # -- learning -----------------------------------------------------------------------------------
    def step(self, actions: torch.Tensor | None):
        """Commit the actions, advance every env, record, learn, update the target network
        (main.py:66-72 + dqn.py:110-124).  Returns (next_state, reward) on the device."""
        n_state, reward = self.memory.step(actions)
        self.t_train += 1
        if self.memory.size > self.batch_size:
            self.learn(self.memory.sample(), self.discount)
        if self.t_train % self.update_freq == 0:
            self.target_update(self.Q, self.Q_target, self.tau)
        return n_state, reward

    def learn(self, experiences, discount: float):
        """One TD(0) update on a sampled batch (dqn.py:137-155)."""
        states, actions, rewards, next_states = experiences
        with torch.no_grad():
            max_next_q = self.Q_target(next_states).max(dim=1, keepdim=True)[0]
            target_q = rewards + discount * max_next_q
        q = self.Q(states).gather(1, actions.long())
        loss = F.mse_loss(q, target_q)
        self.optimizer.zero_grad(set_to_none=True)
        loss.backward()
        if self.world_size > 1:                      # mean over ranks == the gradient of the loss over the union batch
            import torch.distributed as dist
            grads = [p.grad for p in self.Q.parameters()]
            work = [dist.all_reduce(g, group=self.group, async_op=True) for g in grads]
            for w in work:
                w.wait()
            torch._foreach_div_(grads, float(self.world_size))
        self.optimizer.step()
        self.target_update(self.Q, self.Q_target, self.tau)
        return loss.detach()

    @torch.no_grad()
    def target_update(self, Q: nn.Module, Q_target: nn.Module, tau: float) -> None:
        """param_target = tau * param_Q + (1 - tau) * param_target (dqn.py:158-172), all tensors in two
        multi-tensor launches."""
        tgt = list(Q_target.parameters())
        src = list(Q.parameters())
        torch._foreach_mul_(tgt, 1.0 - tau)
        torch._foreach_add_(tgt, src, alpha=tau)

    def save(self, name: str = "unnamed") -> None:
        """dqn.py:175-177."""
        torch.save(self.Q.state_dict(), f"Q_{name}.pth")
        torch.save(self.Q_target.state_dict(), f"Q_target_{name}.pth")
