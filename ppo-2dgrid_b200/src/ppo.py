"""PPO with device-resident rollouts (reference src/ppo.py:9-175: same constructor, methods, attributes and
update math; only the data path is rewired).

Two rollout paths behind `collect_rollouts()`:
  * a BatchedMerlinEnv (N envs, one fused CUDA launch per step): observations are rendered by the env kernel
    straight into the rollout buffer, the policy is evaluated once per step for all envs, and the rest of the
    transition -- sample the action, its log-probability, the three rollout stores, the env step, the next
    observation -- is ONE launch (`BatchedMerlinEnv.policy_step`, merlin_env_policy_step).  Nothing crosses PCIe and
    nothing synchronises until the rollout is over; optionally the whole T-step loop is replayed from one CUDA
    graph.  `batch_size` = T * N transitions per rollout.
  * the reference's single-env wrapper stack (`ScenarioCreator.create_env`): the same per-step loop as the
    reference (src/ppo.py:64-105), one env, host observations -- kept so existing scripts run unchanged.
GAE always runs in the CUDA kernel (`merlin_b200.gae`).  With `torch.distributed` initialised, every rank rolls
out its own envs and the flattened gradient is all-reduced once per minibatch step (src/parallel.py).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.optim as optim

from merlin_b200 import BatchedMerlinEnv, gae as gae_kernel
from src.metrics.ppo_metrics import aggregate_ppo_update_metrics

from . import parallel
from .actor_critic import CNNActorCritic, MLPActorCritic, RolloutPolicy
from .rollout_buffer import RolloutBuffer


class PPO:
    def __init__(self, env, lr=3e-4, gamma=0.99, lam=0.95, clip_eps=0.2, update_epochs=10, batch_size=2048,
                 minibatch_size=256, vf_coef=0.5, ent_coef=0.01, device="cpu", use_cuda_graph=False,
                 obs_storage="rgb", amp_dtype=None, minibatch_frames=torch.float32, carry_episodes=None,
                 bootstrap_truncated=False):
        self.env = env
        self.batched = isinstance(env, BatchedMerlinEnv)
        # bootstrap_truncated: an episode cut by the step limit is not a terminal state.  Its last reward gets
        # gamma * V(final observation), the critic's value of the state the limit cut off (Stable-Baselines3's time-limit
        # correction); GAE then treats the step as done as before.  False (default) = the reference: value 0.
        if bootstrap_truncated and not self.batched:
            raise ValueError("bootstrap_truncated needs a BatchedMerlinEnv (final observations come from its step kernel)")
        self.bootstrap_truncated = bool(bootstrap_truncated)
        self.device = env.device if self.batched else torch.device(device)
        self.gamma, self.lam, self.clip_eps = gamma, lam, clip_eps
        self.update_epochs, self.batch_size, self.minibatch_size = update_epochs, batch_size, minibatch_size
        self.vf_coef, self.ent_coef = vf_coef, ent_coef
        # optional reduced-precision policy evaluation in the update (torch.autocast); None = fp32 like the reference
        self.amp_dtype = amp_dtype
        # obs_storage='symbolic' only: what the render kernel hands the policy for a minibatch -- the first layer's
        # float32 input tensor itself (default; same values, so the same update bit for bit), or blocked uint8 pixels
        # that PyTorch casts afterwards
        if minibatch_frames not in (torch.float32, torch.uint8):
            raise ValueError("minibatch_frames must be torch.float32 or torch.uint8")
        self.minibatch_frames = minibatch_frames

        if obs_storage not in ("rgb", "symbolic"):
            raise ValueError("obs_storage must be 'rgb' (56x56x3 frames in the rollout) or 'symbolic' (7x7x3, expanded on read)")
        self.obs_storage = obs_storage if self.batched else "rgb"
        if self.batched:
            self.num_envs = env.num_envs
            act_dim = env.n_actions
            self.use_cnn, self.obs_shape = True, tuple(env.obs.shape[1:])
            if self.obs_storage == "symbolic" and env.obs_symbolic is None:
                raise ValueError("obs_storage='symbolic' needs an env created with want_symbolic=True")
        else:
            self.num_envs = 1
            sample_obs, _ = env.reset()
            act_dim = env.action_space.n
            self.use_cnn = sample_obs.ndim != 1
            self.obs_shape = tuple(sample_obs.shape) if self.use_cnn else (int(np.prod(sample_obs.shape)),)
        if self.use_cnn:
            self.ac = CNNActorCritic(self.obs_shape, act_dim).to(self.device)
        else:
            self.ac = MLPActorCritic(self.obs_shape[0], act_dim).to(self.device)
        parallel.broadcast_parameters(self.ac)
        self.optimizer = optim.Adam(self.ac.parameters(), lr=lr)
        self._grads = parallel.FlatGrads(self.ac.parameters()) if parallel.world_size() > 1 else None

        # 'symbolic': the rollout keeps the 147-byte Grid.encode image per step (64x smaller than the frame); minibatches
        # are rendered on read by merlin_env_render, straight into the blocked layout the first conv layer consumes
        stored_shape = (7, 7, 3) if self.obs_storage == "symbolic" else self.obs_shape
        self.buffer = RolloutBuffer(buffer_size=self.batch_size, obs_shape=stored_shape, device=self.device,
                                    is_discrete=True, num_envs=self.num_envs,
                                    obs_dtype=torch.uint8 if self.batched else torch.float32)
        self.episode_returns = []
        self.episode_lengths = []

        if self.batched:
            T, N = self.buffer.horizon, self.num_envs
            if self.obs_storage == "symbolic":
                self._last_sym = torch.zeros((N, 7, 7, 3), dtype=torch.uint8, device=self.device)
                self._policy_in = torch.zeros((N, 14, 14, 48), dtype=torch.float32, device=self.device)
                self._mb_frames = torch.zeros((min(self.minibatch_size, self.batch_size), 14, 14, 48),
                                              dtype=self.minibatch_frames, device=self.device)
            else:
                self._last_obs = torch.zeros((N,) + self.obs_shape, dtype=torch.uint8, device=self.device)
            self._ep_ret = torch.zeros((T, N), dtype=torch.float32, device=self.device)
            self._ep_len = torch.zeros((T, N), dtype=torch.int32, device=self.device)
            self._last_value = torch.zeros(N, dtype=torch.float32, device=self.device)
            # the step kernel writes reward / done / episode statistics of step t straight into row t of these tensors
            scratch = {k: torch.zeros(N, dtype=torch.bool, device=self.device) for k in ("terminated", "truncated", "stuck")}
            if self.bootstrap_truncated:
                # per-step flags, and the final observation of every episode that ends (u8[T, N, 7, 7, 3])
                self._terminated = torch.zeros((T, N), dtype=torch.bool, device=self.device)
                self._truncated = torch.zeros((T, N), dtype=torch.bool, device=self.device)
                self._final_sym = torch.zeros((T, N, 7, 7, 3), dtype=torch.uint8, device=self.device)
                self._boot_in = torch.zeros((min(self.minibatch_size, T * N), 14, 14, 48), dtype=torch.float32,
                                            device=self.device)

            def row(x, t):
                return x[t] if x.dim() == 2 else x[t:t + 1]
            def flags(t):
                if not self.bootstrap_truncated:
                    return scratch
                return dict(scratch, terminated=self._terminated[t], truncated=self._truncated[t])
            self._rows = [env.make_step_buffers(reward=row(self.buffer.rewards, t), done=row(self.buffer.dones, t),
                                                episode_return=self._ep_ret[t], episode_length=self._ep_len[t],
                                                **flags(t))
                          for t in range(T)]
            # one fused transition per step: logits / value of step t -> action, log-probability, value rows of the buffer
            self._heads = torch.zeros((2, N, act_dim), dtype=torch.float32, device=self.device)
            self._ios = [env.make_policy_io(self._heads[0], self._heads[1, :, 0], action=row(self.buffer.actions, t),
                                            logprob=row(self.buffer.logprobs, t), value_out=row(self.buffer.values, t))
                         for t in range(T)]
            self._rollout_policy = None
        # carry_episodes: a rollout continues the episodes the previous one left unfinished (the usual vectorised-PPO
        # regime) instead of starting from a fresh reset() like the reference's single-env loop (src/ppo.py:65).  With a
        # horizon shorter than the episode cap a fresh reset per rollout would only ever show the policy the first T steps
        # of an episode and would log only the episodes that finished within T steps.  None = automatic: carry exactly then.
        if carry_episodes is None:
            carry_episodes = self.batched and self.buffer.horizon < env.max_steps
        self.carry_episodes = bool(carry_episodes) and self.batched
        self._started = False
        self.unfinished_episodes = 0   # envs in the middle of an episode when the last rollout ended
        self.use_cuda_graph = bool(use_cuda_graph) and self.batched
        self._graph = None

    # ---- helpers ------------------------------------------------------------------------------------------
    def _obs_to_tensor(self, state):
        state_t = torch.as_tensor(state, device=self.device).to(torch.float32)
        return state_t.unsqueeze(0) if self.use_cnn else state_t.view(1, -1)

    def _gae_device(self):
        return self.device if self.device.type == "cuda" else torch.device("cuda", torch.cuda.current_device())

    # ---- rollouts -----------------------------------------------------------------------------------------
    def collect_rollouts(self):
        """One rollout of `batch_size` transitions; returns the bootstrap value (`float` for a single env, a
        `[N]` device tensor for a batched env).  The single-env path starts from a fresh `reset()` like the reference;
        the batched path continues unfinished episodes when `carry_episodes` (see __init__)."""
        return self._collect_batched() if self.batched else self._collect_single()

    def _logits_value_into_heads(self, x, lean):
        """Policy outputs for `x` written to the static `[2, N, A]` head tensor the fused transitions read."""
        if lean:
            if x.dtype == torch.uint8:  # stored frames [N, 56, 56, 3]: to the blocked float layout the fused network reads
                n = x.shape[0]
                x = x.reshape(n, 14, 4, 14, 4, 3).permute(0, 1, 3, 5, 2, 4).reshape(n, 14, 14, 48).float()
            self._rollout_policy(x, out=self._heads)
        else:
            logits, value = self.ac(x)
            self._heads[0].copy_(logits)
            self._heads[1, :, 0].copy_(value)

    def _rollout_body(self, fresh):
        env, buf, T = self.env, self.buffer, self.buffer.horizon
        sym = self.obs_storage == "symbolic"
        lean = self.use_cnn and self.ac.blocked_first_layer
        if lean:
            # the parameters do not change during a rollout: both trunks are packed once into one fused network
            if self._rollout_policy is None:
                self._rollout_policy = RolloutPolicy(self.ac)
            else:
                self._rollout_policy.refresh()
        last = self._last_sym if sym else self._last_obs
        if fresh:
            if sym:
                env.reset(out_symbolic=buf.obs_slot(0), frames=False)
            else:
                env.reset(out_obs=buf.obs_slot(0))
        else:  # continue the running episodes: the observation the last rollout ended on opens this one
            buf.obs_slot(0).copy_(last)

        def policy_input(t):
            src = buf.obs_slot(t) if t < T else last
            if sym:  # the policy's float32 input is rendered from the 147-byte image it is about to act on
                return env.render(src, out=self._policy_in, blocked=True, dtype=torch.float32)
            return src

        for t in range(T):
            self._logits_value_into_heads(policy_input(t), lean)
            nxt = buf.obs_slot(t + 1) if t + 1 < T else last
            fin = self._final_sym[t] if self.bootstrap_truncated else None
            if sym:  # symbolic storage: the symbolic-only kernel runs and writes NO frames
                env.policy_step(self._ios[t], out_symbolic=nxt, out=self._rows[t], frames=False, final_obs=fin)
            else:
                env.policy_step(self._ios[t], out_obs=nxt, out=self._rows[t], final_obs=fin)
        self._logits_value_into_heads(policy_input(T), lean)
        self._last_value.copy_(self._heads[1, :, 0])

    @torch.no_grad()
    def _collect_batched(self):
        fresh = not (self.carry_episodes and self._started)
        if self.use_cuda_graph:
            if self._graph is None or self._graph[0] != fresh:
                side = torch.cuda.Stream(self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):  # warm-up outside capture (cuDNN plans, allocator)
                    x = self._policy_in if self.obs_storage == "symbolic" else self._last_obs
                    lean = self.use_cnn and self.ac.blocked_first_layer
                    if lean and self._rollout_policy is None:
                        self._rollout_policy = RolloutPolicy(self.ac)
                    self._logits_value_into_heads(x, lean)
                torch.cuda.current_stream(self.device).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    self._rollout_body(fresh)
                self._graph = (fresh, graph)
            self._graph[1].replay()
        else:
            self._rollout_body(fresh)
        if self.bootstrap_truncated:
            self._bootstrap_truncated()
        self._started = True
        ended = self._ep_len > 0  # one synchronisation per rollout, for the episode logs
        self.episode_returns.extend(self._ep_ret[ended].tolist())
        self.episode_lengths.extend(self._ep_len[ended].tolist())
        # episodes cut by the end of the rollout: continued next time (carry_episodes) or discarded by the next reset
        self.unfinished_episodes = int((self.buffer.dones[-1].reshape(-1) == 0).sum().item())
        return self._last_value

    def _bootstrap_truncated(self):
        """reward[t, e] += gamma * V(final observation of step t, env e) where step t truncated env e's episode and did
        not terminate it.  Runs after the rollout (eager or replayed), before the parameters change: the frames of those
        final observations are rendered into the policy's float32 input layout and valued in minibatch-sized chunks.
        One host synchronisation (the number of truncated entries)."""
        idx = (self._truncated & ~self._terminated).reshape(-1).nonzero().squeeze(1)
        if idx.numel() == 0:
            return
        finals = self._final_sym.reshape(-1, 7, 7, 3)
        rewards = self.buffer.rewards.reshape(-1)
        for start in range(0, idx.numel(), self._boot_in.shape[0]):
            rows = idx[start: start + self._boot_in.shape[0]]
            x = self.env.render(finals, rows, out=self._boot_in[: rows.numel()], blocked=True, dtype=torch.float32)
            value = self.ac(x)[1].float()
            rewards.index_add_(0, rows, self.gamma * value)

    def _collect_single(self):
        state, _ = self.env.reset()
        ep_return, ep_length = 0, 0
        for _ in range(self.batch_size):
            state_t = self._obs_to_tensor(state)
            with torch.no_grad():
                action, logp, value = self.ac.act(state_t, deterministic=False)
            state, reward, terminated, truncated, _ = self.env.step(action.item())
            done = terminated or truncated
            self.buffer.add(state_t.squeeze(0), action.squeeze(), logp.squeeze(), value.squeeze(),
                            torch.tensor(reward, dtype=torch.float32, device=self.device),
                            torch.tensor(done, dtype=torch.float32, device=self.device))
            ep_return += reward
            ep_length += 1
            if done:
                self.episode_returns.append(ep_return)
                self.episode_lengths.append(ep_length)
                state, _ = self.env.reset()
                ep_return, ep_length = 0, 0
        with torch.no_grad():
            return self.ac.act(self._obs_to_tensor(state))[2].item()

    # ---- GAE ----------------------------------------------------------------------------------------------
    def compute_gae(self, rewards, values, dones, last_value):
        """`[T]` or time-major `[T, N]` tensors -> (adv, returns), computed by the CUDA GAE kernel."""
        dev = rewards.device
        g = self._gae_device()
        adv, ret = gae_kernel(rewards.to(g), values.to(g), dones.to(g), last_value, self.gamma, self.lam)
        return adv.to(dev), ret.to(dev)

    # ---- update -------------------------------------------------------------------------------------------
    def update(self, last_value):
        states, actions, logprobs_old, rewards, values_old, dones = self.buffer.get()
        adv, returns = self.compute_gae(rewards, values_old, dones, last_value)
        mean, std = parallel.global_mean_std(adv)
        adv = (adv - mean) / (std + 1e-8)

        n = self.buffer.horizon * self.num_envs
        if self.obs_storage == "symbolic":
            stored = states.reshape(n, 7, 7, 3)

            def frames(mb):  # minibatch gather + rendering in one kernel
                return self.env.render(stored, mb, out=self._mb_frames[: mb.numel()], blocked=True,
                                       dtype=self.minibatch_frames, normalise=False)
        else:
            stored = states.reshape((n,) + self.obs_shape)

            def frames(mb):
                return stored[mb]
        actions, logprobs_old = actions.reshape(n), logprobs_old.reshape(n)
        adv, returns = adv.reshape(n), returns.reshape(n)

        totals = torch.zeros(6, dtype=torch.float64, device=self.device)
        nbatches = 0
        for _ in range(self.update_epochs):
            idxs = torch.randperm(n, device=self.device)
            for start in range(0, n, self.minibatch_size):
                mb = idxs[start: start + self.minibatch_size]
                with torch.autocast(self.device.type, dtype=self.amp_dtype, enabled=self.amp_dtype is not None):
                    logp_new, entropy, values = self.ac.evaluate(frames(mb), actions[mb])
                logp_new, entropy, values = logp_new.float(), entropy.float(), values.float()
                mb_adv, mb_old = adv[mb], logprobs_old[mb]
                ratio = torch.exp(logp_new - mb_old)
                surr = torch.min(ratio * mb_adv, torch.clamp(ratio, 1 - self.clip_eps, 1 + self.clip_eps) * mb_adv)
                pi_loss = -surr.mean()
                v_loss = ((values - returns[mb]) ** 2).mean()
                ent = entropy.mean()
                loss = pi_loss + self.vf_coef * v_loss - self.ent_coef * ent

                if self._grads is not None:
                    self._grads.zero_()
                else:
                    self.optimizer.zero_grad(set_to_none=True)
                loss.backward()
                if self._grads is not None:
                    self._grads.all_reduce_mean()
                grad_norm = torch.nn.utils.clip_grad_norm_(self.ac.parameters(), 0.5)
                self.optimizer.step()

                with torch.no_grad():
                    kl = (mb_old - logp_new).mean()
                    clipfrac = (torch.abs(ratio - 1.0) > self.clip_eps).float().mean()
                    totals += torch.stack([pi_loss, v_loss, ent, kl, clipfrac, grad_norm]).double()
                nbatches += 1
        return aggregate_ppo_update_metrics(*totals.tolist(), nbatches)  # the only host sync of the update

    def train(self, total_steps=100_000):
        steps_done = 0
        while steps_done < total_steps:
            self.update(self.collect_rollouts())
            steps_done += self.batch_size * parallel.world_size()

