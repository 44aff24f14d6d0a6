"""The rollout caller around the batched environment (SURVEY 8(f) row 1): what ``pg.Agent.run_episode(s)`` and
``pg.TrajectoryBuffer`` do in the reference (deepgroebner/pg.py:81-244, 432-503), restated for N environments
stepping together on device.

* ``PairsPolicy``      -- the weights of ``ParallelMultilayerPerceptron([H])`` (networks.py:522-571) plus a plain
                          torch fp32 forward that is the numerical reference of the fused CUDA head (bb_policy.cuh).
* ``collect``          -- T fused steps of every environment (policy head, categorical sample, step, auto-reset) in
                          one launch (bb_rollout), trajectories kept on device.
* ``TrajectoryBatch``  -- rewards-to-go and generalised advantage estimates per episode segment
                          (pg.discount_rewards / pg.compute_advantages, pg.py:18-78), the "only finished
                          trajectories" rule of TrajectoryBuffer (pg.py:183-226: data up to ``self.start``), the
                          single-action filter and the -1 padded batches the reference networks consume; with
                          the row store of ``collect(rows_per_env=...)`` every state is kept at its own row count,
                          as the reference's buffer keeps it, and ``batches()`` pads each minibatch on its own.
"""
import math

import torch


class PairsPolicy:
    """ParallelMultilayerPerceptron([hidden]): Dense(hidden, relu) per row, Dense(1), log_softmax over rows.

    Weights use the Keras layouts: W1 [cols, hidden], b1 [hidden], w2 [hidden], b2 [1]; initialised like Keras
    (Glorot uniform kernels, zero biases) from ``torch_seed``.  ``seed`` feeds the device sampler."""

    def __init__(self, cols, hidden=128, torch_seed=0, seed=0, device="cpu"):
        assert hidden in (32, 64, 128, 256)
        g = torch.Generator().manual_seed(torch_seed)
        lim1 = math.sqrt(6.0 / (cols + hidden))
        lim2 = math.sqrt(6.0 / (hidden + 1))
        self.cols, self.hidden, self.seed = cols, hidden, seed
        self.W1 = ((torch.rand((cols, hidden), generator=g) * 2 - 1) * lim1).to(device)
        self.b1 = torch.zeros(hidden, device=device)
        self.w2 = ((torch.rand(hidden, generator=g) * 2 - 1) * lim2).to(device)
        self.b2 = torch.zeros(1, device=device)
        self._dev = None

    def parameters(self):
        return [self.W1, self.b1, self.w2, self.b2]

    def device_weights(self, device, cols):
        assert cols == self.cols, "policy was built for %d state columns, environment has %d" % (self.cols, cols)
        ws = tuple(t.detach().to(device=device, dtype=torch.float32).contiguous() for t in self.parameters())
        self._dev = ws  # keep alive while kernels run
        return ws

    def logits(self, obs):
        """obs: int tensor [..., rows, cols] padded with -1 -> (logits [..., rows], mask)."""
        x = obs.to(torch.float32)
        h = torch.relu(x @ self.W1.to(x.device) + self.b1.to(x.device))
        z = h @ self.w2.to(x.device) + self.b2.to(x.device)
        mask = obs[..., -1] != -1  # networks.py:94-95
        return z, mask

    def log_probs(self, obs):
        """The reference forward pass: masked rows get -1e9 before log_softmax (networks.py:455-459)."""
        z, mask = self.logits(obs)
        z = z + (~mask).to(torch.float32) * -1e9
        return torch.log_softmax(z, dim=-1)


def collect(env, net, T, counter0=0, greedy=False, store_obs=None, pmax=64, max_episode_length=None, value=None, gamma=0.99,
            value_rollouts=None, value_seed=0, rows_per_env=None):
    """Runs T steps of every environment of a LeadMonomialsEnv under policy `net` and returns a TrajectoryBatch.
    The environments must have been reset; auto-reset keeps every slot busy.  max_episode_length cuts episodes as
    pg.Agent.run_episode does (pg.py:470-471; train.py's default is 500).  States with more than pmax rows keep their
    action and log-probability but cannot be stored: TrajectoryBatch.get() leaves them out (and counts them).
    value: 'degree', 'sample' or another selection name -- every state's env.value(value, gamma) is computed in the same
    launch (the baseline pg.Agent.run_episode stores with a value model, pg.py:461-462) and finish() / get() use it.
    Pass the `gam` of finish() / get() as gamma, as pg.py passes its own gam to env.value.
    rows_per_env: an int or True (BuchbergerEngine.rollout) -- every state is stored at its own row count, as the
    reference's TrajectoryBuffer stores it, so get() drops none; environments whose rows run out halt (see
    TrajectoryBatch.halted) and continue in the next call.  store_obs (default: only without rows_per_env) adds the
    dense [N, T, pmax, cols] block."""
    eng = env.engine
    eng.set_auto_reset(True)
    if max_episode_length is not None:
        eng.set_max_episode_length(max_episode_length)
    if store_obs is None:
        store_obs = rows_per_env is None
    out = eng.rollout(net, T, counter0=counter0, greedy=greedy, store_obs=store_obs, pmax=pmax, value=value,
                      value_gamma=gamma, value_rollouts=value_rollouts, value_seed=value_seed, rows_per_env=rows_per_env)
    return TrajectoryBatch(out, engine=eng)


def discount_rewards(rewards, done, gam, engine=None):
    """Rewards-to-go within each episode segment: pg.discount_rewards (pg.py:18-39) along the T axis of [N, T]
    tensors, restarting after every done.  With `engine` (cuda tensors) this is ONE kernel (bb_discount); without it,
    a host-side restatement in torch ops used by the CPU tests."""
    N, T = rewards.shape
    if engine is not None and rewards.is_cuda:
        import ctypes as C
        x = rewards.to(torch.float64).contiguous()
        d = done.to(torch.uint8).contiguous()
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            engine._ck(engine.lib.bb_discount(engine.h, N, T, C.c_void_p(x.data_ptr()), C.c_void_p(d.data_ptr()), float(gam),
                                              C.c_void_p(out.data_ptr()),
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream)), "bb_discount")
        return out
    out = torch.empty_like(rewards, dtype=torch.float64)
    run = torch.zeros(N, dtype=torch.float64, device=rewards.device)
    for t in range(T - 1, -1, -1):
        run = rewards[:, t].to(torch.float64) + gam * run * (~done[:, t]).to(torch.float64)
        out[:, t] = run
    return out


def compute_advantages(rewards, values, done, gam, lam, engine=None):
    """Generalised advantage estimates, pg.compute_advantages (pg.py:42-78): delta_t = r_t - v_t + gam * v_{t+1}
    (v after the last step of an episode is 0), discounted by gam * lam within each episode segment."""
    r = rewards.to(torch.float64)
    v = values.to(torch.float64)
    nxt = torch.zeros_like(v)
    nxt[:, :-1] = v[:, 1:]
    nxt = nxt * (~done).to(torch.float64)
    return discount_rewards(r - v + gam * nxt, done, gam * lam, engine)


class TrajectoryBatch:
    """[N, T] trajectories on device with the TrajectoryBuffer post-processing of the reference.  When `out` has "value"
    (rollout(value=...)), finish() and get() called with values=None use those values as the baseline; they should have
    been computed with the gamma later given to finish() / get() as gam (pg.py passes self.gam to env.value).

    States come from `out["rows"]` (rows mode, rollout(rows_per_env=...)) when it is there, else from `out["obs"]`
    (dense mode).  In rows mode every state is kept at its own row count: offsets[e, t] is the first row of step t's
    state in environment e's region, and no sample is dropped for its width."""

    def __init__(self, out, engine=None):
        self.engine = engine   # with it, the discounted sums run as one kernel each (bb_discount)
        self.dropped_wide = 0  # get(): samples left out because their state had more rows than the stored matrices
        self.actions, self.logp = out["actions"], out["logp"]
        self.reward, self.lengths = out["reward"], out["lengths"]
        self.done = out["done"].bool()
        self.obs = out.get("obs")
        self.rows = out.get("rows")
        self.value = out.get("value")
        N, T = self.reward.shape
        # a step belongs to a FINISHED trajectory iff some done follows it (inclusive) inside the window
        later = torch.flip(torch.cummax(torch.flip(self.done, [1]).to(torch.uint8), dim=1).values, [1]).bool()
        self.finished = later & (self.actions >= 0)
        self.offsets, self.halted = None, 0
        if self.rows is not None:
            # bb_rollout_rows' layout: the states of the steps that took an action, back to back in step order
            took = self.lengths.to(torch.int64) * (self.actions >= 0)
            self.offsets = torch.cumsum(took, dim=1) - took
            # environments the row budget stopped: the only outputs with action -1 and done 0
            self.halted = int(((self.actions < 0) & ~self.done).any(dim=1).sum())

    def episode_stats(self):
        """(returns, lengths) of the episodes that finished inside the window, as 1-D tensors."""
        r = self.reward.to(torch.float64) * self.finished
        csum = torch.cumsum(r, dim=1)
        steps = torch.cumsum(self.finished.to(torch.int64), dim=1)
        idx = self.done & self.finished
        ends_r, ends_s = csum[idx], steps[idx]
        # subtract the cumulative value at the previous episode end of the same environment: position of the last
        # episode end strictly before t, by a running maximum over the end positions
        N, T = self.reward.shape
        pos = torch.where(idx, torch.arange(T, device=r.device).expand(N, T), torch.full((N, T), -1, device=r.device))
        last = torch.cummax(pos, dim=1).values
        prev = torch.cat([torch.full((N, 1), -1, device=r.device, dtype=last.dtype), last[:, :-1]], dim=1)
        has = prev >= 0
        at = prev.clamp(min=0)
        prev_r = torch.where(has, torch.gather(csum, 1, at), torch.zeros_like(csum))
        prev_s = torch.where(has, torch.gather(steps, 1, at), torch.zeros_like(steps))
        return ends_r - prev_r[idx], ends_s - prev_s[idx]

    def finish(self, gam=0.99, lam=0.97, values=None):
        """TrajectoryBuffer.finish for every episode segment: returns (rewards_to_go, advantages), float64 [N, T].
        values None: the batch's own values if it has them, else zeros."""
        if values is None:
            values = self.value
        v = torch.zeros_like(self.reward) if values is None else values
        return (discount_rewards(self.reward, self.done, gam, self.engine),
                compute_advantages(self.reward, v, self.done, gam, lam, self.engine))

    def _samples(self, gam, lam, values, normalize_advantages):
        """The training set as (env, step, actions, logprobs, advantages, rewards_to_go), 1-D, in (env, step) order."""
        rtg, adv = self.finish(gam, lam, values)
        keep = self.finished
        a = adv[keep].to(torch.float32)
        if normalize_advantages and a.numel() > 1:
            a = (a - a.mean()) / a.std(unbiased=False)
        multi = self.lengths[keep] != 1
        if self.obs is not None and self.rows is None:   # a state with more rows than were stored cannot be a sample
            fits = self.lengths[keep] <= self.obs.shape[2]
            self.dropped_wide = int((multi & ~fits).sum())
            multi = multi & fits
        e, t = keep.nonzero(as_tuple=True)
        return e[multi], t[multi], self.actions[keep][multi], self.logp[keep][multi], a[multi], rtg[keep][multi].to(torch.float32)

    def states(self, e, t):
        """The state matrices of steps (e[i], t[i]) as [M, rows, cols], padded with -1 to the largest of them."""
        L = self.lengths[e, t].to(torch.int64)
        width = int(L.max()) if L.numel() else 0
        if self.rows is None:
            return self.obs[e, t, :width]
        R, cols = self.rows.shape[1], self.rows.shape[2]
        j = torch.arange(width, device=L.device)
        valid = j < L[:, None]
        at = e.to(torch.int64)[:, None] * R + torch.where(valid, self.offsets[e, t][:, None] + j, 0)
        return torch.where(valid[..., None], self.rows.reshape(-1, cols)[at], -1)

    def get(self, gam=0.99, lam=0.97, values=None, normalize_advantages=True):
        """The flat training set of TrajectoryBuffer.get (pg.py:183-226): steps of finished trajectories whose state
        had more than one row, as (obs [M, rows, cols] padded -1, actions, logprobs, advantages, rewards_to_go).
        Dense mode: rows = pmax, and states wider than pmax are left out (counted in dropped_wide).  Rows mode: rows =
        the largest kept state."""
        e, t, actions, logp, a, rtg = self._samples(gam, lam, values, normalize_advantages)
        if self.rows is not None:
            obs = self.states(e, t)
        else:
            obs = self.obs[e, t] if self.obs is not None else None
        return obs, actions, logp, a, rtg

    def batches(self, batch_size, gam=0.99, lam=0.97, values=None, normalize_advantages=True, seed=None):
        """get()'s training set as minibatches (obs, actions, logprobs, advantages, rewards_to_go) of batch_size
        samples (the last may be smaller); each obs is padded with -1 to the largest state of its own minibatch, as
        the reference pads its batches.  Advantages are normalised over the whole set.  seed None keeps get()'s order;
        an int shuffles the samples with torch.Generator().manual_seed(seed)."""
        e, t, actions, logp, a, rtg = self._samples(gam, lam, values, normalize_advantages)
        M = e.numel()
        order = torch.arange(M) if seed is None else torch.randperm(M, generator=torch.Generator().manual_seed(seed))
        order = order.to(e.device)
        have = self.rows is not None or self.obs is not None
        for i in range(0, M, batch_size):
            s = order[i:i + batch_size]
            yield (self.states(e[s], t[s]) if have else None), actions[s], logp[s], a[s], rtg[s]
