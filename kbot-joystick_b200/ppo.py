"""PPO minibatch update on top of the C-ABI (SURVEY 8f-1, BASELINE configs[3]): kbs_ppo_grad -> gradient all-reduce over
NCCL (the only collective of the path: environments are sharded, weights replicated) -> kbs_grad_norm -> kbs_adamw_step
-> re-pack.

Mirrors ksim's PPOTask.update_model for this Task: the optimiser is optax.adamw(5e-4, weight_decay = 1e-5) -- the branch
get_optimizer takes with the launch configuration (train.py:1059-1065, 95-102, 1761-1791) -- wrapped in ksim's global-norm
gradient clip and non-finite-update skip [U: parameterised, `max_grad_norm`]; hyper-parameters train.py:1763-1770.  torch is
allocation, streams and torch.distributed only."""
from __future__ import annotations

import torch

from . import _lib as L


class NetParams:
    """One network's parameters as ONE flat fp32 tensor (what Adam and the all-reduce see) with eqx-layout views."""

    ORDER = ("w_in", "b_in", "layers", "w_out", "b_out")

    def __init__(self, w: dict, device=None):
        parts = [w["w_in"], w["b_in"]] + [lw[k] for lw in w["layers"] for k in ("w_ih", "w_hh", "b")] + [w["w_out"], w["b_out"]]
        parts = [torch.as_tensor(p, dtype=torch.float32, device=device) for p in parts]
        self.flat = torch.cat([p.reshape(-1) for p in parts]).contiguous()
        self.shapes = [tuple(p.shape) for p in parts]
        self.depth = len(w["layers"])

    def _views(self, flat):
        out, off = [], 0
        for s in self.shapes:
            n = 1
            for d in s:
                n *= d
            out.append(flat[off:off + n].view(s))
            off += n
        return out

    def as_dict(self, flat=None) -> dict:
        v = self._views(self.flat if flat is None else flat)
        layers = [{"w_ih": v[2 + 3 * i], "w_hh": v[3 + 3 * i], "b": v[4 + 3 * i]} for i in range(self.depth)]
        return {"w_in": v[0], "b_in": v[1], "layers": layers, "w_out": v[-2], "b_out": v[-1]}


def allreduce_sum_(flat: torch.Tensor) -> int:
    """Sum the flat gradient over the ranks (NCCL on GPUs; gloo in the CPU test).  Returns the world size."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return 1
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    return dist.get_world_size()


class PpoUpdater:
    """grad -> all-reduce -> global norm -> AdamW (clip folded in) -> re-pack, for the actor and the critic.

    Overlap: kbs_ppo_grad finishes the critic's gradients first and records an event when they are final; the critic's
    slice of the flat gradient is all-reduced on a communication stream while the actor's weight-gradient GEMMs still run,
    the actor's slice follows.  With `capture()` the WHOLE update -- gradients, both all-reduces, norm, AdamW, re-pack --
    is one CUDA graph (the step counter lives on the device).  `epoch()` runs the update phase of a whole PPO epoch on a
    stored rollout (device-shuffled minibatches of whole trajectories); `capture_epoch()` records it as one CUDA graph.
    `iteration()` runs a whole PPO iteration -- rollout, rewards, epoch -- on the rollout the library records, and
    `capture_iteration()` records that as one CUDA graph."""

    def __init__(self, engine, w_actor: dict, w_critic: dict, lr: float = 5e-4, b1: float = 0.9, b2: float = 0.999,
                 eps: float = 1e-8, weight_decay: float = 1e-5, max_grad_norm: float = 10.0, **loss_hyper):
        dev = torch.device("cuda", torch.cuda.current_device())
        self.eng = engine
        self.pa, self.pc = NetParams(w_actor, dev), NetParams(w_critic, dev)
        n = self.pa.flat.numel() + self.pc.flat.numel()
        self.grad = torch.zeros(n, device=dev)            # [actor | critic]
        self.m, self.v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
        self.param = torch.cat([self.pa.flat, self.pc.flat])
        self.na = self.pa.flat.numel()
        self.pa.flat, self.pc.flat = self.param[:self.na], self.param[self.na:]
        self.step_dev = torch.zeros(1, device=dev, dtype=torch.int64)   # updates applied so far (device-side: graph-replayable)
        self.norm = torch.zeros(1, device=dev)                            # global L2 norm of the (summed) gradient
        self.opt = dict(lr=lr, b1=b1, b2=b2, eps=eps, weight_decay=weight_decay, max_grad_norm=max_grad_norm)
        self.loss_hyper = loss_hyper
        self.comm_stream = torch.cuda.Stream(device=dev)
        self.ev_critic, self.ev_comm, self.ev_fork = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        self.ev_critic.record()            # torch creates the cudaEvent_t lazily: make the handle exist before the library sees it
        self._graph = None
        self.pass_dev = torch.zeros(1, device=dev, dtype=torch.int64)    # passes drawn so far (epoch(): one permutation each)
        self._ework, self._epoch_graph = None, None
        self._iwork, self._iter_graph = None, None
        self._repack(sync=True)

    def _repack(self, sync: bool = False):
        """Re-pack both networks' MMA weight images from the flat parameters.  Inside an update (sync=False) the critic's ~15
        small launches run on the communication stream beside the actor's (per-network buffers only)."""
        if sync:
            self.eng.pack_weights(L.NET_ACTOR, self.pa.as_dict(), sync=True)
            self.eng.pack_weights(L.NET_CRITIC, self.pc.as_dict(), sync=True)
            return
        cur = torch.cuda.current_stream()
        self.ev_fork.record(cur)
        with torch.cuda.stream(self.comm_stream):
            self.comm_stream.wait_event(self.ev_fork)
            self.eng.pack_weights(L.NET_CRITIC, self.pc.as_dict(), sync=False)
            self.ev_comm.record(self.comm_stream)
        self.eng.pack_weights(L.NET_ACTOR, self.pa.as_dict(), sync=False)
        cur.wait_event(self.ev_comm)

    def grads(self, batch: dict, n_envs: int, critic_ready=None, loss_fn=None) -> dict:
        ga, gc = self.pa.as_dict(self.grad[:self.na]), self.pc.as_dict(self.grad[self.na:])
        if loss_fn is None:
            return self.eng.ppo_grad(batch, ga, gc, n_envs=n_envs, critic_ready=critic_ready, **self.loss_hyper)
        return self._loss_fn_grads(batch, n_envs, critic_ready, loss_fn, ga, gc)

    VARIABLES = ("log_probs", "values", "entropy", "action_std")

    def _loss_fn_grads(self, batch: dict, n_envs: int, critic_ready, loss_fn, ga: dict, gc: dict) -> dict:
        """The gradient of a caller's loss: kbs_ppo_variables from copies of the minibatch's start carries, the loss and its
        cotangents by torch autograd, then kbs_ppo_variables_vjp.  The loss sees kbs_ppo_variables' forward and the gradient
        is taken at the VJP's own forward; the two agree to fp32 rounding (as epoch() mixes kbs_ppo_variables' old values
        with kbs_ppo_grad's gradients)."""
        T, _, ld = batch["actor_obs"].shape
        dev = batch["actor_obs"].device
        shape = (self.eng.depth, 2, n_envs, self.eng.hidden_size)
        carry = lambda k, s: batch[k].clone() if batch.get(k) is not None else torch.zeros(s, device=dev)
        v = self.eng.ppo_variables(batch["actor_obs"], batch["action"], batch["done"], carry("actor_carry0", shape),
                                   carry("lpf0", (L.NUM_JOINTS, ld)), batch["critic_obs"], carry("critic_carry0", shape),
                                   n_envs=n_envs)
        var = {k: v[k].detach().requires_grad_(True) for k in self.VARIABLES}
        loss = loss_fn(var, batch)
        cts = torch.autograd.grad(loss, [var[k] for k in self.VARIABLES], allow_unused=True)
        out = self.eng.ppo_variables_vjp(batch, {k: c for k, c in zip(self.VARIABLES, cts) if c is not None}, ga, gc,
                                         n_envs=n_envs, critic_ready=critic_ready)
        nan = torch.full((3,), float("nan"), device=dev)
        out["stats"] = torch.cat([loss.detach().reshape(1).float(), nan])
        return out

    def _step(self, batch: dict, n_envs: int, loss_fn=None) -> dict:
        """One whole update, enqueued on the current stream (+ the communication stream, forked from / joined into it)."""
        import torch.distributed as dist

        world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        if world == 1:
            out = self.grads(batch, n_envs, loss_fn=loss_fn)
        else:
            cur = torch.cuda.current_stream()
            out = self.grads(batch, n_envs, critic_ready=self.ev_critic, loss_fn=loss_fn)
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(self.ev_critic)          # the critic's gradients are final: reduce them now
                dist.all_reduce(self.grad[self.na:], op=dist.ReduceOp.SUM)
                self.ev_comm.record(self.comm_stream)
            dist.all_reduce(self.grad[:self.na], op=dist.ReduceOp.SUM)   # the actor's slice, behind its GEMMs
            cur.wait_event(self.ev_comm)
        self.eng.grad_norm(self.grad, out=self.norm)        # of the SUM; kbs_adamw_step applies grad_scale = 1 / world to it
        self.eng.adamw_step(self.param, self.grad, self.m, self.v, grad_norm=self.norm, step_dev=self.step_dev,
                            grad_scale=1.0 / world, **self.opt)
        self._repack()
        return out

    def capture(self, batch: dict, n_envs: int, loss_fn=None) -> None:
        """Record one whole update on `batch` as ONE CUDA graph; later update() calls with the same batch object and loss_fn
        replay it (refill the batch tensors in place between updates).  Call after at least one eager update (allocations,
        NCCL).  A loss_fn is captured with it: it must enqueue device work only."""
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._graph_out = self._step(batch, n_envs, loss_fn)
        self._graph_batch, self._graph_loss_fn = batch, loss_fn
        self.eng.scratch_lock(True)        # the graph holds pointers into the library's scratch: it must not be reallocated

    def update(self, batch: dict, n_envs: int, loss_fn=None) -> dict:
        """One whole update on a minibatch.  loss_fn=None: the library's PPO loss (kbs_ppo_grad).  Otherwise
        loss = loss_fn(vars, batch), a scalar tensor, where vars holds "log_probs", "values", "entropy" [T, ld] and "action_std"
        [T, 20, ld] as tensors that require grad and batch is the minibatch dict (old_log_probs, advantages, ...): its gradient
        comes from torch autograd for the cotangents and kbs_ppo_variables_vjp for the parameters (see _loss_fn_grads).  Only
        columns < n_envs reach the gradient.  Returns the forward outputs and "stats" ([loss, nan, nan, nan] with a loss_fn)."""
        if self._graph is not None and batch is self._graph_batch and loss_fn is self._graph_loss_fn:
            self._graph.replay()
            return self._graph_out
        return self._step(batch, n_envs, loss_fn)

    # ---- the update phase of an epoch -----------------------------------------------------------------------------------------
    def _epoch_work(self, rollout: dict, n_envs: int, batch_size: int, num_passes: int) -> dict:
        """Buffers of one epoch, allocated once per shape and reused across passes and epochs."""
        key = (tuple(rollout["actor_obs"].shape), n_envs, batch_size, num_passes)
        w = self._ework
        if w is not None and w["key"] == key:
            return w
        T, _, ld = rollout["actor_obs"].shape
        dev = self.param.device
        nb = n_envs // batch_size
        f = lambda *s: torch.empty(s, device=dev)
        w = {"key": key, "actor_carry": torch.empty_like(rollout["actor_carry0"]),
             "critic_carry": torch.empty_like(rollout["critic_carry0"]), "lpf": torch.empty_like(rollout["lpf0"]),
             "adv": f(T, ld), "targets": f(T, ld), "stats": f(num_passes * nb, 4), "norms": f(num_passes * nb),
             "perm": torch.empty((num_passes, n_envs), dtype=torch.int32, device=dev),
             "mb": self.eng.minibatch_buffers(T, nb, batch_size, dev)}       # the shuffled copy of the rollout
        self._ework = w
        return w

    def _epoch(self, rollout: dict, n_envs: int, batch_size: int, num_passes: int, seed: int, loss_fn=None) -> dict:
        """One epoch's update phase, enqueued on the current stream (SURVEY 3.1): kbs_ppo_variables from the rollout's start
        carries -> kbs_gae -> per pass: permutation, shuffle into minibatches, one whole update per minibatch."""
        import torch.distributed as dist

        rank = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
        w = self._epoch_work(rollout, n_envs, batch_size, num_passes)
        for k in ("actor_carry", "critic_carry"):          # kbs_ppo_variables advances its carries in place
            w[k].copy_(rollout[k + "0"])
        w["lpf"].copy_(rollout["lpf0"])
        v = self.eng.ppo_variables(rollout["actor_obs"], rollout["action"], rollout["done"], w["actor_carry"], w["lpf"],
                                   rollout["critic_obs"], w["critic_carry"], want_std=False, n_envs=n_envs)
        self.eng.gae(v["values"], rollout["rewards"], rollout["done"], rollout["success"], adv=w["adv"], targets=w["targets"],
                     n_envs=n_envs)
        src = {k: rollout[k] for k in ("actor_obs", "critic_obs", "action", "done", "actor_carry0", "critic_carry0", "lpf0")}
        src.update(old_log_probs=v["log_probs"], advantages=w["adv"], value_targets=w["targets"], old_values=v["values"])
        mb = w["mb"]
        nb = n_envs // batch_size
        for p in range(num_passes):
            self.eng.minibatch_permutation(self.pass_dev, n_envs, seed=seed, env0=rank * n_envs, out=w["perm"][p])
            self.eng.shuffle_minibatches(w["perm"][p], src, n_envs, batch_size, dst=mb)
            for b in range(nb):
                out = self._step({k: t[b] for k, t in mb.items()}, batch_size, loss_fn)
                w["stats"][p * nb + b].copy_(out["stats"])
                w["norms"][p * nb + b:p * nb + b + 1].copy_(self.norm)
        return {"stats": w["stats"], "norms": w["norms"], "perm": w["perm"]}

    def epoch(self, rollout: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3, seed: int = 0, loss_fn=None) -> dict:
        """The update phase of one PPO epoch on a stored rollout: num_passes x (n_envs / batch_size) updates (train.py:1763-1766),
        each on a minibatch of whole trajectories taken from a fresh device-drawn permutation of the env axis.
        rollout: actor_obs [T,65,ld], critic_obs [T,475,ld], action [T,20,ld], done / success u8 [T,ld], rewards [T,ld], and the
        carries at the rollout's first step (snapshot them before kbs_rollout, which advances them): actor_carry0 /
        critic_carry0 [depth,2,n_envs,H], lpf0 [20,ld].  Returns device tensors, overwritten by the next epoch: "stats"
        [P*B, 4] loss statistics and "norms" [P*B] gradient norms per update, "perm" [P, n_envs] the permutations.  No host
        synchronisation.  After capture_epoch, a call on the same rollout object with the same arguments replays the graph.
        loss_fn: as for update(), for every update of the epoch."""
        if self._epoch_graph is not None and rollout is self._epoch_rollout and \
                self._epoch_args == (n_envs, batch_size, num_passes, seed, loss_fn):
            self._epoch_graph.replay()
            return self._epoch_out
        return self._epoch(rollout, n_envs, batch_size, num_passes, seed, loss_fn)

    def capture_epoch(self, rollout: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3, seed: int = 0,
                      loss_fn=None) -> None:
        """Record one whole epoch() on `rollout` as ONE CUDA graph; later epoch() calls with the same rollout object and
        arguments replay it (refill the rollout tensors in place between epochs).  Call after one eager epoch with the same
        arguments: the handle's scratch has then grown to what kbs_ppo_variables and kbs_ppo_grad need, and is locked here."""
        torch.cuda.synchronize()
        self._epoch_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._epoch_graph):
            self._epoch_out = self._epoch(rollout, n_envs, batch_size, num_passes, seed, loss_fn)
        self._epoch_rollout = rollout
        self._epoch_args = (n_envs, batch_size, num_passes, seed, loss_fn)
        self._epoch_graph_work = self._ework       # the graph holds its buffers' addresses: keep them if the shapes change
        self.eng.scratch_lock(True)

    # ---- a whole iteration: rollout -> rewards -> epoch ---------------------------------------------------------------------
    def _iteration_work(self, io: dict, n_envs: int) -> dict:
        """What an iteration keeps besides the caller's io, allocated once per shape: the carries at the rollout's first step,
        the recorded critic observations, the rewards, and done_prev (the previous iteration's done[T-1]; zero before the
        first iteration, which restarts nothing, as no done_prev)."""
        T, _, ld = io["actor_obs"].shape
        key = (T, ld, n_envs, tuple(io["actor_carry"].shape))
        w = self._iwork
        if w is not None and w["key"] == key:
            return w
        dev = self.param.device
        w = {"key": key, "actor_carry0": torch.empty_like(io["actor_carry"]), "critic_carry0": torch.empty_like(io["critic_carry"]),
             "lpf0": torch.empty_like(io["lpf"]), "critic_obs": torch.empty((T, L.CRITIC_OBS, ld), device=dev),
             "rewards": torch.empty((T, ld), device=dev), "done_prev": torch.zeros((ld,), dtype=torch.uint8, device=dev)}
        self._iwork = w
        return w

    def _iteration(self, io: dict, reward_carry: dict, n_envs: int, batch_size: int, num_passes: int, seed: int) -> dict:
        """One PPO iteration, enqueued on the current stream: carry snapshot -> kbs_rollout_record (value, critic_obs,
        done_prev) -> kbs_rewards -> the epoch's update phase -> done[T-1] and command[T] carried into the next iteration."""
        T = io["T"]
        w = self._iteration_work(io, n_envs)
        for k in ("actor_carry", "critic_carry", "lpf"):      # kbs_rollout advances them in place
            w[k + "0"].copy_(io[k])
        self.eng.rollout(dict(io, done_prev=w["done_prev"], critic_obs=w["critic_obs"]), n_envs)
        self.eng.rewards(io["state"], io["command"][:T], io["ctrl"], io["done"], reward_carry, total=w["rewards"], n_envs=n_envs)
        rollout = {"actor_obs": io["actor_obs"], "critic_obs": w["critic_obs"], "action": io["action"], "done": io["done"],
                   "success": io["success"], "rewards": w["rewards"], "actor_carry0": w["actor_carry0"],
                   "critic_carry0": w["critic_carry0"], "lpf0": w["lpf0"]}
        out = self._epoch(rollout, n_envs, batch_size, num_passes, seed)
        w["done_prev"].copy_(io["done"][T - 1])
        io["command"][0].copy_(io["command"][T])
        return dict(out, rewards=w["rewards"])

    def iteration(self, io: dict, reward_carry: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3,
                  seed: int = 0) -> dict:
        """One whole PPO iteration on the device, no host synchronisation: the rollout over io's recorded state (as
        KbotStep.rollout; io needs actor_obs, value and critic_carry), the rewards of that trajectory (reward_carry: t_single,
        airtime, prev_contact, advanced in place), then epoch() on what the rollout recorded.  Afterwards io is ready for the
        next iteration: its carries, lpf and pg_carry are the final ones, command[0] = command[T], and the next rollout gets this
        one's done[T-1], so consecutive iterations are one continuous rollout.  Refill io's state and noise in place between
        iterations.  n_envs <= 16 384 per rank (the permutation's limit).  Returns epoch()'s "stats", "norms", "perm" and
        "rewards" [T, ld], device tensors overwritten by the next iteration.  After capture_iteration, a call with the same io,
        reward_carry and arguments replays the graph."""
        if self._iter_graph is not None and io is self._iter_io and reward_carry is self._iter_reward_carry and \
                self._iter_args == (n_envs, batch_size, num_passes, seed):
            self._iter_graph.replay()
            return self._iter_out
        return self._iteration(io, reward_carry, n_envs, batch_size, num_passes, seed)

    def capture_iteration(self, io: dict, reward_carry: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3,
                          seed: int = 0) -> None:
        """Record one whole iteration() as ONE CUDA graph; later iteration() calls with the same io, reward_carry and
        arguments replay it.  Call after one eager iteration with the same arguments (the handle's scratch has then grown to
        what the rollout and the epoch need, and is locked here)."""
        torch.cuda.synchronize()
        self._iter_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._iter_graph):
            self._iter_out = self._iteration(io, reward_carry, n_envs, batch_size, num_passes, seed)
        self._iter_io, self._iter_reward_carry = io, reward_carry
        self._iter_args = (n_envs, batch_size, num_passes, seed)
        self._iter_graph_work = (self._iwork, self._ework)     # the graph holds their addresses
        self.eng.scratch_lock(True)

    # ---- the online form: one control step per call, the rollout's carries resident on the device ----------------------------
    def begin_iteration(self, io: dict, n_envs: int) -> None:
        """Start an iteration of the online rollout into io's trajectories (command [T+1,16,ld], actor_obs, action, log_prob,
        ctrl, done, success, value; term_codes optional).  The first call makes the step state from io's actor_carry,
        critic_carry, lpf, pg_carry and command[0]; later iterations continue from the state.  Every call snapshots the state's
        carries for the epoch: the iteration's one conversion out of the kernels' layouts."""
        T, _, ld = io["actor_obs"].shape
        key = (id(io), T, ld, n_envs)
        if getattr(self, "_okey", None) != key:
            dev = self.param.device
            # made first: where the handle has no step state (a tensor-core datapath at depth > 2) this raises and the
            # updater keeps no half-made iteration
            self.step_st = self.eng.step_state(n_envs, True, {"actor_carry": io["actor_carry"], "critic_carry": io["critic_carry"],
                                                              "lpf": io["lpf"], "pg_carry": io["pg_carry"],
                                                              "command": io["command"][0]})
            self._okey, self._oio = key, io
            self._owork = {"actor_carry0": torch.empty_like(io["actor_carry"]), "critic_carry0": torch.empty_like(io["critic_carry"]),
                           "lpf0": torch.empty_like(io["lpf"]), "critic_obs": torch.empty((T, L.CRITIC_OBS, ld), device=dev),
                           "rewards": torch.empty((T, ld), device=dev),
                           "traj_state": {k: torch.empty((T, r, ld), device=dev) for k, r in self.REWARD_STATE_ROWS.items()}}
            self._step_graphs, self._substep_graphs = {}, {}
            self.act_st = None
            self._online_iterations = 0
        w = self._owork
        self.eng.step_state_store(self.step_st, {"actor_carry": w["actor_carry0"], "critic_carry": w["critic_carry0"],
                                                 "lpf": w["lpf0"]})

    REWARD_STATE_ROWS = {"qpos": 27, "qvel": 26, "sensordata": 49, "xpos": 72, "xquat": 96, "com_distance": 1}   # kbs_rewards

    def _online_step(self, io_t: dict) -> None:
        io = self._oio
        self.eng.rollout_step(self.step_st, dict(
            {k: io_t.get(k) for k in ("state", "noise", "episode", "eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")},
            **{k: io.get(k) for k in ("command", "actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value")},
            critic_obs=self._owork["critic_obs"], traj_state=self._owork["traj_state"]))

    def step(self, io_t: dict) -> None:
        """One control step into slot t of the iteration's trajectories.  io_t: this step's state / noise / episode (dicts of
        [F, ld] tensors), eps_action, u_switch, cmd_mode, cmd_u6, cmd_u_arms.  After capture_step(io_t), a call with the same
        io_t object replays the graph (refill its tensors in place between steps)."""
        g = self._step_graphs.get(id(io_t))
        if g is not None and g[1] is io_t:
            g[0].replay()
            return
        self._online_step(io_t)

    def capture_step(self, io_t: dict) -> None:
        """Record step(io_t) as ONE CUDA graph, replayed by later step() calls with the same io_t for every t (the state's step
        index lives on the device).  Capturing runs nothing.  The graph holds pointers into the handle's scratch, which is
        locked here, so the scratch must already have grown to what a step AND end_iteration's epoch need: call it after one
        whole eager iteration (begin_iteration, step x T, end_iteration) on this io; before that it raises."""
        if not getattr(self, "_online_iterations", 0):
            raise RuntimeError("capture_step: run one whole eager iteration (begin_iteration, step, end_iteration) first")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._online_step(io_t)
        self._step_graphs[id(io_t)] = (g, io_t)
        self.eng.scratch_lock(True)

    def _online_substep(self, io_k: dict, n_substeps: int, sub_dt: float, drop_prob: float) -> None:
        n = self.step_st.desc.n_envs
        ast = getattr(self, "act_st", None)
        if ast is None or (ast.desc.n_envs, ast.desc.n_substeps) != (n, n_substeps):
            self.act_st = ast = self.eng.actuator_state(n, n_substeps)
        self.eng.actuator_substep(self.step_st, ast, dict(
            {k: io_k.get(k) for k in ("qpos", "qvel", "u_drop", "latency", "episode", "ctrl")}, action=self._oio["action"],
            sub_dt=sub_dt, drop_prob=drop_prob))

    def substep(self, io_k: dict, *, n_substeps: int = 5, sub_dt: float = 0.004, drop_prob: float = 0.05) -> None:
        """One physics sub-step after the control step that step() just ran: ctrl [20, ld] of io_k = the PD torque on io_k's
        qpos [27, ld] / qvel [26, ld] (gains from io_k's episode) of the action the actuators see at this sub-step -- this step's
        action once latency [ld] has elapsed, the previous one before, the previous one throughout where u_drop [ld] <
        drop_prob (kbs_actuator_substep).  Call it n_substeps times per step, before end_iteration.  The actuator state (sub-step
        index, last applied action) is made on first use, from zeros.  After capture_substep(io_k), a call with the same io_k
        object replays the graph (refill its tensors in place between sub-steps)."""
        g = self._substep_graphs.get(id(io_k))
        if g is not None and g[1] is io_k:
            g[0].replay()
            return
        self._online_substep(io_k, n_substeps, sub_dt, drop_prob)

    def capture_substep(self, io_k: dict, *, n_substeps: int = 5, sub_dt: float = 0.004, drop_prob: float = 0.05) -> None:
        """Record substep(io_k) as ONE CUDA graph, replayed by later substep() calls with the same io_k for every sub-step of
        every step (the sub-step and step indices live on the device), with the keyword arguments given here.  Capturing runs
        nothing.  Like capture_step, it needs one whole eager iteration first; before that it raises."""
        if not getattr(self, "_online_iterations", 0):
            raise RuntimeError("capture_substep: run one whole eager iteration (begin_iteration, step, end_iteration) first")
        n = self.step_st.desc.n_envs
        if getattr(self, "act_st", None) is None or (self.act_st.desc.n_envs, self.act_st.desc.n_substeps) != (n, n_substeps):
            self.act_st = self.eng.actuator_state(n, n_substeps)       # made outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._online_substep(io_k, n_substeps, sub_dt, drop_prob)
        self._substep_graphs[id(io_k)] = (g, io_k, self.act_st)      # the graph holds the state's addresses

    def end_iteration(self, reward_carry: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3, seed: int = 0) -> dict:
        """kbs_rewards on the recorded trajectory (reward_carry advanced in place), then epoch() on it; the step state is then
        ready for the next iteration (step index 0; its command and done_prev carry over, as iteration() carries them).
        Returns what iteration() returns."""
        io, w = self._oio, self._owork
        T = io["actor_obs"].shape[0]
        self.eng.rewards(w["traj_state"], io["command"][:T], io["ctrl"], io["done"], reward_carry, total=w["rewards"], n_envs=n_envs)
        rollout = {"actor_obs": io["actor_obs"], "critic_obs": w["critic_obs"], "action": io["action"], "done": io["done"],
                   "success": io["success"], "rewards": w["rewards"], "actor_carry0": w["actor_carry0"],
                   "critic_carry0": w["critic_carry0"], "lpf0": w["lpf0"]}
        out = self._epoch(rollout, n_envs, batch_size, num_passes, seed)
        self.eng.step_state_rewind(self.step_st)
        self._online_iterations += 1
        return dict(out, rewards=w["rewards"])

    @property
    def step_count(self) -> int:
        return int(self.step_dev.item())
