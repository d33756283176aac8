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
    stored rollout (device-shuffled minibatches of whole trajectories); `capture_epoch()` records it as one CUDA graph."""

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

    def grads(self, batch: dict, n_envs: int, critic_ready=None) -> dict:
        return self.eng.ppo_grad(batch, self.pa.as_dict(self.grad[:self.na]), self.pc.as_dict(self.grad[self.na:]), n_envs=n_envs,
                                 critic_ready=critic_ready, **self.loss_hyper)

    def _step(self, batch: dict, n_envs: int) -> dict:
        """One whole update, enqueued on the current stream (+ the communication stream, forked from / joined into it)."""
        import torch.distributed as dist

        world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        if world == 1:
            out = self.grads(batch, n_envs)
        else:
            cur = torch.cuda.current_stream()
            out = self.grads(batch, n_envs, critic_ready=self.ev_critic)
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

    def capture(self, batch: dict, n_envs: int) -> None:
        """Record one whole update on `batch` as ONE CUDA graph; later update() calls with the same batch object replay it
        (refill the batch tensors in place between updates).  Call after at least one eager update (allocations, NCCL)."""
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._graph_out = self._step(batch, n_envs)
        self._graph_batch = batch
        self.eng.scratch_lock(True)        # the graph holds pointers into the library's scratch: it must not be reallocated

    def update(self, batch: dict, n_envs: int) -> dict:
        if self._graph is not None and batch is self._graph_batch:
            self._graph.replay()
            return self._graph_out
        return self._step(batch, n_envs)

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

    def _epoch(self, rollout: dict, n_envs: int, batch_size: int, num_passes: int, seed: int) -> dict:
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
                out = self._step({k: t[b] for k, t in mb.items()}, batch_size)
                w["stats"][p * nb + b].copy_(out["stats"])
                w["norms"][p * nb + b:p * nb + b + 1].copy_(self.norm)
        return {"stats": w["stats"], "norms": w["norms"], "perm": w["perm"]}

    def epoch(self, rollout: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3, seed: int = 0) -> dict:
        """The update phase of one PPO epoch on a stored rollout: num_passes x (n_envs / batch_size) updates (train.py:1763-1766),
        each on a minibatch of whole trajectories taken from a fresh device-drawn permutation of the env axis.
        rollout: actor_obs [T,65,ld], critic_obs [T,475,ld], action [T,20,ld], done / success u8 [T,ld], rewards [T,ld], and the
        carries at the rollout's first step (snapshot them before kbs_rollout, which advances them): actor_carry0 /
        critic_carry0 [depth,2,n_envs,H], lpf0 [20,ld].  Returns device tensors, overwritten by the next epoch: "stats"
        [P*B, 4] loss statistics and "norms" [P*B] gradient norms per update, "perm" [P, n_envs] the permutations.  No host
        synchronisation.  After capture_epoch, a call on the same rollout object with the same arguments replays the graph."""
        if self._epoch_graph is not None and rollout is self._epoch_rollout and \
                self._epoch_args == (n_envs, batch_size, num_passes, seed):
            self._epoch_graph.replay()
            return self._epoch_out
        return self._epoch(rollout, n_envs, batch_size, num_passes, seed)

    def capture_epoch(self, rollout: dict, n_envs: int, batch_size: int = 512, num_passes: int = 3, seed: int = 0) -> None:
        """Record one whole epoch() on `rollout` as ONE CUDA graph; later epoch() calls with the same rollout object and
        arguments replay it (refill the rollout tensors in place between epochs).  Call after one eager epoch with the same
        arguments: the handle's scratch has then grown to what kbs_ppo_variables and kbs_ppo_grad need, and is locked here."""
        torch.cuda.synchronize()
        self._epoch_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._epoch_graph):
            self._epoch_out = self._epoch(rollout, n_envs, batch_size, num_passes, seed)
        self._epoch_rollout = rollout
        self._epoch_args = (n_envs, batch_size, num_passes, seed)
        self._epoch_graph_work = self._ework       # the graph holds its buffers' addresses: keep them if the shapes change
        self.eng.scratch_lock(True)

    @property
    def step_count(self) -> int:
        return int(self.step_dev.item())
