"""
sharded.py - time-slice sharding of ONE GRAPE evaluation across the GPUs of a box (SURVEY.md section 8e).

Magnus + expm of a slice depend only on the controls, so every rank owns a contiguous range of slices; only the
states (forward) and costates (backward) chain.  Protocol per cost+gradient evaluation (all stream-ordered, no
host synchronisation until the result is read):

    1. local   : expm of the local slices, product of the local propagators  -> P_g           (n x n)
       ALLGATHER P_g
    2. local   : incoming state P_{g-1} .. P_0 psi_0, local state sweeps, cost partial
    3. local   : costate at the shard's first state for zero incoming costate  -> b_g          (S x n)
       ALLGATHER b_g                                (affine recursion lam_in(g) = P_{g+1}^T lam_in(g+1) + b_{g+1})
    4. local   : incoming costate, local costate sweeps, expm / Magnus adjoints, gradient scatter
    5. ALLREDUCE [partial grad | partial cost | final states]

The CUDA phases are the `qocb_shard_*` entry points of the C ABI (include/qocb200.h); the collectives are
torch.distributed (NCCL over NVLink / NVSwitch on GPUs; gloo in the CPU protocol tests).  The driver below is
engine-agnostic: `CudaShardEngine` runs the phases on a B200, tests plug a NumPy engine in to exercise the
protocol at world_size 2 on CPU.
"""
import ctypes
import os

import numpy as np

from qoc_b200 import _lib
from qoc_b200.core.plan import SchroedingerPlan
from qoc_b200.models.enums import InterpolationPolicy, MagnusPolicy


def slice_bounds(slice_count, world):
    """contiguous, balanced partition of `slice_count` time slices: rank g owns [b[g], b[g+1])."""
    if world > slice_count:
        raise ValueError("cannot shard {} time slices over {} ranks".format(slice_count, world))
    return [(g * slice_count) // world for g in range(world + 1)]


class CudaShardEngine(object):
    """one rank's phases on its GPU.  Exchange buffers are torch CUDA tensors; their device pointers go through the
    C ABI.  All work is enqueued on the plan's stream (exposed as `self.stream`, a torch ExternalStream)."""

    def __init__(self, rank, world, hamiltonian, initial_states, costs, evolution_time, system_eval_count,
                 control_eval_count=0, control_count=0, complex_controls=False, magnus_policy=MagnusPolicy.M2,
                 cost_eval_step=1, interpolation_policy=InterpolationPolicy.LINEAR, device=0, store_tape=True,
                 chunks_per_member=0, structure=None):
        import torch
        self.torch = torch
        self.rank, self.world = rank, world
        b = slice_bounds(system_eval_count - 1, world)
        self.slice_range = (b[rank], b[rank + 1])
        self.plan = SchroedingerPlan(hamiltonian, initial_states, costs, evolution_time, system_eval_count,
                                     control_eval_count=control_eval_count, control_count=control_count,
                                     complex_controls=complex_controls, magnus_policy=magnus_policy,
                                     cost_eval_step=cost_eval_step, interpolation_policy=interpolation_policy,
                                     device=device, store_tape=store_tape, chunks_per_member=chunks_per_member,
                                     structure=structure, slice_range=self.slice_range)
        p, lib = self.plan, self.plan.lib
        self.lib, self.h = lib, p.handle
        self.GM = lib.qocb_shard_matrix_doubles(self.h)
        self.VS = lib.qocb_shard_vector_doubles(self.h)
        self.RS = lib.qocb_shard_result_doubles(self.h)
        self.NP = self.VS // (2 * p.S)
        self.dev = torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(lib.qocb_stream(self.h), device=self.dev)
        kw = dict(dtype=torch.float64, device=self.dev)
        self.P, self.b, self.result = torch.zeros(self.GM, **kw), torch.zeros(self.VS, **kw), torch.zeros(self.RS, **kw)

    def _ptr(self, t):
        return ctypes.c_void_p(t.data_ptr())

    def upload(self, controls):
        self.plan.upload(controls)

    def forward_local(self, with_grad):
        _lib.check(self.lib.qocb_shard_forward_local(self.h, int(with_grad), self._ptr(self.P)), self.h)
        return self.P

    def forward_finish(self, all_p):
        _lib.check(self.lib.qocb_shard_forward_finish(self.h, self._ptr(all_p), self.rank), self.h)

    def backward_particular(self):
        _lib.check(self.lib.qocb_shard_backward_particular(self.h, self._ptr(self.b)), self.h)
        return self.b

    def backward_finish(self, all_p, all_b):
        _lib.check(self.lib.qocb_shard_backward_finish(self.h, self._ptr(all_p), self._ptr(all_b), self.rank,
                                                       self.world), self.h)

    def pack_result(self, with_grad):
        _lib.check(self.lib.qocb_shard_pack_result(self.h, int(with_grad), self._ptr(self.result)), self.h)
        return self.result

    def flush_l2(self):
        _lib.check(self.lib.qocb_flush_l2(self.h), self.h)

    def unpack(self, host):
        """host: 1-D float64 array [grad M*KR | cost | finals S*2*NP] -> (cost, grad (M x KR), finals (S x n x 1))."""
        p = self.plan
        cnt = p.M * p.KR
        fin = host[cnt + 1:].reshape(p.S, 2, self.NP)
        finals = (fin[:, 0, :p.n] + 1j * fin[:, 1, :p.n])[:, :, None]
        return float(host[cnt]), host[:cnt].reshape(p.M, p.KR).copy(), finals

    def launch_count(self, with_grad=True):
        return self.plan.launch_count(with_grad)

    def close(self):
        # free the exchange tensors while the plan stream still exists: torch's caching allocator records an event
        # on every stream a block was used on when the block is released
        if getattr(self, "plan", None) is None:
            return
        self.stream.synchronize()
        self.P = self.b = self.result = None
        self.torch.cuda.synchronize(self.dev)
        self.plan.close()
        self.plan = None


class TorchDistComm(object):
    """collectives of the protocol on torch.distributed (NCCL on GPUs, gloo on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group

    def all_gather(self, out, inp):
        self.dist.all_gather_into_tensor(out, inp, group=self.group)

    def all_reduce_sum(self, t):
        self.dist.all_reduce(t, group=self.group)


def sharded_evaluate(engine, comm, all_p, all_b, with_grad, mark=None):
    """the protocol of the module docstring for one rank; returns the all-reduced result tensor (device).
    mark: optional callable invoked after every phase (stage timing)."""
    mark = mark or (lambda: None)
    p_loc = engine.forward_local(with_grad)
    mark()
    comm.all_gather(all_p, p_loc)
    mark()
    engine.forward_finish(all_p)
    mark()
    if with_grad:
        b_loc = engine.backward_particular()
        mark()
        comm.all_gather(all_b, b_loc)
        mark()
        engine.backward_finish(all_p, all_b)
        mark()
    res = engine.pack_result(with_grad)
    comm.all_reduce_sum(res)
    mark()
    return res


class ShardedSchroedingerPlan(object):
    """`SchroedingerPlan` interface (cost / cost_and_grad / upload / time_resident / launch_count / close) over
    all ranks of the default torch.distributed group, one process per GPU."""

    def __init__(self, hamiltonian, initial_states, costs, evolution_time, system_eval_count, device=0,
                 group=None, **kw):
        import torch
        import torch.distributed as dist
        self.torch = torch
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.comm = TorchDistComm(group)
        self.engine = CudaShardEngine(self.rank, self.world, hamiltonian, initial_states, costs, evolution_time,
                                      system_eval_count, device=device, **kw)
        e = self.engine
        self.plan = e.plan
        self.KR, self.K, self.M, self.S, self.n, self.E = e.plan.KR, e.plan.K, e.plan.M, e.plan.S, e.plan.n, 1
        self.complex_controls = e.plan.complex_controls
        kwt = dict(dtype=torch.float64, device=e.dev)
        self.all_p = torch.zeros(self.world * e.GM, **kwt)
        self.all_b = torch.zeros(self.world * e.VS, **kwt)
        self.host = torch.zeros(e.RS, dtype=torch.float64).pin_memory()

    def _run(self, with_grad):
        with self.torch.cuda.stream(self.engine.stream):
            res = sharded_evaluate(self.engine, self.comm, self.all_p, self.all_b, with_grad)
        return res

    def _evaluate(self, controls, with_grad):
        e = self.engine
        e.upload(controls)
        with self.torch.cuda.stream(e.stream):
            res = sharded_evaluate(e, self.comm, self.all_p, self.all_b, with_grad)
            self.host.copy_(res, non_blocking=True)
        e.stream.synchronize()
        return e.unpack(self.host.numpy())

    def cost(self, controls):
        cost, _, finals = self._evaluate(controls, False)
        extra, _ = self.plan._control_costs(controls, False) if controls is not None else (0.0, None)
        return cost + extra, finals

    def cost_and_grad(self, controls):
        cost, g, finals = self._evaluate(controls, True)
        grads = g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g
        extra, extra_grad = self.plan._control_costs(np.asarray(controls), True)
        if extra_grad is not None:
            grads = grads + extra_grad
        return cost + extra, grads, finals

    def upload(self, controls):
        self.engine.upload(controls)

    def time_resident(self, with_grad=True, warmup=3, iters=10, flush_l2=True):
        """device time of `iters` resident evaluations (CUDA events on the plan stream; this rank's clock - the
        caller takes the max over ranks).  Stage split is not available across the collectives: stages[0] = total."""
        torch, e = self.torch, self.engine
        for _ in range(warmup):
            self._run(with_grad)
        e.stream.synchronize()
        total = 0.0
        stages = np.zeros(8)
        stage_timing = os.environ.get("QOCB_STAGE_TIMING") == "1"      # extra events: diagnostics, not for bench numbers
        for _ in range(iters):
            if flush_l2:
                e.flush_l2()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            evs = []

            def mark():
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                evs.append(ev)
            with torch.cuda.stream(e.stream):
                t0.record()
                sharded_evaluate(e, self.comm, self.all_p, self.all_b, with_grad, mark if stage_timing else None)
                t1.record()
            e.stream.synchronize()
            total += t0.elapsed_time(t1)
            prev = t0
            for i, ev in enumerate(evs):         # forward_local, gather P, forward_finish, particular, gather b, finish, pack+reduce
                stages[1 + i] += prev.elapsed_time(ev)
                prev = ev
        stages[0] = total
        return total, stages

    def launch_count(self, with_grad=True):
        return self.engine.launch_count(with_grad)

    def close(self):
        if self.engine is None:
            return
        self.engine.stream.synchronize()
        self.all_p = self.all_b = self.host = None
        self.torch.cuda.synchronize()
        self.engine.close()
        self.engine = None


def units_evaluate(engine, comm, with_grad):
    """sharding of INDEPENDENT units - ensemble members, initial states - across ranks (SURVEY.md section 8e): every rank
    runs the whole time loop for its units; there is no data-path exchange except
      * the coherent overlap sums sum_s <t_s|psi_s> of `TargetStateInfidelity` when STATES are sharded (the cost couples the
        states through |sum_s ip_s|^2, targetstateinfidelity.py:53-55): one all-reduce of a few complex numbers between the
        forward and the backward pass (`engine.forward` returns them, empty when nothing couples);
      * one all-reduce of [gradient | cost] at the end (each rank's contribution already weighted).
    Engine interface: forward(with_grad) -> coherent partial sums (tensor, may be empty); backward(coherent_totals);
    pack(with_grad) -> result tensor.  `CudaUnitEngine` runs it on a B200, tests/numpy_unit_engine.py on CPU (gloo)."""
    coh = engine.forward(with_grad)
    if coh is not None and coh.numel() > 0:
        comm.all_reduce_sum(coh)
    if with_grad:
        engine.backward(coh)
    res = engine.pack(with_grad)
    comm.all_reduce_sum(res)
    return res


class CudaUnitEngine(object):
    """one rank's share of an ensemble (members differ in the drift) on its GPU: the unsharded device pipeline over the
    local members, the result [gradient | cost] packed on the device and weighted by members_local / members_total (the
    cost of an ensemble is the mean over its members)."""

    def __init__(self, plan, weight, device):
        import torch
        self.torch, self.plan, self.lib, self.h = torch, plan, plan.lib, plan.handle
        self.dev = torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(self.lib.qocb_stream(self.h), device=self.dev)
        self.count = plan.M * plan.KR
        self.weight = float(weight)
        self.result = torch.zeros(self.lib.qocb_shard_result_doubles(self.h), dtype=torch.float64, device=self.dev)
        self.out = self.result[:self.count + 1]                     # [gradient | cost]; the tail (final states) stays local

    def forward(self, with_grad):
        _lib.check(self.lib.qocb_run_resident(self.h, int(with_grad)), self.h)      # whole pipeline: members are independent
        return None

    def backward(self, coh):
        pass

    def pack(self, with_grad):
        _lib.check(self.lib.qocb_shard_pack_result(self.h, int(with_grad), ctypes.c_void_p(self.result.data_ptr())), self.h)
        self.out.mul_(self.weight)                                  # enqueued on the plan stream (the caller made it current)
        return self.out

    def close(self):
        self.stream.synchronize()
        self.result = self.out = None
        self.torch.cuda.synchronize(self.dev)


class CudaStateEngine(object):
    """one rank's share of the initial STATES on its GPU (`units_evaluate` interface): every rank computes every slice
    propagator and sweeps its own states; the coherent overlap sums of TargetStateInfidelity are the only coupling."""

    def __init__(self, plan, device):
        import torch
        self.torch, self.plan, self.lib, self.h = torch, plan, plan.lib, plan.handle
        self.dev = torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(self.lib.qocb_stream(self.h), device=self.dev)
        self.count = plan.M * plan.KR
        ncoh = self.lib.qocb_state_shard_coherent_doubles(self.h)
        self.coh = torch.zeros(max(ncoh, 0), dtype=torch.float64, device=self.dev)
        self.result = torch.zeros(self.lib.qocb_shard_result_doubles(self.h), dtype=torch.float64, device=self.dev)
        self.out = self.result[:self.count + 1]

    def _coh_ptr(self):
        return ctypes.c_void_p(self.coh.data_ptr()) if self.coh.numel() else None

    def forward(self, with_grad):
        self.with_grad = with_grad
        _lib.check(self.lib.qocb_state_shard_forward(self.h, int(with_grad), self._coh_ptr()), self.h)
        return self.coh

    def backward(self, coh):
        _lib.check(self.lib.qocb_state_shard_finish(self.h, 1, self._coh_ptr()), self.h)

    def pack(self, with_grad):
        if not with_grad:                                           # forward only: the coherent values still need the totals
            _lib.check(self.lib.qocb_state_shard_finish(self.h, 0, self._coh_ptr()), self.h)
        _lib.check(self.lib.qocb_shard_pack_result(self.h, int(with_grad), ctypes.c_void_p(self.result.data_ptr())), self.h)
        return self.out

    def close(self):
        self.stream.synchronize()
        self.coh = self.result = self.out = None
        self.torch.cuda.synchronize(self.dev)


class StateShardedPlan(object):
    """independent initial states sharded across the ranks of the default group (SURVEY.md section 8e; BASELINE north star:
    "independent initial states and ensemble members are also sharded").  Pays off when the state sweeps and the rank-S / dense
    reverse pass weigh against the (replicated) expm work, i.e. many states on a small Hilbert space (cfg5: S = 64, n = 32).
    `cost_and_grad` returns the final states of ALL states (all-gathered)."""

    def __init__(self, hamiltonian, initial_states, costs, evolution_time, system_eval_count, device=0, group=None, **kw):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.group = torch, dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.comm = TorchDistComm(group)
        initial_states = np.asarray(initial_states)
        self.S_total = initial_states.shape[0]
        self.bounds = slice_bounds(self.S_total, self.world)
        sl = (self.bounds[self.rank], self.bounds[self.rank + 1])
        self.plan = SchroedingerPlan(hamiltonian, initial_states, costs, evolution_time, system_eval_count, device=device,
                                     state_slice=sl, **kw)
        p = self.plan
        self.KR, self.K, self.M, self.S, self.n, self.E = p.KR, p.K, p.M, self.S_total, p.n, 1
        self.complex_controls = p.complex_controls
        self.engine = CudaStateEngine(p, device)
        self.host = torch.zeros(p.M * p.KR + 1, dtype=torch.float64).pin_memory()
        self.smax = max(self.bounds[g + 1] - self.bounds[g] for g in range(self.world))
        kwt = dict(dtype=torch.complex128, device=self.engine.dev)
        self.fin_local = torch.zeros(self.smax * p.n, **kwt)
        self.fin_all = torch.zeros(self.world * self.smax * p.n, **kwt)

    def upload(self, controls):
        self.plan.upload(controls)

    def _evaluate(self, controls, with_grad):
        e, p = self.engine, self.plan
        p.upload(controls)
        with self.torch.cuda.stream(e.stream):
            res = units_evaluate(e, self.comm, with_grad)
            self.host.copy_(res, non_blocking=True)
        e.stream.synchronize()
        out = self.host.numpy()
        local = p.final_states()                                    # (S_local, n, 1)
        self.fin_local.zero_()
        self.fin_local[:local.size] = self.torch.from_numpy(np.ascontiguousarray(local).ravel()).to(self.engine.dev)
        self.dist.all_gather_into_tensor(self.fin_all, self.fin_local, group=self.group)
        allf = self.fin_all.cpu().numpy().reshape(self.world, self.smax, p.n)
        finals = np.concatenate([allf[g, :self.bounds[g + 1] - self.bounds[g]] for g in range(self.world)])[:, :, None]
        extra, extra_grad = p._control_costs(np.asarray(controls), with_grad)
        g = out[:-1].reshape(self.M, self.KR).copy()
        grads = g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g
        if with_grad and extra_grad is not None:
            grads = grads + extra_grad
        return float(out[-1]) + extra, grads, finals

    def cost(self, controls):
        err, _, finals = self._evaluate(controls, False)
        return err, finals

    def cost_and_grad(self, controls):
        return self._evaluate(controls, True)

    def time_resident(self, with_grad=True, warmup=3, iters=10, flush_l2=True):
        """device time of `iters` resident evaluations including both all-reduces (this rank's clock)."""
        torch, e = self.torch, self.engine
        for _ in range(warmup):
            with torch.cuda.stream(e.stream):
                units_evaluate(e, self.comm, with_grad)
        e.stream.synchronize()
        total = 0.0
        for _ in range(iters):
            if flush_l2:
                _lib.check(self.plan.lib.qocb_flush_l2(self.plan.handle), self.plan.handle)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(e.stream):
                t0.record()
                units_evaluate(e, self.comm, with_grad)
                t1.record()
            e.stream.synchronize()
            total += t0.elapsed_time(t1)
        stages = np.zeros(8)
        stages[0] = total
        return total, stages

    def launch_count(self, with_grad=True):
        return self.plan.launch_count(with_grad) + 2

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
            self.host = self.fin_local = self.fin_all = None
            self.plan.close()


def member_share(rank, world, **members):
    """rank's block of every per-member argument given (name=[E] sequence or None): (local arguments, (first, end), E).
    The members are block-partitioned as `slice_bounds` partitions slices; ValueError when the arguments disagree on E."""
    given = {k: v for k, v in members.items() if v is not None}
    counts = {k: len(v) for k, v in given.items()}
    if len(set(counts.values())) != 1:
        raise ValueError("the per-member arguments disagree on the member count: " +
                         ", ".join("{} has {}".format(k, v) for k, v in sorted(counts.items())))
    E = next(iter(counts.values()))
    b = slice_bounds(E, world)
    lo, hi = b[rank], b[rank + 1]
    return {k: v[lo:hi] for k, v in given.items()}, (lo, hi), E


class EnsembleShardedPlan(object):
    """robust-control ensembles (cfg5): members that differ in the drift (`ensemble_drifts`) or in drift and control
    operators (`ensemble_hamiltonians`, callables like `hamiltonian`), and optionally in their initial states and cost
    targets (`ensemble_initial_states`, `ensemble_costs`; a shared drift is `ensemble_drifts=[h0] * E`), are independent
    units, block-partitioned across the ranks; one NCCL all-reduce of [gradient | cost] on the plan stream ends the
    evaluation - inside the device-timed region, no host bounce.  Cost = mean over members.  `cost_and_grad` returns the
    final states of the LOCAL members."""

    def __init__(self, hamiltonian, initial_states, costs, evolution_time, system_eval_count, ensemble_drifts=None, device=0,
                 group=None, ensemble_hamiltonians=None, ensemble_initial_states=None, ensemble_costs=None, **kw):
        if (ensemble_drifts is None) == (ensemble_hamiltonians is None):
            raise ValueError("EnsembleShardedPlan needs exactly one of ensemble_drifts and ensemble_hamiltonians")
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.group = torch, dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.comm = TorchDistComm(group)
        local, self.member_range, self.E_total = member_share(
            self.rank, self.world, ensemble_drifts=None if ensemble_drifts is None else np.asarray(ensemble_drifts),
            ensemble_hamiltonians=None if ensemble_hamiltonians is None else list(ensemble_hamiltonians),
            ensemble_initial_states=None if ensemble_initial_states is None else np.asarray(ensemble_initial_states),
            ensemble_costs=None if ensemble_costs is None else list(ensemble_costs))
        self.plan = SchroedingerPlan(hamiltonian, initial_states, costs, evolution_time, system_eval_count, device=device,
                                     **local, **kw)
        p = self.plan
        self.KR, self.K, self.M, self.S, self.n, self.E = p.KR, p.K, p.M, p.S, p.n, p.E
        self.complex_controls = p.complex_controls
        self.engine = CudaUnitEngine(p, float(p.E) / self.E_total, device)
        self.host = torch.zeros(p.M * p.KR + 1, dtype=torch.float64).pin_memory()

    def upload(self, controls):
        self.plan.upload(controls)

    def _evaluate(self, controls, with_grad):
        e = self.engine
        self.plan.upload(controls)
        with self.torch.cuda.stream(e.stream):
            res = units_evaluate(e, self.comm, with_grad)
            self.host.copy_(res, non_blocking=True)
        e.stream.synchronize()
        out = self.host.numpy()
        extra, extra_grad = self.plan._control_costs(np.asarray(controls), with_grad)
        g = out[:-1].reshape(self.M, self.KR).copy()
        grads = g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g
        if with_grad and extra_grad is not None:
            grads = grads + extra_grad
        return float(out[-1]) + extra, grads, self.plan.final_states()

    def cost(self, controls):
        err, _, finals = self._evaluate(controls, False)
        return err, finals

    def cost_and_grad(self, controls):
        """(mean cost, gradient of the mean cost, final states of the LOCAL members)."""
        return self._evaluate(controls, True)

    def time_resident(self, with_grad=True, warmup=3, iters=10, flush_l2=True):
        """device time of `iters` resident evaluations INCLUDING the closing all-reduce (CUDA events on the plan stream, this
        rank's clock; the caller takes the max over ranks).  stages: per-kernel split of the local pipeline from one extra
        evaluation timed by the C ABI, scaled to `iters`."""
        torch, e = self.torch, self.engine
        for _ in range(warmup):
            with torch.cuda.stream(e.stream):
                units_evaluate(e, self.comm, with_grad)
        e.stream.synchronize()
        total = 0.0
        for _ in range(iters):
            if flush_l2:
                _lib.check(self.plan.lib.qocb_flush_l2(self.plan.handle), self.plan.handle)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(e.stream):
                t0.record()
                units_evaluate(e, self.comm, with_grad)
                t1.record()
            e.stream.synchronize()
            total += t0.elapsed_time(t1)
        _, stages = self.plan.time_resident(with_grad, 0, 1, flush_l2)
        return total, np.asarray(stages) * iters

    def launch_count(self, with_grad=True):
        return self.plan.launch_count(with_grad) + 2                # + pack, scale

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
            self.host = None
            self.plan.close()
