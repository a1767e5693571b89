"""Monte-Carlo sample sharding, the one exchange of the forward path, and the heads above it (SURVEY.md 8e, f3, f4).

The reference's ``num_ens`` loop (main_bayesian.py:46-53, validate :75-80; uncertainty_estimation.py:70-78) runs S
independent weight samples of the SAME batch and combines them with logmeanexp of log-softmax.  Samples only differ in
their noise, so rank r of R takes the global sample ids {j : j mod R == r} (Philox stream namespace of sample j:
results do not depend on R) and ONE exchange carries the per-(image, class) partials and the KL.

Two implementations of the same contract:

* ``MCForward`` / ``mc_forward(net, ...)`` -- the product path on the CUDA engine: the local samples run through the
  engine (fused tcgen05 chain where the net allows), then ONE kernel (``bbb_mc_exchange``, csrc/mc_head.cuh) reduces
  them, pushes the partials into every peer's receive buffer over NVLink (CUDA-IPC peer-mapped memory, no NCCL on the
  data path), waits for the peers and finishes logmeanexp, KL/num_ens, the ELBO head (metrics.py:12-14, 23-24) and the
  uncertainty outputs (uncertainty_estimation.py:80-96, softmax or softplus-normalised :73-77) on the device.  The whole
  step is one captured CUDA graph.
* ``mc_forward(forward_fn, ...)`` with a plain callable -- backend-agnostic host logic on torch.distributed (gloo on
  CPU in the tests): same sharding, same exact (max, sum-exp) partials, one all-gather.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import os
import torch

from . import _lib as L
from . import functional as Fn


def local_samples(num_ens: int, world: int, rank: int):
    """Global sample ids owned by `rank` (round-robin; C4: 25 samples over 8 ranks -> 4,3,3,...)."""
    return list(range(rank, num_ens, world))


def get_beta(batch_idx, m, beta_type, epoch=None, num_epochs=None):
    """metrics.py:32-46 (host scalar; it only feeds the `beta` argument of the ELBO head)."""
    if isinstance(beta_type, (int, float)):
        return float(beta_type)
    if beta_type == "Blundell":
        return 2 ** (m - (batch_idx + 1)) / (2 ** m - 1)
    if beta_type == "Soenderby":
        if epoch is None or num_epochs is None:
            raise ValueError("Soenderby method requires both epoch and num_epochs to be passed.")
        return min(epoch / (num_epochs // 4), 1)
    if beta_type == "Standard":
        return 1 / m
    return 0


def _dist_info(group):
    import torch.distributed as dist
    on = dist.is_available() and dist.is_initialized()
    return (dist if on else None), (dist.get_world_size(group) if on else 1), (dist.get_rank(group) if on else 0)


class MCForward:
    """``out = MCForward(net, example_x, num_ens, ...)(x, labels=None)`` -- the sharded MC step on the engine.

    Returns a dict of device tensors (the same objects every call; identical on all ranks):
      log_outputs [B,C], kl (= sum_j kl_j / num_ens), and with ``want_uncertainty`` pred / epistemic / aleatoric [B,C]
      and entropy [B]; with ``with_labels`` head = [loss, nll, accuracy, beta*kl] (metrics.py:12-14, 23-24).
    """

    def __init__(self, net, example_x: torch.Tensor, num_ens: int, group=None, want_uncertainty: bool = False,
                 normalized: bool = False, with_labels: bool = False, train_size: float = 1.0, beta: float = 0.0,
                 seed: Optional[int] = None, graph: bool = True, num_classes: Optional[int] = None,
                 static_inputs=None, first_replay: int = 0, fold: bool = True, overlap: bool = False, inflight: int = 1):
        """``static_inputs``: device tensors the caller fills in place (e.g. targets of its host->device copies, or a
        rotation of resident batches); one graph is captured per tensor and ``self(slot=k)`` runs the step on
        ``static_inputs[k]`` with no staging copy.  ``first_replay``: index of the first replay's noise block.
        ``overlap``: run the exchange kernel of step t on its own stream, beside the first kernels of step t+1 (the
        layer chain of a step does not depend on the previous step's exchange; logits / KL terms / labels are double
        buffered).  The returned tensors are then complete on ``result_stream`` -- call ``wait()`` before using them on the
        current stream (a device synchronize covers it too).  ``inflight=k`` (with ``overlap``): consecutive steps are
        independent, so steps t, t+1, .. t+k-1 run on k streams with their own layer workspaces and Philox counters -- the
        head of step t+1 (parameter preps, first layers) fills the SMs the tail of step t leaves idle.  Results are
        identical to the serial engine; ``wait()`` also covers the inputs (they may be rewritten afterwards)."""
        Fn._require_cuda(example_x, "MCForward")
        lib = L.lib()
        self.net, self.group = net, group
        self.dist, self.world, self.rank = _dist_info(group)
        if self.world > 16:
            raise L.EngineError("MCForward: at most 16 ranks (one node)")
        dev = self.dev = example_x.device
        self.num_ens = int(num_ens)
        self.ids = local_samples(self.num_ens, self.world, self.rank)
        self.B = int(example_x.shape[0])
        self.C = int(num_classes if num_classes is not None else net.num_classes)
        self.flags = (L.MC_MOMENTS if want_uncertainty else 0) | (L.MC_NORMALIZED if normalized else 0)
        self.want_uncertainty, self.with_labels = want_uncertainty, with_labels
        self.train_size, self.beta = float(train_size), float(beta)
        # every rank must draw sample j from the same (seed, stream): share rank 0's seed unless one is given
        if seed is None:
            box = [Fn.current_seed()]
            if self.world > 1:
                self.dist.broadcast_object_list(box, src=self.dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            seed = box[0]
        self.seed = int(seed)
        B, Cc = self.B, self.C
        f32 = dict(dtype=torch.float32, device=dev)
        self.inputs = list(static_inputs) if static_inputs else [example_x.clone()]
        assert all(t.is_cuda and t.shape == example_x.shape and t.is_contiguous() for t in self.inputs)
        self.x = self.inputs[0]
        self.first_replay = int(first_replay)
        self.overlap = bool(overlap) and graph
        self.inflight = max(1, min(int(inflight), 8)) if self.overlap else 1
        self.nbuf = max(2, self.inflight) if self.overlap else 1
        nbuf = self.nbuf
        self.labels_all = torch.zeros(nbuf, B, dtype=torch.int64, device=dev) if with_labels else None
        self.labels = self.labels_all[0] if with_labels else None
        self.logits_all = torch.zeros(nbuf, max(1, len(self.ids)), B, Cc, **f32)
        self.logits = self.logits_all[0]
        self.kl_one_all = torch.zeros(nbuf, **f32)
        self.kl_one = self.kl_one_all[0]
        self.kl_terms_all = torch.zeros(nbuf, 64, **f32)
        self.out = {"log_outputs": torch.empty(B, Cc, **f32), "kl": torch.empty((), **f32)}
        if want_uncertainty:
            for k in ("pred", "epistemic", "aleatoric"):
                self.out[k] = torch.empty(B, Cc, **f32)
            self.out["entropy"] = torch.empty(B, **f32)
        if with_labels:
            self.out["head"] = torch.empty(4, **f32)
        self.state = torch.zeros(int(lib.bbb_mc_state_bytes()), dtype=torch.uint8, device=dev)
        nbytes = int(lib.bbb_mc_buffer_bytes(B, Cc, self.flags, self.world))
        self._imported, self._own = [], None
        if self.world == 1:
            self._buf = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
            ptrs = [self._buf.data_ptr()]
        else:
            ptrs = self._open_peers(nbytes)
        self.peers = (C.c_void_p * self.world)(*ptrs)
        self.base = torch.zeros(1, dtype=torch.int64, device=dev)
        # LRT nets: the local samples differ only in their per-activation noise, so they FOLD into the batch -- one pass
        # of the fused chain over S_local*B rows (what uncertainty_estimation.py:38-41 does by repeating the input), each
        # row drawing from its own sample's Philox stream; the KL is computed once.  BBB nets (a weight draw per sample)
        # and nets the chain cannot take run sample by sample.
        self.fold_steps = None
        from . import fused
        from .modules import _BayesLayer
        kids = list(net.children())
        layers = [m_ for m_ in kids if isinstance(m_, _BayesLayer)]
        all_lrt = bool(layers) and all(m_._variant == L.VARIANT_LRT for m_ in layers) and getattr(net, "fuse", True)
        if fold and len(self.ids) > 1 and all_lrt:
            self.fold = (self.B, self.world << 40)
            self.fold_steps = fused.plan(kids, (len(self.ids) * self.B,) + tuple(example_x.shape[1:]), self.fold)
        self.graph, self.graphs = None, []
        self.result_stream = None                 # overlap mode: the stream the results are complete on
        self.replays = 0
        self.kernels_per_step = None
        if graph:
            self._capture()

    # -- peer-mapped receive buffers (CUDA IPC; handles travel over torch.distributed) -----------------------
    def _open_peers(self, nbytes):
        lib = L.lib()
        torch.cuda.synchronize(self.dev)
        own = C.c_void_p()
        with torch.cuda.device(self.dev):
            L.check(lib.bbb_comm_alloc(C.c_size_t(nbytes), C.byref(own)), "bbb_comm_alloc")
            self._own = own.value
            handle = (C.c_ubyte * 64)()
            L.check(lib.bbb_comm_export(C.c_void_p(self._own), handle), "bbb_comm_export")
            handles = [None] * self.world
            self.dist.all_gather_object(handles, bytes(handle), group=self.group)
            ptrs = []
            for q, h in enumerate(handles):
                if q == self.rank:
                    ptrs.append(self._own)
                    continue
                peer = C.c_void_p()
                L.check(lib.bbb_comm_import((C.c_ubyte * 64).from_buffer_copy(h), C.byref(peer)), f"bbb_comm_import (rank {q})")
                self._imported.append(peer.value)
                ptrs.append(peer.value)
        self.dist.barrier(group=self.group)
        return ptrs

    def timeouts(self) -> int:
        """Exchange waits that gave up because a peer never delivered (results of those steps are invalid)."""
        return int(self.state[8:12].view(torch.int32).item())

    def close(self):
        """Unmap the peers' buffers and free the local one (after every rank is done with them)."""
        lib = L.lib()
        if self.world > 1 and self._own is not None:
            torch.cuda.synchronize(self.dev)
            self.dist.barrier(group=self.group)
            for p in self._imported:
                lib.bbb_comm_unimport(C.c_void_p(p))
            lib.bbb_comm_free(C.c_void_p(self._own))
            self._imported, self._own = [], None

    # -- one step ----------------------------------------------------------------------------------------------
    def _step(self, x, base=None, advance=False):
        """This rank's samples through the engine, then the exchange kernel."""
        kl_ptr, n_kl = self._chain(x, base, advance)
        self._exchange(kl_ptr, n_kl)
        return self.out

    def _chain(self, x, base=None, advance=False, par=0):
        """This rank's samples through the engine into the sample buffer ``par``.  A fused chain writes its logits
        straight into it and hands over its per-layer KL scalars un-summed (fused.direct_output).  Returns the (pointer,
        count) of the floats whose sum is one sample's KL."""
        from . import fused
        from .graph import _STRIDE
        logits_buf = self.logits_all[par]
        kl_buf = self.kl_terms_all[par] if self.overlap else None
        inc = _STRIDE * self.inflight
        with torch.no_grad(), Fn.workspace_slot(par if self.inflight > 1 else Fn.current_workspace_slot()):
            # The Philox base moves at the HEAD of a captured step, BEFORE the prep streams fork.  Measured (B200, captured
            # step, tools/quick_step.py): with this one-thread kernel as the single root of the graph every GEMM kernel of
            # the chain is launched programmatically behind its predecessor (100 us per step); with the fork in front of it
            # (prep kernels as further root nodes) or with no plain kernel at the head, the programmatic edges of the whole
            # chain are lost -- every GEMM then starts ~3 us after its predecessor ends (132 us per step).
            if advance:
                Fn.noise_advance(base, inc)
            kl_ptr, n_kl = None, 0
            if self.fold_steps is not None:
                with Fn.stream_base(base), Fn.mc_sample(self.ids[0], self.seed):
                    _, kls = fused.run(self.fold_steps, x, out=logits_buf.view(len(self.ids) * self.B, self.C), terms=True,
                                       fold=self.fold, kls_out=kl_buf)
                self._kl_terms = kls
                kl_ptr, n_kl = Fn._ptr(kls), kls.numel()
            for k, j in enumerate(self.ids if self.fold_steps is None else ()):
                with Fn.stream_base(base), Fn.mc_sample(j, self.seed), \
                        fused.direct_output(logits_buf[k], kl_buf if k == 0 else None) as hook:
                    logits, kl = self.net(x)
                if not hook.used:
                    logits_buf[k].copy_(logits.reshape(self.B, self.C))
                if k == 0:
                    if hook.used:
                        self._kl_terms = kl                       # per-layer scalars of sample 0 (every sample has the same KL)
                        kl_ptr, n_kl = Fn._ptr(kl), kl.numel()
                    else:
                        one = self.kl_one_all[par:par + 1]
                        one.copy_(torch.as_tensor(kl, dtype=torch.float32, device=self.dev).reshape(1))
                        kl_ptr, n_kl = Fn._ptr(one), 1
            if not self.ids and self.rank == 0:
                raise L.EngineError("MCForward: rank 0 must own a sample")
        return kl_ptr, n_kl

    def _exchange(self, kl_ptr, n_kl, advance_base=None, par=0):
        """The one kernel behind the samples: combine + exchange + heads (bbb_mc_exchange)."""
        from .graph import _STRIDE
        o = self.out
        rc = L.lib().bbb_mc_exchange(
            Fn._ptr(self.logits_all[par]), len(self.ids), self.num_ens, self.B, self.C, kl_ptr, n_kl, self.flags,
            Fn._ptr(self.labels_all[par] if self.labels_all is not None else None), C.c_float(self.train_size), C.c_float(self.beta), self.rank, self.world, self.peers,
            Fn._ptr(self.state), Fn._ptr(o["log_outputs"]), Fn._ptr(o["kl"]), Fn._ptr(o.get("pred")),
            Fn._ptr(o.get("epistemic")), Fn._ptr(o.get("aleatoric")), Fn._ptr(o.get("entropy")), Fn._ptr(o.get("head")),
            Fn._ptr(advance_base), C.c_uint64(_STRIDE if advance_base is not None else 0), Fn._stream(self.dev))
        L.check(rc, "bbb_mc_exchange")

    def _capture(self, warmup: int = 2):
        # several steps in flight: the tap-GEMM layers take their 128-column tiles wherever Cout allows (throughput over the
        # latency of one step; the choice is made at launch = capture time, include/bbb_b200.h bbb_set_wide_tiles)
        prev_wide = L.lib().bbb_set_wide_tiles(1 if self.inflight > 1 else 0)
        try:
            self._capture_graphs(warmup)
        finally:
            L.lib().bbb_set_wide_tiles(prev_wide)

    def _capture_graphs(self, warmup):
        from .graph import _STRIDE
        dev = self.dev
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):                 # eager: creates plans / workspaces; every rank runs the same exchanges
                self._step(self.x, self.base)
            for p_ in range(1, self.inflight):      # the other in-flight steps' own layer workspaces
                self._exchange(*self._chain(self.x, self.base, par=p_), par=p_)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        # GEMM chain on a HIGH-priority stream, parameter preps on the (default-priority) side streams: when both have CTAs
        # pending, the chain's go first -- the preps of later layers no longer keep the first GEMM's CTAs off the SMs
        cap = torch.cuda.Stream(device=dev, priority=-1)
        if self.overlap:
            # two graphs per step: the layer chain (per resident input and buffer parity) and the exchange kernel (per
            # parity); __call__ replays the second on its own stream so that it runs beside the next step's chain
            nb = self.nbuf
            self.chain_graphs, self.exch_graphs = [[] for _ in range(nb)], []
            self.base2 = torch.zeros(nb, dtype=torch.int64, device=dev)
            self._bases = [self.base2[p_:p_ + 1] for p_ in range(nb)] if self.inflight > 1 else [self.base] * nb
            for par in range(nb):
                for xin in self.inputs:
                    g = torch.cuda.CUDAGraph()
                    n0 = L.launch_count()
                    with torch.cuda.graph(g, stream=cap):
                        kl_ptr, n_kl = self._chain(xin, self._bases[par], advance=True, par=par)
                    n_chain = L.launch_count() - n0
                    self.chain_graphs[par].append(g)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=cap):
                    self._exchange(kl_ptr, n_kl, par=par)
                self.exch_graphs.append(g)
            self.kernels_per_step = n_chain + 1
            self.graphs = self.chain_graphs[0]
            # the exchange kernel is tiny and latency-critical (peers wait for it): highest priority the device offers
            lo = getattr(torch.cuda.Stream, "priority_range", lambda: (-1, 0))()
            self.result_stream = torch.cuda.Stream(device=dev, priority=min(lo))
            self._chain_done = [torch.cuda.Event() for _ in range(nb)]
            self._exch_done = [None] * nb
            self._in_ready = [torch.cuda.Event() for _ in range(nb)]
            self.chain_streams = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(nb)] if self.inflight > 1 else None
            # replay r draws noise block first_replay + r: with k counters, counter p starts k blocks back and moves by k
            for p_ in range(nb):
                self.base2[p_] = (self.first_replay + p_ - nb) * _STRIDE
        for xin in (() if self.overlap else self.inputs):
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count()
            with torch.cuda.graph(g, stream=cap):
                self._step(xin, self.base, advance=True)
            self.kernels_per_step = L.launch_count() - n0          # engine kernels captured in one step
            self.graphs.append(g)
        self.graph = self.graphs[0]
        self.base.fill_((self.first_replay - 1) * _STRIDE)

    def __call__(self, x: Optional[torch.Tensor] = None, labels: Optional[torch.Tensor] = None, slot: int = 0):
        if labels is not None and self.labels is None:
            raise L.EngineError("MCForward was built without with_labels=True")
        if self.overlap:
            cur = torch.cuda.current_stream(self.dev)
            par = self.replays % self.nbuf
            run = cur
            if self.inflight > 1:                        # even / odd steps on their own streams, behind the caller's work so far
                run = self.chain_streams[par]
                self._in_ready[par].record(cur)
                run.wait_event(self._in_ready[par])
            if self._exch_done[par] is not None:          # buffers `par` were last read by the exchange of two steps ago
                run.wait_event(self._exch_done[par])
            with torch.cuda.stream(run):
                if labels is not None:
                    self.labels_all[par].copy_(labels, non_blocking=True)
                if x is not None:
                    self.inputs[slot].copy_(x, non_blocking=True)
                self.chain_graphs[par][slot].replay()
                self._chain_done[par].record(run)
            rs = self.result_stream
            rs.wait_event(self._chain_done[par])
            with torch.cuda.stream(rs):
                self.exch_graphs[par].replay()
                ev = self._exch_done[par] = self._exch_done[par] or torch.cuda.Event()
                ev.record(rs)
            self._last = par
            self.replays += 1
            return self.out
        if labels is not None:
            self.labels.copy_(labels, non_blocking=True)
        if self.graph is not None:
            if x is not None:
                self.inputs[slot].copy_(x, non_blocking=True)
            self.graphs[slot].replay()
            self.replays += 1
            return self.out
        return self._step(self.inputs[slot] if x is None else x.to(self.dev))

    def wait(self):
        """Make the current stream wait for the last step's results (a no-op unless built with ``overlap=True``)."""
        if self.overlap and self.replays and self._exch_done[self._last] is not None:
            # exchanges run in step order on one stream and each follows its chain: the last one covers everything before
            torch.cuda.current_stream(self.dev).wait_event(self._exch_done[self._last])
        return self.out

    def input_consumed(self):
        """Event after which the input of the LAST step may be rewritten (its layer chain has read it); None = stream order
        of the current stream already says so."""
        return self._chain_done[self._last] if (self.overlap and self.replays) else None


def _generic_mc_forward(forward_fn: Callable, x: torch.Tensor, num_ens: int, group=None, want_uncertainty: bool = False):
    """Backend-agnostic restatement (any device, any torch.distributed backend): the exact (max, sum-exp) partials of
    logmeanexp per rank and ONE all-gather; returns (log_outputs, kl[, (pred, epistemic, aleatoric, entropy)])."""
    dist, world, rank = _dist_info(group)
    ids = local_samples(num_ens, world, rank)
    parts, shape, dev = None, None, x.device
    for j in ids:
        logits, kl = forward_fn(x, j)
        logits = logits.float()
        shape, dev = logits.shape, logits.device
        lsm = torch.log_softmax(logits, dim=1)
        p = lsm.exp()
        klv = torch.as_tensor(kl, dtype=torch.float32, device=dev).reshape(1)
        if parts is None:
            parts = [lsm.clone(), torch.ones_like(lsm), p.clone(), p * p, logits.clone(), klv.clone()]
        else:
            m = torch.maximum(parts[0], lsm)
            parts[1] = parts[1] * (parts[0] - m).exp() + (lsm - m).exp()
            parts[0] = m
            parts[2] += p; parts[3] += p * p; parts[4] += logits; parts[5] += klv
    if world > 1:
        meta = [tuple(shape) if shape is not None else None]
        metas = [None] * world
        dist.all_gather_object(metas, meta[0], group=group)
        shape = next(s for s in metas if s is not None)
    n = shape[0] * shape[1]
    if parts is None:                                 # a rank with no sample (num_ens < world) still joins the collective
        z = torch.zeros(shape, dtype=torch.float32, device=dev)
        parts = [torch.full(shape, -float("inf"), device=dev), z, z.clone(), z.clone(), z.clone(), torch.zeros(1, device=dev)]
    vec = torch.cat([t.reshape(-1) for t in parts])
    if world > 1:
        allv = [torch.empty_like(vec) for _ in range(world)]
        dist.all_gather(allv, vec, group=group)       # the ONE collective of the forward path
    else:
        allv = [vec]
    S = float(num_ens)
    ms = torch.stack([v[:n] for v in allv])
    as_ = torch.stack([v[n:2 * n] for v in allv])
    M = ms.max(0).values
    tot = (as_ * torch.where(as_ > 0, (ms - M).exp(), torch.zeros_like(ms))).sum(0)
    log_outputs = (M + torch.log(tot / S)).view(shape)         # == logmeanexp_j log_softmax_j (utils.py:14-22), finite
    kl = sum(v[5 * n] for v in allv) / S                      # main_bayesian.py:51
    if not want_uncertainty:
        return log_outputs, kl
    p_bar = (sum(v[2 * n:3 * n] for v in allv) / S).view(shape)
    p2 = (sum(v[3 * n:4 * n] for v in allv) / S).view(shape)
    pred = (sum(v[4 * n:5 * n] for v in allv) / S).view(shape)
    epistemic = p2 - p_bar * p_bar                    # diag((p-pbar)^T (p-pbar))/T  (uncertainty_estimation.py:89-91)
    aleatoric = p_bar - p2                            # diag(diag(pbar) - p^T p / T)  (:94-95)
    entropy = -(p_bar * torch.log(p_bar.clamp_min(1e-38))).sum(1)      # H[pbar]; no reference (SURVEY D3)
    return log_outputs, kl, (pred, epistemic, aleatoric, entropy)


def mc_forward(net_or_fn, x: torch.Tensor, num_ens: int, group=None, want_uncertainty: bool = False,
               normalized: bool = False, labels: Optional[torch.Tensor] = None, train_size: float = 1.0,
               beta: float = 0.0, seed: Optional[int] = None):
    """(log_outputs [B,C], kl) like main_bayesian.py:46-53 -- plus (pred, epistemic, aleatoric, entropy) like
    uncertainty_estimation.py:70-96 with ``want_uncertainty`` and the ELBO head [loss, nll, acc, beta*kl] when
    ``labels`` are given.  ``net_or_fn``: a net built on the engine with CUDA input -> the device path (MCForward,
    cached on the net per shape/options); any ``forward_fn(x, sample_id) -> (logits, kl)`` -> the generic path."""
    from .modules import ModuleWrapper
    if isinstance(net_or_fn, ModuleWrapper) and x.is_cuda:
        net = net_or_fn
        key = (tuple(x.shape), int(num_ens), bool(want_uncertainty), bool(normalized), labels is not None,
               float(train_size), float(beta), seed, id(group))
        cache = net.__dict__.setdefault("_mc_engines", {})
        eng = cache.get(key)
        if eng is None:
            eng = cache[key] = MCForward(net, x, num_ens, group, want_uncertainty, normalized, labels is not None,
                                         train_size, beta, seed)
        out = eng(x, labels)
        res = [out["log_outputs"], out["kl"]]
        if want_uncertainty:
            res.append((out["pred"], out["epistemic"], out["aleatoric"], out["entropy"]))
        if labels is not None:
            res.append(out["head"])
        return tuple(res)
    return _generic_mc_forward(net_or_fn, x, num_ens, group, want_uncertainty)


def engine_forward_fn(net) -> Callable:
    """forward_fn for a net built on the engine: draws Monte-Carlo sample j (and leaves the training stream untouched)."""
    def fn(x, j):
        with Fn.mc_sample(j), torch.no_grad():
            return net(x)
    return fn


class MCTrainStep(MCForward):
    """One SHARDED training step with main_bayesian.train_model's semantics (main_bayesian.py:38-58): every rank runs
    its share of the ``num_ens`` weight samples WITH autograd (layer forward kernels + the engine's backward kernels),
    the exchange kernel combines them into log_outputs / kl / the ELBO (metrics.py:12-14) on every rank, each rank
    back-propagates d loss / d logits_j of ITS samples -- which needs only the combined log_outputs:
        d loss / d logits_j[b,:] = -(train_size / B) * softmax_j[b,y_b] / (S * p_bar[b,y_b]) * (onehot(y_b) - softmax_j[b,:])
    -- plus beta/S of its samples' KL terms, and ONE all-reduce sums the parameter gradients (SURVEY.md 8e "Backward
    sharding").  The caller owns the optimizer: ``out = step(x, labels, beta); optimizer.step()``.

    Noise: sample j of step t draws Philox streams 2^63 + (j << 40) + t * 2^20 + layer, so R ranks == 1 rank."""

    def __init__(self, net, example_x, num_ens, train_size, group=None, seed=None):
        super().__init__(net, example_x, num_ens, group=group, with_labels=True, train_size=train_size, seed=seed,
                         graph=False, fold=False)
        self.params = [p for p in net.parameters() if p.requires_grad]
        self.steps = 0

    def __call__(self, x, labels, beta: float = 0.0):
        from .graph import _STRIDE
        self.beta = float(beta)
        self.labels.copy_(labels, non_blocking=True)
        for p in self.params:
            p.grad = None
        logits, kls = [], []
        for k, j in enumerate(self.ids):
            with Fn.mc_sample(j, self.seed, offset=self.steps * _STRIDE):
                lg, kl = self.net(x)                                   # autograd on: per-layer kernels (no fused chain)
            logits.append(lg)
            kls.append(kl)
            self.logits[k].copy_(lg.detach().reshape(self.B, self.C))
        kl_ptr, n_kl = None, 0
        if self.ids:
            self.kl_one.copy_(kls[0].detach())
            kl_ptr, n_kl = Fn._ptr(self.kl_one), 1
        self._exchange(kl_ptr, n_kl)
        o = self.out
        if self.ids:
            S = float(self.num_ens)
            idx = self.labels.view(-1, 1)
            p_bar_y = o["log_outputs"].gather(1, idx).exp()                 # p_bar[b, y_b]
            grads = []
            for lg in logits:
                sm = torch.softmax(lg.detach().float(), dim=1)
                w = sm.gather(1, idx) / (S * p_bar_y)
                onehot = torch.zeros_like(sm).scatter_(1, idx, 1.0)
                grads.append((-(self.train_size / self.B)) * w * (onehot - sm))
            kl_g = [torch.full_like(k_, self.beta / S) for k_ in kls if torch.is_tensor(k_) and k_.requires_grad]
            kl_t = [k_ for k_ in kls if torch.is_tensor(k_) and k_.requires_grad]
            torch.autograd.backward(logits + kl_t, grads + kl_g)
        if self.world > 1:                                                  # ONE collective: the summed parameter gradients
            for p in self.params:
                if p.grad is None:
                    p.grad = torch.zeros_like(p)
            flat = torch.cat([p.grad.reshape(-1) for p in self.params])
            self.dist.all_reduce(flat, group=self.group)
            off = 0
            for p in self.params:
                n = p.numel()
                p.grad.copy_(flat[off:off + n].view_as(p))
                off += n
        self.steps += 1
        return o
