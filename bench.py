#!/usr/bin/env python
"""bench.py -- BBBAlexNet forward + KL images/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic batch: BBBAlexNet
(CIFAR-10 shape, 3x32x32, batch 512), ONE Monte-Carlo weight sample per GPU,
all six Bayesian layers + the model file's own activation/pool/flatten modules +
the summed KL scalar.  With N GPUs the num_ens MC loop (main_bayesian.py:46-49)
is the shard axis: rank r runs sample r of the SAME batch and one NCCL all-reduce
combines sum_j softmax_j and the KL (SURVEY.md 8e) -> weak scaling, value =
B * N * K / t.  The value times exactly K steps, in one window after the W warm-up
steps (before those, every captured graph is replayed once, untimed: a graph's first
replay uploads it).  Inputs, parameters and noise seeds are fixed, so with the same arguments
--dump-outputs writes the same step outputs (log_outputs, kl, ...) on every run.

Printed JSON (rank 0, one line): the driver contract + `roofline`, `cpu_baseline`,
`e2e`, `clocks`, `gpu_launches`, `per_layer`.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

PRIORS = {"prior_mu": 0, "prior_sigma": 0.1, "posterior_mu_initial": (0, 0.1),
          "posterior_rho_initial": (-5, 0.1)}          # config_bayesian.py:4-9
METRIC = "BBBAlexNet fwd+KL images/sec"
L2_FLUSH_BYTES = 256 << 20


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# --------------------------------------------------------------------------- #
# clocks
# --------------------------------------------------------------------------- #
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML polled every ~2 ms from a thread
    (the timed region lasts tens of milliseconds, too short for `nvidia-smi -lms`)."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index, self.sm, self.mask, self.max_mhz, self.err = index, [], 0, None, None
        self._stop = threading.Event()
        self.thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    except Exception as e:          # keep sampling what we can
                        self.err = str(e)
                    time.sleep(0.002)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception as e:
            self.err = str(e)

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=1)
        reasons = sorted(n for n, bit in self.REASONS.items() if self.mask & bit)
        out = {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": reasons, "samples": len(self.sm)}
        if self.err:
            out["note"] = self.err
        return out


# --------------------------------------------------------------------------- #
# workload
# --------------------------------------------------------------------------- #
def layer_table(batch, classes=10):
    """Algorithmic FLOPs / bytes per Bayesian layer (SURVEY.md 8d, Appendix B)."""
    spec = [("conv1", 3, 32, 64, 11, 4, 5), ("conv2", 64, 4, 192, 5, 1, 2), ("conv3", 192, 2, 384, 3, 1, 1),
            ("conv4", 384, 2, 256, 3, 1, 1), ("conv5", 256, 2, 128, 3, 1, 1), ("classifier", 128, 1, classes, 1, 1, 0)]
    rows = []
    for name, cin, hin, cout, k, s, p in spec:
        ho = (hin + 2 * p - k) // s + 1
        K = cin * k * k
        rows.append({"name": name, "M": batch * ho * ho, "N": cout, "K": K,
                     "flops_mean": 2.0 * batch * ho * ho * cout * K,
                     "x_elems": batch * cin * hin * hin, "y_elems": batch * cout * ho * ho,
                     "params": cout * K + cout})
    return rows


def algorithmic(row, variant, act_bytes=4):
    """SURVEY 8d: F = 2*M*N*K*v; Q = |x|*s + 2*(|W|+|b|)*4 + |y|*s + 4 with s = the run's activation width
    (4 for the fp32 path, 2 for the bf16 chain -- Appendix C's C3 accounting)."""
    v = 2.0 if variant == "lrt" else 1.0
    flops = row["flops_mean"] * v
    byts = row["x_elems"] * act_bytes + 2 * row["params"] * 4 + row["y_elems"] * act_bytes + 4
    return flops, byts


def build_net(variant, classes, device, math, net_type="alexnet", inputs=3):
    import pytorch_bayesiancnn_b200 as bbb  # noqa: F401
    from pytorch_bayesiancnn_b200.models import get_model
    torch.manual_seed(123)
    net = get_model(net_type, inputs, classes, PRIORS, variant, "softplus")
    with torch.no_grad():                       # identical params on every rank, drawn on the CPU generator
        g = torch.Generator().manual_seed(123)
        for name, p in net.named_parameters():
            mean = -5.0 if name.endswith("rho") else 0.0
            p.copy_(torch.empty(p.shape).normal_(mean, 0.1, generator=g))
    net = net.to(device).train()
    net.set_flag("math", math)
    return net


# --------------------------------------------------------------------------- #
# our arm
# --------------------------------------------------------------------------- #
def pin_to_gpu_numa_node(local):
    """Best effort: run this process (and so first-touch its pinned host buffers) on the CPUs of the GPU's NUMA node, so the
    e2e H2D path does not cross the socket interconnect (round 1 saw 2.96 vs 1.39 M img/s for identical code)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and vis.split(",")[local].isdigit() else local
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": None}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:
        return {"numa_node": None, "note": str(e)[:80]}


CONFIGS = {   # BASELINE.json configs restated (SURVEY.md 8d); "headline" = configs[2]'s model/batch, one MC sample per GPU per step
    "headline": dict(net="alexnet", classes=10, inputs=3, batch=512, variant="lrt", samples=None, uncertainty=False),
    "C2": dict(net="lenet", classes=10, inputs=3, batch=256, variant="bbb", samples=1, uncertainty=False),
    "C3": dict(net="alexnet", classes=10, inputs=3, batch=512, variant="lrt", samples=10, uncertainty=False),
    "C4": dict(net="alexnet", classes=100, inputs=3, batch=1024, variant="lrt", samples=25, uncertainty=False),
    "C5": dict(net="3conv3fc", classes=10, inputs=1, batch=2048, variant="lrt", samples=100, uncertainty=True),
}


def run_ours(args):
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import mc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    numa = pin_to_gpu_numa_node(local)
    # The GPU arms do no CPU math: keep the OpenMP pool at one thread, as torch.distributed.run does for N > 1.  Measured
    # (tools/e2e_probe.py, profiles/r2_e2e_probe.txt): with 64 idle-spinning OpenMP workers the pinned H2D path dropped from
    # 53.5 to 17-26 GB/s and the N=1 end-to-end figure was half of one rank's at N=2.  The CPU baseline leg sets its own count.
    torch.set_num_threads(1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        # NCCL is only the rendezvous here (seed / IPC-handle exchange, barriers, the max-over-ranks of the timings): the
        # data path of a step is the engine's own NVLink exchange kernel.  Its banner goes to stdout: keep that clean.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    cfg = dict(CONFIGS[args.config])
    if args.config == "headline":
        cfg.update(batch=args.batch, classes=args.classes, variant=args.variant)
    B, C = cfg["batch"], cfg["classes"]
    S_total = cfg["samples"] if cfg["samples"] is not None else world       # headline: one MC sample per GPU per step
    args.batch, args.classes, args.variant = B, C, cfg["variant"]
    pk = peaks()

    net = build_net(cfg["variant"], C, dev, args.math, cfg["net"], cfg["inputs"])
    gx = torch.Generator().manual_seed(0)
    in_shape = (B, cfg["inputs"], 32, 32)
    in_bytes = B * cfg["inputs"] * 32 * 32 * 4
    n_inputs = 4                                 # pinned host batches (e2e arm)
    n_dev_inputs = max(2, -(-(160 << 20) // in_bytes))   # device-resident arm rotates through > 126 MB (L2) of inputs
    x_host = [torch.randn(*in_shape, generator=gx).pin_memory() for _ in range(n_inputs)]
    gd = torch.Generator(device=dev).manual_seed(123)    # seeded: the same arguments give the same inputs on every run
    x_dev = [torch.randn(*in_shape, device=dev, generator=gd) for _ in range(n_dev_inputs)]
    # The step = the package's public MC step (mc.MCForward): this rank's samples through the engine (fused tcgen05 chain),
    # then ONE kernel that combines them, exchanges the partials with the other ranks over NVLink and finishes
    # logmeanexp / KL (/ uncertainty) on the device -- all in one captured CUDA graph per resident input batch.
    # overlap=True: the exchange kernel of step t runs on its own stream beside the first kernels of step t+1 (the windows
    # below end with eng.wait(), so every timed step's exchange is inside the timed region)
    ovl = os.environ.get("BBB_B200_MC_OVERLAP", "1") == "1"
    # inflight=k: consecutive steps are independent (different batches, same weights), so steps t..t+k-1 run on k streams with
    # their own workspaces / Philox counters; every step still does all of its work inside the timed region and the results
    # are bit-identical to the serial engine (tests/test_gpu_mc.py).  The one-step-at-a-time figure is under serial_step.
    infl = int(os.environ.get("BBB_B200_MC_INFLIGHT", "4")) if ovl else 1
    eng = mc.MCForward(net, x_dev[0], S_total, want_uncertainty=cfg["uncertainty"], seed=2024, static_inputs=x_dev, overlap=ovl, inflight=infl)
    staging = [torch.zeros_like(x_dev[0]) for _ in range(2)]
    eng_e2e = mc.MCForward(net, x_dev[0], S_total, want_uncertainty=cfg["uncertainty"], seed=2024, static_inputs=staging,
                           first_replay=1 << 18, overlap=ovl, inflight=infl)
    S_local = len(eng.ids)
    main = torch.cuda.current_stream(dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def window(fn, nsteps):
        """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream; max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record(main)
        fn(nsteps)
        e1.record(main)
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def prime(engine, slots):
        """Replay every graph the engine captured once, untimed: a graph's first replay uploads it to the device.  Steps
        cycle through the (in-flight buffer, input slot) pairs with period lcm(nbuf, slots)."""
        for i in range(math.lcm(engine.nbuf, slots)):
            engine(slot=i % slots)
        engine.wait()
        sync_all()

    # ---- device-resident throughput: K steps back to back, inputs rotate through > L2 of resident batches ----
    counter = [0]

    def resident(nsteps):
        for _ in range(nsteps):
            eng(slot=counter[0] % n_dev_inputs)
            counter[0] += 1
        eng.wait()

    prime(eng, n_dev_inputs)
    window(resident, args.warmup)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    wall0 = time.perf_counter()
    total_ms = window(resident, args.steps)
    wall = time.perf_counter() - wall0
    last_step = {k: v.cpu() for k, v in eng.out.items()} if args.dump_outputs and rank == 0 else None
    images_per_step = B * S_total                # image-samples of the whole job per step (SURVEY 8d: B*S/t)
    value = images_per_step * args.steps / (total_ms * 1e-3)
    launches = eng.kernels_per_step * args.steps

    # ---- end to end through the public API: pinned host input -> H2D -> MC step -> D2H of the result ----
    out_host = torch.empty(B, C, dtype=torch.float32).pin_memory()
    kl_host = torch.empty(1, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def e2e_steps(nsteps):
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            staging[0].copy_(x_host[0], non_blocking=True)
            ready[0].record(copy_stream)
        for i in range(nsteps):
            s = i & 1
            if i + 1 < nsteps:                  # prefetch the next batch while this one computes
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(consumed[s ^ 1])
                    staging[s ^ 1].copy_(x_host[(i + 1) % n_inputs], non_blocking=True)
                    ready[s ^ 1].record(copy_stream)
            main.wait_event(ready[s])
            out = eng_e2e(slot=s)
            if eng_e2e.input_consumed() is not None:
                consumed[s] = eng_e2e.input_consumed()                 # the step's chain runs on the engine's own stream
            else:
                consumed[s].record(main)
            with torch.cuda.stream(eng_e2e.result_stream or main):     # the stream the step's results are complete on
                out_host.copy_(out["log_outputs"], non_blocking=True)
                kl_host.copy_(out["kl"].reshape(1), non_blocking=True)
        if eng_e2e.result_stream is not None:
            main.wait_stream(eng_e2e.result_stream)

    prime(eng_e2e, len(staging))
    window(e2e_steps, max(3, args.warmup))
    e2e_ms = window(e2e_steps, args.steps)
    e2e_value = images_per_step * args.steps / (e2e_ms * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    timeouts = eng.timeouts() + eng_e2e.timeouts()

    # ---- the same step strictly one at a time (no exchange overlap, one step in flight): the step LATENCY ----
    serial = None
    if ovl:
        eng_s = mc.MCForward(net, x_dev[0], S_total, want_uncertainty=cfg["uncertainty"], seed=2024, static_inputs=x_dev)

        def resident_serial(nsteps):
            for _ in range(nsteps):
                eng_s(slot=counter[0] % n_dev_inputs)
                counter[0] += 1

        prime(eng_s, n_dev_inputs)
        window(resident_serial, args.warmup)
        s_ms = window(resident_serial, args.steps)
        serial = {"ms_per_step": s_ms / args.steps, "value": images_per_step * args.steps / (s_ms * 1e-3), "unit": "images/s",
                  "note": "one step in flight, exchange kernel inside the step's graph (the step latency); the headline value "
                          f"keeps {infl} independent steps in flight"}
        timeouts += eng_s.timeouts()
        eng_s.close()

    # ---- per-layer kernel timing + roofline of the dominant kernel (rank 0, AlexNet only) ----
    per_layer, roof = [], None
    if rank == 0 and cfg["net"] == "alexnet":
        flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
        per_layer, roof = layer_rooflines(net, x_dev[0], args, pk, flush)
        del flush

    in_chain = None
    if rank == 0 and world == 1 and cfg["net"] == "alexnet" and roof is not None:
        try:
            in_chain = in_chain_kernels(net, x_dev[0], dev)
            gem = [r for r in in_chain if r["kernel"].startswith(("conv_s4 ", "tap_gemm", "gemm_tc"))]
            rows_l = layer_table(B, C)
            act_b = 4 if args.math == "fp32" else 2
            for r, row in zip(gem, rows_l):                       # GEMM kernels appear in layer order
                fl, by = algorithmic(row, cfg["variant"], act_b)
                t_roof = max(fl / (pk["tf_burst"] * 1e12), by / (pk["hbm_gbs"] * 1e9))
                r.update(layer=row["name"], tflops=fl / (r["work_us"] * 1e-6) / 1e12, frac_of_roofline=t_roof / (r["work_us"] * 1e-6))
            top = max(gem, key=lambda r: r["work_us"])
            roof["in_chain"] = {"kernel": top["layer"] + " GEMM kernel", "work_us": top["work_us"], "tflops": top["tflops"],
                                "frac": top["frac_of_roofline"],
                                "note": "same kernel inside the captured step: last-CTA exit minus dependencies-satisfied, "
                                        "device %globaltimer, median of 17 replays (the primary figure above is the kernel "
                                        "replayed ALONE after an L2 flush, with CUDA events: cold weights, launch included)"}
        except Exception as e:                                    # a diagnostic, never the reason a bench run fails
            in_chain = [{"note": f"failed: {e}"[:200]}]

    if roof is not None:
        # the whole step against the sum of the per-layer rooflines (SURVEY 8d): what fraction of the step time the
        # algorithmic FLOPs / bytes of its six layers would need at the measured peaks
        step_us = total_ms / args.steps * 1e3
        fl = sum(algorithmic(r, args.variant, 2 if args.math != "fp32" else 4)[0] for r in layer_table(B * S_local, C))
        roof["whole_step"] = {"step_us": step_us, "tflops": fl / (step_us * 1e-6) / 1e12,
                              "frac_of_sum_of_layer_rooflines": roof["net_t_roof_us"] * S_local / step_us if "net_t_roof_us" in roof else None,
                              "note": f"{infl} step(s) in flight; net_t_roof_us is per MC sample of the batch"}

    mc_batched = None
    if rank == 0 and world == 1 and args.config == "headline" and cfg["variant"] == "lrt" and args.mc_batch > 1:
        # configs[2] literally: S = 10 MC samples of the batch.  For LRT the samples differ only in the per-activation
        # noise, so S samples == one launch over S*B rows (what uncertainty_estimation.py:38-41 does); KL computed once.
        S = args.mc_batch
        xb = x_dev[0].repeat(S, 1, 1, 1)
        gb = bbb.GraphedForward(net, xb, first_stream=1 << 40)
        for _ in range(3):
            gb()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(9):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                gb()
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1) / 10)
        ms = statistics.median(ts)
        fl = sum(algorithmic(r, "lrt", 2)[0] for r in layer_table(S * B, C))
        t_roof = sum(max(algorithmic(r, "lrt", 2)[0] / (pk["tf_sustained"] * 1e12), algorithmic(r, "lrt", 2)[1] / (pk["hbm_gbs"] * 1e9))
                     for r in layer_table(S * B, C))
        mc_batched = {"mc_samples": S, "rows_per_launch": S * B, "ms_per_launch": ms,
                      "value": S * B / (ms * 1e-3), "unit": "sample-images/s", "tflops": fl / (ms * 1e-3) / 1e12,
                      "roofline_frac_of_sustained_peak": t_roof / (ms * 1e-3),
                      "note": "configs[2] as written: 10 MC samples of the 512 images in ONE launch (LRT: samples fold into the batch)"}
        del gb, xb

    cpu = incumbent = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference(args, seconds=args.cpu_seconds)
        if cfg["net"] == "alexnet":
            incumbent = gpu_eager_incumbent(args, dev)

    # ---- sharded TRAINING step (row f1): fwd + bwd + ONE gradient all-reduce + Adam, main_bayesian.py:38-58 semantics ----
    train = None
    if args.train_steps > 0 and cfg["net"] == "alexnet":
        ts = mc.MCTrainStep(net, x_dev[0], S_total, train_size=50000.0, seed=2024)
        labels = torch.randint(0, C, (B,), device=dev)
        opt = torch.optim.Adam(net.parameters(), lr=1e-5)

        def tsteps(n):
            for i in range(n):
                ts(x_dev[i % n_dev_inputs], labels, 0.1)
                opt.step()

        window(tsteps, 2)
        tw = [window(tsteps, args.train_steps) for _ in range(3)]
        tms = statistics.median(tw) / args.train_steps
        train = {"value": images_per_step / (tms * 1e-3), "unit": "images/s", "ms_per_step": tms,
                 "what": "forward (tcgen05 layer kernels, autograd on: no fused chain) + backward (wgrad / dgrad as role-swapped "
                         "tcgen05 layer calls, eps regenerated from Philox; BBB_B200_BWD=simt selects the fp32 CUDA-core "
                         "kernels) + MC exchange/ELBO kernel + one gradient all-reduce + Adam; eager launches (no graph)"}
        ts.close()

    if rank == 0:
        dt = {"fp32": "f32", "tf32": "tf32 operands, f32 accumulate"}.get(args.math, "bf16 operands, f32 accumulate")
        out = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak" if cfg["samples"] is None else "strong", "vs_baseline": None, "dtype": dt,
            "data": "synthetic (randn inputs, random-init params N(0,0.1)/rho N(-5,0.1))",
            "config": {"workload": f"BBB{cfg['net']}-{C} {cfg['inputs']}x32x32, batch {B}, {cfg['variant']} layers, softplus, "
                                   f"{S_total} MC sample(s) per step sharded over {world} GPU(s) ({S_local} on rank 0); step = "
                                   f"forward+KL of the local samples + the MC combine/exchange kernel",
                       "named_config": args.config if args.config != "headline" else
                                       ("BASELINE.json configs[2] model/batch (BBBAlexNet CIFAR-10 batch 512 bf16, BBB_LRT): a step is ONE MC "
                                        "sample of the batch per GPU and the metric counts image-samples (B*S/t, SURVEY 8d); the literal "
                                        "single-launch S=10 figure is under mc_batched"),
                       "batch": B, "variant": cfg["variant"], "math": args.math, "mc_samples_total": S_total,
                       "parallelism": f"mc{world}", "steps_in_flight": infl, "exchange_overlapped": ovl,
                       "l2": f"no flush: inputs rotate through {n_dev_inputs} resident batches = {n_dev_inputs * in_bytes >> 20} MB > 126 MB L2",
                       "launch": ("two CUDA graph replays per step (layer chain: noise advance, per-layer prep + GEMM kernels; then the MC "
                                  "exchange kernel over NVLink peer memory on its own stream, beside the next step's chain)" if ovl else
                                  "one CUDA graph replay per step (noise advance, per-layer prep + GEMM kernels, MC exchange kernel over "
                                  "NVLink peer memory)") + "; one captured graph per resident input batch, read in place",
                       "timing": f"{args.steps} steps in one window bracketed by barrier+synchronize, CUDA events, max over ranks"},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": in_bytes,
                    "d2h_bytes_per_step": B * C * 4 + 4, "ms_per_step": e2e_ms / args.steps, "host_numa": numa},
            "gpu_launches": int(launches),
            "serial_step": serial,
            "clocks": clocks,
            "roofline": roof,
            "per_layer": per_layer,
            "in_chain_kernels": in_chain,
            "cpu_baseline": cpu,
            "gpu_eager_incumbent": incumbent,
            "mc_batched": mc_batched,
            "train": train,
            "exchange_timeouts": timeouts,
            "wall_s_timed_loop": wall,
        }
        print(json.dumps(out), flush=True)
        if last_step is not None:
            dump_outputs(last_step, args.dump_outputs)
    sync_all()
    eng.close(); eng_e2e.close()
    if dist is not None:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(out, path):
    """Write each output of the step as <path>/<name>.npy (float32).  Above DUMP_BYTES in all, every [B, ...] output keeps
    the same fixed, seeded sample of batch rows, so that two builds run with the same arguments compare row for row."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = sum(v.numel() * 4 for v in out.values())
    rows = None
    if total > DUMP_BYTES:
        B = next(v.shape[0] for v in out.values() if v.dim() > 0)
        keep = max(1, B * DUMP_BYTES // total)
        rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    for name, v in out.items():
        if rows is not None and v.dim() > 0:
            v = v[rows]
        np.save(os.path.join(path, f"{name}.npy"), v.float().numpy())


def in_chain_kernels(net, x, dev, reps=20):
    """Per-kernel device timestamps INSIDE the captured step (rank 0, single GPU): every engine kernel stamps
    %globaltimer at first-CTA entry, at the moment its launch dependencies are satisfied (griddepcontrol.wait passed:
    kernels launched with programmatic serialization enter early) and at last-CTA exit.  `work_us` = exit - deps-ok is the
    part of the kernel on the step's critical path; medians over `reps` replays of a dedicated capture (not the timed one)."""
    import ctypes as C
    from pytorch_bayesiancnn_b200 import mc, _lib as L
    lib = C.CDLL(L.LIB_PATH)
    lib.bbb_debug_set_timeline.argtypes = [C.c_void_p, C.c_int]
    lib.bbb_debug_timeline_name.restype = C.c_char_p
    lib.bbb_debug_timeline_name.argtypes = [C.c_int]
    CAP = 128
    slots = torch.zeros(CAP, 4, dtype=torch.int64, device=dev)
    lib.bbb_debug_set_timeline(C.c_void_p(slots.data_ptr()), CAP)
    try:
        eng = mc.MCForward(net, x, 1, seed=7, static_inputs=[x.clone()])
        n = lib.bbb_debug_timeline_count()
        names = [lib.bbb_debug_timeline_name(k).decode() for k in range(n)]
    finally:
        lib.bbb_debug_set_timeline(None, 0)
    m = n // 3                                         # two eager warm-up steps + the captured one launch the same sequence
    first = n - m
    init = torch.tensor([[2 ** 62, 0, 2 ** 62, 0]] * CAP, dtype=torch.int64, device=dev)
    rows = {k: [] for k in range(first, n)}
    for _ in range(reps):
        slots.copy_(init)
        eng()
        torch.cuda.synchronize(dev)
        t = slots[:n].cpu()
        t0 = int(t[first:n, 0].min())
        for k in range(first, n):
            ent, ext, dep = int(t[k, 0]), int(t[k, 1]), int(t[k, 2])
            dep = min(dep, ext) if dep < 2 ** 61 else ent
            rows[k].append(((ent - t0) / 1e3, (ext - t0) / 1e3, (dep - t0) / 1e3))
    out = []
    for k in range(first, n):
        med = [statistics.median(r[j] for r in rows[k][3:]) for j in range(3)]
        out.append({"kernel": names[k], "start_us": round(med[0], 2), "end_us": round(med[1], 2),
                    "deps_ok_us": round(med[2], 2), "work_us": round(med[1] - med[2], 2)})
    return sorted(out, key=lambda r: r["start_us"])


def gpu_eager_incumbent(args, dev, reps=12):
    """SURVEY 8d's same-box incumbent: the reference's op sequence in stock PyTorch eager ON THE B200 (the oracle port's
    aten calls with CUDA tensors -- cuDNN conv (TF32 by default, SURVEY D9) + elementwise launches), including what the
    reference does every forward: eps drawn on the CPU generator and copied host->device (BBB/BBBConv.py:63,68)."""
    try:
        from oracle import bbb_oracle as O               # baseline leg only
        params = [{k: v.to(dev) for k, v in p.items()} for p in O.init_params("alexnet", args.classes, 3, PRIORS, seed=123)]
        x = torch.randn(args.batch, 3, 32, 32, generator=torch.Generator().manual_seed(0)).to(dev)
        shapes = O.eps_shapes("alexnet", args.classes, 3, args.variant, args.batch)

        def one():
            with torch.no_grad():
                eps = [torch.empty(s).normal_(0, 1).to(dev) for s in shapes]
                logits, kl = O.net_forward("alexnet", params, x, eps, args.variant, "softplus", 0.0, 0.1, args.classes)
                return float(kl)                          # main_bayesian.py:52 (kl.item(): the per-step host sync)
        for _ in range(3):
            one()
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter(); one(); torch.cuda.synchronize(dev)
            ts.append(time.perf_counter() - t0)
        med = statistics.median(ts)
        return {"value": args.batch / med, "unit": "images/s", "ms_per_step": med * 1e3, "min_ms": min(ts) * 1e3,
                "what": "oracle port's aten ops on the same B200, eager, incl. per-forward CPU eps draw + H2D copy and the "
                        "kl.item() sync (reference semantics); wall clock around synchronize"}
    except Exception as e:
        return {"value": None, "note": f"failed: {e}"[:200]}


def layer_rooflines(net, x, args, pk, flush, reps=20):
    """Time each Bayesian layer call alone: the call (prep + GEMM kernels; fused chain
    step when the net runs fused) is captured in its own CUDA graph so host launch
    overhead stays out, replayed with CUDA events on the launching stream, L2 flushed
    (untimed) before every replay."""
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import fused
    rows = layer_table(args.batch, args.classes)
    act_b = 4 if args.math == "fp32" else 2              # activation width of this run (SURVEY App. C: C3 uses s = 2)
    steps = fused.plan(list(net.children()), tuple(x.shape)) if getattr(net, "fuse", True) else None
    calls = []
    with torch.no_grad():
        if steps is not None:
            cur, cur_sq, pitch = x.contiguous().float(), None, 0
            for i, st in enumerate(steps):
                nxt = steps[i + 1].layer if i + 1 < len(steps) else None
                calls.append((lambda st=st, nxt=nxt, a=cur, b=cur_sq, c=pitch, ph=0: fused.run_step(st, nxt, a, b, c, phase=ph)))
                cur, cur_sq, pitch = fused.run_step(st, nxt, cur, cur_sq, pitch)
        else:
            h = x
            for name, m in net.named_children():
                if hasattr(m, "W_mu"):
                    calls.append((lambda m=m, a=h.contiguous(): m(a)))
                h = m(h)
    def timed(call):
        with torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                call(); call()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                call()
            times = []
            for _ in range(reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); gr.replay(); e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
        return statistics.median(times)

    from pytorch_bayesiancnn_b200 import _lib as L
    out = []
    for row, call in zip(rows, calls):
        ms = timed(call)
        # the two kernels of a fused-chain layer timed alone: parameter-only prep, and the GEMM kernel
        ms_prep = timed(lambda: call(ph=L.FUSED_PREP_ONLY)) if steps is not None else None
        ms_gemm = timed(lambda: call(ph=L.FUSED_SKIP_PREP)) if steps is not None else None
        fl, by = algorithmic(row, args.variant, act_b)
        t_tc = fl / (pk["tf_burst"] * 1e12)
        t_hbm = by / (pk["hbm_gbs"] * 1e9)
        bound = "tensor" if t_tc >= t_hbm else "hbm"
        out.append({"name": row["name"], "gemm": [row["M"], row["N"], row["K"]], "ms": ms,
                    "gflop": fl / 1e9, "mbytes": by / 1e6, "bound": bound,
                    "tflops": fl / (ms * 1e-3) / 1e12, "gbs": by / (ms * 1e-3) / 1e9,
                    "frac": max(t_tc, t_hbm) / (ms * 1e-3), "fused": steps is not None,
                    "ms_prep_kernel": ms_prep, "ms_gemm_kernel": ms_gemm})
    # dominant kernel = the longest single kernel: the GEMM kernel of a layer when the chain runs fused (the
    # layer's flops all execute there; its bytes are the layer's minus the fp32 mu/rho the prep kernel reads,
    # plus the bf16 operand tiles it reads instead), else the one fused fp32 layer kernel
    kt = (lambda r: r["ms_gemm_kernel"]) if steps is not None else (lambda r: r["ms"])
    top = max(out, key=kt)
    t_k = kt(top) * 1e-3
    if top["bound"] == "tensor":
        roof = {"kernel": top["name"] + (" GEMM kernel" if steps is not None else ""), "bound": "tensor",
                "achieved": top["gflop"] / 1e3 / t_k, "peak": pk["tf_burst"],
                "unit": "TFLOP/s", "frac": top["gflop"] / 1e3 / t_k / pk["tf_burst"], "traffic": None,
                "peak_source": pk["source"] + ", burst bf16 (kernel timed alone)",
                "kernel_us": t_k * 1e6, "layer_us_prep_plus_gemm": top["ms"] * 1e3, "layer_frac": top["frac"]}
    else:
        roof = {"kernel": top["name"] + (" GEMM kernel" if steps is not None else ""), "bound": "hbm",
                "achieved": top["mbytes"] / 1e3 / t_k, "peak": pk["hbm_gbs"],
                "unit": "GB/s", "frac": top["mbytes"] / 1e3 / t_k / pk["hbm_gbs"], "traffic": None,
                "peak_source": pk["source"],
                "kernel_us": t_k * 1e6, "layer_us_prep_plus_gemm": top["ms"] * 1e3, "layer_frac": top["frac"]}
    tp = os.path.join(ROOT, "profiles", "r2_ncu_full_traffic.json")      # dram__bytes_read+write of that kernel, one ncu --set full capture
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("variant") == args.variant and tj.get("batch") == args.batch and top["name"] in tj["layers"]:
            roof["traffic"] = tj["layers"][top["name"]]["dram_bytes"]
            roof["traffic_source"] = tj["source"]
    t_roof = sum(max(algorithmic(r, args.variant, act_b)[0] / (pk["tf_burst"] * 1e12),
                     algorithmic(r, args.variant, act_b)[1] / (pk["hbm_gbs"] * 1e9)) for r in rows)
    roof["net_t_roof_us"] = t_roof * 1e6
    roof["net_layer_kernels_us"] = sum(r["ms"] for r in out) * 1e3
    return out, roof


# --------------------------------------------------------------------------- #
# CPU reference arm (the oracle port of the reference's CPU path)
# --------------------------------------------------------------------------- #
def pick_threads(one):
    """The reference arm gets the thread count that serves it best on this host: oneDNN
    on 100+ threads is often slower than on a few dozen for convs this small."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, ncpu // 2, 64, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        one()
        t0 = time.perf_counter(); one(); one()
        dt = (time.perf_counter() - t0) / 2
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_step_fn(args):
    from oracle import bbb_oracle as O               # bench's cpu_baseline leg may use the oracle
    params = O.init_params(args.net_type, args.classes, args.inputs, PRIORS, seed=123)
    x = torch.randn(args.batch, args.inputs, 32, 32, generator=torch.Generator().manual_seed(0))
    shapes = O.eps_shapes(args.net_type, args.classes, args.inputs, args.variant, args.batch)

    def one():
        with torch.no_grad():
            # the reference draws eps on the CPU generator inside every forward (BBB/BBBConv.py:63)
            eps = [torch.empty(s).normal_(0, 1) for s in shapes]
            logits, kl = O.net_forward(args.net_type, params, x, eps, args.variant, "softplus", 0.0, 0.1, args.classes)
            return float(kl) + float(logits[0, 0])
    return one


def cpu_reference(args, seconds=10.0):
    """cpu_baseline leg: the reference arm in a fresh process (no CUDA context, no
    clock sampler competing for cores), bounded to ~`seconds` of CPU work."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "12", "--warmup", "3",
           "--variant", args.variant, "--batch", str(args.batch), "--classes", str(args.classes), "--config", args.config]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT).stdout.strip().splitlines()
        d = json.loads(out[-1])
        return d["cpu_baseline"]
    except Exception as e:                              # a baseline that cannot be taken is reported, not invented
        return {"value": None, "unit": "images/s", "cores": None, "kind": "port", "sample": f"failed: {e}"}


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    one = cpu_step_fn(args)
    steps = min(args.steps, 200)
    cores = pick_threads(one)
    for _ in range(args.warmup):
        one()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter(); one(); ts.append(time.perf_counter() - t0)
    dt = sum(ts)
    val = args.batch * steps / dt
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
           "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"BBB{args.net_type}-{args.classes} {args.inputs}x32x32, batch {args.batch}, "
                                  f"{args.variant} layers, softplus, 1 MC sample per step", "batch": args.batch,
                      "variant": args.variant, "named_config": args.config},
           "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port",
                            "sample": f"{steps} forwards of the full batch-{args.batch} workload (median "
                                      f"{statistics.median(ts) * 1e3:.1f} ms, min {min(ts) * 1e3:.1f} ms); torch-CPU "
                                      f"restatement of the reference incl. its per-forward CPU eps draws; threads "
                                      f"picked as the fastest of a probe",
                            "cpu_model": cpu_model()},
           "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", default="lrt", choices=["lrt", "bbb"])
    ap.add_argument("--math", default=os.environ.get("BBB_B200_MATH", "bf16"), choices=["fp32", "bf16", "tf32", "auto"])
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mc-batch", type=int, default=10, help="also report S MC samples folded into one launch (LRT; 0 = skip)")
    ap.add_argument("--train-steps", type=int, default=5, help="steps per window of the sharded training-step figure (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed step returned in its last step as DIR/<name>.npy (float32, at most 64 MB)")
    ap.add_argument("--config", default="headline", choices=list(CONFIGS),
                    help="headline (default: BBBAlexNet-10 B=512, one MC sample per GPU per step) or one of BASELINE.json's configs restated")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    cfg = CONFIGS[args.config]
    if args.config != "headline":
        args.batch, args.classes, args.variant = cfg["batch"], cfg["classes"], cfg["variant"]
    args.net_type, args.inputs = cfg["net"], cfg["inputs"]
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback); use --impl reference for the CPU arm")
        run_ours(args)


if __name__ == "__main__":
    main()
