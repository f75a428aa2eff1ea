#!/usr/bin/env python
"""bench.py -- forward+backward throughput of the dense hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps 300 --warmup 10                      # own arm, default workload
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --steps 5 --warmup 1                 # the reference's CPU path (oracle port)
    python bench.py --steps 50 --warmup 5 --dump-outputs DIR              # + the last timed step's outputs as DIR/*.npy

Workloads (BASELINE.json configs):
  linear  (default, config 2)  nn::Linear 4096->4096, bf16, batch 4096 per GPU, fwd + bwd (dX, dW, db)
                               N>1: weak scaling, gradient exchange fused into the dW GEMM over NVLink peer memory
  mlp     (config 4)           MLP 1024-4096-4096-10 + ReLU/Softmax, MSE, SGD step; global batch 8192 sharded
                               over the ranks (STRONG scaling), same exchange
  conv    (config 3)           nn::Conv2d 3->64 k3 s1, 224x224, batch 256 per GPU, fwd + bwd (dX, dW, db)
  convnet (config 5)           small ConvNet (Conv2d 3->32, Conv2d 32->64, Linear) on 32x32x3, global batch 4096 sharded
                               over the ranks, SGD step; every convolution kernel is a tcgen05 one

A step of the own arm = zero_grad -> build the define-by-run graph -> forward -> backward (-> exchange -> SGD where the
workload has them) through the package's public API (Var/VarDiff/nn/optim over the C++ graph and the C ABI).  The step
is recorded ONCE into a CUDA graph (Device.capture; the tape is the same every iteration) and replayed with one driver
call per step; `eager_ms_per_step` reports the same step enqueued kernel by kernel.  `value` times the steps with
inputs resident in HBM; `e2e` repeats them with the step's inputs copied from pinned host memory and the loss read back
inside the timed region.  The default workload is `value`; the other three GPU configs are measured in the same process
and reported under `other_configs` (config 4 is the strong-scaling curve north_star asks for).  N > 1 adds
`exchange_parity`: the fused NVLink exchange against an NCCL all-reduce of locally computed gradients.  One JSON line, rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "forward+backward GFLOP/s"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return {"hbm_gbs": float(p["hbm_gbs"]), "tflops_burst": float(p["bf16_tflops"]),
                "tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------- workloads
def workload_spec(name: str, world: int):
    if name == "linear":
        n = fin = fout = 4096
        flops = 3 * 2.0 * n * fin * fout                     # fwd + dX + dW (SURVEY.md 8-d; bias terms < 0.05 %)
        return {"name": "nn::Linear 4096->4096 bf16, batch 4096 per GPU, fwd+bwd (dX+dW+db)", "scaling": "weak",
                "flops_per_rank_step": flops, "samples_per_rank_step": n, "batch": n, "fin": fin, "fout": fout,
                "params": fin * fout + fout, "bound": "tensor", "arena": 1 << 30}
    if name == "mlp":
        gb = 8192
        assert gb % world == 0
        b = gb // world
        sizes = [1024, 4096, 4096, 10]
        fwd = sum(2.0 * b * i * o for i, o in zip(sizes[:-1], sizes[1:]))
        bwd = 2 * fwd - 2.0 * b * sizes[0] * sizes[1]        # dW for all layers, dX for layers 2,3
        return {"name": "MLP 1024-4096-4096-10 ReLU/Softmax MSE SGD step, global batch 8192", "scaling": "strong",
                "flops_per_rank_step": fwd + bwd, "samples_per_rank_step": b, "batch": b, "sizes": sizes,
                "params": sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:])), "bound": "tensor", "arena": 2 << 30}
    if name == "conv":
        n, cin, h, w, cout, k = 256, 3, 224, 224, 64, 3
        ho, wo = h - k + 1, w - k + 1
        fwd = 2.0 * n * cout * ho * wo * cin * k * k
        # algorithmic bytes (bf16, each tensor once): fwd reads x, writes y; bwd reads g (once, fused dX+dW), x, writes dx
        return {"name": "nn::Conv2d 3->64 k3 s1 p0, 224x224, batch 256 per GPU, fwd+bwd (dX+dW+db)",
                "scaling": "weak", "flops_per_rank_step": 3 * fwd, "samples_per_rank_step": n, "batch": n,
                "shape": (n, cin, h, w), "cout": cout, "k": k, "params": cout * cin * k * k + cout,
                "bytes_per_rank_step": 2.0 * (2 * n * cout * ho * wo + 3 * n * cin * h * w), "bound": "hbm",
                "arena": 12 << 30}
    if name == "convnet":
        gb = 4096
        assert gb % world == 0
        b = gb // world
        f1 = 2.0 * b * 32 * 1024 * 27
        f2 = 2.0 * b * 64 * 1024 * 288
        f3 = 2.0 * b * 65536 * 10
        # fwd + dW for every layer, dX for conv2 and the Linear (the network input is not differentiable)
        return {"name": "small ConvNet (Conv2d 3->32 p1, Conv2d 32->64 p1, Linear 65536->10) on 32x32x3, global batch 4096, SGD step",
                "scaling": "strong", "flops_per_rank_step": 2 * f1 + 3 * f2 + 3 * f3, "samples_per_rank_step": b, "batch": b,
                "params": 32 * 27 + 32 + 64 * 288 + 64 + 655360 + 10, "bound": "tensor", "arena": 24 << 30}
    raise SystemExit(f"unknown workload {name}")


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs.  Construct (nvmlInit) and start it
    BEFORE the ranks are aligned: NVML start-up takes milliseconds and differs from process to process."""

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period_s, [], set(), None
        self._halt = threading.Event()
        self._armed = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def arm(self):
        """start recording samples (the thread itself is already running)"""
        self._armed.set()

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._halt.is_set():
            if self._armed.is_set():
                try:
                    self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    if get_reasons:
                        r = int(get_reasons(self.h))
                        for k, bit in names.items():
                            if r & bit:
                                self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------- own arm
class _CAI:
    def __init__(self, arr):
        self.__cuda_array_interface__ = arr.cuda_array_interface()


def as_torch(arr, torch, index):
    t = torch.as_tensor(_CAI(arr), device=f"cuda:{index}")
    return t.view(torch.bfloat16) if arr.dtype == 1 else t


class Env:
    """Per-process plumbing shared by the workloads."""


class Workload:
    """One BASELINE config wired through the public API: parameters (gradients in one bucket), two input sets, the
    step functions, the exchange and the optimizer."""

    def __init__(self, env, name):
        import neuronika_b200 as nk
        from neuronika_b200 import variable as V
        from neuronika_b200.parallel import FusedGradientExchange, GradientBucket, OverlappedAllReduce
        torch, dev, stream, world, rank, args = env.torch, env.dev, env.stream, env.world, env.rank, env.args
        self.env, self.name = env, name
        self.spec = spec = workload_spec(name, world)
        rng = np.random.default_rng(0)              # identical initial weights on every rank
        drng = np.random.default_rng(1000 + rank)   # per-rank data shard
        BF = nk.BF16
        gdt = nk.F32 if args.grad_dtype == "f32" else nk.BF16
        kind = os.environ.get("NK_DP_EXCHANGE", "fused") if world > 1 else "none"
        if gdt != nk.F32 and kind == "fused":
            kind = "nccl"       # the fused reduce-scatter epilogue sums f32 gradients
        self.exchange_kind = kind
        self.fused = None
        self.live = {}
        live = self.live

        def make_bucket(shapes):
            if world == 1:      # no exchange step: let the graph own (and lazily clear) the gradients
                return None, [None] * len(shapes)
            if self.exchange_kind == "fused":
                try:
                    self.fused = FusedGradientExchange(dev, stream, shapes, world, rank,
                                                       reduce_ctas=int(os.environ.get("NK_DP_REDUCE_CTAS", "0")))
                    return self.fused.bucket, self.fused.bucket.views
                except RuntimeError as e:
                    # peer memory could not be set up (the error is collective: every rank gets here together): the
                    # exchange falls back from the fused NVLink path to NCCL all-reduce, and the JSON line says so
                    if rank == 0:
                        print(f"bench: fused exchange unavailable ({e}); using the NCCL all-reduce exchange", file=sys.stderr)
                    self.exchange_kind = "nccl"
            b = GradientBucket(dev, shapes, gdt)
            return b, b.views

        def param(values, grad_view):
            return V.from_ndarray(dev, values, BF).requires_grad(gdt, grad_view)

        def pinned_bf16(arr):
            return torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).to(torch.bfloat16).pin_memory()

        self.opt = None
        if name == "linear":
            n, fin, fout = spec["batch"], spec["fin"], spec["fout"]
            k = 1.0 / np.sqrt(fin)
            self.bucket, (gw, gb) = make_bucket([(fout, fin), (fout,)])
            W = param(rng.uniform(-k, k, (fout, fin)).astype(np.float32), gw)
            b = param(rng.uniform(-k, k, (fout,)).astype(np.float32), gb)
            self.params = [W, b]
            x_host = drng.uniform(-1, 1, (n, fin)).astype(np.float32)
            t_host = drng.uniform(-1, 1, (n, fout)).astype(np.float32)
            px, pt = pinned_bf16(x_host), pinned_bf16(t_host)

            def make_inputs():
                x = V.from_ndarray(dev, x_host, BF).requires_grad()   # input as VarDiff => dX is computed
                t = V.from_ndarray(dev, t_host, BF)
                return {"x": x, "t": t, "copies": [(px, x), (pt, t)]}

            # every step builds its graph anew (define-by-run, as a user of the reference does each iteration: the op
            # nodes and their intermediate tensors / gradients are fresh, the leaves persist)
            def step_resident(inp):         # root = y, backward(seed)
                for p in self.params:
                    p.zero_grad()
                inp["x"].zero_grad()
                y = inp["x"].mm_t(W) + b
                y.forward()
                y.backward(1.0 / (n * fout))
                live["root"] = y

            def step_e2e(inp):              # loss = mse(y, t)
                for p in self.params:
                    p.zero_grad()
                inp["x"].zero_grad()
                loss = (inp["x"].mm_t(W) + b).mse_loss(inp["t"])
                loss.forward()
                loss.backward(1.0)
                live["root"] = loss
        elif name == "mlp":
            sizes, bsz = spec["sizes"], spec["batch"]
            shapes = []
            for i, o in zip(sizes[:-1], sizes[1:]):
                shapes += [(o, i), (o,)]
            self.bucket, gviews = make_bucket(shapes)
            self.params = []
            for li, (i, o) in enumerate(zip(sizes[:-1], sizes[1:])):
                k = 1.0 / np.sqrt(i)
                self.params.append(param(rng.uniform(-k, k, (o, i)).astype(np.float32), gviews[2 * li]))
                self.params.append(param(rng.uniform(-k, k, (o,)).astype(np.float32), gviews[2 * li + 1]))
            params = self.params
            x_host = drng.uniform(-1, 1, (bsz, sizes[0])).astype(np.float32)
            t_host = np.eye(10, dtype=np.float32)[np.argmax(x_host[:, :10], 1)]
            px, pt = pinned_bf16(x_host), pinned_bf16(t_host)

            def make_inputs():
                x = V.from_ndarray(dev, x_host, BF)
                t = V.from_ndarray(dev, t_host, BF)
                return {"x": x, "t": t, "copies": [(px, x), (pt, t)]}
            self.opt = nk.optim.StochasticGD.new(0.01, nk.optim.L2(0.0), grad_scale=1.0 / world,
                                                 master_weights=args.master_weights)
            for p in params:
                self.opt.register(p)

            def step_resident(inp):         # a training iteration as written against the reference: new graph every step
                self.opt.zero_grad()
                h = inp["x"]
                for li in range(3):
                    h = h.mm_t(params[2 * li]) + params[2 * li + 1]
                    h = h.relu() if li < 2 else h.softmax(1)
                loss = h.mse_loss(inp["t"])
                loss.forward()
                loss.backward(1.0)
                live["root"] = loss
            step_e2e = step_resident
        elif name == "convnet":
            bsz = spec["batch"]
            shapes = [(32, 3, 3, 3), (32, 1, 1), (64, 32, 3, 3), (64, 1, 1), (10, 65536), (10,)]
            self.bucket, gviews = make_bucket(shapes)
            self.params = []
            for sh, gv in zip(shapes, gviews):
                fan = int(np.prod(sh[1:])) if len(sh) > 1 and sh[1:] != (1, 1) else {32: 27, 64: 288, 10: 65536}[sh[0]]
                kk = 1.0 / np.sqrt(fan)
                self.params.append(param(rng.uniform(-kk, kk, sh).astype(np.float32), gv))
            params = self.params
            x_host = drng.uniform(0, 1, (bsz, 3, 32, 32)).astype(np.float32)
            t_host = np.eye(10, dtype=np.float32)[drng.integers(0, 10, bsz)]
            px, pt = pinned_bf16(x_host), pinned_bf16(t_host)

            def make_inputs():
                x = V.from_ndarray(dev, x_host, BF)
                t = V.from_ndarray(dev, t_host, BF)
                return {"x": x, "t": t, "copies": [(px, x), (pt, t)]}
            self.opt = nk.optim.StochasticGD.new(0.01, nk.optim.L2(0.0), grad_scale=1.0 / world)
            for p in params:
                self.opt.register(p)

            def step_resident(inp):
                self.opt.zero_grad()
                h = (params[0].convolution(inp["x"].pad((1, 1)), (1, 1), (1, 1), 1) + params[1]).relu()
                h = (params[2].convolution(h.pad((1, 1)), (1, 1), (1, 1), 1) + params[3]).relu()
                h = (h.flatten().mm_t(params[4]) + params[5]).softmax(1)
                loss = h.mse_loss(inp["t"])
                loss.forward()
                loss.backward(1.0)
                live["root"] = loss
            step_e2e = step_resident
        else:  # conv
            n, cin, hh, ww = spec["shape"]
            cout, ks = spec["cout"], spec["k"]
            k = 1.0 / np.sqrt(cin * ks * ks)
            self.bucket, (gw, gb) = make_bucket([(cout, cin, ks, ks), (cout, 1, 1)])
            Wc = param(rng.uniform(-k, k, (cout, cin, ks, ks)).astype(np.float32), gw)
            bc = param(rng.uniform(-k, k, (cout, 1, 1)).astype(np.float32), gb)
            self.params = [Wc, bc]
            x_host = drng.uniform(0, 1, (n, cin, hh, ww)).astype(np.float32)
            px = pinned_bf16(x_host)

            def make_inputs():
                x = V.from_ndarray(dev, x_host, BF).requires_grad()
                return {"x": x, "copies": [(px, x)]}

            def step_resident(inp):
                for p in self.params:
                    p.zero_grad()
                inp["x"].zero_grad()
                y = Wc.convolution(inp["x"], (1, 1), (1, 1), 1) + bc
                y.forward()
                y.backward(1.0 / 1e6)
                live["root"] = y

            def step_e2e(inp):
                for p in self.params:
                    p.zero_grad()
                inp["x"].zero_grad()
                loss = (Wc.convolution(inp["x"], (1, 1), (1, 1), 1) + bc).mean()
                loss.forward()
                loss.backward(1.0)
                live["root"] = loss

        self.step_resident, self.step_e2e = step_resident, step_e2e
        # N > 1: the exchange starts inside backward (gradient-ready hooks / fused GEMM epilogue) on a side stream
        self.sync = None
        if world > 1 and self.fused is not None:
            self.sync = self.fused
            self.sync.attach(self.params)
        elif world > 1:
            self.sync = OverlappedAllReduce(self.bucket, stream, self.params,
                                            max_chunks=int(os.environ.get("NK_DP_CHUNKS", "1")))
        # two sets of input leaves: while step k computes on one, the pinned-host -> HBM copy of step k+1 fills the other
        self.sets = [make_inputs(), make_inputs()]
        self.h2d_views = [[(src, as_torch(var.data_array(), torch, env.local)) for src, var in st["copies"]]
                          for st in self.sets]
        self.h2d_bytes = sum(int(src.numel()) * 2 for src, _ in self.sets[0]["copies"])
        self.graphs = {}

    # ---- one full step
    def full_step(self, compute, inp):
        compute(inp)
        if self.sync is not None:
            self.sync.wait()
        if self.opt is not None:
            self.opt.step()

    def capture(self, key, compute, inp):
        """Record full_step(compute, inp) into a CUDA graph (after it has run eagerly at least once)."""
        dev = self.env.dev
        with dev.capture(self.spec["arena"]) as cap:
            self.full_step(compute, inp)
        self.graphs[key] = cap.graph
        return cap.graph

    def runner(self, key, compute, inp):
        """The per-step callable: a graph replay when capture is on (and supported by the exchange), else eager."""
        use_graph = self.env.args.graph and (self.sync is None or self.fused is not None)
        if not use_graph:
            return lambda: self.full_step(compute, inp), False
        for _ in range(2):
            self.full_step(compute, inp)            # eager first: workspace growth, attribute calls, pools
        self.env.stream.synchronize()
        g = self.capture(key, compute, inp)
        return g.launch, True

    def close(self):
        for g in self.graphs.values():
            g.close()
        self.graphs = {}
        self.live.clear()


def run_own(args):
    import torch
    import torch.distributed as dist

    import neuronika_b200 as nk

    from neuronika_b200 import variable as V
    V.set_fusion(args.fusion)
    env = Env()
    env.args, env.torch, env.dist = args, torch, dist
    world = env.world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = env.rank = int(os.environ.get("RANK", "0"))
    local = env.local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    env.host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        env.host_group = dist.new_group(backend="gloo")     # host-side waits that do not spin a GPU kernel
    stream = env.stream = torch.cuda.Stream(device=local)
    dev = env.dev = nk.Device(local, stream=stream.cuda_stream)
    peaks = load_peaks()
    copy_stream = torch.cuda.Stream(device=local)
    tiny = torch.zeros(1, device=f"cuda:{local}")

    def align_ranks():
        """host barrier, then an on-device rendezvous on the compute stream: every rank leaves the tiny all-reduce at
        (nearly) the same instant, so the timed regions start together"""
        stream.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                dist.all_reduce(tiny)
            stream.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        tt = torch.tensor([v], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def timed(fn, steps, warmup, sampler=None, launches_of=None):
        """warm-up, align, time exactly `steps` calls of fn with an event after every step; returns total ms (max over
        ranks), per-step statistics and the host enqueue time per step"""
        for _ in range(warmup):
            fn()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        align_ranks()
        if sampler:
            sampler.arm()
        l0 = launches_of() if launches_of else 0
        evs[0].record(stream)
        h0 = time.perf_counter()
        for i in range(steps):
            fn()
            evs[i + 1].record(stream)
        host_ms = (time.perf_counter() - h0) * 1e3 / steps
        evs[-1].synchronize()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        launches = (launches_of() - l0) if launches_of else 0
        per = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(steps)])
        total = max_over_ranks(evs[0].elapsed_time(evs[-1]))
        stats = {"median": round(max_over_ranks(float(np.median(per))), 5), "max": round(max_over_ranks(float(per.max())), 5),
                 "min": round(float(per.min()), 5)}
        return total, stats, host_ms, launches, clocks

    def e2e_loop(wl, launchers, steps):
        """`steps` end-to-end iterations: per step the pinned-host -> HBM copy of the inputs (double-buffered on a copy
        stream), the step, and the loss scalar read back to pinned host memory (read one step late)."""
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
        loss_pinned = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]

        def issue_copy(k):
            i = k & 1
            copy_stream.wait_event(consumed[i])          # the step that last read this set has finished with it
            with torch.cuda.stream(copy_stream):
                for src, dst in wl.h2d_views[i]:
                    dst.copy_(src.view(dst.shape), non_blocking=True)
            copied[i].record(copy_stream)

        losses = []
        for i in range(2):
            consumed[i].record(stream)
        issue_copy(0)
        for k in range(steps):
            i = k & 1
            if k + 1 < steps:
                issue_copy(k + 1)
            stream.wait_event(copied[i])
            launchers[i]()
            loss_t = wl.e2e_loss_views[i] if wl.e2e_loss_views else as_torch(wl.live["root"].data_array(), torch, local)
            with torch.cuda.stream(stream):
                loss_pinned[i].copy_(loss_t.view(()), non_blocking=True)
            loss_ready[i].record(stream)
            consumed[i].record(stream)
            if k >= 1:                                   # read the previous step's loss while this one runs
                loss_ready[i ^ 1].synchronize()
                losses.append(float(loss_pinned[i ^ 1]))
        loss_ready[(steps - 1) & 1].synchronize()
        losses.append(float(loss_pinned[(steps - 1) & 1]))
        return losses

    def measure(name, steps, warmup, full, dump_dir=None):
        """resident-loop timing of one workload (+ e2e, eager and sustained legs when `full`); with `dump_dir`, what the
        last timed step computed is written there before any other leg runs"""
        wl = Workload(env, name)
        spec = wl.spec
        sampler = ClockSampler(local) if full else None
        if sampler:
            sampler.start()
        fn, graphed = wl.runner("res", wl.step_resident, wl.sets[0])
        counter = lambda: dev.launches + (wl.sync.launches if hasattr(wl.sync, "launches") and not graphed else 0)
        ms, stats, host_ms, launches, clocks = timed(fn, steps, warmup, sampler, counter)
        if dump_dir and rank == 0:
            dump_outputs(wl, dump_dir, torch, local)
        per_step = ms / steps
        flops_total = spec["flops_per_rank_step"] * world
        out = {"workload": spec["name"], "scaling": spec["scaling"], "steps": steps, "ms_per_step": round(per_step, 5),
               "ms_per_step_stats": stats, "value": round(flops_total / (per_step * 1e-3) / 1e9, 1), "unit": "GFLOP/s",
               "samples_per_s": round(spec["samples_per_rank_step"] * world / (per_step * 1e-3), 1),
               "host_enqueue_ms_per_step": round(host_ms, 5), "gpu_launches": int(launches),
               "cuda_graph": bool(graphed), "exchange": wl.exchange_kind,
               "kernels": {"gemm": dev.last_gemm_kernel, "conv": dev.last_conv_kernel}}
        if graphed:
            out["graph_kernels_per_step"] = wl.graphs["res"].kernel_count
            out["graph_arena_mb"] = round(wl.graphs["res"].arena_used / 2 ** 20, 1)
        # step-level roofline (the kernel-level one for the default workload is computed separately)
        per_rank = per_step * 1e-3
        if spec["bound"] == "hbm":
            ach = spec["bytes_per_rank_step"] / per_rank / 1e9
            out["step_roofline"] = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": round(ach / peaks["hbm_gbs"], 4),
                                    "algorithmic_bytes_per_step": spec["bytes_per_rank_step"],
                                    "note": "algorithmic bytes as SURVEY.md 8-d defines them (x, y, G, x, dx each once, bf16); "
                                            "the resident step seeds the root with backward(seed), whose uniform gradient the "
                                            "backward kernel synthesises instead of reading, so its DRAM traffic is lower"}
        else:
            ach = spec["flops_per_rank_step"] / per_rank / 1e12
            out["step_roofline"] = {"bound": "tensor", "achieved": round(ach, 1), "peak": peaks["tflops_sustained"],
                                    "unit": "TFLOP/s", "frac": round(ach / peaks["tflops_sustained"], 4),
                                    "frac_of_burst": round(ach / peaks["tflops_burst"], 4),
                                    "algorithmic_flops_per_step": spec["flops_per_rank_step"]}
        extra = {"clocks": clocks, "wl": wl, "graphed": graphed}
        if not full:
            return out, extra
        # ---- the same step enqueued kernel by kernel (no graph): what the host costs
        if graphed:
            esteps = max(5, min(steps, 30))
            ems, _, ehost, _, _ = timed(lambda: wl.full_step(wl.step_resident, wl.sets[0]), esteps, 2)
            out["eager_ms_per_step"] = round(ems / esteps, 5)
            out["eager_host_enqueue_ms_per_step"] = round(ehost, 5)
        # ---- sustained behaviour: the same step back to back for ~1.5 s with the clocks sampled
        if args.sustain_s > 0:
            n_s = int(min(20000, max(steps, args.sustain_s * 1e3 / max(per_step, 1e-3))))
            s2 = ClockSampler(local, period_s=0.01)
            s2.start()
            sms, sstats, _, _, sclk = timed(fn, n_s, 0, s2)
            out["sustained"] = {"steps": n_s, "seconds": round(sms / 1e3, 3), "ms_per_step": round(sms / n_s, 5),
                                "sm_mhz": sclk["sm_mhz"] if sclk else None, "reasons": sclk["reasons"] if sclk else None}
        # ---- end to end: inputs from pinned host memory every step, loss read back
        e2e_steps = max(3, min(steps, args.e2e_steps))
        launchers, views = [], []
        for i in range(2):
            f_i, g_i = wl.runner(f"e2e{i}", wl.step_e2e, wl.sets[i])
            launchers.append(f_i)
            # a captured step writes its loss scalar to a fixed address: wrap it once, right after its capture
            views.append(as_torch(wl.live["root"].data_array(), torch, local) if g_i else None)
        wl.e2e_loss_views = views if graphed else None
        e2e_loop(wl, launchers, 3)                          # warm-up (pinned buffers, allocator pools)
        align_ranks()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)                                   # every copy of the run is ordered after this point ...
        losses = e2e_loop(wl, launchers, e2e_steps)
        e1.record(stream)                                   # ... and the last loss read-back before this one
        e1.synchronize()
        torch.cuda.synchronize()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        out["e2e"] = {"value": round(flops_total / (ms_e2e / e2e_steps * 1e-3) / 1e9, 1), "unit": "GFLOP/s",
                      "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": 4,
                      "ms_per_step": round(ms_e2e / e2e_steps, 5), "steps": e2e_steps,
                      "last_loss": round(float(losses[-1]), 6),
                      "what": "per step: pinned host -> HBM copy of the step's inputs (double-buffered on a copy stream, so "
                              "the copy of step k+1 overlaps the compute of step k), the step (graph build, forward, backward"
                              + (", exchange" if world > 1 else "") + (", sgd" if wl.opt is not None else "")
                              + "; replayed from its CUDA graph)" * bool(graphed)
                              + ", loss scalar read back to pinned host memory (read one step late)"}
        return out, extra

    # ---- main workload
    W_ = max(args.warmup, 3)
    main, mx = measure(args.workload, args.steps, W_, full=not args.profile, dump_dir=args.dump_outputs)
    wl = mx["wl"]
    if args.profile:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "profile_only": True, "ms_per_step": main["ms_per_step"],
                              "gpu_launches": main["gpu_launches"], "workload": main["workload"]}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    out = {
        "metric": METRIC, "value": main["value"], "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": W_, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
        "scaling": main["scaling"], "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "samples_per_s": main["samples_per_s"], "ms_per_step_stats": main["ms_per_step_stats"],
        "config": {"workload": main["workload"], "grad_dtype": args.grad_dtype, "parallelism": f"dp{world}",
                   "exchange": main["exchange"], "cuda_graph": main["cuda_graph"], "fusion_level": args.fusion,
                   "step": "zero_grad -> build graph -> forward -> backward"
                           + ({"none": "", "nccl": " (+ overlapped nccl all_reduce of each layer's grad slice)",
                               "fused": " (dW GEMM epilogue reduce-scatters over NVLink peer memory; one barrier+reduce+"
                                        "broadcast kernel per matrix and a peer-memory all-reduce of the small tensors "
                                        "on a side stream)"}[main["exchange"]])
                           + (" -> sgd" if wl.opt is not None else "")
                           + ("; the step is captured once in a CUDA graph and replayed" if main["cuda_graph"] else ""),
                   "l2": "working set per step exceeds the 126 MB L2 (no flush needed)", "kernels": main["kernels"]},
        "gpu_launches": main["gpu_launches"], "host_enqueue_ms_per_step": main["host_enqueue_ms_per_step"],
        "clocks": mx["clocks"], "e2e": main["e2e"], "step_roofline": main["step_roofline"],
    }
    for k in ("eager_ms_per_step", "eager_host_enqueue_ms_per_step", "sustained", "graph_kernels_per_step", "graph_arena_mb"):
        if k in main:
            out[k] = main[k]

    # ---- N > 1: the fused exchange against an NCCL all-reduce of locally computed gradients, in this very process
    if world > 1 and wl.fused is not None:
        out["exchange_parity"] = exchange_parity(env, wl)

    # ---- roofline of the dominant kernel, timed live with CUDA events on the launching stream (rank 0 computes, all wait)
    if rank == 0:
        out["roofline"] = roofline(args, dev, nk, wl.spec, peaks, stream)
    wl.close()
    del wl, mx

    # ---- the other BASELINE configs in the same process
    others = [w for w in args.others.split(",") if w and w != args.workload and w != "none"]
    if others:
        out["other_configs"] = {}
        osteps = max(10, min(args.steps, args.other_steps))
        for w in others:
            try:
                res, ex = measure(w, osteps, 3, full=False)
                ex["wl"].close()
                del ex
                out["other_configs"][w] = res
            except Exception as e:      # noqa: BLE001 -- a failing extra config must not lose the main line
                out["other_configs"][w] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    # ---- CPU baseline on rank 0 while the other ranks wait on the HOST (no GPU kernel spinning)
    torch.cuda.synchronize()
    if rank == 0:
        out["cpu_baseline"] = cpu_baseline(args.workload, budget_s=args.cpu_budget)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier(group=env.host_group)
        dist.destroy_process_group()


PARAM_NAMES = {"linear": ["weight", "bias"], "conv": ["weight", "bias"],
               "mlp": ["linear1_weight", "linear1_bias", "linear2_weight", "linear2_bias", "linear3_weight", "linear3_bias"],
               "convnet": ["conv1_weight", "conv1_bias", "conv2_weight", "conv2_bias", "linear_weight", "linear_bias"]}
DUMP_SAMPLE = 1 << 20           # elements kept of a larger output: a fixed, seeded sample of its flat indices
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(wl, out_dir, torch, index):
    """Write what the step returns to its caller as <out_dir>/<name>.npy (float32): the root's value (the layer output, or
    the loss), the gradient of every leaf that has one, and the parameters where an optimizer updated them.  The inputs
    are seeded, so two builds run with the same arguments can be compared output for output."""
    from neuronika_b200.variable import VarDiff
    arrays = {"output": wl.live["root"].data_array()}
    x = wl.sets[0]["x"]
    if isinstance(x, VarDiff):
        arrays["input_grad"] = x.grad_array()
    for name, p in zip(PARAM_NAMES[wl.name], wl.params):
        arrays[f"{name}_grad"] = p.grad_array()
        if wl.opt is not None:
            arrays[name] = p.data_array()
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, arr in arrays.items():
        t = as_torch(arr, torch, index).reshape(-1)
        if arr.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(arr.size, DUMP_SAMPLE, replace=False))
            host = t[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()
        else:
            host = t.float().cpu().numpy().reshape(arr.shape)
        total += host.nbytes
        np.save(os.path.join(out_dir, f"{name}.npy"), host)
    assert total <= DUMP_MAX_BYTES, total


def exchange_parity(env, wl):
    """One more step with the fused exchange, then the same step with the exchange detached (gradients stay local) and an
    NCCL all-reduce of the local bucket: the two buckets must agree (bit for bit at two ranks, where a + b is order
    independent; to rounding otherwise -- the owner sums in rank order, NCCL in ring order)."""
    torch, dist, stream = env.torch, env.dist, env.stream
    # compute + exchange WITHOUT the optimizer step: the SGD kernel scales the bucket by 1/world in place and moves the
    # weights, so a comparison after a full step would compare different things
    wl.step_resident(wl.sets[0])
    wl.sync.wait()
    stream.synchronize()
    fused = wl.bucket.as_torch().clone()
    wl.fused.detach()
    wl.step_resident(wl.sets[0])
    stream.synchronize()
    ref = wl.bucket.as_torch().clone()
    dist.all_reduce(ref)
    torch.cuda.synchronize()
    wl.fused.attach(wl.params)
    diff = (fused - ref).abs().max().item()
    scale = ref.abs().max().item() + 1e-30
    bit_equal = bool(torch.equal(fused, ref))
    # the GEMM-pushed matrices: one f32 sum per element, a + b at two ranks is order independent -> bit equal there.  The
    # other tensors (bias column sums, the 10-row dW of the skinny kernel) are accumulated with f32 atomics inside each
    # backward, so two runs of the same backward already differ in the last bits: those are compared to rounding.
    lay = wl.fused.layout
    fused_equal = True
    for pi in wl.fused.fused:
        lo, n = lay.offsets[pi], int(np.prod(lay.shapes[pi]))
        fused_equal = fused_equal and bool(torch.equal(fused[lo:lo + n], ref[lo:lo + n]))
    ok = diff <= 1e-5 * scale and (fused_equal or env.world != 2)
    flag = torch.tensor([1 if ok else 0], device=fused.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"ok_all_ranks": bool(int(flag.item()) == 1), "bit_equal_rank0": bit_equal,
            "gemm_pushed_matrices_bit_equal_rank0": fused_equal, "max_abs_diff": diff,
            "max_abs_ref": scale, "elements": int(ref.numel()),
            "what": "fused NVLink exchange vs NCCL all-reduce of the locally computed gradient bucket, same inputs; bound: "
                    "1e-5 * max|ref| everywhere, and at two ranks bit equality of the GEMM-pushed matrices"}


def measured_traffic(key):
    """DRAM bytes per launch measured with ncu for the roofline kernels (profiles/r0N_traffic.json, committed with the
    launch lists they were extracted from); None when no file has the kernel."""
    for f in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", f)) as fh:
                return float(json.load(fh)[key]["bytes_per_launch"])
        except Exception:
            continue
    return None


def roofline(args, dev, nk, spec, peaks, stream):
    from neuronika_b200 import ops
    iters = max(30, min(200, args.steps))
    rng = np.random.default_rng(7)
    if spec["bound"] == "tensor":
        # the three GEMMs of the Linear step as the step runs them, on random operands:
        #   NT  y(bf16)  = x.W^T + b      NN  dX(bf16) = G.W      TN  dW(f32) = G^T.X
        n = 4096
        mk = lambda: dev.from_ndarray(rng.uniform(-1, 1, (n, n)).astype(np.float32), nk.BF16)
        a, b = mk(), mk()
        bias = dev.from_ndarray(rng.uniform(-1, 1, (n,)).astype(np.float32), nk.BF16)
        c16 = nk.CuArray(dev, (n, n), nk.BF16)
        c32 = nk.CuArray(dev, (n, n), nk.F32)
        forms = {}
        for name, kw, c in (("nt_fwd_bias_bf16out", dict(trans_b=True, bias=bias), c16), ("nn_dx_bf16out", dict(), c16),
                            ("tn_dw_f32out", dict(trans_a=True), c32)):
            for _ in range(3):
                ops.gemm(a, b, c, **kw)
            stream.synchronize()
            dev.timer_start()
            for _ in range(iters):
                ops.gemm(a, b, c, **kw)
            forms[name] = dev.timer_stop() / iters
        dur = float(np.mean(list(forms.values())))
        achieved = 2.0 * n ** 3 / (dur * 1e-3) / 1e12
        peak = peaks["tflops_burst"]      # a kernel timed alone in a short loop runs in the burst regime
        return {"bound": "tensor", "achieved": round(achieved, 1), "peak": peak, "unit": "TFLOP/s",
                "frac": round(achieved / peak, 4),
                "frac_of_sustained": round(achieved / peaks["tflops_sustained"], 4),
                "traffic": measured_traffic("gemm_tc_4096"),
                "traffic_note": "tensor-bound kernel: DRAM bytes per launch (ncu) vs 96-128 MB of operands + output",
                "kernel": f"gemm_tc_kernel ({dev.last_gemm_kernel}: tcgen05 cta_group::2, 256x256x64 tiles over CTA pairs, TMA-store "
                          "epilogue); mean of the step's own three 4096^3 launches (NT +bias bf16 out, NN bf16 out, TN f32 out), "
                          "random operands",
                "per_form_ms": {k: round(v, 5) for k, v in forms.items()}, "launches_timed": 3 * iters,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops (burst, {peaks['source']}); sustained {peaks['tflops_sustained']}",
                "algorithmic_flops_per_launch": 2.0 * n ** 3}
    # conv: HBM bound
    nb, cin, h, w = spec["shape"]
    cout, k = spec["cout"], spec["k"]
    x = dev.from_ndarray(rng.uniform(0, 1, (nb, cin, h, w)).astype(np.float32), nk.BF16)
    wt = dev.from_ndarray(rng.uniform(-0.2, 0.2, (cout, cin, k, k)).astype(np.float32), nk.BF16)
    y = nk.CuArray(dev, (nb, cout, h - k + 1, w - k + 1), nk.BF16)
    for _ in range(2):
        ops.conv2d(x, wt, out=y)
    stream.synchronize()
    iters = min(iters, 20)
    dev.timer_start()
    for _ in range(iters):
        ops.conv2d(x, wt, out=y)
    dur = dev.timer_stop() / iters
    bytes_alg = 2.0 * (x.size + y.size)
    achieved = bytes_alg / (dur * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": measured_traffic("conv_fwd_tc"),
            "kernel": f"conv2d forward ({dev.last_conv_kernel})", "ms": round(dur, 5),
            "algorithmic_bytes_per_launch": bytes_alg, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks['source']})"}


# ------------------------------------------------------------------------------------------- CPU arms
def cpu_step_fn(workload: str, sample_batch: int):
    """One forward+backward of the workload on the host with the oracle (the reference's algorithm
    restated in numpy f32 -- the reference itself cannot be built here).  Returns (fn, flops, description)."""
    import oracle as O
    rng = np.random.default_rng(0)
    if workload in ("linear", "mlp"):
        n, fin, fout = sample_batch, 4096, 4096
        k = 1 / 64.0
        x = rng.uniform(-1, 1, (n, fin)).astype(np.float32)
        w = rng.uniform(-k, k, (fout, fin)).astype(np.float32)
        b = rng.uniform(-k, k, (fout,)).astype(np.float32)
        g = (rng.uniform(-1, 1, (n, fout)) / n).astype(np.float32)

        def fn():
            y = O.linear_forward(x, w, b)
            dx, dw, db = np.zeros_like(x), np.zeros_like(w), np.zeros_like(b)
            O.linear_backward(x, w, g, dx, dw, db)
            return y
        what = f"Linear 4096->4096 fwd+bwd, batch {n}" + ("" if n == 4096 else " rows (of 4096)") + ", numpy f32"
        return fn, 3 * 2.0 * n * fin * fout, what
    n = sample_batch
    x = rng.uniform(0, 1, (n, 3, 224, 224)).astype(np.float32)
    w = rng.uniform(-0.19, 0.19, (64, 3, 3, 3)).astype(np.float32)
    b = rng.uniform(-0.19, 0.19, (64, 1, 1)).astype(np.float32)

    def fn():
        y = O.conv2d_layer_forward(x, w, b)
        g = np.full(y.shape, 1.0 / y.size, np.float32)
        dx, dw, db = np.zeros_like(x), np.zeros_like(w), np.zeros_like(b)
        O.conv2d_layer_backward(x, w, g, dx, dw, db)
        return y
    return fn, 3 * 2.0 * n * 64 * 222 * 222 * 27, f"Conv2d 3->64 k3 224x224 fwd+bwd on a batch of {n} (of 256), im2col + sgemm in numpy f32"


def _time_reps(fn, budget_s, max_reps):
    fn()
    t0 = time.perf_counter()
    times = []
    while True:
        s = time.perf_counter()
        fn()
        times.append(time.perf_counter() - s)
        if time.perf_counter() - t0 > budget_s or len(times) >= max_reps:
            break
    return times


def single_thread_baseline(workload: str, budget_s: float = 4.0):
    """The reference's default GEMM (`matrixmultiply`) is single threaded: the same port with BLAS limited to 1 thread."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return None
    sample = 256 if workload != "conv" else 1
    fn, flops, what = cpu_step_fn(workload, sample)
    with threadpool_limits(limits=1):
        times = _time_reps(fn, budget_s, 10)
    dt = float(np.median(times))
    return {"value": round(flops / dt / 1e9, 2), "unit": "GFLOP/s", "cores": 1,
            "sample": f"{what}; {len(times)} repetitions, median {dt:.3f} s, BLAS threads = 1"}


class _all_cores:
    """torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently turn the "all host cores" baseline into a
    single-thread one: set the BLAS pool to the core count explicitly."""

    def __enter__(self):
        try:
            from threadpoolctl import threadpool_limits
            self._ctx = threadpool_limits(limits=os.cpu_count() or 1)
            self._ctx.__enter__()
        except Exception:
            self._ctx = None
        return self

    def __exit__(self, *a):
        if self._ctx is not None:
            self._ctx.__exit__(*a)
        return False


def cpu_baseline(workload: str, budget_s: float = 12.0):
    cores = os.cpu_count() or 1
    sample = 4096 if workload != "conv" else 8
    fn, flops, what = cpu_step_fn(workload, sample)
    with _all_cores():
        times = _time_reps(fn, budget_s, 50)
    dt = float(np.median(times))
    out = {"value": round(flops / dt / 1e9, 2), "unit": "GFLOP/s", "cores": cores, "kind": "port",
           "sample": f"{what}; {len(times)} repetitions, median {dt:.3f} s (min {min(times):.3f}, max {max(times):.3f}), "
                     f"BLAS threads = all {cores} host cores",
           "single_thread": single_thread_baseline(workload)}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Rust crate cannot be
    built in this environment (no rustc/cargo), so this times the oracle port on the host cores, on the SAME config as
    the own arm (full batch for the Linear / MLP workloads; a bounded batch sample of the convolution)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    spec = workload_spec(args.workload, max(1, world))
    cores = os.cpu_count() or 1
    sample = 4096 if args.workload != "conv" else 8
    fn, flops, what = cpu_step_fn(args.workload, sample)
    steps = max(1, min(args.steps, 20))
    times = []
    with _all_cores():
        for _ in range(max(1, min(args.warmup, 2))):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            s = time.perf_counter()
            fn()
            times.append(time.perf_counter() - s)
        dt = (time.perf_counter() - t0) / steps
    val = round(flops / dt / 1e9, 2)
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "GFLOP/s", "n_gpus": args.gpus,
           "steps": steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
           "scaling": spec["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "ms_per_step_stats": {"median": round(float(np.median(times)) * 1e3, 3), "min": round(min(times) * 1e3, 3),
                                 "max": round(max(times) * 1e3, 3)},
           "config": {"workload": spec["name"], "parallelism": "cpu"},
           "cpu_baseline": {"value": val, "unit": "GFLOP/s", "cores": cores, "kind": "port",
                            "sample": f"{what}; one step = one fwd+bwd; BLAS threads = all {cores} host cores",
                            "single_thread": single_thread_baseline(args.workload)},
           "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="linear", choices=["linear", "mlp", "conv", "convnet"])
    ap.add_argument("--others", default="conv,mlp,convnet", help="other BASELINE configs measured in the same process ('none')")
    ap.add_argument("--other-steps", type=int, default=50)
    ap.add_argument("--grad-dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--master-weights", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--sustain-s", type=float, default=1.5)
    ap.add_argument("--fusion", type=int, default=2, choices=[0, 1, 2, 3],
                    help="host-side peephole level (nkg_set_fusion): 2 = also ReLU backward in the dX GEMM epilogue")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="enqueue every step eagerly (no CUDA graph)")
    ap.add_argument("--profile", action="store_true",
                    help="only the warm-up + timed steps (no e2e / roofline / cpu legs): for ncu launch lists")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (rank 0) as DIR/<name>.npy, float32; "
                         f"outputs above {DUMP_SAMPLE} elements as a fixed seeded sample of that many")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
