#!/usr/bin/env python
"""Benchmark of the NoisyNet hot path: CIFAR-10 4-bit NoisyNet (I_max = 1 nA) training images/sec.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)

A "step" = one full training step (forward, loss, backward, AdamW, weight clamp -- noisynet.py:1276-1542)
over one batch of synthetic CIFAR-10-shaped 4-bit data (random-init weights; no dataset on disk).
Workload = BASELINE.json configs[1]: NoisyNet, --current 1 --act_max 5 --w_max1 0.3, --q_a 4 --q_w 4,
batch 512 per GPU.  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FLOP_FWD = {"conv1": 15.288e6, "conv2": 78.0e6, "fc1": 4.68e6, "fc2": 0.0156e6}   # main + sigma^2, per image
FLOP_STEP = 188.3e6                                                                # SURVEY.md section 8a


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    p.add_argument("--no-library-baseline", action="store_true")
    p.add_argument("--no-second-variant", action="store_true")
    p.add_argument("--batch", type=int, default=512, help="per-GPU batch")
    p.add_argument("--variant", default="q4", choices=["q4", "fp"], help="q4: --q_a 4 --q_w 4; fp: README flags")
    p.add_argument("--flow", default="engine", choices=["engine", "fused", "dropin"],
                   help="engine: explicit kernel schedule (NoisyNetEngine); fused/dropin: autograd module paths")
    p.add_argument("--precision", default=os.environ.get("NN_BENCH_PRECISION", "auto"))
    p.add_argument("--optimizer", default="fused", choices=["fused", "torch"])
    p.add_argument("--graph", type=int, default=int(os.environ.get("NN_BENCH_GRAPH", "1")))
    p.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--pool", type=int, default=24, help="distinct resident input batches cycled through")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last one computed (loss; every parameter, its gradient and the "
                        "floating-point buffers it updated) as DIR/<name>.npy; inputs and seeds are fixed by the arguments, "
                        "so two builds can be compared output for output")
    return p.parse_args()


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return d, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML during the timed region."""

    def __init__(self, index=0, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80, "sync_boost": 0x10,
                 "applications_clocks_setting": 0x2}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.ok:
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------ reference / CPU arm
def oracle_arm(batch, variant, steps, warmup, seconds=None):
    """The reference's CPU implementation of the step (oracle port, torch CPU fp32, all host threads)."""
    from oracle import noisynet_oracle as O
    q = 4 if variant == "q4" else 0
    a = O.default_args(q_a=q, q_w=q, quant_max2=5.0, quant_max4=5.0)
    torch.manual_seed(0)
    m = O.OracleNet(a).init_like_reference()
    opt = O.make_optimizer(m, a)
    m.train()
    x, lab = O.synthetic_cifar(batch, seed=0)
    # "all the host threads it can use": oneDNN/ATen oversubscribe badly on large shared hosts, so pick the
    # fastest intra-op thread count among {affinity, 64, 32, 16, 8} with one probe step each.
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    best_t, best_dt = None, None
    xs, ls = x[:min(batch, 64)], lab[:min(batch, 64)]
    for t in sorted({avail, 64, 32, 16, 8}):
        if t > avail:
            continue
        torch.set_num_threads(t)
        O.train_step(m, opt, xs, ls, i=100)
        t0 = time.perf_counter()
        O.train_step(m, opt, xs, ls, i=100)
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best_t, best_dt = t, dt
    torch.set_num_threads(best_t)
    for s in range(warmup):
        O.train_step(m, opt, x, lab, i=100)
    t0 = time.perf_counter()
    n = 0
    while True:
        O.train_step(m, opt, x, lab, i=100)
        n += 1
        el = time.perf_counter() - t0
        if (seconds is not None and el >= seconds) or (seconds is None and n >= steps):
            break
    return {"img_s": n * batch / el, "steps": n, "seconds": el, "cores": torch.get_num_threads(), "batch": batch}


def torch_gpu_arm(batch, variant, steps, warmup, dev):
    """The bar SURVEY.md section 2.2 / BASELINE.md section 3 name: the reference's step in PyTorch-eager on the SAME B200
    (cuDNN / cuBLAS contractions, ATen elementwise + Philox kernels, torch.optim.AdamW) -- the oracle port of the reference
    step moved to the GPU unchanged, inputs resident on the device, timed with CUDA events.  Not the product path."""
    from oracle import noisynet_oracle as O
    q = 4 if variant == "q4" else 0
    a = O.default_args(q_a=q, q_w=q, quant_max2=5.0, quant_max4=5.0)
    torch.manual_seed(0)
    torch.backends.cudnn.benchmark = True          # noisynet.py:319
    m = O.OracleNet(a).init_like_reference().to(dev)
    opt = O.make_optimizer(m, a)
    m.train()
    xs, ls = [], []
    for k in range(8):
        x, lab = O.synthetic_cifar(batch, seed=k)
        xs.append(x.to(dev)); ls.append(lab.to(dev))
    l0 = None
    for s in range(max(warmup, 3)):
        l0, _ = O.train_step(m, opt, xs[s % 8], ls[s % 8], i=100)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        l0, _ = O.train_step(m, opt, xs[s % 8], ls[s % 8], i=100)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    return {"img_s": steps * batch / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "batch": batch,
            "final_loss": float(l0)}


def run_torch_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    r = torch_gpu_arm(args.batch, args.variant, args.steps, args.warmup, dev)
    line = {
        "impl": "torch_gpu", "metric": "NoisyNet CIFAR-10 4-bit training images/sec", "value": r["img_s"], "unit": "img/s",
        "n_gpus": 1, "steps": r["steps"], "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1), "final_loss": r["final_loss"],
        "note": "PyTorch-eager (cuDNN/cuBLAS/ATen) run of the reference step (oracle port) on one B200: the library bar",
    }
    print(json.dumps(line), flush=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = oracle_arm(args.batch, args.variant, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "NoisyNet CIFAR-10 4-bit training images/sec", "value": r["img_s"], "unit": "img/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / r["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": r["img_s"], "unit": "img/s", "cores": r["cores"], "kind": "port",
                         "sample": "%d steps of batch %d (oracle port of the reference step, torch CPU fp32)" % (r["steps"], args.batch)},
        "e2e": {"value": r["img_s"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": "NoisyNet CIFAR-10 (conv5x5x65 - conv5x5x120 - fc390 - fc10), I_max=1nA all layers, act_max=5, w_max1=0.3, "
                        + ("q_a=4 q_w=4 stochastic rounding" if args.variant == "q4" else "README flags (q_a=q_w=0)"),
            "per_gpu_batch": args.batch, "global_batch": args.batch * world, "parallelism": "dp%d" % world,
            "flow": args.flow, "l2_policy": "inputs+activations (>400 MB/step) exceed the 126 MB L2; %d distinct input batches cycled" % args.pool}


# ------------------------------------------------------------------------------------ our arm
def build_model(args, dev, precision):
    from noisynet_b200.net import NoisyNet, default_args, init_like_reference, make_fused_optimizer, make_optimizer, with_quant
    a = default_args()
    if args.variant == "q4":
        with_quant(a, 4, 4)
    m = init_like_reference(NoisyNet(a, fused=(args.flow != "dropin"), precision=precision)).to(dev)
    if args.variant == "q4":      # ranges as after the 5-batch calibration (noisynet.py:1251-1259): fixed running_max
        m.quantize2.running_max = torch.tensor(5.0, device=dev)
        m.quantize4.running_max = torch.tensor(5.0, device=dev)
    m.collect_stats = False       # steady state: i >= 20 (no host-synced side statistics)
    m.train()
    if args.optimizer == "fused":   # nn_adamw_step: AdamW + clamp + max|W| for all tensors in one launch
        return m, a, make_fused_optimizer(m, a, grad_scale=1.0 / max(1, int(os.environ.get("WORLD_SIZE", "1"))))
    return m, a, make_optimizer(m, a, capturable=bool(args.graph))


def time_second_variant(args, dev, precision, variant):
    """Device-resident engine step of the OTHER operand variant (same timing method as `value`)."""
    import copy
    from noisynet_b200 import _lib, ops
    from noisynet_b200.engine import NoisyNetEngine
    a2 = copy.copy(args)
    a2.variant = variant
    model, a, opt = build_model(a2, dev, precision)
    B = args.batch
    gen = torch.Generator().manual_seed(4321)
    xs = [(torch.randint(0, 16, (B, 3, 32, 32), generator=gen).float() / 15).to(dev) for _ in range(args.pool)]
    ys = [torch.randint(0, 10, (B,), generator=gen).to(dev) for _ in range(args.pool)]
    sx, sy = torch.empty_like(xs[0]), torch.empty_like(ys[0])
    engine = NoisyNetEngine(model, B, opt=opt)
    loss_out = torch.zeros((), device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for s in range(3):
            loss_out.copy_(engine.train_step(xs[s], ys[s])[0])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    lib = _lib.load()
    l0 = lib.nn_launch_count()
    engine.train_step(xs[0], ys[0])
    torch.cuda.synchronize()
    launches = int(lib.nn_launch_count() - l0)
    step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)
    graph = torch.cuda.CUDAGraph()
    with ops.graph_rng(step_ctr, seed=99):
        with torch.cuda.graph(graph):
            loss_out.copy_(engine.train_step(sx, sy)[0])
            ops.rng_advance(step_ctr, 1)
    torch.cuda.synchronize()

    def run(i):
        sx.copy_(xs[i % args.pool], non_blocking=True)
        sy.copy_(ys[i % args.pool], non_blocking=True)
        graph.replay()
    for i in range(max(args.warmup, 3)):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    assert ops.error_flag() == 0
    return {"variant": variant, "value": B * args.steps / (ms * 1e-3), "unit": "img/s", "ms_per_step": ms / args.steps,
            "gpu_launches_per_step": launches, "final_loss": loss_out.item(),
            "dtype": "bf16 operands (exact 4-bit codes)" if variant == "q4" else "bf16-rounded operands (README flags q_a=q_w=0), fp32 accumulate",
            "config": workload_config(a2, 1)["workload"]}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, loss, model):
    """The step hands its caller the loss and updates the model in place: writes the loss, every parameter, its gradient
    and the floating-point buffers (BatchNorm running statistics, quantizer ranges) as <out_dir>/<name>.npy."""
    import numpy as np
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        arrays[name] = p
        if p.grad is not None:
            arrays[name + ".grad"] = p.grad
    for name, b in model.named_buffers():
        if b.is_floating_point():
            arrays[name] = b
    host = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        host[name] = (t if t.dtype in (torch.float32, torch.float64) else t.float()).numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    sys.stderr.write("[bench] wrote %d arrays (%d bytes) to %s\n" % (len(host), total, out_dir))


def pick_precision(args, dev):
    """auto: the tcgen05 path (bf16 integer codes for q4, tf32 otherwise) if it passes a self-check, else fp32."""
    if args.precision != "auto":
        return args.precision
    from noisynet_b200 import ops
    want = "bf16"          # q4: exact integer codes in bf16; fp (README flags): bf16-rounded operands, fp32 accumulate
    try:
        x = torch.rand(8, 65, 14, 14, device=dev)
        w = torch.randn(120, 65, 5, 5, device=dev) * 0.05
        y0 = ops.noisy_conv_fwd(x, w, precision="fp32")["y"]
        y1 = ops.noisy_conv_fwd(x, w, precision=want)["y"]
        gy = torch.randn_like(y0)
        ops.conv_dgrad(gy, w, x.shape, precision=want)
        ops.conv_wgrad(gy, x, w.shape, precision=want)
        torch.cuda.synchronize()
        if (y0 - y1).abs().max().item() < 5e-2 * y0.abs().max().item():
            return want
    except Exception as e:  # noqa: BLE001
        sys.stderr.write("[bench] tcgen05 path unavailable (%s); using fp32 CUDA-core kernels\n" % e)
    return "fp32"


def run_b200(args):
    from noisynet_b200 import _lib, dp, ops
    from noisynet_b200.net import bind_absmax
    import torch.distributed as dist
    import torch.nn.functional as F
    rank, world, local = dp.init_from_env()
    assert torch.cuda.is_available(), "bench.py (impl b200) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    torch.manual_seed(dp.rank_seed(0, rank))
    precision = pick_precision(args, dev)
    model, a, opt = build_model(args, dev, precision)
    fused_opt = args.optimizer == "fused"
    red = dp.make_grad_reducer(model, world, early=[[model.linear1.weight, model.linear2.weight], [model.conv2.weight]])
    red.broadcast_parameters(model)
    B = args.batch
    gen = torch.Generator().manual_seed(1234 + rank)
    pool_x = [(torch.randint(0, 16, (B, 3, 32, 32), generator=gen).float() / 15).pin_memory() for _ in range(args.pool)]
    pool_y = [torch.randint(0, 10, (B,), generator=gen).pin_memory() for _ in range(args.pool)]
    dev_x = [t.to(dev) for t in pool_x]
    dev_y = [t.to(dev) for t in pool_y]
    sx, sy = torch.empty_like(dev_x[0]), torch.empty_like(dev_y[0])   # static inputs for the captured graph
    loss_out = torch.zeros((), device=dev)

    engine = None
    if args.flow == "engine":
        if not (fused_opt and precision == "bf16"):
            raise SystemExit("--flow engine needs the tcgen05 path (bf16) and --optimizer fused")
        from noisynet_b200.engine import NoisyNetEngine
        engine = NoisyNetEngine(model, B, opt=opt, reducer=red if world > 1 else None)

    def step_body(x, y):
        if engine is not None:
            loss_out.copy_(engine.train_step(x, y)[0])
            return
        out = model(x, 0, 100)
        loss = F.cross_entropy(out, y)
        red.zero_()
        loss.backward()
        if fused_opt:
            red.all_reduce_sum_()           # the 1/world is folded into the optimizer kernel (grad_scale)
            opt.step()
            bind_absmax(model, opt)
        else:
            red.all_reduce_mean_()
            opt.step()
            model.clamp_weights_()
        loss_out.copy_(loss.detach())

    # eager warm-up (allocator, cudnn heuristics, lazy state)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for s in range(3):
            step_body(dev_x[s % args.pool], dev_y[s % args.pool])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    l0 = lib.nn_launch_count()
    step_body(dev_x[0], dev_y[0])
    torch.cuda.synchronize()
    launches_per_step = int(lib.nn_launch_count() - l0)

    graph = None
    step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)
    if args.graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with ops.graph_rng(step_ctr, seed=dp.rank_seed(0, rank)):
                with torch.cuda.graph(graph):
                    step_body(sx, sy)
                    ops.rng_advance(step_ctr, 1)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            sys.stderr.write("[bench] CUDA-graph capture failed (%s); running eager\n" % e)
            graph = None

    def run_step(i):
        if graph is not None:
            sx.copy_(dev_x[i % args.pool], non_blocking=True)
            sy.copy_(dev_y[i % args.pool], non_blocking=True)
            graph.replay()
        else:
            step_body(dev_x[i % args.pool], dev_y[i % args.pool])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- timed region 1: inputs resident in HBM ("value")
    for i in range(max(args.warmup, 3)):
        run_step(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        run_step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    t_ms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = t_ms.item()
    value = world * B * args.steps / (ms * 1e-3)
    final_loss = loss_out.item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss_out, model)

    # ---------------- timed region 2: end to end through the public API with HOST buffers ("e2e")
    # Every step's input travels host (pinned) -> device inside the timed region; the copy of step i+1 is issued
    # on a side stream while step i computes (double buffering, as the reference's own input pipeline does:
    # timm/data/loader.py:42-64 PrefetchLoader), and the loss is read back to the host every step.
    copy_stream = torch.cuda.Stream()
    bufs = [(torch.empty_like(dev_x[0]), torch.empty_like(dev_y[0])) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    host_loss = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(i):
        k = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])          # the step that last used this buffer has read it
            bufs[k][0].copy_(pool_x[i % args.pool], non_blocking=True)
            bufs[k][1].copy_(pool_y[i % args.pool], non_blocking=True)
            ready[k].record(copy_stream)

    def e2e_step(i, last):
        k = i & 1
        cur = torch.cuda.current_stream()
        cur.wait_event(ready[k])
        if graph is not None:
            sx.copy_(bufs[k][0], non_blocking=True)
            sy.copy_(bufs[k][1], non_blocking=True)
            consumed[k].record(cur)
            if not last:
                prefetch(i + 1)
            graph.replay()
        else:
            if not last:
                prefetch(i + 1)
            step_body(bufs[k][0], bufs[k][1])
            consumed[k].record(cur)
        # device -> host read of every step's result: the copy of THIS step's loss into pinned host memory is enqueued behind
        # the step, and the host reads the PREVIOUS step's value while this one runs (a synchronous .item() per step left the
        # GPU idle for the host's launch time of the next step)
        host_loss[k].copy_(loss_out, non_blocking=True)
        loss_ev[k].record(cur)
        if i > 0:
            loss_ev[k ^ 1].synchronize()
            return float(host_loss[k ^ 1])
        return None

    for k in range(2):
        consumed[k].record(torch.cuda.current_stream())
    prefetch(0)
    for i in range(3):
        e2e_step(i, False)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(3, 3 + args.steps):
        e2e_step(i, i == 2 + args.steps)
    loss_ev[(2 + args.steps) & 1].synchronize()        # the last step's loss is on the host before the clock stops
    e2e_last_loss = float(host_loss[(2 + args.steps) & 1])
    e3.record()
    barrier()
    t2 = torch.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_val = world * B * args.steps / (t2.item() * 1e-3)

    # ---------------- roofline of the dominant kernel: fused noisy conv forward of conv2, timed live
    # with CUDA events on the launch stream, same tensors as the step, inputs cycled (> L2 between reps).
    peaks, peak_kind = load_peaks()
    roof = None
    if rank == 0:
        from noisynet_b200._lib import NOISE_EXTERNAL
        xs = [torch.rand(B, 65, 14, 14, device=dev).mul_(15).round_().div_(3.0) for _ in range(8)]   # codes * 5/15
        w_raw = model.conv2.weight.detach()
        w_eff = ops.quantize_fwd(w_raw, 4, -1.0, 1.0, 0.0) if args.variant == "q4" else w_raw
        scale = ops.tensor_stats(xs[0])[0:1]
        reps = 20
        # CUDA events bracket the main tcgen05 kernel only, on its launch stream (nn_debug_main_kernel_ms); the
        # operand packs that precede it in this standalone call are not part of the engine's step.
        call = lambda i: ops.noisy_conv_fwd(xs[i % 8], w_eff, w_raw, None, 1, 0, noise_mode=NOISE_EXTERNAL, current=1.0,
                                            scale_dev=scale, precision=precision, want_y=False,
                                            a_code_scale=(5.0 / 15.0 if args.variant == "q4" else 0.0),
                                            w_code_scale=(1.0 / 15.0 if args.variant == "q4" else 0.0))
        for i in range(3):
            call(i)
        torch.cuda.synchronize()
        if precision == "fp32":
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for i, (a0, a1) in enumerate(evs):
                a0.record(); call(i); a1.record()
            torch.cuda.synchronize()
            k_ms = sum(a0.elapsed_time(a1) for a0, a1 in evs) / reps
        else:
            lib.nn_debug_main_kernel_ms(1)
            tms = []
            for i in range(reps):
                call(i)
                tms.append(lib.nn_debug_main_kernel_ms(-1))
            lib.nn_debug_main_kernel_ms(0)
            k_ms = sum(tms) / len(tms)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r2_conv2_fwd_traffic.json")) as f:
                tj = json.load(f)
                traffic = {"dram_bytes_per_launch": tj["dram_bytes_per_launch"], "l2_to_sm_bytes_per_launch": tj["l2_to_sm_bytes"],
                           "unit": "B", "from": tj["source"]} if (B == 512 and precision == "bf16") else None
        except Exception:
            traffic = None
        flops = FLOP_FWD["conv2"] * B
        achieved = flops / (k_ms * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops", 1590.0)
        roof = {"kernel": "k_conv_tma<1>: fused noisy conv forward of conv2 (M=%d, N=2x120, K=1625; persistent CTA pairs, "
                          "TMA-im2col operands), precision=%s" % (B * 100, precision),
                "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_kind": peak_kind + " (burst, kernel timed alone)", "kernel_ms": k_ms,
                "flop_per_launch": flops, "traffic": traffic,
                "step_tensor_frac": (world * B * args.steps / (ms * 1e-3)) * FLOP_STEP / world / (peaks.get("bf16_tflops_sustained", 1400.0) * 1e12)}

    if rank != 0:
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = oracle_arm(128, args.variant, 0, 2, seconds=args.cpu_baseline_seconds)
        cpu = {"value": r["img_s"], "unit": "img/s", "cores": r["cores"], "kind": "port",
               "sample": "%d steps of batch 128 in %.1f s (oracle port of the reference training step, torch CPU fp32)" % (r["steps"], r["seconds"])}
    other = None
    if world == 1 and engine is not None and not args.no_second_variant:
        # SURVEY 8d "report both": the other operand variant (q4 <-> README flags q_a = q_w = 0) through the same engine,
        # device-resident, CUDA graph, same K steps
        try:
            other = time_second_variant(args, dev, precision, "fp" if args.variant == "q4" else "q4")
        except Exception as e:  # noqa: BLE001
            other = {"unavailable": str(e)[:300]}
    lib_base = None
    if world == 1 and not args.no_library_baseline:
        try:
            r = torch_gpu_arm(B, args.variant, args.steps, args.warmup, dev)
            lib_base = {"value": r["img_s"], "unit": "img/s", "ms_per_step": r["ms_per_step"], "kind": "pytorch-eager",
                        "sample": "%d steps of batch %d on the same GPU: the reference step (oracle port) in PyTorch eager -- "
                                  "cuDNN / cuBLAS / ATen Philox, fp32" % (args.steps, B)}
        except Exception as e:  # noqa: BLE001
            lib_base = {"unavailable": str(e)[:200]}
    h2d = B * 3 * 32 * 32 * 4 + B * 8
    line = {
        "metric": "NoisyNet CIFAR-10 4-bit training images/sec", "value": value, "unit": "img/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[precision],
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e_val, "unit": "img/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "readback": "loss of every step copied to pinned host memory and read by the host one step later (last one before the clock stops)",
                "last_loss": e2e_last_loss},
        "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
        "cuda_graph": graph is not None, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "library_baseline": lib_base, "second_variant": other,
        "final_loss": final_loss,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_gpu":
        run_torch_gpu(args)
    else:
        run_b200(args)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            # symmetric-memory handles (dp.SymmGradAllReduce) can block the process-group teardown: every rank has printed
            # and synchronised by now, so leave through _exit after a last barrier
            dist.barrier()
            torch.cuda.synchronize()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
    except Exception:
        pass


if __name__ == "__main__":
    main()
