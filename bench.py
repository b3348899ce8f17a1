#!/usr/bin/env python
"""bench.py -- grasps/sec of the PointNet grasp-quality hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config train|infer|tower] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default (`--config train`): one "step" = one pass of the hot path over one batch of synthetic grasp clouds: forward
(PointNetCls, train mode) + nll_loss + backward + the NCCL gradient all-reduce (N>1) + Adam step, exactly the body of
main_1v.py:72-76, at BASELINE config 2: B=512 clouds/GPU x N=1024 points, k=2.  Weak scaling: every rank processes
its own batch.  Other BASELINE configs: `--classes 3` (config 3), `--batch 128 --points 2048` under torchrun x8
(config 4), `--config infer` (config 5: eval forward, B=4096 x N=750), `--config tower` (north_star's tower-only
shape: 1024 clouds x 1024 points through pgpd_tower_forward).

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is produced.

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32 / float64): the
log-probs (infer), the pooled features (tower), or the loss plus every parameter and BatchNorm buffer after the update
(train).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "grasps/s"
CPU_SAMPLE_B = 128        # clouds per step of the CPU arms (a bounded sample of the 512-cloud workload)
DUMP_BUDGET = 64 << 20    # bytes of --dump-outputs in all


def dump_outputs(out_dir, arrays):
    """Write {name: host tensor} as out_dir/<name>.npy.  An array larger than its even share of DUMP_BUDGET is cut to a
    fixed, seeded sample of its rows (sorted, so the order matches the full output), so the dump stays comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BUDGET // max(1, len(arrays))
    for name, t in arrays.items():
        a = t.numpy()
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64).reshape(a.shape or (1,))
        if a.nbytes > share:
            rows = max(1, share // max(1, a[0].nbytes))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], size=rows, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def fwd_flops_per_grasp(N, k):
    """Dense algorithmic flops of one forward (BASELINE.md section 2)."""
    return N * 557842 + 2626048 + 512 * k


def host_threads():
    """Threads for the CPU arms: the physical cores of the box, whatever OMP_NUM_THREADS says (torchrun exports
    OMP_NUM_THREADS=1 to its children, which would time one core)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    try:
        return max(1, len(os.sched_getaffinity(0)) // 2)
    except Exception:
        return max(1, (os.cpu_count() or 2) // 2)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()          # the exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ baseline legs
def port_train_arm(device, B, N, k, steps, warmup, max_seconds=None, tf32=False):
    """The oracle's torch port (the reference's op sequence, oracle/pointnet_torch_port.py) as a training step:
    forward + nll_loss + backward + Adam.  device "cpu": ATen/MKLDNN on all host cores (the `cpu_baseline` /
    `--impl reference` leg).  device cuda: eager PyTorch on the same B200 (`gpu_eager_baseline`, SURVEY.md 8d)."""
    from oracle import pointnet_torch_port as PT
    from pointnetgpd_b200 import synth as W
    import torch.nn.functional as F
    dev = torch.device(device)
    st = W.make_state(0, k=k)
    sd = {kk: v.to(dev) for kk, v in PT.to_torch_state(st, torch.float32).items()}
    for kk, v in sd.items():
        if v.is_floating_point() and not kk.endswith(("running_mean", "running_var")):
            v.requires_grad_(True)
    params = [v for v in sd.values() if v.requires_grad]
    opt = torch.optim.Adam(params, lr=0.005, fused=True) if dev.type == "cuda" else torch.optim.Adam(params, lr=0.005)
    x = torch.tensor(W.make_clouds(1234, B, N, "box")).to(dev)
    y = torch.tensor(W.make_labels(4321, B, k)).to(dev)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32

    def one():
        opt.zero_grad(set_to_none=True)
        logp, _ = PT.pointnetcls_forward(sd, x, training=True)
        loss = F.nll_loss(logp, y)
        loss.backward()
        opt.step()
        return loss.detach()

    try:
        for _ in range(warmup):
            one()
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)
        times = []
        t_all = time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter()
            one()
            if dev.type == "cuda":
                torch.cuda.synchronize(dev)
            times.append(time.perf_counter() - t0)
            if max_seconds is not None and time.perf_counter() - t_all > max_seconds:
                break
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    ms = 1e3 * sum(times) / len(times)
    return {"value": B / (ms / 1e3), "ms_per_step": ms, "steps_done": len(times), "cores": torch.get_num_threads()}


def port_infer_arm(device, B, N, k, steps, warmup, tf32=False):
    from oracle import pointnet_torch_port as PT
    from pointnetgpd_b200 import synth as W
    dev = torch.device(device)
    sd = {kk: v.to(dev) for kk, v in PT.to_torch_state(W.make_state(0, k=k, style="wild"), torch.float32).items()}
    x = torch.tensor(W.make_clouds(5, B, N, "dup")).to(dev)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        with torch.no_grad():
            for _ in range(warmup):
                PT.pointnetcls_forward(sd, x, training=False)
            if dev.type == "cuda":
                torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for _ in range(steps):
                PT.pointnetcls_forward(sd, x, training=False)
            if dev.type == "cuda":
                torch.cuda.synchronize(dev)
            ms = 1e3 * (time.perf_counter() - t0) / steps
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    return {"value": B / (ms / 1e3), "ms_per_step": ms, "steps_done": steps, "cores": torch.get_num_threads()}


def cpu_sample_note(args):
    if args.config == "train":
        return ("CPU arms (cpu_baseline, --impl reference) time the oracle torch port on %d-cloud batches of %d points per "
                "step (a bounded sample of the %d-cloud batch; throughput per cloud is what is compared)" % (CPU_SAMPLE_B, args.points, args.batch))
    return "CPU arms time the oracle torch port (eval forward) on %d-cloud batches of %d points" % (CPU_SAMPLE_B, args.points)


def make_config(args, world):
    B, N, k = args.batch, args.points, args.classes
    if args.config == "train":
        workload = "PointNetCls k=%d train step (fwd+nll+bwd+allreduce+Adam), B=%d clouds/GPU x N=%d pts" % (k, B, N)
    elif args.config == "infer":
        workload = "PointNetCls k=%d eval forward (batched candidate scoring, main_test.py:59-69), B=%d clouds/GPU x N=%d pts" % (k, B, N)
    else:
        workload = "trunk tower 3->64->128->1024 + max-pool, eval forward only (pgpd_tower_forward), B=%d clouds x N=%d pts" % (B, N)
    return {"workload": workload, "global_batch": B * world, "points": N, "classes": k, "parallelism": "dp%d" % world,
            "l2": "per-step working set (saved activations, >= 0.4 GB) >> 126 MB L2; 8 rotating input batches",
            "cpu_sample": cpu_sample_note(args)}


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="train", choices=["train", "infer", "tower"])
    ap.add_argument("--batch", type=int, default=None, help="clouds per GPU (train: 512 = BASELINE config 2; infer: 4096; tower: 1024)")
    ap.add_argument("--points", type=int, default=None, help="points per cloud (train/tower: 1024; infer: 750)")
    ap.add_argument("--classes", type=int, default=2)
    ap.add_argument("--simt", action="store_true", help="force the fp32 CUDA-core kernels")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU / eager-GPU baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.batch is None:
        args.batch = {"train": 512, "infer": 4096, "tower": 1024}[args.config]
    if args.points is None:
        args.points = {"train": 1024, "infer": 750, "tower": 1024}[args.config]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    B, N, k = args.batch, args.points, args.classes
    config = make_config(args, world)
    metric = {"train": "grasps_per_sec_fwd_bwd", "infer": "grasps_per_sec_inference", "tower": "grasps_per_sec_tower_fwd"}[args.config]

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        torch.set_num_threads(host_threads())
        steps, warm = args.steps, max(1, args.warmup)
        if args.config == "train":
            r = port_train_arm("cpu", CPU_SAMPLE_B, N, k, steps, warm)
            what = "fwd+nll+bwd+Adam"
        else:
            r = port_infer_arm("cpu", CPU_SAMPLE_B, N, k, steps, min(warm, 2))
            what = "eval forward"
        line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": r["steps_done"], "warmup": warm, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                 "sample": "oracle torch port (reference op sequence on ATen CPU), %d-cloud batches of %d points, "
                                           "%s per step, %d host threads" % (CPU_SAMPLE_B, N, what, r["cores"])},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch.distributed as dist
    from pointnetgpd_b200 import _abi as A
    from pointnetgpd_b200 import synth as W
    from pointnetgpd_b200.ddp import FlatGradAllReduce
    from pointnetgpd_b200.model.pointnet import PointNetCls
    import torch.nn.functional as F

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (the fused path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = A.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    NBUF = 8
    style = "default" if args.config == "train" else "wild"
    st = W.make_state(0, k=k, style=style)
    model = PointNetCls(num_points=N, input_chann=3, k=k)
    model.load_state_dict({kk: torch.tensor(v) for kk, v in st.items()})
    model = model.to(dev)
    kind = "box" if args.config == "train" else "dup"
    xs_host = [torch.tensor(W.make_clouds(1234 + rank * 100 + i, B, N, kind)).pin_memory() for i in range(NBUF)]
    ys_host = [torch.tensor(W.make_labels(4321 + rank * 100 + i, B, k)).pin_memory() for i in range(NBUF)]
    xs_dev = [t.to(dev) for t in xs_host]
    ys_dev = [t.to(dev) for t in ys_host]
    use_graph = not args.no_graph and not args.simt
    graphed = None
    config_graph = "one graph"
    lib.pgpd_profile_enable(0)
    launches_fn = None
    h2d = B * 3 * N * 4
    d2h = 4

    if args.config == "train":
        model.train()
        opt = torch.optim.Adam(model.parameters(), lr=0.005, fused=True, capturable=True)
        sync = FlatGradAllReduce(list(model.parameters()), world, overlap=os.environ.get("PGPD_DDP_OVERLAP", "1") != "0").install()   # all-reduce issued from inside the backward
        flags_extra = A.F_SIMT if args.simt else 0
        if flags_extra:
            from pointnetgpd_b200.functional import run_module
            fwd = lambda xx: run_module(model, A.PGPD_CLS, xx, k=k, flags_extra=flags_extra)
        else:
            fwd = model

        def eager_step(x, y):
            opt.zero_grad(set_to_none=True)
            logp, _ = fwd(x)
            loss = F.nll_loss(logp, y)
            loss.backward()
            sync.all_reduce()
            opt.step()
            return loss.detach()

        # The step is captured once into a CUDA graph and replayed (pointnetgpd_b200.graph.GraphedTrainStep); the dominant
        # kernel's event pair is recorded INSIDE the graph (external event nodes), so its duration is still measured live.
        if use_graph:
            from pointnetgpd_b200.graph import GraphedTrainStep
            for capture_sync in ((True, False) if world > 1 else (True,)):
                try:
                    graphed = GraphedTrainStep(model, opt, xs_dev[0], ys_dev[0], grad_sync=sync if world > 1 else None, warmup=3,
                                               before_capture=lambda: lib.pgpd_profile_enable(2), capture_sync=capture_sync)
                    config_graph = "one graph incl. NCCL" if (world > 1 and capture_sync) else ("two graphs + eager NCCL" if world > 1 else "one graph")
                    break
                except Exception as e:           # e.g. a collective that cannot be captured: next scheme, finally eager launches
                    sys.stderr.write("CUDA-graph capture (capture_sync=%s) failed (%s: %s)\n" % (capture_sync, type(e).__name__, e))
                    graphed = None
                    lib.pgpd_profile_enable(0)
                    torch.cuda.synchronize(dev)
        dev_step = (lambda i: graphed.step(xs_dev[i % NBUF], ys_dev[i % NBUF])) if graphed is not None else \
                   (lambda i: eager_step(xs_dev[i % NBUF], ys_dev[i % NBUF]))

        staged = graphed.staged_input() if graphed is not None else None

        def e2e_step(i):
            # every step's batch travels pinned host -> device inside the timed region; the copy of batch i+1 is issued on a side
            # stream while step i runs (pointnetgpd_b200.staging), as a DataLoader with pinned memory does for an eager loop
            if graphed is not None:
                if i == 0:
                    staged.prefetch((xs_host[0], ys_host[0]))
                loss = graphed.step_staged()
                if i + 1 < args.steps:
                    staged.prefetch((xs_host[(i + 1) % NBUF], ys_host[(i + 1) % NBUF]))
            else:
                loss = eager_step(xs_host[i % NBUF].to(dev, non_blocking=True), ys_host[i % NBUF].to(dev, non_blocking=True))
            return loss.item()                                              # D2H read of the step's result
        launches_fn = lambda: eager_step(xs_dev[0], ys_dev[0])
        h2d += B * 8
    elif args.config == "infer":
        model.eval()
        sx = torch.empty_like(xs_dev[0])
        out_host = torch.empty((B, k), dtype=torch.float32).pin_memory()
        with torch.no_grad():
            for _ in range(2):
                logp, _ = model(sx)
            torch.cuda.synchronize(dev)
            if use_graph:
                lib.pgpd_profile_enable(2)
                graphed = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graphed):
                    logp, _ = model(sx)

        def fwd_static(x):
            sx.copy_(x, non_blocking=True)
            if graphed is not None:
                graphed.replay()
                return logp
            with torch.no_grad():
                return model(sx)[0]
        dev_step = lambda i: fwd_static(xs_dev[i % NBUF])

        from pointnetgpd_b200.staging import StagedInput
        staged = StagedInput([sx])

        def e2e_step(i):
            if i == 0:
                staged.prefetch((xs_host[0],))
            staged.commit()                                                  # batch i: staged copy -> static input
            if graphed is not None:
                graphed.replay()
                res = logp
            else:
                with torch.no_grad():
                    res = model(sx)[0]
            if i + 1 < args.steps:
                staged.prefetch((xs_host[(i + 1) % NBUF],))                  # batch i+1 travels while batch i is scored
            out_host.copy_(res, non_blocking=True)                           # scores back to the host: what a caller consumes
            torch.cuda.current_stream(dev).synchronize()
            return out_host
        def _one():
            with torch.no_grad():
                model(sx)
        launches_fn = _one
        d2h = B * k * 4
    else:   # tower-only forward through the C ABI (north_star: "fused 64->128->1024 MLP at batch 1024x1024 pts")
        ptrs = {kk: v for kk, v in model.state_dict().items()}
        tw = A.Tower()
        A.fill_tower(tw, A.TOWER_TRUNK, lambda key: ptrs[key].data_ptr())
        flags = A.F_SIMT if args.simt else 0
        nbytes = lib.pgpd_tower_workspace_bytes(B, N, flags)
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        wsp = ws.data_ptr() + ((-ws.data_ptr()) % 256)
        pooled = torch.empty((B, 1024), dtype=torch.float32, device=dev)
        sx = torch.empty_like(xs_dev[0])
        pooled_host = torch.empty((B, 1024), dtype=torch.float32).pin_memory()

        def tower_call():
            rc = lib.pgpd_tower_forward(ctypes.byref(tw), sx.data_ptr(), None, B, N, 0, flags, pooled.data_ptr(), wsp, nbytes,
                                        torch.cuda.current_stream(dev).cuda_stream)
            A.check(lib, rc)
        for _ in range(2):
            tower_call()
        torch.cuda.synchronize(dev)
        if use_graph:
            lib.pgpd_profile_enable(2)
            graphed = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphed):
                tower_call()

        def fwd_static(x):
            sx.copy_(x, non_blocking=True)
            if graphed is not None:
                graphed.replay()
            else:
                tower_call()
            return pooled
        dev_step = lambda i: fwd_static(xs_dev[i % NBUF])

        from pointnetgpd_b200.staging import StagedInput
        staged = StagedInput([sx])

        def e2e_step(i):
            if i == 0:
                staged.prefetch((xs_host[0],))
            staged.commit()
            if graphed is not None:
                graphed.replay()
            else:
                tower_call()
            if i + 1 < args.steps:
                staged.prefetch((xs_host[(i + 1) % NBUF],))
            pooled_host.copy_(pooled, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            return pooled_host
        launches_fn = tower_call
        d2h = B * 1024 * 4

    for i in range(args.warmup):
        dev_step(i)
    barrier()

    # ---- device-timed region: inputs resident in HBM -------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    if graphed is None:
        lib.pgpd_profile_enable(1)
    n0 = lib.pgpd_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = dev_step(i)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    dumped = None
    if args.dump_outputs and rank == 0:
        # snapshot before the end-to-end region below runs further steps on the same model and buffers
        if args.config == "train":
            dumped = {"loss": last.detach().float().cpu()}
            dumped.update({"param." + n: p.detach().cpu().clone() for n, p in model.named_parameters()})
            dumped.update({"buffer." + n: b.detach().cpu().clone() for n, b in model.named_buffers()})
        else:
            dumped = {"logp" if args.config == "infer" else "pooled": last.detach().cpu().clone()}
    launches = int(lib.pgpd_launch_count() - n0)
    nl, tot = ctypes.c_int(0), ctypes.c_float(0.0)
    lib.pgpd_profile_read(ctypes.byref(nl), ctypes.byref(tot))      # graph mode: the event nodes of the LAST replayed step
    lib.pgpd_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None

    # ---- end-to-end region: pinned host inputs -> H2D -> step -> D2H of the result ------------------
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    barrier()
    e2e_ms_total = (time.perf_counter() - t0) * 1e3

    if graphed is not None:
        # replays launch the captured kernels without passing through the library's host code: count them from one eager step
        # (the backward runs on autograd's worker thread; the counter is process-wide)
        n1 = lib.pgpd_launch_count()
        launches_fn()
        torch.cuda.synchronize(dev)
        launches = int(lib.pgpd_launch_count() - n1) * args.steps

    t = torch.tensor([ms_total, e2e_ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms_total = float(t[0]), float(t[1])
    ms_per_step = ms_total / args.steps
    value = B * world / (ms_per_step / 1e3)
    e2e_value = B * world / (e2e_ms_total / args.steps / 1e3)

    if rank == 0:
        peaks, peak_src = load_peaks()
        M = B * N
        fused = args.config != "train" and not args.simt    # eval forward: ONE kernel per tower (layers 1-3 + max-pool, tc_fused.cuh)
        k3_flops = 2.0 * (3 * 64 + 64 * 128 + 128 * 1024) * M if fused else 2.0 * 128 * 1024 * M     # algorithmic flops per launch
        k3_ms = (tot.value / nl.value) if nl.value else None
        # a 20-step timed region lasts ~50 ms: the like-for-like denominator is the burst figure (a kernel timed inside a
        # seconds-long step would use bf16_tflops_sustained)
        peak = float(peaks.get("bf16_tflops", peaks.get("bf16_tflops_sustained")))
        traffic, traffic_src = None, None   # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
        for name in ("r2_l3_traffic.json", "r1_l3_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath) and (B, N) == (512, 1024) and not args.simt:
                with open(tpath) as f:
                    traffic = json.load(f).get("dram_bytes_per_launch")
                traffic_src = "profiles/" + name
                break
        ach = (k3_flops / (k3_ms * 1e-3) / 1e12) if k3_ms else None
        roofline = {"bound": "tensor", "kernel": ("fused tower 3->64->128->1024 + max-pool (eval), one launch per tower forward" if fused else
                                                  "tower layer-3 GEMM (128->1024) + max-pool epilogue, one launch per tower forward"),
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if ach else None,
                    "peak_source": peak_src + " bf16_tflops (burst: the timed region is tens of ms)",
                    "frac_vs_sustained_peak": (ach / float(peaks["bf16_tflops_sustained"])) if ach and "bf16_tflops_sustained" in peaks else None,
                    "kernel_ms": k3_ms, "launches_timed": nl.value, "traffic": traffic, "traffic_source": traffic_src,
                    "impl": "tcgen05" if (lib.pgpd_has_tensor_core_path() and not args.simt) else "cuda-core fp32",
                    "numerics": "fp32-grade 3-pass fp16 operand split: issued tensor work is 3x the algorithmic flops counted here",
                    "timing": ("event pairs recorded as nodes of the replayed CUDA graph (last timed step)" if graphed is not None
                               else "event pairs around every launch in the timed region")}
        if args.config == "train":
            roofline["step_algorithmic_tflops"] = 3.0 * fwd_flops_per_grasp(N, k) * B / (ms_per_step * 1e-3) / 1e12
        elif args.config == "infer":
            roofline["step_algorithmic_tflops"] = fwd_flops_per_grasp(N, k) * B / (ms_per_step * 1e-3) / 1e12
        else:
            tf = 2.0 * (3 * 64 + 64 * 128 + 128 * 1024) * M
            roofline["tower_algorithmic_tflops"] = tf / (ms_per_step * 1e-3) / 1e12
            roofline["tower_frac_of_peak"] = roofline["tower_algorithmic_tflops"] / peak
        line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config, "cuda_graph": (config_graph if graphed is not None else False),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms_total / args.steps,
                        "input_staging": "every step's batch is copied pinned host -> device inside the timed region; the copy of batch i+1 "
                                         "runs on a side stream while step i computes (pointnetgpd_b200.staging); result read back every step"},
                "gpu_launches": launches, "gpu_launches_per_step": launches // max(1, args.steps), "clocks": clocks, "roofline": roofline}
        if world == 1 and not args.no_cpu_baseline:
            graphed = None
            torch.cuda.empty_cache()
            torch.set_num_threads(host_threads())
            if args.config == "train":
                r = port_train_arm("cpu", CPU_SAMPLE_B, N, k, steps=3, warmup=1, max_seconds=25.0)
                line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                        "sample": "oracle torch port on the host CPU: %d timed fwd+nll+bwd+Adam steps on a %d-cloud x %d-point "
                                                  "batch (1 warm-up), %d threads" % (r["steps_done"], CPU_SAMPLE_B, N, r["cores"])}
                # BASELINE.md section 3 case (a) / BASELINE config 1: main_1v.py's CPU shape, B=32 x 750 points
                r1 = port_train_arm("cpu", 32, 750, 2, steps=5, warmup=2, max_seconds=10.0)
                line["cpu_baseline_config1"] = {"value": r1["value"], "unit": UNIT, "cores": r1["cores"], "kind": "port", "ms_per_step": r1["ms_per_step"],
                                                "sample": "BASELINE config 1 (main_1v.py, B=32 x N=750, k=2, fwd+nll+bwd+Adam): %d timed steps" % r1["steps_done"]}
                eg = {}
                for tf32 in (False, True):
                    try:
                        r2 = port_train_arm(str(dev), B, N, k, steps=3, warmup=2, tf32=tf32)
                        eg["tf32" if tf32 else "fp32"] = {"value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"]}
                    except Exception as e:          # e.g. out of memory at unusual shapes: a baseline leg must not kill the line
                        eg["tf32" if tf32 else "fp32"] = {"error": "%s: %s" % (type(e).__name__, e)}
                    torch.cuda.empty_cache()
                eg["what"] = ("eager PyTorch (oracle torch port = the reference's op sequence, cuDNN/cuBLAS) on the same GPU, same "
                              "B=%d x N=%d train step; tf32 fails the 1e-3 parity bar (SURVEY.md 7.2C)" % (B, N))
                line["gpu_eager_baseline"] = eg
            else:
                r = port_infer_arm("cpu", CPU_SAMPLE_B, N, k, steps=3, warmup=1)
                line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                        "sample": "oracle torch port on the host CPU: eval forward of %d clouds x %d points, 3 timed runs" % (CPU_SAMPLE_B, N)}
                if args.config == "infer":
                    r2 = port_infer_arm(str(dev), B, N, k, steps=3, warmup=1, tf32=False)
                    line["gpu_eager_baseline"] = {"fp32": {"value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"]},
                                                  "what": "eager PyTorch (oracle torch port) eval forward on the same GPU, fp32"}
        print(json.dumps(line), flush=True)
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        # the line is out; never let communicator teardown hang the job
        threading.Timer(30.0, lambda: os._exit(0)).start()
        try:
            torch.cuda.synchronize(dev)
            dist.barrier()
            dist.destroy_process_group()
        finally:
            sys.stdout.flush()
            os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
