#!/usr/bin/env python
"""Headline benchmark: 3D-ViT stacking-ensemble path, volumes/s on N B200s.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
    python bench.py --impl reference ...       # the reference's CPU path (oracle port) on the host cores

ONE JSON line on stdout (rank 0).  The headline (`value`, `e2e`, `roofline`, `cpu_baseline`) is BASELINE.json
config 2: conf-5 inference, `model(x)` in eval / no_grad (train_baseline_cv.py:79), batch 1024 per GPU, batch
sharded over the ranks (no data-path collective).  The same run then times short legs of the two north-star
workloads that DO exchange data, reported under `workloads`:

    conf18_train     conf-18 data-parallel training step (train_baseline_cv.py:163-182): forward + backward replayed
                     from a CUDA graph, ONE NCCL all-reduce of the flat gradient arena, fused SGD step
    ensemble_infer   confs 5+9+11 + meta-classifier (models/modeling.py:353-356): (member, batch-slice) work list cut
                     into equal-FLOP chunks, one all-gather of the member logits, meta-head on every rank
    conf5_infer_tf32 the headline workload in the TF32 (1e-3 logit tolerance) mode
    cv_sweep         a bounded sample of the 18 x 5 train_baseline_cv.py sweep as independent jobs packed on the GPUs
                     (replicas only), jobs/s

`value` = volumes/s with the batch resident in HBM; `e2e` = the same through the public module call with pinned HOST
input, H2D copy and D2H read of the result inside the timed region (`e2e.variants.u8`: volumes cross PCIe as the
8-bit images they are, N2 input path).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "ensemble volumes/sec (inference, fwd+bwd train) at 1/2/4/8 B200 vs CPU ref"
UNIT = "volumes/s"
VOL_BYTES = 327680          # one fp32 volume (1,128,128,5)

WORKLOADS = {
    "conf5_infer": dict(name="conf5 (d2048 L6 8x32 H256) inference, model(x) eval/no_grad", confs=[5], train=False, batch=1024),
    "conf18_train": dict(name="conf18 (d3072 L8 16x16 H256) training fwd+bwd+SGD step", confs=[18], train=True, batch=256),
    "ensemble_infer": dict(name="ensemble conf 5+9+11 + meta-classifier inference", confs=[5, 9, 11], train=False, batch=512),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="conf5_infer", choices=list(WORKLOADS))
    ap.add_argument("--legs", default="auto", help="extra workloads timed after the headline: 'auto' (the other two + the "
                    "TF32 mode when the headline is conf5_infer), 'none', or a comma list")
    ap.add_argument("--leg-steps", type=int, default=8, help="timed steps of every extra leg")
    ap.add_argument("--batch", type=int, default=0, help="volumes per GPU per step (0 = workload default)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--vis", type=int, default=1, help="materialise attention probabilities (reference default vis=True)")
    ap.add_argument("--cpu-sample", type=int, default=64, help="volumes per step of the in-run cpu_baseline leg")
    ap.add_argument("--cpu-budget", type=float, default=240.0, help="seconds the --impl reference arm may run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graphs", type=int, default=1, help="replay the step from a CUDA graph (vit3d_b200.graphs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline's last timed step returned as DIR/<name>.npy "
                         "(float32; arrays over their share of 64 MB as a fixed, seeded sample of their elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [v.strip() for v in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local_rank):
    """Best effort: run this rank (and first-touch its pinned staging buffers) on the CPU socket its GPU hangs off,
    so that 8 ranks do not all stream their H2D copies out of one socket's memory.  Returns the number of CPUs
    the rank was bound to, or None when the topology is not visible / nothing changed."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        if not out:
            return None
        bdf = out.lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:      # 00000000:1b:00.0 -> 0000:1b:00.0
            bdf = bdf[4:]
        path = f"/sys/bus/pci/devices/{bdf}/local_cpulist"
        if not os.path.exists(path):
            return None
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        return None
    return None


# ----------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_arm(cfgs, train, steps, warmup, sample, budget_s=None):
    """Times the reference's algorithm on the host cores: the oracle's functional restatement of
    models/modeling.py (torch CPU fp32, all threads).  Stops early when `budget_s` is used up (returns the steps run)."""
    import torch
    from oracle import vit3d_oracle as O
    torch.set_num_threads(os.cpu_count())
    sds = [O.init_state_dict(c, seed=42 + j) for j, c in enumerate(cfgs)]
    x = O.synth_volumes(sample, seed=42)
    y = O.synth_labels(sample)
    w = O.sklearn_pos_weight(y)
    ens_sd = O.ensemble_state_dict(sds) if len(cfgs) > 1 else None

    def step():
        if train:
            O.vit_loss_and_grads(sds[0], cfgs[0], x, y, w)
        elif ens_sd is not None:
            with torch.no_grad():
                O.ensemble_forward(ens_sd, cfgs, x)
        else:
            with torch.no_grad():
                O.vit_forward(sds[0], cfgs[0], x)

    t_start = time.perf_counter()
    warm_done = 0
    for _ in range(warmup):
        step()
        warm_done += 1
        if budget_s is not None and time.perf_counter() - t_start > 0.3 * budget_s:
            break
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.perf_counter() - t_start > budget_s:
            break
    dt = time.perf_counter() - t0
    return sample * done / dt, dt / done * 1e3, done, warm_done


def workload_config(wl, B, world, vis):
    """`config` of the JSON line: identical for the GPU arm and the reference arm of the same workload."""
    units = B if len(wl["confs"]) > 1 else world * B
    if wl["train"]:
        par = f"dp{world}: batch sharded over the ranks, gradients all-reduced (mean) before the SGD step"
    elif len(wl["confs"]) > 1:
        par = f"{world} ranks: (member, batch-slice) work list cut batch-major, members concurrent on a rank, all-gather of member logits, meta-head on every rank"
    else:
        par = f"dp{world} (independent volumes, no data-path collective)"
    return {"workload": wl["name"], "batch_per_gpu": B, "global_batch": units, "vis": bool(vis),
            "l2": "inputs larger than L2 (batch of fp32 volumes = %.0f MB)" % (B * VOL_BYTES / 1e6), "parallelism": par}


# ----------------------------------------------------------------------------- GPU legs
class Ctx:
    pass


def time_region(ctx, fn, steps, warm, counter=None):
    """`warm` untimed calls, then `steps` calls between CUDA events, barrier + synchronize on both sides, max over
    ranks.  Returns (ms, launches of this library inside the timed region)."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    if ctx.dist is not None:
        ctx.dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = counter() if counter else 0
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    n1 = counter() if counter else 0
    ms = e0.elapsed_time(e1)
    if ctx.dist is not None:
        t = torch.tensor([ms], device=ctx.dev)
        ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
        ms = float(t)
        ctx.dist.barrier()
    return ms, n1 - n0


def run_leg(ctx, args, key, steps, warmup, precision, with_u8=True, dump_dir=None):
    """Builds one workload, times its device-resident loop and its end-to-end loop.  Returns a dict.
    `dump_dir`: write the outputs of the last timed device-resident step there (dump_outputs)."""
    import torch
    import vit3d_b200
    from oracle import vit3d_oracle as O          # test infrastructure: synthetic inputs / seeded weights only
    from vit3d_b200.dist import batch_pos_weight
    from vit3d_b200.models.modeling import TransformerEnsemble, VisionTransformer
    wl = WORKLOADS[key]
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    L = vit3d_b200._lib.lib()
    B = args.batch if (args.batch and key == args.workload) else wl["batch"]
    cfgs = [vit3d_b200.north_star_config(c) for c in wl["confs"]]
    train = wl["train"]
    ens = len(cfgs) > 1
    flops_per_vol = sum(O.fwd_flops_per_volume(c) for c in cfgs) * (3.0 if train else 1.0)
    members = []
    for j, c in enumerate(cfgs):
        m = VisionTransformer(c, 128, zero_head=True, num_classes=1, vis=bool(args.vis), precision=precision)
        m.load_state_dict(O.init_state_dict(c, seed=42 + j))
        members.append(m)
    model = members[0] if not ens else TransformerEnsemble(*members, in_features=1)
    model.to(dev)
    model.train(train)
    x_host = O.synth_volumes(B, seed=42 + (rank if not ens else 0)).pin_memory()
    y_host = O.synth_labels(B).pin_memory()
    x_dev = x_host.to(dev)
    y_dev = y_host.to(dev)
    graphed = sharded = opt = None
    collective = None
    bytes_coll = 0
    if train:
        # the reference's optimizer (train_baseline_cv.py:111-114) as one fused launch over a flat arena
        from vit3d_b200.graphs import GraphedTrainStep
        from vit3d_b200.optim import FusedSGD
        opt = FusedSGD(model.parameters(), lr=1e-4, momentum=0.9, weight_decay=1e-2)
        graphed = GraphedTrainStep(model, opt, warmup=2, data_parallel=world > 1)
        if world > 1:
            collective = "all_reduce(flat gradient arena, fp32) after the backward graph, before the fused SGD launch"
            bytes_coll = opt.arena.numel * 4
    elif ens:
        from vit3d_b200.dist import ShardedEnsemble
        sharded = ShardedEnsemble(model, costs=[O.fwd_flops_per_volume(c) for c in cfgs])
        if world > 1:
            collective = "all_gather_into_tensor(member logits of this rank's (member, batch-slice) chunk, fp32)"
            bytes_coll = sharded.gather_bytes(B)
    elif args.graphs:
        from vit3d_b200.graphs import GraphedInference
        graphed = GraphedInference(model)
        x_dev = graphed.input_like(x_dev)       # the resident batch lives in the graph's own input buffer

    def pos_weight():
        # the scripts compute the class weight of every batch on the host from its labels (sklearn,
        # train_baseline_cv.py:168-169); every rank holds the same synthetic labels, so local == global
        return batch_pos_weight(y_host)

    def step_out(x, y):
        """One step; returns what the caller of the timed path receives."""
        if train:
            return graphed(x, y, pos_weight())
        if sharded is not None:
            return sharded(x)
        if graphed is not None:
            return graphed(x)
        with torch.no_grad():
            return model(x)

    def step_dev(x, y):
        out = step_out(x, y)
        return out[0] if isinstance(out, tuple) else out

    def counter():
        n = L.vit3d_launch_count()
        for g in ([graphed] if graphed is not None else []) + (sharded.graph_runners() if sharded is not None else []):
            n += g.replays * g.launches_per_replay
        return n

    last = [None]

    def timed_step():
        last[0] = step_out(x_dev, y_dev)

    ms_dev, launches = time_region(ctx, timed_step, steps, warmup, counter)
    if dump_dir is not None and rank == 0:
        # before the end-to-end loop below overwrites the graphs' static output buffers
        if train:
            arrays = {"loss": last[0], "params": torch.cat([p.detach().reshape(-1) for p in model.parameters()])}
        elif isinstance(last[0], tuple):        # VisionTransformer.forward: (logits, attention weights, encoded)
            logits, attn, enc = last[0]
            arrays = {"logits": logits, **{f"attn_weights_{i}": a for i, a in enumerate(attn)}, "encoded": enc}
        else:                                   # the ensemble's meta-classifier output
            arrays = {"out": last[0]}
        dump_outputs(dump_dir, arrays)
    del last

    # ---- end to end: every step copies ITS batch from pinned host memory (copy stream, double buffered so the copy of
    # step s+1 overlaps the compute of step s), runs the public call and reads the result back before it counts as done
    res_host = torch.empty((B, 1) if not train else (), dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream()

    def e2e_loop(host_x, bufs):
        ybuf = [torch.empty_like(y_dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        nchunk = 4 if host_x.numel() * host_x.element_size() >= (64 << 20) else 1

        def issue_copy(s):
            b = s & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])
                if nchunk == 1:
                    bufs[b].copy_(host_x, non_blocking=True)
                else:                                   # a few large copies keep the copy engine's queue full
                    n = host_x.shape[0]
                    for c in range(nchunk):
                        lo, hi = n * c // nchunk, n * (c + 1) // nchunk
                        bufs[b][lo:hi].copy_(host_x[lo:hi], non_blocking=True)
                if train:
                    ybuf[b].copy_(y_host, non_blocking=True)
                ready[b].record(copy_stream)

        def run(nsteps):
            main = torch.cuda.current_stream()
            for b in range(2):
                consumed[b].record(main)
            issue_copy(0)
            for s in range(nsteps):
                b = s & 1
                main.wait_event(ready[b])
                out = step_dev(bufs[b], ybuf[b] if train else None)
                consumed[b].record(main)
                if s + 1 < nsteps:
                    issue_copy(s + 1)
                res_host.copy_(out.detach().reshape(res_host.shape), non_blocking=True)
                main.synchronize()
        return run

    def timed_e2e(run):
        w = max(3, warmup // 2)
        run(w)
        ms, _ = time_region(ctx, lambda: run(steps), 1, 0)
        return ms

    units = B if ens else world * B
    if sharded is not None:
        # a rank ships only the batch slices of its own (member, slice) chunk
        ms_e2e = timed_e2e(lambda n: sharded_e2e_run(sharded, x_host, res_host, n))
        h2d = sharded.h2d_bytes(B)
    else:
        ms_e2e = timed_e2e(e2e_loop(x_host, [torch.empty_like(x_dev) for _ in range(2)]))
        h2d = int(B * VOL_BYTES + (B * 4 if train else 0))
    e2e = {"value": units * steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": int(res_host.numel() * 4), "ms_per_step": ms_e2e / steps,
           "h2d_gbs_per_rank": h2d / (ms_e2e / steps * 1e-3) / 1e9}
    if with_u8 and not train:
        # N2: the same volumes cross PCIe as uint8 (they ARE 8-bit images minus a mean); (u8 - mean) on the device
        u8_host, mean = O.synth_volumes_u8(B, seed=42 + (rank if not ens else 0))
        u8_host = u8_host.pin_memory()
        for m in members:
            m.input_mean = mean
        if sharded is not None:
            ms_u8 = timed_e2e(lambda n: sharded_e2e_run(sharded, u8_host, res_host, n))
            h2d8 = sharded.h2d_bytes(B) // 4
        else:
            ms_u8 = timed_e2e(e2e_loop(u8_host, [torch.empty(u8_host.shape, dtype=torch.uint8, device=dev) for _ in range(2)]))
            h2d8 = int(B * VOL_BYTES // 4)
        e2e["variants"] = {"u8": {"value": units * steps / (ms_u8 * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d8,
                                  "d2h_bytes_per_step": int(res_host.numel() * 4), "ms_per_step": ms_u8 / steps,
                                  "note": "volumes shipped as uint8 + mean (N2 input path), (u8 - mean) on the device"}}
    value = units * steps / (ms_dev * 1e-3)
    peaks = load_peaks()
    out = {
        "value": value, "unit": UNIT, "ms_per_step": ms_dev / steps, "steps": steps, "warmup": warmup,
        "scaling": "strong" if ens else "weak", "dtype": precision,
        "config": workload_config(wl, B, world, args.vis),
        "exec": {"precision": precision, "cuda_graph": graphed is not None or (sharded is not None and sharded.graphed),
                 "fused_train_step": bool(getattr(graphed, "fused", False)) if train else None},
        "model_tflops": value * flops_per_vol / 1e12,
        "model_frac_of_bf16_sustained": value * flops_per_vol / 1e12 / (world * peaks["bf16_tflops_sustained"]),
        "e2e": e2e, "gpu_launches": int(launches), "launches_per_step": launches / max(1, steps),
        "collective": collective, "bytes_per_collective": int(bytes_coll),
    }
    ctx.last = dict(cfgs=cfgs, B=B, train=train)
    del model, members, graphed, sharded, opt
    torch.cuda.empty_cache()
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes every tensor of `arrays` (name -> tensor) as `path`/<name>.npy in float32, DUMP_BYTES in all.  A tensor
    larger than its share is written as the flat sample of its elements at sorted indices drawn from a generator
    seeded with 0: the same indices for the same shapes, so two builds run with the same arguments compare element
    for element."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).unique()
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def ensemble_small_batch_probe(ctx, args):
    """The reference runs the 3 members back to back (models/modeling.py:354).  At the batch sizes the scripts use
    (4 for training, 1 for validation) one member cannot fill 148 SMs, so the members run on 3 streams here:
    serial vs concurrent time of `ensemble(x)` per batch size, device-resident input."""
    import torch
    import vit3d_b200
    from oracle import vit3d_oracle as O
    from vit3d_b200.dist import ShardedEnsemble
    from vit3d_b200.models.modeling import TransformerEnsemble, VisionTransformer
    cfgs = [vit3d_b200.north_star_config(c) for c in (5, 9, 11)]
    members = []
    for j, c in enumerate(cfgs):
        m = VisionTransformer(c, 128, zero_head=True, num_classes=1, vis=bool(args.vis), precision=args.precision)
        m.load_state_dict(O.init_state_dict(c, seed=42 + j))
        members.append(m)
    ens = TransformerEnsemble(*members, in_features=1).to(ctx.dev).eval()
    costs = [O.fwd_flops_per_volume(c) for c in cfgs]
    out = {}
    for B in (4, 16, 64):
        x = O.synth_volumes(B, seed=1).to(ctx.dev)
        row = {}
        for mode, conc in (("serial", False), ("concurrent", True)):
            se = ShardedEnsemble(ens, costs=costs, concurrent=conc)
            ms, _ = time_region(ctx, lambda: se(x), 20, 5)
            row[mode + "_ms"] = ms / 20
        row["speedup"] = row["serial_ms"] / row["concurrent_ms"]
        row["volumes_per_s"] = B / (row["concurrent_ms"] * 1e-3)
        out[f"B={B}"] = row
    del ens, members
    torch.cuda.empty_cache()
    return out


def cv_sweep_leg(ctx, args, jobs_per_gpu=6):
    """BASELINE.json config 5 (the train_baseline_cv.py sweep: 18 configurations x 5 folds of 100 steps at batch 4,
    validation every 24 steps on 18 volumes) on a bounded sample: `jobs_per_gpu` x world of the 90 jobs, dealt to the
    ranks longest-first, several jobs in flight per GPU (workflow.run_packed_sweep).  Replicas only - no collective.
    The whole 90-job sweep: tools/run_cv_sweep.py."""
    import importlib.util
    import torch
    import vit3d_b200
    from vit3d_b200 import workflow as W
    from vit3d_b200.dist import pack_jobs
    spec = importlib.util.spec_from_file_location("run_cv_sweep", os.path.join(ROOT, "tools", "run_cv_sweep.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    all_jobs = [(c, f) for c in range(1, 19) for f in range(5)]
    pick = all_jobs[::max(1, len(all_jobs) // (jobs_per_gpu * ctx.world))][:jobs_per_gpu * ctx.world]
    costs = []
    for c, _ in pick:
        cfg = vit3d_b200.north_star_config(c)
        costs.append(cfg.transformer["num_layers"] * (4 * 256 + 2 * cfg.transformer["mlp_dim"]))
    mine = [pick[i] for i in pack_jobs(costs, ctx.world)[ctx.rank]]
    if ctx.dist is not None:
        ctx.dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = W.run_packed_sweep(mine, mod.synth_fold, steps=100, batch=4, concurrent=6, device=str(ctx.dev))
    wall = time.perf_counter() - t0
    if ctx.dist is not None:
        t = torch.tensor([wall], device=ctx.dev)
        ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
        wall = float(t)
    n = len(pick)
    torch.cuda.empty_cache()
    return {"jobs": n, "of": len(all_jobs), "wall_s": wall, "jobs_per_s": n / wall, "train_steps_per_s": n * 100 / wall,
            "value": n * 100 * 4 / wall, "unit": UNIT, "concurrent_jobs_per_gpu": 6, "collective": None,
            "rank0_setup_s": res["setup_s"], "rank0_train_steps_per_s_excl_setup": res["train_steps_per_s_excl_setup"],
            "timing": "host wall clock around the whole sample (model construction, graph capture, training, validation), max over ranks",
            "config": {"workload": "train_baseline_cv.py sweep sample: 100 steps at batch 4, validation every 24 steps on 18 volumes, "
                                   "jobs = (configuration, fold) pairs spread over the 18 configurations",
                       "jobs_per_gpu": jobs_per_gpu, "parallelism": f"{ctx.world} ranks: independent jobs packed longest-first, no collective"}}


def sharded_e2e_run(sharded, x_host, res_host, nsteps):
    """End-to-end loop of the sharded ensemble: `stage` ships THIS rank's slice of the host batch on a copy stream, the
    copy of step s+1 overlaps the member forwards of step s, the result is read back before a step counts as done."""
    import torch
    nxt = sharded.stage(x_host)
    for s in range(nsteps):
        cur = nxt
        out = sharded(cur)
        if s + 1 < nsteps:
            nxt = sharded.stage(x_host)
        res_host.copy_(out.reshape(res_host.shape), non_blocking=True)
        torch.cuda.current_stream().synchronize()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    B = args.batch or wl["batch"]

    if args.impl == "reference":
        if rank != 0:
            return
        import vit3d_b200
        cfgs = [vit3d_b200.north_star_config(c) for c in wl["confs"]]
        # like for like: the GPU arm's batch, the driver's --steps / --warmup (cut short only by the time budget)
        # (the reference has no GPU path to put beside `value`: every rank of the GPU arm runs this same batch)
        v, ms, done, warm_done = cpu_arm(cfgs, wl["train"], max(1, args.steps), max(1, args.warmup), B, budget_s=args.cpu_budget)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
            "warmup": warm_done, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if len(wl["confs"]) > 1 else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(wl, B, args.gpus, args.vis),
            "steps_requested": args.steps, "warmup_requested": args.warmup,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                             "sample": f"{done} steps x {B} volumes (one rank's batch), oracle port of models/modeling.py, torch CPU "
                                       f"fp32, {os.cpu_count()} threads; budget {args.cpu_budget:.0f} s"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local_rank)
    ctx = Ctx()
    ctx.rank, ctx.world, ctx.dev = rank, world, torch.device("cuda", local_rank)
    ctx.numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    ctx.dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=ctx.dev)
        ctx.dist = dist
    args.warmup = max(3, args.warmup)           # timing rule: at least 3 untimed warm-up steps

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    head = run_leg(ctx, args, args.workload, args.steps, args.warmup, args.precision, dump_dir=args.dump_outputs)
    clk = clocks.stop() if rank == 0 else None
    head_ctx = ctx.last

    legs = {}
    if args.legs == "auto":
        names = [k for k in WORKLOADS if k != args.workload] + (["conf5_infer_tf32"] if args.workload == "conf5_infer" and
                                                                args.precision == "bf16" else [])
    elif args.legs == "none":
        names = []
    else:
        names = [s for s in args.legs.split(",") if s and s != "cv_sweep"]
    for nm in names:
        try:
            if nm == "conf5_infer_tf32":
                legs[nm] = run_leg(ctx, args, "conf5_infer", args.leg_steps, 3, "tf32", with_u8=False)
            else:
                legs[nm] = run_leg(ctx, args, nm, args.leg_steps, 3, args.precision)
        except Exception as e:          # a failed extra leg must not take the headline down with it
            legs[nm] = {"error": f"{type(e).__name__}: {e}"[:400]}
            if ctx.dist is not None:
                raise

    if world == 1 and args.legs == "auto":
        try:
            legs["ensemble_small_batch"] = ensemble_small_batch_probe(ctx, args)
        except Exception as e:
            legs["ensemble_small_batch"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    if args.legs == "auto" or "cv_sweep" in args.legs.split(","):
        try:
            legs["cv_sweep"] = cv_sweep_leg(ctx, args)
        except Exception as e:
            legs["cv_sweep"] = {"error": f"{type(e).__name__}: {e}"[:400]}
            if ctx.dist is not None:
                raise

    roof = cpu_base = None
    if rank == 0:
        roof = roofline_probe(args, head_ctx["cfgs"][0], head_ctx["B"], ctx.dev, head_ctx["train"])
        if not args.no_cpu_baseline and world == 1:
            sample = min(args.cpu_sample, head_ctx["B"])
            v, ms, done, _ = cpu_arm(head_ctx["cfgs"], head_ctx["train"], 3, 1, sample)
            cpu_base = {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                        "sample": f"{done} steps x {sample} volumes of the same workload, oracle port of models/modeling.py, "
                                  f"torch CPU fp32, {os.cpu_count()} threads"}
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": head["scaling"], "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": head["config"], "exec": head["exec"], "model_tflops": head["model_tflops"],
                "model_frac_of_bf16_sustained": head["model_frac_of_bf16_sustained"], "clocks": clk,
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "launches_per_step": head["launches_per_step"],
                "collective": head["collective"], "bytes_per_collective": head["bytes_per_collective"],
                "numa_bound_cpus": ctx.numa_cpus, "roofline": roof, "cpu_baseline": cpu_base, "workloads": legs}
        print(json.dumps(line))
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["source"] = "measured (MEASURED_PEAKS.json)"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def _time_launches(fn, iters=10, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the `ncu --set full` captures under profiles/
# (valid only for the captured shape: conf 5, batch 1024, bf16; None otherwise)
NCU_TRAFFIC = {"mlp_ln": (162.2e6, "profiles/r02_fused_mlp_fwd_ncu_full_raw.csv"),
               "fc1_gelu": (257.2e6, "profiles/r01_per_kernel_probe_conf5_b1024.log")}


def roofline_probe(args, cfg, B, dev, train=False):
    """Times the dominant kernel alone with CUDA events on the launching stream.

    Inference in BF16 mode: the fused MLP block (fc1 -> GELU -> fc2 -> + residual -> next LayerNorm,
    vit3d_mlp_ln_fwd), 44 % of the step and 75-82 % of the model's FLOPs: tensor bound, 4*S*H*d FLOP per volume
    per launch.  Otherwise (training / other precisions): the fc1 + GELU GEMM.  `others` carries the HBM-bound
    kernels of a layer against the measured copy bandwidth."""
    import torch
    from vit3d_b200 import _lib
    from vit3d_b200._lib import PREC, call, ptr, stream
    peaks = load_peaks()
    L = _lib.lib()
    M, H, d = B * 65, cfg.hidden_size, cfg.transformer["mlp_dim"]
    heads = cfg.transformer["num_heads"]
    prec = args.precision
    lp = prec == "bf16"
    adt = torch.bfloat16 if lp else torch.float32
    xn = (torch.randn(M, H, device=dev) * 0.5).to(adt)
    w1 = torch.randn(d, H, device=dev) * 0.05
    b1 = torch.randn(d, device=dev) * 0.01
    captured = (M == 66560 and d == 2048 and H == 256 and lp)
    others = []
    fused = (not train) and lp and H == 256 and bool(L.vit3d_mlp_ln_supported(M, H, d))
    if fused:
        w1l = w1.to(torch.bfloat16)
        w2h = (torch.randn(H, d, device=dev) / d ** 0.5).to(torch.float16)
        b2 = torch.randn(H, device=dev) * 0.01
        x32 = torch.randn(M, H, device=dev)
        y32 = torch.empty(M, H, device=dev)
        yn = torch.empty(M, H, device=dev, dtype=torch.bfloat16)
        g, be = torch.ones(H, device=dev), torch.zeros(H, device=dev)
        ms = _time_launches(lambda: call("vit3d_mlp_ln_fwd", ptr(xn), ptr(w1l), ptr(b1), ptr(w2h), ptr(b2), ptr(x32), ptr(y32),
                                         ptr(g), ptr(be), 1e-6, ptr(yn), M, H, d, stream()))
        flops = 4.0 * M * H * d
        ach = flops / (ms * 1e-3) / 1e12
        roof = {"kernel": "fused MLP block: fc1 + GELU + fc2 + residual + LayerNorm (vit3d_mlp_ln_fwd, tc_mlp2_kernel, "
                          "M=%d H=%d d=%d, tcgen05)" % (M, H, d),
                "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": ach / peaks["bf16_tflops"],
                "traffic": NCU_TRAFFIC["mlp_ln"][0] if captured else None, "traffic_unit": "bytes per launch",
                "traffic_source": (NCU_TRAFFIC["mlp_ln"][1] + " (ncu --set full capture of this shape; constant, not re-measured "
                                   "by this run)") if captured else None,
                "algorithmic_bytes": float(M * H * (2 + 4 + 4 + 2) + 2 * H * d * 2),
                "algorithmic_flops": flops, "ms_per_launch": ms, "peak_source": peaks.get("source"),
                "how": "kernel timed alone, 10 launches, CUDA events (burst peak applies)"}
        # HBM-bound kernels of the same layer (bytes = what the kernel must read + write once)
        hbm = peaks["hbm_gbs"]
        qkv = (torch.randn(M, 3 * H, device=dev) * 0.5).to(torch.bfloat16)
        ctx = torch.empty(M, H, device=dev, dtype=torch.bfloat16)
        if args.vis:      # the layout the module path uses: probability rows padded to 72 floats (sector-aligned stores)
            probs = torch.empty(B, heads, 65, 72, device=dev)
            t = _time_launches(lambda: call("vit3d_attn_fwd_padded", ptr(qkv), ptr(ctx), ptr(probs), 72, B, 65, heads, H // heads,
                                            stream()))
        else:
            t = _time_launches(lambda: call("vit3d_attn_fwd", ptr(qkv), ptr(ctx), None, B, 65, heads, H // heads,
                                            PREC["bf16"], stream()))
        nb = M * 4 * H * 2 + (B * heads * 65 * 65 * 4 if args.vis else 0)      # payload: the 65 valid floats of a row
        others.append({"kernel": "attention forward (attn_fwd_tc_kernel, vis=%s, probability rows padded to 72 floats)" % bool(args.vis), "bound": "hbm",
                       "achieved": nb / (t * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": nb / (t * 1e-3) / 1e9 / hbm,
                       "ms_per_launch": t})
        wo = (torch.randn(H, H, device=dev) / 16).to(torch.bfloat16)
        t = _time_launches(lambda: call("vit3d_linear_ln_fwd", ptr(ctx), ptr(wo), ptr(b2), ptr(x32), ptr(y32), ptr(g), ptr(be),
                                        1e-6, ptr(yn), None, None, M, H, H, stream()))
        nb = M * H * (2 + 4 + 4 + 2)
        others.append({"kernel": "out-projection + residual + LayerNorm (tc_gemm_res_kernel)", "bound": "hbm",
                       "achieved": nb / (t * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": nb / (t * 1e-3) / 1e9 / hbm,
                       "ms_per_launch": t})
        mean, rstd = torch.empty(M, device=dev), torch.empty(M, device=dev)
        t = _time_launches(lambda: call("vit3d_ln_fwd", ptr(x32), ptr(g), ptr(be), ptr(yn), 1, ptr(mean), ptr(rstd), M, H, 1e-6,
                                        stream()))
        nb = M * H * 6
        others.append({"kernel": "LayerNorm fp32 -> bf16 (ln_fwd_kernel)", "bound": "hbm", "achieved": nb / (t * 1e-3) / 1e9,
                       "peak": hbm, "unit": "GB/s", "frac": nb / (t * 1e-3) / 1e9 / hbm, "ms_per_launch": t})
    # the fc1 + GELU GEMM (training forward; the inference path when the fused block is unavailable)
    wl = w1.to(torch.bfloat16) if lp else None
    y = torch.empty(M, d, device=dev, dtype=adt)
    tc = bool(L.vit3d_tc_supported(PREC[prec], M, d, H))
    ms1 = _time_launches(lambda: call("vit3d_linear_fwd", ptr(xn), H, int(adt == torch.float32), ptr(w1), ptr(wl), ptr(b1), None,
                                      ptr(y), int(adt == torch.float32), None, 1, M, d, H, PREC[prec], stream()))
    flops1 = 2.0 * M * d * H
    fc1 = {"kernel": "fc1+GELU GEMM (vit3d_linear_fwd, M=%d N=%d K=%d, %s)" % (M, d, H, "tcgen05" if tc else "fp32 FMA"),
           "bound": "tensor", "achieved": flops1 / (ms1 * 1e-3) / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
           "frac": flops1 / (ms1 * 1e-3) / 1e12 / peaks["bf16_tflops"],
           "traffic": NCU_TRAFFIC["fc1_gelu"][0] if captured else None, "traffic_unit": "bytes per launch",
           "traffic_source": NCU_TRAFFIC["fc1_gelu"][1] if captured else None,
           "algorithmic_bytes": float(M * H * 2 + d * H * 2 + M * d * 2) if lp else None, "ms_per_launch": ms1,
           "peak_source": peaks.get("source"), "how": "kernel timed alone, 10 launches, CUDA events (burst peak applies)"}
    if not fused:
        return fc1
    others.append(fc1)
    roof["others"] = others
    return roof


if __name__ == "__main__":
    main()
