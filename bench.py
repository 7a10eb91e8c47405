#!/usr/bin/env python
"""bench.py -- icons/sec of one DeepSVG `hierarchical_ordered` train step (forward + SVGLoss + backward
[+ gradient all-reduce]) on N B200s.  Contract: see the task statement / DESIGN.md section "Measurement".

  python bench.py --gpus 1 --steps 20 --warmup 5                       # our arm (CUDA, tcgen05)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference --steps 3 --warmup 1                # CPU arm: the oracle port on the host cores

One JSON line on stdout (rank 0).  `value` = device-resident inputs; `e2e` = through the public module API with host
buffers (pinned H2D of the step's inputs + D2H of the loss inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs -> model_cfg overrides, per-GPU batch, forward GFLOP/icon and its attention+FFN part (SURVEY.md 8d,
# padded shapes; train step = 3x forward)
WORKLOADS = {
    "hier": dict(kind="hierarchical", over=dict(use_vae=False), batch=512, cpu_batch=32, fwd_gflop=2.7052,
                 attn_ffn_gflop=2.2466, configs=(1, 2),
                 desc="hierarchical_ordered train step, G=8 S=30 n_args=11 d_model=256 L=4+4+4+4 H=8 ff=512"),
    "fonts": dict(kind="one_stage", over=dict(use_vae=True, label_condition=True, n_labels=52, max_total_len=50), batch=256,
                  cpu_batch=64, fwd_gflop=0.5479, attn_ffn_gflop=0.4537, configs=(3, 3),
                  desc="one-stage fonts train step, G=1 S=50 52-class label conditioning, VAE, d_model=256 L=4+4 H=8 ff=512"),
    "scaled": dict(kind="hierarchical", over=dict(use_vae=False, d_model=512, n_layers=8, n_layers_decode=8,
                                                  max_num_groups=16, max_seq_len=64), batch=256, cpu_batch=2,
                   fwd_gflop=59.632, attn_ffn_gflop=55.811, configs=(4, 4),
                   desc="scaled hierarchical train step, G=16 S=64 d_model=512 L=8+8+8+8 H=8 (head_dim 64) ff=512"),
}
WEIGHTS = {"kl_tolerance": 0.1, "loss_kl_weight": 1.0, "loss_cmd_weight": 1.0, "loss_args_weight": 2.0,
           "loss_visibility_weight": 1.0}
MASK = np.array([[0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1], [0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1], [0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1],
                 [1, 1, 1, 1, 1, 0, 0, 0, 0, 1, 1], [0] * 11, [0] * 11, [0] * 11], dtype=np.float32)


def synth_icons(n, G=8, S=30, seed=1234, one_stage=False):
    """Vectorised version of the SURVEY.md 8d generator: paths of U{3..S} commands (m then l/c), U{1..G} visible paths.
    one_stage: G = 1 grouped tensors whose single sequence holds 1..3 'm' sub-paths (group index <= 3)."""
    rng = np.random.default_rng(seed)
    L = S + 2
    cmd = np.full((n, G, L), 4.0, dtype=np.float32)
    cmd[:, :, 0] = 5.0
    nvis = rng.integers(1, G + 1, size=(n, 1))
    vis = np.arange(G)[None, :] < nvis
    ln = rng.integers(3, S + 1, size=(n, G))
    pos = np.arange(L)[None, None, :]
    body = rng.integers(1, 3, size=(n, G, L)).astype(np.float32)
    body[:, :, 1] = 0.0
    if one_stage:
        for _ in range(2):      # up to two more sub-paths
            at = rng.integers(2, S + 1, size=(n, G))
            on = rng.integers(0, 2, size=(n, G)).astype(bool)
            body = np.where((pos == at[:, :, None]) & on[:, :, None], 0.0, body).astype(np.float32)
    inside = (pos >= 1) & (pos <= ln[:, :, None]) & vis[:, :, None]
    cmd = np.where(inside, body, cmd)
    vals = rng.integers(0, 256, size=(n, G, L, 11)).astype(np.float32)
    m = MASK[cmd.astype(np.int64)]
    args = vals * m - (1 - m)
    return torch.from_numpy(cmd), torch.from_numpy(args.astype(np.float32))


def workload_inputs(wl, n, seed):
    """(commands, args, label or None) of `n` synthetic icons of workload `wl` (host tensors)."""
    o = wl["over"]
    if wl["kind"] == "one_stage":
        c, a = synth_icons(n, G=1, S=o["max_total_len"], seed=seed, one_stage=True)
        lab = torch.from_numpy(np.random.default_rng(seed + 7).integers(0, o["n_labels"], size=(n,)).astype(np.int64))
        return c, a, lab
    c, a = synth_icons(n, G=o.get("max_num_groups", 8), S=o.get("max_seq_len", 30), seed=seed)
    return c, a, None


def bench_config(wl_name, batch, world):
    """The `config` object of the JSON line -- identical in both arms (ours / --impl reference) for the same command."""
    wl = WORKLOADS[wl_name]
    return {"workload": "%s, dropout 0.1 (train mode), batch %d per GPU (BASELINE configs[%d])"
                        % (wl["desc"], batch, wl["configs"][0 if world == 1 else 1]),
            "global_batch": batch * world, "parallelism": "dp%d" % world,
            "l2": "per-step working set (GBs of activations) >> 126 MB L2, no explicit flush needed"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1427.5)), d.get("bf16_tflops", 1654.1), \
            d.get("hbm_gbs", 6581.6), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel family: launch-count-weighted mean over
    the family's epilogue roles, each captured once with `ncu --set full` at the path-level shape
    (profiles/r*_linear_modes.json, written by tools/summarize_profiles.py from tools/gpu_artifacts.sh's captures)."""
    try:
        import glob
        files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_linear_modes.json")))
        modes = json.load(open(files[-1]))
        n = sum(m["launches_per_step"] for m in modes.values())
        tot = sum(m["launches_per_step"] * m["dram_bytes"] for m in modes.values())
        return (tot / n, "%s: launch-weighted mean over %d epilogue roles (%d path-level launches per step)" % (
            os.path.basename(files[-1]), len(modes), n)) if n else (None, None)
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region, via in-process NVML (spawning nvidia-smi every 100 ms was
    measured to stall CUDA launches for 100-250 ms at a time on a multi-GPU box)."""

    def __init__(self, gpu=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.recording = gpu, [], False, False
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu))
            # one-off firmware queries, synchronously and long before any timed region (they can take 100s of ms and
            # stall kernel submission while they run)
            self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.first = self._reasons()
        except Exception:
            self.nv, self.h = None, None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                pass
        return i

    def _reasons(self):
        nv = self.nv
        try:
            f = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            return int(f(self.h))
        except Exception:
            return 0

    def run(self):
        """During the timed region only the SM clock is polled (a cached register read); the throttle-reason query is an
        RPC to the GPU's firmware that was measured to stall kernel submission on every GPU of the box for 100-250 ms, so
        it is issued once when the region starts being sampled and once when it stops."""
        if self.h is None:
            return
        nv = self.nv
        mx, first = self.mx, self.first
        while not self.stop_flag:
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                if self.recording:
                    self.rows.append((clk, mx, 0))
            except Exception:
                pass
            time.sleep(0.5)
        last = self._reasons()
        self.rows.append((self.rows[-1][0] if self.rows else 0, mx, first | last))

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml unavailable"}
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        seen = sorted(k for k, b in bits.items() if any(r[2] & b for r in self.rows))
        return {"sm_mhz": float(np.median([r[0] for r in self.rows])), "sm_max_mhz": float(self.rows[0][1]),
                "reasons": seen, "samples": len(self.rows), "source": "nvml"}


# ---------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads given to the CPU arm: all host cores up to 32 -- beyond that torch's intra-op parallelism over these small
    GEMMs (K = 256) only adds synchronisation (measured 38 s/step with 128 threads vs ~5 s with 32 on the same box)."""
    return max(1, min(os.cpu_count() or 1, 32))


def port_rate(wl, batch, steps, warmup, threads=None, device="cpu", train_dropout=True):
    """The oracle (torch restatement of the reference path, stock ATen kernels, fp32) timed on `device`: icons/s of
    zero_grad + forward + SVGLoss + backward.  train_dropout=True draws the reference's train-mode dropout masks
    (model.train(), what deepsvg/train.py runs and what the CUDA arm runs); False is eval-mode arithmetic."""
    from oracle import svg_oracle as O
    if threads:
        torch.set_num_threads(threads)
    cfg = O.make_cfg(wl["kind"], **wl["over"])
    params = {k: v.to(device) for k, v in O.make_params(cfg, seed=0).items()}
    cmd, arg, lab = workload_inputs(wl, batch, seed=99)
    cmd, arg = cmd.to(device), arg.to(device)
    lab = lab.to(device) if lab is not None else None
    eps = torch.randn(batch, cfg.dim_z, device=device) if cfg.use_vae else None
    best, times = None, []
    for i in range(warmup + steps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        O.train_step(params, cfg, cmd, arg, label=lab, eps=eps, train_dropout=train_dropout)
        if device != "cpu":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    best = min(times)
    return batch / best, best, float(np.median(times))


def run_reference(a):
    """`--impl reference`: the reference's own implementation of the path on the host cores.  The reference is a pure-Python
    package without setup.py / pyproject (not pip-installable, so no baseline/_ref) and /root/reference does not exist on
    the GPU box: the timed code is the oracle port -- the same ATen CPU kernels the reference dispatches to -- in train-mode
    arithmetic (dropout masks drawn), on a FIXED bounded sample (batch pinned per workload) of the arm's workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[a.config]
    threads = host_threads()
    batch = a.cpu_batch or wl["cpu_batch"]
    rate, dt, med = port_rate(wl, batch, a.steps, a.warmup, threads, "cpu", train_dropout=True)
    sample = ("oracle port (fp32 torch CPU, train-mode arithmetic incl. dropout RNG), %s, fixed batch %d per step, best of "
              "%d steps (median %.3f s)" % (a.config, batch, a.steps, med))
    line = {"impl": "reference", "metric": METRIC % METRIC_NAME[a.config], "value": rate,
            "unit": "icons/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": bench_config(a.config, a.batch or wl["batch"], a.gpus),
            "cpu_baseline": {"value": rate, "unit": "icons/s", "cores": threads, "kind": "port", "sample": sample,
                             "batch_per_step": batch},
            "e2e": {"value": rate, "unit": "icons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


METRIC = "icons/sec train-step (fwd+loss+bwd) %s"
METRIC_NAME = {"hier": "hierarchical_ordered", "fonts": "one_stage_fonts", "scaled": "scaled_hierarchical"}
DUMP_BYTES = 60 << 20       # --dump-outputs: array data; with the .npy headers the files stay under 64 MB


def sample_cap(sizes, budget):
    """The largest per-array element count c with sum(min(n, c) for n in sizes) <= budget; None when all arrays fit."""
    if sum(sizes) <= budget:
        return None
    left, sizes = budget, sorted(sizes)
    for i, n in enumerate(sizes):
        share = left // (len(sizes) - i)
        if n > share:
            return share
        left -= n


def step_results(model, out, losses, budget_bytes):
    """{name: float32 array} of what a caller of the train step receives: the model's outputs ('out.*'), the loss terms
    ('loss.*') and every parameter gradient ('grad.*').  When they pass `budget_bytes` in all, each array larger than a
    common cap is replaced by a fixed seeded sample of that many of its elements (flattened, ascending index order): the
    same shapes give the same indices, so two runs or two builds compare element for element."""
    ts = {"out." + k: v for k, v in out.items() if torch.is_tensor(v) and v.is_floating_point()}
    ts.update(("loss." + k, v) for k, v in losses.items() if torch.is_tensor(v))
    ts.update(("grad." + k, p.grad) for k, p in model.named_parameters() if p.grad is not None)
    cap = sample_cap([t.numel() for t in ts.values()], budget_bytes // 4)
    res = {}
    for name, t in ts.items():
        t = t.detach()
        if cap is not None and t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        res[name] = t.float().cpu().numpy()
    return res


# ---------------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch.distributed as dist
    from deepsvg_b200 import SVGLoss, SVGTransformer, _lib, ops
    from deepsvg_b200.config import Hierarchical, OneStageOneShot
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    wl = WORKLOADS[a.config]
    make_cfg = lambda: (Hierarchical if wl["kind"] == "hierarchical" else OneStageOneShot)(**wl["over"])
    cfg = make_cfg()                                      # e.g. configs/deepsvg/hierarchical_ordered.py:4-9
    torch.manual_seed(1234)
    model = SVGTransformer(cfg, precision=a.precision, process_group=pg).to(dev)
    if world > 1:
        for p in model.parameters():                      # identical replicas
            dist.broadcast(p.data, 0)
    model.train()
    loss_fn = SVGLoss(cfg).to(dev)
    B = a.batch or wl["batch"]
    cmd_h, arg_h, lab_h = workload_inputs(wl, B, seed=1234 + rank)
    cmd_h, arg_h = cmd_h.pin_memory(), arg_h.pin_memory()
    lab_h = lab_h.pin_memory() if lab_h is not None else None
    cmd_d, arg_d = cmd_h.to(dev), arg_h.to(dev)
    lab_d = lab_h.to(dev) if lab_h is not None else None
    # end-to-end input path: the packed batch format (uint8 commands + int16 arguments, deepsvg_b200/data.py) in pinned host
    # memory; per step one H2D copy per tensor and one unpack kernel (the fp32 tensors would be 2.1x the bytes)
    from deepsvg_b200 import pack_tensors
    pb_h = pack_tensors(cmd_h, arg_h, lab_h, pin=True)
    pb_d = pb_h.cuda(dev)
    h2d = pb_h.nbytes
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def make_step(mdl, keep=None):
        def step(c, a_, lab=None):
            mdl.zero_grad(set_to_none=True)
            out = mdl(c, a_, c, a_, label=lab, params={})
            ls = loss_fn(out, None, weights=WEIGHTS)
            ls["loss"].backward()
            if keep is not None:
                keep["out"], keep["losses"] = out, ls
            return ls["loss"]
        return step

    last = {} if a.dump_outputs else None      # the timed path's results of its latest step (for --dump-outputs)
    step = make_step(model, last)
    cmd_in, arg_in = torch.empty_like(cmd_d), torch.empty_like(arg_d)   # device staging for the per-step H2D copies
    lab_in = torch.empty_like(lab_d) if lab_d is not None else None

    def make_e2e(stp):
        def step_e2e():
            pb_h.cuda(out=pb_d)                          # pinned host -> device, every step (packed: 23 B / position)
            pb_d.unpack(out=(cmd_in, arg_in))            # one kernel: uint8 / int16 -> the fp32 tensors forward() takes
            l = stp(cmd_in, arg_in, pb_d.label)
            loss_host.copy_(l.detach(), non_blocking=True)   # device -> pinned host, every step
        return step_e2e

    step_e2e = make_e2e(step)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        import gc
        gc.collect()
        gc.disable()     # a generation-2 collection in the launching thread shows up as a 30-100 ms hole in the GPU queue
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks, host = [], []
        trace = bool(os.environ.get("DSVG_BENCH_TRACE"))
        st0 = torch.cuda.memory_stats() if trace else None
        e0.record()
        for _ in range(steps):
            h0 = time.perf_counter()
            fn()
            if trace:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append(ev)
                host.append((time.perf_counter() - h0) * 1e3)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if marks and rank == 0:
            ts = [e0.elapsed_time(m) for m in marks]
            st1 = torch.cuda.memory_stats()
            sys.stderr.write("per-step ms: " + " ".join("%.1f" % (b - a) for a, b in zip([0.0] + ts[:-1], ts)) + "\n")
            sys.stderr.write("host-side ms: " + " ".join("%.1f" % h for h in host) + "\n")
            sys.stderr.write("allocator: cudaMalloc +%d, retries +%d, segments %d\n" % (
                st1["num_device_alloc"] - st0["num_device_alloc"], st1["num_alloc_retries"] - st0["num_alloc_retries"],
                st1["segment.all.current"]))
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        barrier()
        gc.enable()
        return ms

    def settle(stp, stp_e2e, limit=120):
        """Extended warm-up (untimed): the caching allocator needs a few more iterations to reach its steady-state pool, and
        with NCCL peer mappings every late cudaMalloc costs 100-250 ms.  Continue until five consecutive steps are within
        10 % of the fastest seen AND trigger no new cudaMalloc; at most `limit` extra steps, same count on all ranks."""
        stable, best, extra = 0, None, 0
        n_malloc = torch.cuda.memory_stats()["num_device_alloc"]
        while extra < limit:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            stp(cmd_d, arg_d, lab_d)
            stp_e2e()
            t1.record()
            torch.cuda.synchronize()
            now_malloc = torch.cuda.memory_stats()["num_device_alloc"]
            dt = torch.tensor([t0.elapsed_time(t1), float(now_malloc - n_malloc)], device=dev)
            n_malloc = now_malloc
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dt, grew = dt[0].item(), dt[1].item() > 0
            best = dt if best is None else min(best, dt)
            stable = stable + 1 if (dt <= 1.1 * best and not grew) else 0   # steady = fast AND no new device allocation
            extra += 1
            if stable >= 5 and extra >= 6:
                break
        return extra

    for _ in range(max(a.warmup, 3)):
        step(cmd_d, arg_d, lab_d)
    sampler = ClockSampler(local) if (rank == 0 and not os.environ.get("DSVG_NO_CLOCKS")) else None
    if sampler:
        sampler.start()      # its one-off NVML firmware queries happen during the warm-up below, not in the timed region
    extra = settle(step, step_e2e)
    if sampler:
        sampler.recording = True
    l0 = _lib.launch_count() + model.graph_kernel_launches
    # every step draws its dropout seed from the CUDA generator, and settle() runs a timing-dependent number of steps:
    # reseeding here makes the timed steps' masks, and so the last step's results, a function of the arguments alone
    torch.cuda.manual_seed(1234)
    ms = timed(lambda: step(cmd_d, arg_d, lab_d), a.steps)
    launches = (_lib.launch_count() + model.graph_kernel_launches - l0) / a.steps
    # the step's outputs live in buffers the next (CUDA-graph) step overwrites: sample them before the e2e steps run
    dump = step_results(model, last["out"], last["losses"], DUMP_BYTES) if last is not None else None
    for _ in range(5):
        step_e2e()
    ms_e2e = timed(step_e2e, a.steps)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    final_loss = float(loss_host.item())

    # ---- per-family kernel timing (one extra, untimed step with events around every tensor-core launch) ----
    fam = {}
    ops.PROFILE = [] if rank == 0 else None
    # Park the GPU behind a ~20 ms spin kernel first, so that the (slower, instrumented) host thread has enqueued the launches
    # and event records before the device reaches them: each event pair then brackets pure device time instead of the host's
    # launch latency (which dominated the 8-15 us group-level GEMMs).
    try:
        torch.cuda._sleep(40_000_000)
    except Exception:
        pass
    step(cmd_d, arg_d, lab_d)       # every rank runs it: the step contains collectives
    torch.cuda.synchronize()
    shapes = {}
    if rank == 0:
        for family, flops, e0, e1, shape, nbytes in ops.PROFILE:
            ms_k = e0.elapsed_time(e1)
            f = fam.setdefault(family, [0, 0.0, 0.0, 0.0])
            f[0] += 1
            f[1] += flops
            f[2] += ms_k
            f[3] += nbytes
            if shape is not None:
                g = shapes.setdefault((family,) + tuple(shape), [0, 0.0, 0.0, 0.0])
                g[0] += 1
                g[1] += flops
                g[2] += ms_k
                g[3] += nbytes
    ops.PROFILE = None

    # ---- the tolerance-meeting mode (bf16x3: rtol 1e-3 / atol 1e-4 vs the fp32 reference, tests/test_model_gpu.py) timed too --
    parity = None
    graphed = getattr(model, "_gs", None) is not None
    graph_backward = graphed and model._gs.bwd_a is not None
    if hasattr(model, "release_graphs"):
        model.release_graphs()          # frees the captured step's private pool (one step of activations)
        torch.cuda.empty_cache()
    if a.precision == "bf16" and not a.no_parity_mode:
        pm = SVGTransformer(cfg, precision="bf16x3", process_group=pg).to(dev)
        pm.load_state_dict(model.state_dict())
        pm.train()
        pstep = make_step(pm)
        pe2e = make_e2e(pstep)
        for _ in range(3):
            pstep(cmd_d, arg_d, lab_d)
        settle(pstep, pe2e, limit=20)
        k = a.steps
        pms = timed(lambda: pstep(cmd_d, arg_d, lab_d), k)
        pms_e2e = timed(pe2e, k)
        parity = {"precision": "bf16x3 (split-bf16 operands, 3 tcgen05 products per K step)", "steps": k,
                  "value": world * B * k / (pms / 1e3), "ms_per_step": pms / k,
                  "e2e": world * B * k / (pms_e2e / 1e3), "unit": "icons/s", "final_loss": float(loss_host.item()),
                  "cuda_graphs": getattr(pm, "_gs", None) is not None,
                  "tolerance": "logits/loss rtol 1e-3 atol 1e-4 vs the fp32 reference; argmax identical wherever the "
                               "reference's own top-2 margin exceeds 2e-4 (tests/test_model_gpu.py)"}
        pm.release_graphs()
        del pm, pstep, pe2e
        torch.cuda.empty_cache()

    # ---- data-parallel self-check (N > 1): all-reduced per-rank gradients == single-process gradient of the global batch --
    ddp = None
    if world > 1 and not a.no_ddp_check:
        ddp = ddp_check(cfg, wl, model, loss_fn, pg, dev, rank, world)

    # ---- stock PyTorch (the oracle port, fp32 ATen CUDA kernels) on the same GPU, same batch: "reference on the same box" --
    ref_gpu = None
    if world == 1 and not a.no_cpu_baseline and not a.no_ref_gpu:
        try:
            torch.backends.cuda.matmul.allow_tf32 = False
            del model
            torch.cuda.empty_cache()
            nb = min(B, 128 if a.config == "scaled" else B)
            r, dt, med = port_rate(wl, nb, 3, 2, None, dev, train_dropout=True)
            ref_gpu = {"value": r, "unit": "icons/s", "kind": "port", "dtype": "fp32 (TF32 off)", "batch": nb,
                       "ms_per_step": dt * 1e3,
                       "what": "oracle port = the reference's op sequence on stock ATen CUDA kernels, train-mode dropout, "
                               "same GPU, wall clock with synchronize, best of 3"}
        except Exception as e:   # an out-of-memory here must not lose the measured line
            ref_gpu = {"unavailable": repr(e)[:200]}
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ips = world * B * a.steps / (ms / 1e3)
    ips_e2e = world * B * a.steps / (ms_e2e / 1e3)
    sus, burst, hbm, src = peaks()
    train_gflop = 3 * wl["fwd_gflop"]
    step_tflops = ips * train_gflop / 1e3 / world
    af_tflops = ips * 3 * wl["attn_ffn_gflop"] / 1e3 / world
    lin = fam.get("linear", [1, 0.0, 1.0, 0.0])
    lin_tflops = lin[1] / (lin[2] / 1e3) / 1e12 if lin[2] > 0 else 0.0
    cpu_threads = host_threads()
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        cb = a.cpu_batch or wl["cpu_batch"]
        r_tr, dt_tr, _ = port_rate(wl, cb, 2, 1, cpu_threads, "cpu", train_dropout=True)
        r_ev, dt_ev, _ = port_rate(wl, cb, 2, 1, cpu_threads, "cpu", train_dropout=False)
        cpu = {"value": r_tr, "unit": "icons/s", "cores": cpu_threads, "kind": "port",
               "sample": "oracle port (fp32 torch CPU, train-mode arithmetic incl. dropout RNG), fixed batch %d, best of 2 "
                         "steps (%.2f s each)" % (cb, dt_tr),
               "eval_mode_value": r_ev,
               "why_port": "the reference is a setup-less pure-Python package: not pip-installable, and /root/reference is "
                           "absent on the GPU box"}
    traffic, traffic_src = ncu_traffic()
    cfgd = bench_config(a.config, B, world)
    line = {
        "metric": METRIC % METRIC_NAME[a.config], "value": ips, "unit": "icons/s",
        "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if a.precision == "bf16" else "bf16x3(split-bf16, fp32-accurate)", "data": "synthetic",
        "config": cfgd,
        "run": {"final_loss": final_loss, "extra_untimed_warmup_steps": extra,
                "cuda_graphs": {"forward": graphed, "backward": graph_backward,
                                "note": "gpu_launches counts the kernels inside the replayed graphs plus the eager loss kernels"},
                "argmax_note": "bit-exact argmax is asserted (parity mode) where the reference's top-2 margin > 2e-4"},
        "e2e": {"value": ips_e2e, "unit": "icons/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / a.steps,
                "input_format": "packed uint8 commands + int16 arguments in pinned host memory, unpacked on the GPU"},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "kernel": "dsvg::linear_kernel (tcgen05 X.W^T, all forward + dgrad GEMMs)",
                     "achieved": lin_tflops, "peak": sus, "unit": "TFLOP/s", "frac": lin_tflops / sus if sus else None,
                     "peak_source": src + " (bf16_tflops_sustained)", "launches_per_step": lin[0],
                     "ms_per_step_in_kernel": lin[2], "traffic": traffic, "traffic_source": traffic_src,
                     "step": {"achieved": step_tflops, "frac": step_tflops / sus, "gflop_per_icon": train_gflop},
                     "attn_ffn": {"achieved": af_tflops, "frac": af_tflops / sus, "gflop_per_icon": 3 * wl["attn_ffn_gflop"],
                                  "what": "north-star fraction: attention+FFN FLOPs of the step / step time / peak"},
                     # the same family against the OTHER roof: algorithmic bytes (operands read once, outputs written once)
                     # of its launches / their time / the measured copy bandwidth.  d_model 256 puts these GEMMs at
                     # ~190 FLOP/B, under the ridge (sustained peak / copy bandwidth = 217): whichever fraction is larger
                     # names the roof the family actually leans on
                     "hbm": {"achieved": lin[3] / (lin[2] / 1e3) / 1e9 if lin[2] > 0 else 0.0, "peak": hbm, "unit": "GB/s",
                             "frac": lin[3] / (lin[2] / 1e3) / 1e9 / hbm if (lin[2] > 0 and hbm) else None,
                             "gbytes_per_step": lin[3] / 1e9},
                     "families": {k: {"launches": v[0], "ms": v[2], "tflops": (v[1] / (v[2] / 1e3) / 1e12 if v[2] else 0),
                                      "gbs": (v[3] / (v[2] / 1e3) / 1e9 if v[2] else 0)}
                                  for k, v in fam.items()},
                     # the six most expensive GEMM shapes of the step, each with its own achieved rate (live CUDA events)
                     "top_shapes": [{"kernel": k[0], "MNK": list(k[1:]), "launches": v[0], "ms": round(v[2], 4),
                                     "tflops": round(v[1] / (v[2] / 1e3) / 1e12, 1),
                                     "frac_of_peak": round(v[1] / (v[2] / 1e3) / 1e12 / sus, 3),
                                     "gbs": round(v[3] / (v[2] / 1e3) / 1e9, 1),
                                     "frac_of_hbm": round(v[3] / (v[2] / 1e3) / 1e9 / hbm, 3) if hbm else None}
                                    for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][2])[:6]]},
        "clocks": sampler.summary() if sampler else None,
    }
    if parity is not None:
        line["parity_mode"] = parity
    if ddp is not None:
        line["ddp_check"] = ddp
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if ref_gpu is not None:
        line["ref_gpu"] = ref_gpu
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def ddp_check(cfg, wl, model, loss_fn, pg, dev, rank, world, n_per_rank=4):
    """One untimed eval-mode bf16x3 step per rank on its own shard (gradients all-reduced by the product path) against the
    single-process step on the concatenated global batch (reference semantics: nn.DataParallel gathers the logits, SVGLoss
    normalises by GLOBAL masked counts, loss.py:53-54 under train.py:74).  Reports the worst relative L2 gradient error."""
    import torch.distributed as dist
    from deepsvg_b200 import SVGTransformer
    sd = model.state_dict()
    ours = SVGTransformer(cfg, precision="bf16x3", process_group=pg).to(dev)
    ours.load_state_dict(sd)
    ours.eval()
    single = SVGTransformer(cfg, precision="bf16x3", process_group=None).to(dev)
    single.load_state_dict(sd)
    single.eval()
    if cfg.use_vae:
        ours._eps_override = torch.zeros(n_per_rank, cfg.dim_z, device=dev)
        single._eps_override = torch.zeros(n_per_rank * world, cfg.dim_z, device=dev)
    c, a_, lab = workload_inputs(wl, n_per_rank, seed=4321 + rank)
    c, a_ = c.to(dev), a_.to(dev)
    lab = lab.to(dev) if lab is not None else None

    def run(mdl, cc, aa, ll, group):
        mdl.zero_grad(set_to_none=True)
        out = mdl(cc, aa, cc, aa, label=ll, params={})
        loss_fn.process_group = None
        ls = loss_fn(out, None, weights=WEIGHTS)
        ls["loss"].backward()
        return ls["loss"].detach(), [p.grad.detach().clone() for p in mdl.parameters()]

    l_dp, g_dp = run(ours, c, a_, lab, pg)

    def gather(t):
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous(), group=pg)
        return torch.cat(parts, 0)

    cg, ag = gather(c), gather(a_)
    lg = gather(lab) if lab is not None else None
    l_1, g_1 = run(single, cg, ag, lg, None)
    worst, worst_name, num, den = 0.0, "", 0.0, 0.0
    for (name, _), gd, g1 in zip(single.named_parameters(), g_dp, g_1):
        d2, n2 = (gd - g1).double().pow(2).sum().item(), g1.double().pow(2).sum().item()
        num, den = num + d2, den + n2
        e = (d2 / (n2 + 1e-300)) ** 0.5
        if e > worst:
            worst, worst_name = e, name
    res = torch.tensor([worst, (num / (den + 1e-300)) ** 0.5, abs(l_dp.item() - l_1.item()) / abs(l_1.item())], device=dev)
    dist.all_reduce(res, op=dist.ReduceOp.MAX, group=pg)
    return {"max_rel_grad_err": res[0].item(), "global_rel_grad_err": res[1].item(), "rel_loss_err": res[2].item(),
            "worst_tensor": worst_name, "icons_per_rank": n_per_rank, "mode": "eval, bf16x3",
            "what": "NCCL-all-reduced per-rank gradients vs the single-process gradient of the concatenated batch"}


def main():
    import signal
    signal.alarm(int(os.environ.get("DSVG_BENCH_TIMEOUT", "900")))   # a hung collective must not hold the box
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("DSVG_BENCH_CONFIG", "hier"), choices=sorted(WORKLOADS),
                    help="hier = BASELINE configs[1]/[2] (the headline), fonts = configs[3], scaled = configs[4]")
    ap.add_argument("--batch", type=int, default=0, help="icons per GPU per step (default: the workload's)")
    ap.add_argument("--precision", default=os.environ.get("DSVG_PRECISION", "bf16"))
    ap.add_argument("--cpu-batch", type=int, default=0, help="icons per CPU-arm step (default: pinned per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-mode", action="store_true")
    ap.add_argument("--no-ddp-check", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's logits, losses and parameter gradients to DIR/<name>.npy (float32; "
                         "a fixed sample of each large array; under 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
