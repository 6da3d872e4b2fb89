#!/usr/bin/env python
"""bench.py — patch-pairs/s of the train step (BASELINE.json configs[1]: synthetic rho=45, 128x128 2-channel patches,
per-GPU batch 128, loss_type=h_loss, Adam lr 5e-4), one process per GPU.

  python bench.py --gpus 1 --steps K --warmup W                      # our CUDA path (default numeric mode: see --numeric)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...                               # the restated reference (oracle/) on the host CPU
  python bench.py ... --dump-outputs DIR                             # also write the last timed step's outputs as DIR/*.npy

A step = one full pass of the hot path over one batch: regressor forward (dropout on), h4p losses, DLT, fused warp +
all six photometric diagnostics (the reference fetches them every step, homography_CNN_synthetic.py:345), backward of
h_loss, gradient allreduce (N > 1), TF-Adam update.  `value` is timed with inputs resident in HBM; `e2e` goes through
the host-facing HostStepper API with pinned host inputs (H2D + D2H inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "patch-pairs/sec (128x128) per train step"
PER_GPU_BATCH = 128
# MACs per pair of each conv layer's forward (SURVEY §8a row C)
CONV_MACS = [18.87e6, 603.98e6, 150.99e6, 150.99e6, 75.50e6, 150.99e6, 37.75e6, 37.75e6]
FWD_FLOP_PER_PAIR = 2.5208e9
TRAIN_FLOP_PER_PAIR = 7.525e9


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be >= 1, got %d" % v)
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="number of timed train steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--numeric", default=os.environ.get("UDH_NUMERIC", "auto"), choices=["auto", "fp32", "bf16", "bf16x3"],
                    help="auto = bf16x3, the tensor-core mode the parity tests certify (tests/test_gpu_x3.py)")
    ap.add_argument("--loss_type", default="h_loss")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dp-diag", default="", choices=["", "nocomm"], help="multi-GPU diagnosis only: 'nocomm' skips the gradient allreduce")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short BASELINE configs[2]/[3] side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned on rank 0 (and a fixed sample of the updated "
                         "weights) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


# Seeded sample of the updated flat parameters written by --dump-outputs: the full 137 MB buffer is too large to keep.
PARAM_SAMPLE = 1 << 20


def snapshot_outputs(out, params):
    """Host copies of what one train step hands its caller: every public entry of the returned dict and a fixed seeded
    sample of the updated parameters (about 13 MB in all at batch 128)."""
    import numpy as np
    import torch
    snap = {}
    for k, v in out.items():
        if k.startswith("_"):
            continue
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        snap[k] = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
    idx = np.sort(np.random.default_rng(0).integers(0, params.numel(), PARAM_SAMPLE))
    snap["params_sample"] = params[torch.from_numpy(idx).to(params.device)].cpu().numpy().astype(np.float32)
    return snap


def write_outputs(d, snap):
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for k, a in snap.items():
        np.save(os.path.join(d, k + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """All the host threads this process may actually use: min(affinity, cgroup cpu quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def cpu_oracle_pairs_per_s(sample_b, steps, warmup, loss_type):
    """The restated reference (oracle/, PyTorch-CPU fp32, all host threads) on a bounded sample of the workload."""
    import torch
    from oracle import oracle as O
    from unsuperviseddeephomographyral2018_b200 import params as P
    torch.set_num_threads(host_threads())
    specs = P.param_specs()
    flat = torch.tensor(P.init_flat(0))
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    batch = O.make_batch(0, sample_b)
    g = torch.Generator().manual_seed(0)
    s = 128 // 8
    times = []
    for i in range(warmup + steps):
        keep = (torch.bernoulli(torch.full((sample_b, s, s, 128), 0.5), generator=g), torch.bernoulli(torch.full((sample_b, 1024), 0.5), generator=g))
        t0 = time.perf_counter()
        flat, m, v, out, _ = O.train_step(flat, m, v, i, batch, specs, loss_type=loss_type, lr=5e-4, keep_masks=keep)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return sample_b * len(times) / tot, tot / len(times) * 1e3, torch.get_num_threads()


def workload(loss_type):
    """The same string in both arms (the driver compares the arms' configs)."""
    return "train step (BASELINE configs[1]): synthetic rho=45, 128x128 2-ch patches, batch 128 per GPU, loss_type=%s" % loss_type


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_b = 4
    steps, warmup = args.steps, max(0, args.warmup)
    val, ms, cores = cpu_oracle_pairs_per_s(sample_b, steps, warmup, args.loss_type)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": workload(args.loss_type),
                   "sample": "each step = %d pairs of the 128-pair batch on the host CPU" % sample_b},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": "%d pairs/step x %d steps, oracle/ (PyTorch-CPU fp32 restatement; the TF1 reference cannot be installed here)" % (sample_b, steps)},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from unsuperviseddeephomographyral2018_b200 import _lib, engine, synthetic, trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_MAX_CTAS", "32")                  # bound the allreduce kernel to the SMs the conv4_x backward leaves free
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
        if args.dp_diag == "nocomm":
            # DIAGNOSTIC ONLY (the line is labelled and is not a bench value): skip the gradient allreduce so that the
            # per-rank step times show the GPU-to-GPU spread the collective otherwise hides behind its implicit barrier.
            _real_all_reduce = dist.all_reduce
            torch.distributed.all_reduce = lambda t, op=dist.ReduceOp.SUM, group=None, async_op=False: (
                _real_all_reduce(t, op=op, group=group) if op == dist.ReduceOp.MAX else None)
    numeric = args.numeric
    if numeric == "auto":
        numeric = "bf16x3"       # the parity-certified tensor-core mode is the headline; single-pass bf16 is a labelled side number
    B = PER_GPU_BATCH
    eng = engine.HomographyEngine(B, numeric=numeric, seed=0, loss_type=args.loss_type, lr=5e-4, device=dev, process_group=pg, world_size=world)
    # Training amplifies rounding: the gradient sums use fp32 atomics, whose order varies from run to run, and TF-Adam
    # normalises near-zero gradients to steps of about lr, so two runs drift apart within a few steps.  The last timed step
    # therefore starts again from the seeded initial state (restored outside the timed windows): its inputs are then the
    # same in every run and its outputs (--dump-outputs) agree to rounding.
    init_state = dict(params=eng.params.clone(), adam_m=eng.adam_m.clone(), adam_v=eng.adam_v.clone(), global_step=eng.global_step)
    nb = 3
    batches = [synthetic.make_batch(B, seed=1000 * rank + i, device=dev) for i in range(nb)]
    W, K = max(3, args.warmup), args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled (nvidia-smi, 100 ms) from the warm-up to the end of the e2e loop: the timed region itself can be
    # shorter than one sampling period
    sampler = ClockSampler(local); sampler.start()
    for i in range(W):
        eng.train_step(batches[i % nb])
    barrier()
    # ---- the timed region: exactly K steps, nothing else on the stream (no per-phase events); two windows, K - 1 steps
    # and the last one, with the restore of the initial state between them ----
    launches0 = _lib.lib.udh_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K - 1):
        eng.train_step(batches[i % nb])
    r0.record()
    eng.load_state_dict(init_state)
    del init_state
    r1.record()
    out = eng.train_step(batches[(K - 1) % nb])
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(r0) + r1.elapsed_time(e1)
    launches = _lib.lib.udh_launch_count() - launches0
    # the step's results live in the engine's static buffers: copy them before the next step overwrites them
    dumped = snapshot_outputs(out, eng.params) if args.dump_outputs and rank == 0 else None
    # ---- the same K steps again with the library's per-phase CUDA-event brackets (udh_prof_*): per-kernel durations for the
    # roofline.  Kept out of the headline region because ~80 event records per step serialise kernel boundaries. ----
    _lib.lib.udh_prof_enable(1); _lib.lib.udh_prof_reset()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(K):
        eng.train_step(batches[i % nb])
    p1.record()
    barrier()
    ms_step_instrumented = p0.elapsed_time(p1) / K
    phases = _lib.prof_read_all()
    _lib.lib.udh_prof_enable(0)
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    ms_ranks = [ms_total / K]
    if world > 1:
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        ms_ranks = [float(x.item()) / K for x in g]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / K
    value = B * world * K / (ms_total * 1e-3)

    # ---- end to end through the host-facing API (pinned host inputs, H2D + D2H every step) ----
    e2e = None
    if not args.no_e2e:
        host = [trainer.pin_batch(b) for b in batches]
        stepper = trainer.HostStepper(eng)
        for i in range(3):
            stepper.step(host[i % nb])
        stepper.flush(); barrier()
        t0 = time.perf_counter()
        e0.record()
        for i in range(K):
            stepper.step(host[i % nb])
        last = stepper.flush()
        e1.record(); barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms_e = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms_e, wall], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e = float(t[0].item())
        e2e = {"value": B * world * K / (ms_e * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": stepper.h2d_bytes * world,
               "d2h_bytes_per_step": stepper.d2h_bytes * world, "ms_per_step": ms_e / K, "wall_ms_per_step": float(t[1].item()) / K,
               "api": "trainer.HostStepper.step(pinned post-dataloader fp32 tensors, the reference's feed)", "last_h_loss": last["h_loss"] if last else None}
        # variant: the host hands over the decoded uint8 images; normalise / gray / patch gather run on the device
        host8 = [trainer.pin_batch_u8(b["I_u8"], b["I_prime_u8"], b["pts1"], b["gt"]) for b in batches]
        for i in range(3):
            stepper.step_u8(host8[i % nb])
        stepper.flush(); barrier()
        e0.record()
        for i in range(K):
            stepper.step_u8(host8[i % nb])
        last8 = stepper.flush()
        e1.record(); barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e["uint8_input_variant"] = {"value": B * world * K / (float(t.item()) * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": stepper.h2d_bytes * world,
                                      "d2h_bytes_per_step": stepper.d2h_bytes * world, "ms_per_step": float(t.item()) / K,
                                      "api": "trainer.HostStepper.step_u8(pinned decoded uint8 images; device-side normalise/gray/crop)",
                                      "last_h_loss": last8["h_loss"] if last8 else None}

    clocks = sampler.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    # ---- roofline of the dominant kernel family (by measured share of the step) ----
    layers = ["conv1_1", "conv1_2", "conv2_1", "conv2_2", "conv3_1", "conv3_2", "conv4_1", "conv4_2"]
    fam = {}          # family -> [ms total, launches, algorithmic flops, algorithmic bytes]

    def add(f, ms, n, flops=0.0, byts=0.0):
        e = fam.setdefault(f, [0.0, 0, 0.0, 0.0]); e[0] += ms; e[1] += n; e[2] += flops; e[3] += byts
    tc = numeric in ("bf16", "bf16x3")
    for name, (tms, cnt) in phases.items():
        head, _, kind = name.partition(".")
        if head in layers:
            li = layers.index(head)
            flops = 2.0 * CONV_MACS[li] * B * cnt
            if li == 0 or not tc:
                add("conv3x3 fp32 CUDA-core kernels" if not tc else "conv1_1 CUDA-core kernels", tms, cnt, flops)
            elif kind == "wgrad":
                add("tc_wgrad%s_kernel (tcgen05 weight gradient, conv1_2..conv4_2)" % ("_x3" if numeric == "bf16x3" else ""), tms, cnt, flops)
            else:
                add("tc_conv%s_kernel (tcgen05 implicit-GEMM conv fwd+dgrad, conv1_2..conv4_2)" % ("_x3" if numeric == "bf16x3" else ""), tms, cnt, flops)
        elif name == "adam":
            add("adam_kernel", tms, cnt, 0.0, 28.0 * 34192264 * cnt)
        elif name.startswith("fc"):
            add("fc1/fc2 GEMMs", tms, cnt, 2.0 * 33.56e6 * B * cnt * (1 if name == "fc.fwd" else 2))
        else:
            add(name, tms, cnt)
    roof = None
    if fam:
        name, (tms, cnt, flops, byts) = max(fam.items(), key=lambda kv: kv[1][0])
        share = tms / K / ms_step
        if flops:
            ach = flops / (tms * 1e-3) / 1e12
            peak = peaks["bf16_tflops_sustained"]
            roof = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "traffic": None, "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "launches_per_step": cnt / K, "ms_per_step": tms / K, "share_of_step": share,
                    "algorithmic_work": "2*MAC(layer)*B per launch, MACs from SURVEY 8a row C" +
                                        ("; the two-limb mode issues THREE tensor-core MACs per algorithmic MAC (lo.hi + hi.hi + hi.lo), so the "
                                         "tensor pipe is busy for 3x this fraction: frac_of_issued_macs = %.3f" % (3.0 * ach / peak) if numeric == "bf16x3" else "")}
        else:
            ach = byts / (tms * 1e-3) / 1e9 if byts else None
            roof = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / peaks["hbm_gbs"] if ach else None, "traffic": None, "peak_source": peaks["source"],
                    "launches_per_step": cnt / K, "ms_per_step": tms / K, "share_of_step": share}
        tr = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if roof and os.path.exists(tr):
            try:
                roof["traffic"] = json.load(open(tr)).get(name.split(" ")[0])
            except Exception:
                pass
    extras = None
    if world == 1 and not args.no_extras:
        extras = other_configs(torch, _lib, engine, synthetic, numeric, peaks, dev)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        sb = 8
        v, ms_cpu, cores = cpu_oracle_pairs_per_s(sb, 2, 1, args.loss_type)
        cpu = {"value": v, "unit": "pairs/s", "cores": cores, "kind": "port",
               "sample": "%d-pair sample of the 128-pair batch, 1 warm-up + 2 timed train steps of oracle/ (PyTorch-CPU fp32 restatement)" % sb}
    dtype = {"bf16x3": "bf16x3 (two bf16 limbs per fp32 value, lo.hi + hi.hi + hi.lo on tcgen05, fp32 TMEM accumulation: fp32-grade, parity-certified)",
             "bf16": "bf16 (single pass, fp32 accumulation: throughput mode, NOT parity-certified)", "fp32": "fp32 (CUDA cores)"}[numeric]
    parity = None
    if world == 1 and not args.no_extras:
        parity = parity_check(torch, engine, numeric, dev)
    line = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
        "ms_per_step_ranks": [round(x, 4) for x in ms_ranks], "dp_diag": args.dp_diag or None,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic", "parity": parity,
        "config": {"workload": workload(args.loss_type),
                   "per_gpu_batch": B, "global_batch": B * world, "parallelism": "dp%d" % world, "numeric_mode": numeric,
                   "dropout": "on (keep 0.5)", "optimizer": "TF-Adam lr 5e-4 staircase",
                   "l2_policy": "inputs larger than L2: %d rotating batches, 135 MB of inputs + ~1.7 GB of activations touched per step (L2 = 126 MB)" % nb},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
        "tflops_algorithmic": TRAIN_FLOP_PER_PAIR * B * world / (ms_step * 1e-3) / 1e12,
        "phases_ms_per_step": {k: round(v[0] / K, 4) for k, v in sorted(phases.items(), key=lambda kv: -kv[1][0])},
        "phases_note": "per-phase CUDA-event brackets, measured live in a second pass of the same %d steps (%.4f ms/step with the ~80 event "
                       "records per step on the stream; the headline region carries none)" % (K, ms_step_instrumented),
        "other_configs": extras,
    }
    print(json.dumps(line))
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def other_configs(torch, _lib, engine, synthetic, numeric, peaks, dev):
    """Short side measurements of BASELINE configs[2] (inference CNN+DLT forward, B=512) and configs[3] (fused warp + L1 on
    the full 320x240 grid, B=64) — reported next to the headline, not as the headline."""
    import ctypes
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for other, label in (("fp32", "configs[1] in the fp32 CUDA-core mode (UDH_NUMERIC_FP32)"),
                         ("bf16", "configs[1] in single-pass bf16 (UDH_NUMERIC_BF16: throughput mode, not parity-certified)"),
                         ("bf16x3", "configs[1] in the two-limb tensor-core mode (UDH_NUMERIC_BF16X3, parity-certified)")):
        if other == numeric:
            continue
        try:
            eng = engine.HomographyEngine(PER_GPU_BATCH, numeric=other, seed=0, loss_type="h_loss", lr=5e-4, device=dev)
            bs = [synthetic.make_batch(PER_GPU_BATCH, seed=900 + i, device=dev) for i in range(2)]
            for i in range(3):
                eng.train_step(bs[i % 2])
            e0, e1 = ev(), ev(); torch.cuda.synchronize(); e0.record()
            n = 5 if other == "fp32" else 20
            for i in range(n):
                eng.train_step(bs[i % 2])
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n
            out[label] = {"pairs_per_s": PER_GPU_BATCH / (ms * 1e-3), "ms_per_step": ms}
            if other != "fp32":
                out[label]["parity"] = parity_check(torch, engine, other, dev)
            del eng, bs
            torch.cuda.empty_cache()
        except Exception as e:
            out[label + " error"] = repr(e)[:200]
    try:
        B3 = 512
        eng = engine.HomographyEngine(B3, numeric=numeric, seed=0, device=dev)
        b = synthetic.make_batch(B3, seed=77, device=dev)
        h4p = torch.empty(B3, 8, device=dev); H = torch.empty(B3, 9, device=dev)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

        def fwd():
            _lib.check(_lib.lib.udh_cnn_fwd(p(eng.params), p(b["I1_aug"]), p(b["I2_aug"]), p(h4p), p(eng.ws), eng.ws_bytes, B3, 128, 0, 0, eng.numeric, st), "cnn_fwd")
            _lib.check(_lib.lib.udh_dlt_fwd(p(b["pts1"]), p(h4p), p(H), B3, st), "dlt")
        for _ in range(3):
            fwd()
        e0, e1 = ev(), ev(); torch.cuda.synchronize(); e0.record()
        n = 10
        for _ in range(n):
            fwd()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out["configs[2] inference CNN+DLT forward, B=512"] = {"pairs_per_s": B3 / (ms * 1e-3), "ms_per_batch": ms,
                                                               "tflops_algorithmic": FWD_FLOP_PER_PAIR * B3 / (ms * 1e-3) / 1e12,
                                                               "frac_of_bf16_peak": FWD_FLOP_PER_PAIR * B3 / (ms * 1e-3) / 1e12 / peaks["bf16_tflops"]}
        del eng, b
        torch.cuda.empty_cache()
    except Exception as e:                                     # side measurement only
        out["configs[2] error"] = repr(e)[:200]
    try:
        B4, Hh, W = 64, 240, 320
        nb = 4                                                 # 4 x 39.3 MB of inputs rotate through the 126 MB L2
        g = torch.Generator(device=dev).manual_seed(5)
        src = [torch.randn(B4, Hh, W, 1, device=dev, generator=g) for _ in range(nb)]
        tgt = [torch.randn(B4, Hh, W, 1, device=dev, generator=g) for _ in range(nb)]
        pts = torch.tensor([[96., 56., 224., 56., 224., 184., 96., 184.]], device=dev).repeat(B4, 1).contiguous()
        hh = (torch.rand(B4, 8, device=dev, generator=g) * 20 - 10).contiguous()
        Hm = torch.empty(B4, 9, device=dev); sums = torch.zeros(8, device=dev, dtype=torch.float64)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.lib.udh_dlt_fwd(p(pts), p(hh), p(Hm), B4, st), "dlt")

        def warp(i):
            _lib.check(_lib.lib.udh_warp_loss_fwd_ex(p(src[i % nb]), 1, Hh, W, p(Hm), p(tgt[i % nb]), None, 0, W, Hh, None, p(sums), 0, B4, st), "warp")
        for i in range(4):
            warp(i)
        e0, e1 = ev(), ev(); torch.cuda.synchronize(); e0.record()
        n = 40
        for i in range(n):
            warp(i)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        byts = 614400.0 * B4
        out["configs[3] fused warp+L1, full 320x240 grid, B=64"] = {
            "pairs_per_s": B4 / (ms * 1e-3), "us_per_launch": ms * 1e3,
            "roofline": {"bound": "hbm", "achieved": byts / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": byts / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": byts,
                         "l2_policy": "4 rotating input sets of 39.3 MB (157 MB > 126 MB L2)"}}
    except Exception as e:
        out["configs[3] error"] = repr(e)[:200]
    return out


def parity_check(torch, engine, numeric, dev, B=8, seed=0):
    """Measured live: pred_h4p and the mean corner error of `numeric` against the fp32 CUDA-core engine on the LARGE-OUTPUT
    parity weights (params.init_flat_large: |pred_h4p| of tens of pixels, like a trained net) and seeded synthetic inputs.
    The fp32 engine itself is pinned to the CPU oracle by tests/test_gpu_parity.py; the oracle comparison of this mode is
    tests/test_gpu_x3.py."""
    from unsuperviseddeephomographyral2018_b200 import params as P, synthetic
    try:
        flat = P.init_flat_large(seed)
        b = synthetic.make_batch(B, seed=4242, device=dev)
        e32 = engine.HomographyEngine(B, numeric="fp32", seed=None, device=dev); e32.load_flat(flat)
        em = engine.HomographyEngine(B, numeric=numeric, seed=None, device=dev); em.load_flat(flat)
        o32, om = e32.forward(b, train=False), em.forward(b, train=False)
        scale = o32["pred_h4p"].abs().max().item()
        d = (om["pred_h4p"] - o32["pred_h4p"]).abs().max().item()
        l32, lm = e32.losses_dict(o32), em.losses_dict(om)
        return {"fixture": "params.init_flat_large(seed=%d), synthetic.make_batch(B=%d)" % (seed, B), "max_abs_pred_h4p_px": scale,
                "max_err_pred_h4p_px": d, "rel_err_pred_h4p": d / scale,
                "mean_corner_error_px": {"fp32": l32["bounded_h_loss"], numeric: lm["bounded_h_loss"]},
                "abs_err_mean_corner_error_px": abs(l32["bounded_h_loss"] - lm["bounded_h_loss"]),
                "abs_err_h_loss_px": abs(l32["h_loss"] - lm["h_loss"]),
                "within_1e-3_px": bool(abs(l32["bounded_h_loss"] - lm["bounded_h_loss"]) <= 1e-3 and abs(l32["h_loss"] - lm["h_loss"]) <= 1e-3),
                "reference": "fp32 CUDA-core engine (UDH_NUMERIC_FP32) on identical inputs and weights"}
    except Exception as e:
        return {"error": repr(e)[:200]}


def _bf16_available(_lib):
    """The tensor-core mode is the default when this build carries it (probe: tiny forward returns OK, not UDH_ENOSUP)."""
    import ctypes
    import torch
    try:
        B = 2
        ws_bytes = _lib.lib.udh_cnn_workspace_bytes(B, 128, _lib.NUMERIC_BF16)
        ws = torch.empty(ws_bytes, device="cuda", dtype=torch.uint8)
        p = torch.zeros(_lib.lib.udh_param_total_floats(128), device="cuda")
        x = torch.zeros(B, 128, 128, device="cuda"); h = torch.zeros(B, 8, device="cuda")
        rc = _lib.lib.udh_cnn_fwd(ctypes.c_void_p(p.data_ptr()), ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(x.data_ptr()),
                                  ctypes.c_void_p(h.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws_bytes, B, 128, 0, 0, _lib.NUMERIC_BF16,
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return rc == 0
    except Exception:
        return False


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
