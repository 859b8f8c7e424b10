#!/usr/bin/env python
"""bench.py - headline benchmark of the hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU arm

metric   utterances/sec of a full training step (train.py:28-35 of the reference:
         zero_grad -> model.loss(batch) -> backward -> [all-reduce] -> clip(200) -> SGD step)
workload SURVEY.md §8d north-star config: global batch B=64, T=1000 frames, F=80 features,
         28 symbols + blank, conv [[32,5,8,2],[32,5,8,2]], 5-layer biGRU-1024 (84.9 M parameters),
         synthetic data, random-init weights, dropout 0.
value    device-timed (CUDA events) with the input batch already resident in HBM.
e2e      the same step through the public API with HOST numpy inputs: every step pads its
         batch into pinned memory, copies it to the device and reads the loss back, all inside the
         timed region.  `value` uses the input pipeline a training loop would use
         (loader.BatchPrefetcher: the worker thread stages batch i+1 on a copy stream while step i
         computes, so K timed steps still contain K host->device copies); `value_no_prefetch` is
         the reference's own loop shape, `model.loss((inputs, labels))` collating on the training
         thread.
outputs  `--dump-outputs DIR` writes what the last device-timed step computed (dump_outputs);
         the inputs and initial weights are seeded, so two builds can be compared output for
         output.
Under torchrun (N>1) the global batch is sharded B/N per rank (strong scaling), gradients are
summed over ranks with NCCL all-reduces (per GRU layer, overlapped with backward); time is the max
over ranks.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL_CFG = {"dropout": 0.0,
             "encoder": {"conv": [[32, 5, 8, 2], [32, 5, 8, 2]],
                         "rnn": {"dim": 1024, "bidirectional": True, "layers": 5}}}
GLOBAL_B, T_IN, F_IN, VOCAB = 64, 1000, 80, 28
WORKLOAD = "LibriSpeech-clean-100 CTC: 5-layer biGRU-1024, |V|=29, B=64, T=1000, 80 feat (synthetic)"
METRIC = "utterances/sec (training step, B=64,T=1000,80-feat)"


def bench_config(n_gpus):
    """`config` of the JSON line: identical for this repo's arm and the reference arm."""
    return {"workload": WORKLOAD, "global_batch": GLOBAL_B, "seq_len": T_IN,
            "parallelism": "dp%d" % n_gpus,
            "l2": "no flush: one step touches ~10 GB of activations, far above the 126 MB L2"}


_T0 = time.perf_counter()


def _log(msg):
    if os.environ.get("SB_BENCH_VERBOSE"):
        sys.stderr.write("[bench %.1fs] %s\n" % (time.perf_counter() - _T0, msg))
        sys.stderr.flush()


def synth_batch(nutt, seed=0):
    rng = np.random.RandomState(seed)
    inputs = [rng.randn(T_IN, F_IN).astype(np.float32) for _ in range(GLOBAL_B)]
    labels = [rng.randint(0, VOCAB, size=rng.randint(40, 121)).tolist() for _ in range(GLOBAL_B)]
    return inputs[:nutt], labels[:nutt]


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, from the committed
# `ncu --set full` captures of this same workload (profiles/r02_summary.md; B=64 per GPU)
NCU_TRAFFIC_BYTES = {"gru_bwd": 793.56e6 + 215.58e6, "gru_fwd": 409.71e6 + 661.25e6,
                     "gemm_bf16_tn": 172.35e6 + 353.05e6, "ctc_fwd_bwd": 3.13e6}


def flops_per_step(nutt):
    """Algorithmic FLOPs of one training step for `nutt` utterances (SURVEY §8d: 126.7 GF/utt)."""
    return 126.7e9 * nutt


# ------------------------------------------------------------------------------------------------
# clocks sampling (recipe: /opt/skills/guides/B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx = [], []
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm restated over torch CPU ops (oracle/model_ref.py)
# ------------------------------------------------------------------------------------------------
def cpu_step_time(nutt, iters, warm, threads, layers=None):
    from oracle.model_ref import RefCTC
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    cfg = MODEL_CFG
    if layers is not None:
        cfg = json.loads(json.dumps(MODEL_CFG))
        cfg["encoder"]["rnn"]["layers"] = layers
    m = RefCTC(F_IN, VOCAB, cfg)
    inputs, labels = synth_batch(nutt)
    x = torch.from_numpy(np.stack(inputs))
    flat = torch.tensor([t for l in labels for t in l], dtype=torch.int32)
    llen = torch.tensor([len(l) for l in labels], dtype=torch.int32)
    opt = torch.optim.SGD(m.parameters(), lr=1e-3, momentum=0.0)
    times = []
    for i in range(warm + iters):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = m.loss(x, flat, llen)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 200)
        opt.step()
        _ = loss.item()
        if i >= warm:
            times.append(time.perf_counter() - t0)
    return times


def host_cores():
    ncpu = os.cpu_count() or 1
    try:
        ncpu = min(ncpu, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return ncpu


def pick_threads(nutt=GLOBAL_B):
    """Thread count for the CPU arm: the fastest of all power-of-two candidates UP TO EVERY host
    core, probed on the full batch with a 1-layer model (all hardware threads is often not the
    fastest for the T'-serial GRU on a many-core host, so the baseline gets the best setting
    rather than the largest; the probe stops once a candidate is 1.5x slower than the best)."""
    ncpu = host_cores()
    cands = sorted({c for c in (8, 16, 32, 64, 128, 256) if c < ncpu} | {ncpu})
    best, best_t = cands[0], None
    for c in cands:
        t = sum(cpu_step_time(nutt, 1, 0, c, layers=1))
        _log("cpu probe: %d threads -> %.2f s" % (c, t))
        if best_t is None or t < best_t:
            best, best_t = c, t
        elif t > 1.5 * best_t:
            break      # oversubscription only gets worse
    return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = pick_threads()
    # The metric's own configuration: the FULL B=64 minibatch per step (one step is ~10-20 s of
    # host time, so the warm-up is capped at 1 step; the cap is stated in the line).
    nutt = GLOBAL_B
    steps = args.steps
    warm = max(0, min(args.warmup, 1))
    times = cpu_step_time(nutt, steps, warm, threads)
    total = sum(times)
    val = nutt * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC,
        "value": val, "unit": "utt/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "steps_timed": len(times), "warmup_done": warm,
        "warmup_cap": "full B=64 batch per step; warm-up capped at 1 step "
                      "(one CPU step is 10-20 s)",
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": bench_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": "utt/s", "cores": threads,
                         "host_cores": host_cores(), "kind": "port",
                         "sample": "the full B=%d batch per step, %d warm-up + %d timed steps "
                                   "(oracle/model_ref.py: the ATen CPU conv+GRU+fc+ctc_loss "
                                   "fwd+bwd+clip+SGD the reference's train.py:28-35 runs on the "
                                   "host; /root/reference is not present on the GPU box and its "
                                   "warp-ctc dependency is un-vendored, so the reference's own "
                                   "classes cannot be driven here)" % (nutt, warm, len(times))},
        "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# this repo
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from speech_b200 import _lib, ops
    from speech_b200.models import CTC
    from speech_b200.optim import FlatSGD

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert GLOBAL_B % world == 0
    nutt = GLOBAL_B // world

    torch.manual_seed(0)
    model = CTC(F_IN, VOCAB, MODEL_CFG).cuda()
    model.set_train()
    # clip(200) + SGD(lr 1e-3, momentum 0) of train.py:32-35,95-97, fused over flat buffers;
    # step() also completes the data-parallel gradient all-reduce (per-layer buckets started
    # during backward, the remainder here)
    opt = FlatSGD(model, lr=1e-3, momentum=0.0, max_grad_norm=200.0, world_size=world)
    inputs, labels = synth_batch(GLOBAL_B)
    inputs = inputs[rank * nutt:(rank + 1) * nutt]
    labels = labels[rank * nutt:(rank + 1) * nutt]
    batch = (tuple(inputs), tuple(labels))
    x_dev, y, x_lens, y_lens = model.collate(*batch)     # device-resident copy of the inputs
    x_host = x_dev                                        # (sizes only, for the byte counts)
    last = {}                                             # results of the latest step_device()

    def step_device():
        opt.zero_grad(set_to_none=False)
        out = model.forward_impl(x_dev)
        loss = model.ctc_loss(out, y, x_lens, y_lens)
        loss.backward()
        last["grad_norm"] = opt.step()
        # detached: holding the graph would keep this step's activations alive into the next
        last["logits"], last["loss"] = out.detach(), loss.detach()
        return loss

    def step_e2e():
        opt.zero_grad(set_to_none=False)
        loss = model.loss(batch)          # host numpy in: pinned staging + H2D inside
        loss.backward()
        opt.step()
        return loss.item()                # D2H read of the step's result

    staged = {}

    def step_e2e_prefetch():
        if "it" not in staged:
            import itertools
            from speech_b200.loader import BatchPrefetcher
            staged["pf"] = BatchPrefetcher(model, itertools.repeat(batch))
            staged["it"] = iter(staged["pf"])
        opt.zero_grad(set_to_none=False)
        loss = model.loss(next(staged["it"]))   # staged by the worker thread during the last step
        loss.backward()
        opt.step()
        return loss.item()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm):
        for _ in range(warm):
            fn()
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    if args.profile:
        for _ in range(max(1, args.warmup)):
            step_device()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for _ in range(args.steps):
            step_device()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profile_run": True, "steps": args.steps}))
        return

    # ---- device-resident value, with per-kernel CUDA events and clock sampling ----
    _log("model built; warm-up")
    for i in range(args.warmup):
        step_device()
        torch.cuda.synchronize()
        _log("warm-up step %d done" % i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.profile_begin()
    _lib.launch_count = 0
    ms_dev = timed(step_device, args.steps, 0)
    launches = _lib.launch_count
    prof = ops.profile_end()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, opt)
    loss_val = float(step_device().item())
    _log("device-timed region done: %.2f ms/step" % (ms_dev / args.steps))

    # ---- end to end through the public API ----
    ms_e2e_serial = timed(step_e2e, args.steps, 2)
    _log("e2e (no prefetch) region done: %.2f ms/step" % (ms_e2e_serial / args.steps))
    ms_e2e = timed(step_e2e_prefetch, args.steps, 3)
    staged["pf"].close()
    _log("e2e region done: %.2f ms/step" % (ms_e2e / args.steps))

    # ---- data-parallel correctness (N > 1): replicas must stay bit-identical, and the sharded
    # gradient must equal the single-rank gradient of the global batch ----
    dp = dp_check(model, opt, dev, world, rank) if world > 1 else None
    weak = weak_scaling(model, opt, world, rank, dev, timed) if world > 1 else None
    rnnt_dp = rnnt_dp_measurement(world, rank, timed) if world in (2, 4) else None

    if rank == 0:
        utt = GLOBAL_B * args.steps
        value = utt / (ms_dev * 1e-3)
        # the input pipeline that is faster at this N is the headline end-to-end number (the
        # prefetcher's worker thread competes with the launch thread when the step is short)
        e2e_pipeline = "loader.BatchPrefetcher, 1 batch ahead on a copy stream"
        if ms_e2e_serial < ms_e2e:
            ms_e2e, ms_e2e_serial = ms_e2e_serial, ms_e2e
            e2e_pipeline = "model.loss(batch): collate + pinned staging + H2D on the training thread"
        e2e = utt / (ms_e2e * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else \
            "fallback (B200_PROFILING.md sustained)"
        kernels = {}
        for name, (n, ms, fl) in prof.items():
            kernels[name] = {"launches_per_step": n / args.steps, "ms_per_step": ms / args.steps,
                             "tflops": (fl / 1e12) / (ms * 1e-3) if ms > 0 else None,
                             "frac_of_peak": ((fl / 1e12) / (ms * 1e-3)) / peak_tf if ms > 0 else None}
        dom = max(prof.items(), key=lambda kv: kv[1][1])[0] if prof else None
        roof = None
        if dom:
            n, ms, fl = prof[dom]
            ach = (fl / 1e12) / (ms * 1e-3)
            roof = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": peak_tf,
                    "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "traffic": NCU_TRAFFIC_BYTES.get(dom) if nutt == GLOBAL_B else None,
                    "traffic_source": "profiles/r02_summary.md (ncu --set full, bytes per launch)",
                    "peak_source": peak_src,
                    "avg_launch_ms": ms / n if n else None,
                    "note": "per-step latency-bound recurrence (see DESIGN.md 4.2): tensor pipe "
                            "and HBM are both far from saturated by construction at B=64"}
        line = {
            "metric": METRIC,
            "value": value, "unit": "utt/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": bench_config(world),
            "notes": {"precision": "bf16 tensor-core operands, fp32 accumulate/state/master weights"},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "utt/s", "ms_per_step": ms_e2e / args.steps,
                    "value_other_pipeline": utt / (ms_e2e_serial * 1e-3),
                    "input_pipeline": e2e_pipeline,
                    "h2d_bytes_per_step": int(x_host.numel() * 4 + y.numel() * 4 + 8 * nutt) * world,
                    "d2h_bytes_per_step": 4 * world},
            "gpu_launches": launches,
            "gru_cluster": int(_lib.load().sb_debug_gru_cluster(0)),
            "loss": loss_val,
            "step_tflops": flops_per_step(GLOBAL_B) / 1e12 / (ms_dev / args.steps * 1e-3),
            "roofline": roof,
            "kernels": kernels,
        }
        if dp is not None:
            line["dp_check"] = dp
        if weak is not None:
            line["secondary"] = {"weak_scaling": weak}
        if rnnt_dp is not None:
            line["secondary"]["rnnt_dp"] = rnnt_dp
        if world == 1 and not args.no_secondary:
            line["secondary"] = secondary_measurements(model, batch, dev)
        if world == 1 and not args.no_cpu_baseline:
            threads = pick_threads()
            nb = GLOBAL_B
            times = cpu_step_time(nb, 1, 1, threads)
            line["cpu_baseline"] = {
                "value": nb * len(times) / sum(times), "unit": "utt/s", "cores": threads,
                "host_cores": host_cores(), "kind": "port",
                "sample": "the full B=%d batch, 1 warm-up + 1 timed step "
                          "(oracle/model_ref.py on the host cores)" % nb}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_SAMPLE = 1 << 20   # entries of the flat parameter and gradient vectors --dump-outputs writes


def dump_outputs(d, last, opt):
    """--dump-outputs: what the last timed step computed (rank 0's shard when N > 1), as float32
    .npy files under `d`: the summed CTC loss, the gradient norm clip(200) saw, the logits, and a
    fixed sample (seed 0, the same indices in every run) of the updated parameters and of the
    gradients - the full flat vectors are 340 MB each."""
    os.makedirs(d, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(opt.n, min(DUMP_SAMPLE, opt.n), replace=False))
    idx = torch.from_numpy(idx).to(opt.flat_p.device)
    arrays = {"loss": last["loss"], "grad_norm": last["grad_norm"], "logits": last["logits"],
              "params_sample": opt.flat_p[idx], "grads_sample": opt.flat_g[idx]}
    for name, t in arrays.items():
        np.save(os.path.join(d, name + ".npy"), t.detach().float().cpu().numpy())


def dp_check(model, opt, dev, world, rank):
    """N > 1 only.  (1) after the timed steps every rank must hold bit-identical parameters (same
    reduced gradients, same clip, same update): compare a float64 checksum and the first 1024
    words across ranks.  (2) on a small model, the all-reduced gradient of the sharded minibatch
    must equal the gradient rank 0 computes for the WHOLE minibatch alone (sum reduction makes
    this exact up to fp32 add order)."""
    import torch.distributed as dist
    from speech_b200 import ops
    from speech_b200.models import CTC
    from speech_b200.optim import FlatSGD
    out = {}
    chk = torch.stack([opt.flat_p.double().sum(), opt.flat_p[:1024].double().abs().sum()])
    allc = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    allc = torch.stack(allc)
    out["param_checksum_spread"] = float((allc.max(0).values - allc.min(0).values).abs().max())
    out["replicas_identical"] = out["param_checksum_spread"] == 0.0
    # (2) sharded vs single-rank gradients, small config, 16 utterances
    cfg = {"dropout": 0.0, "encoder": {"conv": [[8, 5, 8, 2], [8, 5, 8, 2]],
                                       "rnn": {"dim": 64, "bidirectional": True, "layers": 2}}}
    rng = np.random.RandomState(1)
    nb = 16
    inputs = [rng.randn(200, F_IN).astype(np.float32) for _ in range(nb)]
    labels = [rng.randint(0, VOCAB, size=12).tolist() for _ in range(nb)]
    torch.manual_seed(1)
    small = CTC(F_IN, VOCAB, cfg).cuda()
    small.set_train()
    sopt = FlatSGD(small, lr=1e-3, world_size=world)
    per = nb // world
    sopt.zero_grad()
    small.loss((tuple(inputs[rank * per:(rank + 1) * per]),
                tuple(labels[rank * per:(rank + 1) * per]))).backward()
    sopt.all_reduce()
    g_dp = sopt.flat_g.clone()
    ops.set_grad_ready_hook(None)
    sopt2 = FlatSGD(small, lr=1e-3, world_size=1)
    sopt2.zero_grad()
    small.loss((tuple(inputs), tuple(labels))).backward()
    torch.cuda.synchronize()
    rel = ((g_dp - sopt2.flat_g).norm() / sopt2.flat_g.norm()).item()
    out["sharded_vs_single_rank_grad_rel_l2"] = rel
    # restore the hooks of the benchmark's optimizer
    ops.set_grad_sink(True)
    if world > 1:
        ops.set_grad_ready_hook(opt._grads_ready, guard=opt._guard_second_backward)
    return out


def rnnt_dp_measurement(world, rank, timed):
    """BASELINE.json configs[4] data-parallel: the B=32 RNN-T minibatch sharded over the ranks,
    gradients all-reduced by FlatSGD (same machinery as the headline step)."""
    from speech_b200 import ops
    from speech_b200.optim import FlatSGD
    per = 32 // world
    m, batch = rnnt_workload(per, rank * per)
    m.set_train()
    ops.set_grad_ready_hook(None)
    opt = FlatSGD(m, lr=1e-4, momentum=0.0, max_grad_norm=200.0, world_size=world)

    def step():
        opt.zero_grad()
        loss = m.loss(batch)
        loss.backward()
        opt.step()
        return loss

    steps = 3
    ms = timed(step, steps, 2)
    ops.set_grad_ready_hook(None)
    return {"global_batch": 32, "world": world, "ms_per_step": ms / steps,
            "utt_per_s": 32 * steps / (ms * 1e-3)}


def weak_scaling(model, opt, world, rank, dev, timed):
    """N > 1 only: B=64 per rank (global batch 64 N), same step otherwise: shows the gradient
    all-reduce overlap separately from the chain-bound strong-scaling number."""
    inputs, labels = synth_batch(GLOBAL_B, seed=rank + 1)
    x_dev, y, x_lens, y_lens = model.collate(tuple(inputs), tuple(labels))

    def step():
        opt.zero_grad(set_to_none=False)
        loss = model.ctc_loss(model.forward_impl(x_dev), y, x_lens, y_lens)
        loss.backward()
        opt.step()
        return loss

    steps = 5
    ms = timed(step, steps, 2)
    return {"per_rank_batch": GLOBAL_B, "global_batch": GLOBAL_B * world,
            "ms_per_step": ms / steps, "utt_per_s": GLOBAL_B * world * steps / (ms * 1e-3)}


def secondary_measurements(model, batch, dev):
    """SURVEY.md section 8d secondary numbers, N=1 only (outside the timed regions):
       - CTC loss delta vs the reference model restated on the CPU (oracle/model_ref.py) with the
         SAME weights and inputs (8 utterances): the effect of the bf16 tensor-core operands;
       - CTC kernel-only delta: our kernel vs torch's CPU float64 CTC on OUR logits;
       - standalone CTC micro-benchmark at B=64, T=1000, V=29 (algorithmic bytes / time);
       - decode throughput: CTC.infer (prefix beam search on the GPU), beam 1 and 8."""
    from oracle.model_ref import RefCTC
    from speech_b200.functions.ctc import ctc_costs_and_grads
    out = {}
    inputs, labels = batch
    sub = (tuple(inputs[:8]), tuple(labels[:8]))
    torch.set_num_threads(min(16, os.cpu_count() or 1))

    def loss_pair(m):
        with torch.no_grad():
            mine = float(m.loss(sub).item())
            x, y, x_lens, y_lens = m.collate(*sub)
            lg = m.forward_impl(x)
        ref = RefCTC(F_IN, VOCAB, MODEL_CFG)
        ref.load_from_dropin({k: v.detach().float().cpu() for k, v in m.state_dict().items()})
        with torch.no_grad():
            theirs = float(ref.loss(torch.from_numpy(np.stack(sub[0])), y, y_lens).item())
        return mine, theirs, lg, y, y_lens

    # ---- loss delta on the north-star state: torch.manual_seed(0) random-init weights ----
    from speech_b200.models import CTC
    torch.manual_seed(0)
    fresh = CTC(F_IN, VOCAB, MODEL_CFG).cuda()
    fresh.set_eval()
    ours, ref_loss, logits, y, y_lens = loss_pair(fresh)
    out["ctc_loss_ours_8utt"] = ours
    out["ctc_loss_cpu_reference_8utt"] = ref_loss
    out["ctc_loss_rel_delta"] = abs(ours - ref_loss) / abs(ref_loss)
    del fresh
    # ---- same comparison on the weights the timed SGD steps above left behind (noise labels at
    # lr 1e-3 drive the recurrent weights up, which amplifies the bf16 operand rounding) ----
    t_ours, t_ref, _, _, _ = loss_pair(model)
    out["ctc_loss_rel_delta_after_timed_steps"] = abs(t_ours - t_ref) / abs(t_ref)
    # ---- the same loss in PARITY MODE (split-bf16 GEMMs + fp32 recurrence, inference only): the
    # measuring stick for the bf16 operand path, on the trained weights as well ----
    for tag, mm in (("seed0", None), ("after_timed_steps", model)):
        if mm is None:
            torch.manual_seed(0)
            mm = CTC(F_IN, VOCAB, MODEL_CFG).cuda()
        was = mm.training
        mm.set_eval()
        mm.parity_mode = True
        p_ours, p_ref, _, _, _ = loss_pair(mm)
        mm.parity_mode = False
        if was:
            mm.set_train()
        out["ctc_loss_rel_delta_parity_mode_" + tag] = abs(p_ours - p_ref) / abs(p_ref)
    # ---- kernel-only delta on our logits ----
    lg = logits.detach().double().cpu()
    lp = torch.log_softmax(lg, 2).transpose(0, 1)
    T = lg.shape[1]
    c64 = torch.nn.functional.ctc_loss(lp, y.long(), torch.full((8,), T, dtype=torch.long),
                                       y_lens.long(), blank=VOCAB, reduction="sum").item()
    out["ctc_kernel_rel_delta_vs_f64"] = abs(ours - c64) / abs(c64)
    # ---- standalone CTC micro-benchmark ----
    rng = np.random.RandomState(0)
    acts = torch.from_numpy(rng.randn(GLOBAL_B, T_IN, VOCAB + 1).astype(np.float32)).to(dev)
    llen = torch.tensor([len(l) for l in labels], dtype=torch.int32)
    flat = torch.tensor([t for l in labels for t in l], dtype=torch.int32)
    alen = torch.full((GLOBAL_B,), T_IN, dtype=torch.int32)
    for _ in range(3):
        ctc_costs_and_grads(acts, flat, alen, llen)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ctc_costs_and_grads(acts, flat, alen, llen)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    algo = 2.0 * GLOBAL_B * T_IN * (VOCAB + 1) * 4
    out["ctc_standalone"] = {"shape": [GLOBAL_B, T_IN, VOCAB + 1], "ms": ms,
                             "algorithmic_bytes": algo, "GB_per_s": algo / ms / 1e6,
                             "note": "includes the host->device copy of the label arrays; bound "
                                     "by the T-step dependency chain (float64 lattice)"}
    # ---- decode throughput ----
    model.set_eval()
    for beam in (1, 8):
        model.infer(batch, beam_size=beam)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.infer(batch, beam_size=beam)
        torch.cuda.synchronize()
        out["infer_beam%d_utt_per_s" % beam] = len(inputs) / (time.perf_counter() - t0)
    model.set_train()
    # ---- featuriser (SURVEY 8f rank 2): 64 utterances of 10 s int16 PCM at 16 kHz -> the
    # (64, 1000, 161) normalised log-spectrogram, host PCM in, device features out ----
    try:
        from oracle.specgram_ref import log_specgram as ref_specgram
        from speech_b200.features import log_specgram_batch
        rng = np.random.RandomState(1)
        audios = [(rng.randn(160160) * 3000).astype(np.int16) for _ in range(GLOBAL_B)]
        mean = np.zeros(161, np.float32)
        std = np.ones(161, np.float32)
        feats, n_frames = log_specgram_batch(audios, 16000, mean=mean, std=std)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            feats, n_frames = log_specgram_batch(audios, 16000, mean=mean, std=std)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 5
        t0 = time.perf_counter()
        refs = [ref_specgram(a, 16000) for a in audios[:4]]
        dt_cpu = (time.perf_counter() - t0) / 4
        err = max(float(np.abs(feats[e, :n_frames[e]].cpu().numpy() - refs[e]).max())
                  for e in range(4))
        out["featuriser"] = {"utt_per_s": GLOBAL_B / dt, "ms_per_batch_of_64x10s": dt * 1e3,
                             "frames": int(n_frames[0]), "cpu_oracle_utt_per_s_1core": 1.0 / dt_cpu,
                             "max_abs_err_vs_f64_oracle": err,
                             "note": "host int16 PCM in (pinned copy + H2D inside), device "
                                     "features out"}
    except Exception as e:      # never let a secondary number take the bench line down
        out["featuriser"] = {"error": repr(e)}
    try:
        out["other_configs"] = other_config_measurements(dev)
    except Exception as e:
        out["other_configs"] = {"error": repr(e)}
    return out


def _time_train_steps(m, batch, steps=3, warm=2):
    """utt/s of zero_grad -> loss -> backward -> clip + SGD on one GPU (device events)"""
    from speech_b200.optim import FlatSGD
    m.set_train()
    opt = FlatSGD(m, lr=1e-4, momentum=0.0, max_grad_norm=200.0)

    def step():
        opt.zero_grad()
        loss = m.loss(batch)
        loss.backward()
        opt.step()
        return loss
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "utt_per_s": len(batch[0]) / (ms * 1e-3), "loss": float(loss.item())}


WSJ_CONV = [[32, 5, 8, 2], [32, 5, 8, 2]]


def other_config_measurements(dev):
    """The other workloads BASELINE.json `configs` names (synthetic data, random-init weights,
    1 GPU; outside the timed regions of the headline metric):
      [1] TIMIT CTC: 4-layer biGRU-512, 80 features, 61 phones, B=32 (training step)
      [3] WSJ attention model: conv + 3x biGRU-512 encoder (training step B=16; greedy and beam-8
          decode through the device-resident loops)
      [4] RNN-Transducer: 3x biGRU-1024 encoder + GRU-1024 prediction net (the reference class
          ties both dims, transducer_model.py:20-25), B=32, fused joint + lattice loss"""
    from speech_b200.models import CTC, Seq2Seq, Transducer
    out = {}
    rng = np.random.RandomState(2)
    # ---- configs[1]: TIMIT CTC ----
    torch.manual_seed(0)
    cfg = {"dropout": 0.0, "encoder": {"conv": WSJ_CONV,
                                       "rnn": {"dim": 512, "bidirectional": True, "layers": 4}}}
    m = CTC(F_IN, 61, cfg).cuda()
    batch = (tuple(rng.randn(300, F_IN).astype(np.float32) for _ in range(32)),
             tuple(rng.randint(0, 61, size=rng.randint(20, 40)).tolist() for _ in range(32)))
    out["timit_ctc_bigru512x4_B32_T300"] = _time_train_steps(m, batch)
    del m
    # ---- configs[3]: WSJ attention model ----
    torch.manual_seed(0)
    cfg = {"dropout": 0.0, "encoder": {"conv": WSJ_CONV,
                                       "rnn": {"dim": 512, "bidirectional": True, "layers": 3}},
           "decoder": {"embedding_dim": 512, "layers": 1, "log_t": True}}
    V = 32
    m = Seq2Seq(F_IN, V, cfg).cuda()
    lab = lambda: [V - 1] + rng.randint(0, V - 2, size=rng.randint(60, 100)).tolist() + [V - 2]
    batch = (tuple(rng.randn(800, F_IN).astype(np.float32) for _ in range(16)),
             tuple(lab() for _ in range(16)))
    res = _time_train_steps(m, batch)
    m.set_eval()
    m.infer(batch, max_len=100)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.infer(batch, max_len=100)
    torch.cuda.synchronize()
    res["greedy_decode_utt_per_s_B16_100steps"] = 16 / (time.perf_counter() - t0)
    one = ((batch[0][0],), (batch[1][0],))
    m.beam_search(one, beam_size=8, max_len=100)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for e in range(4):
        m.beam_search(((batch[0][e],), (batch[1][e],)), beam_size=8, max_len=100)
    torch.cuda.synchronize()
    res["beam8_decode_utt_per_s_100steps"] = 4 / (time.perf_counter() - t0)
    out["wsj_seq2seq_bigru512x3_B16_T800"] = res
    del m
    # ---- configs[4]: RNN-Transducer ----
    out["rnnt_bigru1024x3_pred1024_B32_T1000"] = _time_train_steps(*rnnt_workload(32, 0))
    return out


def rnnt_workload(nutt, first):
    """(model, batch) of the RNN-T configuration, utterances first .. first+nutt of a B=32 batch"""
    from speech_b200.models import Transducer
    torch.manual_seed(0)
    cfg = {"dropout": 0.0, "encoder": {"conv": WSJ_CONV,
                                       "rnn": {"dim": 1024, "bidirectional": True, "layers": 3}},
           "decoder": {"embedding_dim": 256, "layers": 1}}
    m = Transducer(F_IN, VOCAB, cfg).cuda()
    rng = np.random.RandomState(3)
    inputs = [rng.randn(T_IN, F_IN).astype(np.float32) for _ in range(32)]
    labels = [rng.randint(0, VOCAB, size=rng.randint(40, 100)).tolist() for _ in range(32)]
    return m, (tuple(inputs[first:first + nutt]), tuple(labels[first:first + nutt]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the secondary measurements (loss delta vs the CPU reference model, "
                         "standalone CTC micro-benchmark, decode throughput)")
    ap.add_argument("--profile", action="store_true",
                    help="profiling run (ncu): 1 warm-up + --steps device steps, nothing else; "
                         "prints no benchmark value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                         "(float32: loss, grad_norm, logits, and a seeded sample of the updated "
                         "parameters and of the gradients); the inputs are the same in every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.profile):
        ap.error("--dump-outputs writes the outputs of this repo's timed steps: it takes neither "
                 "--impl reference nor --profile")
    if args.warmup < 3 and args.impl == "ours" and not args.profile:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
