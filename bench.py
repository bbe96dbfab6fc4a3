#!/usr/bin/env python
"""bench.py -- train images/sec of an EAD-GAN training step on N B200s, the dominant kernel's roofline and the
reference's CPU path as baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config celeba|dsprites|colored] [--batch B_per_gpu]
                  [--global-batch B] [--impl ours|reference] [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
              --master-port P bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json `configs`):
  celeba   (default)  CelebA 64x64 G + D/Q step, three phases, three Adams (celebA/EAD-GAN_celebA.py:296-401);
                      1024 images per GPU, weak scaling (configs[3]); --batch sweeps configs[4];
                      --global-batch fixes the GLOBAL batch instead (strong scaling, e.g. 1024 over 8 GPUs)
  dsprites            dSprites rp.py stage-2 step, batch 256 (configs[1]; dSprites/rp.py:362-482)
  colored             colored-dSprites rp_color.py step, GLOBAL batch 512 split over the GPUs (configs[2], strong
                      scaling; colored_dSprites/rp_color.py:362-516)

One JSON line on rank 0.  `value`: images resident in HBM, CUDA-event timed, barrier + synchronize on both sides,
max over ranks.  `e2e`: the same step called with the HOST (pinned) image batch -- its H2D copy and the D2H read of
the losses inside the timed region; the latent draws (z, code, labels) are sampled on the device inside the step
(csrc/sample.cu, replacing the reference's host NumPy draws), so nothing else crosses PCIe.  `parity` (N = 1,
celeba): the first step at the TIMED batch size checked against the oracle outside the timed region.  `dp_parity`
(N > 1): the N-rank step against the single-device step on the same global batch.
Data is synthetic, weights random-init (no datasets / checkpoints offline).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # useful algorithmic GFLOP / image / step and ideal-fusion bf16 activation bytes / image / step: SURVEY.md section 8d
    "celeba": {"metric": "train images/sec (G+D+E step, 64x64 CelebA)", "gflop": 18.865, "mb": 20.2, "batch": 1024,
               "workload": "CelebA EAD-GAN_celebA 64x64 RGB G/D step, 3 phases + 3 Adam (BASELINE configs[3]/[4])"},
    "dsprites": {"metric": "train images/sec (D + G/E step, 64x64 dSprites rp.py)", "gflop": 0.489, "mb": 4.56, "batch": 256,
                 "workload": "dSprites rp.py 64x64 grayscale encoder + G/D step, 2 phases + 2 Adam (BASELINE configs[1])"},
    "colored": {"metric": "train images/sec (D + G/E step, 64x64 colored dSprites rp_color.py)", "gflop": 0.546, "mb": 4.93,
                "batch": 512, "workload": "colored_dSprites rp_color.py 64x64 RGB step, 2 phases + 2 Adam (BASELINE configs[2])"},
}


def ncu_traffic(entry_name):
    """DRAM bytes per launch of this entry point's kernel from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_summarize.py), or None when it was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f).get(entry_name)
        return None if t is None else {"bytes": t["dram_bytes_per_launch"], "capture": t["capture"],
                                       "tensor_pipe_pct": t.get("tensor_pipe_pct")}
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sust": p["bf16_tflops_sustained"],
                "src": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sust": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
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
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def config_block(args, world):
    """identical in both arms (`--impl ours` and `--impl reference`): it names the WORKLOAD, nothing about the arm"""
    c = CONFIGS[args.config]
    B, Bg = batch_sizes(args, world)
    return {"workload": c["workload"], "batch_per_gpu": B, "global_batch": Bg, "parallelism": f"dp{world}",
            "l2": "inputs + activations per step >> 126 MB L2 (no flush needed)" if Bg * c["mb"] > 512 else
                  "working set is L2-sized: a 256 MB buffer is overwritten between timed steps",
            "weights": "random-init seed 0", "latents": "z ~ N(0,1), code ~ U(-1,1), labels ~ randint, drawn per step"}


def batch_sizes(args, world):
    c = CONFIGS[args.config]
    if args.global_batch:
        Bg = args.global_batch
    elif args.batch:
        Bg = args.batch * world
    elif args.config == "colored":
        Bg = c["batch"]                       # configs[2]: 512 GLOBAL, data-parallel over 2 / 4 / 8 GPUs
    else:
        Bg = c["batch"] * world
    if Bg % world:
        raise SystemExit(f"bench.py: global batch {Bg} is not divisible by {world} GPUs")
    return Bg // world, Bg


def scaling_kind(args):
    return "strong" if (args.global_batch or (args.config == "colored" and not args.batch)) else "weak"


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline leg: the oracle restatement of the reference step (stock torch.nn, fp32) on the host
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference(config, batch, steps, warmup):
    from oracle import torch_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    rs = np.random.RandomState(0)
    if config == "celeba":
        st = O.build_celeba(seed=0, device="cpu")
        imgs = O.synth_celeba_images(batch, 0)
        run = lambda: O.step_celeba(st, imgs, O.sample_celeba(rs, batch), record=False)
    elif config == "dsprites":
        st = O.build_dsprites(seed=0, device="cpu")
        imgs = O.synth_dsprites_images(batch, 0)
        run = lambda: O.step_dsprites(st, imgs, O.sample_dsprites(rs, batch), record=False)
    else:
        st = O.build_dsprites(seed=0, device="cpu", colored=True)
        imgs = O.synth_dsprites_images(batch, 0)
        run = lambda: O.step_colored(st, imgs, O.sample_colored(rs, batch), record=False)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        run()
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
    med = statistics.median(times)
    return batch / med, med


def cpu_sample_batch(args):
    if args.cpu_batch:
        return args.cpu_batch
    return 16 if args.config == "celeba" else 128


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    Bs = cpu_sample_batch(args)
    ips, med = cpu_reference(args.config, Bs, max(1, args.steps), max(1, args.warmup))
    line = {"impl": "reference", "metric": c["metric"], "value": ips, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": scaling_kind(args), "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args, world),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": f"each timed step is the reference's full training step on a {Bs}-image sample of the "
                                       f"configured batch ({args.steps} steps after {args.warmup} warm-up; oracle/torch_oracle.py, "
                                       "pinned bit for bit to the executed reference scripts; the reference has no native code "
                                       "to compile). CPU images/s is flat in batch size (SURVEY.md section 6), so the sample "
                                       "rate is the rate at the full batch",
                             "device": "host CPU, stock torch (oneDNN), all host threads"},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _OUT.emit(json.dumps(line))


class _QuietStdout:
    """Everything written to fd 1 before the result (NCCL prints its version banner there, libraries may print
    warnings) goes to stderr, so that stdout carries exactly ONE line: the JSON result."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


_OUT = None


def main():
    global _OUT
    with _QuietStdout() as _OUT:
        _main()


# ---------------------------------------------------------------------------------------------------------------
# parity of the timed configuration (outside the timed region; the oracle is the checker, never the thing measured)
# ---------------------------------------------------------------------------------------------------------------
def parity_block(config, B, dev):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import step_util as U
    if config == "celeba":
        import gates
        out = gates.celeba_forced(dev, B, "bf16" if os.environ.get("EADGAN_PRECISION", "bf16") == "bf16" else "fp32",
                                  oracle_dtypes=(torch.float32,))
        ref, free = out["forced"][0], out["free"]
        names = U.grad_names(out["step"])
        rep = {"batch": B, "oracle": "oracle/torch_oracle.py on this GPU, stock torch fp32 (cuDNN/cuBLAS, TF32 off)",
               "loss_rel_err": {k: abs(out["losses"][k] - free["losses"][k]) / max(1.0, abs(free["losses"][k]))
                                for k in free["losses"]},
               "gate_flips": out["flips"], "gates": out["gates"], "phases": []}
        for ph in range(3):
            forced = U.phase_errors(names[ph], out["ours"][ph]["grads"], ref["phases"][ph]["grads"])
            unforced = U.phase_errors(names[ph], out["ours"][ph]["grads"], free["phases"][ph]["grads"])
            l2s = [v[1] for v in unforced.values() if isinstance(v[2], float)]
            cos = [v[2] for v in unforced.values() if isinstance(v[2], float)]
            rep["phases"].append({"forced_gates_worst_tensor_err": max(v[0] for v in forced.values()),
                                  "own_gates_worst_l2_rel": max(l2s), "own_gates_min_cosine": min(cos)})
        rep["bound"] = "2e-2 (north_star bf16): losses, and every gradient tensor max|a-b|/max|b| on common gates"
        rep["pass"] = bool(max(rep["loss_rel_err"].values()) <= 2e-2 and
                           all(p["forced_gates_worst_tensor_err"] <= 2e-2 for p in rep["phases"]))
        return rep
    run = U.run_pair_dsprites if config == "dsprites" else U.run_pair_colored
    ref, rec, losses, st, ours = run(dev, B, os.environ.get("EADGAN_PRECISION", "bf16"), oracle_dtype=torch.float32)
    names = U.dsprites_grad_names(ours)
    rep = {"batch": B, "oracle": "oracle/torch_oracle.py on this GPU, stock torch fp32 (cuDNN/cuBLAS, TF32 off)",
           "loss_rel_err": {k: abs(losses[k] - ref["losses"][k]) / max(1.0, abs(ref["losses"][k])) for k in ref["losses"]},
           "phases": []}
    for ph in range(2):
        errs = U.phase_errors(names[ph], rec[ph]["grads"], ref["phases"][ph]["grads"], U.DSPRITES_ZERO_GRAD)
        rep["phases"].append({"own_gates_worst_l2_rel": max(v[1] for v in errs.values() if isinstance(v[2], float)),
                              "own_gates_min_cosine": min(v[2] for v in errs.values() if isinstance(v[2], float))})
    rep["bound"] = "2e-2 on the losses; gradients by direction / L2 on each run's own gates"
    rep["pass"] = bool(max(rep["loss_rel_err"].values()) <= 2e-2)
    return rep


def build_step(config, dev, rank, B):
    """-> (step object taking host/device images + explicit draws, SampledStep drawing its latents on the device,
    list of R distinct host image batches (pinned), images-per-step)"""
    from eadgan_b200 import synthetic
    from eadgan_b200.sampling import DeviceSampler, SampledStep
    world = int(os.environ.get("WORLD_SIZE", "1"))
    Bg = B * world
    if config == "celeba":
        from eadgan_b200.steps.celeba import CelebAStep
        step = CelebAStep(seed=0, device=dev)
        host = [synthetic.celeba_images(Bg, i)[rank * B:(rank + 1) * B].contiguous().pin_memory() for i in range(2)]
    elif config == "dsprites":
        from eadgan_b200.steps.dsprites import DSpritesStep
        step = DSpritesStep(seed=0, device=dev)
        host = [synthetic.dsprites_images(Bg, i)[rank * B:(rank + 1) * B].contiguous().pin_memory() for i in range(2)]
    else:
        from eadgan_b200.steps.colored import ColoredDSpritesStep
        step = ColoredDSpritesStep(seed=0, device=dev)
        host = [synthetic.dsprites_images(Bg, i)[rank * B:(rank + 1) * B].contiguous().pin_memory() for i in range(2)]
    sampled = SampledStep(step, DeviceSampler(seed=1234, device=dev, row0=rank * B), config)
    return step, sampled, host


DUMP_SAMPLE = 1 << 20     # elements: a larger tensor is dumped as a seeded sample
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, losses, step):
    """What the last timed step hands its caller: the losses it returns and the model state it leaves behind (every
    floating-point parameter and buffer of the step's networks), as out_dir/<name>.npy in float32 (float64 where the
    state is float64).  A tensor of more than DUMP_SAMPLE elements is written flattened, as the same seeded sample of
    its elements on every run, so that the dumps of two builds compare element for element."""
    arrays = {k: v.detach().float().cpu().numpy().reshape(1) for k, v in losses.items()}
    for mname, m in sorted(vars(step).items()):
        if not isinstance(m, torch.nn.Module):
            continue
        for k, t in m.state_dict().items():
            if not t.is_floating_point():
                continue
            t = t.detach()
            if t.numel() > DUMP_SAMPLE:
                idx = np.sort(np.random.RandomState(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
                t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
            arrays[f"{mname}.{k}"] = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="celeba", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (weak scaling); default: the configuration's")
    ap.add_argument("--global-batch", type=int, default=0, help="fix the GLOBAL batch instead (strong scaling)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=0, help="image sample per CPU step (default 16 celeba / 128 dsprites)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity / dp_parity checks in front of the timing")
    ap.add_argument("--profile-out", default=None, help="write the per-entry-point time table here (json)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying "
                    "the captured whole-step CUDA graph")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the losses of the last timed step and the model state it left as "
                         "DIR/<name>.npy (tensors over 2^20 elements as a seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path (--impl ours); the reference arm writes nothing")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    from eadgan_b200 import _lib, parallel
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sm_100a path has no CPU fallback")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    parallel.init_from_env()
    precision = os.environ.get("EADGAN_PRECISION", "bf16")
    cfg = CONFIGS[args.config]
    B, Bg = batch_sizes(args, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- parity of the timed configuration, before anything is timed ----------------------------------------
    parity = dp_par = None
    if not args.no_parity:
        if world == 1:
            if B <= 2048:
                parity = parity_block(args.config, B, dev)
            else:
                parity = {"skipped": f"batch {B}: the stock-torch fp32 oracle keeps ~10 MB of activations per image; parity "
                                     "is checked at batches <= 2048 (tests/test_b1024_gpu.py and the default bench line)"}
        elif args.config == "celeba":
            from tools.dp_parity import dp_parity
            dp_par = dp_parity(B, dev, seed=0)
        from eadgan_b200 import tc
        tc.clear_pool()
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        barrier()

    eager_step, sampled, host = build_step(args.config, dev, rank, B)
    ablate = os.environ.get("EADGAN_DP_ABLATE", "")     # experiments: which exchange costs what (profiles/r02*_dp_ablation)
    if world > 1 and "grads" in ablate:
        parallel.detach(*eager_step.optimizers())       # no gradient all-reduce (replicas diverge: timing only)
    if world > 1 and "syncbn" in ablate:
        from eadgan_b200 import functional as _Fn
        _Fn.set_allreduce(None, 1)                       # BatchNorm statistics stay local (timing only)
    R = len(host)
    resident = [h.to(dev) for h in host]
    h2d_bytes = host[0].numel() * host[0].element_size()
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8) if Bg * cfg["mb"] <= 512 else None

    use_graph = not args.no_graph   # under DP the NCCL all-reduces (gradient buckets, SyncBN) are captured too
    step = sampled
    if use_graph:
        from eadgan_b200.graph import GraphedStep
        step = GraphedStep(sampled, [resident[0]], warmup=args.warmup)   # warm-up steps run inside, eagerly
    for i in range(args.warmup):
        step(resident[i % R])
    # ---- device-resident timing -------------------------------------------------------------------------------
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    k0 = _lib.lib().eadgan_kernel_launches()
    window = os.environ.get("EADGAN_PROFILE_WINDOW") == "1"   # ncu --profile-from-start off: only the timed steps
    if window:
        torch.cuda.profiler.start()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            last = step(resident[i % R])
        e1.record()
        torch.cuda.synchronize()
        ms_local = e0.elapsed_time(e1)
    else:   # small working set: overwrite an L2-sized buffer between steps, time every step on its own
        evs = []
        for i in range(args.steps):
            flush.fill_(i & 0xff)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last = step(resident[i % R])
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms_local = sum(a.elapsed_time(b) for a, b in evs)
    if window:
        torch.cuda.profiler.stop()
    launches = _lib.lib().eadgan_kernel_launches() - k0
    if use_graph:
        launches = step.kernels_per_replay * args.steps   # replays do not pass through the C-ABI launch counter
    barrier()
    ms = max_over_ranks(ms_local)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:    # before the e2e replays overwrite the graph's outputs and step the models on
        dump_outputs(args.dump_outputs, last, eager_step)

    # ---- end-to-end: HOST image batch in, losses out, every step -------------------------------------------------
    # graph: while replay i runs, the pinned host batch of step i + 1 is copied on a copy stream (every step's H2D
    # copy and the D2H read of its losses are inside the timed region; only the very first batch is staged before)
    def e2e_step(i):
        if use_graph:
            return step(host[i % R], prefetch=[host[(i + 1) % R]])
        return step(host[i % R].to(dev, non_blocking=True))

    for i in range(2):
        e2e_step(i)
    barrier()
    d2h_bytes = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = e2e_step(2 + i)
        vals = torch.stack([v.reshape(()) for v in out.values()]).cpu()
        d2h_bytes = vals.numel() * vals.element_size()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    losses = dict(zip(out.keys(), (float(v) for v in vals)))

    # ---- per-entry-point profile of one step -> dominant kernel roofline ---------------------------------------------
    _lib.profile_start()
    sampled(resident[0])          # per-call CUDA events need the eager launch path
    prof = _lib.profile_stop()
    pk = peaks()
    conv = {k: v for k, v in prof.items() if v["flops"] > 0}
    total_ms = sum(v["ms"] for v in prof.values())
    roof = None
    if conv and args.config == "celeba":
        name, r = max(conv.items(), key=lambda kv: kv[1]["ms"])
        ach = r["flops"] / (r["ms"] * 1e-3) / 1e12
        tr = ncu_traffic(name)
        roof = {"bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sust"], "traffic": None if tr is None else tr["bytes"],
                "traffic_source": None if tr is None else f"profiles/{tr['capture']} (ncu --set full, dram read + write per launch)",
                "ncu_tensor_pipe_pct": None if tr is None else tr["tensor_pipe_pct"],
                "algorithmic_flops_per_launch": r["flops"] / r["calls"],
                "kernel": name, "launches": r["calls"],
                "avg_launch_ms": r["ms"] / r["calls"], "share_of_step": r["ms"] / total_ms if total_ms else None,
                "peak_source": pk["src"] + ", sustained bf16 (kernel timed inside a long step)",
                "all_gemm_entry_points": {k: {"tflops": v["flops"] / (v["ms"] * 1e-3) / 1e12, "ms": v["ms"], "calls": v["calls"]}
                                          for k, v in sorted(conv.items(), key=lambda kv: -kv[1]["ms"])}}
    # HBM-bound roofline: the fused multi-tensor Adam, 28 B per parameter update (read p, g, m, v; write p, m, v),
    # timed ALONE: the three optimiser steps of an iteration back to back, 5 times, one event pair (1.45 GB per
    # iteration at CelebA size: far beyond L2).  Per-call events in an eager step also time launch gaps.
    opts = eager_step.optimizers()
    saved_dp = [o._dp for o in opts]
    parallel.detach(*opts)                           # local timing: no collective
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep_i in range(6):
        if rep_i == 1:
            a0.record()
        for o in opts:
            o.step()
    a1.record()
    torch.cuda.synchronize()
    for o, d in zip(opts, saved_dp):
        o._dp = d
    adam_ms = a0.elapsed_time(a1) / 5
    n_updates = sum(p.numel() for o in opts for g in o.param_groups for p in g["params"] if p.grad is not None)
    gbs = 28.0 * n_updates / (adam_ms * 1e-3) / 1e9 if adam_ms > 0 else 0.0
    main_hbm = {"bound": "hbm", "kernel": "adam_kernel (eadgan_adam_step), all optimiser steps of one iteration",
                "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                "algorithmic_bytes_per_step": 28.0 * n_updates, "ms_per_iteration": adam_ms, "peak_source": pk["src"],
                "how": "timed alone, 5 iterations' worth back to back between one CUDA-event pair"}
    if args.profile_out and rank == 0:
        with open(args.profile_out, "w") as f:
            json.dump({"config": args.config, "batch_per_gpu": B, "precision": precision, "step_ms_sum": total_ms,
                       "entry_points": dict(sorted(prof.items(), key=lambda kv: -kv[1]["ms"]))}, f, indent=1)

    if rank != 0:
        return
    ips = Bg * args.steps / (ms * 1e-3)
    ips_e2e = Bg * args.steps / (ms_e2e * 1e-3)
    if roof is None:   # dSprites-class steps are HBM / latency bound (SURVEY.md section 8d): whole-step algorithmic bytes
        gb = cfg["mb"] * 1e6 * ips / 1e9 / world
        roof = {"bound": "hbm", "achieved": gb, "peak": pk["hbm"], "unit": "GB/s", "frac": gb / pk["hbm"], "traffic": None,
                "kernel": "whole step (ideal-fusion bf16 activation bytes per image x images/s per GPU)",
                "algorithmic_bytes_per_image": cfg["mb"] * 1e6, "peak_source": pk["src"]}
    line = {
        "metric": cfg["metric"], "value": ips, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling_kind(args),
        "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
        "config": config_block(args, world),
        "impl_detail": {"precision": precision,
                        "launch": "whole-step CUDA graph replay" if use_graph else "eager (one C-ABI call per kernel)",
                        "latent_sampling": "device Philox4x32-10 inside the step (csrc/sample.cu)",
                        "timing": "one CUDA-event pair around all steps" if flush is None else
                                  "per-step CUDA events, 256 MB L2 flush between steps"},
        "clocks": clocks,
        "e2e": {"value": ips_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_e2e / args.steps,
                "input_pipeline": ("step i+1's pinned host image batch is copied on a copy stream while step i's graph replays; "
                                   "every step's H2D copy and loss read-back are inside the timed region; latents are drawn on "
                                   "the device") if use_graph else "synchronous H2D copy in front of every step"},
        "gpu_launches": int(launches),
        "roofline": roof,
        "roofline_hbm": main_hbm,
        "step_tensor_frac": {"achieved_tflops": cfg["gflop"] * 1e9 * ips / 1e12,
                             "peak_tflops": pk["tf_sust"] * world, "frac": cfg["gflop"] * 1e9 * ips / 1e12 / (pk["tf_sust"] * world)},
        "losses_last_step": losses,
    }
    if parity is not None:
        line["parity"] = parity
    if dp_par is not None:
        line["dp_parity"] = dp_par
    if world == 1 and not args.no_cpu_baseline:
        Bs = cpu_sample_batch(args)
        cb, med = cpu_reference(args.config, Bs, 4, 2)
        line["cpu_baseline"] = {"value": cb, "unit": "images/s", "cores": os.cpu_count(), "kind": "port",
                                "sample": f"4 steps on a {Bs}-image sample of the batch after 2 warm-up on the host CPU "
                                          "(oracle/torch_oracle.py; CPU images/s is flat in batch size)"}
    _OUT.emit(json.dumps(line))


if __name__ == "__main__":
    main()
