"""Eval-mode CelebA generator: sampling (no-grad forward) and latent-space projection (forward + backward to z).

    python tools/bench_eval.py [--batches 100,1024] [--out FILE] [--profile FILE]

Paths, all on the same seeded inputs and generator state (random running statistics, .eval()):
  ours_bf16       eadgan_b200 with EADGAN_PRECISION=bf16 (tcgen05 chain, eval-mode BatchNorm on the chain)
  ours_fp32       eadgan_b200 with EADGAN_PRECISION=fp32 (the fp32 SIMT per-operator path)
  torch_tf32      the stock oracle module through cuDNN with TF32 allowed
  torch_bf16_amp  the stock oracle module under torch.autocast(dtype=torch.bfloat16)

Each case is warmed up, then timed with CUDA events over a window of at least --window seconds.  One JSON line per case
goes to stdout (and to --out); the first line names the device and its power limit.  --profile writes a
torch.profiler kernel list of ONE bf16 eval forward at the largest batch (a separate run, after the timing)."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:   # read-only query
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unknown"
    return info


def make_nets(dev):
    from eadgan_b200.steps import celeba as CS
    from oracle import torch_oracle as O
    torch.manual_seed(0)
    ref = O.CelebAGenerator()
    g = torch.Generator().manual_seed(0)
    for m in ref.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.3)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
    ref = ref.to(dev).eval()
    ours = CS.Generator().to(dev)
    ours.load_state_dict(ref.state_dict())
    ours.eval()
    for p in list(ref.parameters()) + list(ours.parameters()):
        p.requires_grad_(False)
    return ours, ref


def inputs(B, dev):
    g = torch.Generator().manual_seed(B)
    z = torch.randn(B, 200, generator=g).to(dev)
    lab = torch.eye(10)[torch.randint(0, 10, (B,), generator=g)].to(dev)
    code = (torch.rand(B, 8, generator=g) * 2 - 1).to(dev)
    go = torch.randn(B, 3, 64, 64, generator=g).to(dev)
    return z, lab, code, go


def make_fn(path, mode, ours, ref, z, lab, code, go):
    net = ours if path.startswith("ours") else ref

    def run():
        ctx = (torch.autocast("cuda", dtype=torch.bfloat16) if path == "torch_bf16_amp"
               else torch.autocast("cuda", enabled=False))
        if mode == "forward":
            with torch.no_grad(), ctx:
                return net(z, lab, code)
        zz = z.clone().requires_grad_()
        with ctx:
            y = net(zz, lab, code)
        y.float().backward(go)
        return zz.grad
    return run


def set_path(path):
    os.environ["EADGAN_PRECISION"] = "fp32" if path == "ours_fp32" else "bf16"
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = path == "torch_tf32"


def time_case(fn, window):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    est = e0.elapsed_time(e1) / 3 / 1e3
    iters = max(10, int(1.2 * window / max(est, 1e-6)) + 1)
    while True:
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        total = e0.elapsed_time(e1) / 1e3
        if total >= window:
            return total / iters, iters, total
        iters = int(iters * 1.5 * window / total) + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="100,1024")
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_eval.py needs a CUDA device")
    dev = torch.device("cuda:0")
    ours, ref = make_nets(dev)
    lines = [dict(device_info(), what="CelebA generator, eval mode, random running statistics")]
    print(json.dumps(lines[0]), flush=True)
    paths = ("ours_bf16", "ours_fp32", "torch_tf32", "torch_bf16_amp")
    for B in [int(b) for b in args.batches.split(",")]:
        z, lab, code, go = inputs(B, dev)
        outs = {}
        for mode in ("forward", "forward_backward_z"):
            for path in paths:     # results first: every path is compared with the fp32 one
                set_path(path)
                outs[(mode, path)] = make_fn(path, mode, ours, ref, z, lab, code, go)().float()
            base = outs[(mode, "ours_fp32")]
            for path in paths:
                set_path(path)
                sec, iters, total = time_case(make_fn(path, mode, ours, ref, z, lab, code, go), args.window)
                rec = {"batch": B, "mode": mode, "path": path, "ms": round(sec * 1e3, 4),
                       "samples_per_s": round(B / sec, 1), "iters": iters, "window_s": round(total, 3)}
                if path != "ours_fp32":
                    rec["max_rel_err_vs_ours_fp32"] = float((outs[(mode, path)] - base).abs().max() / base.abs().max())
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    os.environ["EADGAN_PRECISION"] = "bf16"
    if args.out:
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        z, lab, code, _ = inputs(max(int(b) for b in args.batches.split(",")), dev)
        with torch.no_grad():
            ours(z, lab, code)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                ours(z, lab, code)
                torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type.name == "CUDA"]
        with open(args.profile, "w") as f:
            f.write(f"# {json.dumps(lines[0])}\n# one bf16 eval forward of the CelebA generator, batch {z.shape[0]}, "
                    f"warm pack cache; {len(evs)} device activities in launch order (us, name)\n")
            for e in evs:
                f.write(f"{e.device_time:10.1f}  {e.name}\n")


if __name__ == "__main__":
    main()
