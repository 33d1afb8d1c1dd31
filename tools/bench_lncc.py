"""Local NCC at 256^3: the kernels (trb_lncc_forward + trb_lncc_backward) against the fp32 torch restatement, and the LNCC
direct-flow epoch next to the fused MSE + NCC epoch, timed with CUDA events.

    python tools/bench_lncc.py [--out FILE.json] [--reps N] [--win W]

Every timed window is preceded, outside it, by a 256 MB write that evicts the 126 MB L2, so each call reads its inputs
from HBM.  Reported: median us of --reps windows, algorithmic bytes / time, and that as a fraction of the measured HBM
copy peak (DESIGN.md section 4).  Algorithmic bytes per voxel: forward 20 (I, J read; alpha, beta, gamma written),
backward 24 (alpha, beta, gamma, I, J read; dL/dJ written).  LNCC epoch: warp 20 (flow, moving read; J written) +
forward 20 + backward 24 + update 32 (flow, dL/dJ, moving read; flow written) = 96 with SGD; Adam adds 48 (m, v read and
written) and smoothing needs the stats pass, 20 more.  The fused MSE + NCC epoch: 32 (SGD), 80 (Adam).  The torch
restatement (loss + autograd backward, TF32 off) is charged the kernels' 44 bytes."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torchregister_b200.functional as TF            # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tests"))
import lncc_reference as lref                           # noqa: E402
from torchregister_b200.synth import make_pair, smooth_flow      # noqa: E402

HBM_PEAK_GBS = 6549.8
DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, reps, flush, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--win", type=int, default=9)
    ap.add_argument("--size", type=int, default=256)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_lncc needs a CUDA device"
    S, win = args.size, args.win
    vox = S ** 3
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=DEV)
    rows = []

    def report(name, us, bytes_per_voxel, **extra):
        gbs = bytes_per_voxel * vox / us / 1e3
        rows.append(dict({"case": name, "us": round(us, 1), "B_per_voxel": bytes_per_voxel, "GB/s": round(gbs, 0),
                          "frac_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)}, **extra))
        print("%-52s %9.1f us  %3d B/vox  %6.0f GB/s  %.3f of HBM peak %s" % (name, us, bytes_per_voxel, gbs, gbs / HBM_PEAK_GBS,
                                                                           extra or ""), flush=True)

    mov, tgt = (v.to(DEV) for v in make_pair((S, S, S), "flow"))
    flow0 = (0.3 * smooth_flow((S, S, S), 1.0)).to(DEV)
    warped = TF.warp_flow(mov, flow0)

    # ---- the kernels against the torch restatement
    us_f = timed(lambda: TF.lncc_forward(tgt, warped, win), args.reps, flush)
    report("lncc_forward (win %d)" % win, us_f, 20)
    _, coef = TF.lncc_forward(tgt, warped, win)
    us_b = timed(lambda: TF.lncc_backward(tgt, warped, coef, win), args.reps, flush)
    report("lncc_backward (win %d)" % win, us_b, 24)
    us_fb = timed(lambda: TF.lncc_loss_grad(warped, tgt, win), args.reps, flush)
    report("lncc_loss_grad = forward + backward (win %d)" % win, us_fb, 44)

    def torch_lncc():
        w = warped.detach().requires_grad_(True)
        lref.lncc_loss(tgt, w, win).backward()
        return w.grad

    torch.backends.cudnn.allow_tf32 = False
    us_t = timed(torch_lncc, max(5, args.reps // 3), flush)
    report("torch fp32: lncc_loss + autograd backward (win %d)" % win, us_t, 44)
    loss_k, grad_k = TF.lncc_loss_grad(warped, tgt, win)
    w = warped.detach().requires_grad_(True)
    loss_t = lref.lncc_loss(tgt, w, win)
    loss_t.backward()
    agree = {"loss_kernel": loss_k.item(), "loss_torch": loss_t.item(),
             "grad_l2_rel": ((grad_k - w.grad).norm() / w.grad.norm()).item()}
    print("kernel vs torch fp32:", agree)

    # ---- epochs: LNCC direct flow next to the fused MSE + NCC epoch
    per = 5

    def epoch_case(name, opt, lr, smooth, bpv, w_mse=0.0, w_ncc=0.0, w_lncc=0.0):
        prob = TF.DirectFlowProblem(mov, tgt, per * (args.reps + 4), flow0=flow0, optimiser=opt)
        us = timed(lambda: prob.run(per, lr, w_mse, w_ncc, smooth, w_lncc=w_lncc, lncc_win=win), args.reps, flush) / per
        report(name, us, bpv, losses_first_last=[round(float(prob.losses[0]), 6), round(float(prob.losses[-1]), 6)])

    epoch_case("LNCC epoch, SGD", "sgd", 500.0, 0.0, 96, w_lncc=1.0)
    epoch_case("LNCC epoch, Adam + smoothness", "adam", 0.05, 2.0, 164, w_lncc=1.0)
    epoch_case("fused MSE+NCC epoch, SGD", "sgd", 0.5, 0.0, 32, w_mse=0.5, w_ncc=0.5)
    epoch_case("fused MSE+NCC epoch, Adam + smoothness", "adam", 0.05, 2.0, 80, w_mse=0.5, w_ncc=0.5)
    name = card()
    print("card:", name)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": name, "size": S, "win": win, "hbm_peak_GBs": HBM_PEAK_GBS, "reps": args.reps,
                       "kernel_vs_torch": agree, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
