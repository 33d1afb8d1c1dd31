"""Transform algebra at 256^3 (affine -> flow, theta-then-flow and flow-then-flow composition, flow inversion), timed
with CUDA events against fp32 torch restatements.

    python tools/bench_transforms.py [--out FILE.json] [--reps N]

Every timed call is preceded, outside its event window, by a 256 MB write that evicts the 126 MB L2, so each call reads
its inputs from HBM.  Reported per call: median us, algorithmic bytes / time, and that as a fraction of the measured HBM
copy peak (DESIGN.md section 4).  Algorithmic bytes per voxel: affine -> flow 12 (written); theta first 24 (u read, w
written); flow first 36 (u, f read once, w written); inverse 24 (u read once, v written: the floor for any number of
iterations, whose gathers hit L1 / L2).  The torch restatements are charged the same bytes."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torchregister_b200 as tr                       # noqa: E402
from torchregister_b200.synth import affine_theta_star, smooth_flow      # noqa: E402

HBM_PEAK_GBS = 6549.8
DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, reps, flush):
    for _ in range(3):
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


def voxel_grid(S):
    r = torch.arange(S, dtype=torch.float32, device=DEV)
    return torch.stack(torch.meshgrid(r, r, r, indexing="ij"))[None]         # [1, 3, S, S, S], (z, y, x)


def affine_terms(theta, S):
    """A = M - I and c of theta's voxel-unit map in flow channel order (cube of side S: M = theta's linear part
    reversed), fp64 on the host, as fp32 device tensors."""
    th = theta.double()
    A = th[:, :3].flip(0).flip(1) - torch.eye(3, dtype=torch.float64)
    c = torch.stack([S / 2 * (th[r, 3] + 1 - th[r, :3].sum() * (1 - 1 / S)) - 0.5 for r in (2, 1, 0)])
    return A.float().to(DEV), c.float().to(DEV).view(1, 3, 1, 1, 1)


def torch_border(f, q, S):
    """f~(q) for a cube of side S: grid_sample(border, align_corners=True) at voxel positions q [1, 3, ...]."""
    g = (q * (2.0 / (S - 1)) - 1).flip(1).permute(0, 2, 3, 4, 1)
    return F.grid_sample(f, g, mode="bilinear", padding_mode="border", align_corners=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_transforms needs a CUDA device"
    S = 256
    vox = S ** 3
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=DEV)
    rows = []

    def report(name, us, bytes_per_voxel, **extra):
        gbs = bytes_per_voxel * vox / us / 1e3
        rows.append(dict({"case": name, "us": round(us, 1), "GB/s": round(gbs, 0), "frac_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)},
                         **extra))
        print("%-46s %8.1f us  %6.0f GB/s  %.3f of HBM peak %s" % (name, us, gbs, gbs / HBM_PEAK_GBS, extra or ""), flush=True)

    theta = affine_theta_star(3).float()
    th_dev = theta.to(DEV)
    u = smooth_flow((S, S, S), 3.0, device=DEV).contiguous()
    f = smooth_flow((S, S, S), 2.0, device=DEV).flip(1).contiguous()
    p = voxel_grid(S)
    A, c = affine_terms(theta, S)

    us = timed(lambda: tr.affine_to_flow(th_dev, (S, S, S)), args.reps, flush)
    report("affine_to_flow", us, 12)
    us = timed(lambda: torch.einsum("ij,bj...->bi...", A, p) + c, args.reps, flush)
    report("torch: A p + c", us, 12)

    us = timed(lambda: tr.compose_flow(th_dev, u), args.reps, flush)
    report("compose_flow(theta, u)", us, 24)
    us = timed(lambda: u + torch.einsum("ij,bj...->bi...", A, p + u) + c, args.reps, flush)
    report("torch: u + A (p + u) + c", us, 24)

    us = timed(lambda: tr.compose_flow(f, u), args.reps, flush)
    report("compose_flow(f, u)", us, 36)
    us = timed(lambda: u + torch_border(f, p + u, S), args.reps, flush)
    report("torch: u + grid_sample(f, p + u, border)", us, 36)

    _, info = tr.invert_flow(u)
    us = timed(lambda: tr.invert_flow(u), args.reps, flush)
    report("invert_flow (incl. one D2H read)", us, 24, mean_iterations=round(info["mean_iterations"], 3),
           n_not_converged=info["n_not_converged"], max_residual=info["max_residual"])

    def torch_invert(tol=1e-3, max_iter=50):
        v = -u
        for k in range(max_iter):
            s = torch_border(u, p + v, S)
            if k == max_iter - 1 or float((v + s).abs().amax()) <= tol:
                return v, k + 1
            v = -s

    _, iters = torch_invert()
    us = timed(torch_invert, max(5, args.reps // 3), flush)
    report("torch: the fixed point, stop on max residual", us, 24, iterations=iters)
    name = card()
    print("card:", name)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"card": name, "size": S, "hbm_peak_GBs": HBM_PEAK_GBS, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
