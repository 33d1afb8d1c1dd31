"""Label-map warps (nearest against bilinear) and the flow Jacobian at 256^3, timed with CUDA events.

    python tools/bench_labels.py [--out FILE.json] [--reps N]

Every timed call is preceded, outside its event window, by a 256 MB write that evicts the 126 MB L2, so each call reads
its inputs from HBM.  Reported per call: median us, algorithmic bytes / time, and that as a fraction of the measured HBM
copy peak (DESIGN.md section 4).  Algorithmic bytes per voxel: nearest or bilinear affine warp 8 per channel; flow warp
12 + 8 per channel; Jacobian 12 (stats only) or 16 (with the fp32 field)."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torchregister_b200 as tr                       # noqa: E402
import torchregister_b200.functional as TF            # noqa: E402
from torchregister_b200 import _lib                   # noqa: E402
from torchregister_b200.synth import smooth_flow      # noqa: E402

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


def torch_jacobian(flow):
    """fp32 torch restatement: torch.gradient per channel (numpy.gradient's differences), 3x3 determinant, statistics."""
    g = [torch.gradient(flow[0, i]) for i in range(3)]
    J = [[g[i][j] + (1.0 if i == j else 0.0) for j in range(3)] for i in range(3)]
    det = (J[0][0] * (J[1][1] * J[2][2] - J[1][2] * J[2][1]) - J[0][1] * (J[1][0] * J[2][2] - J[1][2] * J[2][0])
           + J[0][2] * (J[1][0] * J[2][1] - J[1][1] * J[2][0]))
    L = torch.log(det.clamp(1e-9, 1e9))
    return torch.stack([(det <= 0).sum().float(), det.mean(), det.std(unbiased=False), L.std(unbiased=False)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_labels needs a CUDA device"
    S = 256
    vox = S ** 3
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=DEV)
    rows = []

    def report(name, us, bytes_per_voxel):
        gbs = bytes_per_voxel * vox / us / 1e3
        rows.append({"case": name, "us": round(us, 1), "GB/s": round(gbs, 0), "frac_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)})
        print("%-44s %8.1f us  %6.0f GB/s  %.3f of HBM peak" % (name, us, gbs, gbs / HBM_PEAK_GBS), flush=True)

    small = torch.tensor([[1.01, .02, -.01, .01], [-.02, .99, .01, 0.], [.01, -.01, 1., .02]], device=DEV)
    flow = smooth_flow((S, S, S), 3.0, device=DEV).contiguous()
    g = torch.Generator(device=DEV).manual_seed(0)
    for C in (1, 4):
        labels = torch.randint(0, 20, (1, C, S, S, S), device=DEV, generator=g).float()
        for path, large in (("tma", False), ("gather", True)):
            for mode in ("bilinear", "nearest"):
                us = timed(lambda: TF.warp_affine(small, labels, large_rotation=large, mode=mode), args.reps, flush)
                report("affine %s %s C=%d" % (path, mode, C), us, 8 * C)
        grid_shape = [1, C, S, S, S]
        us = timed(lambda: F.grid_sample(labels, F.affine_grid(small[None], grid_shape, align_corners=False), mode="nearest",
                                         padding_mode="zeros", align_corners=False), args.reps, flush)
        report("torch affine_grid+grid_sample nearest C=%d" % C, us, 8 * C)
        for mode in ("bilinear", "nearest"):
            us = timed(lambda: TF.warp_flow(labels, flow, mode=mode), args.reps, flush)
            report("flow %s C=%d" % (mode, C), us, 12 + 8 * C)
    fold = flow.clone()
    fold[0, 2, 100:140, 100:140, 100:140] *= -4.0
    for field in (False, True):
        us = timed(lambda: tr.jacobian_determinant(fold, return_field=field), args.reps, flush)
        report("jacobian_determinant%s (incl. one D2H read)" % (" +field" if field else ""), us, 16 if field else 12)
    ws = TF._flow_ws(fold.device)
    stats = torch.empty(8, dtype=torch.float64, device=DEV)
    det = torch.empty(1, 1, S, S, S, device=DEV)
    lib = _lib.load()
    for field in (False, True):
        out = det.data_ptr() if field else None
        us = timed(lambda: _lib.check(lib.trb_flow_jacobian(3, fold.data_ptr(), S, S, S, out, stats.data_ptr(), ws.data_ptr(),
                                                            ws.numel(), TF._stream(fold.device)), "flow_jacobian"), args.reps, flush)
        report("trb_flow_jacobian kernel%s" % (" +field" if field else ""), us, 16 if field else 12)
    us = timed(lambda: torch_jacobian(fold), max(5, args.reps // 3), flush)
    report("torch fp32 torch.gradient restatement", us, 12)
    name = card()
    print("card:", name)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": name, "size": S, "hbm_peak_GBs": HBM_PEAK_GBS, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
