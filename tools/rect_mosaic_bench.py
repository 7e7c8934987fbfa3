"""Square against rectangular mosaics of the same window count, one GPU, in one process.
    python tools/rect_mosaic_bench.py [--out FILE] [--steps K] [--warmup W] [--rounds R]
ViT-S/8 in fp16 (bench.py's segmentation defaults: window 224, stride 112, chunk and tile batch 2048, random-init weights of seed 0)
segments, alternating, round after round:
  - bench.py's 4096^2 mosaic: 35 x 35 = 1225 windows, extent 4032^2;
  - a 3024 x 5712 mosaic: 25 x 49 = 1225 windows, extent 2912 x 5600.
Each step is MosaicSegmenter.segment on the device-resident mosaic, timed with CUDA events; the L2 is flushed between steps; the
warm-up runs the requested steps and then (untimed, at most 12 more) until two consecutive steps agree within 3 %, as bench.py's.
Reported per case and round: ms per step, tiles/s and MP/s of the stitched extent; per case, the device time of each pass of the
post-processing (stitched gray image, pass 1 stitch + min/max, pass 2 histograms, Otsu, pass 3 masks) by CUDA events around the
C entry points on the case's own low-res maps.  The card's name and power limit are read in the same run.  One JSON line per record
is printed and appended to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vitocm_b200 as vob  # noqa: E402
from vitocm_b200 import sw_processing as sw  # noqa: E402
from vitocm_b200 import synthetic as SY  # noqa: E402
from vitocm_b200._lib import check, cur_stream, ptr  # noqa: E402

WINDOW, STRIDE, PATCH = 224, 112, 8
CASES = {"square_4096": (4096, 4096), "rect_3024x5712": (3024, 5712)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def step(seg, mosaic, flush):
    flush.fill_(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = seg.segment(mosaic, want=("th", "th3"))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def timed(seg, mosaic, flush, steps, warmup):
    prev, extra, i = None, 0, 0
    while warmup > 0 and (i < warmup or extra < 12):
        cur, _ = step(seg, mosaic, flush)
        i += 1
        settled = prev is not None and abs(cur - prev) <= 0.03 * prev
        prev = cur
        if i >= warmup:
            if settled:
                break
            extra += 1
    ms = [step(seg, mosaic, flush)[0] for _ in range(steps)]
    return ms, max(i - warmup, 0)


def pass_times(seg, mosaic, out, reps):
    """Device ms of each post-processing pass of the whole extent, mean over `reps` (CUDA events around each entry point)."""
    lib = vob._lib.load_library()
    (ny, nx), (Ey, Ex) = out["grid_shape"], out["extent_shape"]
    H, Wd = mosaic.shape
    lh = WINDOW // PATCH
    low = out["lowres"].contiguous()
    wtab = sw._wtab(WINDOW, STRIDE, mosaic.device)
    st = cur_stream()
    gray = torch.empty(Ey, Ex, dtype=torch.uint8, device=mosaic.device)
    amap = torch.empty(Ey, Ex, dtype=torch.float32, device=mosaic.device)
    mm = torch.empty(2, dtype=torch.int32, device=mosaic.device)
    hists = torch.zeros(3, 256, dtype=torch.int64, device=mosaic.device)
    thr = torch.empty(3, dtype=torch.int32, device=mosaic.device)
    th = torch.empty(Ey, Ex, dtype=torch.uint8, device=mosaic.device)
    th3 = torch.empty_like(th)
    passes = {
        "stitch_gray": lambda: check(lib.vitocm_stitch_gray_grid(ptr(mosaic), H, Wd, mosaic.stride(0), ny, nx, WINDOW, STRIDE, ptr(wtab),
                                                                 0, Ey, ptr(gray), st)),
        "pass1_stitch_minmax": lambda: (check(lib.vitocm_minmax_init(ptr(mm), st)),
                                        check(lib.vitocm_stitch_minmax_grid(ptr(low), ny, nx, WINDOW, STRIDE, lh, lh, ptr(wtab), 0, Ey,
                                                                            ptr(mm), ptr(amap), None, st))),
        "pass2_hist": lambda: (hists.zero_(),
                               check(lib.vitocm_stitch_hist_grid(ptr(low), ny, nx, WINDOW, STRIDE, lh, lh, ptr(wtab), ptr(gray), ptr(mm), 0,
                                                                 Ey, ptr(hists), ptr(amap), st))),
        "otsu": lambda: check(lib.vitocm_otsu(ptr(hists), 3, ptr(thr), st)),
        "pass3_mask": lambda: check(lib.vitocm_stitch_mask_grid(ptr(low), ny, nx, WINDOW, STRIDE, lh, lh, ptr(wtab), ptr(gray), ptr(mm),
                                                                ptr(thr), 0, Ey, ptr(th), None, ptr(th3), ptr(amap), st)),
    }
    res = {k: 0.0 for k in passes}
    for r in range(reps + 1):           # the first round is a warm-up
        for k, fn in passes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if r:
                res[k] += e0.elapsed_time(e1) / reps
    # the passes in isolation reproduce segment()'s masks
    same = bool(torch.equal(th, out["th"]) and torch.equal(th3, out["th3"]))
    return res, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_rect_mosaic.jsonl"))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--precision", default="fp16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rect_mosaic_bench needs a CUDA device")
    dev = torch.device("cuda")
    recs = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        recs.append(rec)

    emit({"record": "setup", "card": card(), "torch": torch.__version__, "precision": args.precision, "window": WINDOW, "stride": STRIDE,
          "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "time": time.strftime("%Y-%m-%dT%H:%M:%S")})
    torch.manual_seed(0)
    model = vob.vit_small(patch_size=PATCH, num_classes=0, precision=args.precision, chunk_tiles=2048).cuda().eval()
    seg = vob.MosaicSegmenter(model, window=WINDOW, stride=STRIDE, tile_batch=2048)
    mosaics = {}
    for name, (H, Wd) in CASES.items():
        full = SY.synthetic_mosaic_u8(max(H, Wd), seed=4321)
        mosaics[name] = torch.from_numpy(np.ascontiguousarray(full[:H, :Wd])).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    outs = {}
    summary = {name: [] for name in CASES}
    for rnd in range(args.rounds):
        for name, mosaic in mosaics.items():
            ms, extra = timed(seg, mosaic, flush, args.steps, args.warmup)
            _, out = step(seg, mosaic, flush)
            outs[name] = out
            (ny, nx), (Ey, Ex) = out["grid_shape"], out["extent_shape"]
            mean = float(np.mean(ms))
            summary[name].append(ny * nx / (mean / 1e3))
            emit({"record": "step", "case": name, "round": rnd, "mosaic": list(mosaic.shape), "grid": [ny, nx], "extent": [Ey, Ex],
                  "tiles": ny * nx, "ms_per_step": mean, "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)),
                  "tiles_per_s": ny * nx / (mean / 1e3), "mp_per_s": Ey * Ex / 1e6 / (mean / 1e3), "extra_warmup": extra})
    for name, mosaic in mosaics.items():
        res, same = pass_times(seg, mosaic, outs[name], 20)
        (Ey, Ex) = outs[name]["extent_shape"]
        emit({"record": "post_passes", "case": name, "extent": [Ey, Ex], "ms": res, "ms_total": sum(res.values()),
              "ns_per_px_total": sum(res.values()) * 1e6 / (Ey * Ex), "masks_equal_segment": same})
    tps = {k: (float(np.mean(v)), float(np.min(v)), float(np.max(v))) for k, v in summary.items()}
    emit({"record": "summary", "card": card(), "tiles_per_s_mean_min_max": tps,
          "rect_over_square": tps["rect_3024x5712"][0] / tps["square_4096"][0]})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
