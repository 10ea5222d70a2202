"""Timing of the training route: a BG-mix batch finished from native-size frames with the two-stage geometry
(Resize(scale=(-1, 256)) -> MultiScaleCrop -> Resize(224, 224) -> Normalize -> blend) against the crops route, whose workers
run Resize + MultiScaleCrop on the host and ship the crops; plus what the workers no longer run, on one host core, and
the bytes each route carries across PCIe.

Workload: configs[4]-shaped, B = 64 clips x T = 8 frames -> 224x224, native 240x320 (UCF101), MultiScaleCrop(224,
scales=(1, .875, .75, .66), max_wh_scale_gap=1, num_fixed_crops=13) drawn per clip; mix probability 0.5.  Pools: dense
(64 fp32 images 256x341) and ragged (64 uint8 images of four widths, Resize(256) inside the launch).  Outputs: fp32 NTCHW and
bf16 channels-last.  Device timing: the two routes alternated, a 256 MB L2 flush before each CUDA-event bracket, 4 batches
per bracket, median of 15 brackets; the geometry upload is inside the bracket, the H2D copy is not.  Both routes' outputs
are compared bit for bit.
usage: python tools/perf_train_batch.py [out.txt]      (default profiles/r3_perf_train.txt)"""
import pathlib
import random
import subprocess
import sys
import time

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))
import cv2                                                   # noqa: E402
import numpy as np                                           # noqa: E402
import torch                                                 # noqa: E402

import bgdebias_b200.ops as ops                              # noqa: E402
from bgdebias_b200.comix_loader import TrainPipeline         # noqa: E402
from bgdebias_b200.pool import RaggedPool                    # noqa: E402

MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
B, T, H, W, REPS, BRACKETS = 64, 8, 224, 224, 4, 15
STEPS = [dict(type="Resize", scale=(-1, 256)),
         dict(type="MultiScaleCrop", input_size=224, scales=(1, 0.875, 0.75, 0.66), random_crop=False, max_wh_scale_gap=1,
              num_fixed_crops=13),
         dict(type="Resize", scale=(224, 224), keep_ratio=False),
         dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


def host_steps(clip, Hr, Wr, y0, x0, ch, cw):
    """What a crops-route worker runs per clip: cv2 Resize(scale=(-1, 256)) of every frame and the MultiScaleCrop slice."""
    return np.stack([cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR)[y0:y0 + ch, x0:x0 + cw] for f in clip])


def main():
    out_path = pathlib.Path(sys.argv[1]) if len(sys.argv) > 1 else pathlib.Path("profiles/r3_perf_train.txt")
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    rng = np.random.default_rng(0)
    random.seed(0)
    tp = TrainPipeline(STEPS)
    clips = [rng.integers(0, 256, (T, 240, 320, 3), dtype=np.uint8) for _ in range(B)]
    wins = [tp.draw(240, 320) for _ in range(B)]

    cpu_t = []
    for _ in range(3):
        t0 = time.perf_counter()
        crops = [host_steps(c, *w) for c, w in zip(clips, wins)]
        cpu_t.append((time.perf_counter() - t0) * 1e3 / B)
    cpu_ms = sorted(cpu_t)[1]

    nat_buf, g5 = ops.pack_clips(clips, pin=True)
    geom11 = torch.cat([g5, torch.tensor(wins, dtype=torch.int64)], 1)
    crop_buf, geom5 = ops.pack_clips(crops, pin=True)
    nat_srcs = [nat_buf.to(dev) for _ in range(REPS)]
    crop_srcs = [crop_buf.to(dev) for _ in range(REPS)]

    lut = ops.make_fg_lut(MEAN, STD, dev)
    mean_t, std_t = torch.tensor(MEAN), torch.tensor(STD)
    d32 = lambda a: torch.tensor(np.asarray(a), dtype=torch.int32, device=dev)       # noqa: E731
    app = torch.tensor(rng.integers(0, 2, B), dtype=torch.uint8, device=dev)
    P = 64
    dense = torch.rand((P, 3, 256, 341), device=dev, generator=torch.Generator(dev).manual_seed(1)) * 255.0
    d_idx, d_top, d_left = d32(rng.integers(0, P, B)), d32(rng.integers(0, 33, B)), d32(rng.integers(0, 118, B))
    g = torch.Generator().manual_seed(2)
    sizes = [(240, 320), (240, 427), (240, 352), (240, 426)]
    rp = RaggedPool(256, dev)
    rp.append([torch.randint(0, 256, (3,) + sizes[k % 4], dtype=torch.uint8, generator=g) for k in range(P)])
    r_idx = rng.integers(0, P, B)
    r_hw = [rp.hw(int(k)) for k in r_idx]
    r_idx_d = d32(r_idx)
    r_top, r_left = d32([rng.integers(0, h - H + 1) for h, w in r_hw]), d32([rng.integers(0, w - W + 1) for h, w in r_hw])

    def route(pool_kind, src, geom, layout, dt):
        if pool_kind == "dense":
            return torch.ops.bgdebias.bgmix_resize_blend(src, geom, T, H, W, dense, d_idx, d_top, d_left, app, lut, mean_t,
                                                         std_t, 0.5, layout, dt)
        fg = torch.ops.bgdebias.resize_bilinear(src, geom, T, H, W)
        return torch.ops.bgdebias.bgmix_blend_ragged(fg, rp.data, rp.slots_tensor, rp.tables.tensor, r_idx_d, r_top, r_left, app,
                                                     lut, mean_t, std_t, 0.5, layout, dt)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lines = [f"device: {smi}  (name, power limit, max SM clock)",
             f"torch {torch.__version__}, CUDA {torch.version.cuda}; B = {B} clips x T = {T} frames of 240x320 -> {H}x{W}",
             f"timing: routes alternated, {REPS} batches per CUDA-event bracket, 256 MB L2 flush before each, median of "
             f"{BRACKETS}; geometry upload inside, H2D copy outside the bracket",
             "two-stage: native frames + 11-column geometry; crops: host Resize + MultiScaleCrop, packed crops + 5-column geometry",
             f"host steps the two-stage route removes from a worker (cv2 at 1 thread, one core): {cpu_ms:.3f} ms per clip "
             f"({cpu_ms * B:.1f} ms per batch)",
             f"H2D bytes per batch: two-stage {nat_buf.numel() / 1e6:.2f} MB, crops {crop_buf.numel() / 1e6:.2f} MB "
             f"({nat_buf.numel() / crop_buf.numel():.2f}x)",
             "",
             f"{'pool':<7} {'output':<22} {'two-stage ms':>13} {'crops ms':>9} {'ratio':>6}  output check"]
    print("\n".join(lines), flush=True)
    for pool_kind in ("dense", "ragged"):
        for label, layout, dt in (("fp32 NTCHW", "NTCHW", torch.float32), ("bf16 channels-last", "NTHWC", torch.bfloat16)):
            runs = {"two": lambda i: route(pool_kind, nat_srcs[i], geom11, layout, dt),
                    "crops": lambda i: route(pool_kind, crop_srcs[i], geom5, layout, dt)}
            for fn in runs.values():
                for i in range(REPS):
                    fn(i)
            torch.cuda.synchronize()
            ts = {k: [] for k in runs}
            outs = {}
            for _ in range(BRACKETS):
                for k, fn in runs.items():
                    flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    outs[k] = [fn(i) for i in range(REPS)]
                    b.record()
                    torch.cuda.synchronize()
                    ts[k].append(a.elapsed_time(b) / REPS)
            med = {k: sorted(v)[len(v) // 2] for k, v in ts.items()}
            same = torch.equal(outs["two"][0], outs["crops"][0])
            lines.append(f"{pool_kind:<7} {label:<22} {med['two']:>13.4f} {med['crops']:>9.4f} {med['two'] / med['crops']:>6.2f}  "
                         f"{'bit-equal' if same else 'MISMATCH'}")
            print(lines[-1], flush=True)
            if not same:
                raise SystemExit("the two routes differ")
    lines += ["", "not measured: DataLoader throughput with N workers (JPEG decode included), and the PCIe copy time itself"]
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text("\n".join(lines) + "\n")
    print(f"wrote {out_path}")


if __name__ == "__main__":
    main()
