"""Timing of the evaluation route: resize_crop_normalize (Resize(scale=(-1, 256)) -> CenterCrop(224) / ThreeCrop(256) ->
Normalize -> FormatShape('NCHW'), one launch per batch) against the same tail run per clip on one host core, and the
bytes a batch carries across PCIe as decoded uint8 frames instead of the fp32 tensor the workers build today.

Workloads: B = 16 videos of one native size (240x320 as UCF101 / HMDB51 decode, 240x427 as Sth-Sth-v2), T = 8 and 16,
both crops, fp32 and bf16.  Device timing: 4 batches with their own inputs and outputs back to back per CUDA-event bracket,
a 256 MB L2 flush before each bracket, median of 9 brackets; the geometry upload is inside the bracket.  Every GPU output
is compared bit for bit with the CPU pipeline of the same batch (bf16: with its fp32 result rounded by torch).
usage: python tools/perf_eval_batch.py [out.txt]      (default profiles/r3_perf_eval.txt)"""
import pathlib
import subprocess
import sys
import time

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))
import cv2                                                   # noqa: E402
import numpy as np                                           # noqa: E402
import torch                                                 # noqa: E402

import bgdebias_b200.ops as ops                              # noqa: E402
from bgdebias_b200.comix_loader import EvalPipeline          # noqa: E402

MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
B, REPS, BRACKETS = 16, 4, 9


def steps(crop, size):
    return [dict(type="Resize", scale=(-1, 256)), dict(type=crop, crop_size=size),
            dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


def cpu_clip(clip, ev):
    """The worker-side tail of one clip, as mmaction runs it: cv2 resize, crop slices, mmcv-style normalise, transpose."""
    Hr, Wr, wins = ev.windows(clip.shape[1], clip.shape[2])
    ch, cw = ev.crop_hw
    resized = [cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR) for f in clip]
    mean, stdinv = np.float64(np.asarray(MEAN).reshape(1, -1)), 1 / np.float64(np.asarray(STD).reshape(1, -1))
    out = []
    for top, left in wins:
        for r in resized:
            x = r[top:top + ch, left:left + cw].astype(np.float32)
            cv2.subtract(x, mean, x)
            cv2.multiply(x, stdinv, x)
            out.append(x)
    return np.ascontiguousarray(np.stack(out).transpose(0, 3, 1, 2))


def main():
    out_path = pathlib.Path(sys.argv[1]) if len(sys.argv) > 1 else pathlib.Path("profiles/r3_perf_eval.txt")
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    lut = ops.make_fg_lut(MEAN, STD, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(0)
    lines = [f"device: {smi}  (name, power limit, max SM clock)",
             f"torch {torch.__version__}, CUDA {torch.version.cuda}; B = {B} videos of one native size per batch",
             f"timing: {REPS} batches back to back per CUDA-event bracket, 256 MB L2 flush before each, median of {BRACKETS}; "
             "CPU: the per-clip tail on one host core (cv2 and torch at 1 thread), median of 3 batches",
             "GB/s counts the native uint8 source bytes plus the output bytes; H2D: the bytes of one batch across PCIe",
             "",
             f"{'native':>8} {'T':>3} {'crop':<14} {'dtype':<5} {'ms/batch':>9} {'GB/s':>7} {'H2D u8 MB':>10} {'fp32 MB':>8} "
             f"{'ratio':>6} {'CPU ms/batch':>13}  output check"]
    for h, w in ((240, 320), (240, 427)):
        for T in (8, 16):
            clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for _ in range(B)]
            buf, g5 = ops.pack_clips(clips, pin=True)
            srcs = [buf.to(dev) for _ in range(REPS)]
            for crop, size in (("CenterCrop", 224), ("ThreeCrop", 256)):
                ev = EvalPipeline(steps(crop, size))
                geom = ev.geometry(g5)
                K, (ch, cw) = ev.n_crops, ev.crop_hw
                cpu_t, ref = [], None
                for _ in range(3):
                    t0 = time.perf_counter()
                    ref = np.stack([cpu_clip(c, ev) for c in clips])
                    cpu_t.append((time.perf_counter() - t0) * 1e3)
                cpu_ms = sorted(cpu_t)[1]
                ref_t = torch.from_numpy(ref)
                fp32_bytes = ref.nbytes
                for dt in (torch.float32, torch.bfloat16):
                    run = lambda s: torch.ops.bgdebias.resize_crop_normalize(s, geom, T, ch, cw, lut, "NTCHW", dt)  # noqa: E731
                    for s in srcs:
                        run(s)
                    torch.cuda.synchronize()
                    ts = []
                    for _ in range(BRACKETS):
                        flush.zero_()
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        outs = [run(s) for s in srcs]
                        b.record()
                        torch.cuda.synchronize()
                        ts.append(a.elapsed_time(b) / REPS)
                    ms = sorted(ts)[len(ts) // 2]
                    got = outs[0].view(B, K * T, 3, ch, cw).cpu()
                    same = torch.equal(got, ref_t.to(dt))
                    moved = buf.numel() + got.numel() * got.element_size()
                    lines.append(f"{h}x{w:<4} {T:>3} {f'{crop}({size})':<14} {str(dt)[6:]:<5} {ms:>9.4f} {moved / ms / 1e6:>7.0f} "
                                 f"{buf.numel() / 1e6:>10.2f} {fp32_bytes / 1e6:>8.2f} {fp32_bytes / buf.numel():>6.1f} "
                                 f"{cpu_ms:>13.1f}  {'bit-equal to the CPU pipeline' if same else 'MISMATCH'}")
                    print(lines[-1], flush=True)
                    if not same:
                        raise SystemExit("GPU output differs from the CPU pipeline")
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text("\n".join(lines) + "\n")
    print(f"wrote {out_path}")


if __name__ == "__main__":
    main()
