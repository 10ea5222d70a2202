"""Output dtype / layout of the batch blends on the GPU: {fp32, bf16, fp16} x {NTCHW, NTHWC} for the three kernel families
the dataset uses, at bench.py's configs[4] shape (64 clips x 8 x 224 x 224 uint8, alpha 0.5), every sample mixed and a
Bernoulli(0.25) draw of mixed samples:

  dense    fp32 pool of 1,024 backgrounds of 240x320 after Resize(256) (256 x 341), bgd_bgmix_blend_out
  ragged   uint8 pool of 1,024 backgrounds of 240x{320,427,352,426}, Resize(256) inside the launch, bgd_bgmix_blend_ragged_out
  resize   MultiScaleCrop-sized packed crops (168..256 px) resized inside the launch, dense pool, bgd_bgmix_resize_blend_out

Timing as bench.py's time_back_to_back: 4 batches with their own inputs and outputs back to back in one CUDA-event bracket,
a 256 MB L2 flush before each bracket, median of the brackets, ms per batch.  Algorithmic bytes count the output at its
element size.  Two consumer legs show what the model side saves: the fp32 NTCHW batch followed by .to(torch.bfloat16),
and followed by .contiguous(memory_format=torch.channels_last) of its [B*T, 3, H, W] view, against the blend writing that
tensor directly.  Every 16-bit / NTHWC output is checked against the fp32 NTCHW output converted by torch, at the timed size.

usage: python tools/perf_mix_out.py [--reps 9] [--out FILE]
"""
import argparse
import ctypes
import pathlib
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch        # noqa: E402

import bgdebias_b200.ops as ops                    # noqa: E402
from bgdebias_b200 import _cabi                    # noqa: E402
from bgdebias_b200.pool import RaggedPool          # noqa: E402
from bench import time_back_to_back                # noqa: E402

DTYPES = {"fp32": (torch.float32, _cabi.OUT_F32), "bf16": (torch.bfloat16, _cabi.OUT_BF16), "fp16": (torch.float16, _cabi.OUT_F16)}
LAYOUTS = {"NTCHW": _cabi.LAYOUT_NTCHW, "NTHWC": _cabi.LAYOUT_NTHWC}
B, T, H, W, P = 64, 8, 224, 224, 1024
MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]


def device_context(dev) -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=60)
        if q.returncode == 0 and q.stdout.strip():
            return "device: " + q.stdout.strip() + "  (name, power limit, max SM clock)"
    except (OSError, subprocess.SubprocessError):
        pass
    return f"device: {torch.cuda.get_device_name(dev)} (power limit not readable)"


def shape_of(layout):
    return (B, T, 3, H, W) if layout == "NTCHW" else (B, T, H, W, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    L = _cabi.lib()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(device_context(dev))
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}; workload configs[4]: fg uint8 [{B},{T},{H},{W},3], alpha 0.5")
    say("timing: 4 batches with their own inputs/outputs back to back per CUDA-event bracket, 256 MB L2 flush before each "
        f"bracket, median of {args.reps} brackets")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cur = torch.cuda.current_stream(dev).cuda_stream
    gm = torch.Generator(device=dev).manual_seed(4)
    fgs = [torch.randint(0, 256, (B, T, H, W, 3), dtype=torch.uint8, device=dev, generator=gm) for _ in range(4)]
    lut = ops.make_fg_lut(MEAN, STD, dev)
    c_mean, c_std = _cabi.f32x3(MEAN), _cabi.f32x3(STD)
    rs = np.random.default_rng(9)
    apply_sets = {"all mixed": torch.ones(B, dtype=torch.uint8, device=dev),
                  "Bernoulli(0.25)": torch.from_numpy((rs.random(B) < 0.25).astype(np.uint8)).to(dev)}
    d32 = lambda a: torch.tensor(np.asarray(a), dtype=torch.int32, device=dev)   # noqa: E731

    # ---- the three families: launch(i, app, layout, code, out) blends batch i into out ----
    pool = torch.rand((P, 3, 256, 341), device=dev, generator=gm) * 255.0
    idx = d32(rs.integers(0, P, B)); top = d32(rs.integers(0, 33, B)); left = d32(rs.integers(0, 118, B))

    def dense(i, app, layout, code, out):
        _cabi.check(L.bgd_bgmix_blend_out(fgs[i].data_ptr(), B, T, H, W, pool.data_ptr(), 0, P, 256, 341, idx.data_ptr(),
                                          top.data_ptr(), left.data_ptr(), app.data_ptr(), lut.data_ptr(), c_mean, c_std, 0.5,
                                          layout, code, out.data_ptr(), cur))

    g = torch.Generator().manual_seed(6)
    sizes = [(240, 320), (240, 427), (240, 352), (240, 426)]
    rp = RaggedPool(256, dev)
    imgs = [torch.randint(0, 256, (3,) + sizes[k % 4], dtype=torch.uint8, generator=g) for k in range(64)]
    for _ in range(16):
        rp.append(imgs)
    r_idx = rs.integers(0, len(rp), B)
    r_hw = [rp.hw(int(k)) for k in r_idx]
    r_top = d32([rs.integers(0, h - H + 1) for h, w in r_hw]); r_left = d32([rs.integers(0, w - W + 1) for h, w in r_hw])
    r_idx_d = d32(r_idx)
    r_bg_bytes = []                                   # source window of each crop, as bench.py counts it
    for k, (Hb, Wb) in zip(r_idx, r_hw):
        s_ = rp.slots[int(k)]
        r_bg_bytes.append(3 * int(np.ceil(H * int(s_["h"]) / Hb + 2)) * int(np.ceil(W * int(s_["w"]) / Wb + 2)))

    def ragged(i, app, layout, code, out):
        _cabi.check(L.bgd_bgmix_blend_ragged_out(fgs[i].data_ptr(), B, T, H, W, rp.data.data_ptr(), rp.slots_tensor.data_ptr(),
                                                 len(rp), rp.tables.tensor.data_ptr(), r_idx_d.data_ptr(), r_top.data_ptr(),
                                                 r_left.data_ptr(), app.data_ptr(), lut.data_ptr(), c_mean, c_std, 0.5, layout,
                                                 code, out.data_ptr(), cur))

    csizes = [(256, 256), (224, 256), (256, 224), (224, 224), (192, 224), (224, 192), (192, 192), (168, 192), (192, 168), (168, 168)]
    gc = torch.Generator().manual_seed(4)
    crops = [torch.randint(0, 256, (T, *csizes[k % len(csizes)], 3), dtype=torch.uint8, generator=gc) for k in range(B)]
    buf, geom = ops.pack_clips(crops)
    bufs = [buf.to(dev)] + [buf.to(dev) for _ in range(3)]
    gptr = ctypes.cast(geom.data_ptr(), ctypes.POINTER(ctypes.c_int64))
    crop_bytes = sum(c.numel() for c in crops)

    def resize(i, app, layout, code, out):
        _cabi.check(L.bgd_bgmix_resize_blend_out(bufs[i].data_ptr(), bufs[i].numel(), gptr, B, T, H, W, pool.data_ptr(), 0, P, 256,
                                                 341, idx.data_ptr(), top.data_ptr(), left.data_ptr(), app.data_ptr(), lut.data_ptr(),
                                                 c_mean, c_std, 0.5, layout, code, out.data_ptr(), cur))

    fg_bytes = B * T * H * W * 3
    families = [("dense", dense, fg_bytes, [H * W * 3 * 4] * B),          # per sample: background bytes read when mixed
                ("ragged", ragged, fg_bytes, r_bg_bytes),
                ("resize", resize, crop_bytes, [H * W * 3 * 4] * B)]
    out_elems = B * T * 3 * H * W

    say()
    say(f"{'family':8s} {'apply':16s} {'dtype':5s} {'layout':6s} {'ms/batch':>9s} {'MB/batch':>9s} {'GB/s':>7s}  output check")
    ok_all = True
    for fam, launch, in_bytes, bg_bytes in families:
        for app_name, app in apply_sets.items():
            outs32 = [torch.empty(shape_of("NTCHW"), dtype=torch.float32, device=dev) for _ in range(4)]
            for i in range(4):
                launch(i, app, _cabi.LAYOUT_NTCHW, _cabi.OUT_F32, outs32[i])
            torch.cuda.synchronize()
            for dname, (dt, code) in DTYPES.items():
                for lname, lay in LAYOUTS.items():
                    outs = outs32 if (dname, lname) == ("fp32", "NTCHW") else \
                        [torch.empty(shape_of(lname), dtype=dt, device=dev) for _ in range(4)]
                    calls = [(lambda i=i, o=o: launch(i, app, lay, code, o)) for i, o in enumerate(outs)]
                    ms = time_back_to_back(calls, flush, args.reps, torch)
                    by = in_bytes + sum(n for n, a in zip(bg_bytes, app.tolist()) if a) + out_elems * dt.itemsize
                    check = "reference"
                    if (dname, lname) != ("fp32", "NTCHW"):
                        exp = outs32[0].to(dt)
                        if lname == "NTHWC":
                            exp = exp.permute(0, 1, 3, 4, 2).contiguous()
                        ok = bool(torch.equal(outs[0].view(torch.int16 if dt.itemsize == 2 else torch.int32),
                                              exp.view(torch.int16 if dt.itemsize == 2 else torch.int32)))
                        ok_all &= ok
                        check = "bit-equal to fp32 NTCHW converted by torch" if ok else "MISMATCH"
                    say(f"{fam:8s} {app_name:16s} {dname:5s} {lname:6s} {ms:9.4f} {by / 1e6:9.2f} {by / (ms * 1e-3) / 1e9:7.0f}  {check}")
                    if outs is not outs32:
                        del outs
            del outs32
            torch.cuda.empty_cache()

    # ---- consumer legs: the dense blend + the conversion the model side would otherwise run ----
    say()
    say("consumer legs (dense family, all mixed): ms per batch, blend + conversion kernels together")
    app = apply_sets["all mixed"]
    outs32 = [torch.empty(shape_of("NTCHW"), dtype=torch.float32, device=dev) for _ in range(4)]
    direct = {name: [torch.empty(shape_of(lname), dtype=DTYPES[dname][0], device=dev) for _ in range(4)]
              for name, dname, lname in (("bf16 NTCHW", "bf16", "NTCHW"), ("fp32 NTHWC", "fp32", "NTHWC"),
                                         ("bf16 NTHWC", "bf16", "NTHWC"))}

    def blend32(i):
        dense(i, app, _cabi.LAYOUT_NTCHW, _cabi.OUT_F32, outs32[i])
        return outs32[i]

    def blend_direct(i, name):
        dname, lname = name.split()
        dense(i, app, LAYOUTS[lname], DTYPES[dname][1], direct[name][i])

    legs = [("fp32 NTCHW out, then .to(torch.bfloat16)", lambda i: blend32(i).to(torch.bfloat16)),
            ("bf16 NTCHW out", lambda i: blend_direct(i, "bf16 NTCHW")),
            ("fp32 NTCHW out, then [B*T,3,H,W].contiguous(channels_last)",
             lambda i: blend32(i).flatten(0, 1).contiguous(memory_format=torch.channels_last)),
            ("fp32 NTHWC out", lambda i: blend_direct(i, "fp32 NTHWC")),
            ("fp32 NTCHW out, then .to(bfloat16) and channels_last",
             lambda i: blend32(i).flatten(0, 1).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)),
            ("bf16 NTHWC out", lambda i: blend_direct(i, "bf16 NTHWC"))]
    for name, fn in legs:
        ms = time_back_to_back([(lambda i=i: fn(i)) for i in range(4)], flush, args.reps, torch)
        say(f"  {name:62s} {ms:8.4f} ms")
    say()
    say("all output checks passed" if ok_all else "OUTPUT CHECK FAILED")
    if args.out:
        pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(args.out).write_text("\n".join(lines) + "\n")
    return 0 if ok_all else 1


if __name__ == "__main__":
    sys.exit(main())
