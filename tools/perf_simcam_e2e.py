"""sim_cam extraction on the device: the batched RandomResizedCrop kernel alone, and the CLI end to end.

1. Kernel: torch.ops.bgdebias.resized_crop_aa over one slab -- V folders, T ~ U[50, 150], 240x320 frames, draws replayed
   from a seed -- CUDA events, 2 warm-up launches, median of 7.  Algorithmic bytes = crop-window bytes read + 120,000 B
   written per frame (the input, ~6 GB, is far larger than the L2).
2. End to end: a seeded tree of JPEG frame folders; `--method sim_cam` through the staged path (decoder threads, pinned
   slabs, two launches per slab) and through the per-folder drop-in loop (sim_cam_motion_bg_extract folder by folder, the
   path the CLI took before the staged one; kept here only as a baseline), alternating, same host, same seed; both arms
   must write identical JPEG bytes.  Also the reference's procedure on the host (read_image, RandomResizedCrop(100),
   np.nanmedian; one process per core) on a bounded sample of the folders.
usage: python tools/perf_simcam_e2e.py [V=256] [folders=64] [frames=150]"""
import json, os, pathlib, subprocess, sys, tempfile, time, warnings
sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))
import cv2, numpy as np, torch

H, W = 240, 320
V = int(sys.argv[1]) if len(sys.argv) > 1 else 256
n_folders = int(sys.argv[2]) if len(sys.argv) > 2 else 64
T_e2e = int(sys.argv[3]) if len(sys.argv) > 3 else 150


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_alone():
    from bgdebias_b200 import extract_background as eb
    from bgdebias_b200.pool import AATables
    rng = np.random.default_rng(0)
    Ts = rng.integers(50, 151, V)
    n = int(Ts.sum())
    frame = 3 * H * W
    src = torch.randint(0, 256, (n * frame,), dtype=torch.uint8, device="cuda")
    torch.manual_seed(0)
    draws = eb.crop_draws([(H, W)] * n)
    tables = AATables("cuda")
    desc = eb.crop_descriptors([(k * frame, H, W) for k in range(n)], draws, tables)
    tab = tables.tensor
    op = torch.ops.bgdebias.resized_crop_aa
    for _ in range(2):
        out = op(src, desc, tab, 100, 100)
    torch.cuda.synchronize()
    ts, host = [], []
    for _ in range(7):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record(); out = op(src, desc, tab, 100, 100); b.record()
        host.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = sorted(ts)[len(ts) // 2]
    read = sum(3 * h * w for _, _, h, w in draws)
    written = n * 100 * 100 * 3 * 4
    return {"leg": "kernel", "folders": V, "frames": n, "frame": f"{H}x{W}", "ms": round(ms, 4), "ms_all": [round(t, 4) for t in ts],
            "frames_per_s": round(n / ms * 1e3), "algorithmic_GB_per_s": round((read + written) / ms / 1e6, 1),
            "read_MB": round(read / 1e6, 1), "written_MB": round(written / 1e6, 1),
            "host_ms_per_call_median": round(sorted(host)[len(host) // 2] * 1e3, 2), "out_shape": list(out.shape)}


def _make_tree(root: pathlib.Path):
    rng = np.random.default_rng(1)
    t0 = time.perf_counter()
    for v in range(n_folders):
        d = root / f"v{v:04d}"
        d.mkdir(parents=True)
        base = cv2.GaussianBlur(rng.integers(0, 256, (H + 64, W + 64, 3), dtype=np.uint8), (21, 21), 0)
        for t in range(T_e2e):
            dy, dx = (3 * t) % 64, (5 * t + v) % 64                   # a camera pan over a smooth scene
            f = base[dy:dy + H, dx:dx + W].copy()
            f[(7 * t) % (H - 40):(7 * t) % (H - 40) + 40, (11 * t) % (W - 40):(11 * t) % (W - 40) + 40] = 255 - (t % 5)
            cv2.imwrite(str(d / f"img_{t + 1:05d}.jpg"), f)
    return time.perf_counter() - t0


def _dropin_loop(paths, out):
    from bgdebias_b200 import extract_background as eb
    for p in paths:
        eb.sim_cam_motion_bg_extract(p, (out / p.name).with_suffix(".jpg"), False, 1, 500, 0, device=0)


def _one_thread():
    torch.set_num_threads(1)                                           # one process per core, as the reference's workers


def _reference_one(path):
    from torchvision.io import read_image
    from torchvision.transforms import Compose, RandomResizedCrop
    pipe = Compose([RandomResizedCrop(size=100)])
    files = sorted(pathlib.Path(path).glob("*"))
    frames = []
    for i, f in enumerate(files[:-1:1]):
        if i == 500:
            break
        x = pipe(read_image(str(f)).float()).permute(1, 2, 0).numpy()
        x[x == 0] = np.nan
        frames.append(x)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        np.nanmedian(frames, axis=0).astype(np.uint8)
    return len(frames)


def _log(msg):
    print(msg, file=sys.stderr, flush=True)


def end_to_end():
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    from bgdebias_b200 import extract_background as eb
    cores = len(os.sched_getaffinity(0))
    res = {"leg": "end_to_end", "folders": n_folders, "frames_per_folder": T_e2e, "frame": f"{H}x{W} JPEG", "host_cores": cores}
    with tempfile.TemporaryDirectory() as tmp:
        root = pathlib.Path(tmp)
        res["tree_write_s"] = round(_make_tree(root / "in"), 1)
        _log(f"tree written in {res['tree_write_s']} s")
        paths = sorted((root / "in").iterdir())
        n = sum(len(list(p.iterdir())) - 1 for p in paths)
        argv = lambda out: ["--video_dir", str(root / "in"), "--output_dir", str(out), "--num_workers", "1",  # noqa: E731
                            "--method", "sim_cam", "--decode_threads", str(cores)]
        outs = {"staged": root / "staged", "dropin": root / "dropin"}
        times = {"staged": [], "dropin": []}
        for rnd in range(3):                                           # round 0 warms both arms up
            for arm in ("staged", "dropin"):
                out = outs[arm]
                if out.exists():
                    for f in out.iterdir():
                        f.unlink()
                out.mkdir(exist_ok=True)
                torch.manual_seed(0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if arm == "staged":
                    eb.main(argv(out))
                else:
                    _dropin_loop(paths, out)
                torch.cuda.synchronize()
                _log(f"round {rnd} {arm}: {time.perf_counter() - t0:.3f} s")
                if rnd:
                    times[arm].append(time.perf_counter() - t0)
        same = all((outs["staged"] / (p.name + ".jpg")).read_bytes() == (outs["dropin"] / (p.name + ".jpg")).read_bytes()
                   for p in paths)
        sample = paths[:min(len(paths), 2 * cores)]
        # spawned workers: a fork of this process (CUDA context, torch thread pools) is not safe
        with ProcessPoolExecutor(cores, mp_context=mp.get_context("spawn"), initializer=_one_thread) as ex:
            list(ex.map(_reference_one, sample[:cores]))               # warm-up
            _log("reference arm warmed up")
            t0 = time.perf_counter(); n_ref = sum(ex.map(_reference_one, sample)); t_ref = time.perf_counter() - t0
    best = {a: min(t) for a, t in times.items()}
    res.update({"frames": n, "staged_s": [round(t, 3) for t in times["staged"]], "dropin_s": [round(t, 3) for t in times["dropin"]],
                "staged_frames_per_s": round(n / best["staged"], 1), "dropin_frames_per_s": round(n / best["dropin"], 1),
                "speedup_staged_over_dropin": round(best["dropin"] / best["staged"], 2), "identical_jpegs": same,
                "reference_procedure_sample": f"{len(sample)} folders, {n_ref} frames, {cores} processes",
                "reference_frames_per_s": round(n_ref / t_ref, 1)})
    return res


if __name__ == "__main__":
    import bgdebias_b200.ops  # noqa: F401
    print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
    _log("kernel leg")
    print(json.dumps(kernel_alone()), flush=True)
    torch.cuda.empty_cache()
    print(json.dumps(end_to_end()), flush=True)
