"""Buffer creation with augmentation (use_aug=True) from JPEG frames: the CPU oracle loader (oracle/image_ref.py, the
reference's per-image pipeline with a numpy rotation standing in for scikit-image's) against the GPU image path
(acezero_b200/imageprep.py + csrc/imageprep.cu).

Per frame size: write N JPEG frames, then time `TrainerACE.create_training_buffer` (one pass, W loader workers) for each
path, after a short warm-up fill of the same path. Reported per path:
  fill_images_per_s      images / wall time of the fill (ends in a device synchronise)
  main_cpu_ms_per_image  CPU time of the main thread during the fill / images (the per-image host work of the loop)
and, measured separately on already decoded items:
  prep_kernel_us_per_image   GPU path: CUDA events around the prep kernels + the mask-cells kernel, one image per call
  cpu_item_ms_per_image      oracle path: one worker's time for one item (decode + PIL + torchvision + numpy rotate)

    python tools/bench_image_prep.py [--frames 512] [--workers 12] [--out result.json]

The result is printed as one JSON line; `--out` also writes it to a file (profiles/bench_image_prep_r03.json came from
this tool).
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def options(out_dir, workers, samples):
    import train_ace
    o = train_ace.build_parser().parse_args(["frames", str(Path(out_dir) / "map.pt")])
    from acezero_b200.weights import random_encoder_state
    o.encoder_state_dict = random_encoder_state(77)
    o.num_data_workers = workers
    o.max_dataset_passes = 1
    o.samples_per_image = samples
    o.use_aug = True
    return o


def fill(ds, out_dir, workers, samples):
    from ace_trainer import TrainerACE
    tr = TrainerACE(options(out_dir, workers, samples), dataset=ds)
    torch.cuda.synchronize()
    t0, c0 = time.perf_counter(), time.thread_time()
    tr.create_training_buffer()
    torch.cuda.synchronize()
    wall, cpu = time.perf_counter() - t0, time.thread_time() - c0
    n = tr.images_encoded
    del tr
    torch.cuda.empty_cache()
    return {"images": n, "wall_s": wall, "fill_images_per_s": n / wall, "main_cpu_ms_per_image": 1e3 * cpu / n}


def prep_kernel_time(base, n_items=64, reps=5):
    from acezero_b200.encoder import out_hw
    from acezero_b200.imageprep import GpuImageDataset, ImagePrep
    ds = GpuImageDataset(base)
    items = []
    for i in range(n_items):
        it = ds[[i % len(ds)]]
        it["pixels"] = it["pixels"].pin_memory()
        items.append(it)
    prep = ImagePrep(torch.device("cuda"))
    outs = [torch.empty((1, 1) + tuple(it["size"]), dtype=torch.float16, device="cuda") for it in items]
    srcs = [it["pixels"].cuda() for it in items]   # device-resident sources: time the kernels, not the upload
    for it, s in zip(items, srcs):
        it["pixels"] = s

    def run():
        for it, o in zip(items, outs):
            prep.mask_cells(it, *out_hw(*it["size"]))
            prep.prepare([it], o)

    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    e1.synchronize()
    us = 1e3 * e0.elapsed_time(e1) / (reps * n_items)
    return {"prep_kernel_us_per_image": us, "items": n_items,
            "note": "CUDA events around mask-cells + prep kernels (incl. launch gaps), sources already on the device"}


def cpu_item_time(base, n_items=16):
    from oracle.image_ref import ImageRefDataset
    ds = ImageRefDataset(base)
    ds[[0]]
    t0 = time.perf_counter()
    for i in range(n_items):
        ds[[i % len(ds)]]
    return {"cpu_item_ms_per_image": 1e3 * (time.perf_counter() - t0) / n_items}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--workers", type=int, default=12)
    ap.add_argument("--samples", type=int, default=1024)
    ap.add_argument("--sizes", default="480x640,1080x1920")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    from acezero_b200.imageprep import GpuImageDataset
    from acezero_b200.synthetic import FrameDataset, write_frames
    from oracle.image_ref import ImageRefDataset
    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "frames": a.frames, "workers": a.workers, "samples_per_image": a.samples,
              "cpu_baseline": "oracle loader; rotation by the numpy restatement, not scikit-image", "sizes": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for spec in a.sizes.split(","):
            H, W = map(int, spec.split("x"))
            focal = 525.0 * H / 480
            files, poses = write_frames(Path(tmp) / spec, a.frames, H=H, W=W, focal=focal, ext="jpg", device="cuda")
            base = FrameDataset(files, poses, focal=focal)
            warm = FrameDataset(files[:24], poses[:24], focal=focal)
            r = {}
            for name, wrap in (("oracle_cpu", ImageRefDataset), ("gpu", GpuImageDataset)):
                fill(wrap(warm), tmp, a.workers, a.samples)
                r[name] = fill(wrap(base), tmp, a.workers, a.samples)
                print(spec, name, json.dumps(r[name]), flush=True)
            r["gpu"].update(prep_kernel_time(base))
            r["oracle_cpu"].update(cpu_item_time(base))
            result["sizes"][spec] = r
    result["gpu_after"] = gpu_info()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(result, indent=1))
    print(json.dumps(result))


if __name__ == "__main__":
    main()
