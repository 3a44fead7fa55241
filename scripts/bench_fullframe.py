"""What coding whole images costs: full-frame containers (partial edge blocks, masked pixels not coded) against the
reference's cropped format and against naive padding.  One JSON line on stdout; writes nothing.

    python scripts/bench_fullframe.py [--images 100 --steps 3 --warmup 1 --lanes 4]

Workload: the crop benchmark's images (scripts/bench_crop.synthetic_crop_images(100, seed=0), H and W ~ U{224..512}) on
one GPU, the imagenetcrop model with random-init weights (imagenetcrop4 preset, tensor-core nets, free-running 4-lane
PipelinedCodec), every image ONE chain over its blocks, step = compress_images + decompress_images of every image.
Three arms, alternating inside every timed step:
  crop   compress_images(crop=True): h and w cropped to multiples of 32 (the reference's demo format; loses pixels)
  full   compress_images(crop=False): the whole image, partial edge blocks masked (only their valid pixels are coded)
  naive  every image edge-padded to multiples of 32 in numpy and coded with crop=True (the padding is coded too)
Per arm: pixels coded, Mpixel/s end to end (pixels coded / time), bits/dim over the dims that arm coded, and for the
full-frame arms bits per dim of the true image.  Random-init weights: the rates are not the paper's.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def power_limit_w():
    """The card's enforced power limit in W (read-only nvidia-smi query), or None."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                             text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:                                         # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=100)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--lanes", type=int, default=4)
    args = ap.parse_args()

    from bitswap_b200 import synthetic
    from bitswap_b200.config import preset
    from bitswap_b200.codec import PipelinedCodec, Bins
    from bitswap_b200.container import compress_images, decompress_images
    from scripts.bench_crop import synthetic_crop_images

    assert torch.cuda.is_available(), "needs a GPU (no CPU fallback for the product path)"
    torch.cuda.set_device(0)
    cfg = preset("imagenetcrop4")
    images = synthetic_crop_images(args.images, seed=0)
    padded = [np.pad(im, ((0, -im.shape[0] % 32), (0, -im.shape[1] % 32), (0, 0)), mode="edge") for im in images]
    crops = [im[:im.shape[0] - im.shape[0] % 32, :im.shape[1] - im.shape[1] % 32] for im in images]
    sd = synthetic.synthetic_state_dict(cfg, seed=50, varied=False)
    zend, zcen = synthetic.synthetic_bins(cfg, seed=0)
    lanes = max(1, min(args.lanes, len(images)))
    codec = PipelinedCodec(cfg, sd, Bins(cfg, zend, zcen), len(images), lanes=lanes, use_tensor_cores=True, free_running=True)
    arms = {"crop": (images, True, crops), "full": (images, False, images), "naive": (padded, True, padded)}

    def run(arm):
        ims, crop, _ = arms[arm]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        conts = compress_images(codec, ims, crop=crop)
        back = decompress_images(codec, conts)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, conts, back

    for _ in range(max(args.warmup, 1)):
        for arm in arms:
            run(arm)
    secs = {a: 0.0 for a in arms}
    last = {}
    for _ in range(args.steps):
        for arm in arms:                                      # alternating arms inside every step
            dt, conts, back = run(arm)
            secs[arm] += dt
            last[arm] = (conts, back)
    true_px = sum(im.shape[0] * im.shape[1] for im in images)
    res = {}
    for arm, (ims, crop, want) in arms.items():
        conts, back = last[arm]
        assert all(np.array_equal(a, b) for a, b in zip(want, back)), f"{arm}: round trip failed"
        px = sum(w.shape[0] * w.shape[1] for w in want)       # pixels this arm coded
        bits = sum(32 * (len(c) - 5) for c in conts)          # container words without the 5-word tail
        res[arm] = {"pixels_coded": int(px), "Mpixel_s": px * args.steps / secs[arm] / 1e6,
                    "ms_per_step": 1e3 * secs[arm] / args.steps, "bits_per_dim_coded": bits / (3 * px),
                    "bits_per_true_dim": bits / (3 * true_px) if arm != "crop" else None,
                    "containers_words": int(sum(len(c) for c in conts)), "roundtrip_ok": True}
    line = {"metric": "full-frame vs cropped vs naively padded whole-image coding (Bit-Swap, one GPU)",
            "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
            "images": args.images, "true_pixels": int(true_px), "steps": args.steps, "warmup": max(args.warmup, 1),
            "lanes": lanes, "model": "imagenetcrop4, random-init weights (seed 50), tensor-core nets", "data": "synthetic",
            "bits_note": "container bits include the borrowed initial-state words, as bench.py --config crop reports them",
            "arms": res,
            "full_vs_naive_bits_saved_per_padded_subpixel":
                (res["naive"]["containers_words"] - res["full"]["containers_words"]) * 32
                / max(1, 3 * (res["naive"]["pixels_coded"] - true_px))}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
