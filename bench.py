#!/usr/bin/env python
"""bench.py -- Bit-Swap encode+decode throughput on B200 (BASELINE.json metric).

A "step" = one pass of the hot path over one batch: Bit-Swap ENCODE of B images (one per ANS stream)
followed by Bit-Swap DECODE of the same B images, CIFAR-shaped 32x32x3 uint8, 8-latent VAE
(configs[1] of BASELINE.json: batch 1024 per GPU).  Decode restores every stream to its initial
state, so steps repeat without re-initialisation.

  value        Mpixel/s (pixel = H*W, 1024 per image) over encode+decode, inputs resident in HBM,
               CUDA-event timed, max over ranks; whole-job aggregate over N GPUs (weak scaling:
               per-GPU batch fixed, streams sharded by rank).  At N > 1 every step also gathers the
               produced bitstreams of all ranks over NCCL (device-resident, trimmed) between the
               encode and the decode -- the path's only collective, inside the timed region.
  e2e          same metric through the public Python/C-ABI API with HOST buffers: pinned uint8 pixels
               -> device -> encode -> trimmed bitstream to host -> back to device -> decode -> pixels
               to host, all copies inside the timed region.
  roofline     dominant kernel category, from CUDA events around every launch in a replay of the
               timed steps with the SAME launch shapes (the lanes run back to back instead of
               concurrently); traffic / FP64 instruction counts from the tracked ncu summary.
  cpu_baseline the oracle port of the reference path (torch-CPU nets + float64 tables + Python-loop
               ANS) on this box's host cores: latency mode with the 5-way time split and
               throughput mode (cores/16 processes of 16 threads, one chain each), bounded samples.

`--impl reference` times that CPU path as its own arm (the reference is pure Python and cannot be
pip-installed/travel; DESIGN.md).  `--config crop` is BASELINE configs[4]: 100 variable-size images as
chained 32x32 block streams over the GPUs, next to gzip/bz2/lzma/PNG/WebP on the host.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bitswap_b200 import synthetic                        # noqa: E402
from bitswap_b200.config import preset                    # noqa: E402

METRIC = "Mpixels/sec encode+decode (Bit-Swap, 32x32x3, 8-latent VAE)"
UNIT = "Mpixel/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def ncu_facts():
    """Per-kernel facts taken from the tracked ncu captures (profiles/ncu_facts_r2.json, written by
    scripts/ncu_summary.py facts): dram bytes per launch, FP64-pipe instructions per launch, streams per launch."""
    p = os.path.join(ROOT, "profiles", "ncu_facts_r2.json")
    return json.load(open(p)) if os.path.exists(p) else {}


# ----------------------------------------------------------------------------------------------------
# work accounting (DESIGN.md 5; SURVEY.md 6.3 / 8d)
# ----------------------------------------------------------------------------------------------------
def conv_flops(cfg):
    """Algorithmic 2*MAC of the UNPADDED reference convs per image and direction."""
    W, zc, C = cfg.reswidth, cfg.zchannels, cfg.xs[0]
    px = 256
    rd = cfg.level_resdepth
    d3 = 2 * px * W * 9 * W          # one 3x3 W->W conv
    d5 = 2 * px * W * 25 * W
    n3 = 2 * sum(rd) * 2             # infer+gen, conv1+conv2 per layer
    n5 = 2 * cfg.nprocessing * 2
    small = 2 * px * (4 * C * 25 * W) + (2 * cfg.nz - 1) * 2 * px * (zc * 9 * W) \
        + (2 * cfg.nz - 1) * 2 * px * (W * 9 * 2 * zc) + 2 * px * (W * 9 * 4 * C * (2 if cfg.cond_xscale else 1))
    return dict(dense3=d3, n3=n3, dense5=d5, n5=n5, small=small, total=n3 * d3 + n5 * d5 + small)


def ans_bytes(cfg):
    """Compulsory HBM bytes per image and direction: mu,sigma float32 + int16 symbol per symbol-op
    (x-level sigma is a shared parameter unless cond_xscale; the prior has neither)."""
    z, x, nz = cfg.zdim, cfg.xdim, cfg.nz
    return dict(pop_z=nz * z * 10, push_z=(nz - 1) * z * 10, push_x=x * (10 if cfg.cond_xscale else 6), prior=z * 2)


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw = [], [], []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        counts = {n: 0 for n in names}
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for nm, v in zip(names, r[3:7]):
                if "Active" in v and "Not" not in v:
                    counts[nm] += 1
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "power_w_median_under_load": float(np.median([p for p in pw if p > 0.5 * max(pw)] or pw)),
                "samples": len(sm), "reasons": sorted(n for n, c in counts.items() if c), "reason_samples": counts}


# ----------------------------------------------------------------------------------------------------
# CPU reference path (oracle port) -- bounded samples
# ----------------------------------------------------------------------------------------------------
_W = {}


def _cpu_setup(config, threads, coder="port"):
    from oracle import oracle as O
    torch.set_num_threads(threads)
    cfg = preset(config)
    sd = synthetic.synthetic_state_dict(cfg, seed=50, varied=False)
    zend, zcen = synthetic.synthetic_bins(cfg, seed=0)
    bs = O.BitSwapOracle(cfg, O.ModelOracle(cfg, sd), zend, zcen, coder=coder, pmf="torch")
    return cfg, bs, O


def cpu_chain(config, nimg, threads, seed=7, timers=False):
    """One chain of `nimg` images, encode then decode, on `threads` torch threads.  Returns
    (seconds_encode, seconds_decode, net bits/dim, split dict or None)."""
    key = (config, threads)
    if key not in _W:
        _W[key] = _cpu_setup(config, threads)
    cfg, bs, O = _W[key]
    torch.set_num_threads(threads)
    bs.timers = {} if timers else None
    imgs = synthetic.synthetic_images(cfg, nimg, seed=seed)
    w, head = synthetic.initial_words(4096, seed=100)
    st = [int(v) for v in w] + [head]
    n0 = len(st)
    t0 = time.perf_counter()
    for i in range(nimg):
        st = bs.encode_image(st, imgs[i])
    t1 = time.perf_counter()
    n1 = len(st)
    for i in reversed(range(nimg)):
        st, x = bs.decode_image(st)
        assert np.array_equal(x, imgs[i].reshape(-1))
    t2 = time.perf_counter()
    split = None
    if timers:
        tot = sum(bs.timers.values()) or 1.0
        split = {k: v / tot for k, v in sorted(bs.timers.items())}
    return t1 - t0, t2 - t1, 32.0 * (n1 - n0) / (cfg.xdim * nimg), split


def _tp_worker(args):
    """Throughput-mode worker: one process with `threads` torch threads = one chain of one image, encode + decode."""
    config, seed, threads = args
    e, d, _, _ = cpu_chain(config, 1, threads, seed=seed)
    return e + d


def _tp_init(config, threads):
    os.environ["OMP_NUM_THREADS"] = str(threads)
    torch.set_num_threads(threads)
    _W[(config, threads)] = _cpu_setup(config, threads)
    cpu_chain(config, 1, threads)                             # warm-up inside the worker (first-call costs)


class ThroughputPool:
    """All host cores on the reference's CPU path (BASELINE.md 3, throughput mode): `procs` worker processes of `threads`
    torch threads each, procs x threads = cores, every worker its own chain.  16 threads per chain is where the path's torch
    ops stop scaling for one chain.  One single-threaded process per core was measured too and is the stronger aggregate
    (profiles/bench_r2_reference_arm_1thread.json: 0.0026 against 0.0018 Mpixel/s on 128 cores) but needs 48 s per image,
    i.e. 20 minutes for the 25-step arm the driver launches; the line says so (`single_thread_per_core`)."""

    def __init__(self, config, procs, threads):
        import multiprocessing as mp
        self.config, self.procs, self.threads = config, procs, threads
        self.pool = mp.get_context("spawn").Pool(procs, initializer=_tp_init, initargs=(config, threads))

    def step(self, step_index=0):
        """Every worker codes one image (encode + decode); returns (wall seconds, images)."""
        t0 = time.perf_counter()
        self.pool.map(_tp_worker, [(self.config, 1000 + step_index * self.procs + i, self.threads) for i in range(self.procs)], chunksize=1)
        return time.perf_counter() - t0, self.procs

    def close(self):
        self.pool.close()
        self.pool.join()


def host_procs(threads=16):
    """(worker processes, threads per worker) covering the host cores (bounded by free memory: ~2 GB per worker)."""
    cores = os.cpu_count() or 1
    threads = max(1, min(threads, cores))
    n = max(1, cores // threads)
    try:
        import psutil
        n = min(n, max(1, int(psutil.virtual_memory().available // (2 << 30))))
    except Exception:
        pass
    return n, threads


def run_reference_arm(args, cfg, rank, world):
    """The reference's own CPU implementation of the path, with all the host threads it can use: `procs` processes of
    16 threads, each coding its own chain (the reference is strictly batch 1).  A step = every worker encodes and decodes one
    image (about 1.5 s of wall time, so a 25-step arm ends within a minute)."""
    if rank != 0:
        return
    procs, threads = host_procs()
    if args.ref_procs:
        procs = args.ref_procs
    pool = ThroughputPool(args.config, procs, threads)
    for i in range(args.warmup):
        pool.step(10000 + i)
    wall, imgs = 0.0, 0
    for i in range(args.steps):
        w, n = pool.step(i)
        wall += w; imgs += n
    pool.close()
    e, d, bpd, split = cpu_chain(args.config, 2, threads, timers=True)
    val = imgs * 1024 / wall / 1e6
    sample = (f"throughput mode: {procs} worker processes x {threads} torch threads (of {os.cpu_count()} host cores), each step every "
              f"worker encodes + decodes one image of its own chain (the reference is strictly batch 1)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 tables / f32 nets / int64 coder", "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfg.xs[1]}x{cfg.xs[2]}x{cfg.xs[0]} uint8, nz={cfg.nz}, W={cfg.reswidth}; {sample}",
                       "what_runs": "oracle port of the reference path (torch-CPU nets, torch float64 logistic tables, "
                                    "Python-loop ANS with Python ints) -- the reference itself is pure Python and cannot travel"},
            "bits_per_dim": bpd,
            "latency_mode": {"threads": threads, "encode_s_per_image": e / 2, "decode_s_per_image": d / 2,
                             "Mpixel_s": 2 * 1024 / (e + d) / 1e6, "time_split": split,
                             "sample": "one 2-image chain alone on the box"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs * threads, "kind": "port", "sample": sample,
                             "single_thread_per_core": "measured once on this pool's 128-core host: 0.0026 Mpixel/s, 48 s per step "
                                                       "(profiles/bench_r2_reference_arm_1thread.json) -- 1.45x this arm's rate"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline_block(config, images, tp_steps):
    """cpu_baseline of the GPU arm's line: latency mode (one chain alone on the box, 16 threads, 5-way split) + throughput
    mode (all cores: processes x 16 threads, one chain each)."""
    procs, threads = host_procs()
    cpu_chain(config, 1, threads)
    e, d, bpd, split = cpu_chain(config, images, threads, timers=True)
    out = {"unit": UNIT, "kind": "port",
           "latency_mode": {"threads": threads, "Mpixel_s": images * 1024 / (e + d) / 1e6, "encode_s_per_image": e / images,
                            "decode_s_per_image": d / images, "bits_per_dim": bpd, "time_split": split,
                            "sample": f"one {images}-image chain (batch 1), encode then decode"}}
    pool = ThroughputPool(config, procs, threads)
    pool.step(999)
    wall, imgs = 0.0, 0
    for i in range(tp_steps):
        w, n = pool.step(i)
        wall += w; imgs += n
    pool.close()
    out.update(value=imgs * 1024 / wall / 1e6, cores=procs * threads,
               single_thread_per_core="measured once on this pool's 128-core host: 0.0026 Mpixel/s "
                                      "(profiles/bench_r2_reference_arm_1thread.json)",
               sample=f"throughput mode: {procs} processes x {threads} torch threads x {tp_steps} image(s) each, encode + decode "
                      f"({os.cpu_count()} host cores); latency mode beside it")
    return out


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
def states_digest(ss, first=0, count=None):
    """sha256 over (word count, head, words) of the streams -- what H3 / SURVEY 8e say must not depend on G."""
    words, offs, heads, _ = ss.export(first, count)
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(offs).tobytes()); h.update(np.ascontiguousarray(heads).tobytes()); h.update(np.ascontiguousarray(words).tobytes())
    return h.hexdigest()[:16]


DUMP_BYTES = 64 << 20


def dump_outputs(path, codec, ss, x_dev, out_dev, digest):
    """Writes what the last timed step handed its caller, as DIR/<name>.npy, so that two builds can be compared output
    for output:
      pixels   float32 [n, C, H, W]  the decoded images of the last step (still in out_dev)
      words    float64 [sum]         each stream's trimmed bitstream (the words above the lowest depth it reached), concatenated
      lengths  float64 [n]           words per stream in `words`
      base     float64 [n]           that lowest depth: the seed words below it are not part of the bitstream
      heads    float64 [n, 2]        the 64-bit ANS heads as (low, high) 32-bit halves
      streams  float64 [n]           which streams these are
    The step's decode consumed the bitstreams its encode produced, so they are produced again here, outside the timed
    region, by encoding the same images onto the same initial states; their digest must equal that of the untimed first
    encode, i.e. every step coded the same words.  n is every stream unless 64 MB cannot hold them (bounded by the stream
    capacity, so n depends on the arguments only); then it is a fixed seeded sample."""
    B = ss.n
    pixels = out_dev.cpu().numpy()
    codec.encode(ss, x_dev)
    torch.cuda.synchronize()
    ss.raise_on_error()
    assert states_digest(ss) == digest, "the re-encoded streams differ from the first encode of the same images"
    words, offs, heads, base = (a.copy() for a in ss.export_packed(trim=True))
    codec.decode(ss, B, out=out_dev)
    torch.cuda.synchronize()
    ss.raise_on_error()
    assert torch.equal(out_dev, x_dev), "round trip failed"
    n = min(B, DUMP_BYTES // (8 * ss.capacity + 8 * 5 + 4 * pixels[0].size))
    idx = np.arange(B) if n == B else np.sort(np.random.RandomState(0).choice(B, n, replace=False))
    arrays = {"pixels": pixels[idx].astype(np.float32),
              "words": np.concatenate([words[offs[i]:offs[i + 1]] for i in idx]).astype(np.float64),
              "lengths": np.diff(offs)[idx].astype(np.float64),
              "base": base[idx].astype(np.float64),
              "heads": np.stack([heads[idx] & 0xffffffff, heads[idx] >> 32], axis=1).astype(np.float64),
              "streams": idx.astype(np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cifar8", help="cifar8 (BASELINE configs[1], default), imagenet4, mnist2, ..., or crop (configs[4])")
    ap.add_argument("--batch", type=int, default=0, help="streams (= images per step) PER GPU (default 1024; imagenet4: 4096)")
    ap.add_argument("--tensor-cores", type=int, default=-1, help="-1 auto, 0 SIMT fp32 convs, 1 tcgen05")
    ap.add_argument("--ref-procs", type=int, default=0, help="worker processes (of 16 threads) of the CPU reference arm (0 = cores / 16)")
    ap.add_argument("--cpu-baseline-images", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=4, help="sub-batches coded concurrently on separate CUDA streams (1 = off)")
    ap.add_argument("--lane-size", type=int, default=0, help="streams per lane (0 = batch/lanes); the last lane takes the remainder")
    ap.add_argument("--free-running", type=int, default=1, help="1: the lanes are joined once at the end of the timed region instead of after "
                    "every encode/decode call (keeps their phase offsets); forced off when a collective needs all lanes (N > 1)")
    ap.add_argument("--dual-stream", type=int, default=-1, help="codec stream mode (bsw_codec_set_dual_stream); -1 = library default")
    ap.add_argument("--fused-coder", action="store_true", help="one-warp-per-stream fused coder kernels instead of the two-phase coder")
    ap.add_argument("--crop-images", type=int, default=100)
    ap.add_argument("--hwc-quirk", action="store_true", help="crop: feed blocks as imagenetcrop_compress.py:130 does")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the pixels and bitstreams of the last step "
                    "as DIR/<name>.npy (float32/float64, at most 64 MB; rank 0's streams)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "crop"):
        ap.error("--dump-outputs writes the outputs of the GPU arm's per-image configurations (not --impl reference or --config crop)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config == "crop":
        from scripts.bench_crop import run_crop
        return run_crop(args, rank, world, local)
    cfg = preset(args.config)

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank, world)
        return

    import torch.distributed as dist
    from bitswap_b200.model import Model
    from bitswap_b200.codec import BitSwapCodec, Bins, PipelinedCodec
    from bitswap_b200.streams import StreamSet
    from bitswap_b200 import _lib, parallel

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    peaks = measured_peaks()
    facts = ncu_facts()

    B = args.batch or (4096 if args.config == "imagenet4" else 1024)
    use_tc = args.tensor_cores
    if use_tc < 0:
        use_tc = 1 if (_lib.has_tensor_core_path() and (cfg.reswidth + 63) // 64 * 64 == 256) else 0
    sd = synthetic.synthetic_state_dict(cfg, seed=50, varied=False)          # default-init distribution (SURVEY.md 8d)
    zend, zcen = synthetic.synthetic_bins(cfg, seed=0)
    bins = Bins(cfg, zend, zcen)
    lanes = max(1, args.lanes)
    codec = PipelinedCodec(cfg, sd, bins, B, lanes=lanes, use_tensor_cores=bool(use_tc), lane_size=args.lane_size)
    free_running = bool(args.free_running) and world == 1 and lanes > 1
    two_phase = not args.fused_coder
    codec.set_two_phase(two_phase)
    if args.dual_stream >= 0:
        codec.set_dual_stream(args.dual_stream)
    INIT_WORDS = 4096
    ss = StreamSet(B, INIT_WORDS + 2048)
    w, head = synthetic.initial_words(INIT_WORDS, seed=100)
    ss.fill(w, head)
    # images are seeded by the GLOBAL stream index block: rank r codes exactly what a 1-GPU run with seed 7+r codes
    x_host = torch.from_numpy(synthetic.synthetic_images(cfg, B, seed=7 + rank)).pin_memory()
    x_dev = x_host.to(dev)
    out_dev = torch.empty_like(x_dev)
    out_host = torch.empty_like(x_host).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- correctness outside the timed region: round trip, bits/dim, digest of the coded streams ---------------
    n0, _, _ = ss.sizes()
    codec.encode(ss, x_dev)
    torch.cuda.synchronize()
    n1, _, f1 = ss.sizes()
    launches_enc = codec.last_launches
    acct = ss.bit_accounting(INIT_WORDS, cfg.xdim, 1)
    digest = states_digest(ss)
    sample_n = min(16, B)
    digest_head = states_digest(ss, 0, sample_n)               # first streams of this rank (cross-rank determinism check below)
    codec.decode(ss, B, out=out_dev)
    torch.cuda.synchronize()
    n2, h2, f2 = ss.sizes()
    launches_dec = codec.last_launches
    roundtrip_ok = bool(torch.equal(out_dev, x_dev) and np.array_equal(n2, n0) and not f1.any() and not f2.any()
                        and (h2 == np.uint64(head)).all())
    assert roundtrip_ok, "round trip failed"

    # ---- device-resident timing --------------------------------------------------------------------------------
    def gather_step():
        """The path's only collective: every rank receives every rank's PRODUCED words (trimmed), device to device."""
        wd, od, hd, bd = ss.pack_device(trim=True)
        lens = od[1:] - od[:-1]
        return parallel.gather_packed(wd, lens, hd, bd)

    for _ in range(max(args.warmup, 3)):
        codec.encode(ss, x_dev)
        if world > 1:
            gather_step()
        codec.decode(ss, B, out=out_dev)
    barrier()
    # free-running lanes: every lane chains its own encode -> decode -> encode ...; ONE join before the closing event, so the
    # timed region still contains all the work of its K steps (per-direction times are then not separable: a lane may be
    # decoding while its neighbour encodes)
    codec.free_running = free_running
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * args.steps + 1)]
    ev[0].record()
    gathered_words = 0
    for i in range(args.steps):
        codec.encode(ss, x_dev)
        ev[3 * i + 1].record()
        if world > 1:
            W, M, counts = gather_step()
        ev[3 * i + 2].record()
        codec.decode(ss, B, out=out_dev)
        if free_running and i == args.steps - 1:
            codec.join()
        ev[3 * i + 3].record()
    torch.cuda.synchronize()
    codec.free_running = False
    total_ms = ev[0].elapsed_time(ev[-1])
    enc_ms = sum(ev[3 * i].elapsed_time(ev[3 * i + 1]) for i in range(args.steps))
    gat_ms = sum(ev[3 * i + 1].elapsed_time(ev[3 * i + 2]) for i in range(args.steps))
    dec_ms = sum(ev[3 * i + 2].elapsed_time(ev[3 * i + 3]) for i in range(args.steps))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, codec, ss, x_dev, out_dev, digest)
    gather_info = None
    if world > 1:
        gathered_words = int(counts[:, 0].sum())
        # what arrived must be what was sent: every rank's slice re-imported into fresh streams decodes to that rank's pixels
        # (checked on rank 0 for the LAST rank's shard: a different GPU coded it)
        gather_info = {"words_gathered_per_step": gathered_words, "bytes_per_image": 4.0 * gathered_words / (B * world),
                       "streams": int(counts[:, 1].sum())}
    # ---- per-kernel times: the same steps with the lanes run back to back (identical launch shapes) ---------------
    codec.serial = True
    codec.set_dual_stream(0)
    for _ in range(1):
        codec.encode(ss, x_dev)
        codec.decode(ss, B, out=out_dev)
    codec.profile(True)
    for i in range(args.steps):
        codec.encode(ss, x_dev)
        codec.decode(ss, B, out=out_dev)
    prof = codec.profile(False)
    torch.cuda.synchronize()
    assert torch.equal(out_dev, x_dev)
    codec.serial = False
    if args.dual_stream > 0:
        codec.set_dual_stream(args.dual_stream)
    barrier()
    t = torch.tensor([total_ms, enc_ms, dec_ms, gat_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, enc_ms, dec_ms, gat_ms = t.tolist()
    px_job = world * B * 1024 * args.steps
    value = px_job / (total_ms * 1e-3) / 1e6

    # ---- end to end with host buffers (trimmed bitstreams both ways) ---------------------------------------------
    def e2e_step():
        x_d = x_host.to(dev, non_blocking=True)                                   # H2D pixels
        codec.encode(ss, x_d)
        words, offs, heads, base = ss.export_packed(trim=True)                    # device gather + D2H produced words, offsets, heads, bases
        nbytes = int(words.nbytes + offs.nbytes + heads.nbytes + base.nbytes)
        ss.import_packed_fast(words, offs, heads, base=base)                      # H2D + device scatter (the receiver's side: it holds the seed words)
        o = codec.decode(ss, B, out=out_dev)
        out_host.copy_(o, non_blocking=True)                                      # D2H pixels
        torch.cuda.synchronize()
        return nbytes

    bs_bytes = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        bs_bytes = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = t.item()
    e2e_val = px_job / e2e_s / 1e6
    assert torch.equal(out_host, x_host)
    _, _, f3 = ss.sizes()
    assert not f3.any()

    # ---- cross-G determinism (H3, SURVEY 8e): the streams a rank coded == what ANOTHER GPU codes for the same seeds ----
    digests, determinism = [digest], None
    if world > 1:
        objs = [None] * world
        dist.all_gather_object(objs, {"rank": rank, "digest": digest, "head": digest_head})
        digests = [o["digest"] for o in objs]
        if rank == 0:
            peer = world - 1
            xs = torch.from_numpy(synthetic.synthetic_images(cfg, B, seed=7 + peer)[:sample_n]).to(dev)
            m2 = Model.from_config(cfg, max_batch=sample_n, use_tensor_cores=bool(use_tc)).load_state_dict(sd)
            m2.compress()
            c2 = BitSwapCodec(cfg, m2, bins, sample_n)
            s2 = StreamSet(sample_n, INIT_WORDS + 2048)
            s2.fill(w, head)
            c2.encode(s2, xs)
            torch.cuda.synchronize()
            mine = states_digest(s2)
            determinism = {"peer_rank": peer, "streams": sample_n, "peer_digest": objs[peer]["head"], "recoded_here_digest": mine,
                           "equal": mine == objs[peer]["head"], "note": "other GPU, other batch size (16 vs the lane size), other position"}
            assert determinism["equal"], "stream states depend on which GPU / batch coded them"

    # ---- roofline for the dominant kernel category ---------------------------------------------------------------
    fl, ab = conv_flops(cfg), ans_bytes(cfg)
    fp64_peak = _lib.measure_fp64_peak()                                     # DFMA lanes/s, measured on this GPU
    Bl = codec.per                                                           # images per kernel launch (lane size)
    per_launch = {
        "conv_dense5x5": ("tensor", fl["dense5"] * Bl), "conv_dense3x3": ("tensor", fl["dense3"] * Bl),
        "rows_z": ("hbm", cfg.zdim * 10 * Bl), "rows_x": ("hbm", ab["push_x"] * Bl),
        "pop_z": ("hbm", cfg.zdim * 10 * Bl), "push_z": ("hbm", cfg.zdim * 10 * Bl),
        "pop_x": ("hbm", ab["push_x"] * Bl), "push_x": ("hbm", ab["push_x"] * Bl),
    }
    kernels = {}
    tot_ms = max(sum(v[0] for v in prof.values()), 1e-9)
    for k, (ms, n) in prof.items():
        if n == 0:
            continue
        rec = {"ms_per_step": ms / args.steps, "launches_per_step": n / args.steps, "avg_ms": ms / n, "share": ms / tot_ms}
        if k in per_launch:
            bound, work = per_launch[k]
            sec = ms / n * 1e-3
            if bound == "tensor":
                rec.update(bound="tensor", achieved=work / sec / 1e12, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                           mma_tflops_issued=3 * work * (256 / cfg.reswidth) ** 2 / sec / 1e12 if use_tc else None)
            else:
                rec.update(bound="hbm", achieved=work / sec / 1e9, peak=peaks["hbm_gbs"], unit="GB/s", algorithmic_bytes_per_launch=work)
            rec["frac"] = rec["achieved"] / rec["peak"]
            fk = facts.get(k)
            if fk and fk.get("streams_per_launch"):
                scale = Bl / fk["streams_per_launch"]
                rec["traffic"] = fk["dram_bytes_per_launch"] * scale
                rec["traffic_source"] = fk.get("source")
                if fk.get("fp64_inst_per_launch"):
                    lanes_per_s = 32.0 * fk["fp64_inst_per_launch"] * scale / sec
                    rec["fp64"] = {"warp_instructions_per_launch": fk["fp64_inst_per_launch"] * scale, "achieved_lanes_per_s": lanes_per_s,
                                   "peak_measured_dfma_lanes_per_s": fp64_peak, "frac": lanes_per_s / fp64_peak,
                                   "source": "sm__inst_executed_pipe_fp64 of " + str(fk.get("source"))}
        kernels[k] = rec
    # dominant kernel: among the THROUGHPUT kernels (tables, convs).  The serial coder kernels are latency-bound -- their
    # duration does not depend on the stream count, so the lane-by-lane replay counts them once per lane although in the
    # timed region the lanes' copies run side by side.
    dom = max((k for k in kernels if "bound" in kernels[k] and (k.startswith("conv") or k.startswith("rows"))),
              key=lambda k: kernels[k]["ms_per_step"])
    roofline = {"kernel": dom, "bound": kernels[dom]["bound"], "achieved": kernels[dom]["achieved"], "peak": kernels[dom]["peak"],
                "unit": kernels[dom]["unit"], "frac": kernels[dom]["frac"], "traffic": kernels[dom].get("traffic"),
                "traffic_source": kernels[dom].get("traffic_source"),
                "peak_source": peaks["source"] + (" bf16_tflops_sustained" if kernels[dom]["bound"] == "tensor" else " hbm_gbs"),
                "share_of_step": kernels[dom]["share"], "streams_per_launch": Bl}
    if "fp64" in kernels[dom]:
        roofline["fp64"] = kernels[dom]["fp64"]
    if kernels[dom]["bound"] == "hbm":
        roofline["note"] = ("the coder's table kernel is bound by float64 arithmetic, not HBM ((S-1) float64 logistic values per "
                            "symbol-op, SURVEY.md 8d/H2): the hbm fraction is the contract's figure; `fp64` is the FP64-pipe "
                            "instruction count of the tracked ncu capture against the measured DFMA peak")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 tables / int64 coder / " + ("bf16x3 split tcgen05" if use_tc else "f32 SIMT") + " convs",
            "coder": "two-phase (parallel f64 row tables + serial integer coder)" if two_phase else "fused one-warp-per-stream",
            "lanes": codec.lanes,
            "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfg.xs[1]}x{cfg.xs[2]}x{cfg.xs[0]} uint8, nz={cfg.nz}, W={cfg.reswidth}, q={cfg.quantbits}; "
                                   f"{B} independent ANS streams per GPU x 1 image per step; step = Bit-Swap encode"
                                   + (" + NCCL gather of the produced bitstreams" if world > 1 else "") + " + decode",
                       "streams_per_gpu": B, "global_batch": B * world, "weights": "seeded random init (reference default-init distribution)",
                       "bins": "synthetic uniform grids + float32 equal-mass top level", "images": "iid uniform uint8",
                       "l2": "per-step working set (3 x 268 MB activations + streams) >> 126 MB L2: no explicit flush needed",
                       "parallelism": f"streams sharded over {world} GPU(s); within a GPU {codec.lanes} sub-batches of {Bl} on separate CUDA streams"},
            "encode_Mpixel_s": None if free_running else px_job / (enc_ms * 1e-3) / 1e6,
            "decode_Mpixel_s": None if free_running else px_job / (dec_ms * 1e-3) / 1e6,
            "lanes_free_running": free_running,
            "Mdim_s": value * cfg.xs[0],
            "bits_per_dim": float(acct["net_bits_per_dim"].mean()),
            "bits": {"net_bits_per_dim": float(acct["net_bits_per_dim"].mean()),
                     "cma_bits_per_dim_incl_initial_bits": float(acct["cma_bits_per_dim"].mean()),
                     "total_bits_per_stream": float(acct["total_bits"].mean()),
                     "definition": "cifar_compress.py:253-259: net = (len(state) - len(initialstate)) * 32 / xdim; "
                                   "cma = (len(state) - (len(restbits) - 1)) * 32 / (xdim * images), restbits = state after the first pop; "
                                   "1 image per chain here, so cma is the reference's CMA@1"},
            "roundtrip_ok": roundtrip_ok, "stream_digests": digests,
            "gpu_launches": (launches_enc + launches_dec + (2 if world > 1 else 0)) * args.steps,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(x_host.numel() + bs_bytes),
                    "d2h_bytes_per_step": int(bs_bytes + out_host.numel()), "ms_per_step": 1e3 * e2e_s / args.steps,
                    "bitstream_bytes_per_image": bs_bytes / B},
            "roofline": roofline, "kernels": kernels, "clocks": clocks,
            "kernels_timing": (f"CUDA events around every launch in a replay of the same {args.steps} steps with the {codec.lanes} lanes run back "
                               f"to back on one stream: identical kernels and launch shapes ({Bl} streams per launch) as the timed region, "
                               "which runs the lanes concurrently (there per-kernel event times overlap and cannot be attributed)")}
    if world > 1:
        line["bitstream_gather"] = dict(gather_info, ms_per_step=gat_ms / args.steps, inside_timed_region=True,
                                        how="StreamSet.pack_device(trim) -> parallel.gather_packed: 3 all_gather_into_tensor (NCCL), device resident")
        line["bitstream_gather_ms"] = gat_ms / args.steps
        line["cross_gpu_determinism"] = determinism
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        del codec
        torch.cuda.empty_cache()
        line["cpu_baseline"] = cpu_baseline_block(args.config, args.cpu_baseline_images, 3)
    if world > 1:
        dist.barrier()
    if rank == 0:
        sys.stdout.flush()
        print(json.dumps(line), flush=True)                  # LAST thing on stdout (NCCL is free to print its banner before)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
