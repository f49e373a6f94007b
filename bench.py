#!/usr/bin/env python
"""Benchmark of the sam_road tiled-inference hot path on B200 (see DESIGN.md).

    python bench.py --gpus 1 --steps 20 --warmup 3                # this framework (CUDA, sm_100a)
    python bench.py --dump-outputs DIR                            # + the last timed step's results as DIR/*.npy
    python bench.py --workload c4                                 # another BASELINE configuration
    python bench.py --impl reference --steps 3 --warmup 1         # reference algorithm on host CPU cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Default workload (BASELINE.json configs[1], `toponet_vitb_512_cityscale`): one "step" is one pass of the
hot path over one INFER_BATCH_SIZE=64 batch of synthetic 512x512 RGB tiles per GPU: ViT-B encoder + naive
mask decoder + TopoNet on 256 keypoints x 16 neighbour pairs per tile.  Weights are seeded random
tensors with the reference's state_dict layout; data is synthetic (no network for datasets/ckpts).

Printed JSON (one line, rank 0):
  value      tiles/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the host-buffer C-ABI call (pinned host tiles in, results out), the two
             staging slots alternating so that a batch's downloads overlap the next batch's upload + compute
  e2e_scene  whole scenes through the drop-in `infer_one_img` (uint8 scene in host memory -> nodes, edges
             and the two uint8 masks in host memory): tiles/s = tiles of the scene / wall time
  roofline   dominant kernel class: algorithmic FLOPs / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (port of the reference algorithm) timed on this box's host cores
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_BASE = dict(USE_SAM_DECODER=False, ENCODER_LORA=False, TOPONET_VERSION="normal", NO_SAM=False,
             INFER_BATCH_SIZE=64)
TOPO_FLOP_PER_POINT = 10.89e6 + 65.5e3      # per 16-pair sample + feature_proj per keypoint (SURVEY.md §8d)
# BASELINE.json configs; algorithmic FLOPs per tile from SURVEY.md §8d (encoder + decoder), TopoNet added per point
WORKLOADS = {
    "c1": dict(name="toponet_vitb_256", cfg=dict(_BASE, SAM_VERSION="vit_b", PATCH_SIZE=256), points=0,
               flop_tile=46.33e9, metric="256x256 ViT-B tiles/sec",
               note="encoder + mask head only (the reference's CPU-runnable case), 64 tiles per step"),
    "c2": dict(name="toponet_vitb_512_cityscale", cfg=dict(_BASE, SAM_VERSION="vit_b", PATCH_SIZE=512),
               points=256, flop_tile=195.34e9, metric="512x512 ViT-B tiles/sec",
               note="encoder + decoder + TopoNet, 256 keypoints x 16 pairs per tile"),
    "c3": dict(name="toponet_vitb_256_spacenet", cfg=dict(_BASE, SAM_VERSION="vit_b", PATCH_SIZE=256),
               points=64, flop_tile=46.33e9, metric="256x256 ViT-B tiles/sec",
               note="encoder + decoder + TopoNet, 64 keypoints x 16 pairs per tile"),
    "c4": dict(name="toponet_vitb_512_cityscale_8x8", cfg=dict(_BASE, SAM_VERSION="vit_b", PATCH_SIZE=512),
               points=1024, flop_tile=195.34e9, metric="512x512 ViT-B tiles/sec",
               note="dense TopoNet: 1024 keypoints x 16 pairs per tile (16 384 sequences of 16)"),
    "c5": dict(name="toponet_vith_256", cfg=dict(_BASE, SAM_VERSION="vit_h", PATCH_SIZE=256), points=0,
               flop_tile=330.98e9, metric="256x256 ViT-H tiles/sec",
               note="ViT-H encoder + mask head (head_dim 80)"),
    "c2_samdec": dict(name="toponet_vitb_512_cityscale + USE_SAM_DECODER",
                      cfg=dict(_BASE, SAM_VERSION="vit_b", PATCH_SIZE=512, USE_SAM_DECODER=True), points=256,
                      flop_tile=194.50e9 + 0.91e9, metric="512x512 ViT-B tiles/sec",
                      note="SAM TwoWayTransformer mask decoder instead of the naive decoder"),
}
# scene-level legs (e2e_scene): the grids of the reference's inference configs
SCENES = {
    "c2": [dict(tag="cityscale_2048_16x16", size=2048, per_edge=16, margin=64)],
    "c3": [dict(tag="spacenet_400_16x16", size=400, per_edge=16, margin=0)],
    "c4": [dict(tag="cityscale_2048_8x8", size=2048, per_edge=8, margin=64)],
}
SCENE_KEYS = dict(TOPO_THRESHOLD=0.5, ITSC_NMS_RADIUS=8, ROAD_NMS_RADIUS=16, NEIGHBOR_RADIUS=64,
                  MAX_NEIGHBOR_QUERIES=16)


def flop_per_tile(w):
    return w["flop_tile"] + w["points"] * TOPO_FLOP_PER_POINT


DUMP_MAX_VALUES = 4 << 20       # per output (16 MiB of float32): the three outputs stay below 64 MB together


def dump_outputs(out_dir, outputs):
    """Write each result of the last timed step as out_dir/<name>.npy in float32 (None: the workload has
    no such output).  An output with more than DUMP_MAX_VALUES elements is stored as a fixed sample: the
    values at seeded random flat indices, in ascending index order, so that two builds run with the same
    arguments write comparable files."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if t is None:
            continue
        t = t.detach().float()
        if t.numel() > DUMP_MAX_VALUES:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_VALUES]
            t = t.reshape(-1)[idx.sort().values.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=float(p["bf16_tflops_sustained"]), tflops_burst=float(p["bf16_tflops"]),
                    hbm=float(p["hbm_gbs"]), source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0,
                source="fallback (B200_PROFILING.md)")


def load_ncu_metrics():
    """Per-kernel-class ncu numbers (DRAM bytes per launch, tensor-pipe %) written by tools/ncu_extract.py
    from the `--set full` captures of tools/gpu/profile_r02.sh, stamped with the digest of the kernel sources
    they were taken from.  Returned only when that digest is the one of the library being run."""
    path = os.path.join(ROOT, "profiles", "ncu_metrics.json")
    dig = os.path.join(ROOT, "sam_road_b200", "_build", "digest.txt")
    if not (os.path.exists(path) and os.path.exists(dig)):
        return None, "no profiles/ncu_metrics.json for this build"
    m = json.load(open(path))
    if m.get("digest") != open(dig).read().strip():
        return None, "profiles/ncu_metrics.json was captured from other kernel sources (digest differs)"
    return m, m.get("source", "profiles/ncu_metrics.json")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML every 10 ms when the binding
    is importable (nvidia-ml-py), else one nvidia-smi query per 150 ms."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None
        self.source = "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
            self.source = "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
        try:
            watts = n.nvmlDeviceGetPowerUsage(self._h) / 1000.0
        except Exception:
            watts = float("nan")
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        bits = [getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)]
        self.rows.append([str(sm), str(self._max), str(watts)] +
                         ["Active" if mask & b else "Not Active" for b in bits])

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True,
                                         text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.01 if self._nvml is not None else 0.15)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        def num(x):
            try:
                return float(x)
            except Exception:
                return None
        sm = sorted(v for v in (num(r[0]) for r in self.rows if r) if v is not None)
        reasons = set()
        for r in self.rows:
            for n, v in zip(self.NAMES, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max((v for v in (num(r[1]) for r in self.rows if len(r) > 1) if v is not None), default=None)
        pw = [v for v in (num(r[2]) for r in self.rows if len(r) > 2) if v is not None and v == v]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "sm_mhz_min": sm[0] if sm else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "source": self.source}



# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle (CPU port of the reference algorithm) on host cores
# ------------------------------------------------------------------------------------------------
def time_cpu_oracle(w, n_tiles: int, steps: int, warmup: int):
    import torch
    from oracle import samroad_oracle as O          # the only place bench.py executes oracle/
    from sam_road_b200 import synth
    cfg, P, NP = w["cfg"], w["cfg"]["PATCH_SIZE"], w["points"]
    spec = O.ModelSpec.from_config(cfg)
    sd = synth.make_state_dict(cfg, seed=0)
    rgb = synth.make_tiles(n_tiles, P, seed=11, dtype=torch.float32)
    topo = synth.make_topo_inputs(n_tiles, P, NP, seed=12, ragged=False) if NP else None
    # all the host threads the process can really use: the affinity mask / cgroup quota may be far
    # below os.cpu_count() on a shared box, and oversubscribed eager PyTorch is several times slower,
    # so probe a few thread counts on one tile and keep the fastest
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            avail = max(1, min(avail, int(int(quota) / int(period))))
    except Exception:
        pass
    cands = sorted({avail, min(avail, 64), min(avail, 32), min(avail, 16), min(avail, 8)}, reverse=True)
    best_t, cores = None, avail
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            O.image_encoder(O.normalize_rgb(rgb[:1]), sd, spec)          # warm
            t0 = time.perf_counter()
            O.image_encoder(O.normalize_rgb(rgb[:1]), sd, spec)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best_t, cores = dt, c
    torch.set_num_threads(cores)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            _, feat = O.infer_masks_and_img_features(sd, spec, rgb)
            if topo:
                O.infer_toponet(sd, spec, feat, *topo)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    total = sum(times)
    return dict(value=n_tiles * len(times) / total, ms_per_step=1e3 * total / len(times), cores=cores,
                sample=f"{n_tiles} tiles of {P}x{P}" + (f" + TopoNet ({NP} keypoints x 16 pairs)" if NP else "") +
                       f" per step, {len(times)} timed steps after {warmup} warm-up, fp32, "
                       f"torch.set_num_threads({cores})")


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = time_cpu_oracle(w, n_tiles=args.ref_tiles, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": w["metric"], "value": r["value"], "unit": "tiles/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"], "tiles_per_step": args.ref_tiles,
                   "points_per_tile": w["points"], "pairs_per_point": 16,
                   "note": "reference algorithm (oracle port pinned against the unmodified reference, fp32 "
                           "PyTorch eager) on host CPU cores; each step is a bounded sample of the workload"},
        "cpu_baseline": {"value": r["value"], "unit": "tiles/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "tiles/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
def _mem_line(tag, dev):
    import torch
    free, total = torch.cuda.mem_get_info(dev)
    try:
        import psutil
        rss = psutil.Process().memory_info().rss / 2**30
        avail = psutil.virtual_memory().available / 2**30
    except Exception:
        rss = avail = float("nan")
    sys.stderr.write(f"[bench mem] {tag}: rank {os.environ.get('RANK', '0')} device used "
                     f"{(total - free) / 2**30:.1f} GiB of {total / 2**30:.0f} (torch reserved "
                     f"{torch.cuda.memory_reserved(dev) / 2**30:.1f}), host rss {rss:.1f} GiB, host available "
                     f"{avail:.0f} GiB\n")
    sys.stderr.flush()


def run_scenes(args, w, wl, dev, rank, world, barrier):
    """e2e_scene: `infer_one_img` on whole synthetic scenes.  Thresholds are set from the scene's own
    fused masks (random weights give noise-like masks) so that ~0.4 % of the pixels are intersection
    candidates and ~5 % road candidates, the density of a real road mask."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from sam_road_b200 import SAMRoad, synth
    from sam_road_b200.inferencer import infer_one_img
    out = {}
    for sc in SCENES.get(wl, []):
        cfg = dict(w["cfg"], SAMPLE_MARGIN=sc["margin"], INFER_PATCHES_PER_EDGE=sc["per_edge"], **SCENE_KEYS,
                   ITSC_THRESHOLD=2.0, ROAD_THRESHOLD=2.0)
        net = SAMRoad(cfg)
        net.load_state_dict(synth.make_state_dict(cfg, seed=0, logit_gain=6.0), strict=True)
        net.eval().to(dev)
        img = np.random.RandomState(17).randint(0, 256, size=(sc["size"], sc["size"], 3)).astype(np.uint8)
        _, _, kp, road = infer_one_img(net, img, cfg, device=dev)       # probe: masks only (also the warm-up)
        cfg.update(ITSC_THRESHOLD=float(np.quantile(kp, 0.996)) / 255, ROAD_THRESHOLD=float(np.quantile(road, 0.95)) / 255)
        n_tiles = sc["per_edge"] ** 2
        res = {"scene": f"{sc['size']}x{sc['size']} uint8, {n_tiles} tiles of {cfg['PATCH_SIZE']}^2, margin {sc['margin']}, "
                        f"INFER_BATCH_SIZE {cfg['INFER_BATCH_SIZE']}", "unit": "tiles/s",
               "h2d_bytes_per_scene": int(img.nbytes)}
        for tie in ("numpy", "stable"):
            tm = {}
            infer_one_img(net, img, cfg, device=dev, nms_tie_order=tie)                  # warm-up
            infer_one_img(net, img, cfg, device=dev, nms_tie_order=tie, timings=tm)      # stage split (with syncs)
            times = []
            for _ in range(args.scene_runs):
                barrier()
                t0 = time.perf_counter()
                nodes, edges, kp, road = infer_one_img(net, img, cfg, device=dev, nms_tie_order=tie)
                barrier()
                times.append(time.perf_counter() - t0)
            sec = sorted(times)[len(times) // 2]
            if world > 1:
                t = torch.tensor([sec], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                sec = t.item()
            res[tie] = {"value": n_tiles / sec, "ms_per_scene": 1e3 * sec, "runs": len(times),
                        "n_points": int(nodes.shape[0]), "n_edges": int(edges.shape[0]),
                        "d2h_bytes_per_scene": int(kp.nbytes + road.nbytes + nodes.nbytes + edges.nbytes),
                        "stages_ms": {k: round(1e3 * v, 3) for k, v in tm.items() if k.endswith("_s")},
                        "graph_stats": {k: v for k, v in tm.get("graph_stats", {}).items()},
                        "topo_samples": tm.get("topo_samples")}
        res["value"] = res["numpy"]["value"]
        res["note"] = ("'numpy': this host's np.argsort decides the visiting order of equal scores in the greedy "
                       "NMS (bit-exact with the reference on this host); 'stable': device-only sort")
        res["scaling"] = "strong (one scene sharded over the ranks)" if world > 1 else "single GPU"
        out[sc["tag"]] = res
        del net
        torch.cuda.empty_cache()
    return out


def run_native(args, w, wl):
    import torch
    import torch.distributed as dist
    from sam_road_b200 import SAMRoad, _lib, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        from sam_road_b200.exchange import limit_nccl_ctas
        limit_nccl_ctas(world)          # only matters on the NCCL fallback of the exchange (sam_road_b200/exchange.py)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    CONFIG = w["cfg"]
    B, P, NP = args.batch, CONFIG["PATCH_SIZE"], w["points"]
    FLOP_PER_TILE = flop_per_tile(w)

    net = SAMRoad(CONFIG)
    net.load_state_dict(synth.make_state_dict(CONFIG, seed=0), strict=True)
    net.eval().to(dev)

    # R distinct resident input batches: R * B * P^2 * 3 B of uint8 tiles; the step's own activations
    # (>1 GB at 64 tiles of 512^2) exceed the 126 MB L2 many times over, so no explicit flush is needed.
    R = 3
    tiles = [synth.make_tiles(B, P, seed=100 * rank + r).to(dev) for r in range(R)]
    topo_host = [synth.make_topo_inputs(B, P, NP, seed=100 * rank + r, ragged=False) for r in range(R)] if NP else None
    topo = [[t.to(dev) for t in th] for th in topo_host] if NP else None

    # exchange step of the path (SURVEY.md §8e): per-tile mask scores and topology scores to every rank,
    # double-buffered and asynchronous -- step i's exchange runs under step i+1's compute, on the copy
    # engines over NVLink peer memory when symmetric memory is available (sam_road_b200/exchange.py).
    ex_sc = ex_ts = None
    if world > 1:
        from sam_road_b200.exchange import TileExchange
        ex_sc = TileExchange(B, (P, P, 2), torch.float32, dev, slots=2, prefer_copy_engine=not args.nccl_exchange)
        if NP:
            ex_ts = TileExchange(B, (NP, 16, 1), torch.float32, dev, slots=2, prefer_copy_engine=not args.nccl_exchange)
    _mem_line("native arm, inputs resident", dev)

    def step(i):
        r, sl = i % R, i % 2
        if world > 1:      # results are produced straight into this rank's block of the gather buffer
            ex_sc.wait(sl)
            scores, feat = net._encode(tiles[r], False, out_scores=ex_sc.local_block(sl))[::2]
            ts = None
            if NP:
                ex_ts.wait(sl)
                ts = net.infer_toponet(feat, *topo[r], out=ex_ts.local_block(sl))
            if not args.no_exchange:
                ex_sc.publish(sl)
                if NP:
                    ex_ts.publish(sl)
            return scores, feat, ts
        scores, feat = net.infer_masks_and_img_features(tiles[r])
        ts = net.infer_toponet(feat, *topo[r]) if NP else None
        return scores, feat, ts

    def drain():
        for ex in (ex_sc, ex_ts):
            if ex is not None:
                ex.drain()

    def barrier():
        drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    if args.debug_gemm_mode:
        lib.samroad_debug_disable_2cta_gemm(args.debug_gemm_mode)
    handle = net._handle(dev)
    _lib.check(lib.samroad_timing_enable(handle, 1), "timing_enable")
    lib.samroad_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        e0.record()
        for i in range(args.steps):
            results = None              # a step's results are released before the next step, as in warm-up
            results = step(args.warmup + i)
        drain()                                            # the last steps' gathers belong to the timed region
        e1.record()
        barrier()
    launches = int(lib.samroad_launch_count(0))
    ms = e0.elapsed_time(e1)
    buf = C.create_string_buffer(1 << 16)
    _lib.check(lib.samroad_timing_read(handle, buf, len(buf)), "timing_read")
    kernels = json.loads(buf.value.decode())
    _lib.check(lib.samroad_timing_enable(handle, 0), "timing_disable")
    if args.dump_outputs and rank == 0:
        scores, feat, ts = results
        dump_outputs(args.dump_outputs, dict(mask_scores=scores, image_embeddings=feat, topo_scores=ts))
    del results
    ms_ranks = [ms]
    if world > 1:
        allms = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms], device=dev))
        ms_ranks = [float(x.item()) for x in allms]
        ms = max(ms_ranks)               # the slowest rank decides
    value = world * B * args.steps / (ms / 1e3)

    # ---- e2e: the host-buffer C-ABI call, pinned host tiles in, results out, every step ----------
    h_tiles = [t.cpu().pin_memory() for t in tiles]
    h_topo = [[t.contiguous().pin_memory() for t in (th[0], th[1], th[2].view(torch.uint8))]
              for th in topo_host] if NP else None
    exchange_backend = (f"{ex_sc.backend}, barrier: {getattr(ex_sc, 'barrier_kind', 'n/a')}" +
                        (f" ({ex_sc.note})" if ex_sc.note else "")) if ex_sc is not None else None
    del tiles, topo                                      # the e2e leg owns its own (staged) device buffers
    ex_sc = ex_ts = None
    torch.cuda.empty_cache()
    h_scores = [torch.empty((B, P, P, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_emb = [torch.empty((B, 256, P // 16, P // 16), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_ts = [torch.empty((B, max(NP, 1), 16), dtype=torch.float32).pin_memory() for _ in range(2)]
    _mem_line("native arm, e2e leg", dev)

    def e2e_submit(i):
        r, sl = i % R, i % 2
        if NP:
            p, q, v = h_topo[r]
            pp, qp, vp, ts = p.data_ptr(), q.data_ptr(), v.data_ptr(), h_ts[sl].data_ptr()
        else:
            pp = qp = vp = ts = None
        _lib.check(lib.samroad_infer_batch_host_async(
            handle, sl, h_tiles[r].data_ptr(), _lib.U8, B, pp, _lib.I64, qp, _lib.I64, vp, NP, NP, 16,
            h_scores[sl].data_ptr(), h_emb[sl].data_ptr(), ts), "samroad_infer_batch_host_async")

    def e2e_run(n, first):
        # a streaming consumer: batch i is submitted, then batch i-1's results are awaited and "read"
        for i in range(n):
            e2e_submit(first + i)
            if i >= 1:
                _lib.check(lib.samroad_infer_batch_host_wait(handle, (first + i - 1) % 2), "wait")
        _lib.check(lib.samroad_infer_batch_host_wait(handle, (first + n - 1) % 2), "wait")

    e2e_run(max(2, min(3, args.warmup)), 0)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps, 0)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
    e2e_value = world * B * args.steps / e2e_s
    h2d = sum(x.numel() * x.element_size() for x in ((h_tiles[0], *h_topo[0]) if NP else (h_tiles[0],)))
    d2h = sum(x.numel() * x.element_size() for x in ((h_scores[0], h_emb[0], h_ts[0]) if NP else (h_scores[0], h_emb[0])))
    del net
    torch.cuda.empty_cache()

    # ---- e2e_scene: whole scenes through infer_one_img -----------------------------------------------
    scenes = None
    if not args.no_scene:
        scenes = run_scenes(args, w, wl, dev, rank, world, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel class ---------------------------------------------------
    ncu, ncu_src = load_ncu_metrics()
    ncu_ok = ncu is not None and args.batch == 64 and wl == ncu.get("workload", "c2")
    peaks = load_peaks()
    gemm_like = {k: v for k, v in kernels.items() if v["flops"] > 0}
    dom = max(gemm_like, key=lambda k: gemm_like[k]["ms"]) if gemm_like else None
    roofline = None
    if dom:
        d = kernels[dom]
        per_launch_ms = d["ms"] / d["launches"]
        achieved = d["flops"] / d["launches"] / (per_launch_ms * 1e-3) / 1e12
        roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peaks["tflops"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                    "traffic": (ncu["kernels"].get(dom, {}).get("dram_bytes_per_launch") if ncu_ok else None),
                    "traffic_source": ncu_src if ncu_ok else f"not reported: {ncu_src}",
                    "peak_source": peaks["source"], "launches": d["launches"],
                    "avg_launch_ms": per_launch_ms,
                    "algorithmic_flops_per_launch": d["flops"] / d["launches"]}
    total_kernel_ms = sum(v["ms"] for v in kernels.values())
    shares = {k: {"ms_per_step": v["ms"] / args.steps, "share": v["ms"] / total_kernel_ms,
                  "tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["ms"] > 0 else 0.0,
                  "gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else 0.0,
                  "launches_per_step": v["launches"] / args.steps}
              for k, v in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = time_cpu_oracle(w, n_tiles=2, steps=3, warmup=1)
        cpu = {"value": r["value"], "unit": "tiles/s", "cores": r["cores"], "kind": "port",
               "sample": r["sample"]}

    line = {
        "metric": w["metric"], "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "ms_per_step_by_rank": [round(x / args.steps, 4) for x in ms_ranks], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate",
        "data": "synthetic",
        "config": {"workload": w["name"], "workload_key": wl, "what": w["note"], "tiles_per_step_per_gpu": B,
                   "patch_size": P, "points_per_tile": NP, "pairs_per_point": 16, "input_dtype": "uint8",
                   "l2_policy": f"{R} rotating resident input batches and >1 GB of activations per step "
                                "(> 126 MB L2); no explicit flush",
                   "parallelism": f"tile-sharded dp{world}" +
                                  (" + all-gather of mask scores and topology scores, double-buffered, overlapped with "
                                   "the next step" if world > 1 else ""),
                   "exchange": "SKIPPED (--no-exchange, A/B only)" if args.no_exchange else exchange_backend},
        "e2e": {"value": e2e_value, "unit": "tiles/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / args.steps,
                "call": "samroad_infer_batch_host_async / _wait, two staging slots (pinned host uint8 tiles -> mask "
                        "scores, embeddings, topology scores on host; batch i's downloads overlap batch i+1)",
                "timer": "perf_counter"},
        "e2e_scene": scenes,
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "roofline": roofline,
        "path_tensor_frac": value / world * FLOP_PER_TILE / 1e12 / peaks["tflops"],
        "algorithmic_gflop_per_tile": FLOP_PER_TILE / 1e9,
        # BASELINE's third metric: sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active per kernel class
        # from the committed ncu --set full captures of THIS build (null when the captures are of another build)
        "tensor_pipe_pct_ncu": ({k: v.get("tensor_pipe_pct") for k, v in ncu["kernels"].items()} if ncu_ok else None),
        "tensor_pipe_pct_source": ncu_src,
        "kernels": shares,
        "cpu_baseline": cpu,
    }
    emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


class _JsonStdout:
    """Keep stdout clean for the single JSON line: libraries (NCCL prints its version banner on the
    first communicator) write to fd 1, so fd 1 is pointed at stderr for the run and the JSON line goes
    to the saved original stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.fd = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line: str):
        os.write(self.fd, (line + "\n").encode())

    def __exit__(self, *a):
        # fd 1 stays pointed at stderr for the rest of the process: NCCL (NCCL_DEBUG=INFO) still prints
        # while the communicator is torn down at interpreter exit
        sys.stdout.flush()
        os.close(self.fd)


_OUT = None


def emit(line: str):
    if _OUT is not None:
        _OUT.emit(line)
    else:
        print(line, flush=True)


def main():
    global _OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="BASELINE.json configuration (default c2 = toponet_vitb_512_cityscale)")
    ap.add_argument("--batch", type=int, default=64, help="tiles per step per GPU (INFER_BATCH_SIZE)")
    ap.add_argument("--ref-tiles", type=int, default=4,
                    help="tiles per step of the CPU reference arm (bounded sample)")
    ap.add_argument("--scene-runs", type=int, default=5, help="timed infer_one_img runs per scene and tie order")
    ap.add_argument("--no-scene", action="store_true", help="skip the e2e_scene legs")
    ap.add_argument("--no-exchange", action="store_true",
                    help="A/B only: skip the exchange step at N > 1 (attributes a slow step to the slowest GPU or to the exchange)")
    ap.add_argument("--nccl-exchange", action="store_true",
                    help="A/B: force the NCCL all-gather fallback of the exchange step (default: copy engines)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--debug-gemm-mode", type=int, default=0,
                    help="A/B only: samroad_debug_disable_2cta_gemm bit mask (16 = no snake traversal)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's mask scores, image embeddings and topology scores to "
                         "DIR/<name>.npy (float32; outputs above 4 Mi values as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")
    w = WORKLOADS[args.workload]
    with _JsonStdout() as out:
        _OUT = out
        if args.impl == "reference":
            run_reference(args, w)
        else:
            run_native(args, w, args.workload)


if __name__ == "__main__":
    main()
