#!/usr/bin/env python
"""bench.py -- headline benchmark of the two DetectorFreeSfM hot paths on B200 (DESIGN.md).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the reference's CPU path: the oracle port, bounded sample)
  python bench.py ... --dump-outputs DIR                   (also write what the last timed step of every leg returned, as .npy)

One "step" = one pass of HP-1 over the demo-scene workload C2: 8 synthetic 832x832 images, exhaustive pairing = 28 image
pairs, each pair -> (M,5) matches (BASELINE.json configs[1]).  `value` = image-pairs/s with the images resident in HBM and
the backbone run for both images of every pair (exactly the work the reference does per pair); `e2e` = the same through the
plugin call (B200LoFTR.forward on a dict) from pinned HOST images with the match arrays copied back.  `hp2` carries the second
hot path: tracks/s of one refinement chunk (C3: 2000 tracks, <= 9 query views).  With N ranks every rank processes its own
scene (weak scaling) and the per-pair match arrays are gathered to rank 0 inside the timed region.
"""
import argparse
import itertools
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tests import util  # noqa: E402  (seeded synthetic inputs shared with the tests)

HW = 832
N_IMAGES = 8
METRIC = "image-pairs/s coarse-match (hp2: tracks/s refinement)"
NOISE = 0.025
WORKLOAD = (f"C2 demo scene: {N_IMAGES} overlapping synthetic views {HW}x{HW} (crops of one low-pass noise image at 8-px-aligned offsets + "
            f"N(0,{NOISE}) per view), exhaustive 28 pairs per rank, LoFTR coarse_only, shipped thr 0.2 / temperature 0.1, BN-calibrated "
            "seeded weights (tests/weights.py) -> O(10^3) matches per pair; the step ends with the match->keypoint merge of its own matches")


def conv_gemm_flops(H, W):
    """Algorithmic FLOPs (2*MAC, true channel counts) of the backbone GEMM convolutions feeding x3_out for one HxW image
    (ResNetFPN_8_2 coarse sub-graph without the 7x7 stem, resnet_fpn.py:100-108)."""
    p2, p4, p8 = (H // 2) * (W // 2), (H // 4) * (W // 4), (H // 8) * (W // 8)
    f = 4 * p2 * 9 * 128 * 128
    f += p4 * (9 * 128 * 196 + 9 * 196 * 196 + 128 * 196 + 2 * 9 * 196 * 196)
    f += p8 * (9 * 196 * 256 + 9 * 256 * 256 + 196 * 256 + 2 * 9 * 256 * 256 + 256 * 256)
    return 2.0 * f


def pair_flops(H, W):
    L = (H // 8) * (W // 8)
    stem = 2.0 * (H // 2) * (W // 2) * 128 * 49
    backbone = 2 * (conv_gemm_flops(H, W) + stem)
    transformer = 16 * L * 1.343e6
    sim = 3 * 2.0 * L * L * 256       # two statistics passes + one confidence pass
    return backbone + transformer + sim


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_threads():
    """PyTorch-CPU threads for the reference arm: all host cores up to 32 -- measured on the 128-core B200 host the oracle runs
    3.4 s/pair at 32 threads, 3.7 s at 64 and 26 s at 128 (oversubscribed intra-op pools), so 32 is the reference's best."""
    return max(1, min(os.cpu_count() or 1, 32))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tflops": d["bf16_tflops_sustained"], "hbm": d["hbm_gbs"], "src": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    return {"tflops": 1590.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


DUMP_MAX_ELEMS = 1 << 20      # per array; the at most 16 arrays written stay under 64 MB in all


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float32 (float64 for integer arrays, exact below 2^53).  An array of more than
    DUMP_MAX_ELEMS elements is replaced by a fixed, seeded sample of its flattened elements (sorted indices), so that two builds
    given the same arguments can be compared file by file."""
    assert len(arrays) <= 16
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64)
        if a.size > DUMP_MAX_ELEMS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def profile_report(lib):
    n = lib.dfsfm_profile_report(None, 0)
    buf = ctypes.create_string_buffer(n + 16)
    lib.dfsfm_profile_report(buf, n + 16)
    out = {}
    for line in buf.value.decode().splitlines():
        label, cnt, ms = line.split()
        out[label] = (int(cnt), float(ms))
    return out


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's CPU implementation of HP-1 (the oracle port, validated bit-exact against the reference modules in
    tests/test_oracle_vs_reference.py), all host threads, on a bounded sample: one 832x832 pair per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import loftr_oracle as lo
    from oracle import postprocess_oracle as po
    from tests import weights
    torch.set_num_threads(cpu_threads())
    sd = weights.loftr_state_dict(0, calibrated=True)
    images, _ = util.synth_scene(N_IMAGES, HW, HW, 1000, noise=NOISE)
    data = {"image0": images[0], "image1": images[1], "scale0": torch.ones(1, 2), "scale1": torch.ones(1, 2)}
    ref_cfg = {"compute_unused_fine_branch": True}  # the reference evaluates the unused 1/2-res FPN branch too

    def ref_step():
        out = lo.loftr_forward(data, sd, ref_cfg)
        m = np.concatenate([out["mkpts0_f"].numpy(), out["mkpts1_f"].numpy(), out["mconf"].numpy()[:, None]], -1).astype(np.float32)
        po.merge_keypoints({"im0 im1": m}, ["im0", "im1"], " ")
        return m.shape[0]

    for _ in range(min(args.warmup, 1)):
        ref_step()
    steps = max(1, min(args.steps, 3))
    t0 = time.perf_counter()
    for _ in range(steps):
        n_matches = ref_step()
    dt = time.perf_counter() - t0
    v = steps / dt
    hp2 = None if args.skip_hp2 else hp2_cpu_baseline(256)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "sample": "bounded: 1 pair of the workload per step (+ the merge of its matches), PyTorch CPU fp32"},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{steps} x one {HW}x{HW} pair ({n_matches} matches), oracle/loftr_oracle.py + postprocess_oracle.py (PyTorch CPU fp32 / numpy)"},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
        "matches_per_pair": n_matches, "hp2": hp2,
    }))


def hp2_chunk(tracks, seed):
    return util.synth_chunk(M=tracks, n_img=10, max_views=9, hw=(600, 800), seed=seed, scales=torch.ones(1, 10, 2))


def chunk_slice(chunk, sl):
    """a contiguous slice of tracks of a chunk dict (tracks stay sorted by valid-view count)"""
    sub = dict(chunk)
    for k in ("query_points", "query_img_idxs", "query_movable_mask"):
        sub[k] = chunk[k][:, sl].contiguous()
    for k in ("reference_points_coarse", "track_valid_mask", "reference_img_idxs", "scales_relative", "view_point_vector"):
        sub[k] = chunk[k][:, :, sl].contiguous()
    return sub


def hp2_cpu_baseline(n_sub):
    """HP-2 reference CPU path (SURVEY 8d): the oracle port (validated against the reference MultiviewMatcher) + the reference's own
    RoIAlign C++ when oracle/_ref holds it, on an n_sub-track slice taken from the middle of the C3 chunk (tracks are sorted by
    view count, so the middle slice has the chunk's mean patches per track to within a few %)."""
    from oracle import multiview_oracle as mo
    from tests import weights
    torch.set_num_threads(cpu_threads())
    sd = weights.multiview_state_dict(0)
    chunk = hp2_chunk(2000, 11)
    lo_ = (2000 - n_sub) // 2
    sub = chunk_slice(chunk, slice(lo_, lo_ + n_sub))
    patches_sub = int(sub["track_valid_mask"].sum()) + n_sub
    patches_full = int(chunk["track_valid_mask"].sum()) + 2000
    t0 = time.perf_counter()
    reps = 0
    while reps < 2 and (reps == 0 or time.perf_counter() - t0 < 20):
        mo.multiview_forward(sub, sd, 15, 7)
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    kind = "C restatement of the reference RoIAlign, pinned bit-exact to oracle/_ref"
    return {"value": n_sub / dt, "unit": "tracks/s", "cores": torch.get_num_threads(), "kind": "port",
            "value_patch_scaled": (patches_sub / dt) * (2000.0 / patches_full),
            "sample": f"{reps} x a {n_sub}-track slice ({patches_sub} patches; full chunk {patches_full}) of the C3 chunk, oracle/multiview_oracle.py "
                      f"(PyTorch CPU fp32; {kind}); value_patch_scaled = tracks/s of the full chunk at the same patches/s"}



# ------------------------------------------------------------------------------ BASELINE configs[3] / configs[4]: sharded scenes
def _timed_region(fn, steps, dev, D):
    D.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    D.barrier()
    return D.max_over_ranks(e0.elapsed_time(e1), dev), out


def run_c4(args):
    """C4: one scene of --c4-images overlapping 832x832 views, EXHAUSTIVE pairs (101 -> 5050), strong scaling: the pair list is dealt
    to the ranks by image locality (dist.shard_pairs_by_image), every rank matches its pairs with the per-image feature cache, the
    match -> keypoint merge runs sharded by image owner (postprocess_dist.merge_keypoints_sharded: one all_to_all of [x,y,conf] rows and
    one of the ids over NCCL), and only rank 0 receives the per-pair keypoint-id arrays (gather_varlen_to)."""
    from detectorfreesfm_b200 import B200LoFTR
    from detectorfreesfm_b200 import dist as D
    from detectorfreesfm_b200.postprocess_dist import merge_keypoints_sharded
    from tests import weights
    rank, world, local = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n_img = args.c4_images
    names = [f"scene/img_{i:04d}.jpg" for i in range(n_img)]
    pairs = list(itertools.combinations(range(n_img), 2))
    mine = D.shard_pairs_by_image(pairs, rank, world)
    images = util.synth_scene(n_img, HW, HW, 77, noise=NOISE, max_shift=256)[0]          # same scene on every rank (seeded)
    touched = sorted({i for k in mine for i in pairs[k]})
    dev_images = {i: images[i].to(dev) for i in touched}
    matcher = B200LoFTR(util.loftr_config(thr=0.2, temperature=0.1), feature_cache_size=n_img + 1).cuda(local).eval()
    matcher.load_state_dict(weights.loftr_state_dict(0, calibrated=True))
    ones = torch.ones(1, 2, device=dev)
    stats = {}

    def step():
        matcher.clear_cache()
        local_matches = {}
        for k in mine:
            i, j = pairs[k]
            data = {"image0": dev_images[i], "image1": dev_images[j], "scale0": ones, "scale1": ones, "pair_key": ((names[i],), (names[j],))}
            matcher(data)
            local_matches[f"{names[i]} {names[j]}"] = torch.cat([data["mkpts0_f"], data["mkpts1_f"], data["mconf"][:, None]], -1)
        fk, fs, upd = merge_keypoints_sharded(local_matches, mine, names, " ", device=dev)
        ids = [torch.from_numpy(upd[k].astype(np.float32)).to(dev) for k in local_matches]
        got = D.gather_varlen_to(ids, dst=0)
        stats["matches"] = int(sum(v.shape[0] for v in local_matches.values()))
        stats["keypoints"] = int(sum(v.shape[0] for v in fk.values()))
        stats["gathered_pairs"] = None if got is None else sum(len(g) for g in got)
        return got

    W, K = max(1, min(args.warmup, 1)), max(1, min(args.steps, 2))
    for _ in range(W):
        step()
    ms, _ = _timed_region(step, K, dev, D)
    total_matches = int(D.sum_over_ranks(stats["matches"], dev))
    pairs_max = int(D.max_over_ranks(len(mine), dev))
    if rank == 0:
        print(json.dumps({
            "metric": "image-pairs/s coarse-match, C4 full pair graph", "value": len(pairs) * K / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16x2-split (fp32-grade), fp32 accumulate", "data": "synthetic",
            "config": {"workload": f"C4: {n_img} overlapping synthetic {HW}x{HW} views, exhaustive {len(pairs)} pairs sharded by image locality over "
                                   f"{world} rank(s), per-image feature cache, sharded keypoint merge over NCCL, ids gathered to rank 0",
                       "pairs_on_slowest_rank": pairs_max, "matches_total": total_matches, "keypoints": stats["keypoints"],
                       "gathered_pairs_on_rank0": stats["gathered_pairs"]}}))
    if world > 1:
        torch.distributed.destroy_process_group()


def run_c5(args):
    """C5: --c5-chunks refinement chunks of 2000 tracks (500 -> 1e6 tracks) dealt round-robin to the ranks (chunks never interact;
    dist.shard), every chunk dict travelling host -> device and its refined points back, [K,4]-sized results gathered to rank 0."""
    from detectorfreesfm_b200 import B200MultiviewMatcher
    from detectorfreesfm_b200 import dist as D
    from tests import weights
    rank, world, local = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    rm = B200MultiviewMatcher(util.multiview_config(15, 7), test=True).cuda(local).eval()
    rm.load_state_dict(weights.multiview_state_dict(0))
    mine = D.shard(args.c5_chunks, rank, world)
    pool = [hp2_chunk(2000, 100 + s) for s in range(4)]                                 # 4 distinct synthetic chunks, reused cyclically
    pool = [{k: ([im.pin_memory() for im in v] if isinstance(v, list) else (v.pin_memory() if torch.is_tensor(v) else v)) for k, v in c.items()}
            for c in pool]

    def step():
        res = []
        for c in mine:
            h = pool[c % len(pool)]
            d = {k: ([im.to(dev, non_blocking=True) for im in v] if isinstance(v, list) else (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v))
                 for k, v in h.items()}
            rm(d)
            mask = d["track_valid_mask"][0]
            res.append(torch.cat([d["query_points_refined"][0], d["reference_points_refined"][-1][0][mask]], 0))   # the [K,2] part of matchWorker's rows
        return D.gather_varlen_to(res, dst=0)

    step_small = mine[:2]
    for _ in range(1):                                                                   # warm-up on two chunks
        saved, mine[:] = list(mine), step_small
        step()
        mine[:] = saved
    ms, _ = _timed_region(step, 1, dev, D)
    tracks = args.c5_chunks * 2000
    if rank == 0:
        print(json.dumps({
            "metric": "tracks/s refinement, C5 chunks sharded", "value": tracks / (ms * 1e-3), "unit": "tracks/s", "n_gpus": world, "steps": 1,
            "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16x2-split (fp32-grade), fp32 accumulate", "data": "synthetic",
            "config": {"workload": f"C5: {args.c5_chunks} chunks x 2000 tracks ({tracks} tracks, <= 9 query views, 10 images of 600x800 per chunk) "
                                   f"round-robin over {world} rank(s), host chunk dict -> device per chunk, refined points gathered to rank 0"}}))
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workers-per-gpu", type=int, default=int(os.environ.get("DFSFM_BENCH_WORKERS", "1")),
                    help="concurrent pair workers per GPU, each with its own matcher (engine handle + workspaces) and CUDA stream -- the reference's "
                         "built-in config shares a GPU between Ray workers the same way (n_gpus_per_worker: 0.5, src/coarse_match/coarse_match.py:53). "
                         "Default 1: three workers measured +27 %% pairs/s (profiles/r02_worker_pool.txt) but a bench invocation with three "
                         "workers at 832x832 hung intermittently on the GPU (profiles/r02_pool_hang.txt, unresolved), so the pool is opt-in")
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 (default): the headline line, one demo scene per rank; c4: IMC-style full pair graph (5050 pairs of 101 images) sharded "
                         "over the ranks, strong scaling; c5: Bridge-scale refinement, --c5-chunks chunks of 2000 tracks sharded over the ranks")
    ap.add_argument("--c4-images", type=int, default=101)
    ap.add_argument("--c5-chunks", type=int, default=500)
    ap.add_argument("--hp2-tracks", type=int, default=2000)
    ap.add_argument("--skip-hp2", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-post", action="store_true")
    ap.add_argument("--skip-img", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each leg returned as DIR/<name>.npy (float32 / float64; "
                         "arrays over 2^20 elements as a fixed seeded sample): hp1_* the per-pair matches and their keypoint merge, hp2_* "
                         "the refined chunk, post_* the keypoint merge, image_* the resized images; rank 0 only.  bench_outputs/ in "
                         "the repository is git-ignored for this")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "c2"):
        ap.error("--dump-outputs writes the outputs of the default workload (--impl b200 --config c2)")
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "c4":
        return run_c4(args)
    if args.config == "c5":
        return run_c5(args)

    from detectorfreesfm_b200 import B200LoFTR, B200MultiviewMatcher, KeypointMerger, _lib
    from detectorfreesfm_b200 import dist as D
    from tests import weights
    rank, world, local = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load_library()
    W = max(args.warmup, 3)
    K = args.steps
    outputs = {}      # --dump-outputs: name -> host array of the last timed step

    # ------------------------------------------------------------------ HP-1 workload: one scene per rank
    matcher = B200LoFTR(util.loftr_config(thr=0.2, temperature=0.1), feature_cache_size=2 * N_IMAGES).cuda(local).eval()
    matcher.load_state_dict(weights.loftr_state_dict(0, calibrated=True))
    host_images = [im.pin_memory() for im in util.synth_scene(N_IMAGES, HW, HW, 1000 * (rank + 1), noise=NOISE)[0]]
    dev_images = [im.to(dev) for im in host_images]
    pairs = [(i, j) for i in range(N_IMAGES) for j in range(i + 1, N_IMAGES)]
    ones = torch.ones(1, 2, device=dev)
    merger = KeypointMerger(dev)
    pair_img = torch.tensor(pairs, dtype=torch.int32, device=dev)
    m_stats = {}

    def merge_step(out):
        """the match -> keypoint -> index merge (coarse_match.py:203-237) of THIS step's matches, still on the device"""
        counts = torch.tensor([0] + [int(o.shape[0]) for o in out], dtype=torch.int64)
        m_stats["counts"] = counts[1:].tolist()
        return merger.merge(torch.cat(out, 0), torch.cumsum(counts, 0), pair_img, N_IMAGES)

    # optional: several pair workers per GPU (threads; the C ABI calls and the per-pair count read-back release the GIL).  One pair at a time
    # offers only 43 / 86 CTA-pair tiles per encoder launch to 74 CTA pairs; two independent pairs in flight fill the gaps.
    n_workers = max(1, args.workers_per_gpu)
    workers = [(matcher, torch.cuda.current_stream(dev))]
    for _ in range(1, n_workers):
        mw = B200LoFTR(util.loftr_config(thr=0.2, temperature=0.1), feature_cache_size=2 * N_IMAGES).cuda(local).eval()
        mw.load_state_dict(weights.loftr_state_dict(0, calibrated=True))
        workers.append((mw, torch.cuda.Stream(device=dev)))
    from detectorfreesfm_b200.coarse_stage import pool_thread_begin, pool_thread_end   # what coarse_stage.match_workers does per thread

    def run_pairs(widx, todo, cached, out):
        mw, stream = workers[widx]
        torch.cuda.set_device(local)
        pool_thread_begin(n_workers)
        with torch.cuda.stream(stream):
            for k in todo:
                i, j = pairs[k]
                data = {"image0": dev_images[i], "image1": dev_images[j], "scale0": ones, "scale1": ones}
                if cached:
                    data["pair_key"] = ((f"im{i}",), (f"im{j}",))
                mw(data)
                out[k] = torch.cat([data["mkpts0_f"], data["mkpts1_f"], data["mconf"][:, None]], -1)
        pool_thread_end()

    def step_resident(cached):
        """inputs resident in HBM; returns the per-pair (M,5) device arrays"""
        nonlocal n_workers
        out = [None] * len(pairs)
        for mw, _ in workers:
            mw.clear_cache()
        if n_workers == 1:
            run_pairs(0, range(len(pairs)), cached, out)
        else:
            main = torch.cuda.current_stream(dev)
            start = torch.cuda.Event()
            start.record(main)
            ths = []
            for w in range(1, n_workers):
                workers[w][1].wait_event(start)
                ths.append(threading.Thread(target=run_pairs, args=(w, range(w, len(pairs), n_workers), cached, out)))
                ths[-1].start()
            run_pairs(0, range(0, len(pairs), n_workers), cached, out)
            for t in ths:
                t.join()
            for w in range(1, n_workers):
                done = torch.cuda.Event()
                done.record(workers[w][1])
                main.wait_event(done)
        m_stats["merged"] = merge_step(out)
        return out

    h2d = d2h = 0

    def run_pairs_e2e(widx, todo, cached, res, dev_out, counts):
        """one pair worker of the end-to-end leg: the plugin call from HOST buffers -- pinned images -> device, matcher(data), the
        (M,5) match array back to the host -- on the worker's own stream"""
        mw, stream = workers[widx]
        torch.cuda.set_device(local)
        pool_thread_begin(n_workers)
        up = down = 0
        with torch.cuda.stream(stream):
            for k in todo:
                i, j = pairs[k]
                a, b = host_images[i].to(dev, non_blocking=True), host_images[j].to(dev, non_blocking=True)
                up += a.numel() * 4 + b.numel() * 4
                data = {"image0": a, "image1": b, "scale0": ones, "scale1": ones}
                if cached:
                    data["pair_key"] = ((f"im{i}",), (f"im{j}",))
                mw(data)
                md = torch.cat([data["mkpts0_f"], data["mkpts1_f"], data["mconf"][:, None]], -1)
                dev_out[k] = md
                m = md.cpu().numpy()
                down += m.nbytes + 4  # + the match-count readback that sizes the arrays
                res[k] = m
        pool_thread_end()
        counts[widx] = (up, down)

    def step_e2e(cached):
        """the plugin call from HOST buffers for every pair (+ the merge of the step's matches, results to the host)"""
        nonlocal h2d, d2h
        for mw, _ in workers:
            mw.clear_cache()
        res, dev_out, counts = [None] * len(pairs), [None] * len(pairs), [None] * n_workers
        ths = [threading.Thread(target=run_pairs_e2e, args=(w, range(w, len(pairs), n_workers), cached, res, dev_out, counts))
               for w in range(1, n_workers)]
        for t in ths:
            t.start()
        run_pairs_e2e(0, range(0, len(pairs), n_workers), cached, res, dev_out, counts)
        for t in ths:
            t.join()                                  # every worker has read its last match array back: its stream is drained
        h2d = sum(c[0] for c in counts)
        d2h = sum(c[1] for c in counts)
        kp = [t.cpu() for t in merge_step(dev_out)]   # keypoints, scores, per-image offsets, per-match keypoint ids -> host
        d2h += sum(t.numel() * t.element_size() for t in kp)
        return res

    def timed(fn, steps, gather):
        """-> (max over ranks of the ms the steps took, what the last step returned)"""
        D.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
            if gather and world > 1:
                D.gather_varlen_to([o if torch.is_tensor(o) else torch.from_numpy(o).to(dev) for o in out], dst=0)   # only rank 0 receives
        e1.record()
        torch.cuda.synchronize()
        D.barrier()
        return D.max_over_ranks(e0.elapsed_time(e1), dev), out

    for _ in range(W):
        warm = step_resident(False)
        if world > 1:   # the first point-to-point op creates its NCCL communicator: keep that out of the timed region
            D.gather_varlen_to(warm, dst=0)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = lib.dfsfm_launch_count()
    ms_cold, last = timed(lambda: step_resident(False), K, True)
    launches = lib.dfsfm_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        kp, score, img_off, ids = m_stats["merged"]
        outputs.update(hp1_matches=torch.cat(last, 0), hp1_match_counts=torch.tensor([o.shape[0] for o in last]), hp1_keypoints=kp,
                       hp1_keypoint_scores=score, hp1_image_keypoint_offsets=img_off, hp1_match_keypoint_ids=ids)
        outputs = {k: v.cpu() for k, v in outputs.items()}
    ms_cold_1w = None
    if n_workers > 1:     # the same step with ONE pair in flight (per-pair latency view; explains what the pair workers buy)
        saved_w, n_workers = n_workers, 1
        step_resident(False)
        ms_cold_1w, _ = timed(lambda: step_resident(False), K, False)
        n_workers = saved_w
    step_resident(True)   # every variant gets its own untimed warm-up step (allocator growth, feature-cache storage)
    ms_cached, _ = timed(lambda: step_resident(True), K, True)
    step_e2e(False)
    ms_e2e, _ = timed(lambda: step_e2e(False), K, True)
    step_e2e(True)
    ms_e2e_cached, _ = timed(lambda: step_e2e(True), K, True)
    n_pairs = len(pairs) * world

    # ------------------------------------------------------------------ roofline attribution of the dominant kernel
    lib.dfsfm_profile_enable(1)
    saved_workers, n_workers = n_workers, 1       # per-kernel attribution: one pair at a time (concurrent pairs overlap their kernels)
    step_resident(False)
    n_workers = saved_workers
    prof = profile_report(lib)
    lib.dfsfm_profile_enable(0)
    peaks = measured_peaks()
    conv_cnt, conv_ms = prof.get("conv", (0, 0.0))
    conv_alg = conv_gemm_flops(HW, HW) * 2 * len(pairs)
    achieved = conv_alg / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else None
    total_ms = sum(v[1] for v in prof.values())
    roofline = {"bound": "tensor", "kernel": "gemm_tc2_kernel<BN,split,ConvEpi> (backbone implicit-GEMM convolutions, persistent CTA pairs)",
                "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": (achieved / peaks["tflops"]) if achieved else None,
                "traffic": 238.0e6 / 1e9 if conv_ms else None, "traffic_unit": "GB per launch of the largest conv (layer1 3x3 with residual; ncu dram read+write, profiles/r01_ncu_conv_summary.txt; algorithmic 0.267 GB)",
                "peak_source": peaks["src"], "passes": 3,
                "executed": (3 * achieved) if achieved else None, "executed_frac": (3 * achieved / peaks["tflops"]) if achieved else None,
                "note": "achieved = algorithmic FLOPs (true channel counts, 1 pass); the kernel executes 3 fp16 MMA passes per K-step "
                        "(split-fp16 operands for fp32-grade parity): `executed` = 3 x achieved is the fp16 tensor-pipe rate (padding and halo rows not counted)",
                "launches": conv_cnt, "avg_launch_ms": conv_ms / conv_cnt if conv_cnt else None, "share_of_step": conv_ms / total_ms if total_ms else None,
                "kernel_ms_per_step": {k: round(v[1], 3) for k, v in sorted(prof.items())}}

    # the kernel north_star sets the 70 % target for: the LoFTR encoder layer (SURVEY 8d: 1.343 MFLOP per token per layer call)
    enc_keys = ("lin", "kv", "kv_final", "attn", "fold", "kvproj", "enc_fused")
    enc_ms = sum(prof[k][1] for k in enc_keys if k in prof)
    L_tok = (HW // 8) ** 2
    enc_alg = 16 * L_tok * 1.343e6 * len(pairs)
    enc_tiles = 4 * (2 * ((L_tok + 255) // 256)) + 8 * ((L_tok + 255) // 256)        # 256-token CTA-pair tiles per pair: 4 self + 8 cross calls
    enc_rounds = 4 * -(-(2 * ((L_tok + 255) // 256)) // 74) + 8 * -(-((L_tok + 255) // 256) // 74)
    roofline_encoder = {
        "bound": "tensor", "kernel": "LoFTR encoder layer: KvEpi k/v projection + state reduction, kvp_fold, enc256_fused_kernel (or the GEMM-per-linear schedule)",
        "achieved": enc_alg / (enc_ms * 1e-3) / 1e12 if enc_ms else None, "peak": peaks["tflops"], "unit": "TFLOP/s",
        "frac": enc_alg / (enc_ms * 1e-3) / 1e12 / peaks["tflops"] if enc_ms else None, "passes": 3,
        "executed_frac": 3 * enc_alg / (enc_ms * 1e-3) / 1e12 / peaks["tflops"] if enc_ms else None,
        "ms_per_step": enc_ms, "kernels": {k: round(prof[k][1], 3) for k in enc_keys if k in prof},
        "tile_occupancy": enc_tiles / (enc_rounds * 74.0),
        "note": "algorithmic = 1.343 MFLOP/token/layer-call x 16 calls x 10816 tokens per pair; 3 fp16 passes executed (split-fp16); one pair at a "
                "time gives 43 (cross) / 86 (self) 256-token tiles per launch for 74 CTA pairs: tile_occupancy is the resulting upper bound on SM use"}
    roofline["encoder_layer"] = roofline_encoder

    # ------------------------------------------------------------------ HP-2: one refinement chunk (C3)
    hp2 = None
    if not args.skip_hp2:
        multiview_config, to_cuda = util.multiview_config, util.to_cuda
        rm = B200MultiviewMatcher(multiview_config(15, 7), test=True).cuda(local).eval()
        rm.load_state_dict(weights.multiview_state_dict(0))
        chunk = hp2_chunk(args.hp2_tracks, 11 + rank)
        n_patches = int(chunk["track_valid_mask"].sum()) + args.hp2_tracks
        cd = to_cuda(chunk)
        # the chunk as MatchingMultiviewData + DataLoader hand it over: every tensor on the HOST (pinned)
        host_chunk = {k: ([im.pin_memory() for im in v] if isinstance(v, list) else (v.pin_memory() if torch.is_tensor(v) else v))
                      for k, v in chunk.items()}
        h2d_2 = sum(t.numel() * t.element_size() for v in host_chunk.values() for t in (v if isinstance(v, list) else [v]) if torch.is_tensor(t))

        def chunk_resident():
            d = dict(cd)
            rm(d)
            return d

        d2h_2 = 0

        def chunk_e2e():
            """what matchWorker does per chunk (multiview_match_worker.py:111-150): the whole host dict -> device, matcher, results -> host"""
            nonlocal d2h_2
            d = {k: ([im.to(dev, non_blocking=True) for im in v] if isinstance(v, list) else (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v))
                 for k, v in host_chunk.items()}
            rm(d)
            outs = (d["query_points_refined"].cpu(), d["reference_points_refined"][-1].cpu(), d["std"][-1].cpu())
            d2h_2 = sum(t.numel() * t.element_size() for t in outs)
            return outs

        for _ in range(2):
            chunk_resident()
        ms2, last = timed(chunk_resident, K, False)
        if args.dump_outputs:
            outputs.update(hp2_query_points_refined=last["query_points_refined"].cpu(),
                           hp2_reference_points_refined=last["reference_points_refined"][-1].cpu(), hp2_std=last["std"][-1].cpu())
        ms2_e2e, _ = timed(chunk_e2e, K, False)
        lib.dfsfm_profile_enable(1)
        chunk_resident()
        prof2 = profile_report(lib)
        lib.dfsfm_profile_enable(0)
        pc_cnt, pc_ms = prof2.get("pconv", (0, 0.0))
        # algorithmic FLOPs per patch of the GEMM convolutions as the reference executes them (SURVEY 8d: 1.024 GFLOP/patch
        # incl. the 4.2 MFLOP conv1_1 which is a SIMT kernel here)
        pconv_alg = n_patches * (1.024e9 - 2 * 35 * 35 * 27 * 64)
        hp2 = {"metric": "tracks/s refinement", "value": args.hp2_tracks * K * world / (ms2 * 1e-3), "unit": "tracks/s",
               "ms_per_chunk": ms2 / K, "tracks_per_chunk": args.hp2_tracks, "patches_per_chunk": n_patches,
               "e2e": {"value": args.hp2_tracks * K * world / (ms2_e2e * 1e-3), "unit": "tracks/s",
                       "h2d_bytes_per_step": h2d_2, "d2h_bytes_per_step": d2h_2,
                       "note": "host chunk dict (pinned) -> device, matcher call, refined points + std -> host; inside the call the shim reads the "
                               "small per-track arrays back ONCE as one packed buffer (the C ABI builds its patch records on the host; ~0.5 MB, "
                               "not in these counts) and leaves the results on the device"},
               "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel<BN,split,ConvEpi> (S2DNet patch convolutions, persistent CTA pairs)",
                            "achieved": pconv_alg / (pc_ms * 1e-3) / 1e12 if pc_ms else None, "peak": peaks["tflops"], "unit": "TFLOP/s",
                            "frac": pconv_alg / (pc_ms * 1e-3) / 1e12 / peaks["tflops"] if pc_ms else None,
                            "note": "algorithmic = FLOPs the reference executes (1.02 GFLOP/patch); the engine skips the part of the 5x5 "
                                    "adapter outside the centre window and runs 3 fp16 passes",
                            "kernel_ms_per_chunk": {k: round(v[1], 3) for k, v in sorted(prof2.items())}}}
        if rank == 0 and world == 1 and not args.skip_cpu:
            hp2["cpu_baseline"] = hp2_cpu_baseline(256)

    # ------------------------------------------------------------------ match -> keypoint -> index post-processing (SURVEY 8(f) row 1)
    post = None
    if not args.skip_post:
        try:
            n_img, m_pair = 64, 2000
            pairs = list(itertools.combinations(range(n_img), 2))
            pm, names = util.synth_matches(n_img, pairs, m_pair, seed=5 + rank, dup=0.25)
            rows_host = torch.from_numpy(np.concatenate(list(pm.values()), 0)).pin_memory()
            rows_dev = rows_host.to(dev)
            counts = np.array([v.shape[0] for v in pm.values()], dtype=np.int64)
            pair_off = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)).to(dev)
            index = {n: i for i, n in enumerate(names)}
            pair_img = torch.tensor([[index[k.split(" ")[0]], index[k.split(" ")[1]]] for k in pm], dtype=torch.int32, device=dev)
            n_obs = 2 * int(rows_dev.shape[0])

            def post_resident():
                return merger.merge(rows_dev, pair_off, pair_img, n_img)

            def post_e2e():
                out = merger.merge(rows_host.to(dev, non_blocking=True), pair_off, pair_img, n_img)
                return [o.cpu() for o in out]

            for _ in range(2):
                post_resident()
            ms3, last = timed(post_resident, K, False)
            if args.dump_outputs:
                outputs.update({"post_" + n: t.cpu() for n, t in zip(("keypoints", "keypoint_scores", "image_keypoint_offsets",
                                                                       "match_keypoint_ids"), last)})
            ms3_e2e, _ = timed(post_e2e, K, False)
            lib.dfsfm_profile_enable(1)
            kp = post_resident()
            prof3 = profile_report(lib)
            lib.dfsfm_profile_enable(0)
            sc_cnt, sc_ms = prof3.get("post_scatter", (0, 0.0))
            rec_bytes = 24.0 * n_obs   # one pass streams every 12-byte (key, value) record in and out once
            post = {"metric": "match end points/s merged into key points", "value": n_obs * K * world / (ms3 * 1e-3), "unit": "observations/s",
                    "ms_per_call": ms3 / K, "observations": n_obs, "pairs": len(pairs), "images": n_img, "keypoints": int(kp[0].shape[0]),
                    "e2e": {"value": n_obs * K * world / (ms3_e2e * 1e-3), "unit": "observations/s", "h2d_bytes_per_step": rows_host.numel() * 4,
                            "d2h_bytes_per_step": int(kp[0].numel() * 4 + kp[1].numel() * 4 + kp[3].numel() * 4)},
                    "roofline": {"bound": "hbm", "kernel": "rs_scatter_kernel (one 8-bit LSD radix pass over the observation records)",
                                 "achieved": rec_bytes / (sc_ms / sc_cnt * 1e-3) / 1e9 if sc_cnt else None, "peak": peaks.get("hbm"), "unit": "GB/s",
                                 "frac": (rec_bytes / (sc_ms / sc_cnt * 1e-3) / 1e9 / peaks["hbm"]) if sc_cnt and peaks.get("hbm") else None,
                                 "traffic": 0.3396, "traffic_unit": "GB per launch of the first pass over the 8.06 M observation records (ncu dram read+write, "
                                                                    "profiles/r02_ncu_post_summary.txt; algorithmic 0.1935 GB: the per-digit offsets / histograms and "
                                                                    "write-allocate reads account for the rest)", "launches": sc_cnt,
                                 "kernel_ms_per_call": {k: round(v[1], 3) for k, v in sorted(prof3.items())}}}
            if rank == 0 and world == 1 and not args.skip_cpu:
                from oracle import postprocess_oracle as po
                sub_pairs = list(itertools.combinations(range(12), 2))
                sub, sub_names = util.synth_matches(12, sub_pairs, m_pair, seed=5, dup=0.25)
                t0 = time.perf_counter()
                reps = 0
                while reps < 3 and time.perf_counter() - t0 < 15:
                    po.merge_keypoints(sub, sub_names, " ")
                    reps += 1
                dt = time.perf_counter() - t0
                post["cpu_baseline"] = {"value": 2 * len(sub_pairs) * m_pair * reps / dt, "unit": "observations/s", "cores": 1, "kind": "port",
                                        "sample": f"{reps} x 12 images / {len(sub_pairs)} pairs x {m_pair} matches, oracle/postprocess_oracle.py "
                                                  "(numpy np.unique/bincount/argsort restatement, pinned to the reference functions; the "
                                                  "reference itself adds per-match Python dict look-ups)"}
        except Exception as e:  # the secondary leg must never take the headline line down with it
            post = {"error": repr(e)}

    # ------------------------------------------------------------------ host image pipeline: PIL-LANCZOS resize + /255 (SURVEY 8(f) row 3)
    img_leg = None
    if not args.skip_img:
        try:
            from detectorfreesfm_b200.image_pipeline import GpuImageReader, process_resize
            rd = GpuImageReader(dev)
            src_hw = (3000, 4000)                       # a 12 MP photo, demo config: longest side -> 1200, df = 8
            photo = util.synth_photo(src_hw[0], src_hw[1], seed=3 + rank)
            size = process_resize(src_hw[1], src_hw[0], (1200,), 8)
            photo_dev = torch.from_numpy(photo).to(dev)
            n_img = 8

            def img_resident():
                return [rd.resize_gray(photo_dev, size) for _ in range(n_img)]

            def img_e2e():
                return [rd.resize_gray(photo, size) for _ in range(n_img)]      # pinned staging + H2D inside

            for _ in range(2):
                img_resident()
            ms4, last = timed(img_resident, K, False)
            if args.dump_outputs:
                outputs["image_resized"] = torch.stack(last, 0).cpu()
            ms4_e2e, _ = timed(img_e2e, K, False)
            lib.dfsfm_profile_enable(1)
            img_resident()
            prof4 = profile_report(lib)
            lib.dfsfm_profile_enable(0)
            h_cnt, h_ms = prof4.get("resize_h", (0, 0.0))
            alg_bytes = float(src_hw[0] * src_hw[1] + src_hw[0] * size[0])      # horizontal pass: bytes in + intermediate bytes out
            img_leg = {"metric": "images/s resized (12 MP gray -> longest side 1200, PIL-LANCZOS parity) + /255", "value": n_img * K * world / (ms4 * 1e-3),
                       "unit": "images/s", "ms_per_image": ms4 / (K * n_img), "src_hw": list(src_hw), "out_wh": list(size),
                       "e2e": {"value": n_img * K * world / (ms4_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": n_img * photo.size,
                               "d2h_bytes_per_step": 0},
                       "roofline": {"bound": "hbm", "kernel": "lanczos_h_kernel (horizontal pass over the full-resolution image)",
                                    "achieved": alg_bytes / (h_ms / h_cnt * 1e-3) / 1e9 if h_cnt else None, "peak": peaks["hbm"], "unit": "GB/s",
                                    "frac": alg_bytes / (h_ms / h_cnt * 1e-3) / 1e9 / peaks["hbm"] if h_cnt else None,
                                    "traffic": 0.01212, "traffic_unit": "GB per launch (ncu dram read; the 3.6 MB intermediate stays in L2; profiles/r02_ncu_post_summary.txt)",
                                    "kernel_ms_per_step": {k: round(v[1], 3) for k, v in sorted(prof4.items())}}}
            if rank == 0 and world == 1 and not args.skip_cpu:
                from PIL import Image
                t0 = time.perf_counter()
                reps = 0
                while reps < 8 and time.perf_counter() - t0 < 10:
                    np.asarray(Image.fromarray(photo).resize(size, resample=Image.LANCZOS), dtype=np.uint8).astype("float32") / 255.
                    reps += 1
                img_leg["cpu_baseline"] = {"value": reps / (time.perf_counter() - t0), "unit": "images/s", "cores": 1, "kind": "reference",
                                           "sample": f"{reps} x PIL.Image.resize(LANCZOS) + /255 of the same photo (the reference's own call, Pillow)"}
        except Exception as e:
            img_leg = {"error": repr(e)}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        from oracle import loftr_oracle as lo
        torch.set_num_threads(cpu_threads())
        sd = weights.loftr_state_dict(0, calibrated=True)
        data = {"image0": host_images[0], "image1": host_images[1], "scale0": torch.ones(1, 2), "scale1": torch.ones(1, 2)}
        t0 = time.perf_counter()
        n_cpu = 0
        while n_cpu < 2 and time.perf_counter() - t0 < 25:
            lo.loftr_forward(data, sd, {"compute_unused_fine_branch": True})
            n_cpu += 1
        dt = time.perf_counter() - t0
        cpu = {"value": n_cpu / dt, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{n_cpu} x one {HW}x{HW} pair of the workload, oracle/loftr_oracle.py (PyTorch CPU fp32, validated bit-exact vs the reference; incl. the unused FPN branch the reference also runs)"}

    total_launches = int(D.sum_over_ranks(launches, dev))
    if rank == 0:
        value = n_pairs * K / (ms_cold * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_cold / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16x2-split (fp32-grade), fp32 accumulate",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "l2": "per-step working set (activations of one 832x832 image ~0.4 GB) exceeds the 126 MB L2; no explicit flush",
                       "backbone": "run for both images of every pair in `value`/`e2e` (as the reference does); *_cached keys use the exact per-image feature cache",
                       "parallelism": f"pairs sharded over {world} rank(s), one scene per rank, final gather of (M,5) arrays",
                       "pair_workers_per_gpu": n_workers},
            "value_cached": n_pairs * K / (ms_cached * 1e-3),
            "value_one_pair_in_flight": (n_pairs * K / (ms_cold_1w * 1e-3)) if ms_cold_1w else None,
            "e2e": {"value": n_pairs * K / (ms_e2e * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "value_cached": n_pairs * K / (ms_e2e_cached * 1e-3)},
            "matches_per_pair": {"mean": float(np.mean(m_stats["counts"])), "min": int(min(m_stats["counts"])), "max": int(max(m_stats["counts"])),
                                 "keypoints_merged": int(m_stats["merged"][0].shape[0])},
            "gpu_launches": total_launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "algorithmic_gflop_per_pair": pair_flops(HW, HW) / 1e9, "hp2": hp2, "post": post, "image_pipeline": img_leg,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
