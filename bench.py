#!/usr/bin/env python
"""bench.py -- image-pairs matched(+verified)/s on N B200s (BASELINE.json metric).

    python bench.py --gpus 1 --steps 2 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference          # the reference's CPU algorithm on the host cores
    python bench.py --steps 2 --warmup 1 --dump-outputs out/   # + what the last timed step computed, as .npy

A "step" is one pass of the hot path (exhaustive matching [+ two-view verification]) over every
image pair of the synthetic scene.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


# BASELINE.json configs[1..4] (SURVEY.md section 8(d)); the scene and the pair list are the same for every GPU
# count (strong scaling): ranks own contiguous image ranges for the upload + all-gather and every k-th pair.
CONFIGS = {
    "c2": dict(images=1000, feats=8192, verify=0, pairs="exhaustive", guided=0, baseline_index=1),
    "c3": dict(images=1000, feats=8192, verify=1, pairs="exhaustive", guided=0, baseline_index=2),
    "c4": dict(images=5000, feats=4096, verify=1, pairs="exhaustive", guided=0, baseline_index=3),
    "c5": dict(images=10000, feats=4096, verify=1, pairs="sequential", guided=1, baseline_index=4),
}


def log(msg):
    """Progress on stderr (stdout carries exactly one JSON line)."""
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS),
                    help="BASELINE.json configs[1..4]: c2 match only, c3 (default) + verification, c4 5000 x 4096, "
                         "c5 10000 images sequential (overlap 20) + guided matching")
    ap.add_argument("--images", type=int, default=0, help="override the config's image count (fixed for every --gpus: strong scaling)")
    ap.add_argument("--feats", type=int, default=0, help="override the config's descriptors per image")
    ap.add_argument("--verify", type=int, default=-1, help="override: 1 match + two-view verification, 0 match only")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--pair-batch", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's pairs, a seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline(desc_np, n_feat, pairs, budget_s, verify, kpts_np=None, cam=None, full_frac=None):
    """The reference's CPU algorithm (oracle port) on a bounded sample of the same workload, all host threads, one pair
    per thread at a time (like upstream's FeatureMatcherWorker / VerifierWorker pools).  Matching: the AVX-512-VNNI
    brute-force matcher (oracle/oracle_match.c).  Verification (when `verify`): the scalar fp64 SEQUENTIAL LO-RANSAC of
    oracle/ransac_seq.cpp (E / F / H + decision tree, the C++ path BASELINE.md section 3 describes) on the sampled pairs
    that have >= 15 matches.  pairs/s = cores / (core-seconds per matched pair + verified fraction x core-seconds per
    verification)."""
    import oracle
    cores = os.cpu_count() or 1
    rng = np.random.default_rng(123)
    probe = pairs[rng.choice(len(pairs), min(len(pairs), 2 * cores), replace=False)]
    t0 = time.perf_counter()
    oracle.fast_match_pairs(desc_np, n_feat, probe, n_threads=cores)
    dt = max(time.perf_counter() - t0, 1e-6)
    rate = len(probe) / dt
    n = int(min(len(pairs), max(2 * cores, rate * budget_s * 0.7)))
    sample = pairs[rng.choice(len(pairs), n, replace=False)]
    t0 = time.perf_counter()
    res = oracle.fast_match_pairs(desc_np, n_feat, sample, n_threads=cores)
    dt = time.perf_counter() - t0
    out = {"value": n / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
           "match_pairs_per_s": n / dt,
           "sample": f"{n} random pairs of the same scene, oracle.fast_match_pairs ({oracle.fast_isa()}), {dt:.1f} s"}
    if verify and kpts_np is not None:
        from oracle import ransac_seq
        K = int(n_feat[0])
        cand = [k for k in range(n) if len(res[k]) >= 15]
        frac = len(cand) / max(n, 1)
        if cand:
            def jobs_of(idx):
                return [(cam, kpts_np[sample[k, 0] * K:(sample[k, 0] + 1) * K].astype(np.float64), cam,
                         kpts_np[sample[k, 1] * K:(sample[k, 1] + 1) * K].astype(np.float64), res[k]) for k in idx]
            probe_idx = cand[: min(len(cand), cores)]
            t0 = time.perf_counter()
            ransac_seq.verify_pairs(jobs_of(probe_idx), seed=1, n_threads=cores)
            per_wave = max(time.perf_counter() - t0, 1e-3)
            waves = max(1, min(int(0.3 * budget_s / per_wave), (len(cand) + cores - 1) // cores))
            idx = cand[: waves * cores]
            t0 = time.perf_counter()
            got, scored = ransac_seq.verify_pairs(jobs_of(idx), seed=1, n_threads=cores)
            wall = time.perf_counter() - t0
            out["verify_sample"] = [(k, int(r[0]), int(r[4])) for k, r in zip(idx, got)]
            core_s_verify = wall * min(cores, len(idx)) / len(idx)
            core_s_match = cores * dt / n
            out["verify_core_seconds_per_pair"] = core_s_verify
            out["verify_models_scored_per_pair"] = scored / len(idx)
            # the sample comes from the first images of the scene (denser in overlapping pairs than the
            # whole exhaustive set): weight with the verified fraction of the FULL workload when known
            use = frac if full_frac is None else full_frac
            out["verified_fraction_of_pairs"] = use
            out["verified_fraction_in_sample"] = frac
            out["value"] = cores / (core_s_match + use * core_s_verify)
            out["sample"] += (f"; + oracle/ransac_seq.cpp (scalar fp64 sequential LO-RANSAC, E/F/H + decision) on {len(idx)} "
                              f"of the sampled pairs with >= 15 matches ({min(cores, len(idx))} threads, {wall:.1f} s)")
    return out, sample, res


def resolve_config(args):
    cfg = dict(CONFIGS[args.config])
    if args.images:
        cfg["images"] = args.images
    if args.feats:
        cfg["feats"] = args.feats
    if args.verify >= 0:
        cfg["verify"] = args.verify
        cfg["guided"] = cfg["guided"] and args.verify
    what = ("exhaustive matching" if cfg["pairs"] == "exhaustive" else
            "sequential matching (overlap 20, quadratic_overlap)")
    cfg["workload"] = (f"{cfg['images']} images x {cfg['feats']} SIFT-like uint8 128-D descriptors, {what}"
                       + (" + two-view verification (E/F/H LO-RANSAC)" if cfg["verify"] else "")
                       + (" + guided matching" if cfg["guided"] else "")
                       + f"; BASELINE configs[{cfg['baseline_index']}]")
    cfg["metric"] = "image-pairs matched+verified/sec" if cfg["verify"] else "image-pairs matched/sec"
    return cfg


def pair_list(pb, cfg):
    n = cfg["images"]
    if cfg["pairs"] == "sequential":   # SequentialFeatureMatcher (images already in name order), SURVEY.md row P2
        return np.ascontiguousarray(pb.sequential_pairs(n, 20, True))
    # every unordered pair once, visited block by block like ExhaustiveFeatureMatcher::Run with the default
    # block_size = 50 (U:controllers/feature_matching.cc): a 50 x 50 block re-uses 100 images, which stay L2-resident
    return np.ascontiguousarray(np.concatenate(pb.exhaustive_pair_blocks(n, 50)))


DUMP_BYTES = 64 * 10 ** 6    # everything --dump-outputs writes, .npy headers included
DUMP_SUMMARY_PAIRS = 32768


def dump_outputs(out_dir, res, pairs, feats, verify):
    """--dump-outputs: what the caller of match_pairs received, one float .npy per array under out_dir.

    The pairs are a seeded sample that depends on the pair count alone, never on the results, so that two builds
    dump the same pairs.  For up to DUMP_SUMMARY_PAIRS of them, in pair-list order: `pairs` (image indices),
    `num_matches` and, with verification, `config`, `num_inliers`, `E`, `F`, `H`, `cam2_from_cam1` (3 x 4) and
    `tri_angle`.  For as many of those pairs as fit DUMP_BYTES even when every pair had `feats` matches (the most
    one image can have), flagged by `has_lists`: their `matches` and `inlier_matches` concatenated in the same order
    (`num_matches` / `num_inliers` of the flagged pairs split them)."""
    order = np.random.default_rng(0).permutation(len(pairs))
    summary = np.sort(order[:DUMP_SUMMARY_PAIRS])
    ks = summary.tolist()
    out = {"pairs": pairs[summary].astype(np.float64),
           "num_matches": np.array([len(res.matches(k)) for k in ks], np.float64)}
    if verify:
        geoms = [res.two_view_geometry(k) for k in ks]
        out["config"] = np.array([int(g.config) for g in geoms], np.float64)
        out["num_inliers"] = np.array([len(g.inlier_matches) for g in geoms], np.float64)
        for m in ("E", "F", "H"):
            out[m] = np.stack([getattr(g, m) for g in geoms]).astype(np.float64)
        out["cam2_from_cam1"] = np.stack([g.cam2_from_cam1.matrix() for g in geoms]).astype(np.float64)
        out["tri_angle"] = np.array([g.tri_angle for g in geoms], np.float64)
    fixed = sum(a.nbytes for a in out.values()) + len(summary) * 8 + (1 << 16)   # + has_lists, headers
    per_pair = feats * 2 * 4 * (2 if verify else 1)                                # <= feats rows x 2, float32
    listed = np.isin(summary, order[:max(0, (DUMP_BYTES - fixed) // per_pair)])
    out["has_lists"] = listed.astype(np.float64)
    pos = np.flatnonzero(listed)
    out["matches"] = np.concatenate([res.matches(ks[i]) for i in pos] + [np.zeros((0, 2))]).astype(np.float32)
    if verify:
        out["inlier_matches"] = np.concatenate([geoms[i].inlier_matches for i in pos]
                                               + [np.zeros((0, 2))]).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return sum(a.nbytes for a in out.values())


def reference_arm(args, cfg, rank):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself cannot be built here,
    DESIGN.md section 0) on the host cores, bounded sample of the same workload per step."""
    if rank != 0:
        return
    from pycolmap_b200 import synthetic as syn
    n_img, K, verify = cfg["images"], cfg["feats"], cfg["verify"]
    n_small = min(n_img, 64)
    scene = syn.make_scene(n_img, K, seed=0, device="cpu", image_range=(0, n_small))
    desc = scene["desc"].numpy().reshape(-1, 128)
    nf = np.full(n_small, K, np.int32)
    pairs = syn.exhaustive_pairs(n_small) if cfg["pairs"] == "exhaustive" else np.array(
        [(i, j) for i in range(n_small) for j in range(i + 1, min(n_small, i + 20))], np.int32)
    vals, step_ms = [], []
    # verified fraction of the full workload from the scene geometry: images further apart than
    # 2 x window_images (default 24) share no points (pycolmap_b200/synthetic.py)
    full_frac = min(1.0, 2.0 * (2 * 24 - 1) / max(n_img - 1, 1)) if cfg["pairs"] == "exhaustive" else 0.7
    for it in range(args.warmup + args.steps):
        t_step = time.perf_counter()
        cb, _, _ = cpu_baseline(desc, nf, pairs, max(2.0, args.cpu_seconds / 2), verify,
                                scene["kpts"].numpy().reshape(-1, 2), scene["cameras"][0], full_frac=full_frac)
        if it >= args.warmup:
            vals.append(cb)
            step_ms.append((time.perf_counter() - t_step) * 1e3)
    v = float(np.mean([c["value"] for c in vals])) if vals else 0.0
    cb = vals[-1] if vals else {"cores": os.cpu_count(), "kind": "port", "sample": "none"}
    cb["value"] = v
    cb.pop("verify_sample", None)
    print(json.dumps({
        "impl": "reference", "metric": cfg["metric"], "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(step_ms)) if step_ms else None,  # wall time of one bounded sample
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": cfg["workload"], "note": "first 64 images of the same scene; bounded sample per step",
                   "cpu_model": cpu_model()},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip() + f" ({os.cpu_count()} logical cores)"
    except OSError:
        pass
    return f"unknown ({os.cpu_count()} logical cores)"


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = resolve_config(args)
    n_img, K, verify, guided = cfg["images"], cfg["feats"], cfg["verify"], cfg["guided"]

    if args.impl == "reference":
        reference_arm(args, cfg, rank)
        return

    import torch
    import torch.distributed as dist
    import pycolmap_b200 as pb
    from pycolmap_b200 import synthetic as syn

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- the library's own communicator (NCCL behind the C ABI): rank 0 makes the id, the launcher's store carries it
    ctx = pb.Context(device=local_rank, pair_batch=args.pair_batch)
    if world > 1:
        box = [pb.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init_rank(world, rank, box[0])

    # ---- data: every rank synthesises ONLY the images it owns; they stay resident in its HBM (device leg) and in
    # pinned host memory (e2e leg).  Making the whole set resident everywhere is part of every step.
    first, count = pb.comm_image_range(n_img, world, rank)
    scene = syn.make_scene(n_img, K, seed=0, device=dev, image_range=(first, first + count))
    d_desc = scene["desc"].reshape(-1, 128).contiguous()
    d_kpts = scene["kpts"].reshape(-1, 2).contiguous()
    torch.cuda.synchronize()
    if rank == 0:
        log(f"scene ready: {n_img} images x {K} features, {count} images on this rank ({world} rank(s))")
    cam = dict(model=0, width=1600, height=1200, params=[1200.0, 800.0, 600.0], has_prior_focal_length=1)
    cams = [cam] * n_img if verify else None
    nfeat = np.full(n_img, K, np.int32)
    all_pairs = pair_list(pb, cfg)
    my_pairs = np.ascontiguousarray(all_pairs[rank::world])       # independent units: no data-path collective after the gather
    sift = pb.SiftMatchingOptions(guided_matching=bool(guided), max_num_matches=max(32768, K))
    tvg = pb.TwoViewGeometryOptions() if verify else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(host=None, keep=False):
        """One pass of the hot path: shard -> whole set resident on this GPU (copy + ONE all-gather) -> match
        (+ verify) this rank's pairs.  `host`: (desc, kpts) pinned host arrays of the local shard (e2e leg).
        `keep`: hand the result object back as out["res"] instead of freeing it."""
        w0 = time.perf_counter()
        if host is None:
            ctx.set_images_sharded(nfeat, first, count, d_desc.data_ptr(), d_kpts.data_ptr() if verify else None, cams,
                                   bool(verify))
        else:
            ctx.set_images_sharded(nfeat, first, count, host[0], host[1] if verify else None, cams, bool(verify))
        w1 = time.perf_counter()
        res = ctx.match_pairs(my_pairs, sift, tvg)
        w2 = time.perf_counter()
        st = ctx.stats()
        out = dict(dev_ms=st["last_upload_ms"] + st["last_allgather_ms"] + st["last_total_ms"], k1_ms=st["last_k1_ms"],
                   k1_n=st["last_k1_launches"], matches=res.total_matches, ver_ms=st["last_verify_ms"],
                   n_ver=res.num_verified, ag_ms=st["last_allgather_ms"], ag_bytes=st["last_allgather_bytes"],
                   up_ms=st["last_upload_ms"])
        if host is not None:                  # touch the result object like a caller would
            _ = res.matches(len(my_pairs) - 1)
            if verify:
                _ = res.two_view_geometry(len(my_pairs) - 1)
        if keep:
            out["res"] = res
        else:
            res.free()
        out["wall_ms"] = dict(upload=(w1 - w0) * 1e3, match_pairs=(w2 - w1) * 1e3, read_and_free=(time.perf_counter() - w2) * 1e3)
        return out

    for _ in range(args.warmup):
        one_step()
    barrier()
    if rank == 0:
        log("warm-up done")
    ctx.reset_stats()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    t_wall0 = time.perf_counter()
    acc = dict(dev_ms=0.0, k1_ms=0.0, k1_n=0, ver_ms=0.0, ag_ms=0.0, up_ms=0.0)
    last = None
    for i in range(args.steps):
        last = one_step(keep=bool(args.dump_outputs) and i == args.steps - 1)
        for k in acc:
            acc[k] += last[k]
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    if rank == 0:
        log(f"timed region done: {wall_ms / max(args.steps, 1):.0f} ms/step")
    clk = clocks.stop() if rank == 0 else None
    st_end = ctx.stats()
    launches = st_end["kernel_launches"]
    if args.dump_outputs:
        if rank == 0:
            nbytes = dump_outputs(args.dump_outputs, last["res"], my_pairs, K, verify)
            log(f"outputs of the last timed step: {nbytes / 1e6:.1f} MB in {args.dump_outputs}")
        last["res"].free()

    t = torch.tensor([acc["dev_ms"], wall_ms, acc["k1_ms"], acc["ag_ms"]], dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(len(my_pairs)), float(launches), float(last["n_ver"]), float(last["matches"])],
                       dtype=torch.float64, device=dev)
    ag_min = torch.tensor([acc["ag_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        dist.all_reduce(ag_min, op=dist.ReduceOp.MIN)
    ag_ms_min = ag_min.item()
    dev_ms_max, wall_ms_max, k1_ms_max, ag_ms_max = t.tolist()
    pairs_total, launches_total, verified_total, matches_total = cnt.tolist()
    verified_fraction = verified_total / max(pairs_total, 1) if verify else 0.0
    ms_per_step = dev_ms_max / args.steps
    value = pairs_total / (ms_per_step / 1e3)

    # ---- e2e: the same step from PINNED HOST buffers of the local shard (H2D inside), results read on the host
    e2e = None
    if not args.no_e2e:
        h_desc = torch.empty(d_desc.shape, dtype=torch.uint8, pin_memory=True)
        h_desc.copy_(d_desc)
        h_kpts = torch.empty(d_kpts.shape, dtype=torch.float32, pin_memory=True)
        h_kpts.copy_(d_kpts)
        host = (h_desc.numpy(), h_kpts.numpy())
        one_step(host)
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(1, min(args.steps, 3))
        for _ in range(n_e2e):
            r = one_step(host)
        barrier()
        e2e_s = (time.perf_counter() - t0) / n_e2e
        te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        by = torch.tensor([float(count * K * (128 + (8 if verify else 0)) + len(my_pairs) * 8),
                           float(r["matches"] * 8 + len(my_pairs) * 12)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dist.all_reduce(by, op=dist.ReduceOp.SUM)
        e2e = {"value": pairs_total / te.item(), "unit": "pairs/s", "h2d_bytes_per_step": int(by[0].item()),
               "d2h_bytes_per_step": int(by[1].item()), "steps": n_e2e,
               "wall_ms_last_step_rank0": {k: round(v, 1) for k, v in r["wall_ms"].items()},
               "note": "per step: b2m_set_images_sharded from pinned host memory (each rank uploads its 1/N of the images, "
                       "NCCL all-gather) + b2m_match_pairs + results read on the host; wall clock, max over ranks; "
                       "byte counts summed over ranks"}

    if rank != 0:
        if world > 1:
            ctx.comm_destroy()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (K1: int8 GEMM + fused top-2), tensor-bound
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bf16 = peaks.get("bf16_tflops_sustained")
    peak_src = "2 x MEASURED_PEAKS.json bf16_tflops_sustained (derived int8 peak: kind::i8 runs at twice the bf16 rate)"
    if not bf16:
        bf16, peak_src = 1400.0, "2 x fallback sustained bf16 1.4 PFLOP/s (B200_PROFILING.md), derived int8 peak"
    peak = 2.0 * bf16
    try:
        # measured on this pool's B200 by tools/microbench.cu (tcgen05.mma.kind::i8 issue loop, all SMs)
        mb = json.load(open(os.path.join(ROOT, "profiles", "r01_microbench_tmem_i8mma.json")))
        peak = float(mb["i8_mma_n256_chip_TOPS"])
        peak_src = ("measured int8 tcgen05 peak, tools/microbench.cu on this pool's B200 "
                    "(profiles/r01_microbench_tmem_i8mma.json, burst, 1965 MHz)")
    except Exception:
        pass
    # K1 is timed INSIDE a long step (the board sits at its power cap): the applicable peak is the SUSTAINED one
    # (B200_PROFILING.md: burst for a kernel timed alone, sustained for a kernel inside a long step) -- the same MMA
    # loop back to back for 4 s, tools/microbench.cu.  The burst figure and the fraction against it are kept beside it
    # (round 1 quoted the burst fraction).
    peak_burst, peak_burst_src = peak, peak_src
    try:
        mb = json.load(open(os.path.join(ROOT, "profiles", "r02_microbench_sustained.json")))
        peak = float(mb["i8_mma_n256_chip_TOPS_sustained"])
        peak_burst = float(mb["i8_mma_n256_chip_TOPS"])
        peak_src = ("measured SUSTAINED int8 tcgen05 peak: tools/microbench.cu MMA loop back to back for 4 s on this pool's "
                    "B200, last second timed (profiles/r02_microbench_sustained.json; 1725-1760 MHz at the 1 kW power cap); "
                    "burst in the same run %.1f TOP/s at 1965 MHz" % peak_burst)
    except Exception:
        pass
    ops_per_pair = 2.0 * K * K * 128
    k1_avg_ms = acc["k1_ms"] / max(acc["k1_n"], 1)
    pairs_per_launch = len(my_pairs) * args.steps / max(acc["k1_n"], 1)
    achieved = ops_per_pair * pairs_per_launch / (k1_avg_ms / 1e3) / 1e12
    dir1_mode = int(st_end["k1_dir1_mode"])
    split = dir1_mode in (1, 4, 6, 7)
    gathered = dir1_mode in (6, 7)
    # api.cu match_pairs_impl: resolve + gather of batch b next to the RANSAC kernels of batch b - 1
    overlapped = (gathered and bool(verify) and not guided and "B2M_NO_OVERLAP" not in os.environ
                  and len(my_pairs) > pairs_per_launch)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch of the schedule in use (profiles/, ncu --set full)
        tr = json.load(open(os.path.join(ROOT, "profiles", "k1_traffic.json")))
        key = f"{'gather' if gathered else 'split' if split else 'full'}_{K}"
        traffic = tr[key]["bytes_per_pair"] * pairs_per_launch if key in tr else None
    except Exception:
        pass
    roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s", "frac": achieved / peak,
            "traffic": traffic,
            "kernel": ("b2m_k1_filter_kernel x2 per batch: row direction of all pairs + column direction of the MATCHED columns "
                       "(gathered); " + ("overlapped order: K1 time = the two GEMM launches alone, CUDA events around each"
                                         if overlapped else
                                         "the exact resolve of the row direction and the gather run between the two and are "
                                         "inside the K1 time") if gathered else
                       "b2m_k1_filter_kernel x2 per batch (row direction of all pairs + column direction of the live pairs)"
                       if split else "b2m_k1_filter_kernel"),
            "k1_dir1_mode": dir1_mode, "avg_launch_ms": k1_avg_ms,
            "pairs_per_launch": pairs_per_launch, "peak_source": peak_src,
            "peak_burst": peak_burst, "frac_burst": achieved / peak_burst,
            "whole_step_frac": ops_per_pair * len(my_pairs) / (ms_per_step / 1e3) / 1e12 / peak,
            "algorithmic": "2*K1*K2*128 int8 ops per pair (one GEMM; the transposed GEMM of the cross-check "
                           "direction is not counted)"}
    roof_verify = None
    if verify:
        # kernel-side counters (b2m_stats.verify_*): models scored x matches of the pair, per model kind.
        # Flops per residual as fixed in DESIGN.md: Sampson 33 (E, F), forward transfer 19 (H).
        res_e, res_f, res_h = st_end["verify_residuals"]
        flops = 33.0 * (res_e + res_f) + 19.0 * res_h
        ver_s = acc["ver_ms"] / 1e3
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
        roof_verify = {"bound": "alu", "residual_evaluations_per_s": (res_e + res_f + res_h) / max(ver_s, 1e-9),
                       "achieved": flops / max(ver_s, 1e-9) / 1e12, "unit": "TFLOP/s",
                       "peak": fp32_peak, "frac": flops / max(ver_s, 1e-9) / 1e12 / fp32_peak,
                       "peak_fp64": 37.0,
                       "peak_source": "nominal: fp32 148 SMs x 128 lanes x 2 x 1.965 GHz (the hypothesis-scoring loop is fp32 "
                                      "with an exact fp64 recheck of borderline points); fp64 37 TFLOP/s (B200 datasheet)",
                       "models_scored": list(st_end["verify_models_scored"]), "residuals": [res_e, res_f, res_h],
                       "ms_per_step": acc["ver_ms"] / args.steps,
                       "note": "time = resolve + cross-check compaction + E/F/H LO-RANSAC + decision kernels of this rank"}

    log("e2e leg done; cpu baseline ...")
    cb = None
    if not args.no_cpu:
        n_small = min(count, 48)
        sub_pairs = syn.exhaustive_pairs(n_small)
        cb, sample, cpu_res = cpu_baseline(d_desc[: n_small * K].cpu().numpy(), np.full(n_small, K, np.int32),
                                           sub_pairs, args.cpu_seconds, verify,
                                           d_kpts[: n_small * K].cpu().numpy(), cam,
                                           full_frac=verified_fraction if verify else None)
        cb["cpu_model"] = cpu_model()
        # the same sample through the GPU path must be bit-identical (matching) and agree on the verification outcome
        c2 = pb.Context(device=local_rank)
        c2.set_images([d_desc[i * K:(i + 1) * K].cpu().numpy() for i in range(n_small)],
                      [d_kpts[i * K:(i + 1) * K].cpu().numpy() for i in range(n_small)], [cam] * n_small)
        chk = c2.match_pairs(sample, pb.SiftMatchingOptions(), tvg)
        same = all(np.array_equal(chk.matches(k), cpu_res[k] if (not verify or len(cpu_res[k]) >= 15) else cpu_res[k][:0])
                   for k in range(len(sample)))
        cb["gpu_bit_exact_on_sample"] = bool(same)
        if verify and cb.get("verify_sample") is not None:
            agree = []
            for k, cfg_cpu, n_inl_cpu in cb.pop("verify_sample"):
                g = chk.two_view_geometry(k)
                ok = int(g.config) == (cfg_cpu if n_inl_cpu >= 15 else 0)
                agree.append(ok and abs(len(g.inlier_matches) - (n_inl_cpu if n_inl_cpu >= 15 else 0))
                             <= max(2, int(0.01 * n_inl_cpu)))
            cb["gpu_verification_agrees_on_sample"] = f"{sum(agree)}/{len(agree)} pairs: same configuration, inliers within +-1 %"
        chk.free()
        c2.close()

    out = {
        "metric": cfg["metric"], "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": cfg["workload"], "config": args.config, "images": n_img, "features_per_image": K,
                   "pairs_per_step": int(pairs_total), "matches_per_step": int(matches_total),
                   "verified_pairs_fraction": verified_fraction, "guided_matching": bool(guided),
                   "parallelism": f"images sharded x{world} for the upload, ONE NCCL all-gather per step, pairs dealt round-robin x{world}",
                   "pair_batch": args.pair_batch or "library default",
                   "l2": "inputs (descriptor set %.2f GB) larger than L2" % (n_img * K * 128 / 1e9),
                   "timing": "CUDA events on the library stream: b2m_set_images_sharded (copy + all-gather) + "
                             "b2m_match_pairs of every step, max over ranks"},
        "wall_ms_per_step": wall_ms_max / args.steps, "k1_ms_per_step": acc["k1_ms"] / args.steps,
        "compact_verify_ms_per_step": acc["ver_ms"] / args.steps,
        # max over ranks = what the step pays (it includes waiting for the slowest rank to ARRIVE: the ranks are not
        # synchronised between steps); min over ranks = the last rank to arrive = the transfer itself
        "allgather": {"ms_per_step": ag_ms_max / args.steps, "transfer_ms_per_step": ag_ms_min / args.steps,
                      "bytes_received_per_rank": int(last["ag_bytes"]),
                      "GBps_per_rank": (last["ag_bytes"] / 1e9) / max(ag_ms_min / args.steps / 1e3, 1e-9) if world > 1 else None,
                      "share_of_step": ag_ms_max / max(dev_ms_max, 1e-9),
                      "nvlink_peak_GBps": 900.0 if world > 1 else None},
        "upload_ms_per_step": acc["up_ms"] / args.steps,
        "gpu_launches": int(launches_total), "clocks": clk,
        "roofline": roof, "roofline_verify": roof_verify, "cpu_baseline": cb, "e2e": e2e,
    }
    print(json.dumps(out))
    if world > 1:
        ctx.comm_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
