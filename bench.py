#!/usr/bin/env python
"""bench.py -- shape-pair distance queries/sec on a 1M-pair batch (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            (our arm; torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...   (CPU reference arm)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (+ the last timed step's records as .npy)

One "step" = one pass of the hot path (distance(): closed form / GJK / EPA + witness
points) over one batch of synthetic pairs.  Workload at every N: BASELINE config 2,
`--pairs` (default 1M) mixed primitive pairs PER GPU (weak scaling), distinct
seeds per rank, as a scene: 100 k objects and the 1 M object pairs whose relative
pose falls in config 2's box.  `value` = pairs/s with the expanded pair rows resident
in HBM; `e2e` = the same pairs through the host C-ABI call of the scene form
(hfb_batch_distance_objects) with pinned HOST buffers, H2D and D2H inside the timed
region.  For N>1 geometry is broadcast once over NCCL and the per-rank result buffers
are all-gathered inside the timed step.  At N=1 the line also carries, under
`workloads`, BASELINE configs 3 and 4 at their own sizes (value / e2e / roofline /
cpu_baseline each) and the convex-support kernel's roofline.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "shape_pair_distance_queries_per_sec"
UNIT = "pairs/s"
# algorithmic bytes per pair of the phase-1 kernel (DESIGN.md "roofline"):
#   2 handles (8) + 2 poses (192) + 2 shape records (80) + 1 result record (96)
BYTES_PER_PAIR = 8 + 192 + 80 + 96


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config4", "config5"])
    ap.add_argument("--variant", type=int, default=None,
                    help="0 DefaultGJK, 1 Polyak, 2 NesterovAcceleration (default: 0; config3: 2, as BASELINE names it)")
    ap.add_argument("--cpu-sample", type=int, default=400_000)
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU arm (0: calibrated)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64; rows in pair order, "
                         "config5's candidate pairs sorted by (first, second); a fixed sample of rows when the whole "
                         "exceeds 64 MB), so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.variant is None:
        a.variant = 2 if a.workload == "config3" else 0
    if a.workload == "config4" and a.pairs == 1_000_000:
        a.pairs = 100_000  # BASELINE config 4 is quoted on 100k capsules
    if a.workload == "config5" and a.pairs == 1_000_000:
        a.pairs = 100_000  # BASELINE config 5: 100 k moving boxes (objects; about 1 M candidate pairs)
    if a.cpu_sample == 400_000:
        a.cpu_sample = {"config2": 400_000, "config3": 100_000, "config4": 20_000, "config5": 200_000}[a.workload]
    return a


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.rows = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


DUMP_BYTES = 64_000_000


def dump_outputs(directory, columns):
    """columns: name -> array with one row per output row (records of the last timed step, split into fields), in an
    order that does not depend on the run.  Every column is written as float64 (integer fields are exact there); when
    all of them together exceed DUMP_BYTES, the same seeded sample of rows is taken from each and its row numbers are
    written as `row`."""
    n = len(next(iter(columns.values())))
    row_bytes = sum(8 * int(np.prod(a.shape[1:])) for a in columns.values())
    budget = DUMP_BYTES - 256 * (len(columns) + 1)  # (the .npy headers)
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        columns = dict({k: a[rows] for k, a in columns.items()}, row=rows)
    os.makedirs(directory, exist_ok=True)
    for k, a in columns.items():
        np.save(os.path.join(directory, k + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def record_columns(rec):
    return {f: rec[f] for f in rec.dtype.names if not f.startswith("_")}


def make_workload(args, rank, workload=None, pairs=None):
    """-> (w, name): w holds the geometry to register and the batch in POOL indices: rows h1/tf1/h2/tf2 (every
    workload) and, for config 2, the scene they were expanded from (obj_h, obj_tf, first, second)."""
    from hppfcl_b200 import workloads as W
    workload = workload or args.workload
    pairs = pairs or args.pairs
    if workload == "config2":
        # BASELINE config 2 as a scene: 1 M pairs over pairs / 10 objects, relative poses with config 2's statistics
        s = W.config2_scene(max(pairs // 10, 2000), pairs, seed=0xFC1 + 2 + 1000 * rank)
        w = dict(shapes=s["shapes"], obj_h=s["obj_h"], obj_tf=s["obj_tf"], first=s["first"], second=s["second"],
                 h1=s["obj_h"][s["first"]], h2=s["obj_h"][s["second"]],
                 tf1=np.ascontiguousarray(s["obj_tf"][s["first"]]), tf2=np.ascontiguousarray(s["obj_tf"][s["second"]]))
        name = ("config2: %d mixed primitive pairs (sphere/capsule/box/cylinder) of a %d-object scene, GJK distance + "
                "witness points" % (pairs, len(s["obj_h"])))
    elif workload == "config3":
        w = W.config3_convex_pairs(pairs, seed=0xFC1 + 3 + 1000 * rank)
        name = "config3: %d ConvexBase(64) x ConvexBase(64) pairs, %s GJK distance + EPA penetration/contact points" % (
            pairs, {0: "default", 1: "Polyak-accelerated", 2: "Nesterov-accelerated"}[variant_of(args, workload)])
    else:
        c = W.config4_mesh_vs_capsules(pairs, seed=0xFC1 + 4 + 1000 * rank)
        # handle table: [mesh] + capsule pool; pair k = (mesh, capsule hc[k])
        w = dict(verts=c["verts"], tris=c["tris"], capsules=c["capsules"],
                 h1=np.zeros(pairs, dtype=np.uint32), h2=(1 + c["hc"]).astype(np.uint32),
                 tf1=c["tf_mesh"], tf2=c["tf_caps"])
        name = "config4: %d-triangle OBBRSS BVH mesh vs %d capsules, distance + nearest points" % (len(c["tris"]), pairs)
    return w, name


def variant_of(args, workload):
    """GJK variant of a workload: --variant for the main one; BASELINE names Nesterov for config 3"""
    if workload == args.workload and args.variant is not None:
        return args.variant
    return 2 if workload == "config3" else 0


DEFAULT_PAIRS = {"config2": 1_000_000, "config3": 1_000_000, "config4": 100_000}
CPU_SAMPLE = {"config2": 400_000, "config3": 100_000, "config4": 20_000}


def register(eng_or_orc, w, workload, oracle=False):
    from hppfcl_b200 import _pod as P
    if workload == "config2":
        return eng_or_orc.register_shapes(w["shapes"])
    if workload == "config4":
        if oracle:  # the oracle builds the tree with its restatement of the reference builder
            bid, _ = eng_or_orc.register_bvh(w["verts"], w["tris"])
        else:       # the product builds it with its own host builder (hfb_bvh_build_obbrss)
            bid = eng_or_orc.register_bvh_obbrss(None, w["verts"], w["tris"])
        hm = eng_or_orc.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]))
        hc = eng_or_orc.register_shapes(w["capsules"])
        return np.concatenate([hm, hc])
    cids = []
    for pts, tris in w["hulls"]:
        cids.append(eng_or_orc.register_convex(pts, tris) if oracle else eng_or_orc.register_convex(pts))
    return eng_or_orc.register_shapes(P.make_shapes([P.GEOM_CONVEX] * len(cids), np.zeros((len(cids), 3)), data=cids))


def cpu_arm_kind():
    from oracle import oracle_lib
    return "reference" if oracle_lib.ref_available() else "port"


_CAL = {}  # thread count of the CPU arm, calibrated once per (workload, variant) and process


def cpu_reference_rate(args, w, workload, n_sample, threads=0):
    """The reference's CPU path on a bounded sample of the same workload: oracle/_ref (the reference's own
    sources compiled in place, see oracle/Makefile `ref`) when it was built, else the oracle's restatement."""
    from hppfcl_b200 import _pod as P
    from oracle import oracle_lib
    key = (workload, variant_of(args, workload))
    if "scene" not in _CAL.setdefault(key, {}):
        orc = oracle_lib.RefScene(P) if oracle_lib.ref_available() else oracle_lib.OracleScene(P)
        _CAL[key]["scene"] = (orc, register(orc, w, workload, oracle=True))
    orc, hs = _CAL[key]["scene"]
    n = min(n_sample, len(w["h1"]))
    h1, h2 = hs[w["h1"][:n] % len(hs)], hs[w["h2"][:n] % len(hs)]
    req = P.DistanceRequestPOD(gjk_variant=variant_of(args, workload))
    # "all the host threads it can use": torchrun exports OMP_NUM_THREADS=1 and the box exposes 128 logical
    # CPUs of which oversubscribing hurts (measured: 128 threads 6e6 pairs/s, 64 threads 3.4e7), so the
    # thread count is calibrated ONCE on a short sample among {affinity, affinity/2, affinity/4, OpenMP's default}
    if threads == 0:
        threads = _CAL[key].get("threads", 0)
    if threads == 0:
        aff = len(os.sched_getaffinity(0))
        cands = sorted({c for c in (aff, max(1, aff // 2), max(1, aff // 4), oracle_lib.lib().oracle_max_threads()) if c >= 1})
        m = min(n, 50000 if workload != "config4" else 4000)
        best, best_t = 1, None
        for c in cands:
            orc.batch_distance(h1[:m], w["tf1"][:m], h2[:m], w["tf2"][:m], req, nthreads=c)  # spin the team up
            t0 = time.perf_counter()
            orc.batch_distance(h1[:m], w["tf1"][:m], h2[:m], w["tf2"][:m], req, nthreads=c)
            dtc = time.perf_counter() - t0
            if best_t is None or dtc < best_t:
                best, best_t = c, dtc
        threads = _CAL[key]["threads"] = best
    t0 = time.perf_counter()
    orc.batch_distance(h1, w["tf1"][:n], h2, w["tf2"][:n], req, nthreads=threads)
    dt = time.perf_counter() - t0
    return n / dt, threads, n


def run_reference(args):
    rank, local, world = env_rank()
    if rank != 0:
        return
    if args.workload == "config5":
        c = cpu_config5(args, args.pairs, args.cpu_sample)
        line = {"metric": METRIC, "value": c["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
                "config": {"workload": "config5: %d moving boxes, broadphase -> narrow phase (collide)" % args.pairs},
                "cpu_baseline": c, "e2e": {"value": c["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return
    w, name = make_workload(args, 0)
    rates = []
    n = args.cpu_sample
    cores = 1
    for it in range(args.warmup + args.steps):
        r, cores, n = cpu_reference_rate(args, w, args.workload, args.cpu_sample, threads=args.cpu_threads)
        if it >= args.warmup:
            rates.append(r)
    v = float(np.mean(rates))
    # whole-job figure under weak scaling: the CPU box is one host regardless of N
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * n / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "reference", "config": {"workload": name, "sample_pairs_per_step": n,
                                            "gjk_variant": variant_of(args, args.workload)},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": cpu_arm_kind(),
                             "sample": "%d pairs of the same seeded workload per step, OpenMP static over pairs" % n},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def support_kernel_roofline(eng_factory, peak, n_hulls=786432, nv=64, n_queries=1 << 21):
    """The north_star's convex-support kernel: batched ConvexBase support argmax over DISTINCT hulls
    (1.2 GB of vertices, ten times the 126 MB L2, each hull queried 2.7 times on average, so the
    algorithmic bytes are close to what DRAM delivers), one warp per query, coalesced SoA rows.
    Algorithmic bytes per query: 24*nv vertices + 24 B direction + 28 B output + 4 B id (SURVEY 8d:
    1 588 B at nv = 64)."""
    import torch
    from hppfcl_b200 import _pod as P
    rng = np.random.default_rng(99)
    eng = eng_factory(torch.cuda.current_device())
    v = rng.normal(size=(n_hulls, nv, 3))
    v /= np.linalg.norm(v, axis=2, keepdims=True)
    v *= 0.05 + 0.95 * rng.random((n_hulls, 1, 3))
    assert eng.register_convex_batch(v) == 0
    eng.commit()
    ids = rng.permutation(n_queries).astype(np.uint32) % n_hulls
    dirs = rng.normal(size=(n_queries, 3))
    d_ids = torch.from_numpy(ids).cuda()
    d_dirs = torch.from_numpy(dirs).cuda()
    d_idx = torch.empty(n_queries, dtype=torch.int32, device="cuda")
    d_sup = torch.empty((n_queries, 3), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(3):
        eng.batch_convex_support_device(n_queries, d_ids.data_ptr(), d_dirs.data_ptr(), d_idx.data_ptr(), d_sup.data_ptr(), stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        eng.batch_convex_support_device(n_queries, d_ids.data_ptr(), d_dirs.data_ptr(), d_idx.data_ptr(), d_sup.data_ptr(), stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    bytes_per = 24 * nv + 24 + 28 + 4
    achieved = bytes_per * n_queries / (ms * 1e-3) / 1e9
    # spot check against numpy
    k = 4096
    got = d_idx[:k].cpu().numpy()
    want = np.argmax(np.einsum("qvc,qc->qv", v[ids[:k]], dirs[:k]), axis=1)
    return {"kernel": "k_convex_support", "supports_per_s": n_queries / (ms * 1e-3), "kernel_ms": ms,
            "bytes_per_support": bytes_per, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "distinct_hulls": n_hulls, "vertices": nv, "queries": n_queries,
            "matches_numpy_argmax": bool(np.array_equal(got, want))}


def _peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    return peak, src


def _traffic(workload, n, variant):
    """DRAM bytes of the dominant kernel per full-size launch, from the committed ncu capture of this command
    (profiles/r02_dominant_kernel_traffic.json; a profiler run, not measured live)"""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_dominant_kernel_traffic.json")))
        e = tj[workload]
        if n == e.get("pairs") and variant == e.get("variant", variant):
            return e["traffic"], e.get("source")
    except Exception:
        pass
    return None, None


def measure(args, workload, rank, local, world, dist, steps, warmup, clocks=False):
    """One workload on this rank's GPU: device-resident rate (`value`), end-to-end rate through the host C-ABI with
    pinned host buffers (`e2e`), the per-kernel times of a SEPARATE profiled pass, roofline of the dominant kernel."""
    import torch
    import hppfcl_b200 as hf
    from hppfcl_b200 import _pod as P

    n = args.pairs if workload == args.workload else DEFAULT_PAIRS[workload]
    variant = variant_of(args, workload)
    w, name = make_workload(args, rank, workload, n)
    eng = hf.Engine(local)
    hs = register(eng, w, workload)
    eng.commit()
    h1 = hs[w["h1"] % len(hs)].astype(np.uint32)
    h2 = hs[w["h2"] % len(hs)].astype(np.uint32)
    req = P.DistanceRequestPOD(gjk_variant=variant)

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()

    d_h1, d_h2, d_tf1, d_tf2 = dev(h1), dev(h2), dev(w["tf1"]), dev(w["tf2"])
    out_bytes = n * P.distance_result_dtype.itemsize
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda") if world == 1 else None
    stream = torch.cuda.current_stream().cuda_stream
    # config 4's working set (34 MB) fits the 126 MB L2: flush it between steps by overwriting 256 MB
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if workload == "config4" else None
    if world > 1:
        # the product's communicator: every step's records are all-gathered by the library (NCCL, on its own stream,
        # overlapping the next step's kernels) into one of two buffers the context owns
        from hppfcl_b200 import sharding
        sharding.init_engine_comm(eng)

    def step():
        if flush is not None:
            flush.zero_()
        if world > 1:
            eng.batch_distance_sharded_device(n, d_h1.data_ptr(), d_tf1.data_ptr(), d_h2.data_ptr(), d_tf2.data_ptr(), req,
                                              stream=stream)
        else:
            eng.batch_distance_device(n, d_h1.data_ptr(), d_tf1.data_ptr(), d_h2.data_ptr(), d_tf2.data_ptr(),
                                      d_out.data_ptr(), req, stream=stream)

    def drain():
        if world > 1:
            eng.comm_wait(stream)  # the timed region ends when the last all-gather has landed

    def barrier():
        if world > 1:
            drain()
            torch.cuda.synchronize()
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    st0 = eng.stats()
    sampler = ClockSampler(local) if clocks else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        step()
    drain()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    st1 = eng.stats()
    if args.dump_outputs and workload == args.workload:
        dump_outputs(args.dump_outputs, record_columns(d_out.cpu().numpy().view(P.distance_result_dtype)))
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * n * steps / (ms * 1e-3)

    # ---- per-kernel times: a separate pass with the event hooks on (they are off in the timed region) ----
    prof_steps = 3
    eng.set_profiling(True)
    eng.kernel_times(reset=True)
    sp0 = eng.stats()
    for _ in range(prof_steps):
        step()
    barrier()
    kt = eng.kernel_times(reset=True)
    eng.set_profiling(False)
    sp1 = eng.stats()

    # ---- e2e: the host C-ABI call with pinned host buffers, H2D + D2H inside the timed region ----
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).pin_memory()
        return t, t.numpy().view(a.dtype).reshape(a.shape)

    keep = []
    t_out = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    host_out = t_out.numpy().view(P.distance_result_dtype)
    if workload == "config2":
        # the scene form (hfb_batch_distance_objects): object table + index pairs in, full result records out
        ph = []
        for a in (hs[w["obj_h"] % len(hs)].astype(np.uint32), w["obj_tf"], w["first"], w["second"]):
            t, v = pinned(a)
            keep.append(t)
            ph.append(v)
        h2d = int(ph[0].nbytes + ph[1].nbytes + ph[2].nbytes + ph[3].nbytes)
        api = "hfb_batch_distance_objects (object table + index pairs; full 96-byte records back)"

        def e2e_call():
            eng.batch_distance_objects(ph[0], ph[1], ph[2], ph[3], req, out=host_out)
    else:
        ph = []
        for a in (h1, w["tf1"], h2, w["tf2"]):
            t, v = pinned(a)
            keep.append(t)
            ph.append(v)
        h2d = int(n * 200)
        api = "hfb_batch_distance (pair rows)"

        def e2e_call():
            eng.batch_distance(ph[0], ph[1], ph[2], ph[3], req, out=host_out)

    def time_e2e(call, k):
        for _ in range(2):
            call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            call()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return world * n * k / dt

    e2e_steps = max(3, min(steps, 10))
    e2e_value = time_e2e(e2e_call, e2e_steps)
    checksum = float(np.nansum(host_out["min_distance"][:: max(1, n // 4096)]))
    res = {"workload": workload, "name": name, "n": n, "variant": variant, "value": value, "ms_per_step": ms / steps,
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(out_bytes),
                   "steps": e2e_steps, "checksum": checksum, "api": api},
           "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]),
           "watchdog_trips": int(st1["watchdog_trips"])}
    if workload == "config2":
        # secondary e2e figures: the pair-row form of round 1 (200 B per pair up), and distances only (8 B per pair down)
        ph2 = []
        for a in (h1, w["tf1"], h2, w["tf2"]):
            t, v = pinned(a)
            keep.append(t)
            ph2.append(v)
        res["e2e_pair_rows"] = {"value": time_e2e(lambda: eng.batch_distance(ph2[0], ph2[1], ph2[2], ph2[3], req, out=host_out), 3),
                                "unit": UNIT, "h2d_bytes_per_step": int(n * 200), "d2h_bytes_per_step": int(out_bytes),
                                "api": "hfb_batch_distance (pair rows)"}
        t_min = torch.empty(n, dtype=torch.float64).pin_memory()
        res["e2e_min_distance_only"] = {
            "value": time_e2e(lambda: eng.batch_distance_objects(ph[0], ph[1], ph[2], ph[3], req, out=t_min.numpy(), min_only=True), 3),
            "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(8 * n),
            "api": "hfb_batch_distance_objects, min_distance_out (8 bytes per pair back)"}
    if sampler:
        res["clocks"] = sampler.summary()

    # ---- workload statistics + roofline of the dominant kernel ----
    path = (host_out["status"] >> 16) & 0xff
    gjk_it = (host_out["iterations"] & 0xffff)[path == 0]
    epa_it = (host_out["iterations"] >> 16)[path == 0]
    peak, peak_src = _peak()
    if workload in ("config2", "config3"):
        ws = {"gjk_routed_pairs": int((path == 0).sum()), "closed_form_pairs": int((path == 1).sum()),
              "gjk_iterations_mean": float(gjk_it.mean()) if len(gjk_it) else 0.0,
              "gjk_iterations_max": int(gjk_it.max()) if len(gjk_it) else 0,
              "epa_pairs": int((epa_it > 0).sum()),
              "epa_iterations_mean": float(epa_it[epa_it > 0].mean()) if (epa_it > 0).any() else 0.0}
        res["workload_stats"] = ws
    if workload == "config2":
        # the passes are ONE unit of work over the GJK-routed pairs (several launches, timed in two scopes): per step
        dom, dom_ms, dom_launches = "GJK passes k_gjk_first/_more/_end (primitive pairs)", kt["pairs_ms"], prof_steps
        units = float((path == 0).sum())
        bpp = BYTES_PER_PAIR
    elif workload == "config4":
        # SURVEY 8d: 136 B per BV test (node header + RSS half), 96 B per leaf test (indices + vertices),
        # 232 B per query (capsule record + poses + result); counts from the device counters
        bv = (sp1["bv_tests"] - sp0["bv_tests"]) / prof_steps
        lf = (sp1["leaf_tests"] - sp0["leaf_tests"]) / prof_steps
        dom, dom_ms, dom_launches = "k_bvhq (+ k_bvhq_prep)", kt["bvh_ms"], max(1, kt["bvh_launches"] // 2)
        units = float(n)
        bpp = (136 * bv + 96 * lf) / n + 232
        res["workload_stats"] = {"bv_tests_per_query": bv / n, "leaf_tests_per_query": lf / n}
    else:
        dom, dom_ms, dom_launches = "k_pairs<G,CAPS_ALL,0,PATH_BOTH>", kt["convex_ms"], kt["convex_launches"]
        units = float(n)
        bpp = 2 * 1536 + 192 + 8 + 96
    k_ms = dom_ms / max(1, dom_launches)
    achieved = bpp * units / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    traffic, tsrc = _traffic(workload, n, variant)
    res["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                       "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": tsrc,
                       "bytes_per_pair": bpp, "pairs_per_launch": units, "kernel_ms": k_ms, "peak_source": peak_src,
                       "timing": "CUDA events around the kernel's launches on the launching stream, in a separate pass "
                                 "of %d steps after the timed region" % prof_steps}
    res["kernels"] = {"gjk_pairs_ms_per_step": kt["pairs_ms"] / prof_steps,
                      "closed_pairs_ms_per_step": kt["closed_ms"] / prof_steps,
                      "convex_pairs_ms_per_step": kt["convex_ms"] / prof_steps,
                      "bin_sort_ms_per_step": kt["other_ms"] / prof_steps,
                      "epa_ms_per_step": kt["epa_ms"] / prof_steps,
                      "bvh_ms_per_step": kt["bvh_ms"] / prof_steps,
                      "epa_pairs_per_step": (sp1["epa_pairs"] - sp0["epa_pairs"]) / prof_steps}
    if workload in ("config2", "config3") and res["kernels"]["gjk_pairs_ms_per_step" if workload == "config2" else "convex_pairs_ms_per_step"] > 0:
        # secondary view: FP64 issue.  ~450 flop per GJK iteration on primitives (SURVEY 8d estimate; the
        # convex kernels add 6 flop per hull vertex and support call); nominal B200 FP64 (non-tensor) 37 TFLOP/s
        it_flop = 450.0 if workload == "config2" else 450.0 + 2 * 64 * 6
        gsec = res["kernels"]["gjk_pairs_ms_per_step" if workload == "config2" else "convex_pairs_ms_per_step"] * 1e-3
        res["fp64_view"] = {"flop_per_gjk_iteration_estimate": it_flop,
                            "achieved_tflops_estimate": res["workload_stats"]["gjk_routed_pairs"] * res["workload_stats"]["gjk_iterations_mean"] * it_flop / gsec / 1e12,
                            "nominal_fp64_tflops": 37.0}
    if workload == "config2":
        names = {P.GEOM_SPHERE: "sphere", P.GEOM_CAPSULE: "capsule", P.GEOM_BOX: "box", P.GEOM_CYLINDER: "cylinder"}
        t1, t2 = w["shapes"]["type"][w["h1"]], w["shapes"]["type"][w["h2"]]
        res["workload_stats"]["type_histogram"] = {"%s-%s" % (names[a], names[b]): int(((t1 == a) & (t2 == b)).sum())
                                                   for a in names for b in names}
    res["l2"] = ("L2 flushed between steps (256 MB overwrite inside the timed region)" if flush is not None else
                 "inputs+outputs per step (%d MB) exceed the 126 MB L2; no explicit flush" % ((n * (BYTES_PER_PAIR - 80)) >> 20))
    del eng
    return res


def measure_config5(args, rank, local, world, dist, steps, warmup, n_objects=None):
    """BASELINE config 5: 100 k moving boxes, broadphase -> batched narrow phase (collide()).  One scene cut over the
    ranks by ranges of objects (STRONG scaling): every rank holds all the poses, computes the boxes and the grid, sweeps
    the candidate pairs of its own objects and runs collide() on them.  value: candidate pairs/s with the poses
    resident in HBM (boxes + grid + sweep + narrow phase inside the timed region); e2e: hfb_scene_collide with pinned
    host poses in, the colliding pairs' records out."""
    import torch
    import hppfcl_b200 as hf
    from hppfcl_b200 import _pod as P, workloads as W
    n = n_objects or args.pairs
    w = W.config5_moving_boxes(n, seed=0xFC1 + 5)
    eng = hf.Engine(local)
    hb = eng.register_shapes(w["shapes"])
    eng.commit()
    oh = hb[w["obj_h"]].astype(np.uint32)
    nposes = 4
    poses = [w["step"](k) for k in range(nposes)]
    lo, cnt = (n * rank) // world, (n * (rank + 1)) // world - (n * rank) // world
    req = P.CollisionRequestPOD()

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()

    d_h = dev(oh)
    d_tf = [dev(p) for p in poses]
    d_bb = torch.empty(n * 6, dtype=torch.float64, device="cuda")
    cap = int(2.0 * 1_000_000 * (n / 100_000.0) / world) + 65536
    d_f = torch.empty(cap, dtype=torch.int32, device="cuda")
    d_s = torch.empty(cap, dtype=torch.int32, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int32, device="cuda")
    d_out = torch.empty(cap * P.contact_dtype.itemsize, dtype=torch.uint8, device="cuda")
    h_n = torch.zeros(1, dtype=torch.int32).pin_memory()
    stream = torch.cuda.current_stream().cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    acc = {"pairs": 0, "bp_ms": 0.0, "np_ms": 0.0}

    def step(k, timed=False):
        t = d_tf[k % nposes]
        if timed:
            ev[0].record()
        eng.scene_aabbs_device(n, d_h.data_ptr(), t.data_ptr(), d_bb.data_ptr(), stream)
        eng.broadphase_pairs_device(n, d_bb.data_ptr(), d_f.data_ptr(), d_s.data_ptr(), cap, d_n.data_ptr(), stream,
                                    first_object=lo, num_first_objects=cnt)
        h_n.copy_(d_n, non_blocking=True)
        if timed:
            ev[1].record()
        torch.cuda.current_stream().synchronize()  # the narrow phase is launched for the number of candidates found
        k_pairs = int(h_n.item())
        assert k_pairs <= cap, "candidate buffer too small"
        eng.batch_collide_objects_device(n, d_h.data_ptr(), t.data_ptr(), k_pairs, d_f.data_ptr(), d_s.data_ptr(),
                                         d_out.data_ptr(), req, stream=stream)
        if timed:
            ev[2].record()
            torch.cuda.synchronize()
            acc["bp_ms"] += ev[0].elapsed_time(ev[1])
            acc["np_ms"] += ev[1].elapsed_time(ev[2])
        return k_pairs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(max(warmup, 3)):
        step(k)
    barrier()
    st0 = eng.stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for k in range(steps):
        acc["pairs"] += step(k)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    st1 = eng.stats()
    if args.dump_outputs and n_objects is None:
        # the sweep appends candidates through atomics, in no fixed order: sort them by (first, second) so that two
        # runs, and two builds, dump the same pairs in the same rows
        kp = int(d_n.item())
        cols = dict(first=d_f[:kp].cpu().numpy(), second=d_s[:kp].cpu().numpy(),
                    **record_columns(d_out[:kp * P.contact_dtype.itemsize].cpu().numpy().view(P.contact_dtype)))
        order = np.lexsort((cols["second"], cols["first"]))
        dump_outputs(args.dump_outputs, {k: a[order] for k, a in cols.items()})
    pairs = acc["pairs"]
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        t = torch.tensor([float(pairs)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        pairs = int(t.item())
    value = pairs / (ms * 1e-3)
    for k in range(3):  # broadphase / narrow phase split, separate pass
        step(k, timed=True)
    # ---- e2e: hfb_scene_collide, pinned host poses in, colliding pairs out ----
    pin = [torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).reshape(-1)).pin_memory() for p in poses]
    hp = [t.numpy().view(P.transform_dtype) for t in pin]
    ccap = 4 * n
    bufs = tuple(torch.empty(ccap * it, dtype=torch.uint8).pin_memory().numpy().view(dt) for it, dt in
                 ((4, np.uint32), (4, np.uint32), (P.contact_dtype.itemsize, P.contact_dtype)))
    tot = {"cand": 0, "hit": 0}

    def e2e_step(k):
        f, s2, rec, ncand, nhit = eng.scene_collide(oh, hp[k % nposes], req, capacity=ccap, first_object=lo, num_first_objects=cnt,
                                                    bufs=bufs)
        tot["cand"] += ncand
        tot["hit"] += nhit

    for k in range(2):
        e2e_step(k)
    barrier()
    tot["cand"] = tot["hit"] = 0
    e2e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        e2e_step(k)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    cand = tot["cand"]
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        t = torch.tensor([float(cand)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        cand = int(t.item())
    hits_per_step = tot["hit"] / e2e_steps
    res = {"workload": "config5", "n": n,
           "name": "config5: %d moving Box(5,10,20) objects, uniform-grid broadphase on the device -> batched narrow phase "
                   "(collide), about %d candidate pairs per step" % (n, pairs // max(1, steps)),
           "value": value, "ms_per_step": ms / steps, "candidate_pairs_per_step": pairs / steps,
           "e2e": {"value": cand / dt, "unit": UNIT, "h2d_bytes_per_step": int(n * 100), "steps": e2e_steps,
                   "d2h_bytes_per_step": int(hits_per_step * (8 + P.contact_dtype.itemsize) / max(1, world)),
                   "api": "hfb_scene_collide (poses in; colliding pairs + contact records out)",
                   "colliding_pairs_per_step": hits_per_step * (world if world > 1 else 1)},
           "split_ms_per_step": {"boxes_grid_sweep": acc["bp_ms"] / 3, "narrow_phase": acc["np_ms"] / 3},
           "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]),
           "scaling": "strong", "env_scale": w["env_scale"]}
    del eng
    return res


def cpu_config5(args, n_objects, sample_pairs):
    """CPU arm of config 5 (rank 0): the product's HOST pair finder on one thread (hpp-fcl's managers do not build
    here: boost::function) + the reference's collide() over a bounded sample of the candidates, all cores"""
    import hppfcl_b200 as hf
    from hppfcl_b200 import _pod as P, workloads as W
    from oracle import oracle_lib
    w = W.config5_moving_boxes(n_objects, seed=0xFC1 + 5)
    tf = w["step"](0)
    local = np.array([-2.5, -5, -10, 2.5, 5, 10.0])
    R = tf["R"].reshape(-1, 3, 3).transpose(0, 2, 1)
    mn = np.minimum(R * local[None, None, :3], R * local[None, None, 3:]).sum(axis=2)
    mx = np.maximum(R * local[None, None, :3], R * local[None, None, 3:]).sum(axis=2)
    bb = np.concatenate([tf["T"] + mn, tf["T"] + mx], axis=1)
    t0 = time.perf_counter()
    f, s2 = hf.broadphase_pairs(bb)
    t_bp = time.perf_counter() - t0
    orc = oracle_lib.RefScene(P) if oracle_lib.ref_available() else oracle_lib.OracleScene(P)
    hb = orc.register_shapes(w["shapes"])
    m = min(sample_pairs, len(f))
    h1 = np.full(m, hb[0], dtype=np.uint32)
    req = P.CollisionRequestPOD()
    aff = len(os.sched_getaffinity(0))
    best = None
    for c in sorted({aff, max(1, aff // 2), max(1, aff // 4)}):
        orc.batch_collide(h1[:20000], tf[f[:20000]], h1[:20000], tf[s2[:20000]], req, nthreads=c)
        t0 = time.perf_counter()
        orc.batch_collide(h1, tf[f[:m]], h1, tf[s2[:m]], req, nthreads=c)
        dtc = time.perf_counter() - t0
        if best is None or dtc < best[0]:
            best = (dtc, c)
    rate_np = m / best[0]
    total = t_bp + len(f) / rate_np
    return {"value": len(f) / total, "unit": UNIT, "cores": best[1], "kind": cpu_arm_kind(),
            "sample": "host pair finder of the product on 1 thread over %d objects (%.1f ms, %d candidates) + the "
                      "reference's collide() on %d of them, %d threads" % (n_objects, 1e3 * t_bp, len(f), m, best[1]),
            "narrow_phase_only_value": rate_np, "broadphase_ms": 1e3 * t_bp}


def cpu_arm(args, workload, sample, threads):
    """the CPU arm in a process of its own: this one has torch's OpenMP runtime loaded next to the system one, and
    the reference's per-call heap traffic is sensitive to that (measured 4e6 vs 2e7)"""
    n = args.pairs if workload == args.workload else DEFAULT_PAIRS[workload]
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload,
           "--pairs", str(n), "--variant", str(variant_of(args, workload)), "--steps", "2", "--warmup", "1",
           "--cpu-sample", str(sample), "--cpu-threads", str(threads)]
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS",)}
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1200).stdout
    for ln in out.splitlines():
        if ln.startswith("{"):
            d = json.loads(ln)
            return d["value"], d["cpu_baseline"]["cores"], sample
    raise RuntimeError("CPU arm produced no line")


def cpu_baseline_block(args, workload):
    sample = min(args.cpu_sample, CPU_SAMPLE[workload]) if workload != args.workload else args.cpu_sample
    v, cores, ns = cpu_arm(args, workload, sample, 0)
    v1, _, _ = cpu_arm(args, workload, max(1000, sample // 8), 1)
    return {"value": v, "unit": UNIT, "cores": cores, "kind": cpu_arm_kind(),
            "sample": "%d pairs of the same workload, %s, OpenMP over pairs" % (
                ns, "hpp-fcl's own sources (oracle/_ref)" if cpu_arm_kind() == "reference"
                else "oracle (CPU restatement of hpp-fcl)"),
            "single_thread_value": v1}


def run_ours(args):
    import torch
    import hppfcl_b200 as hf

    rank, local, world = env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes one GPU's records; run it with --gpus 1")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hf.build_extension()
    if args.workload == "config5":
        m = measure_config5(args, rank, local, world, dist, args.steps, max(args.warmup, 3))
        if rank == 0:
            line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True,
                    "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                    "config": {"workload": m["name"], "objects": m["n"], "env_scale": m["env_scale"],
                               "l2": "poses, boxes, pairs and records of a step (%d MB) exceed the 126 MB L2" % (
                                   (m["n"] * 150 + int(m["candidate_pairs_per_step"]) * 350) >> 20),
                               "parallelism": "one scene over %d rank(s): every rank sweeps and collides the pairs of its own range of objects" % world},
                    "e2e": m["e2e"], "gpu_launches": m["gpu_launches"], "split_ms_per_step": m["split_ms_per_step"],
                    "candidate_pairs_per_step": m["candidate_pairs_per_step"]}
            if world == 1:
                line["cpu_baseline"] = cpu_config5(args, args.pairs, args.cpu_sample)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    m = measure(args, args.workload, rank, local, world, dist, args.steps, max(args.warmup, 3), clocks=True)
    if rank == 0:
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": m["name"], "pairs_per_gpu": m["n"], "gjk_variant": m["variant"], "l2": m["l2"],
                       "parallelism": "pairs sharded over %d rank(s); results all-gathered per step by the library (hfb_batch_distance_sharded_device: NCCL on the communicator's stream, overlapped with the next step's kernels)" % world},
            "e2e": m["e2e"], "gpu_launches": m["gpu_launches"], "clocks": m.get("clocks"),
            "roofline": m["roofline"], "kernels": m["kernels"],
        }
        for k in ("e2e_pair_rows", "e2e_min_distance_only", "workload_stats", "fp64_view", "watchdog_trips"):
            if k in m:
                line[k] = m[k]
        if world == 1:
            line["cpu_baseline"] = cpu_baseline_block(args, args.workload)
            # the other BASELINE configurations that fit one GPU, at their BASELINE sizes, each with its own
            # value / e2e / roofline / cpu_baseline (fewer steps: they are reported, not the headline)
            others = {}
            for wl in ("config3", "config4"):
                if wl == args.workload:
                    continue
                try:
                    o = measure(args, wl, rank, local, world, dist, 5, 3)
                    o["cpu_baseline"] = cpu_baseline_block(args, wl)
                    o["config"] = {"workload": o.pop("name"), "pairs": o.pop("n"), "gjk_variant": o.pop("variant"), "l2": o.pop("l2")}
                    o.pop("workload", None)
                    o["metric"], o["unit"], o["steps"], o["warmup"] = METRIC, UNIT, 5, 3
                    others[wl] = o
                except Exception as ex:  # a failing side workload must not take the headline line with it
                    others[wl] = {"error": "%s: %s" % (type(ex).__name__, ex)}
            try:  # config 5 at one GPU (its own line at 1 -> 8 GPUs: --workload config5)
                o = measure_config5(args, rank, local, world, dist, 5, 3, n_objects=100_000)
                o["cpu_baseline"] = cpu_config5(args, 100_000, 200_000)
                o["config"] = {"workload": o.pop("name"), "objects": o.pop("n"), "env_scale": o.pop("env_scale")}
                o["metric"], o["unit"], o["steps"], o["warmup"] = METRIC, UNIT, 5, 3
                others["config5"] = o
            except Exception as ex:
                others["config5"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
            line["workloads"] = others
            peak, _ = _peak()
            line["convex_support_kernel"] = support_kernel_roofline(eng_factory=hf.Engine, peak=peak)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
