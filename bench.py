#!/usr/bin/env python
"""bench.py -- flow-rows/s classified per model on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload gnb|logistic|kmeans|forest|forest_hbm|knn|svc]
                    [--impl reference] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

Headline workload (`value`): BASELINE.json configs[1] -- GaussianNB.predict on 1M synthetic 8-feature flow rows
per GPU (weak scaling: every rank classifies its own 1M-row batches; no data-path collective, SURVEY 8e).
A "step" is one pass of the hot path over one batch.  Batches rotate through a ring larger than L2, rows are
float32 and already resident in HBM for `value`; `e2e` goes through the public estimator call with pinned HOST
buffers (H2D rows + D2H labels inside the timed region).  The other models/configs are measured in the same run
and reported under "models" (each with its own roofline and e2e), so the single line carries every model.
`--steps K` is the number of timed steps of every model's device-resident measurement.  `--dump-outputs DIR` writes
the labels of each model's last timed step; inputs and models are seeded, so two builds run with the same arguments
can be compared output for output.
`cpu_baseline` / `--impl reference` time scikit-learn -- the library whose predict() the reference calls at
traffic_classifier.py:106 -- on the box's host cores.
"""
from __future__ import annotations

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
sys.dont_write_bytecode = True   # the bench leaves the tree as it found it (it may be read-only)

L2_BYTES = 126 << 20
# the arithmetic each kernel computes in (a description, not a precision claim: labels are the fp64 definition's everywhere)
DTYPES = {"gnb": "f32 certified pre-pass + f64 re-evaluation of uncertified rows", "linear": "f64", "kmeans": "f64",
          "forest": "f32 compares (exact) + f64 accumulation", "knn": "bf16x3 tensor-core filter + f64 exact re-evaluation",
          "svc": "bf16x3 tensor-core distances + f32 exp/sums with a certificate + f64 re-evaluation of uncertified rows"}
OPTIONS = []   # (key, value) pairs for tcsdn_set_option on every estimator the bench creates (--set-option)
WORKLOADS = ("gnb", "gnb_100m", "logistic", "kmeans", "forest", "forest_hbm", "forest_hbm2", "knn", "svc")
# --dump-outputs keeps at most this many rows' labels per workload: 4 MiB of float32 each, nine workloads stay under 64 MiB
DUMP_ROWS = 1 << 20


# ----------------------------------------------------------------------------- workload definitions
_WORKLOAD_CACHE = {}


def build_workload(name, quick=False):
    if (name, quick) not in _WORKLOAD_CACHE:
        w = _build_workload(name, quick)
        w["name"] = name
        w["full_rows"] = _FULL_ROWS[name]
        _WORKLOAD_CACHE[(name, quick)] = w
    return dict(_WORKLOAD_CACHE[(name, quick)])


_FULL_ROWS = {"gnb": 1_000_000, "gnb_100m": 100_000_000, "logistic": 10_000_000, "kmeans": 10_000_000, "forest": 12_500_000, "forest_hbm": 2_000_000,
              "forest_hbm2": 1_000_000, "knn": 10_000_000, "svc": 10_000_000}


def _build_workload(name, quick=False):
    """-> dict(spec, d, rows (per GPU per step), bytes_per_row, flops_per_row, desc, cpu_sample_rows)"""
    from traffic_classifier_sdn_b200 import synth
    from traffic_classifier_sdn_b200.modelio import spec_from_estimator
    seed = 20260921
    if name == "gnb_100m":   # SURVEY 8(d): the 1M-row step is launch-scale (12 us); the same kernel on a batch that is not
        w = _build_workload("gnb", quick)
        w["rows"] = 100_000_000 if not quick else 10_000_000
        w["desc"] = "GaussianNB predict, 100M synthetic 8-feature flow rows (the headline model on a batch that amortises launch)"
        return w
    if name in ("gnb", "logistic", "kmeans"):
        d = 8 if name == "gnb" else 12
        Xtr, ytr = synth.make_flows(200_000, seed=seed + 1, d=d)
        if name == "gnb":
            from sklearn.naive_bayes import GaussianNB
            sk = GaussianNB().fit(Xtr, ytr)
            desc = "GaussianNB predict, 1M synthetic 8-feature flow rows (BASELINE configs[1])"
            rows = 1_000_000
        elif name == "logistic":
            from sklearn.linear_model import LogisticRegression
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                sk = LogisticRegression(max_iter=100).fit(Xtr, ytr)
            desc = "LogisticRegression predict, 10M synthetic 12-feature flow rows"
            rows = 10_000_000
        else:
            from sklearn.cluster import KMeans
            sk = KMeans(6, n_init=1, random_state=0).fit(Xtr[:50_000])
            desc = "KMeans predict (6 centers), 10M synthetic 12-feature flow rows"
            rows = 10_000_000
        spec = spec_from_estimator(sk)
        C = len(spec["classes"])
        return dict(spec=spec, sk=sk, d=d, rows=rows if not quick else rows // 10, bytes_per_row=4 * d + 4,
                    flops_per_row=(3 * d * C + C) if name == "gnb" else 2 * d * C, desc=desc, bound="hbm",
                    cpu_sample_rows=1_000_000)
    if name == "forest":
        from sklearn.ensemble import RandomForestClassifier
        Xtr, ytr = synth.make_flows(60_000, seed=seed + 4)
        sk = RandomForestClassifier(n_estimators=100, max_depth=16, random_state=0, n_jobs=-1).fit(Xtr.astype(np.float32), ytr)
        spec = spec_from_estimator(sk)
        return dict(spec=spec, sk=sk, d=12, rows=12_500_000 if not quick else 1_000_000, bytes_per_row=52, flops_per_row=0,
                    desc="RandomForestClassifier 100 trees depth<=16 (sklearn-fitted), 12.5M rows per GPU "
                         "(BASELINE configs[4]: 100M rows over 8 GPUs)", bound="hbm", cpu_sample_rows=400_000)
    if name == "forest_hbm":
        spec = synth.random_forest_spec(n_trees=100, depth=16, seed=seed + 5, full=True)
        return dict(spec=spec, sk=None, d=12, rows=2_000_000 if not quick else 200_000, bytes_per_row=52, flops_per_row=0,
                    desc="adversarial forest: 100 complete depth-16 trees (13.1M nodes, 105 MB: L2-resident), 2M rows",
                    bound="hbm", cpu_sample_rows=100_000, visits_per_row=100 * 17.0)
    if name == "forest_hbm2":
        # the regime the "fraction of HBM peak" target is about: the node array (268 MB) does not fit the 126 MB L2
        # (uniform thresholds and uniform rows: every leaf is reached, the walk's working set is the whole array; with
        # flow-shaped rows the same forest is touched on 58 MB only -- ncu r02 -- and stays in L2)
        spec = synth.random_forest_spec(n_trees=256 if not quick else 32, depth=16, seed=seed + 6, full=True, uniform=True)
        return dict(spec=spec, sk=None, d=12, rows=1_000_000 if not quick else 100_000, bytes_per_row=52, flops_per_row=0,
                    desc="adversarial forest, HBM-resident: 256 complete depth-16 trees (33.6M nodes, 268 MB > 126 MB L2), uniform "
                         "thresholds, 1M rows uniform in [0,1)^12 (every leaf reached)",
                    bound="hbm", cpu_sample_rows=20_000, visits_per_row=256 * 17.0, rows_kind="uniform")
    if name == "knn":
        Xtr, ytr = synth.make_flows(50_000, seed=seed + 2)
        spec = dict(kind="knn", fit_X=Xtr, y=ytr.astype(np.int32), k=5, classes=synth.CLASSES, n_features=12)
        return dict(spec=spec, sk=None, d=12, rows=10_000_000 if not quick else 200_000, bytes_per_row=52,
                    flops_per_row=2 * 12 * 50_000, issued_mma_flops_per_row=2 * 80 * 64 * ((50_000 + 63) // 64),
                    desc="KNeighbors k=5 (sklearn's brute-force neighbour votes; the engine prunes far tiles exactly), 10M queries x 50k train rows "
                    "(BASELINE configs[2])", bound="tensor", cpu_sample_rows=20_000)
    if name == "svc":
        # SURVEY 8(d): a real libsvm fit (sklearn.svm.SVC(), defaults: C=1, gamma='scale') on synthetic flows, sized so that
        # about 20k rows become support vectors (29 % of the training rows do on this generator); ~40 s of host time
        from sklearn.svm import SVC
        Xtr, ytr = synth.make_flows(70_000 if not quick else 8_000, seed=seed + 3)
        t0 = time.perf_counter()
        sk = SVC().fit(Xtr, ytr)
        spec = spec_from_estimator(sk)
        nsv, C = len(spec["sv"]), len(spec["classes"])
        nsup = np.asarray(spec["n_support"])
        return dict(spec=spec, sk=sk, d=12, rows=10_000_000 if not quick else 200_000, bytes_per_row=52,
                    flops_per_row=2 * 12 * nsv + 2 * (C - 1) * nsv, exp_per_row=nsv,
                    issued_mma_flops_per_row=2 * 80 * 64 * int(sum((int(c) + 63) // 64 for c in nsup)),   # classes padded to tiles
                    desc=f"SVC(rbf) 10M flows x {nsv} support vectors (sklearn.svm.SVC().fit on {len(Xtr)} synthetic flows, "
                    f"{time.perf_counter() - t0:.0f} s), {C} classes (BASELINE configs[3])", bound="tensor", cpu_sample_rows=4_000)
    raise ValueError(name)


def sklearn_model(w):
    """A live scikit-learn estimator for the workload (the reference arm / cpu_baseline)."""
    if w.get("sk") is not None:
        return w["sk"]
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from sk_rebuild import sklearn_from_spec
    return sklearn_from_spec(w["spec"])


def synth_rows(n, d, seed, device=None, kind="flows"):
    """kind="uniform": n float32 rows uniform in [0, 1)^d (the HBM-resident forest's cache-hostile input).  Otherwise
    n float32 rows: a seeded 1M-row synthetic base resampled with replacement (bootstrap) to n rows.  With a device the
    base rows are derived ON the GPU by the reference's own feature derivation (synth.make_flows_device ->
    tcsdn_flow_update, SURVEY 8d); the host variant is the bit-identical closed form."""
    import torch
    from traffic_classifier_sdn_b200 import synth
    if kind == "uniform":
        g = torch.Generator().manual_seed(seed)
        t = torch.rand((n, d), generator=g, dtype=torch.float32)
        return t.to(device) if device is not None else t
    nb = min(n, 1_000_000)
    if device is not None:
        base = synth.make_flows_device(nb, seed=seed, d=d, dtype="float32", device=device)
        if n <= nb:
            return base
        g = torch.Generator().manual_seed(seed)
        pick = torch.randint(0, nb, (n,), generator=g)
        return base[pick.to(device)].contiguous()
    base = torch.from_numpy(synth.make_flows(nb, seed=seed, d=d, dtype=np.float32, return_labels=False))
    if n <= nb:
        return base
    g = torch.Generator().manual_seed(seed)
    pick = torch.randint(0, nb, (n,), generator=g)
    return base[pick].contiguous()


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 is None or (t0 - 0.05 <= t <= t1 + 0.15)] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- measurement
def ring_size(rows, row_bytes):
    """distinct batches the timed steps rotate through, so that consecutive steps never find their rows in the 126 MiB L2"""
    if rows * row_bytes >= L2_BYTES * 1.25:
        return 1
    return min(12, max(2, int(np.ceil((L2_BYTES * 1.25) / (rows * row_bytes))) + 1))


def make_config(w, world):
    """the `config` object, identical in the b200 and the reference arm (it describes the workload, not the implementation)"""
    ring = ring_size(w["rows"], 4 * w["d"])
    return {"workload": w["desc"], "rows_per_gpu_per_step": w["rows"], "n_features": w["d"],
            "input": "float32 rows: resident in HBM for `value`, in page-locked host memory for `e2e`",
            "parallelism": f"row-sharded x{world}: every rank classifies its own rows with its own model replica, no collective on the "
                           "data path; `value_with_gather` adds the one all-gather of per-shard label vectors (uint8 on the wire)",
            "l2": (f"{ring} distinct batches rotate ({ring * w['rows'] * 4 * w['d'] >> 20} MiB > 126 MiB L2)" if ring > 1 else
                   f"one batch of {w['rows'] * 4 * w['d'] >> 20} MiB > 126 MiB L2")}


def bind_to_gpu_numa_node(index):
    """Pin this process (and so its page-locked staging buffers, first touch) to the NUMA node the GPU hangs off: with
    eight ranks streaming host rows at once, buffers on the far socket cross the inter-socket link and the root complexes
    contend (e2e efficiency 0.81 at N = 8 in round 1).  Returns a short description; silently does nothing when the
    topology is not exposed (containers, single-node hosts)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0"
        node = int(open(os.path.join(path, "numa_node")).read().strip())
        if node < 0:
            return "numa_node=-1 (not exposed)"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        ids &= os.sched_getaffinity(0)
        if not ids:
            return f"node {node}: no allowed cpu"
        os.sched_setaffinity(0, ids)
        return f"node {node} ({len(ids)} cpus)"
    except Exception as exc:
        return f"unavailable ({type(exc).__name__})"


def dist_env():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world, device):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_with_gather(w, steps, world, device):
    """SURVEY 8(e): the N-GPU step WITH the one collective of the path -- every rank classifies its block, then ONE all-gather
    of the per-shard label vectors puts the full vector on every rank (tcsdn_allgather_labels_u8: class indices travel as
    bytes).  predict + gather are enqueued on one stream with no host synchronisation and the K steps are captured into
    ONE CUDA graph, like the gather-free measurement."""
    import torch
    from traffic_classifier_sdn_b200 import from_spec
    from traffic_classifier_sdn_b200.parallel import Communicator
    est = from_spec(w["spec"])
    rows, d = w["rows"], w["d"]
    n_classes = len(w["spec"]["classes"])
    rank = dist_env()[0]
    x = synth_rows(rows, d, seed=4000 + rank, device=device)
    lab = torch.empty(rows, dtype=torch.int32, device=device)
    allv = torch.empty(rows * world, dtype=torch.int32, device=device)
    comm = Communicator()
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):                       # warm-up outside the capture (also sizes the communicator's staging buffer)
            est.predict_indices(x, out=lab)
            comm.allgather_labels(lab, rows, n_classes=n_classes, out=allv)
    torch.cuda.synchronize()
    mode = "cuda-graph"
    graph = None
    try:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(steps):
                est.predict_indices(x, out=lab)
                comm.allgather_labels(lab, rows, n_classes=n_classes, out=allv)
        graph.replay()
        torch.cuda.synchronize()
    except Exception as exc:
        graph, mode = None, f"eager ({type(exc).__name__}: {exc})"
        torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    torch.cuda.synchronize()
    ev0.record()
    if graph is not None:
        graph.replay()
    else:
        for _ in range(steps):
            est.predict_indices(x, out=lab)
            comm.allgather_labels(lab, rows, n_classes=n_classes, out=allv)
    ev1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms = max_over_ranks(ev0.elapsed_time(ev1), world, device)
    ok = bool(torch.equal(allv[rank * rows:(rank + 1) * rows], lab))   # this rank's block of the gathered vector is its own labels
    del graph
    nccl = {"value": rows * world * steps / (ms * 1e-3), "unit": "flow-rows/s", "ms_per_step": ms / steps,
            "gathered_bytes_per_step_per_rank": (1 if n_classes <= 255 else 4) * rows * world, "wire": "uint8" if n_classes <= 255 else "int32",
            "timed_region": mode, "own_block_matches": ok,
            "how": "predict + tcsdn_allgather_labels_u8 (pack, ncclAllGather of bytes, unpack) per step on one stream"}
    # ---- the exchange FUSED into the classification kernel: labels stored straight into every rank's buffer over NVLink
    fused = None
    try:
        comm.gather_buffer(rows)
        with torch.cuda.stream(side):
            for _ in range(3):
                got = comm.predict_gathered(est, x)
        torch.cuda.synchronize()
        barrier(world)
        graph2, mode2 = None, "cuda-graph"
        try:
            graph2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph2, stream=side):
                for _ in range(steps):
                    got = comm.predict_gathered(est, x)
        except Exception as exc:
            graph2, mode2 = None, f"eager ({type(exc).__name__}: {exc})"
            torch.cuda.synchronize()
        barrier(world)
        if graph2 is not None:       # every rank replays the same number of barrier epochs: one untimed replay each
            graph2.replay()
        torch.cuda.synchronize()
        barrier(world)
        ev0.record()
        if graph2 is not None:
            graph2.replay()
        else:
            for _ in range(steps):
                got = comm.predict_gathered(est, x)
        ev1.record()
        torch.cuda.synchronize()
        barrier(world)
        ms2 = max_over_ranks(ev0.elapsed_time(ev1), world, device)
        full = torch.cat([got[r, :rows] for r in range(world)])
        ok2 = bool(torch.equal(full[rank * rows:(rank + 1) * rows].to(torch.int32), est.predict_indices(x)))
        fused = {"value": rows * world * steps / (ms2 * 1e-3), "unit": "flow-rows/s", "ms_per_step": ms2 / steps, "timed_region": mode2,
                 "own_block_matches": ok2, "peer_bytes_stored_per_step_per_rank": rows * world,
                 "how": "tcsdn_predict_gathered: the scoring kernel stores each label byte into all ranks' buffers (CUDA IPC peer "
                        "memory over NVLink), then a peer-memory barrier kernel; no NCCL call in the step"}
        del graph2
    except Exception as exc:
        fused = {"error": f"{type(exc).__name__}: {exc}"}
    comm.close()
    best = fused if fused and fused.get("value", 0) > nccl["value"] else nccl
    return dict(best, nccl_allgather=nccl, fused_peer_memory=fused)


def dump_sample(rows):
    """Row indices --dump-outputs keeps of a `rows`-row step: None (all of them) up to DUMP_ROWS, else a fixed, seeded,
    sorted sample of DUMP_ROWS rows (the same rows on every run with the same arguments)."""
    if rows <= DUMP_ROWS:
        return None
    return np.sort(np.random.default_rng(0).choice(rows, DUMP_ROWS, replace=False))


def measure_gpu(w, steps, warmup, world, device, peaks, extras_light=False, clock_probe_s=0.0, keep_labels=False):
    """Device-resident timing (`value`) + end-to-end timing (`e2e`) of one workload on this rank.  keep_labels: also
    return the label indices of the last timed step (the rows dump_sample picks) as float32, for --dump-outputs."""
    import torch
    from traffic_classifier_sdn_b200 import from_spec
    est = from_spec(w["spec"])
    for key, val in OPTIONS:          # --set-option K=V (tuning sweeps; defaults are the measured best)
        est.set_option(key, val)
    rows, d = w["rows"], w["d"]
    row_bytes = 4 * d
    ring = ring_size(rows, row_bytes)
    rank = dist_env()[0]
    batches = [synth_rows(rows, d, seed=1000 + 17 * rank + i, device=device, kind=w.get("rows_kind", "flows")) for i in range(ring)]
    torch.cuda.synchronize()
    lab_dev = torch.empty(rows, dtype=torch.int32, device=device)
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(warmup):
            est.predict_indices(batches[i % ring], out=lab_dev)
        est.sync_check()
    launches_per_step = int(est.stats()[0])
    torch.cuda.current_stream().wait_stream(side)
    # the K timed steps are captured once into a CUDA graph (1M-row steps last microseconds: eager launches
    # would time the Python interpreter, not the GPU); replay = K back-to-back passes over the batch ring
    graph, mode = None, "cuda-graph"
    try:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(steps):
                est.predict_indices(batches[i % ring], out=lab_dev)
        graph.replay()   # one untimed replay (graph upload)
        torch.cuda.synchronize()
    except Exception as exc:
        graph, mode = None, f"eager ({type(exc).__name__})"
        torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    torch.cuda.synchronize()
    try:
        # a short busy-wait kernel goes first, so that the replay below is already queued on the device when the first
        # event fires: the timed region then holds K steps of GPU work, not the host's graph-launch latency (which would
        # otherwise weigh on a K = 5 run of 10 us steps far more than on a K = 20 run)
        torch.cuda._sleep(400_000)
    except Exception:
        pass
    ev0.record()
    if graph is not None:
        graph.replay()
    else:
        for i in range(steps):
            est.predict_indices(batches[i % ring], out=lab_dev)
    ev1.record()
    torch.cuda.synchronize()
    barrier(world)
    est.sync_check()
    ms = ev0.elapsed_time(ev1)
    kernel_ms = ms / steps
    labels = None
    if keep_labels:   # lab_dev still holds the last timed step's result (batch (steps - 1) % ring)
        pick = dump_sample(rows)
        kept = lab_dev if pick is None else lab_dev[torch.from_numpy(pick).to(device)]
        labels = kept.cpu().numpy().astype(np.float32)
    # keep the very same work running for ~1.5 s so that nvidia-smi (100 ms period) sees the clocks under this load
    load_window = None
    if clock_probe_s > 0:
        t_a = time.time()
        while time.time() - t_a < clock_probe_s:
            if graph is not None:
                graph.replay()
            else:
                for i in range(steps):
                    est.predict_indices(batches[i % ring], out=lab_dev)
            torch.cuda.synchronize()
        load_window = (t_a, time.time())
    ms = max_over_ranks(ms, world, device)
    value = rows * world * steps / (ms * 1e-3)

    # end to end through the PUBLIC call a user of the reference makes -- labels = model.predict(X) on host rows
    # (traffic_classifier.py:106): H2D of the rows, kernels, D2H of the class indices and classes_.take (the labels are
    # materialised as the estimator's classes_ dtype, exactly what the sklearn arm pays for too) inside the timed region.
    # Three variants: rows in page-locked memory (the headline `value`), the same through predict_indices with a
    # page-locked int32 result buffer (no label materialisation: what a pipeline that keeps indices would see), and
    # rows in ordinary pageable memory.
    e2e_steps = max(3, min(steps, 10)) if not extras_light else 3
    host = [torch.empty((rows, d), dtype=torch.float32).pin_memory() for _ in range(min(ring, 3))]
    for h, b in zip(host, batches):
        h.copy_(b)
    host_np = [h.numpy() for h in host]
    lab_host = torch.empty(rows, dtype=torch.int32).pin_memory().numpy()   # page-locked result buffer (out=)

    def timed(fn, n_steps):
        fn(0)                                  # untimed first call (allocations, page faults of result arrays)
        barrier(world)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n_steps):
            out = fn(i)
        dt = max_over_ranks(time.perf_counter() - t0, world, device)
        assert out.shape == (rows,)
        return rows * world * n_steps / dt

    e2e_predict = timed(lambda i: est.predict(host_np[i % len(host_np)]), e2e_steps)
    e2e_indices = timed(lambda i: est.predict_indices(host_np[i % len(host_np)], out=lab_host), e2e_steps)
    pageable = np.array(host_np[0], copy=True)                            # ordinary (pageable) memory
    e2e_pageable = timed(lambda i: est.predict(pageable), max(2, e2e_steps // 2))
    del pageable
    e2e = e2e_predict

    peak = peaks["hbm_gbs"] if w["bound"] == "hbm" else peaks["bf16_tflops"]
    if w["bound"] == "hbm":
        achieved = rows * w["bytes_per_row"] / (kernel_ms * 1e-3) / 1e9
        unit = "GB/s"
    else:
        achieved = rows * w["flops_per_row"] / (kernel_ms * 1e-3) / 1e12
        unit = "TFLOP/s"
    copy_at_size = None
    if w["bound"] == "hbm" and rows * w["bytes_per_row"] < (1 << 30) and not extras_light:
        # context for a launch-scale step: what a plain device copy moving the SAME number of bytes per step reaches when it is
        # timed the same way (K copies in one CUDA graph, rotating through buffers larger than L2) -- the measured-peak
        # denominator comes from a 2 GB copy, which amortises the launch; a 36 MB step cannot
        try:
            half = rows * w["bytes_per_row"] // 2
            nbuf = max(2, int(np.ceil(L2_BYTES * 1.25 / (2 * half))) + 1)
            src = [torch.empty(half, dtype=torch.uint8, device=device) for _ in range(nbuf)]
            dst = [torch.empty(half, dtype=torch.uint8, device=device) for _ in range(nbuf)]
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(3):
                    dst[i % nbuf].copy_(src[i % nbuf])
            torch.cuda.synchronize()
            gcopy = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gcopy, stream=side):
                for i in range(steps):
                    dst[i % nbuf].copy_(src[i % nbuf])
            gcopy.replay()
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(); gcopy.replay(); c1.record()
            torch.cuda.synchronize()
            us = c0.elapsed_time(c1) / steps * 1e3
            copy_at_size = {"bytes_per_step": 2 * half, "us_per_step": us, "gbs": 2 * half / (us * 1e-6) / 1e9,
                            "how": "torch copy_ of the same bytes per step, K copies in one CUDA graph"}
            del gcopy, src, dst
        except Exception as exc:
            copy_at_size = {"error": f"{type(exc).__name__}: {exc}"}
    tr = load_traffic(w["name"])
    if tr is not None:
        # the capture was taken on the full-size workload; scale if this run uses another batch size (--quick)
        tr = dict(tr, bytes=tr["bytes"] * rows / w["full_rows"])
    roofline = dict(bound=w["bound"], achieved=achieved, peak=peak, unit=unit, frac=achieved / peak,
                    traffic=None if tr is None else tr["bytes"], traffic_source=None if tr is None else tr["source"],
                    peak_source=peaks["source"])
    if copy_at_size is not None:
        roofline["copy_at_this_size"] = copy_at_size
        if "gbs" in copy_at_size:
            roofline["frac_of_copy_at_this_size"] = achieved / copy_at_size["gbs"]
    if w["bound"] == "tensor":
        # SURVEY 8(d): next to the algorithmic flops, the flops the tensor cores are actually ISSUED (bf16 x 3 split:
        # K = 80 per pair instead of d = 12, reference rows padded to 64-row tiles) and the ncu tensor-pipe figure
        issued_per_row = w["issued_mma_flops_per_row"]
        if w["name"] == "knn":
            # the engine leaves out the reference tiles that are too far for all 512 rows of a pass (exact: DESIGN 4): what the
            # tensor cores are issued is the tiles actually multiplied (the engine's own counter), `achieved` stays the
            # brute-force-equivalent rate (every pair counted, as sklearn's brute force computes them)
            st = est.stats()
            n_tiles = (50_000 + 63) // 64
            tiles = st[4] / 1000.0 if st[4] > 0 else float(n_tiles)
            issued_per_row = 2 * 80 * 64 * tiles
            roofline.update(tiles_multiplied_per_pass=tiles, tiles_total=n_tiles,
                            achieved_is="brute-force-equivalent flops (all 10M x 50k pairs) per second; issued_mma counts the tiles actually multiplied",
                            tie_rows_rerun_in_index_order=int(st[7]))
        issued = rows * issued_per_row / (kernel_ms * 1e-3) / 1e12
        roofline.update(issued_mma=issued, issued_mma_frac=issued / peak, tensor_pipe_pct_ncu=load_summary_field(w["name"], "tensor_pipe_pct"))
        if w.get("exp_per_row"):
            # SVC is bound by the MUFU unit, not the tensor pipe (SURVEY 8d): one ex2 per (row, support vector) pair against
            # 16 lanes/clk/SM (measured, tools/tmem_probe.cu) x 148 SMs x the SM clock
            exp_s = rows * w["exp_per_row"] / (kernel_ms * 1e-3)
            exp_peak = 16.0 * 148 * (peaks.get("sm_max_mhz") or 1965.0) * 1e6
            roofline.update(exp_per_s=exp_s, exp_peak=exp_peak, exp_frac=exp_s / exp_peak, xu_pipe_pct_ncu=load_summary_field(w["name"], "xu_pipe_pct"))
    return dict(value=value, ms_per_step=ms / steps, kernel_ms=kernel_ms, rows=rows, ring=ring, mode=mode, traffic=tr,
                launches_per_step=launches_per_step, load_window=load_window,
                e2e=dict(value=e2e, unit="flow-rows/s", h2d_bytes_per_step=rows * row_bytes, d2h_bytes_per_step=rows * 4,
                         call="estimator.predict(X): float32 rows in page-locked host memory -> numpy labels (classes_.take included)",
                         indices_value=e2e_indices, indices_call="estimator.predict_indices(X, out=page-locked int32): no label materialisation",
                         pageable_value=e2e_pageable, pageable_call="estimator.predict(X) on rows in pageable host memory",
                         bound="PCIe: host rows cross at ~48-55 GB/s per GPU; the streaming models' kernels are 50-100x faster than the copy"),
                roofline=roofline, est=est, batch0=batches[0], labels=labels)


def _threadpools():
    try:
        from threadpoolctl import threadpool_info
        return [{k: p.get(k) for k in ("user_api", "internal_api", "num_threads", "version")} for p in threadpool_info()]
    except Exception as exc:
        return [{"error": f"{type(exc).__name__}: {exc}"}]


class _SvcPool:
    """SVC.predict row-chunked over a pool of worker processes: libsvm's predict is one serial loop over the rows
    (sk:svm/src/libsvm/libsvm_helper.c:315-332), so all-core scikit-learn means one chunk per worker.  The pool is created
    once (workers and their copy of the model stay alive across calls, like a serving process would keep them)."""

    def __init__(self, sk, jobs):
        from joblib import Parallel
        self.sk, self.jobs = sk, jobs
        self.par = Parallel(n_jobs=jobs, backend="loky")
        self.par.__enter__()

    def predict(self, X):
        from joblib import delayed
        parts = self.par(delayed(self.sk.predict)(c) for c in np.array_split(X, self.jobs) if len(c))
        return np.concatenate(parts)

    def close(self):
        self.par.__exit__(None, None, None)
        # joblib keeps loky's workers alive for reuse after the Parallel block: stop them, so none outlives the bench
        from joblib.externals.loky import get_reusable_executor
        get_reusable_executor(reuse=True).shutdown(wait=True)


def cpu_reference(w, max_seconds=20.0, steps=2, warmup=1):
    """scikit-learn predict on the host cores, on a bounded sample of the workload's rows -- two columns (BASELINE.md 3):
    `as_shipped`: the estimator exactly as the reference's notebooks construct it (defaults: KNN kd_tree with n_jobs=None,
    RandomForest n_jobs=None, SVC's single-threaded libsvm loop); `value`: best effort on all cores (n_jobs=-1 for
    RandomForest and KNN, KNN algorithm='brute' = the work the GPU does, SVC row-chunked over a process pool).
    `warmup` untimed calls, then `steps` timed calls; rows/s = rows * steps / time."""
    import warnings
    kind = w["spec"]["kind"]
    sk = sklearn_model(w)
    n = min(w["cpu_sample_rows"], w["rows"])
    X = synth_rows(n, w["d"], seed=1000, kind=w.get("rows_kind", "flows")).numpy()
    if kind != "forest":
        X = X.astype(np.float64)   # sklearn validates these estimators to float64 anyway
    cores = os.cpu_count() or 1
    jobs = min(cores, 64)

    def run(predict, Xs, budget):
        """-> (rows/s, rows used): sample shrunk so that warmup + steps calls fit the time budget"""
        t0 = time.perf_counter()
        predict(Xs[: max(1, len(Xs) // 20)])
        probe = (time.perf_counter() - t0) * 20
        m = len(Xs)
        if probe * (steps + warmup) > budget:
            m = max(64, int(m * budget / (probe * (steps + warmup))))
        Xs = Xs[:m]
        for _ in range(warmup):
            predict(Xs)
        t0 = time.perf_counter()
        for _ in range(steps):
            predict(Xs)
        return m * steps / (time.perf_counter() - t0), m

    out = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        # ---- as shipped
        shipped = sk
        note = "defaults"
        if kind == "knn":
            from sklearn.neighbors import KNeighborsClassifier
            shipped = KNeighborsClassifier(int(w["spec"]["k"])).fit(w["spec"]["fit_X"], w["spec"]["y"])   # algorithm='auto' -> kd_tree
            note = f"algorithm='auto' -> {shipped._fit_method}, n_jobs=None"
        elif kind == "forest":
            sk.n_jobs = None
            note = "n_jobs=None"
        elif kind == "svc":
            note = "single-threaded libsvm loop"
        v_shipped, m_shipped = run(shipped.predict, X, max_seconds * 0.4)
        # ---- all cores, best effort
        if kind == "knn":
            from sklearn.neighbors import KNeighborsClassifier
            allc = KNeighborsClassifier(int(w["spec"]["k"]), algorithm="brute", n_jobs=-1).fit(w["spec"]["fit_X"], w["spec"]["y"])
            v_all, m_all = run(allc.predict, X, max_seconds * 0.6)
            how = "algorithm='brute' (the GPU's work), n_jobs=-1"
        elif kind == "forest":
            sk.n_jobs = -1
            v_all, m_all = run(sk.predict, X, max_seconds * 0.6)
            how = "n_jobs=-1"
        elif kind == "svc":
            try:
                pool = _SvcPool(sk, jobs)
                Xp = synth_rows(min(w["rows"], max(n, jobs * 300)), w["d"], seed=1000).numpy().astype(np.float64)
                pool.predict(Xp[: jobs * 4])                      # spawn the workers outside the timed calls
                v_all, m_all = run(pool.predict, Xp, max(max_seconds * 0.6, 25.0))
                pool.close()
                how = f"rows chunked over a pool of {jobs} worker processes (joblib/loky, workers kept alive across calls)"
            except Exception as exc:
                v_all, m_all, how = v_shipped, m_shipped, f"process pool failed ({type(exc).__name__}: {exc}); single thread"
        else:
            v_all, m_all, how = v_shipped, m_shipped, "same call (numpy/OpenBLAS/OpenMP use the threads they use: see threadpools)"
    best, m_best = (v_all, m_all) if v_all >= v_shipped else (v_shipped, m_shipped)
    out = dict(value=best, unit="flow-rows/s", cores=cores, kind="reference",
               sample=f"sklearn {type(sk).__name__}.predict on {m_best} of the workload's rows, {warmup} warm-up + {steps} timed calls; "
                      f"all-core column: {how}",
               as_shipped=dict(value=v_shipped, rows=m_shipped, how=note), all_cores=dict(value=v_all, rows=m_all, how=how),
               threadpools=_threadpools())
    if kind == "forest":
        # SURVEY 8(d): the traversal accounting needs the MEASURED mean number of node visits per row (V-bar)
        try:
            m = min(n, 2000)
            out["node_visits_per_row"] = float(sk.decision_path(X[:m])[0].nnz) / m
        except Exception as exc:
            out["node_visits_per_row"] = None
            out["node_visits_error"] = f"{type(exc).__name__}: {exc}"
    return out


def per_row_call_pattern(w, est, seconds=1.0):
    """The reference's literal call pattern (traffic_classifier.py:103-106): model.predict([[12 floats]]) once per flow.
    Calls per second of scikit-learn's estimator and of this package's estimator (one-row host call: H2D, kernel, D2H)."""
    import warnings
    rows = synth_rows(256, w["d"], seed=77).numpy().astype(np.float64).tolist()
    out = {"what": "model.predict([[d floats]]) once per flow, as traffic_classifier.py:103-106 does"}
    for name, model in (("sklearn_calls_per_s", sklearn_model(w)), ("gpu_calls_per_s", est)):
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model.predict([rows[0]])
                t0, k = time.perf_counter(), 0
                while time.perf_counter() - t0 < seconds:
                    model.predict([rows[k % len(rows)]])
                    k += 1
                out[name] = k / (time.perf_counter() - t0)
        except Exception as exc:
            out[name] = f"{type(exc).__name__}: {exc}"
    return out


def load_traffic(name):
    """DRAM bytes per launch of the workload's dominant kernel, from the committed ncu capture (profiles/)."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    if os.path.isdir(pdir):
        for f in sorted(os.listdir(pdir)):
            if f.endswith("_ncu_summary.json"):
                j = json.load(open(os.path.join(pdir, f)))
                if name in j and j[name].get("dram_bytes"):
                    best = {"bytes": j[name]["dram_bytes"], "source": f"profiles/{f}"}
    return best


def load_summary_field(name, field):
    """Latest committed ncu summary's value of `field` for the workload (profiles/*_ncu_summary.json), or None."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    if os.path.isdir(pdir):
        for f in sorted(os.listdir(pdir)):
            if f.endswith("_ncu_summary.json"):
                j = json.load(open(os.path.join(pdir, f)))
                if name in j and j[name].get(field) is not None:
                    best = j[name][field]
    return best


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=float(j["hbm_gbs"]), bf16_tflops=float(j.get("bf16_tflops", 1590.0)), sm_max_mhz=float(j.get("sm_max_mhz", 1965.0)),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="gnb", choices=WORKLOADS)
    ap.add_argument("--no-extras", action="store_true", help="measure only the headline workload")
    ap.add_argument("--extras", default="gnb_100m,logistic,kmeans,forest,forest_hbm,forest_hbm2,knn,svc")
    ap.add_argument("--quick", action="store_true", help="10x smaller batches (debugging)")
    ap.add_argument("--gpu-only", action="store_true", help="skip the scikit-learn baselines (tuning sweeps)")
    ap.add_argument("--set-option", action="append", default=[], metavar="KEY=VALUE",
                    help="tcsdn_set_option on every estimator (include/tcsdn.h TCSDN_OPT_*), e.g. 4=3")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the label indices each workload's last timed step computed as "
                         "DIR/<workload>_labels.npy (float32; a fixed, seeded sample of 1Mi rows where a step has more)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    for kv in args.set_option:
        OPTIONS.append((int(kv.split("=")[0]), int(kv.split("=")[1])))
    args.warmup = max(args.warmup, 3)
    rank, world, local = dist_env()
    peaks = load_peaks()

    if args.impl == "reference":
        if rank != 0:
            return 0
        w = build_workload(args.workload, args.quick)
        t0 = time.perf_counter()
        res = cpu_reference(w, max_seconds=90.0, steps=args.steps, warmup=args.warmup)
        wall = time.perf_counter() - t0
        line = {"impl": "reference", "metric": "flow-rows/sec classified (GaussianNB, 1M x 8 synthetic flow rows per GPU)"
                if args.workload == "gnb" else f"flow-rows/sec classified ({args.workload})",
                "value": res["value"], "unit": "flow-rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * w["rows"] / res["value"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": make_config(w, args.gpus),
                "cpu_baseline": res,
                "e2e": {"value": res["value"], "unit": "flow-rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "wall_s": wall}
        print(json.dumps(line))
        return 0

    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: bench.py measures the GPU path and has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    w = build_workload(args.workload, args.quick)
    sampler = ClockSampler(local)
    sampler.start()
    dump = bool(args.dump_outputs) and rank == 0
    outputs = {}
    head = measure_gpu(w, args.steps, args.warmup, world, device, peaks, clock_probe_s=1.5, keep_labels=dump)
    outputs[args.workload] = head["labels"]
    clocks = sampler.stop(*head["load_window"])
    clocks["how"] = "nvidia-smi -lms 100 over a 1.5 s continuation of the timed CUDA graph (same kernels, same batches)"

    models = {}
    if not args.no_extras:
        for name in [x for x in args.extras.split(",") if x and x != args.workload]:
            try:
                wx = build_workload(name, args.quick)
                r = measure_gpu(wx, args.steps, 3, world, device, peaks, extras_light=True, keep_labels=dump)
                outputs[name] = r["labels"]
                entry = {"workload": wx["desc"], "dtype": DTYPES.get(wx["spec"]["kind"]), "value": r["value"], "unit": "flow-rows/s", "rows_per_gpu_per_step": r["rows"],
                         "ms_per_step": r["ms_per_step"], "e2e": r["e2e"], "roofline": r["roofline"],
                         "gpu_launches_per_step": r["launches_per_step"], "engine_stats": r["est"].stats().tolist(),
                         "timed_region": r["mode"]}
                if rank == 0 and world == 1 and not args.gpu_only:
                    entry["cpu_baseline"] = cpu_reference(wx, max_seconds=8.0)
                vbar = (entry.get("cpu_baseline") or {}).get("node_visits_per_row") or wx.get("visits_per_row")
                if vbar and wx["spec"]["kind"] == "forest":   # rows/s x (52 + 8 V-bar) next to the compulsory-bytes figure
                    tb = r["value"] * (wx["bytes_per_row"] + 8.0 * vbar) / 1e9
                    entry["roofline"].update(traversal_bytes_per_row=wx["bytes_per_row"] + 8.0 * vbar, traversal_achieved=tb,
                                             traversal_frac=tb / peaks["hbm_gbs"])
                models[name] = entry
                del r
                torch.cuda.empty_cache()
            except Exception as exc:  # keep the headline line even if a secondary workload fails
                models[name] = {"error": f"{type(exc).__name__}: {exc}"}

    cpu = cpu_reference(w, max_seconds=15.0) if (rank == 0 and world == 1 and not args.gpu_only) else None
    call_pattern = per_row_call_pattern(w, head["est"]) if (rank == 0 and world == 1 and not args.gpu_only) else None
    gathered = None
    if world > 1:
        try:
            gathered = measure_with_gather(w, args.steps, world, device)
        except Exception as exc:   # the headline line must survive a failure of this extra
            gathered = {"error": f"{type(exc).__name__}: {exc}"}
    if rank == 0:
        line = {"metric": "flow-rows/sec classified (GaussianNB, 1M x 8 synthetic flow rows per GPU)"
                if args.workload == "gnb" else f"flow-rows/sec classified ({args.workload})",
                "value": head["value"], "unit": "flow-rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPES.get(w["spec"]["kind"], "f64"), "data": "synthetic",
                "config": make_config(w, world), "timed_region": head["mode"], "numa_binding": numa,
                "e2e": head["e2e"], "gpu_launches": head["launches_per_step"] * args.steps,
                "roofline": head["roofline"], "kernel_ms": head["kernel_ms"], "clocks": clocks, "models": models}
        vbar = (cpu or {}).get("node_visits_per_row") or w.get("visits_per_row")
        if vbar and w["spec"]["kind"] == "forest":
            tb = head["value"] / world * (w["bytes_per_row"] + 8.0 * vbar) / 1e9
            line["roofline"].update(traversal_bytes_per_row=w["bytes_per_row"] + 8.0 * vbar, traversal_achieved=tb, traversal_frac=tb / peaks["hbm_gbs"])
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if call_pattern is not None:
            line["reference_call_pattern"] = call_pattern
        if gathered is not None:
            # first-class: the same job with the path's one collective, and how much of the gather-free rate it keeps
            line["with_label_allgather"] = gathered
            if "value" in gathered:
                line["value_with_gather"] = gathered["value"]
                line["gather_efficiency"] = gathered["value"] / head["value"]
        if dump:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, labels in outputs.items():
                if labels is not None:
                    np.save(os.path.join(args.dump_outputs, f"{name}_labels.npy"), labels)
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
