#!/usr/bin/env python3
"""bench.py — shared_tree build throughput (Gbp/s) on B200, BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--bases 3100000000] [--repeat-permille 500] [--seed 42] [--dump-outputs DIR]

A "step" is one full shared_tree build (pack + canonicalise + hash-cons every level, ids
final) of the synthetic genome-shaped sequence of BASELINE.json config 3 (`--bases`
random ACGT + planted repeats, DESIGN.md §6).  `value` = bases / device time with the
ASCII body already resident in HBM; `e2e` = the same build through the public C-ABI call
with the text in pinned HOST memory (H2D inside the timed region, result counters read
back).  One JSON line on stdout.

--impl reference times the reference's own CPU build (oracle/_ref when it was compiled,
else the oracle port) on a bounded sample of the same workload.

--dump-outputs DIR writes the tree of the last timed build as DIR/*.npy (see dump_outputs), so that two
builds of the project can be compared output for output on the same seeded input.  With N > 1 GPUs it is the
tree rank 0 gathers from one more sharded build of the same input after the timed steps (builds are
deterministic, so it equals the last timed one).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree may be read-only; nothing is cached in it

DNA = 12
METRIC = "shared_tree_build_gbp_per_s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bases", type=int, default=3_100_000_000)
    ap.add_argument("--repeat-permille", type=int, default=500)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--cpu-sample-bases", type=int, default=0, help="0 = auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="skip sort/serialize/decode/random-access timings")
    ap.add_argument("--option", action="append", default=[], metavar="NAME=VALUE",
                    help="stb_set_option on the build handle (experiments; the defaults are what is reported)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the tree of the last timed build to DIR/*.npy (float64, a seeded sample of the large tables); "
                         "with N > 1 GPUs, rank 0's gathered tree of one more build of the same input")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU build computed; --impl reference has no such output")
    return args


def workload_config(args, extra=None):
    cfg = {
        "workload": "config 3: synthetic human-genome-shaped sequence, random ACGT + planted repeats, one shared_tree build",
        "bases": args.bases, "dna_size": DNA, "repeat_permille": args.repeat_permille, "seed": args.seed,
        "repeat_lengths": "300*2^k+r, k in 0..9, capped at 200000",
        "repeat_alignment": "4/8 forward at a multiple of 12*1024 bases, 1/8 reverse-complement aligned, 3/8 arbitrary",
        "l2_policy": "inputs (>= 1 B/base of text + multi-GB tables) are far larger than the 126 MB L2",
    }
    if extra:
        cfg.update(extra)
    return cfg


# ---------------------------------------------------------------------------- clocks
def nvml_handle(index):
    """NVML handle of CUDA device `index` of this process (matched by UUID: NVML's own numbering
    ignores CUDA_VISIBLE_DEVICES)."""
    import pynvml
    import torch
    pynvml.nvmlInit()
    uuid = str(torch.cuda.get_device_properties(index).uuid)
    if not uuid.startswith("GPU-"):
        uuid = "GPU-" + uuid
    return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid)


class ClockSampler:
    """SM clock and throttle reasons while the timed region runs: NVML polled every few
    milliseconds from a thread (the timed region of a multi-GPU run lasts tens of milliseconds,
    too short for an nvidia-smi loop); `nvidia-smi -lms` only when NVML cannot be loaded."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0, period_s=0.004):
        self.index, self.period = index, period_s
        self.proc = self.nvml = None
        self.lines, self.sm, self.reason_bits = [], [], 0
        self.stop_flag = threading.Event()

    def start(self):
        try:
            self.nvml, self.handle = nvml_handle(self.index)
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            time.sleep(self.period)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            n, bits = self.nvml, self.reason_bits
            flags = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz, "samples": len(self.sm),
                    "reasons": sorted(k for k, v in flags.items() if bits & v), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(self.NAMES, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def bind_to_gpu_numa_node(index):
    """One process per GPU: run (and first-touch pinned host buffers) on the cores NVML reports as
    local to the GPU, so that the host-to-device copies of the e2e figure do not cross sockets."""
    try:
        pynvml, handle = nvml_handle(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, mask in enumerate(words) for b in range(64) if (int(mask) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ---------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_build_once(text: bytes):
    """Times one CPU build of `text` with the unmodified reference when it is available
    (oracle/_ref/libref.so: shared_tree{path}, i.e. loader thread + build thread exactly as
    ./compress runs it), else with the oracle port.  Returns (seconds, kind, cores)."""
    from oracle import pyoracle
    if pyoracle.have_ref():
        ref = pyoracle.Ref()
        with tempfile.NamedTemporaryFile(suffix=".fa", delete=False) as f:
            f.write(text)
            path = f.name
        try:
            t0 = time.perf_counter()
            tree = ref.build_file(path, DNA)
            dt = time.perf_counter() - t0
            assert tree.width() == len(text) // DNA
        finally:
            os.unlink(path)
        return dt, "reference", 2  # one build thread + one loader thread (NullMutex hash maps)
    orc = pyoracle.Oracle()
    t0 = time.perf_counter()
    leaves = orc.fasta_to_leaves(text, DNA)
    orc.build(leaves, DNA)
    return time.perf_counter() - t0, "port", 1


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle
    orc = pyoracle.Oracle()
    sample = args.cpu_sample_bases or 24_000_000
    sample = min(sample, args.bases)
    text = orc.synth(args.bases, args.seed, args.repeat_permille, first=0, count=sample).tobytes()
    for _ in range(args.warmup):
        cpu_build_once(text[: max(DNA * 1024, sample // 16)])
    times = []
    kind, cores = "port", 1
    for _ in range(args.steps):
        dt, kind, cores = cpu_build_once(text)
        times.append(dt)
    total = sum(times)
    value = sample * len(times) / total / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, {"sample": f"first {sample} bases of the {args.bases}-base sequence per step"}),
        "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": cores, "kind": kind,
                         "sample": f"first {sample} bases, {len(times)} timed builds", "host_cpus": os.cpu_count(),
                         # the reference's build of the WHOLE workload, timed once when the golden was made (not on this box)
                         "full_size": full_size_reference(golden_record(args))},
        "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------- reference goldens
def golden_record(args, variant="plain"):
    """What the UNMODIFIED reference produced for this exact workload (tests/golden/synth.json, written by
    oracle/gen_golden_synth.py in the build container), or None when the workload has no golden."""
    path = ROOT / "tests" / "golden" / "synth.json"
    if not path.exists():
        return None
    for name, rec in json.loads(path.read_text()).items():
        if (rec["bases"], rec["seed"], rec["repeat_permille"], rec["variant"], rec["dna_size"]) == (
                args.bases, args.seed, args.repeat_permille, variant, DNA):
            return dict(rec, name=name)
    return None


def full_size_reference(gold):
    """The reference's own build of the WHOLE workload (not a sample), timed once when the golden was made."""
    if not gold or "reference_timing" not in gold:
        return None
    rt = gold["reference_timing"]
    return {"value": rt["gbp_per_s"], "unit": "Gbp/s", "construct_s": rt["construct_s"], "sort_s": rt["sort_s"], "threads": rt["threads"],
            "host": rt["host"], "how": rt["how"], "source": "tests/golden/synth.json (oracle/gen_golden_synth.py)"}


def check_against_golden(rec, what, got, want):
    if got != want:
        raise SystemExit(f"bench.py: {what} differs from the reference's ({rec['name']} in tests/golden/synth.json): "
                         f"got {got}, the reference has {want}")


def sha256_of_device_bytes(t, nbytes):
    import hashlib
    return hashlib.sha256(t[:nbytes].cpu().numpy().tobytes()).hexdigest()


# ---------------------------------------------------------------------------- --dump-outputs
DUMP_ROWS = 1 << 20  # rows of leaves.npy and of nodes.npy at most: 16 + 32 MiB in float64


def _sample(n: int, k: int, seed):
    """Sorted positions of `k` rows out of `n` (all of them when n <= k), a fixed function of (n, k, seed)."""
    import numpy as np
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))


def dump_outputs(tree, out_dir: Path, seed: int):
    """What a build hands its caller, as float64 arrays (every value is below 2^53, so each is exact):
    counts.npy        width, depth, leaf_count, node_count, root pointer
    layer_counts.npy  nodes per layer, bottom-up
    leaves.npy        (position, leaf word) rows of the leaf table
    nodes.npy         (layer, position, left pointer, right pointer) rows of the node layers
    Tables longer than DUMP_ROWS are sampled at seeded positions: the leaf table as a whole, the node layers
    with an equal share each so that the short top layers are always complete."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    counts = tree.layer_counts()
    leaves = tree.leaves()
    pos = _sample(len(leaves), DUMP_ROWS, [seed, 0])
    leaf_rows = np.stack([pos.astype(np.float64), leaves[pos].astype(np.float64)], axis=1)
    assert len(leaves) == 0 or int(leaves[pos].max()) < (1 << 53), "leaf words wider than a float64 mantissa"
    del leaves
    node_rows, share = [], DUMP_ROWS // max(1, len(counts))
    for k in range(len(counts)):
        layer = tree.layer(k)
        pos = _sample(len(layer), share, [seed, 1, k])
        node_rows.append(np.concatenate([np.full((len(pos), 1), k, np.float64), pos[:, None].astype(np.float64),
                                         layer[pos].astype(np.float64)], axis=1))
        del layer
    arrays = {
        "counts": np.array([tree.width(), tree.depth(), tree.leaf_count(), tree.node_count(), tree.root()], dtype=np.float64),
        "layer_counts": np.array(counts, dtype=np.float64),
        "leaves": leaf_rows,
        "nodes": np.concatenate(node_rows) if node_rows else np.zeros((0, 4), np.float64),
    }
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


# ---------------------------------------------------------------------------- algorithmic bytes
def algorithmic_bytes(n0: int, leaf_unique: int, layer_unique: list[int]):
    """Compulsory HBM bytes per kernel class for one build (DESIGN.md §4): streams only;
    hash-table probes are reported separately as non-compulsory traffic."""
    levels = [n0]
    while levels[-1] > 1 or len(levels) == 1:
        levels.append((levels[-1] + 1) // 2)
    node_pos = levels[1:]
    uniq = [leaf_unique] + list(layer_unique)
    pos = [n0] + node_pos
    node_level = [4 * a + 4 * b + b // 8 for a, b in zip(levels[:-1], levels[1:])]
    resolve_level = [p // 8 + 8 * (p - u) for p, u in zip(pos, uniq)]
    out = {
        "leaf_insert": n0 * DNA + 4 * n0 + n0 // 8,
        "node_insert": sum(node_level),
        "assign_ids": sum(p // 8 + 16 * u for p, u in zip(pos, uniq)),
        "resolve_ids": sum(resolve_level),
    }
    out["build_total"] = sum(out.values())
    # the first node layer is deduplicated on chip (csrc/bucket.cu: two partition passes + one dedup kernel), and its
    # first pass also resolves the leaf level's later occurrences: that group of launches against the streams of both
    out["layer0_dedup"] = node_level[0] + resolve_level[0]
    out["node_insert_above_layer0"] = sum(node_level[1:])
    out["resolve_ids_above_leaves"] = sum(resolve_level[1:])
    return out


# ---------------------------------------------------------------------------- own arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        return run_b200_dist(args, world, rank, local_rank)
    torch.cuda.set_device(local_rank)
    pkg = load_package()
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peak_gbs, peak_src = 6650.0, "fallback"
    if peaks_path.exists():
        peak_gbs, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "measured"

    n_bases = args.bases
    stream = torch.cuda.current_stream()
    text = torch.empty(n_bases, dtype=torch.uint8, device="cuda")
    pkg.synth_genome(text, n_bases, seed=args.seed, repeat_permille=args.repeat_permille, device=local_rank,
                     stream=stream.cuda_stream)
    tree = pkg.SharedTree(DNA, device=local_rank, stream=stream.cuda_stream)
    for opt in args.option:
        name, value = opt.split("=")
        tree.set_option(name, int(value))

    for _ in range(args.warmup):
        tree.build_from_body(text)
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = pkg.kernel_launches()
    tree.profile(True)
    tree.profile_reset()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.steps):
        tree.build_from_body(text)
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    total_ms = ev0.elapsed_time(ev1)
    prof = tree.profile_read()
    tree.profile(False)
    launches = pkg.kernel_launches() - launches0
    if args.dump_outputs:
        dump_outputs(tree, args.dump_outputs, args.seed)
    ms_per_step = total_ms / args.steps
    bases_used = tree.width() * DNA
    value = bases_used / (ms_per_step * 1e-3) / 1e9

    n0 = tree.width()
    counts = tree.layer_counts()
    alg = algorithmic_bytes(n0, tree.leaf_count(), counts)
    kernels = {}
    for name, rec in prof.items():
        per_step_ms = rec["ms"] / args.steps
        k = {"ms_per_step": round(per_step_ms, 4), "launches_per_step": rec["launches"] // args.steps}
        if name in alg and per_step_ms > 0:
            k["algorithmic_bytes"] = alg[name]
            k["achieved_gbs"] = round(alg[name] / (per_step_ms * 1e-3) / 1e9, 1)
            k["frac_of_peak"] = round(k["achieved_gbs"] / peak_gbs, 4)
        kernels[name] = k
    bucket_classes = [n for n in ("bucket_partition", "bucket_dedup", "bucket_exact", "bucket_fallback") if n in kernels]
    if bucket_classes:
        # roofline classes follow what the launches do: the bucket kernels together are layer 0's emplace_node plus the
        # leaf level's resolve; node_insert / resolve_ids cover the levels above
        ms = sum(kernels[n]["ms_per_step"] for n in bucket_classes)
        g = {"ms_per_step": round(ms, 4), "launches_per_step": sum(kernels[n]["launches_per_step"] for n in bucket_classes),
             "algorithmic_bytes": alg["layer0_dedup"], "classes": bucket_classes}
        g["achieved_gbs"] = round(g["algorithmic_bytes"] / (ms * 1e-3) / 1e9, 1)
        g["frac_of_peak"] = round(g["achieved_gbs"] / peak_gbs, 4)
        kernels["layer0_dedup"] = g
        for name, key in (("node_insert", "node_insert_above_layer0"), ("resolve_ids", "resolve_ids_above_leaves")):
            if name in kernels and kernels[name]["ms_per_step"] > 0:
                k = kernels[name]
                k["algorithmic_bytes"] = alg[key]
                k["achieved_gbs"] = round(alg[key] / (k["ms_per_step"] * 1e-3) / 1e9, 1)
                k["frac_of_peak"] = round(k["achieved_gbs"] / peak_gbs, 4)
    timed = {n: k for n, k in kernels.items() if "algorithmic_bytes" in k}
    dom = max(timed, key=lambda n: timed[n]["ms_per_step"])
    traffic = None
    tpath = ROOT / "profiles" / "traffic.json"
    if tpath.exists():
        tj = json.loads(tpath.read_text())
        traffic = sum(tj.get(n, 0) for n in bucket_classes) if dom == "layer0_dedup" else tj.get(dom)
    roofline = {
        "bound": "hbm", "kernel": dom,
        "achieved": timed[dom]["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s",
        "frac": round(timed[dom]["achieved_gbs"] / peak_gbs, 4), "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes_per_step": timed[dom]["algorithmic_bytes"],
        "launches_per_step": timed[dom]["launches_per_step"],
        "avg_launch_ms": round(timed[dom]["ms_per_step"] / max(1, timed[dom]["launches_per_step"]), 4),
        "whole_build": {"algorithmic_bytes": alg["build_total"],
                        "achieved": round(alg["build_total"] / (ms_per_step * 1e-3) / 1e9, 1),
                        "frac": round(alg["build_total"] / (ms_per_step * 1e-3) / 1e9 / peak_gbs, 4)},
    }

    # ---- end to end: pinned host text -> C-ABI build -> counters back on the host ----
    e2e = None
    if not args.no_e2e:
        host = torch.empty(n_bases, dtype=torch.uint8, pin_memory=True)
        host.copy_(text)
        torch.cuda.synchronize()
        tree.build_from_body(host)  # warm the staging allocation
        t0 = time.perf_counter()
        reps = max(1, min(args.steps, 3))
        for _ in range(reps):
            tree.build_from_body(host)
            _ = (tree.width(), tree.leaf_count(), tree.node_count(), tree.root())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        e2e = {"value": bases_used / dt / 1e9, "unit": "Gbp/s", "h2d_bytes_per_step": n_bases,
               "d2h_bytes_per_step": 4 * (len(counts) + 1) + 4 + 16, "ms_per_step": dt * 1e3, "steps": reps}
        del host

    # ---- the rest of the path at the same size: sort_tree, bytes/serialize, decode, random access ----
    # every stage with its own roofline (SURVEY §8d algorithmic bytes), and the tree itself checked
    # against what the unmodified reference built from the same text (tests/golden/synth.json)
    gold = golden_record(args)
    parity = {"golden": gold["name"] if gold else None}
    pipeline = None
    if not args.no_pipeline:
        def timed(fn, reps=1):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(stream)
            for _ in range(reps):
                out = fn()
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps, out

        def kernel_sum(fn):
            tree.profile(True)
            tree.profile_reset()
            ms, out = timed(fn)
            per_kernel = {k: round(r["ms"], 4) for k, r in tree.profile_read().items()}
            tree.profile(False)
            return ms, per_kernel, out

        def stage(ms, alg_bytes):
            gbs = alg_bytes / (ms * 1e-3) / 1e9
            return {"ms": round(ms, 3), "algorithmic_bytes": int(alg_bytes), "achieved_gbs": round(gbs, 1), "frac_of_peak": round(gbs / peak_gbs, 4)}

        tree.build_from_body(text)
        U = [tree.leaf_count()] + tree.layer_counts()     # unique items: leaves, then node layers bottom-up
        nodes_total = sum(U[1:])
        stream_pre = tree.bytes()
        dag = torch.empty(max(stream_pre, 16) + (64 << 20), dtype=torch.uint8, device="cuda")
        tree.serialize_into(dag)
        parity["pre_sort_sha256"] = sha256_of_device_bytes(dag, stream_pre)
        sort_first_ms, _ = timed(tree.sort)   # first sort on this handle (its scratch was reserved by the build)
        tree.build_from_body(text)
        sort_ms, sort_kernels, _ = kernel_sum(tree.sort)
        plan_ms, stream_bytes = timed(tree.bytes)
        ser_ms, _ = timed(lambda: tree.serialize_into(dag))
        parity["post_sort_sha256"] = sha256_of_device_bytes(dag, stream_bytes)
        parity["layer_counts"] = U[1:]
        parity["leaves"] = U[0]
        out = torch.empty(n0 * DNA, dtype=torch.uint8, device="cuda")
        dec_first_ms, _ = timed(lambda: tree.decode_ascii(out=out))
        dec_ms, dec_kernels, _ = kernel_sum(lambda: tree.decode_ascii(out=out))
        roundtrip_ok = bool(torch.equal(out, text[: n0 * DNA]))
        del out
        leaves_out = torch.empty(n0, dtype=torch.int64, device="cuda")
        decl_ms, _ = timed(lambda: tree.decode(out=leaves_out))
        q = 10_000_000
        idx_host = pkg.query_indices(args.seed, q, n0)   # BASELINE.json config 5: seeded, reproducible on the CPU
        idx = torch.from_numpy(idx_host.astype("int64")).cuda()
        got = torch.empty(q, dtype=torch.int64, device="cuda")
        ra_ms, _ = timed(lambda: tree.random_access(idx, out=got), reps=3)
        ra_ok = bool(torch.equal(got, leaves_out[idx]))
        import hashlib
        parity["query_answers_sha256"] = hashlib.sha256(got.cpu().numpy().astype("<u8").tobytes()).hexdigest()
        del leaves_out, idx, got
        depth = tree.depth()
        # SURVEY §8(d): sort = histogram read + permute/rewire (read + write) of every node layer and the leaf
        # table + (freq, index) radix passes, here counted as one 8-byte pass per item; serialize = tables in,
        # stream out; decode = node layers 0-2 once + 8 B per leaf lookup + text out; random access = depth
        # node reads + leaf + index + answer per query
        sort_alg = 8 * nodes_total + 2 * 8 * (nodes_total + U[0]) + 8 * (nodes_total + U[0])
        ser_alg = 8 * (nodes_total + U[0]) + stream_bytes
        dec_alg = 8 * sum((n0 + (1 << k) - 1) >> k for k in (1, 2, 3)) + 8 * n0 + n0 * DNA
        ra_alg = q * (8 * (depth - 1) + 8 + 8 + 8)
        pipeline = {
            "sort_tree": dict(stage(sort_ms, sort_alg), first_call_ms=round(sort_first_ms, 3), kernels_ms=sort_kernels),
            "bytes_plan_ms": round(plan_ms, 3),
            "serialize": dict(stage(ser_ms + plan_ms, ser_alg), emit_ms=round(ser_ms, 3), stream_bytes=int(stream_bytes),
                              out_gbs=round(stream_bytes / (ser_ms * 1e-3) / 1e9, 1)),
            "bits_per_base": round(8.0 * stream_bytes / bases_used, 4),
            "decode_ascii": dict(stage(dec_ms, dec_alg), first_call_ms=round(dec_first_ms, 3), kernels_ms=dec_kernels,
                                 gbp_s=round(bases_used / (dec_ms * 1e-3) / 1e9, 1), roundtrip_equal=roundtrip_ok),
            "decode_leaves_ms": round(decl_ms, 3),
            "random_access": dict(stage(ra_ms, ra_alg), queries=q, mq_s=round(q / (ra_ms * 1e-3) / 1e6, 1), equal_to_decode=ra_ok),
        }

        # ---- the whole `compress` path end to end (compress.cpp:182-200): pinned host text -> build -> sort_tree ->
        # bytes -> .dag bytes back in pinned host memory; and the way back: host .dag -> deserialize -> text on the host
        if not args.no_e2e:
            host = torch.empty(n_bases, dtype=torch.uint8, pin_memory=True)
            host.copy_(text)
            dag_host = torch.empty(stream_bytes + 16, dtype=torch.uint8, pin_memory=True)
            torch.cuda.synchronize()

            def compress_once():
                t0 = time.perf_counter()
                tree.build_from_body(host)
                tree.sort()
                nb_ = tree.bytes()
                tree.serialize_to_host(dag_host)
                torch.cuda.synchronize()
                return time.perf_counter() - t0, nb_
            cold_s, _ = compress_once()
            warm = [compress_once()[0] for _ in range(max(3, min(args.steps, 5)))]
            warm_s = statistics.median(warm)  # a repetition that has to grow the memory pool takes several times longer: all are listed
            parity["e2e_compress_sha256"] = __import__("hashlib").sha256(dag_host[:stream_bytes].numpy().tobytes()).hexdigest()
            text_host = torch.empty(n0 * DNA, dtype=torch.uint8, pin_memory=True)
            back = pkg.SharedTree(DNA, device=local_rank, stream=stream.cuda_stream)

            def decompress_once():
                t0 = time.perf_counter()
                back.deserialize(dag_host[:stream_bytes].numpy())
                back.decode_ascii_to_host(text_host)
                torch.cuda.synchronize()
                return time.perf_counter() - t0
            dcold_s = decompress_once()
            dwarm = [decompress_once() for _ in range(3)]
            dwarm_s = statistics.median(dwarm)
            e2e_roundtrip = bool(torch.equal(text_host, host[: n0 * DNA]))
            ref_t = (gold or {}).get("reference_timing")
            pipeline["e2e_compress"] = {
                "value": bases_used / warm_s / 1e9, "unit": "Gbp/s", "ms": round(warm_s * 1e3, 2), "first_call_ms": round(cold_s * 1e3, 2),
                "reps_ms": [round(w * 1e3, 2) for w in warm], "statistic": "median of the warm repetitions",
                "h2d_bytes": n_bases, "d2h_bytes": int(stream_bytes), "path": "stb_build_from_body(HOST) + stb_sort_tree + stb_bytes + stb_serialize(HOST)",
                "reference_s": round(ref_t["construct_s"] + ref_t["sort_s"], 1) if ref_t else None}
            pipeline["e2e_decompress"] = {
                "value": bases_used / dwarm_s / 1e9, "unit": "Gbp/s", "ms": round(dwarm_s * 1e3, 2), "first_call_ms": round(dcold_s * 1e3, 2),
                "reps_ms": [round(w * 1e3, 2) for w in dwarm], "h2d_bytes": int(stream_bytes), "d2h_bytes": n0 * DNA, "roundtrip_equal": e2e_roundtrip,
                "path": "stb_deserialize(host bytes) + stb_decode_ascii(HOST)"}
            # ---- BASELINE.json config 3 as a FASTA file: a '>' header line and 60-column lines, from pinned host memory.
            # Same body, so the same tree: the stream must equal the reference's again.  (stb_build_from_fasta(STB_HOST):
            # chunked copy, body extraction with the line automaton's state carried across chunks, build behind the copy.)
            import numpy as np
            body_np = host[: (n_bases // 60) * 60].numpy().reshape(-1, 60)
            header = np.frombuffer(b">synthetic genome, config 3\n", dtype=np.uint8)
            rest = host[(n_bases // 60) * 60:].numpy()
            fasta_len = header.size + body_np.shape[0] * 61 + rest.size + 1
            fasta_host = torch.empty(fasta_len, dtype=torch.uint8, pin_memory=True)
            fview = fasta_host.numpy()
            fview[: header.size] = header
            lines = fview[header.size: header.size + body_np.shape[0] * 61].reshape(-1, 61)
            lines[:, :60] = body_np
            lines[:, 60] = 10
            fview[header.size + body_np.shape[0] * 61: fasta_len - 1] = rest
            fview[fasta_len - 1] = 10
            del body_np, lines, fview
            tree.build_from_fasta(fasta_host)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            reps_f = max(1, min(args.steps, 3))
            for _ in range(reps_f):
                tree.build_from_fasta(fasta_host)
                _ = (tree.width(), tree.node_count())
            torch.cuda.synchronize()
            fasta_s = (time.perf_counter() - t0) / reps_f
            fasta_counts = tree.layer_counts()
            tree.sort()
            tree.serialize_to_host(dag_host)
            parity["e2e_fasta_sha256"] = __import__("hashlib").sha256(dag_host[:stream_bytes].numpy().tobytes()).hexdigest()
            pipeline["e2e_fasta"] = {
                "value": bases_used / fasta_s / 1e9, "unit": "Gbp/s", "ms": round(fasta_s * 1e3, 2), "h2d_bytes": int(fasta_len),
                "layout": "one '>' header line, 60-column lines", "vs_bare_body_e2e": round(fasta_s * 1e3 / e2e["ms_per_step"], 3) if e2e else None,
                "layer_counts_equal": fasta_counts == U[1:], "path": "stb_build_from_fasta(STB_HOST)"}
            del fasta_host
            # ---- the "real genome" variant of config 3: runs of N (1 % of the bases) and soft-masked lower case laid
            # over the same sequence (DESIGN.md §6), built from device and from pinned host memory; its own reference golden
            gold_n = golden_record(args, "nruns")
            pkg.synth_mask(text, seed=args.seed, device=local_rank, stream=stream.cuda_stream)
            host.copy_(text)
            torch.cuda.synchronize()
            for _ in range(3):  # a tree of another shape: the first builds re-size the handle's buffers
                tree.build_from_body(text)
            nrun_reps = [timed(lambda: tree.build_from_body(text))[0] for _ in range(5)]
            nrun_ms = statistics.median(nrun_reps)
            tree.build_from_body(host)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps_f):
                tree.build_from_body(host)
                _ = (tree.width(), tree.node_count())
            torch.cuda.synchronize()
            nrun_host_s = (time.perf_counter() - t0) / reps_f
            nrun_counts = tree.layer_counts()
            tree.sort()
            nrun_bytes = tree.bytes()
            tree.serialize_to_host(dag_host)
            parity["nruns_sha256"] = __import__("hashlib").sha256(dag_host[:nrun_bytes].numpy().tobytes()).hexdigest()
            parity["nruns_golden"] = gold_n["name"] if gold_n else None
            pipeline["nruns"] = {
                "build_ms": round(nrun_ms, 3), "build_reps_ms": [round(r, 3) for r in nrun_reps], "value": bases_used / (nrun_ms * 1e-3) / 1e9, "unit": "Gbp/s",
                "vs_plain_build": round(nrun_ms / ms_per_step, 3), "e2e_ms": round(nrun_host_s * 1e3, 2),
                "e2e_value": bases_used / nrun_host_s / 1e9, "vs_bare_body_e2e": round(nrun_host_s * 1e3 / e2e["ms_per_step"], 3) if e2e else None,
                "layout": "N runs of 1..16384 bases in 8 % of the 64 Ki-base blocks, lower case in half of the 4 Ki-base blocks",
                "stream_bytes": int(nrun_bytes), "path": "stb_build_from_body(DEVICE | HOST)"}
            if gold_n:
                check_against_golden(gold_n, "per-layer node counts (N-run variant)", nrun_counts, gold_n["layer_counts"])
                check_against_golden(gold_n, "stream sha256 after sort_tree (N-run variant)", parity["nruns_sha256"], gold_n["post_sha256"])
                parity["nruns_equal_to_reference"] = True
            pkg.synth_genome(text, n_bases, seed=args.seed, repeat_permille=args.repeat_permille, device=local_rank, stream=stream.cuda_stream)
            tree.build_from_body(text)
            del host, dag_host, text_host, back
        del dag
        if gold:
            check_against_golden(gold, "per-layer node counts", parity["layer_counts"], gold["layer_counts"])
            check_against_golden(gold, "leaf count", parity["leaves"], gold["leaves"])
            check_against_golden(gold, "stream sha256 before sort_tree", parity["pre_sort_sha256"], gold["pre_sha256"])
            check_against_golden(gold, "stream sha256 after sort_tree", parity["post_sort_sha256"], gold["post_sha256"])
            check_against_golden(gold, "stream length", int(stream_bytes), gold["post_bytes"])
            check_against_golden(gold, "sha256 of the 10 M operator[] answers", parity["query_answers_sha256"], gold["query_answers_sha256"])
            if "e2e_fasta_sha256" in parity:
                check_against_golden(gold, "stream sha256 of the FASTA-file build (header + 60-column lines)", parity["e2e_fasta_sha256"], gold["post_sha256"])
            if "e2e_compress_sha256" in parity:
                check_against_golden(gold, "stream sha256 of the end-to-end compress path", parity["e2e_compress_sha256"], gold["post_sha256"])
            parity["equal_to_reference"] = True
    elif gold:
        counts_now = tree.layer_counts()
        check_against_golden(gold, "per-layer node counts", counts_now, gold["layer_counts"])
        parity["layer_counts"] = counts_now

    cpu = None
    if not args.no_cpu_baseline:
        sample = args.cpu_sample_bases or 120_000_000
        sample = min(sample, n_bases)
        chunk = text[:sample].cpu().numpy().tobytes()
        dt, kind, cores = cpu_build_once(chunk)
        cpu = {"value": sample / dt / 1e9, "unit": "Gbp/s", "cores": cores, "kind": kind,
               "sample": f"first {sample} bases of the same sequence, one build, {dt:.1f} s", "host_cpus": os.cpu_count(),
               "full_size": full_size_reference(gold)}

    line = {
        "parity": parity,
        "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": workload_config(args), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels, "pipeline": pipeline,
        "tree": {"width": n0, "leaves": tree.leaf_count(), "nodes": tree.node_count(), "depth": tree.depth(),
                 "first_layer_nodes": [int(c) for c in counts[:6]]},  # compare with "sharded_layer_nodes" of the N > 1 lines
    }
    print(json.dumps(line), flush=True)


def run_b200_dist(args, world, rank, local_rank):
    """N > 1: the sharded build behind one C-ABI call per rank (csrc/shard.cu, include/shared_tree_b200_dist.h).
    Strong scaling: the same 3.1 Gbp sequence split over the ranks by leaf range; per level the partition kernel
    stores the (key, position) records straight into their hash owner's memory over NVLink, the owner deduplicates
    them on chip and answers with plain REDs into the home rank's words; NCCL carries three barriers and one small
    all-gather per level.  torch.distributed only hands the communicator id around and reduces the timings."""
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package

    # NCCL prints its version banner on stdout when the box exports NCCL_DEBUG=VERSION; this
    # program owes its caller exactly one JSON line there, so stdout points at stderr until the
    # communicators exist.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        warm = torch.zeros(1, device="cuda")
        dist.all_reduce(warm)
        torch.cuda.synchronize()
        pkg = load_package()
        from genome_compression_b200 import shard
        stream = torch.cuda.current_stream()
        me = shard.create_nccl(DNA, device=local_rank, stream=stream.cuda_stream)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    for opt in args.option:
        name, value = opt.split("=")
        me.set_option(name, int(value))
    local_cpus = bind_to_gpu_numa_node(local_rank)

    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peak_gbs, peak_src = 6650.0, "fallback"
    if peaks_path.exists():
        peak_gbs, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "measured"
    n_bases = args.bases
    n_leaves = n_bases // DNA
    first, count = me.range(n_bases)
    body = torch.empty(max(16, count), dtype=torch.uint8, device="cuda")
    if count:
        pkg.synth_genome(body, n_bases, first=first, count=count, seed=args.seed, repeat_permille=args.repeat_permille,
                         device=local_rank, stream=stream.cuda_stream)
    for _ in range(args.warmup):
        me.build_from_body(body, n_bases)
    torch.cuda.synchronize()
    dist.barrier()
    # rank 0 alone polls NVML, and sparsely (its GPU's clocks go into the line): eight processes
    # polling every 4 ms contend for the driver and doubled the step time at N = 8 in round 1
    sampler = ClockSampler(local_rank, period_s=0.012) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = pkg.kernel_launches()
    me.profile_reset()
    me.profile(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    dist.barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        me.build_from_body(body, n_bases)
    ev1.record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = torch.tensor([pkg.kernel_launches() - launches0], device="cuda", dtype=torch.int64)
    dist.all_reduce(launches, op=dist.ReduceOp.SUM)
    prof = me.profile_read()
    me.profile(False)
    if os.environ.get("STB_RANK_PROFILES"):  # per-rank kernel classes, for finding the rank the others wait for
        out_dir = ROOT / "gpurun_out"
        out_dir.mkdir(exist_ok=True)
        (out_dir / f"rank_profile_{os.environ['STB_RANK_PROFILES']}_n{world}_r{rank}.json").write_text(json.dumps(
            {k: round(v["ms"] / args.steps, 4) for k, v in prof.items()}))
    ms_per_step = float(ms.item()) / args.steps
    bases_used = n_leaves * DNA
    value = bases_used / (ms_per_step * 1e-3) / 1e9

    # end to end: every rank's text shard starts in pinned host memory (H2D inside the call)
    e2e = None
    if not args.no_e2e:
        host = torch.empty(body.numel(), dtype=torch.uint8, pin_memory=True)
        host.copy_(body)
        torch.cuda.synchronize()
        me.build_from_body(host, n_bases)
        torch.cuda.synchronize()
        dist.barrier()
        reps = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(reps):
            me.build_from_body(host, n_bases)
            _ = me.layer_totals()
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - t0) / reps], device="cuda", dtype=torch.float64)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        # for the record: the copies alone, all ranks at once (what PCIe and the host memory give)
        staging = torch.empty_like(body)
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            staging.copy_(host, non_blocking=True)
        torch.cuda.synchronize()
        ct = torch.tensor([(time.perf_counter() - t0) / reps], device="cuda", dtype=torch.float64)
        dist.all_reduce(ct, op=dist.ReduceOp.MAX)
        del staging, host
        e2e = {"value": bases_used / float(dt.item()) / 1e9, "unit": "Gbp/s", "h2d_bytes_per_step": n_bases,
               "d2h_bytes_per_step": 4 * 48 * world, "ms_per_step": float(dt.item()) * 1e3, "steps": reps,
               "h2d_copy_alone_ms": round(float(ct.item()) * 1e3, 3), "host_cores_bound_per_rank": local_cpus,
               "path": "stb_shard_build_from_body(STB_HOST) on every rank"}

    # parity, outside the timed region: the tree gathered on rank 0, sorted, serialized, compared with the reference's
    me.build_from_body(body, n_bases)
    totals = me.layer_totals()
    del body
    tree = me.gather(stream=stream.cuda_stream)
    parity = None
    if rank == 0:
        if args.dump_outputs:  # gathered from the build above, which repeats the last timed one on the same input
            dump_outputs(tree, args.dump_outputs, args.seed)
        gold = golden_record(args)
        parity = {"golden": gold["name"] if gold else None, "leaves": tree.leaf_count(), "layer_counts": tree.layer_counts()}
        nb_pre = tree.bytes()
        dag = torch.empty(nb_pre + (64 << 20), dtype=torch.uint8, device="cuda")
        tree.serialize_into(dag)
        parity["pre_sort_sha256"] = sha256_of_device_bytes(dag, nb_pre)
        tree.sort()
        nb_post = tree.bytes()
        tree.serialize_into(dag)
        parity["post_sort_sha256"] = sha256_of_device_bytes(dag, nb_post)
        parity["stream_bytes"] = nb_post
        del dag
        if gold:
            check_against_golden(gold, "per-layer node counts (sharded build)", parity["layer_counts"], gold["layer_counts"])
            check_against_golden(gold, "leaf count (sharded build)", parity["leaves"], gold["leaves"])
            check_against_golden(gold, "stream sha256 before sort_tree (sharded build)", parity["pre_sort_sha256"], gold["pre_sha256"])
            check_against_golden(gold, "stream sha256 after sort_tree (sharded build)", parity["post_sort_sha256"], gold["post_sha256"])
            parity["equal_to_reference"] = True
        kernels = {name: {"ms_per_step": round(rec["ms"] / args.steps, 4), "launches_per_step": rec["launches"] // args.steps}
                   for name, rec in prof.items()}
        # the dominant stage of rank 0 and the record streams it moves (bytes per position of the sharded node levels:
        # children 8 + record out 12 for the partition; record in 12 + out 12 for the owner's split; record in 12 for the dedup)
        sharded_node_positions = sum(-(-n_leaves // (1 << l)) for l in range(1, len(totals))) // world
        per_position = {"shard_partition": 20, "shard_partition2": 24, "shard_dedup": 12, "assign_ids": 20, "shard_resolve": 8, "count_firsts": 1}
        stage_names = [k for k in kernels if k in per_position]
        dom = max(stage_names or list(kernels), key=lambda k: kernels[k]["ms_per_step"])
        alg = per_position.get(dom, 12) * sharded_node_positions
        ach = alg / (kernels[dom]["ms_per_step"] * 1e-3) / 1e9
        line = {
            "parity": parity,
            "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": workload_config(args, {"sharding": f"{world} ranks, contiguous power-of-two aligned leaf ranges; records to their hash owner and "
                                                         f"answers back through peer-mapped memory (NVLink); {len(totals)} sharded levels, the rest on rank 0"}),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches.item()),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak_gbs, "unit": "GB/s",
                         "frac": round(ach / peak_gbs, 4), "traffic": None, "peak_source": peak_src,
                         "note": "rank 0's launches of its dominant stage kernel; algorithmic bytes = the record streams of its share of the sharded levels"},
            "cpu_baseline": None, "kernels": kernels,
            "sync_per_level": {"nccl_collectives": 0, "peer_exchange_kernels": 4, "what": "barrier + a few counts stored into every peer's arena over NVLink (csrc/shard.cu)"},
            "tree": {"width": n_leaves, "leaves": totals[0], "sharded_layer_nodes": totals[1:]},
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    me.close()
    dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
