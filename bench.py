#!/usr/bin/env python
"""bench.py — k-mer recruitment read-bases/s on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cenx|cen6|stream] [--scale S]
                    [--dump-outputs DIR]

Workloads (config.workload), all drawn from genomes made by the reference's own simulate_tandem_repeat.py
(tests/golden/genomes/, oracle/make_genomes.py) with reads from centroflye_b200.synth:

  cenx    BASELINE.json configs[1] (the default, the configuration the metric is quoted on): DXZ1 x 1500 (3.08 Mb array,
          seed 1) at 50x long reads with 6 % errors, k = 19, --coverage 32; one step = the whole recruitment path
          (document frequency -> rare band -> per-unit clouds -> unit-distance pair graph -> edge filter).  At N GPUs
          (weak scaling) the read set is that of N such arrays -- array j >= 2 from the reference simulator too, on its
          own unit (DXZ1 with 30 % of the bases substituted: arrays of ONE unit share their error k-mers, which at
          N x 50x enter the rare band and nearly double the pair increments per array, so the work per GPU would not be
          fixed) -- every rank holding the reads i = rank mod N of every array; counts, rare set and distance graph
          stay global.
  cen6    configs[2]: D6Z1 x 1000 (3.2 Mb, seed 4), 50x, 12 % errors, --kmer-survival-rate 0.09 --coverage 50; the ONE
          read set sharded over the N ranks (strong scaling).
  stream  configs[4]: a stream of independent 155-Mbase batches drawn like configs[1] (batch b = read seed 3 + b, batch 0
          IS configs[1]) through the stage-A kernel pair, complete count table written per batch, batches dealt
          round-robin to the N GPUs, no collective; the HBM-roofline figure of the north star.

`value` times a step with inputs resident in HBM; `e2e` times the same call from pinned host buffers (H2D inside) to
host-resident results (D2H inside); `e2e_cli` is the drop-in command line from a report file on disk to the two output
files.  --scale shrinks the array multiplicity (parity / smoke use); 1.0 is the configuration the metric is quoted on.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned (cenx / cen6: rare k-mers, clouds,
edges, recruited k-mers, counters; stream: the rare k-mers and count table of the last batch) in a canonical order as
float64 .npy files, arrays beyond 12 MB as a fixed, seeded sample of their rows (DIR/manifest.json says which).  The
inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "cenx": dict(params=dict(k=19, coverage=32, min_coverage=4, min_d=1, max_d=150, bottom=0.9, top=3.0,
                             kmer_survival_rate=0.34, max_nonuniq=3),
                 data=dict(genome="cenx_dxz1_m1500_s{seed}", genome_more="cenx_like_u{seed}_m1500_s{seed}", genome_seed=1,
                           read_coverage=50, error_rate=0.06, read_seed=3),
                 label="configs[1]: cenX-like array, reference simulator DXZ1_rc x 1500 (3.08 Mb, div-rate 0.01, seed 1) "
                       "+ 2 x 200 kb flanks, 50x reads, 6% errors, k=19, coverage=32, max_d=150: full recruitment + "
                       "read_kmer_cloud build"),
    "cen6": dict(params=dict(k=19, coverage=50, min_coverage=4, min_d=1, max_d=150, bottom=0.9, top=3.0,
                             kmer_survival_rate=0.09, max_nonuniq=3),
                 data=dict(genome="cen6_d6z1_m1000_s{seed}", genome_seed=4, read_coverage=50, error_rate=0.12, read_seed=5),
                 label="configs[2]: cen6-like array, reference simulator D6Z1 x 1000 (3.2 Mb, div-rate 0.01, seed 4) "
                       "+ 2 x 200 kb flanks, 50x reads, 12% errors, k=19, coverage=50, kmer-survival-rate 0.09: full "
                       "recruitment + read_kmer_cloud build"),
}
CONFIGS["stream"] = dict(CONFIGS["cenx"], label="configs[4]: stream of independent 155-Mbase batches drawn like "
                         "configs[1] (batch b = read seed 3 + b) through the stage-A kernels (document frequency of every "
                         "k-mer + rare band), count table written per batch")
PARAMS = CONFIGS["cenx"]["params"]  # (tools/ import these)
# algorithmic bytes per unit of work, fixed before the first measurement (BASELINE.md §4 / SURVEY.md §8d)
BYTES_PER_KMER_A = 32.25
BYTES_PER_INCREMENT_C = 32.0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def simulate(config, scale, rank=0, world=1, n_arrays=None, read_seed_shift=0, keep_reads=False, first_array=0):
    """-> (unit, ReadBatch, UnitIndex[, reads]).  cenx at world > 1: array j (genome seed 1 + j, read seed 3 + j) for
    j < world, this rank's share of every array; cen6 at world > 1: this rank's share of the one array."""
    from centroflye_b200 import synth
    from centroflye_b200.ingest import batch_from_synth
    D = CONFIGS[config]["data"]
    n_arrays = (world if config != "cen6" else 1) if n_arrays is None else n_arrays
    reads, unit = [], None
    for j in range(first_array, first_array + n_arrays):
        genome, a0, alen, unit_j = synth.load_genome((D["genome"] if j == 0 else D["genome_more"]).format(seed=D["genome_seed"] + j))
        unit = unit or unit_j
        if scale != 1.0:  # fewer copies of the unit: the left flank, the first copies, the right flank
            keep = max(8, int(round(alen / len(unit_j) * scale))) * len(unit_j)
            genome = np.concatenate([genome[:a0 + keep], genome[a0 + alen:]])
            alen = keep
        reads += synth.simulate_reads(genome, a0, alen, unit_j, D["read_coverage"], D["error_rate"],
                                      D["read_seed"] + j + read_seed_shift, id_prefix="read" if j == 0 else f"a{j}_read",
                                      shard=(rank, world) if world > 1 else None)
    batch, units = batch_from_synth(reads, len(unit))
    return (unit, batch, units, reads) if keep_reads else (unit, batch, units)


def make_inputs(scale, rank=0, world=1):
    """configs[1] (tools/ and tests use this)."""
    return simulate("cenx", scale, rank, world)


def band(params=None):
    from centroflye_b200.engine import band_to_int
    P = PARAMS if params is None else params
    left = P["bottom"] * P["coverage"] * P["kmer_survival_rate"]
    right = P["top"] * P["coverage"] * P["kmer_survival_rate"]
    return band_to_int(left, right)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  A step lasts tens
    of milliseconds, so the sampler reads NVML directly (nvidia_ml_py) and falls back to polling nvidia-smi only if
    NVML cannot be loaded.  One GPU: every 5 ms (no measurable effect on the step).  Several ranks: ONLY rank 0
    samples, every GPU of the job, every 25 ms -- eight processes polling NVML every 5 ms stretched the collectives of
    a 12.5 ms step to 19.9 ms (measured, configs[2] on 8 B200s: the host threads that enqueue them were held up)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, world=1, rank=0):
        self.period = float(os.environ.get("CFK_CLOCK_PERIOD_MS", "5" if world == 1 else "25")) * 1e-3
        self.sm, self.mx, self.reasons, self.index = [], [], set(), index
        self.indices = [index] if world == 1 else list(range(world))  # one node: local ranks 0..world-1
        self.active = rank == 0
        self.stop, self.source = threading.Event(), "nvml"
        self.th = threading.Thread(target=self._run, daemon=True)

    def _nvml_handle(self, idx=None):
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = self.index if idx is None else idx
        if vis:
            ent = vis.split(",")[idx].strip()
            if ent.isdigit():
                idx = int(ent)
            else:
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(ent)
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)

    def _run(self):
        try:
            handles = [self._nvml_handle(i) for i in self.indices]
            nv = handles[0][0]
            handles = [h for _, h in handles]
            for h in handles:
                self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown")
                    else nv.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop.is_set():
                for h in handles:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = int(get_reasons(h))
                    for name, bit in bits.items():
                        if r & int(bit):
                            self.reasons.add(name)
                self.stop.wait(self.period)
            return
        except Exception as e:  # noqa: BLE001 - any NVML problem: poll nvidia-smi instead
            self.source = f"nvidia-smi ({type(e).__name__})"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                r = [x.strip() for x in out.split(",")] if out else []
                if r and r[0].replace(".", "").isdigit():
                    self.sm.append(float(r[0]))
                if len(r) > 1 and r[1].replace(".", "").isdigit():
                    self.mx.append(float(r[1]))
                for name, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        if self.active:
            self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.active:
            self.th.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source,
                "gpus_sampled": len(self.indices), "period_ms": self.period * 1e3}


def ncu_traffic(kernel):
    """DRAM bytes (read + write) of one launch of `kernel` from the newest committed `ncu --set full` summary under
    profiles/ (tools/ncu_summary.py output); (None, None) if no capture names the kernel."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_summary.txt")),
                       key=lambda p: [int(x) for x in re.findall(r"\d+", os.path.basename(p))], reverse=True):
        cur, vals = None, {}
        for ln in open(path):
            if ln.startswith("## "):
                cur = ln.strip().split("::")[-1]
            elif cur == kernel:
                m = re.match(r"\s*(dram__bytes_(?:read|write)\.sum)\s+([0-9.]+)\s+(\S+)", ln)
                if m:
                    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(3), None)
                    if mult:
                        vals[m.group(1)] = float(m.group(2)) * mult
        if len(vals) == 2:
            return sum(vals.values()), os.path.relpath(path, ROOT)
    return None, None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def sm_clock_hz():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f).get("sm_max_mhz", 1965.0)) * 1e6
    return 1965.0e6


def init_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    return world, rank, local


def make_barrier(world):
    import torch
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    return barrier


def max_over_ranks(x, world, device):
    import torch
    import torch.distributed as dist
    if world == 1:
        return float(x)
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(xs, world, device):
    import torch
    import torch.distributed as dist
    if world == 1:
        return [int(x) for x in xs]
    t = torch.tensor([int(x) for x in xs], dtype=torch.int64, device=device)
    dist.all_reduce(t)
    return [int(x) for x in t.tolist()]


# ---- --dump-outputs: what the timed path returned in its last step, for output-by-output comparison of two builds ----
DUMP_BYTES_PER_ARRAY = 12 << 20  # five arrays of that size at most per run, so a dump stays under 64 MB
DUMP_SEED = 20261020


def sorted_rows(a):
    """Rows of a 2-D integer array in lexicographic order (the device returns edges and table slots unordered)."""
    return a[np.lexsort(a.T[::-1])] if a.shape[0] else a


def dump_outputs(dirname, arrays, rank=0, world=1):
    """arrays: name -> integer numpy array in a canonical order.  Written as float64 (exact for the integers here:
    2-bit k-mer codes of k <= 26, ids, counts), each one cut to DUMP_BYTES_PER_ARRAY by a fixed, seeded choice of rows
    that depends only on the number of rows, so equal outputs give equal files.  manifest.json records the full shapes
    and which rows were kept.  At several ranks every rank writes its own shard as <name>_rank<r>.npy."""
    os.makedirs(dirname, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    manifest = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out = a.astype(np.float64)
        row_bytes = max(out[:1].nbytes, 8)
        entry = {"shape": list(a.shape), "source_dtype": str(a.dtype), "rows": "all"}
        if out.nbytes > DUMP_BYTES_PER_ARRAY:
            keep = DUMP_BYTES_PER_ARRAY // row_bytes
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(a.shape[0], size=keep, replace=False))
            out = out[rows]
            entry["rows"] = (f"{keep} of {a.shape[0]}: np.sort(np.random.default_rng({DUMP_SEED}).choice({a.shape[0]}, "
                             f"size={keep}, replace=False))")
        np.save(os.path.join(dirname, f"{name}{suffix}.npy"), out)
        manifest[name] = entry
    with open(os.path.join(dirname, f"manifest{suffix}.json"), "w") as f:
        json.dump(manifest, f, indent=1)


# ---- parity leg: a down-scaled instance of the same kind at THIS world size against the C oracle ------------------
def parity_check(eng, world, rank, config):
    """Sharded (or single-GPU) recruitment on a ~1-Mbase instance == oracle/c on the whole read set: rare set, clouds
    of this rank, increment count, edge set, recruited k-mers.  The oracle is the checker here, nothing is timed."""
    import torch
    import torch.distributed as dist
    from centroflye_b200 import synth
    from centroflye_b200.engine import band_to_int
    from centroflye_b200.ingest import batch_from_synth
    from oracle import c_oracle
    P = CONFIGS[config]["params"]
    D = CONFIGS[config]["data"]
    genome, a0, alen, unit = synth.load_genome(D["genome"].format(seed=D["genome_seed"]))
    keep = 80 * len(unit)  # 80 copies of the unit and 5 kb of each flank
    genome = np.concatenate([genome[a0 - 5000:a0 + keep], genome[a0 + alen:a0 + alen + 5000]])
    kw = dict(median_len=9000, sigma=0.4, min_len=5200, max_len=30000)
    cov = 24
    whole = synth.simulate_reads(genome, 5000, keep, unit, cov, D["error_rate"], 11, **kw)
    mine = synth.simulate_reads(genome, 5000, keep, unit, cov, D["error_rate"], 11,
                                shard=(rank, world) if world > 1 else None, **kw)
    k = P["k"]
    lo, hi = band_to_int(P["bottom"] * cov * P["kmer_survival_rate"], P["top"] * cov * P["kmer_survival_rate"])
    batch, units = batch_from_synth(mine, len(unit))
    if world > 1:
        from centroflye_b200.dist import ShardedRecruiter
        rec = ShardedRecruiter(eng, batch, units, k, rank, world)
        index, csr, res = rec.step(lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"])
    else:
        index, csr, res = eng.recruit(eng.upload_reads(batch, k), eng.upload_units(units, k), k, lo, hi, P["max_nonuniq"],
                                      P["min_d"], P["max_d"], P["min_coverage"])
    whole_batch, whole_units = batch_from_synth(whole, len(unit))
    keys = index.sorted_keys.cpu().numpy().view(np.uint64)
    ok, detail = True, {}
    want_rare = None
    if rank == 0:
        want = c_oracle.recruit(whole_batch, whole_units, k, lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"],
                                P["min_coverage"], threads=min(8, os.cpu_count() or 1))
        want_rare = want["rare"]
        got = res.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)
        canon = lambda e: e[np.lexsort((e[:, 3], e[:, 2], e[:, 1], e[:, 0]))]  # noqa: E731
        detail = {"rare_equal": bool(np.array_equal(keys, want["rare"])),
                  "increments_equal": bool(res.n_increments == want["n_increments"]),
                  "edges_equal": bool(got.shape == want["edges"].shape and np.array_equal(canon(got), canon(want["edges"]))),
                  "unique_kmers_equal": bool(np.array_equal(np.sort(res.selected.cpu().numpy().view(np.uint32)), want["selected"])),
                  "read_bases": int(whole_batch.n_bases), "rare": int(keys.size), "edges": int(got.shape[0]),
                  "unique_kmers": int(res.selected.numel())}
        ok = all(v for k_, v in detail.items() if k_.endswith("_equal"))
    # every rank: its own clouds against the oracle's clouds of its reads (the rare set is the same everywhere)
    my_ptr, my_ids = c_oracle.clouds(c_oracle.unpacked_codes(batch), units, k, keys)
    clouds_ok = bool(np.array_equal(csr.unit_ptr.cpu().numpy()[: units.n_units + 1], my_ptr) and
                     np.array_equal(csr.ids.cpu().numpy().view(np.uint32)[: my_ids.size], my_ids))
    flags = torch.tensor([int(ok), int(clouds_ok)], dtype=torch.int64, device=eng.device)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    detail["clouds_equal_all_ranks"] = bool(flags[1].item())
    detail["checker"] = "oracle/c (C restatement of the reference, pinned to the reference's golden outputs)"
    return bool(flags[0].item()) and bool(flags[1].item()), detail


# ---- the recruitment configs (cenx, cen6) ---------------------------------------------------------------------
def run_recruit(args):
    import torch
    from centroflye_b200.engine import Engine
    world, rank, local = init_dist()
    eng = Engine(f"cuda:{local}")
    C = CONFIGS[args.config]
    P = C["params"]
    k = P["k"]
    lo, hi = band(P)
    barrier = make_barrier(world)

    t0 = time.time()
    unit, batch, units, reads_list = simulate(args.config, args.scale, rank, world, keep_reads=True)
    log(f"[bench] rank {rank}: inputs in {time.time() - t0:.1f}s: {batch.n_reads} reads, {batch.n_bases} bases, "
        f"{units.n_units} units")
    parity_ok, parity = (None, None)
    if args.check:
        parity_ok, parity = parity_check(eng, world, rank, args.config)
        log(f"[bench] rank {rank}: parity leg {'ok' if parity_ok else 'FAILED'}")

    runner = None
    if world > 1:
        from centroflye_b200.dist import ShardedRecruiter
        runner = ShardedRecruiter(eng, batch, units, k, rank, world)

    def device_step(reads, dunits):
        if runner is not None:
            return runner.step(lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"],
                               gather=False)  # edges stay sharded by source k-mer, like the work
        return eng.recruit(reads, dunits, k, lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"])

    def e2e_step():
        if runner is not None:
            return runner.e2e_step(lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"])
        reads = eng.upload_reads(batch, k)
        dunits = eng.upload_units(units, k)
        early = {}
        # the rare set and the clouds are final after stage B: they travel to the host on a side stream while the
        # distance graph is computed; edges and endpoints follow when it is done
        index, csr, res = eng.recruit(reads, dunits, k, lo, hi, P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"],
                                      on_clouds=lambda index, csr: early.update(eng.start_host_copy(
                                          unit_ptr=csr.unit_ptr, ids=csr.ids, rare_keys=index.sorted_keys)))
        out = eng.to_host(selected=res.selected, edges=res.edges)  # pinned result buffers; synchronises
        eng.finish_host_copies()
        out.update(early)
        d2h = sum(t.numel() * t.element_size() for t in out.values())
        return reads.h2d_bytes + dunits.h2d_bytes, d2h

    reads = eng.upload_reads(batch, k) if runner is None else None
    dunits = eng.upload_units(units, k) if runner is None else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)

    for _ in range(args.warmup):
        res = device_step(reads, dunits)
    barrier()
    n_bases_total = batch.n_bases if runner is None else runner.n_bases_total

    step_ms, launches0 = [], eng.launch_count()
    stage_ms = {}
    with ClockSampler(local, world, rank) as clk:
        for _ in range(args.steps):
            flush.fill_(1)  # evict L2 between timed steps (inputs alone would fit the 126 MB L2)
            barrier()
            eng.events = []
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            res = device_step(reads, dunits)
            b.record()
            barrier()
            step_ms.append(a.elapsed_time(b))
            for name, ms in eng.stage_times_ms().items():
                stage_ms.setdefault(name, []).append(ms)
            eng.events = None
    launches = (eng.launch_count() - launches0) / max(args.steps, 1)
    if args.dump_outputs:
        index, csr, dres = res
        dump_outputs(args.dump_outputs, {
            "rare_kmers": index.sorted_keys.cpu().numpy().view(np.uint64),
            "cloud_unit_ptr": csr.unit_ptr.cpu().numpy()[: csr.n_units + 1],
            "cloud_ids": csr.ids.cpu().numpy()[: csr.n_entries].view(np.uint32),
            "edges": sorted_rows(dres.edges.cpu().numpy().view(np.uint32).reshape(-1, 4)),
            "unique_kmers": np.sort(dres.selected.cpu().numpy().view(np.uint32)),
            "counts": np.array([dres.n_increments, dres.n_candidates, dres.n_pair_candidates], dtype=np.int64)},
            rank, world)
    ms = max_over_ranks(float(np.mean(step_ms)), world, eng.device)
    last = res[2]
    n_edges_total, = sum_over_ranks([int(last.edges.shape[0])], world, eng.device)

    # end to end: pinned host buffers -> host results, same call
    e2e_ms, h2d, d2h = [], 0, 0
    e2e_step()
    for _ in range(max(2, min(args.steps, 3))):
        barrier()
        t1 = time.perf_counter()
        h2d, d2h = e2e_step()
        barrier()
        e2e_ms.append((time.perf_counter() - t1) * 1e3)
    e2e = max_over_ranks(float(np.mean(e2e_ms)), world, eng.device)
    h2d, d2h = sum_over_ranks([h2d, d2h], world, eng.device)  # every rank moves its own shard

    if rank != 0:
        return
    peak, peak_src = peaks()
    clock = sm_clock_hz()
    mean = lambda name: float(np.mean(stage_ms.get(name, [0.0])))  # noqa: E731
    dc_ms = mean("pair_candidates")
    n_incr = last.n_increments
    pair_kernel = getattr(eng, "last_pair_kernel", "pair_candidates_kernel")
    traffic, traffic_src = ncu_traffic(pair_kernel)
    incr_launch = n_incr / world  # per launch: sources (hence increments) are dealt evenly
    # Stage C keeps its counters in shared memory: its ceilings are on chip.  Algorithmic work per increment, fixed in
    # DESIGN.md: one byte counter read + one write = 2 shared-memory lane accesses = 2/32 conflict-free wavefronts
    # (1 wavefront per clock per SM), and 55 warp instructions per 128 cloud entries = 0.43 (4 per clock per SM).
    n_sm = eng.n_sms
    smem_peak = n_sm * clock  # wavefronts/s
    smem_ach = (2.0 / 32.0) * incr_launch / (dc_ms * 1e-3) if dc_ms > 0 else 0.0
    issue_peak = 4.0 * n_sm * clock
    issue_ach = (55.0 / 128.0) * incr_launch / (dc_ms * 1e-3) if dc_ms > 0 else 0.0
    eff_hbm = BYTES_PER_INCREMENT_C * incr_launch / (dc_ms * 1e-3) / 1e9 if dc_ms > 0 else 0.0
    if "docfreq_emit" in stage_ms:  # two kernels: the stage-A figure is their sum
        stage_ms["docfreq"] = [x + y for x, y in zip(stage_ms.get("docfreq_emit", []), stage_ms.get("docfreq_count", []))]
    df_kernel = {"stream": "docfreq_emit_kernel+docfreq_count_kernel", "resident": "docfreq_resident_kernel"}.get(
        eng.docfreq_mode, "docfreq_kernel")
    n_k = int(batch.n_bases - batch.n_reads * (k - 1))
    n_ku = int(units.unit_len.astype(np.int64).sum() - units.n_units * (k - 1))
    csr_last = res[1]
    stage_rooflines = []
    for kern, stage, nbytes, what in (
            (df_kernel, "docfreq", BYTES_PER_KMER_A * n_k, "32.25 B per k-mer occurrence (rank 0's reads)"),
            ("cloud_build_warp_kernel", "cloud_build", 16.25 * n_ku + 4.0 * csr_last.n_entries + 8.0 * units.n_units,
             "16.25 B per k-mer inside a unit + 4 B per cloud entry + 8 B per unit (rank 0's units)"),
            ("pair_join_kernel", "pair_join", 32.0 * last.n_pair_candidates / world + 16.0 * int(last.edges.shape[0]),
             "32 B per pair candidate + 16 B per edge (rank 0's sources)")):
        t_ms = mean(stage)
        if t_ms <= 0:
            continue
        gbs = nbytes / (t_ms * 1e-3) / 1e9
        tr = tr_src = None
        for kk in kern.split("+"):
            x, src = ncu_traffic(kk)
            if x is not None:
                tr, tr_src = (tr or 0.0) + x, src
        stage_rooflines.append({"kernel": kern, "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                "frac": gbs / peak, "traffic": tr, "traffic_source": tr_src, "kernel_ms": t_ms,
                                "algorithmic_bytes": nbytes, "note": what})
    sharding = "single GPU"
    if world > 1:
        sharding = ("reads sharded by record; stage A: phase-1 records all-to-all by hash-partition range, phase 2 on the "
                    "owned partitions, rare keys all-gathered; cloud CSR all-gathered; source k-mers dealt round-robin, "
                    "edges stay with their source's rank")
    workload = C["label"]
    if world > 1:
        workload += (f"; weak scaling: {world} such arrays (reference simulator, seeds 1..{world}; arrays 2.. on their own units, "
                     f"DXZ1 with 30% of the bases substituted), reads of every array dealt to {world} ranks"
                     if args.config == "cenx" else f"; strong scaling: the one read set sharded over {world} ranks")
    line = {
        "metric": "k-mer recruitment read-bases/s", "value": n_bases_total / (ms * 1e-3), "unit": "read-bases/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if args.config == "cenx" else "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload, "scale": args.scale, "read_bases": int(n_bases_total),
                   "reads_rank0": int(batch.n_reads), "units_rank0": int(units.n_units), "rare_kmers": int(res[0].n),
                   "cloud_entries_rank0": int(csr_last.n_entries), "pair_increments": int(n_incr),
                   "candidates": int(last.n_candidates), "pair_candidates": int(last.n_pair_candidates),
                   "edges": n_edges_total, "unique_kmers": int(last.selected.numel()),
                   "l2": "256 MiB flush write between timed steps", "sharding": sharding},
        "roofline": {"kernel": pair_kernel, "bound": "smem", "achieved": smem_ach / 1e9, "peak": smem_peak / 1e9,
                     "unit": "Gwavefronts/s", "frac": smem_ach / smem_peak, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": "148 SMs x 1 shared-memory wavefront per clock at the measured max SM clock",
                     "kernel_ms": dc_ms, "algorithmic_units": incr_launch,
                     "issue": {"achieved_ginst_s": issue_ach / 1e9, "peak_ginst_s": issue_peak / 1e9,
                               "frac": issue_ach / issue_peak, "note": "55 warp instructions per 128 cloud entries"},
                     "effective_hbm": {"achieved": eff_hbm, "peak": peak, "unit": "GB/s", "frac": eff_hbm / peak,
                                       "peak_source": peak_src,
                                       "note": "32 B per pair increment (BASELINE.md §4) -- an EFFECTIVE figure: the "
                                               "counters never leave the SM (DRAM traffic, `traffic`, is ~1000x lower), "
                                               "so it is not a roofline fraction"},
                     "note": "2 shared-memory lane accesses per pair increment = 1/16 conflict-free wavefront; the kernel "
                             "lives on shared memory and issue slots (profiles/), not on HBM"},
        "roofline_other_kernels": stage_rooflines,
        "stage_ms": {name: float(np.mean(v)) for name, v in stage_ms.items()},
        "e2e": {"value": n_bases_total / (e2e * 1e-3), "unit": "read-bases/s", "ms_per_step": e2e,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": launches, "clocks": clk.summary(),
    }
    if parity_ok is not None:
        line["parity_ok"], line["parity"] = parity_ok, parity
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(batch, units, P, bounded_s=args.cpu_seconds)
        with tempfile.TemporaryDirectory() as tmp:
            report_fn = os.path.join(tmp, "report.ncrf")
            from centroflye_b200 import synth
            synth.write_ncrf_report(report_fn, reads_list, unit)
            line["e2e_cli"] = e2e_cli(report_fn, tmp, P, n_bases_total)
            line["cpu_baseline_t0"] = cpu_baseline_t0(reads_list, unit, tmp, P)
    print(json.dumps(line), flush=True)


def e2e_cli(report_fn, tmp, P, n_bases):
    """The drop-in command line, report file on disk -> the two output files (dbkr.py:174-208), wall clock."""
    from centroflye_b200 import distance_based_kmer_recruitment as dbkr
    outdir = os.path.join(tmp, "out")
    argv = ["--ncrf", report_fn, "--coverage", str(P["coverage"]), "--min-coverage", str(P["min_coverage"]),
            "--outdir", outdir, "-k", str(P["k"]), "--max-distance", str(P["max_d"]), "--bottom", str(P["bottom"]),
            "--top", str(P["top"]), "--kmer-survival-rate", str(P["kmer_survival_rate"]), "--max-nonuniq", str(P["max_nonuniq"])]
    best = None
    for _ in range(2):  # the second call has warm allocator pools and file cache, like the second read of a pipeline
        t = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):  # the command line is verbose by default, like the reference's
            dbkr.main(argv)
        dt = time.perf_counter() - t
        if best is None or dt < best[0]:
            best = (dt, dict(dbkr.LAST_TIMINGS))
    sizes = {f: os.path.getsize(os.path.join(outdir, f)) for f in sorted(os.listdir(outdir))}
    return {"value": n_bases / best[0], "unit": "read-bases/s", "seconds": best[0], "stage_s": best[1],
            "report_bytes": os.path.getsize(report_fn), "output_bytes": sizes,
            "what": "centroflye_b200.distance_based_kmer_recruitment.main(argv): NCRF report on disk -> "
                    "unique_kmers_*.txt + unique_edges_*.txt on disk; best of 2 calls"}


def cpu_baseline(batch, units, P, bounded_s=20.0, threads=1):
    """The oracle's C restatement (oracle/c) timed on the host on a bounded sample of the same workload."""
    from oracle import c_oracle
    return c_oracle.timed_sample(batch, units, P, band(P), bounded_s=bounded_s, threads=threads)


def cpu_baseline_t0(reads_list, unit, tmp, P):
    """The UNMODIFIED reference (baseline/_ref) on one core, stage by stage, on a bounded sample of the same reads."""
    from baseline import t0
    if not t0.available():
        return {"kind": "reference", "unavailable": "baseline/_ref is missing (python baseline/make_ref.py in the build container)"}
    from centroflye_b200 import synth
    fn = os.path.join(tmp, "t0_sample.ncrf")
    synth.write_ncrf_report(fn, reads_list[:64], unit)
    out = t0.run(fn, P["k"], P["max_nonuniq"], P["min_d"], P["max_d"], P["min_coverage"])
    out["sample"] = ("first 60 records of the bench's own report for stage A, first 12 for stage B, stage C/D on the "
                     "clouds of the first reads with max_d cut to keep the increments bounded; rates, not a whole-job time")
    return out


# ---- the streaming config (stage A only) ------------------------------------------------------------------------
def run_stream(args):
    import torch
    from centroflye_b200.engine import Engine
    world, rank, local = init_dist()
    eng = Engine(f"cuda:{local}")
    C = CONFIGS["stream"]
    P = C["params"]
    k = P["k"]
    lo, hi = band(P)
    barrier = make_barrier(world)
    n_distinct = max(1, min(args.stream_batches, args.steps))
    t0 = time.time()
    batches = []
    for j in range(n_distinct):  # global batch index of this rank's j-th batch: rank + j * world
        unit, batch, units = simulate("stream", args.scale, 0, 1, n_arrays=1, read_seed_shift=rank + j * world)
        batches.append((batch, eng.upload_reads(batch, k)))
    log(f"[bench] rank {rank}: {n_distinct} batches in {time.time() - t0:.1f}s: "
        f"{[b.n_bases for b, _ in batches]} bases")
    n_k_max = max(int(b.n_bases - b.n_reads * (k - 1)) for b, _ in batches)
    table_buf = torch.empty(2 * n_k_max, dtype=torch.int64, device=eng.device)  # distinct k-mers <= occurrences
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=eng.device)
    bnd = (lo, hi, P["max_nonuniq"])

    def step(i):
        batch, reads = batches[i % n_distinct]
        out = eng.docfreq_stream(reads, k, band=bnd, want_table=True, table_buf=table_buf)
        if out is None:
            raise SystemExit("stage A fell back to the single-kernel form: not the streaming path")
        return batch, out

    parity = None
    if args.check:  # batch 0 of rank 0 is configs[1]: the streaming kernels against the single-kernel form on it
        batch, (rare, table) = step(0)
        eng.docfreq_mode = "resident"
        want = eng.rare_kmers(batches[0][1], k, lo, hi, P["max_nonuniq"])
        tr = eng.count_docfreq(batches[0][1], k)
        eng.docfreq_mode = "stream"
        srt = lambda x: np.sort(x.cpu().numpy().view(np.uint64))  # noqa: E731
        ks, rs, ms_ = (x.cpu().numpy() for x in eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True))
        kr, rr, mr = (x.cpu().numpy() for x in eng.table_select(tr, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True))
        o1, o2 = np.argsort(ks.view(np.uint64)), np.argsort(kr.view(np.uint64))
        parity = {"rare_equal": bool(np.array_equal(srt(rare), srt(want))),
                  "table_equal": bool(np.array_equal(ks[o1], kr[o2]) and np.array_equal(rs[o1], rr[o2]) and
                                      np.array_equal(ms_[o1], mr[o2])),
                  "distinct_kmers": int(ks.size), "rare_kmers": int(rare.numel()),
                  "checker": "docfreq_resident_kernel (the single-kernel form, itself checked against the oracle in tests/)"}
        del tr
    tables = [table_buf, torch.empty_like(table_buf)]
    prev = None
    for i in range(args.warmup + 1):  # warm-up through the pipelined path (allocator pools, partition-buffer sizes)
        h = eng.docfreq_stream_launch(batches[i % n_distinct][1], k, band=bnd, table_buf=tables[i & 1])
        if prev is not None:
            eng.docfreq_stream_finish(prev)
        prev = h
    eng.docfreq_stream_finish(prev)
    barrier()
    # The timed region is ONE stream of K batches: batch i + 1 is enqueued before batch i's counters are read back (two
    # count tables alternate), so the GPU never waits for the host.  No L2 flush in here: a batch's working set (0.9 GB
    # of records + 38 MB of packed reads) is several times the 126 MB L2.
    stage_ms, bases, kmers = {}, 0, 0
    launches0 = eng.launch_count()
    with ClockSampler(local, world, rank) as clk:
        flush.fill_(1)
        barrier()
        eng.events = []
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        prev = None
        for i in range(args.steps):
            batch, reads = batches[i % n_distinct]
            h = eng.docfreq_stream_launch(reads, k, band=bnd, table_buf=tables[i & 1])
            if prev is not None:
                eng.docfreq_stream_finish(prev)
            prev = h
            bases += batch.n_bases
            kmers += int(batch.n_bases - batch.n_reads * (k - 1))
        last = eng.docfreq_stream_finish(prev)
        b.record()
        barrier()
        step_ms = [a.elapsed_time(b) / max(args.steps, 1)] * args.steps
        for name, ms in eng.stage_times_ms().items():
            stage_ms[name] = [ms / max(args.steps, 1)]
        eng.events = None
        if getattr(eng, "stream_fallbacks", 0):
            raise SystemExit("stage A fell back to the single-kernel form inside the timed region")
    launches = (eng.launch_count() - launches0) / max(args.steps, 1)
    if args.dump_outputs:  # the last batch's rare keys and its whole count table (key, n_reads, n_multi)
        rare, table = last
        keys, n_reads, n_multi = (x.cpu().numpy().view(np.uint32 if x.element_size() == 4 else np.uint64)
                                  for x in eng.table_select(table, 0, 0xFFFFFFFF, 0xFFFFFFFF, with_counts=True))
        dump_outputs(args.dump_outputs, {
            "rare_kmers": np.sort(rare.cpu().numpy().view(np.uint64)),
            "count_table": sorted_rows(np.stack([keys, n_reads.astype(np.uint64), n_multi.astype(np.uint64)], axis=1))},
            rank, world)
    # end to end: the batch's packed reads from pinned host memory, the rare keys and the table's size back
    e2e_ms, h2d, d2h = [], 0, 0
    for i in range(1 + max(2, min(args.steps, 3))):
        barrier()
        t1 = time.perf_counter()
        batch = batches[i % n_distinct][0]
        reads = eng.upload_reads(batch, k)
        rare, table = eng.docfreq_stream(reads, k, band=bnd, want_table=True, table_buf=table_buf)
        home = eng.to_host(rare_keys=rare)
        barrier()
        if i:
            e2e_ms.append((time.perf_counter() - t1) * 1e3)
        h2d, d2h = reads.h2d_bytes, sum(t.numel() * t.element_size() for t in home.values())
    total_s = max_over_ranks(float(np.sum(step_ms)) * 1e-3, world, eng.device)
    e2e_s = max_over_ranks(float(np.mean(e2e_ms)) * 1e-3, world, eng.device)
    bases_all, kmers_all, h2d_all, d2h_all = sum_over_ranks([bases, kmers, h2d, d2h], world, eng.device)
    if rank != 0:
        return
    peak, peak_src = peaks()
    mean = lambda name: float(np.mean(stage_ms.get(name, [0.0])))  # noqa: E731
    kern_ms = mean("docfreq_emit") + mean("docfreq_count")
    alg = BYTES_PER_KMER_A * kmers / max(args.steps, 1)  # per batch of rank 0
    ach = alg / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
    tr = None
    tr_src = None
    for kk in ("docfreq_emit_kernel", "docfreq_count_kernel"):
        x, src = ncu_traffic(kk)
        if x is not None:
            tr, tr_src = (tr or 0.0) + x, src
    line = {
        "metric": "k-mer recruitment read-bases/s", "value": bases_all / total_s, "unit": "read-bases/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_s * 1e3 / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": C["label"] + f"; batches dealt round-robin to {world} GPU(s), no collective; {n_distinct} "
                   f"distinct batch(es) per GPU resident in HBM and cycled over {args.steps} steps", "scale": args.scale,
                   "bases_per_batch": int(bases / max(args.steps, 1)), "batches": int(args.steps * world),
                   "l2": "inputs larger than L2: a batch's working set is 0.9 GB of records + 38 MB of packed reads (L2: 126 MB); "
                         "one 256 MiB flush write before the timed stream",
                   "pipelining": "batch i + 1 is enqueued before batch i's counters are read back; two count tables alternate",
                   "sharding": "replicas only: independent batches, one process per GPU"},
        "roofline": {"kernel": "docfreq_emit_kernel+docfreq_count_kernel", "bound": "hbm", "achieved": ach, "peak": peak,
                     "unit": "GB/s", "frac": ach / peak if peak else None, "traffic": tr, "traffic_source": tr_src,
                     "peak_source": peak_src, "kernel_ms": kern_ms, "algorithmic_bytes": alg,
                     "frac_of_nominal_8TBs": ach / 8000.0,
                     "note": "32.25 B per k-mer occurrence (SURVEY.md §8d): 0.25 B of packed read + one 16-byte slot read "
                             "and written; the kernels move less than that (traffic) because the per-read sets and the "
                             "per-partition tables live in shared memory -- they are bound by issue slots and "
                             "shared-memory atomics, see profiles/"},
        "stage_ms": {name: float(np.mean(v)) for name, v in stage_ms.items()},
        "e2e": {"value": bases_all / max(args.steps, 1) / e2e_s, "unit": "read-bases/s", "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all)},
        "gpu_launches": launches, "clocks": clk.summary(),
    }
    if parity is not None:
        line["parity_ok"], line["parity"] = bool(parity["rare_equal"] and parity["table_equal"]), parity
    print(json.dumps(line), flush=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle
    cfg = "cenx" if args.config == "stream" else args.config
    P = CONFIGS[cfg]["params"]
    world = max(1, args.gpus)
    threads = os.cpu_count() or 1
    # The whole job's input.  cenx at N GPUs = N arrays that share no k-mers (their own units), so the job IS N independent
    # recruitments and its CPU time is the sum of theirs: step i times array i mod N in full for stages A and B and a
    # bounded sample of its stage C/D (the memory of one array), and reports the rate.  The stage-C budget per step is cut
    # so that the whole --steps K --warmup W run stays within a few minutes.
    n_jobs = world if cfg == "cenx" else 1
    inputs = [simulate(cfg, args.scale, 0, 1, n_arrays=1, first_array=j)[1:] for j in range(n_jobs)]
    budget = max(2.0, min(args.cpu_seconds, 120.0 / max(1, args.warmup + args.steps)))
    vals = []
    for i in range(args.warmup + args.steps):
        batch, units = inputs[i % n_jobs]
        res = c_oracle.timed_sample(batch, units, P, band(P), bounded_s=budget, threads=threads)
        if i >= args.warmup:
            if n_jobs > 1:
                res["sample"] = (f"array {i % n_jobs} of the {n_jobs} independent arrays of the job (step i takes array i mod "
                                 f"{n_jobs}; the job's CPU time is the sum over its arrays, its rate the one reported): " + res["sample"])
            res["read_bases"] = int(batch.n_bases)
            vals.append(res)
    batch_bases = sum(int(b.n_bases) for b, _ in inputs)
    if args.config == "stream":  # stage A only
        v = float(np.mean([r["read_bases"] / r["stage_s"]["A"] for r in vals]))
        ms = float(np.mean([r["stage_s"]["A"] for r in vals])) * 1e3
    else:
        v = float(np.mean([r["value"] for r in vals]))
        ms = float(np.mean([r["ms"] for r in vals]))
    if n_jobs > 1:  # the job = all its arrays: its time is the sum over arrays (estimated from the ones timed), same rate
        ms = ms * n_jobs
        v = batch_bases / (ms * 1e-3)
    line = {"impl": "reference", "metric": "k-mer recruitment read-bases/s", "value": v, "unit": "read-bases/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak" if args.config != "cen6" else "strong", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": CONFIGS[args.config]["label"] + (f"; {world} such arrays" if world > 1 and cfg == "cenx" else "")
                       + " (bounded sample, see cpu_baseline.sample)", "scale": args.scale, "read_bases": int(batch_bases)},
            "cpu_baseline": dict(vals[-1], value=v),
            "e2e": {"value": v, "unit": "read-bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cenx", choices=sorted(CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", dest="check", action="store_false", help="skip the parity leg")
    ap.add_argument("--stream-batches", type=int, default=2, help="distinct batches per GPU kept resident (stream)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path returns: use it with --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "stream":
        run_stream(args)
    else:
        run_recruit(args)


if __name__ == "__main__":
    main()
