#!/usr/bin/env python
"""bench.py — reads/sec of the mtsv-binner read-assignment hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle on all host cores

Workload (BASELINE.json configs[1]): one ~1 Gbp MG-index chunk (200 synthetic genomes x 5 Mbp, 10 % of
each genome shared with an earlier genome at 1 % divergence, 0.1 % N), default binner flags, 150 bp
reads (90 % from the reference with 2 % substitutions and 0.5 % indels, half reverse-complemented; 10 %
random).  The index is replicated on every GPU and each GPU bins its own 10 M reads per step (weak
scaling, no data-path collective: reads are independent units).  One step = one pass of the hot path
over one such batch.  `value` = reads/s with the reads already resident in HBM (mtsvgpu_bin_batch_device);
`e2e` = the same through mtsvgpu_bin_batch with pinned HOST buffers, H2D of the reads and D2H of the
hits inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (n_genomes, genome_len, shared_frac, divergence, reads, read_len, flags)
    "cfg2": dict(n_seqs=200, seq_len=5_000_000, shared=0.10, div=0.01, reads=10_000_000, read_len=150,
                 flags={}, label="cfg2: 1 Gbp chunk (200 x 5 Mbp), 150 bp reads, default flags"),
    "cfg1": dict(n_seqs=52, seq_len=192_308, shared=0.0, div=0.0, reads=100_000, read_len=150,
                 flags={}, label="cfg1: 10 Mbp reference, 100k x 150 bp reads, default flags"),
    # config 4: 75 bp reads against a highly redundant reference (500 near-identical strains, distinct TaxIDs):
    # large SA intervals, tune-max-hits doubling, hundreds of candidates per read
    "cfg4": dict(n_seqs=500, seq_len=2_000_000, shared=0.0, div=0.0, strains=dict(base_len=2_000_000, div=0.003),
                 reads=2_000_000, read_len=75, flags={},
                 label="cfg4: 500 strains x 2 Mbp at 0.3 % divergence, 75 bp reads, default flags"),
    # config 4 with the strains filed under 50 species TaxIDs (ten genomes each), the way reference databases carry
    # many assemblies per TaxID: the reference stops a TaxID at its first passing window (src/index.rs:393-396)
    "cfg4b": dict(n_seqs=500, seq_len=2_000_000, shared=0.0, div=0.0, strains=dict(base_len=2_000_000, div=0.003),
                  per_taxid=10, reads=2_000_000, read_len=75, flags={},
                  label="cfg4b: 500 strains x 2 Mbp at 0.3 % divergence under 50 TaxIDs, 75 bp reads, default flags"),
    # config 5: 250 bp reads at edit-rate 0.2 with dense seeding: verifier stress
    "cfg5": dict(n_seqs=40, seq_len=5_000_000, shared=0.10, div=0.01, reads=2_000_000, read_len=250,
                 flags=dict(edit_rate=0.2, seed_gap=3), read_sub=0.12,
                 label="cfg5: 200 Mbp chunk, 250 bp reads mutated 12 %, --edit-rate 0.2 --seed-interval 3"),
    "cfg2s": dict(n_seqs=40, seq_len=5_000_000, shared=0.10, div=0.01, reads=2_000_000, read_len=150,
                  flags={}, label="cfg2s: 200 Mbp chunk (40 x 5 Mbp), 150 bp reads, default flags"),
}
CACHE_DIR = os.environ.get("MTSV_B200_CACHE", os.path.join(tempfile.gettempdir(), "mtsv_b200_cache"))


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------
# data
# ------------------------------------------------------------------------------------------------
def make_reference_torch(cfg, seed, device):
    """i.i.d. ACGT genomes + shared diverged segments + N runs, generated on `device`."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    n_seqs, seq_len = cfg["n_seqs"], cfg["seq_len"]
    total = n_seqs * seq_len
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=device)
    cat = torch.empty(total, dtype=torch.uint8, device=device)
    step = 1 << 28
    for b in range(0, total, step):
        e = min(total, b + step)
        cat[b:e] = acgt[torch.randint(0, 4, (e - b,), generator=g, device=device)]
    rng = np.random.default_rng(seed)
    if cfg.get("strains"):
        # every sequence is a mutated copy of the first one (near-identical strains)
        base = cat[:seq_len].clone()
        nmut = int(seq_len * cfg["strains"]["div"])
        for i in range(1, n_seqs):
            piece = base.clone()
            pos = torch.randint(0, seq_len, (nmut,), generator=g, device=device)
            piece[pos] = acgt[torch.randint(0, 4, (nmut,), generator=g, device=device)]
            cat[i * seq_len:(i + 1) * seq_len] = piece
    if cfg["shared"] > 0:
        seg = int(seq_len * cfg["shared"])
        for i in range(1, n_seqs):
            src = int(rng.integers(0, i))
            so = int(rng.integers(0, seq_len - seg + 1))
            do = int(rng.integers(0, seq_len - seg + 1))
            piece = cat[src * seq_len + so: src * seq_len + so + seg].clone()
            nmut = int(seg * cfg["div"])
            if nmut:
                pos = torch.randint(0, seg, (nmut,), generator=g, device=device)
                piece[pos] = acgt[torch.randint(0, 4, (nmut,), generator=g, device=device)]
            cat[i * seq_len + do: i * seq_len + do + seg] = piece
    # N runs: 0.1 % of the bases in runs of 10-50
    n_runs = int(total * 0.001 / 30)
    if n_runs:
        pos = torch.randint(0, total - 64, (n_runs,), generator=g, device=device)
        ln = torch.randint(10, 51, (n_runs,), generator=g, device=device)
        idx = pos[:, None] + torch.arange(50, device=device)[None, :]
        m = torch.arange(50, device=device)[None, :] < ln[:, None]
        cat[idx[m]] = ord("N")
    off = np.arange(n_seqs + 1, dtype=np.uint64) * np.uint64(seq_len)
    gi = np.arange(1, n_seqs + 1, dtype=np.uint32)
    tax = (1000 + np.arange(n_seqs) // cfg.get("per_taxid", 1)).astype(np.uint32)
    return cat, off, gi, tax


def index_file_path(name, cfg):
    return os.path.join(CACHE_DIR, "%s_seed%d.index" % (name, cfg.get("seed", 3)))


def ensure_index_file(name, cfg, local_rank, rank, barrier):
    """The workload's `.index` file, as mtsv-build would leave it: reference generated on the GPU, index built by
    the library's device builder (mtsvgpu_index_build: hand-written suffix sort + BWT kernels) and written as the
    bincode MGIndex a reference mtsv-binner reads (mtsvgpu_index_write).  Cached per box under CACHE_DIR."""
    import torch
    from mtsv_tools_b200 import MGIndex
    path = index_file_path(name, cfg)
    done = path + ".done.json"
    if rank == 0 and not os.path.exists(done):
        os.makedirs(CACHE_DIR, exist_ok=True)
        t0 = time.time()
        cat, off, gi, tax = make_reference_torch(cfg, cfg.get("seed", 3), "cuda:%d" % local_rank)
        torch.cuda.synchronize()
        t1 = time.time()
        with MGIndex.build(cat.data_ptr(), off, gi, tax, device=local_rank, ktab_k=0xFFFFFFFF) as g:
            del cat
            torch.cuda.empty_cache()
            t2 = time.time()
            info = g.info()
            g.write(path, 64, 32)
        t3 = time.time()
        meta = {"reference_gen_seconds": t1 - t0, "build_seconds": info["build_seconds"],
                "build_call_seconds": t2 - t1, "write_seconds": t3 - t2, "text_len": info["text_len"],
                "file_bytes": os.path.getsize(path)}
        log("index built on the GPU: %s" % meta)
        json.dump(meta, open(done, "w"))
    barrier()
    return path, json.load(open(done))


def index_file_text_and_bins(path):
    """Header of the bincode MGIndex (src/index.rs:60-68): sequences (memory-mapped) and the bins."""
    n = int(np.fromfile(path, dtype="<u8", count=1)[0])
    text = np.memmap(path, dtype=np.uint8, mode="r", offset=8, shape=(n,))
    nb = int(np.fromfile(path, dtype="<u8", count=1, offset=8 + n)[0])
    rec = np.fromfile(path, dtype=np.dtype([("gi", "<u4"), ("tax", "<u4"), ("start", "<u8"), ("end", "<u8")]),
                      count=nb, offset=16 + n)
    ref_off = np.concatenate([rec["start"], rec["end"][-1:]]).astype(np.uint64)
    return text, rec, ref_off


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------------------------------------
# shared by both arms
# ------------------------------------------------------------------------------------------------
METRIC = "reads/sec binned (150 bp)"


def config_dict(name, cfg, n_reads):
    """Identical in the GPU arm and the reference arm: what the workload IS (not how an arm ran it)."""
    return {"workload": cfg["label"], "config": name, "reads_per_gpu_per_step": int(n_reads),
            "read_len": cfg["read_len"], "index_mbp": cfg["n_seqs"] * cfg["seq_len"] / 1e6,
            "flags": cfg["flags"] or "defaults", "index_replicated": True,
            "l2_note": "index and per-step read batch exceed the 126 MB L2 (different reads every sub-batch)"}


def make_reads(cfg, ref_t, ref_off, n_reads, seed, dev, ragged=False):
    """Reads of the workload on `dev`: (uint8 bytes tensor, int64 offsets tensor).  ragged: every read trimmed
    at its 3' end to a length drawn uniformly from [2/3 L, L] (adapter / quality trimming)."""
    import torch
    from mtsv_tools_b200 import synth
    L = cfg["read_len"]
    flat = synth.make_reads_torch(ref_t, ref_off, n_reads, L, seed, dev, sub=cfg.get("read_sub", 0.02))
    if not ragged:
        return flat, torch.arange(n_reads + 1, dtype=torch.int64, device=dev) * L
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 991)
    lens = torch.randint(2 * L // 3, L + 1, (n_reads,), generator=g, device=dev)
    keep = torch.arange(L, device=dev)[None, :] < lens[:, None]
    out = flat.view(n_reads, L)[keep]
    off = torch.zeros(n_reads + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(lens, 0)
    return out.contiguous(), off


def oracle_rate(oix, pyoracle, reads_np, off_np, params, seconds, cores, counters=None):
    """Times the CPU restatement on a bounded prefix of (reads_np, off_np): about `seconds` of work."""
    n_all = len(off_np) - 1
    probe = min(n_all, 1000)
    t0 = time.time()
    oix.bin_reads((reads_np[:int(off_np[probe])], off_np[:probe + 1]), params, threads=cores)
    rate = probe / max(time.time() - t0, 1e-6)
    if rate * seconds > 8 * probe:  # a probe that short under-estimates a fast config: probe again, longer
        probe = min(n_all, 20000)
        t0 = time.time()
        oix.bin_reads((reads_np[:int(off_np[probe])], off_np[:probe + 1]), params, threads=cores)
        rate = probe / max(time.time() - t0, 1e-6)
    ns = int(min(n_all, max(probe, rate * seconds)))
    t0 = time.time()
    h, _ = oix.bin_reads((reads_np[:int(off_np[ns])], off_np[:ns + 1]), params, threads=cores, counters=counters)
    dt = time.time() - t0
    return ns, dt, len(h)


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def run_reference_arm(args, name, cfg, rank, world):
    """The reference's CPU implementation of the path = the oracle (the Rust binary cannot be built in
    this image: no cargo/rustc), with the reference's own ssw.c, on all host cores."""
    if rank != 0:
        return
    import torch
    from oracle import pyoracle
    cores = os.cpu_count() or 1
    path, _meta = ensure_index_file(name, cfg, 0, 0, lambda: None)
    t0 = time.time()
    oix = pyoracle.Index.read(path)
    log("oracle index read from %s in %.1fs" % (path, time.time() - t0))
    text, _bins, ref_off = index_file_text_and_bins(path)
    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    ref_t = torch.from_numpy(np.array(text[:-1])).to(dev)
    n_reads = args.reads or cfg["reads"]
    params = pyoracle.default_params(**cfg["flags"])
    # same generator, same seed as rank 0 of the GPU arm: the sample is a prefix of the very same reads
    n_gen = int(min(n_reads, 1 << 21))  # (whole generator chunks: the same reads as the GPU arm's first 2 Mi)
    r_t, o_t = make_reads(cfg, ref_t, ref_off, n_gen, 4, dev)
    reads, off = r_t.cpu().numpy(), o_t.cpu().numpy().astype(np.uint64)
    del ref_t, r_t, o_t
    ns, dt1, _ = oracle_rate(oix, pyoracle, reads, off, params, args.ref_seconds, cores)
    sub = (reads[:int(off[ns])], off[:ns + 1])
    for _ in range(min(args.warmup, 1)):
        oix.bin_reads((reads[:int(off[min(ns, 20000)])], off[:min(ns, 20000) + 1]), params, threads=cores)
    t0 = time.time()
    n_hits = 0
    for _ in range(args.steps):
        h, o = oix.bin_reads(sub, params, threads=cores)
        n_hits = len(h)
    dt = time.time() - t0
    value = ns * args.steps / dt
    sample = "first %d of the step's %d reads (same generator, seed and index file as the GPU arm)" % (ns, n_reads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "reads/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32 integer", "data": "synthetic",
        "config": config_dict(name, cfg, n_reads),
        "run": {"sampled_reads_per_step": ns, "threads": cores, "hits_per_step": n_hits,
                "note": "the CPU arm does not depend on --gpus: one host, all its cores"},
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "C++ restatement of src/index.rs:258-432 + reference ssw.c (oracle/); "
                                 "the Rust mtsv-binner cannot be built here (no cargo/rustc)"},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's host threads (and, by first touch, its page-locked buffers) to the CPUs NVML reports as
    local to its GPU: at N = 8 the uploads of 8 ranks otherwise cross the socket interconnect."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode() if hasattr(bus, "encode") else bus)
        n = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = [i for i in range(n) if (int(mask[i // 64]) >> (i % 64)) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return "%d cpus local to %s" % (len(allowed), bus)
    except Exception as e:  # no NVML / no affinity support: run unbound
        return "unbound (%s)" % (e,)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, rank, world, local_rank):
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dev = "cuda:%d" % local_rank

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def max_over_ranks(self, vals):
        if self.world == 1:
            return [float(v) for v in vals]
        import torch
        import torch.distributed as dist
        t = torch.tensor(list(vals), dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]


class Workload:
    """One config on one rank: the index opened from its `.index` file, this rank's reads on the device and in
    page-locked host memory."""

    def __init__(self, args, name, cfg, ctx, ragged=False, n_reads=None):
        import torch
        from mtsv_tools_b200 import MGIndex, Params
        self.name, self.cfg, self.ctx, self.ragged = name, cfg, ctx, ragged
        self.path, self.build_meta = ensure_index_file(name, cfg, ctx.local_rank, ctx.rank, ctx.barrier)
        t0 = time.time()
        # the drop-in's own way in: mtsvgpu_index_open on the `.index` file (parse, upload, re-layout; nothing rebuilt)
        self.gix = MGIndex.from_file(self.path, device=ctx.local_rank, sa_rate=args.sa_rate, ktab_k=args.ktab_k,
                                     batch_reads=args.batch_reads)
        self.info = self.gix.info()
        log("rank %d: %s opened in %.1fs (relayout %.2fs), %.2f GB HBM, sa_rate %d, ktab k=%d" %
            (ctx.rank, self.path, time.time() - t0, self.info["relayout_seconds"], self.info["device_bytes"] / 1e9,
             self.info["device_sa_rate"], self.info["ktab_k"]))
        text, _bins, ref_off = index_file_text_and_bins(self.path)
        self.L = cfg["read_len"]
        self.n_reads = n_reads or args.reads or cfg["reads"]
        ref_t = torch.from_numpy(np.array(text[:-1])).to(ctx.dev)
        t0 = time.time()
        self.d_reads, self.d_off = make_reads(cfg, ref_t, ref_off, self.n_reads, 4 + 17 * ctx.rank, ctx.dev, ragged)
        del ref_t
        torch.cuda.synchronize()
        log("rank %d: %d reads generated on device in %.1fs" % (ctx.rank, self.n_reads, time.time() - t0))
        # pinned host copies for the end-to-end leg
        self.h_reads = torch.empty(self.d_reads.numel(), dtype=torch.uint8, pin_memory=True)
        self.h_reads.copy_(self.d_reads)
        self.h_off = torch.empty(self.n_reads + 1, dtype=torch.int64, pin_memory=True)
        self.h_off.copy_(self.d_off)
        torch.cuda.synchronize()
        self.params = Params(**cfg["flags"])
        self.stream = torch.cuda.current_stream()
        self.gix.set_stream(self.stream.cuda_stream)
        self.oix = None

    def host_views(self, n=None):
        n = self.n_reads if n is None else n
        ho = self.h_off.numpy().view(np.uint64)[:n + 1]
        return self.h_reads.numpy()[:int(ho[n])], ho

    def oracle(self):
        if self.oix is None:
            from oracle import pyoracle
            self.oix = pyoracle.Index.read(self.path)
        return self.oix

    def close(self):
        import torch
        self.gix.close()
        self.oix = None
        del self.d_reads, self.d_off, self.h_reads, self.h_off
        torch.cuda.empty_cache()


def parity_gate(args, w):
    """GPU vs oracle on a prefix of rank 0's reads before any timing: bit-exact or no number."""
    from oracle import pyoracle
    ns = min(args.parity_reads if w.name in ("cfg2", "cfg1") else min(args.parity_reads, 20000), w.n_reads)
    t0 = time.time()
    oix = w.oracle()
    sub = w.host_views(ns)
    octr = pyoracle.Counters()
    want_h, want_o = oix.bin_reads(sub, pyoracle.default_params(**w.cfg["flags"]), threads=os.cpu_count(), counters=octr)
    got_h, got_o = w.gix.bin_reads(sub, w.params)
    gst = w.gix.last_batch_stats()
    ok = np.array_equal(want_o, got_o) and all(np.array_equal(want_h[f], got_h[f])
                                               for f in ("tax_id", "gi", "offset", "edit"))
    oc = octr.as_dict()
    # work cross-check against the reference algorithm's own counters: rows located and candidates verified
    # (the GPU path skips strands that cannot be accepted: more N than the edit budget, core.cuh::query_hopeless)
    parity = {"reads": ns, "hits": int(len(want_h)), "bit_exact": bool(ok),
              "rows_located": {"oracle": int(oc["rows_located"]), "gpu": gst["n_seed_hits"]},
              "candidates": {"oracle_built": int(oc["candidates"]), "oracle_verified": int(oc["sw_calls"]),
                             "gpu_verified": gst["n_candidates"]}}
    log("parity gate %s: %s (%.1fs)" % (w.name, parity, time.time() - t0))
    if not ok:
        raise SystemExit("bench.py: GPU results differ from the oracle on %s — refusing to report a number" % w.name)
    return parity


def time_device(w, steps, warmup, n=None, profile=True, on_last=None):
    """Device-resident leg: reads already in HBM, results left there.  Returns (ms, stats, stage_ms, launches).
    on_last: called after the timed region with what the last timed step returned (device hits, offsets, count)."""
    import torch
    from mtsv_tools_b200 import load_library
    lib = load_library()
    n = w.n_reads if n is None else n

    def step():
        return w.gix.bin_reads_device(w.d_reads.data_ptr(), w.d_off.data_ptr(), n, w.params)

    w.gix.set_profiling(profile)  # (before the warm-up: the profiled mode runs other slice sizes on one lane)
    for _ in range(warmup):
        step()
    launches0 = lib.mtsvgpu_launch_count()
    torch.cuda.synchronize()
    w.ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms, stats = {}, None
    e0.record(w.stream)
    last = None
    for _ in range(steps):
        last = step()
        if profile:
            stats = w.gix.last_batch_stats()
            for k, v in stats["ms"].items():
                stage_ms[k] = stage_ms.get(k, 0.0) + v
    e1.record(w.stream)
    torch.cuda.synchronize()
    w.ctx.barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.mtsvgpu_launch_count() - launches0
    if on_last is not None:
        on_last(last)  # (before any other call on the handle: the results live in its buffers until then)
    w.gix.set_profiling(False)
    if stats is None:
        stats = w.gix.last_batch_stats()
    return ms, stats, {k: v / steps for k, v in stage_ms.items()}, int(launches)


DUMP_READS = 1 << 16
DUMP_BYTES = 64 << 20


def _device_array(ptr, shape, typestr, dev):
    """A torch view of memory the library owns on `dev` (no copy)."""
    import torch

    class View:
        __cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
    return torch.as_tensor(View(), device=dev)


def dump_outputs(out_dir, w, last):
    """Writes what the timed device-resident call returned in its last step as float64 .npy files under out_dir:
    a fixed, seeded sample of DUMP_READS reads (whole reads, in read order, cut where DUMP_BYTES would be exceeded).
    read_index: the sampled reads; hit_count: hits of each; tax_id, gi, offset, edit: their hits, read by read."""
    import torch
    from mtsv_tools_b200.index import HIT_DTYPE
    d_hits, d_off, n_hits = last
    n = w.n_reads
    off = _device_array(d_off, (n + 1,), "<i8", w.ctx.dev).cpu().numpy().astype(np.int64)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_READS), replace=False))
    cnt = off[idx + 1] - off[idx]
    keep = np.cumsum(2 * 8 + 4 * 8 * cnt) <= DUMP_BYTES
    idx, cnt = idx[keep], cnt[keep]
    pos = np.repeat(off[idx] - np.cumsum(cnt) + cnt, cnt) + np.arange(int(cnt.sum()))
    hits = np.zeros(0, dtype=HIT_DTYPE)
    if len(pos):
        rows = _device_array(d_hits, (int(n_hits), HIT_DTYPE.itemsize), "|u1", w.ctx.dev)
        hits = rows[torch.from_numpy(pos).to(w.ctx.dev)].cpu().numpy().reshape(-1).view(HIT_DTYPE)
    os.makedirs(out_dir, exist_ok=True)
    cols = {"read_index": idx, "hit_count": cnt}
    cols.update((f, hits[f]) for f in ("tax_id", "gi", "offset", "edit"))
    for name, a in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    log("outputs of the last timed step: %d of %d reads, %d hits -> %s" % (len(idx), n, len(hits), out_dir))


def time_e2e(w, steps, n=None):
    """End-to-end leg: mtsvgpu_bin_batch_pinned — pinned host reads in, hits in pinned host memory out, wall clock."""
    import torch
    hr, ho = w.host_views(n)
    for _ in range(2):
        w.gix.bin_reads_pinned((hr, ho), w.params)
    torch.cuda.synchronize()
    w.ctx.barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(steps):
        hits, offs = w.gix.bin_reads_pinned((hr, ho), w.params)
        d2h = hits.nbytes + offs.nbytes
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    # bytes the library actually uploaded per call (seq_off of equal-length slices is generated on the device)
    h2d = int(w.gix.last_batch_stats().get("h2d_bytes", 0)) or int(hr.nbytes + ho.nbytes)
    w.ctx.barrier()
    return e2e_s * 1e3, h2d, int(d2h)


def time_e2e_packed(w, steps, n=None):
    """End-to-end through mtsvgpu_bin_batch_packed.  `packed`: the raw reads start in host memory and the host-side
    pack (mtsvgpu_pack_reads, this rank's share of the host threads) is INSIDE the timed region, every step.
    `prepacked`: the records already exist (a parser that packs while it scans), only the call is timed."""
    import torch
    from mtsv_tools_b200.index import pack_reads_planes
    from mtsv_tools_b200 import load_library
    import ctypes as C
    hr, ho = w.host_views(n)
    n_reads = len(ho) - 1
    nbytes = int(load_library().mtsvgpu_packed_size(C.c_void_p(ho.ctypes.data), n_reads))
    buf_t = torch.empty(max(1, nbytes), dtype=torch.uint8, pin_memory=True)
    buf = buf_t.numpy()
    threads = max(1, (len(os.sched_getaffinity(0)) or 1) // max(1, w.ctx.world if w.ctx.world > 1 else 1))

    def step(pack):
        if pack:
            pack_reads_planes((hr, ho), threads=threads, out=buf)
        return w.gix.bin_reads_packed(buf[:nbytes], ho, w.params)

    out = {}
    for name, pack in (("packed", True), ("prepacked", False)):
        for _ in range(2):
            step(True)
        torch.cuda.synchronize()
        w.ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            hits, offs = step(pack)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        w.ctx.barrier()
        out[name] = (dt * 1e3, int(w.gix.last_batch_stats().get("h2d_bytes", 0)), int(hits.nbytes + offs.nbytes))
    t0 = time.perf_counter()
    pack_reads_planes((hr, ho), threads=threads, out=buf)
    out["pack_ms"] = (time.perf_counter() - t0) * 1e3
    out["pack_threads"] = threads
    del buf, buf_t
    return out


def h2d_ceiling(w):
    """What this box gives plain page-locked uploads: every rank copies its reads buffer host -> device with
    nothing else going on (torch copy_ = one cudaMemcpyAsync), all ranks at once and rank 0 alone."""
    import torch
    nbytes = w.h_reads.numel()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=w.ctx.dev)

    def run(active):
        for _ in range(1):
            if active:
                dst.copy_(w.h_reads, non_blocking=True)
        torch.cuda.synchronize()
        w.ctx.barrier()
        t0 = time.perf_counter()
        if active:
            for _ in range(3):
                dst.copy_(w.h_reads, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        w.ctx.barrier()
        return dt

    dt_all = w.ctx.max_over_ranks([run(True)])[0]
    dt_alone = w.ctx.max_over_ranks([run(w.ctx.rank == 0)])[0]
    del dst
    return {"bytes_per_copy": int(nbytes), "all_ranks_gbs_aggregate": 3 * nbytes * w.ctx.world / dt_all / 1e9,
            "all_ranks_gbs_per_gpu": 3 * nbytes / dt_all / 1e9, "one_rank_alone_gbs": 3 * nbytes / dt_alone / 1e9,
            "how": "3 back-to-back cudaMemcpyAsync of the rank's pinned reads buffer, wall clock, max over ranks"}


def rooflines(w, stats, per_step, ms_per_step, clocks):
    """DESIGN.md §4.  Memory kernels: algorithmic bytes per launch / mean launch duration against the measured HBM
    copy bandwidth.  Verifier: executed ALU-pipe warp instructions / time against the SM integer issue roof."""
    peaks, peak_kind = measured_peaks()
    L = w.L
    n_sub = max(1, int(stats.get("n_sub_batches", 0)) or 1)
    window_cols = float(stats["window_bytes"])  # reference columns (bases) the verifier walks, summed over candidates
    alg_bytes = {
        # index sectors needed (k-mer table + FmBlock sectors, counted in-kernel) + 2 plane words in + 8 B out
        "seed_search": 32.0 * stats["rank_queries"] + (48.0 + 8.0) * stats["n_seed_slots"],
        # one 32-B SA sector per located row + 8 B key out
        "locate": (32.0 + 8.0) * stats["n_seed_hits"],
        # the fast verifier reads the 4-bit text (0.5 B per reference column) + the read's planes + 4 B result
        "verify": 0.5 * window_cols + (24.0 * ((L + 63) // 64) + 4.0) * stats["n_candidates"],
    }
    traffic = {}
    for tp in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tpath):
            try:
                traffic, tsrc = json.load(open(tpath)), tp
                break
            except Exception:
                pass
    fast = L <= 253 and os.environ.get("MTSV_B200_VERIFIER") != "legacy"
    kernel_of = {"verify": "verify_warp_kernel" if fast else "verify_kernel"}

    def hbm_roof(stage, extra):
        ms_k = per_step.get(stage, 0.0)
        ach = alg_bytes[stage] / (ms_k * 1e-3) / 1e9 if ms_k > 0 else 0.0
        kname = kernel_of.get(stage, stage + "_kernel")
        t = traffic.get(kname, {})
        r = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
             "frac": ach / peaks["hbm_gbs"], "traffic": t.get("dram_bytes_per_launch"),
             "peak_source": "%s MEASURED_PEAKS.json hbm_gbs (streaming copy)" % peak_kind,
             "algorithmic_bytes_per_launch": alg_bytes[stage] / n_sub, "launches_per_step": n_sub,
             "kernel_ms_per_launch": ms_k / n_sub, "share_of_step": ms_k / ms_per_step if ms_per_step else None}
        if t:
            r["ncu"] = {k: t.get(k) for k in ("dram_throughput_pct_of_peak", "alu_pipe_pct_of_peak",
                                              "fma_pipe_pct_of_peak", "issue_active_pct")}
            r["ncu"]["source"] = "profiles/%s" % tsrc
            if r["traffic"]:
                r["frac_in_dram_bytes"] = r["traffic"] / (ms_k / n_sub * 1e-3) / 1e9 / peaks["hbm_gbs"] if ms_k else None
        r.update(extra)
        return r

    def alu_roof():
        # SM integer roof: the ALU pipe issues one warp instruction per 2 cycles per scheduler (16 lanes each):
        # 148 SMs x 4 schedulers x 0.5 x clock warp-instructions/s
        ms_k = per_step.get("verify", 0.0)
        kname = kernel_of["verify"]
        t = traffic.get(kname, {})
        mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        peak = 148 * 4 * 0.5 * mhz * 1e6 / 1e9  # G warp-inst/s
        word_steps = ((L + 63) // 64) * window_cols  # SURVEY §8(d): bit-vector word-steps of the full matrices
        r = {"bound": "alu", "kernel": kname, "unit": "G warp-inst/s (ALU pipe)", "peak": peak,
             "peak_source": "148 SMs x 4 schedulers x 1 ALU-pipe warp instruction per 2 cycles x %.0f MHz "
                            "(SM clock sampled under load)" % mhz,
             "traffic": t.get("dram_bytes_per_launch"), "launches_per_step": n_sub,
             "kernel_ms_per_launch": ms_k / n_sub, "share_of_step": ms_k / ms_per_step if ms_per_step else None,
             "algorithmic_word_steps_per_launch": word_steps / n_sub,
             "algorithmic_word_steps_per_s": word_steps / (ms_k * 1e-3) if ms_k else None,
             "hbm_view": {"achieved_gbs": alg_bytes["verify"] / (ms_k * 1e-3) / 1e9 if ms_k else None,
                          "frac_of_hbm_peak": alg_bytes["verify"] / (ms_k * 1e-3) / 1e9 / peaks["hbm_gbs"] if ms_k else None,
                          "note": "memory is not what bounds this kernel"},
             "bound_actual": "SM integer issue: the Myers/Hyyro bit-vector recurrence is LOP3/IADD3/SHF on the ALU pipe"}
        ipc = t.get("alu_warp_inst_per_candidate")
        if ipc and ms_k:
            ach = ipc * stats["n_candidates"] / (ms_k * 1e-3) / 1e9
            r.update({"achieved": ach, "frac": ach / peak,
                      "achieved_how": "ALU-pipe warp instructions per candidate (ncu, profiles/%s) x candidates "
                                      "verified in the timed region / kernel time (CUDA events)" % tsrc})
        elif t.get("alu_pipe_pct_of_peak"):
            f = t["alu_pipe_pct_of_peak"] / 100.0
            r.update({"achieved": f * peak, "frac": f,
                      "achieved_how": "ncu sm__inst_executed_pipe_alu pct_of_peak_sustained_active (profiles/%s)" % tsrc})
        else:
            r.update({"achieved": None, "frac": None})
        return r

    notes = {
        "seed_search": {"bound_actual": "HBM random access: every miss fills a whole 128-B line on this part "
                                        "(tools/randbench2.cu), so DRAM traffic is a multiple of the algorithmic "
                                        "sectors; frac_in_dram_bytes is the share of the copy peak the kernel really moves",
                        "random_line_ceiling_per_s": 4.6e10},
        "locate": {"bound_actual": "HBM random access (128-B line fills), see seed_search"},
    }
    dom = max(alg_bytes, key=lambda k: per_step.get(k, 0.0))
    roofline = alu_roof() if dom == "verify" else hbm_roof(dom, notes.get(dom, {}))
    mem_dom = max(("seed_search", "locate"), key=lambda k: per_step.get(k, 0.0))
    return roofline, hbm_roof(mem_dom, notes.get(mem_dom, {}))


def cpu_baseline(args, w, seconds):
    from oracle import pyoracle
    cores = os.cpu_count() or 1
    hr, ho = w.host_views(min(w.n_reads, 1 << 21))
    ctr = pyoracle.Counters()
    ns, dt, _ = oracle_rate(w.oracle(), pyoracle, hr, ho, pyoracle.default_params(**w.cfg["flags"]), seconds, cores,
                            counters=ctr)
    c = ctr.as_dict()
    return {"value": ns / dt, "unit": "reads/s", "cores": cores, "kind": "port",
            "sample": "first %d of the step's %d reads, %.1f s" % (ns, w.n_reads, dt),
            "reference_algorithm_sectors_per_read":
                (2 * c["bs_steps"] + c["lf_steps"] + c["rows_located"] + c["window_bytes"] / 128.0) / ns}


def measure(args, name, cfg, ctx, steps, warmup, ragged=False, n_reads=None, cpu_seconds=None, full=False,
            dump_dir=None):
    """One workload on this rank set: parity gate, device-resident leg, end-to-end leg, CPU baseline.
    dump_dir: rank 0 writes there what the last step of the device-resident leg computed (dump_outputs).
    Returns (summary dict on rank 0 / None elsewhere, Workload)."""
    w = Workload(args, name, cfg, ctx, ragged=ragged, n_reads=n_reads)
    parity = parity_gate(args, w) if (ctx.rank == 0 and not args.no_parity) else None
    ctx.barrier()
    # clocks and throttle reasons are sampled from before the warm-up steps of the device-resident leg to the end of
    # the end-to-end leg (both timed regions and the identical load around them; the legs themselves last ~0.1-0.2 s)
    clocks = ClockSampler(ctx.local_rank) if full else None
    # `value`: the call as a user makes it (no per-stage timers; the library then runs its slices on two lanes).
    # A second, identical leg with the per-stage CUDA-event timers on (one lane, so that kernels are timed alone)
    # gives the stage times and the roofline's kernel durations; its own step time is reported beside them.
    dump = (lambda last: dump_outputs(dump_dir, w, last)) if dump_dir and ctx.rank == 0 else None
    ms, _, _, launches = time_device(w, steps, max(3, warmup), profile=False, on_last=dump)
    ms_prof, stats, per_step, _ = time_device(w, 1 if args.no_profile else steps, 2, profile=True)
    prof_steps = 1 if args.no_profile else steps
    e2e_ms, h2d, d2h = time_e2e(w, steps)
    clk = clocks.stop() if clocks else None
    pk = time_e2e_packed(w, steps) if full else None
    ms, e2e_ms, ms_prof = ctx.max_over_ranks([ms, e2e_ms, ms_prof])
    total = w.n_reads * ctx.world * steps
    out = {"value": total / (ms * 1e-3), "ms_per_step": ms / steps,
           "profiled_leg": {"ms_per_step": ms_prof / prof_steps, "steps": prof_steps,
                            "note": "same steps with mtsvgpu_set_profiling(1): per-stage CUDA events, one lane; "
                                    "stages_ms_per_step, work_per_step and the rooflines come from this leg"},
           "e2e": {"value": total / (e2e_ms * 1e-3), "unit": "reads/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / steps,
                   "h2d_gbs_achieved_per_gpu": h2d / (e2e_ms / steps * 1e-3) / 1e9},
           "gpu_launches": launches, "clocks": clk, "stages_ms_per_step": per_step,
           "work_per_step": {k: stats[k] for k in ("n_queries", "n_seed_slots", "n_seed_hits", "n_candidates",
                                                    "n_hits", "window_bytes", "rank_queries", "n_sub_batches")},
           "parity": parity, "index_load_seconds": w.info["load_seconds"], "index_hbm_gb": w.info["device_bytes"] / 1e9,
           "device_sa_rate": w.info["device_sa_rate"], "ktab_k": w.info["ktab_k"],
           "index_build": w.build_meta, "_stats": stats}
    if pk:
        pm, ppm, pack_ms = ctx.max_over_ranks([pk["packed"][0], pk["prepacked"][0], pk["pack_ms"]])
        out["e2e_packed"] = {
            "value": total / (pm * 1e-3), "unit": "reads/s", "ms_per_step": pm / steps,
            "h2d_bytes_per_step": pk["packed"][1], "d2h_bytes_per_step": pk["packed"][2],
            "host_pack_ms_per_step": pack_ms, "host_pack_threads": pk["pack_threads"],
            "prepacked_value": total / (ppm * 1e-3), "prepacked_ms_per_step": ppm / steps,
            "note": "mtsvgpu_bin_batch_packed: 3 bit planes per read (57 B per 150 bases) instead of raw bytes. `value` "
                    "starts from the same raw host reads as e2e and packs them on the host inside the timed region "
                    "(mtsvgpu_pack_reads); prepacked_value is the call alone, for a parser that emits records directly"}
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, w, cpu_seconds or args.cpu_seconds)
    else:
        out["cpu_baseline"] = None
    return out, w


def strip(d):
    return {k: v for k, v in d.items() if not k.startswith("_")}


def run_gpu_arm(args, name, cfg, ctx):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this implementation has no CPU path "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(ctx.local_rank)
    numa = bind_to_gpu_numa_node(ctx.local_rank) if ctx.world > 1 else "single rank: unbound"
    log("rank %d: host affinity: %s" % (ctx.rank, numa))
    world = ctx.world
    m, w = measure(args, name, cfg, ctx, args.steps, args.warmup, full=True, dump_dir=args.dump_outputs)
    roofline, roofline_mem = rooflines(w, m["_stats"], m["stages_ms_per_step"], m["profiled_leg"]["ms_per_step"], m["clocks"])
    L = w.L
    line = {
        "metric": METRIC, "value": m["value"], "unit": "reads/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": m["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 integer",
        "data": "synthetic", "config": config_dict(name, cfg, w.n_reads),
        "run": {"device_sa_rate": m["device_sa_rate"], "ktab_k": m["ktab_k"], "index_hbm_gb": m["index_hbm_gb"],
                "batch_reads": args.batch_reads or "default (1<<22 device-resident; host input: ramped slices up to 1<<20 on two lanes)",
                "hits_per_step": int(m["work_per_step"]["n_hits"]), "profiling_events_in_value_leg": False},
        "e2e": m["e2e"], "e2e_packed": m.get("e2e_packed"), "profiled_leg": m["profiled_leg"],
        "gpu_launches": m["gpu_launches"], "clocks": m["clocks"], "roofline": roofline,
        "roofline_memory_kernel": roofline_mem, "cpu_baseline": m["cpu_baseline"],
        "stages_ms_per_step": m["stages_ms_per_step"], "work_per_step": m["work_per_step"],
        "parity": m["parity"], "index_load_seconds": m["index_load_seconds"],
        "index_build": dict(m["index_build"], note="mtsvgpu_index_build + mtsvgpu_index_write on this box (device "
                            "suffix sort); index_load_seconds = mtsvgpu_index_open of that file"),
    }
    cpu = m["cpu_baseline"]
    if cpu:
        # SURVEY §8(d): the layout-independent work of the reference algorithm (32-byte index sectors per read,
        # counted by the instrumented oracle) over this implementation's time — it exceeds the HBM peak because the
        # k-mer table, the dense suffix array and the pruned verifier avoid most of that work rather than do it faster
        spr = cpu["reference_algorithm_sectors_per_read"]
        line["reference_work_equivalent"] = {
            "sectors_per_read": spr, "bytes_per_read": 32.0 * spr + 2 * L,
            "gbs_at_value": (32.0 * spr + 2 * L) * m["value"] / 1e9,
            "gbs_at_e2e": (32.0 * spr + 2 * L) * m["e2e"]["value"] / 1e9}

    # ---- what bounds the end-to-end number: the box's own upload ceiling, measured here ----
    if not args.only_main:
        line["h2d"] = h2d_ceiling(w)
        line["h2d"]["e2e_achieved_gbs_aggregate"] = m["e2e"]["h2d_gbs_achieved_per_gpu"] * world
        line["h2d"]["e2e_over_ceiling"] = line["h2d"]["e2e_achieved_gbs_aggregate"] / line["h2d"]["all_ranks_gbs_aggregate"]

    # ---- strong scaling: the workload's reads (10 M at cfg2) split N ways, as BASELINE configs[1] states ----
    if world > 1 and not args.only_main:
        n_s = max(1, (args.reads or cfg["reads"]) // world)
        ms_s, _, _, _ = time_device(w, args.steps, 3, n=n_s, profile=False)
        e2e_s, h2d_s, _ = time_e2e(w, args.steps, n=n_s)
        pk_s = time_e2e_packed(w, args.steps, n=n_s)
        ms_s, e2e_s, pk_ms, ppk_ms = ctx.max_over_ranks([ms_s, e2e_s, pk_s["packed"][0], pk_s["prepacked"][0]])
        tot = n_s * world * args.steps
        line["strong_scaling"] = {
            "reads_total_per_step": n_s * world, "reads_per_gpu_per_step": n_s,
            "value": tot / (ms_s * 1e-3), "ms_per_step": ms_s / args.steps,
            "e2e_value": tot / (e2e_s * 1e-3), "e2e_ms_per_step": e2e_s / args.steps,
            "e2e_packed_value": tot / (pk_ms * 1e-3), "e2e_prepacked_value": tot / (ppk_ms * 1e-3),
            "note": "same index, the step's reads divided among the ranks; compare with the N=1 line's value / e2e"}
    if world == 1 and name == "cfg2" and not args.only_main or args.mode == "cli":
        try:
            line["cli_e2e"] = run_cli(args, w)
        except SystemExit:
            raise
        except Exception as e:
            line["cli_e2e"] = {"error": repr(e)}
    w.close()

    # ---- the other BASELINE configs and a ragged-read batch, shorter runs attached to the same line (N=1) ----
    if world == 1 and name == "cfg2" and not args.only_main:
        others = {}
        rw_m, rw = measure(args, "cfg2", cfg, ctx, max(2, args.steps // 2), 3, ragged=True, n_reads=args.reads or cfg["reads"],
                           cpu_seconds=0)
        rw.close()
        rw_m.pop("cpu_baseline", None)
        others["cfg2_ragged"] = dict(strip(rw_m), note="cfg2 with every read trimmed to 100-150 bases: per-slot offsets, "
                                     "non-uniform verifier, seq_off uploaded")
        for oname in ("cfg1", "cfg4", "cfg4b", "cfg5"):
            try:
                om, ow = measure(args, oname, CONFIGS[oname], ctx, max(2, args.steps // 2), 3, cpu_seconds=args.other_cpu_seconds)
                ow.close()
                others[oname] = dict(strip(om), config=config_dict(oname, CONFIGS[oname], ow.n_reads))
            except SystemExit:
                raise
            except Exception as e:  # a side config must not cost the headline line
                others[oname] = {"error": repr(e)}
        line["other_configs"] = others

    if world > 1 and not args.only_main and not args.no_chunk:
        try:
            line["chunk_sharded"] = run_chunk_arm(args, ctx, as_dict=True)
        except SystemExit:
            raise
        except Exception as e:
            line["chunk_sharded"] = {"error": repr(e)}
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)


def write_fastq(path, reads_np, n, L, gz=False):
    """Uniform-length reads -> 4-line FASTQ (fixed-width ids), built as one byte matrix."""
    hdr = np.frombuffer(b"@read_", dtype=np.uint8)
    width = len(hdr) + 9 + 1 + L + 3 + L + 1
    rows = np.empty((n, width), dtype=np.uint8)
    rows[:, :len(hdr)] = hdr
    idx = np.arange(n)
    for d in range(9):
        rows[:, len(hdr) + 8 - d] = 48 + (idx // 10 ** d) % 10
    c = len(hdr) + 9
    rows[:, c] = 10
    rows[:, c + 1:c + 1 + L] = reads_np[:n * L].reshape(n, L)
    rows[:, c + 1 + L:c + 4 + L] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    rows[:, c + 4 + L:c + 4 + 2 * L] = ord("I")
    rows[:, -1] = 10
    if gz:
        import gzip
        with gzip.open(path, "wb", compresslevel=1) as f:
            f.write(rows.tobytes())
    else:
        rows.tofile(path)
    return ["read_%09d" % i for i in range(n)] if n <= 200000 else None


def run_cli(args, w, n_plain=2_000_000, n_gz=500_000, n_check=100_000):
    """The drop-in binary itself: FASTQ file -> results file through mtsv_tools_b200/bin/mtsv-binner (reader thread,
    parser pool packing straight into bit planes, mtsvgpu_bin_batch_packed, formatter pool, ordered writer), wall
    clock of the process and the query time the binary reports (the reference's own timer starts after index
    deserialisation, src/binner.rs:63,72,143).  Results of the first reads are compared with the oracle's lines."""
    from oracle import pyoracle
    exe = os.path.join(ROOT, "mtsv_tools_b200", "bin", "mtsv-binner")
    cores = len(os.sched_getaffinity(0)) or 1
    hr, ho = w.host_views(min(w.n_reads, n_plain))
    n_plain = len(ho) - 1
    L = w.L
    out = {}
    want = None
    for kind, n, gz in (("fastq", n_plain, False), ("fastq_gz", min(n_gz, n_plain), True)):
        path = os.path.join(CACHE_DIR, "cli_reads_%d.fq%s" % (n, ".gz" if gz else ""))
        res = path + ".results"
        write_fastq(path, hr, n, L, gz)
        runs = []
        for _ in range(2):  # (the first start of the binary on a fresh box also pays for cold files; both are reported)
            t0 = time.time()
            pr = subprocess.run([exe, "--fastq", path, "--index", w.path, "--results", res, "--force-overwrite",
                                 "--threads", str(cores)], capture_output=True, text=True)
            wall = time.time() - t0
            if pr.returncode != 0:
                raise SystemExit("bench.py: mtsv-binner failed (%d): %s" % (pr.returncode, pr.stderr[-400:]))
            took = None
            for ln in pr.stderr.splitlines():
                if "Took" in ln:
                    took = float(ln.split("Took")[1].split()[0])
            runs.append((wall, took))
        first_run = {"wall_seconds": runs[0][0], "query_seconds": runs[0][1]}
        wall, took = runs[1]
        lines = open(res).read().splitlines(True)
        if want is None:
            nc = min(n_check, n)
            names = ["read_%09d" % i for i in range(nc)]
            oh, oo = w.oracle().bin_reads((hr[:nc * L], ho[:nc + 1]), pyoracle.default_params(**w.cfg["flags"]),
                                          threads=os.cpu_count())
            want = pyoracle.results_lines(names, oh, oo, False)
        last = "read_%09d" % (min(n_check, n) - 1)
        got = [l for l in lines if l.split(":")[0] <= last]
        ok = got == want
        if not ok:
            raise SystemExit("bench.py: mtsv-binner results differ from the oracle's lines (%s)" % kind)
        out[kind] = {"reads": n, "file_bytes": os.path.getsize(path), "wall_seconds": wall, "query_seconds": took,
                     "first_run": first_run,
                     "reads_per_s_wall": n / wall, "reads_per_s_query": n / took if took else None,
                     "result_lines": len(lines), "parity_lines_checked": len(got), "bit_exact": True}
        os.unlink(path)
        os.unlink(res)
    out["threads"] = cores
    out["note"] = ("wall includes process start, CUDA context and mtsvgpu_index_open of the %.1f GB .index; query_seconds "
                   "is the binary's own timer (starts after the index is loaded, like the reference's)" %
                   (os.path.getsize(w.path) / 1e9))
    return out


def run_chunk_arm(args, ctx, as_dict=False):
    """BASELINE config 3: every rank holds a DIFFERENT MG-index chunk (4 Gbp by default: rows beyond 2^31), every
    read visits every chunk, the per-read TaxID sets are brought together over NVLink by the library's own exchange
    (mtsvgpu_bin_batch_chunked: peer-memory stores + flag barrier + device collapse, min edit per TaxID).
    value = reads/s binned against ALL chunks.  With --hybrid-chunks C < N the N ranks form N/C groups of C chunks,
    each group working on its own shard of the reads (SURVEY §8e row 3)."""
    import torch
    import torch.distributed as dist
    from mtsv_tools_b200 import MGIndex, Params, load_library, chunked
    from mtsv_tools_b200._lib import LibraryError
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.cuda.set_device(ctx.local_rank)
    lib = load_library()
    n_chunks = args.hybrid_chunks or world
    groups = chunked.hybrid_groups(world, n_chunks)
    shard, chunk_id = rank // n_chunks, rank % n_chunks
    group = None
    if len(groups) > 1:
        for g in groups:  # (every rank creates every group, as torch.distributed requires)
            pg = dist.new_group(g)
            if rank in g:
                group = pg
    chunk_mbp = args.chunk_mbp or 4000
    base = CONFIGS["cfg2"]
    cfgc = dict(base, n_seqs=max(1, chunk_mbp // 5), seed=5 + chunk_id)
    L = base["read_len"]
    n_reads = args.reads or base["reads"]  # per group per step
    # ---- this rank's chunk, built where it will be used (nothing goes through the host) ----
    t0 = time.time()
    cat, off, gi, tax = make_reference_torch(cfgc, cfgc["seed"], dev)
    tax = tax + np.uint32(100000 * chunk_id)  # distinct TaxIDs per chunk, except ...
    src_rank = shard * n_chunks
    # ... the first 2 % of chunk 0's genomes, which every other chunk of the group also carries at 0.5 % divergence
    # under the same TaxIDs (strains of one species filed in different chunks): reads from there hit several chunks
    # with different edit distances, which is what the min-edit merge is for
    n_sh = max(1, len(tax) // 50)
    sh_len = int(off[n_sh])
    shared = cat[:sh_len].clone()
    if world > 1:
        dist.broadcast(shared, src=src_rank, group=group)
    if chunk_id != 0:
        g = torch.Generator(device=dev)
        g.manual_seed(900 + chunk_id)
        pos = torch.randint(0, sh_len, (int(sh_len * 0.005),), generator=g, device=dev)
        shared[pos] = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)[
            torch.randint(0, 4, (len(pos),), generator=g, device=dev)]
        cat[:sh_len] = shared
        tax[:n_sh] = (1000 + np.arange(n_sh)).astype(np.uint32)
    del shared
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    # the batch is a metagenome spread over the whole database: every chunk contributes an equal share of the reads
    # (generated from its own genomes), all ranks of the group then hold the same n_reads reads
    per = n_reads // n_chunks
    n_reads = per * n_chunks
    mine, _ = make_reads(base, cat, off, per, 4 + 17 * rank, dev)
    d_reads = torch.empty(n_reads * L, dtype=torch.uint8, device=dev)
    if world > 1:
        dist.all_gather_into_tensor(d_reads, mine, group=group)
    else:
        d_reads.copy_(mine)
    del mine
    # interleave the chunks' shares so that every rank's range of the reads is the same mix
    d_reads = d_reads.view(n_chunks, per, L).transpose(0, 1).contiguous().view(-1)
    torch.cuda.empty_cache()
    t0 = time.time()
    gix = MGIndex.build(cat.data_ptr(), off, gi, tax, device=ctx.local_rank, sa_rate=args.sa_rate, ktab_k=args.ktab_k,
                        batch_reads=args.batch_reads)
    del cat
    torch.cuda.empty_cache()
    info = gix.info()
    log("rank %d: chunk %d (%.2f Gbp) generated in %.1fs, built in %.1fs (suffix array + BWT %.1fs), %.1f GB HBM, k=%d" %
        (rank, chunk_id, info["text_len"] / 1e9, t_gen, time.time() - t0, info["build_seconds"],
         info["device_bytes"] / 1e9, info["ktab_k"]))
    d_off = torch.arange(n_reads + 1, dtype=torch.int64, device=dev) * L
    torch.cuda.synchronize()
    params = Params(**base["flags"])
    stream = torch.cuda.current_stream()
    gix.set_stream(stream.cuda_stream)
    n_local = -(-n_reads // n_chunks)
    comm = chunked.ChunkComm(ctx.local_rank, max_local_reads=n_local, max_hits_per_source=4 * n_local + (1 << 20),
                             group=group)

    # ---- parity gate on a sample, before any timing ----
    parity = None
    if not args.no_parity:
        from oracle import pyoracle
        ns = min(20000, n_reads)
        sub_r, sub_o = d_reads[: ns * L], d_off[: ns + 1]
        first, pairs, offs = comm.bin_reads_tensors(gix, sub_r, sub_o, ns, params)
        fused = (first, pairs.cpu().numpy().astype(np.uint32), offs.cpu().numpy().astype(np.uint64))
        h_sub = (sub_r.cpu().numpy(), sub_o.cpu().numpy().astype(np.uint64))
        local_h, local_o = gix.bin_reads(h_sub, params)  # this chunk alone, through the plain host entry point
        gathered = [None] * n_chunks if chunk_id == 0 else None
        dist.gather_object((fused, local_h, local_o), gathered, dst=src_rank, group=group) if world > 1 else None
        if world == 1:
            gathered = [(fused, local_h, local_o)]
        ok_merge, ok_chunk, t_or = True, None, 0.0
        if chunk_id == 0:
            # (1) exchange + merge == mtsv-collapse's rule (oracle restatement) over the chunks' own hit lists
            want_pairs, want_off = pyoracle.collapse_taxid([(g[1], g[2]) for g in gathered])
            bounds = chunked.read_ranges(ns, n_chunks)
            for r, g in enumerate(gathered):
                f, pr, of = g[0]
                a, e = int(want_off[bounds[r]]), int(want_off[bounds[r + 1]])
                ok_merge &= f == bounds[r] and np.array_equal(pr, want_pairs[a:e]) and \
                    np.array_equal(of, want_off[bounds[r]:bounds[r + 1] + 1] - want_off[bounds[r]])
        if rank == 0 and not args.no_chunk_oracle:
            # (2) this chunk's hits == the CPU oracle on the very same index fields (rows beyond 2^31 at 4 Gbp)
            t1 = time.time()
            parts = gix.export_parts(32)
            b_gi, b_tax = gi, tax
            order = np.argsort(b_tax, kind="stable")
            st = np.zeros(len(order), np.uint64)
            lens = (off[1:] - off[:-1])[order]
            st[1:] = np.cumsum(lens[:-1], dtype=np.uint64)
            oix = pyoracle.Index.from_parts(parts["text"], (b_gi[order], b_tax[order], st, st + lens), parts["bwt"],
                                            parts["sa_sample"], 32)
            del parts
            want_h, want_o = oix.bin_reads(h_sub, pyoracle.default_params(**base["flags"]), threads=os.cpu_count())
            ok_chunk = bool(np.array_equal(want_o, local_o) and all(np.array_equal(want_h[f], local_h[f])
                                                                    for f in ("tax_id", "gi", "offset", "edit")))
            del oix
            t_or = time.time() - t1
        flags = torch.tensor([1.0 if ok_merge else 0.0, 1.0 if ok_chunk in (None, True) else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        parity = {"reads": ns, "merged_pairs": int(len(fused[1])), "exchange_and_merge_bit_exact": bool(flags[0] > 0),
                  "chunk0_vs_oracle_bit_exact": ok_chunk, "chunk0_hits": int(len(local_h)), "oracle_gate_seconds": t_or}
        log("rank %d: chunk parity gate: %s" % (rank, parity))
        if not (flags[0] > 0 and flags[1] > 0):
            raise SystemExit("bench.py: chunk-sharded results differ from the oracle — refusing to report a number")

    def step():
        return comm.bin_reads(gix, d_reads.data_ptr(), d_off.data_ptr(), n_reads, params)

    def step_local():
        return gix.bin_reads_device(d_reads.data_ptr(), d_off.data_ptr(), n_reads, params)

    def timed(fn, steps):
        torch.cuda.synchronize()
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            r = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ctx.barrier()
        return e0.elapsed_time(e1), r

    clocks = ClockSampler(ctx.local_rank)  # (from the warm-up steps on: the timed legs are ~0.1 s each)
    for _ in range(max(3, args.warmup)):
        step()
    launches0 = lib.mtsvgpu_launch_count()
    ms, last = timed(step, args.steps)
    launches = lib.mtsvgpu_launch_count() - launches0
    ms_local, _ = timed(step_local, args.steps)
    clk = clocks.stop()
    n_pairs = float(last[4])
    ms, ms_local = ctx.max_over_ranks([ms, ms_local])
    if world > 1:
        t = torch.tensor([n_pairs], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        n_pairs = float(t[0])
    comm.close()
    gix.close()
    del d_reads, d_off
    torch.cuda.empty_cache()
    n_shards = world // n_chunks
    out = {
        "value": n_reads * n_shards * args.steps / (ms * 1e-3), "unit": "reads/s (each read binned against all %d chunks)" % n_chunks,
        "ms_per_step": ms / args.steps, "exchange_and_merge_ms": (ms - ms_local) / args.steps,
        "local_binning_ms": ms_local / args.steps,
        "workload": "cfg3: %d chunks x %.1f Gbp%s, every read visits every chunk, hits stored into the owning rank's "
                    "buffer over NVLink peer memory (own kernels, CUDA IPC), one flag barrier, device collapse "
                    "(min edit per TaxID)" % (n_chunks, info["text_len"] / 1e9,
                                              " x %d read shards (hybrid)" % n_shards if n_shards > 1 else ""),
        "reads_per_step": n_reads * n_shards, "reference_gbp_total": n_chunks * info["text_len"] / 1e9,
        "collapsed_taxid_hits_per_step": n_pairs, "chunk_build_seconds": info["build_seconds"],
        "chunk_hbm_gb": info["device_bytes"] / 1e9, "gpu_launches": int(launches), "clocks": clk, "parity": parity,
        "scaling_note": "reference size grows with the number of chunks (one chunk per GPU); reads per step fixed",
    }
    if as_dict:
        return out
    if rank == 0:
        line = {"metric": METRIC, "value": out["value"], "unit": "reads/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": out["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 integer", "data": "synthetic",
                "config": {"workload": out["workload"], "reads_per_step": out["reads_per_step"]},
                "chunk_sharded": out, "e2e": None, "gpu_launches": int(launches), "clocks": clk, "roofline": None,
                "cpu_baseline": None}
        print(json.dumps(line), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="reads", choices=["reads", "chunk", "cli"],
                    help="reads: index replicated, reads sharded (default); chunk: one index chunk per GPU; "
                         "cli: reads + the mtsv-binner binary on a FASTQ file (also part of the default N=1 run)")
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU per step (default: the config's)")
    ap.add_argument("--sa-rate", type=int, default=0)
    ap.add_argument("--ktab-k", type=int, default=0)
    ap.add_argument("--batch-reads", type=int, default=0)
    ap.add_argument("--parity-reads", type=int, default=50000)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--other-cpu-seconds", type=float, default=5.0)
    ap.add_argument("--ref-seconds", type=float, default=10.0)
    ap.add_argument("--chunk-mbp", type=int, default=0, help="chunk mode: Mbp per chunk (default 4000)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-chunk", action="store_true", help="N>1: skip the chunk-sharded leg")
    ap.add_argument("--no-chunk-oracle", action="store_true", help="chunk mode: skip the CPU-oracle check of chunk 0")
    ap.add_argument("--hybrid-chunks", type=int, default=0, help="chunk mode: chunks per copy of the database (< N: hybrid)")
    ap.add_argument("--only-main", action="store_true", help="only the headline workload (no side configs / legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (a seeded sample of the reads' hits, float64 .npy, "
                         "at most 64 MB) to DIR, to compare two builds on identical inputs (reads mode)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode == "chunk" or args.impl == "reference"):
        ap.error("--dump-outputs writes the outputs of the reads mode of this implementation")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, args.config, cfg, rank, world)
        return
    ctx = Ctx(rank, world, local_rank)
    if world > 1 or args.mode == "chunk":
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    try:
        if args.mode == "chunk":
            run_chunk_arm(args, ctx)
        else:
            run_gpu_arm(args, args.config, cfg, ctx)
    finally:
        if world > 1 or args.mode == "chunk":
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
