"""bin vs assign on one GPU: the Hit-record output of mtsvgpu_bin_batch_* against the merged (TaxID, edit) output of
mtsvgpu_assign_batch_* on bench.py's configs, through the pinned, pre-packed and device-resident paths, alternating
the two kinds.  Per leg: ms per step, reads/s, bytes copied device -> host per step and merged records per read.  The
profiled leg gives the device time the merge adds (stage "emit").  At the timed sizes the assign output is checked
against a reduction of the bin output computed with torch (each TaxID of a read once, with its minimum edit).

    python tools/assign_bench.py --out DIR [--configs cfg2,cfg4,cfg4b,cfg5] [--steps 5]
                                 [--cli-binaries A,B] [--cli-reads 2000000,500000]

--cli-binaries: mtsv-binner executables to time on FASTQ files of cfg2 and cfg4 reads (alternated, twice each); the
results files of all binaries must be byte-identical.  Writes DIR/assign_bench.json."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from mtsv_tools_b200 import load_library  # noqa: E402
from mtsv_tools_b200._lib import check  # noqa: E402
from mtsv_tools_b200.index import pack_reads_planes  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def call_pinned(w, kind, hr, ho):
    """One pinned-result call without copying the results; returns (records, offsets, n_records, record_bytes)."""
    L = load_library()
    ps = w.params.c_struct(2)
    rp, op, nr = C.c_void_p(), C.c_void_p(), C.c_uint64()
    fn = L.mtsvgpu_bin_batch_pinned if kind == "bin" else L.mtsvgpu_assign_batch_pinned
    n = len(ho) - 1
    check(fn(w.gix._h, C.c_void_p(hr.ctypes.data), C.c_void_p(ho.ctypes.data), n, C.byref(ps), C.byref(rp),
             C.byref(op), C.byref(nr)))
    return rp.value, op.value, int(nr.value), 24 if kind == "bin" else 8


def call_packed(w, kind, buf, ho):
    if kind == "bin":
        h, o = w.gix.bin_reads_packed(buf, ho, w.params)
        return None, None, len(h), 24
    t, o = w.gix.assign_reads_packed(buf, ho, w.params)
    return None, None, len(t), 8


def call_device(w, kind):
    fn = w.gix.bin_reads_device if kind == "bin" else w.gix.assign_reads_device
    d, do, n = fn(w.d_reads.data_ptr(), w.d_off.data_ptr(), w.n_reads, w.params)
    return d, do, int(n), 24 if kind == "bin" else 8


def timed(fn, steps):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps, out


def device_tensor(ptr, nbytes):
    import torch
    from mtsv_tools_b200.chunked import _DevArray
    return torch.as_tensor(_DevArray(ptr, max(1, nbytes)), device="cuda")[:nbytes]


def reduce_hits_torch(d_hits, n_hits, d_off, n_reads, chunk=1 << 20):
    """Per read each TaxID once with its minimum edit, by TaxID, from device Hit records -> (records int32 [n, 2]
    on the device, offsets int64)."""
    import torch
    h = device_tensor(d_hits, n_hits * 24).view(torch.int32).reshape(-1, 6)
    off = device_tensor(d_off, (n_reads + 1) * 8).view(torch.int64)
    recs, counts = [], []
    for r0 in range(0, n_reads, chunk):
        r1 = min(n_reads, r0 + chunk)
        a, b = int(off[r0]), int(off[r1])
        cnt = off[r0 + 1:r1 + 1] - off[r0:r1]
        read = torch.repeat_interleave(torch.arange(r1 - r0, device="cuda"), cnt)
        tax = h[a:b, 0].to(torch.int64) & 0xffffffff
        edit = h[a:b, 4].to(torch.int64)
        assert int(edit.max()) < 256 if b > a else True
        key, _ = torch.sort((read << 40) | (tax << 8) | edit)
        first = torch.ones_like(key, dtype=torch.bool)
        first[1:] = (key[1:] >> 8) != (key[:-1] >> 8)
        k = key[first]
        recs.append(torch.stack([((k >> 8) & 0xffffffff).to(torch.int64), k & 0xff], 1))
        counts.append(torch.bincount(k >> 40, minlength=r1 - r0))
    rec = torch.cat(recs).to(torch.int64) if recs else torch.zeros(0, 2, dtype=torch.int64, device="cuda")
    o = torch.zeros(n_reads + 1, dtype=torch.int64, device="cuda")
    if counts:
        o[1:] = torch.cumsum(torch.cat(counts), 0)
    return rec, o


def measure_config(args, name, ctx):
    import torch
    cfg = bench.CONFIGS[name]
    wargs = types.SimpleNamespace(sa_rate=0, ktab_k=0, batch_reads=0, reads=0)
    w = bench.Workload(wargs, name, cfg, ctx)
    n = w.n_reads
    hr, ho = w.host_views()
    nbytes = int(load_library().mtsvgpu_packed_size(C.c_void_p(ho.ctypes.data), n))
    buf_t = torch.empty(max(1, nbytes), dtype=torch.uint8, pin_memory=True)
    buf = buf_t.numpy()[:nbytes]
    pack_reads_planes((hr, ho), out=buf)
    legs = {"pinned": lambda k: call_pinned(w, k, hr, ho), "prepacked": lambda k: call_packed(w, k, buf, ho),
            "device": lambda k: call_device(w, k)}
    res = {"label": cfg["label"], "reads": n, "legs": {}}
    for leg, fn in legs.items():
        for kind in ("bin", "assign"):
            for _ in range(args.warmup):
                fn(kind)
        runs = {"bin": [], "assign": []}
        recs = {}
        for _ in range(args.rounds):  # bin and assign alternate
            for kind in ("bin", "assign"):
                ms, out = timed(lambda: fn(kind), args.steps)
                runs[kind].append(ms)
                recs[kind] = out
        d = {}
        for kind in ("bin", "assign"):
            n_rec, rec_bytes = recs[kind][2], recs[kind][3]
            ms = min(runs[kind])
            d[kind] = {"ms_per_step": ms, "ms_runs": runs[kind], "reads_per_s": n / ms * 1e3,
                       "records": n_rec, "records_per_read": n_rec / n}
            if leg != "device":
                d[kind]["d2h_bytes_per_step"] = n_rec * rec_bytes + (n + 1) * 8
        d["assign_over_bin"] = d["assign"]["ms_per_step"] / d["bin"]["ms_per_step"]
        res["legs"][leg] = d
        bench.log("%s %s: bin %.1f ms, assign %.1f ms (runs %s / %s)" % (name, leg, d["bin"]["ms_per_step"],
                                                                        d["assign"]["ms_per_step"], runs["bin"],
                                                                        runs["assign"]))
    # profiled leg (device-resident input): per-stage device time of one call of each kind
    w.gix.set_profiling(True)
    prof = {}
    for kind in ("bin", "assign"):
        call_device(w, kind)
        torch.cuda.synchronize()
        prof[kind] = w.gix.last_batch_stats()["ms"]
    w.gix.set_profiling(False)
    res["profiled_stage_ms"] = prof
    res["assign_adds_device_ms"] = sum(prof["assign"].values()) - sum(prof["bin"].values())
    res["assign_adds_emit_ms"] = prof["assign"]["emit"] - prof["bin"]["emit"]
    # the outputs at the timed size: assign == the reduction of bin, through every path
    d, do, nh, _ = call_device(w, "bin")
    want_rec, want_off = reduce_hits_torch(d, nh, do, n)
    checks = {}
    for leg in ("device", "pinned", "prepacked"):
        if leg == "device":
            t, to, nt, _ = call_device(w, "assign")
            got = device_tensor(t, nt * 8).view(torch.int32).reshape(-1, 2).to(torch.int64) & 0xffffffff
            got_off = device_tensor(to, (n + 1) * 8).view(torch.int64)
        else:
            if leg == "pinned":
                t, to, nt, _ = call_pinned(w, "assign", hr, ho)
                arr = np.frombuffer((C.c_uint8 * max(1, nt * 8)).from_address(t), dtype=np.uint32)[:nt * 2]
                offs = np.frombuffer((C.c_uint8 * ((n + 1) * 8)).from_address(to), dtype=np.int64)
            else:
                tt, oo = w.gix.assign_reads_packed(buf, ho, w.params)
                arr, offs = tt.view(np.uint32), oo.view(np.int64)
            got = torch.from_numpy(arr.astype(np.int64).reshape(-1, 2)).cuda()
            got_off = torch.from_numpy(offs.copy()).cuda()
        ok = bool(torch.equal(got_off, want_off) and torch.equal(got, want_rec))
        checks[leg] = ok
        if not ok:
            raise SystemExit("assign_bench: %s %s output differs from the reduction of the bin output" % (name, leg))
    res["assign_equals_reduced_bin"] = checks
    res["merged_records"] = int(want_rec.shape[0])
    del buf, buf_t
    return w, res


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 24), b""):
            h.update(b)
    return h.hexdigest()


def run_cli(args, w, name, n_reads):
    hr, ho = w.host_views(min(w.n_reads, n_reads))
    n = len(ho) - 1
    fq = os.path.join(bench.CACHE_DIR, "assign_bench_%s_%d.fq" % (name, n))
    bench.write_fastq(fq, hr, n, w.L)
    cores = len(os.sched_getaffinity(0)) or 1
    out = {"reads": n, "runs": {}}
    digests = {}
    for rnd in range(2):
        for exe in args.cli_binaries.split(","):
            res = fq + ".results"
            t0 = time.time()
            pr = subprocess.run([exe, "--fastq", fq, "--index", w.path, "--results", res, "--force-overwrite",
                                 "--threads", str(cores)], capture_output=True, text=True)
            wall = time.time() - t0
            if pr.returncode != 0:
                raise SystemExit("assign_bench: %s failed: %s" % (exe, pr.stderr[-400:]))
            took = [float(ln.split("Took")[1].split()[0]) for ln in pr.stderr.splitlines() if "Took" in ln]
            out["runs"].setdefault(exe, []).append({"query_seconds": took[0] if took else None, "wall_seconds": wall})
            digests.setdefault(exe, set()).add(sha256(res))
            out["result_bytes"] = os.path.getsize(res)
            os.unlink(res)
    os.unlink(fq)
    all_digests = set().union(*digests.values())
    out["results_identical"] = len(all_digests) == 1
    if len(all_digests) != 1:
        raise SystemExit("assign_bench: the binaries' results files differ on %s" % name)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="cfg2,cfg4,cfg4b,cfg5")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--cli-binaries", default="")
    ap.add_argument("--cli-reads", default="2000000,500000", help="reads of the cfg2 and cfg4 FASTQ files")
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    ctx = bench.Ctx(0, 1, 0)
    out = {"gpu": gpu_info(), "steps": args.steps, "rounds": args.rounds, "configs": {}, "cli": {}}
    cli_reads = dict(zip(("cfg2", "cfg4"), (int(x) for x in args.cli_reads.split(","))))
    for name in args.configs.split(","):
        w, res = measure_config(args, name, ctx)
        out["configs"][name] = res
        if args.cli_binaries and name in cli_reads:
            out["cli"][name] = run_cli(args, w, name, cli_reads[name])
        w.close()
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "assign_bench.json"), "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
