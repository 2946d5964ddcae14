"""Chunk-sharded operation (SURVEY §8e): the collapse rule's KATs, the device collapse against the oracle's
restatement of mtsv-collapse's merge rule, and the fused exchange (mtsvgpu_bin_batch_chunked) against the oracle."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mtsv_tools_b200 import chunked

HIT_DTYPE = np.dtype([("tax_id", "<u4"), ("gi", "<u4"), ("offset", "<u8"), ("edit", "<u4"), ("reserved", "<u4")])


def test_collapse_rule_kats():
    """src/collapse.rs:788-817 collapse_edit_distances_min_edit: r1:1=5,2=9 + r1:1=2,2=10 -> r1:1=2,2=9."""
    from oracle import pyoracle

    def mk(lists):
        hits = np.zeros(sum(len(x) for x in lists), dtype=HIT_DTYPE)
        offs = np.zeros(len(lists) + 1, dtype=np.uint64)
        k = 0
        for i, l in enumerate(lists):
            for t, e in l:
                hits[k]["tax_id"], hits[k]["edit"] = t, e
                k += 1
            offs[i + 1] = k
        return hits, offs
    a = mk([[(1, 5), (2, 9)], [(3, 4)]])
    b = mk([[(1, 2), (2, 10)], [(3, 1)]])
    pairs, offs = pyoracle.collapse_taxid([a, b])
    assert pairs.tolist() == [[1, 2], [2, 9], [3, 1]] and offs.tolist() == [0, 2, 3]


def test_collapse_rule_kat_taxid_gi():
    """src/collapse.rs:804-817 collapse_edit_distances_taxid_gi_min_edit:
    r1:1-5-3=7,1-5-2=4 | r2:2-9-1=3  +  r1:1-5-4=5,2-8-1=6 | r2:2-9-1=2  ->  r1:1-5-2=4,2-8-1=6 | r2:2-9-1=2."""
    from oracle import pyoracle

    def mk(lists):
        hits = np.zeros(sum(len(x) for x in lists), dtype=HIT_DTYPE)
        offs = np.zeros(len(lists) + 1, dtype=np.uint64)
        k = 0
        for i, l in enumerate(lists):
            for t, g, off, e in l:
                hits[k]["tax_id"], hits[k]["gi"], hits[k]["offset"], hits[k]["edit"] = t, g, off, e
                k += 1
            offs[i + 1] = k
        return hits, offs
    a = mk([[(1, 5, 3, 7), (1, 5, 2, 4)], [(2, 9, 1, 3)]])
    b = mk([[(1, 5, 4, 5), (2, 8, 1, 6)], [(2, 9, 1, 2)]])
    out, offs = pyoracle.collapse_taxid_gi([a, b])
    got = [(int(h["tax_id"]), int(h["gi"]), int(h["offset"]), int(h["edit"])) for h in out]
    assert got == [(1, 5, 2, 4), (2, 8, 1, 6), (2, 9, 1, 2)] and offs.tolist() == [0, 2, 3]
    # ties on the edit go to the smaller offset (:622)
    c = mk([[(1, 5, 9, 4)], []])
    out, offs = pyoracle.collapse_taxid_gi([c, a])
    assert (int(out[0]["offset"]), int(out[0]["edit"])) == (2, 4)


@pytest.mark.gpu
def test_collapse_device_taxid_gi_vs_oracle(oracle):
    """Device merge in mode TaxIdGi == oracle restatement, on two chunks that share sequence (same TaxID/GI reached
    from both) plus the reference's KAT."""
    from mtsv_tools_b200 import MGIndex, Params, synth
    refs = [synth.make_reference(6, 20000, seed=s, n_frac=0.001, shared_frac=0.1, taxids=[5, 6, 7, 8, 9, 10])
            for s in (31, 32)]
    refs[1][0][:30000] = refs[0][0][:30000]  # same GIs (1..6) in both chunks: groups meet across parts
    idx = [oracle.Index.build((r[0], r[1]), r[2], r[3], 64, 32) for r in refs]
    reads = synth.make_reads(np.concatenate([refs[0][0], refs[1][0]]),
                             np.concatenate([refs[0][1], refs[1][1][1:] + refs[0][1][-1]]), 4000, 150, seed=33)
    parts_o = [ix.bin_reads(reads, oracle.default_params(), threads=4) for ix in idx]
    want, want_off = oracle.collapse_taxid_gi(parts_o)
    parts_h = [torch.from_numpy(np.frombuffer(h.tobytes(), dtype=np.uint8).copy()).cuda() for h, _ in parts_o]
    parts_c = [torch.from_numpy((o[1:] - o[:-1]).astype(np.int32)).cuda() for _, o in parts_o]
    hits, offs = chunked.collapse_parts_device_taxid_gi(0, None, parts_h, parts_c, 4000)
    got = np.frombuffer(hits.cpu().numpy().tobytes(), dtype=HIT_DTYPE)
    assert np.array_equal(offs.cpu().numpy().astype(np.uint64), want_off)
    for f in ("tax_id", "gi", "offset", "edit"):
        assert np.array_equal(got[f], want[f]), f
    assert len(want) > 3000
    # the reference's own KAT through the device kernel
    a = np.zeros(3, dtype=HIT_DTYPE)
    a["tax_id"], a["gi"], a["offset"], a["edit"] = [1, 1, 2], [5, 5, 9], [3, 2, 1], [7, 4, 3]
    b = np.zeros(3, dtype=HIT_DTYPE)
    b["tax_id"], b["gi"], b["offset"], b["edit"] = [1, 2, 2], [5, 8, 9], [4, 1, 1], [5, 6, 2]
    ph = [torch.from_numpy(np.frombuffer(x.tobytes(), dtype=np.uint8).copy()).cuda() for x in (a, b)]
    pc = [torch.tensor([2, 1], dtype=torch.int32).cuda(), torch.tensor([2, 1], dtype=torch.int32).cuda()]
    hits, offs = chunked.collapse_parts_device_taxid_gi(0, None, ph, pc, 2)
    got = np.frombuffer(hits.cpu().numpy().tobytes(), dtype=HIT_DTYPE)
    assert [(int(h["tax_id"]), int(h["gi"]), int(h["offset"]), int(h["edit"])) for h in got] == \
        [(1, 5, 2, 4), (2, 8, 1, 6), (2, 9, 1, 2)]
    assert offs.cpu().tolist() == [0, 2, 3]


@pytest.mark.gpu
def test_collapse_device_vs_oracle(oracle):
    """Two different chunks, the same reads: device merge == oracle merge of the two oracle runs."""
    from mtsv_tools_b200 import MGIndex, Params, synth
    refs = [synth.make_reference(6, 20000, seed=s, n_frac=0.001, shared_frac=0.1, taxids=[5, 6, 7, 8, 9, 10])
            for s in (31, 32)]
    # chunk 2 shares some sequence with chunk 1 so that the same TaxIDs are reached from both chunks
    refs[1][0][:30000] = refs[0][0][:30000]
    idx = [oracle.Index.build((r[0], r[1]), r[2], r[3], 64, 32) for r in refs]
    reads = synth.make_reads(np.concatenate([refs[0][0], refs[1][0]]),
                             np.concatenate([refs[0][1], refs[1][1][1:] + refs[0][1][-1]]), 4000, 150, seed=33)
    parts_o = [ix.bin_reads(reads, oracle.default_params(), threads=4) for ix in idx]
    want_pairs, want_off = oracle.collapse_taxid(parts_o)
    parts_h, parts_c = [], []
    for ix in idx:
        with MGIndex.from_parts(ix.text, ix.bins(), ix.bwt, ix.sa_sample, ix.sa_sample_rate) as g:
            h, o = g.bin_reads(reads, Params())
        parts_h.append(torch.from_numpy(np.frombuffer(h.tobytes(), dtype=np.uint8).copy()).cuda())
        parts_c.append(torch.from_numpy((o[1:] - o[:-1]).astype(np.int32)).cuda())
    pairs, offs = chunked.collapse_parts_device(0, None, parts_h, parts_c, 4000)
    assert np.array_equal(offs.cpu().numpy().astype(np.uint64), want_off)
    assert np.array_equal(pairs.cpu().numpy().astype(np.uint32), want_pairs)
    assert len(want_pairs) > 3000


# ------------------------------------------------------------------------------------------------
# the fused path: mtsvgpu_comm_* / mtsvgpu_bin_batch_chunked (csrc/chunked.cu)
# ------------------------------------------------------------------------------------------------
def test_hybrid_groups():
    assert chunked.hybrid_groups(8, 8) == [[0, 1, 2, 3, 4, 5, 6, 7]]
    assert chunked.hybrid_groups(8, 2) == [[0, 1], [2, 3], [4, 5], [6, 7]]
    with pytest.raises(ValueError):
        chunked.hybrid_groups(8, 3)
    assert chunked.read_ranges(10, 4) == [0, 3, 6, 9, 10]


def _handles_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        mine = bytes([rank + 1]) * chunked.HANDLE_BYTES
        out.put((rank, chunked.gather_handles(mine)))
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_handle_exchange_gloo_world2():
    """The host's part of the communicator setup: every rank ends up with all handles in rank order."""
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_handles_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = b"".join(bytes([r + 1]) * chunked.HANDLE_BYTES for r in range(world))
    assert got[0] == want and got[1] == want


def _chunk_refs(world):
    from mtsv_tools_b200 import synth
    refs = [synth.make_reference(6, 20000, seed=40 + s, n_frac=0.001, shared_frac=0.1, taxids=[5, 6, 7, 8, 9, 10])
            for s in range(world)]
    for s in range(1, world):  # shared sequence: the same TaxIDs are reached from several chunks
        refs[s][0][:30000] = refs[0][0][:30000]
    cat = np.concatenate([r[0] for r in refs])
    off = np.concatenate([[0]] + [r[1][1:] + i * refs[0][1][-1] for i, r in enumerate(refs)]).astype(np.uint64)
    return refs, cat, off


def _hybrid_worker(rank, world, n_chunks, port, n_reads, out):
    """Hybrid operation: rank r holds chunk r % n_chunks and works on read shard r // n_chunks; each shard's ranks
    form their own exchange group (a torch.distributed sub-group and a communicator of n_chunks ranks)."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from mtsv_tools_b200 import MGIndex, Params, synth
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        groups = chunked.hybrid_groups(world, n_chunks)
        group = None
        for g in groups:
            pg = dist.new_group(g)
            if rank in g:
                group = pg
        shard, chunk = rank // n_chunks, rank % n_chunks
        refs, cat, off = _chunk_refs(n_chunks)
        r = refs[chunk]
        with MGIndex.build(r[0], r[1], r[2], r[3], device=dev) as gix:
            comm = chunked.ChunkComm(dev, max_local_reads=-(-n_reads // n_chunks), max_hits_per_source=200000, group=group)
            try:
                reads, roff = synth.make_reads(cat, off, n_reads, 150, seed=80 + shard)
                first, pairs, offs = comm.bin_reads_tensors(gix, torch.from_numpy(reads).cuda(),
                                                            torch.from_numpy(roff.astype(np.int64)).cuda(), n_reads, Params())
                out.put((rank, (first, pairs.cpu().numpy().astype(np.uint32), offs.cpu().numpy().astype(np.uint64))))
            finally:
                comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_hybrid_chunk_groups_times_read_shards(oracle):
    """4 ranks = 2 chunks x 2 read shards (SURVEY §8e row 3): every shard's reads meet both chunks inside their own
    group; results equal the oracle's merge per shard."""
    from mtsv_tools_b200 import synth
    world, n_chunks, n_reads = 4, 2, 2000
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_hybrid_worker, args=(r, world, n_chunks, port, n_reads, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    refs, cat, off = _chunk_refs(n_chunks)
    idx = [oracle.Index.build((r[0], r[1]), r[2], r[3], 64, 32) for r in refs]
    for shard in range(world // n_chunks):
        reads = synth.make_reads(cat, off, n_reads, 150, seed=80 + shard)
        want_pairs, want_off = oracle.collapse_taxid([ix.bin_reads(reads, oracle.default_params(), threads=4) for ix in idx])
        bounds = chunked.read_ranges(n_reads, n_chunks)
        for c in range(n_chunks):
            first, pairs, offs = got[shard * n_chunks + c]
            assert first == bounds[c]
            a, e = int(want_off[bounds[c]]), int(want_off[bounds[c + 1]])
            assert np.array_equal(pairs, want_pairs[a:e]) and len(pairs) > 100
            assert np.array_equal(offs, want_off[bounds[c]:bounds[c + 1] + 1] - want_off[bounds[c]])


def _fused_worker(rank, world, port, n_batches, n_reads, cap, out):
    """One rank of the fused chunk-sharded path.  With fewer GPUs than ranks the ranks share device 0: CUDA IPC
    works between processes on one device too, the peer stores are then local stores."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from mtsv_tools_b200 import MGIndex, Params, synth, LibraryError
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        refs, cat, off = _chunk_refs(world)
        r = refs[rank]
        res = []
        with MGIndex.build(r[0], r[1], r[2], r[3], device=dev) as gix:
            comm = chunked.ChunkComm(dev, max_local_reads=-(-n_reads // world), max_hits_per_source=cap)
            try:
                for b in range(n_batches):
                    nb = n_reads if b % 2 == 0 else n_reads - 37  # (ragged last range on odd batches)
                    reads, roff = synth.make_reads(cat, off, nb, 150, seed=50 + b)
                    d_reads = torch.from_numpy(reads).cuda()
                    d_off = torch.from_numpy(roff.astype(np.int64)).cuda()
                    try:
                        first, pairs, offs = comm.bin_reads_tensors(gix, d_reads, d_off, nb, Params())
                        res.append((first, pairs.cpu().numpy().astype(np.uint32), offs.cpu().numpy().astype(np.uint64)))
                    except LibraryError as e:
                        res.append(("error", e.code))
            finally:
                comm.close()
        out.put((rank, res))
    finally:
        dist.destroy_process_group()


def _run_fused(world, n_batches, n_reads, cap):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_fused_worker, args=(r, world, port, n_batches, n_reads, cap, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_fused_chunk_exchange_vs_oracle(oracle, world):
    """mtsvgpu_bin_batch_chunked on `world` ranks == mtsv-collapse's merge (oracle restatement) of `world`
    independent oracle runs, range by range, over several consecutive batches (both buffer parities)."""
    from mtsv_tools_b200 import synth
    n_batches, n_reads = 3, 3000
    got = _run_fused(world, n_batches, n_reads, cap=200000)
    refs, cat, off = _chunk_refs(world)
    idx = [oracle.Index.build((r[0], r[1]), r[2], r[3], 64, 32) for r in refs]
    for b in range(n_batches):
        nb = n_reads if b % 2 == 0 else n_reads - 37
        reads = synth.make_reads(cat, off, nb, 150, seed=50 + b)
        want_pairs, want_off = oracle.collapse_taxid([ix.bin_reads(reads, oracle.default_params(), threads=4) for ix in idx])
        bounds = chunked.read_ranges(nb, world)
        assert len(want_pairs) > 1000
        for r in range(world):
            first, pairs, offs = got[r][b]
            assert first == bounds[r]
            a, e = int(want_off[bounds[r]]), int(want_off[bounds[r + 1]])
            assert np.array_equal(offs, want_off[bounds[r]:bounds[r + 1] + 1] - want_off[bounds[r]]), (b, r)
            assert np.array_equal(pairs, want_pairs[a:e]), (b, r)


@pytest.mark.gpu
def test_fused_chunk_exchange_overflow_fails_on_every_rank():
    """A range that does not fit its slot fails the batch with ELIMIT on all ranks (nothing truncated), and the
    communicator stays usable."""
    got = _run_fused(2, 1, 3000, cap=50)
    assert got[0] == [("error", -7)] and got[1] == [("error", -7)]
