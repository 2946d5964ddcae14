"""Chunk-sharded operation (SURVEY.md §8e, BASELINE config 3): GPU g holds MG-index chunk g, every read
visits every chunk, and the per-read hit lists are merged the way ``mtsv-collapse`` merges the per-chunk
results files (src/collapse.rs:543-654, mode TaxId: minimum edit per TaxID, :597-602).

``ChunkComm`` = mtsvgpu_comm_* / mtsvgpu_bin_batch_chunked — the exchange and the merge run inside the library
(csrc/chunked.cu: hits stored straight into the owning rank's buffer over NVLink peer memory, one flag barrier,
collapse as the epilogue); the host only moves `world` 128-byte handles once.  ``collapse_parts_device`` and
``collapse_parts_device_taxid_gi`` run the library's merge on hit lists the caller already holds on the device.
"""
import ctypes as C

from . import _lib
from ._lib import check

HANDLE_BYTES = 128  # MTSVGPU_COMM_HANDLE_BYTES


def gather_handles(my_handle, group=None):
    """The host's part of the communicator setup: move every rank's opaque 128-byte handle to every rank, in
    rank order.  Any channel would do; here it is one all_gather (NCCL on GPU boxes, gloo in the CPU tests)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    backend = dist.get_backend(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    mine = torch.frombuffer(bytearray(my_handle), dtype=torch.uint8).to(dev)
    allh = torch.empty(world * HANDLE_BYTES, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(allh, mine, group=group)
    return bytes(allh.cpu().numpy().tobytes())


class ChunkComm:
    """mtsvgpu_comm: the peer-memory communicator of the chunk-sharded mode (include/mtsv_b200.h).  `group` is the
    torch.distributed group whose ranks hold the chunks of ONE copy of the database: the whole world in plain
    chunk-sharded operation, a sub-group in hybrid operation (chunk groups x read shards)."""

    def __init__(self, device, max_local_reads, max_hits_per_source, group=None):
        import torch.distributed as dist
        L = _lib.load_library()
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = device
        self._c = C.c_void_p()
        blob = (C.c_uint8 * HANDLE_BYTES)()
        check(L.mtsvgpu_comm_create(device, self.rank, self.world, max_local_reads, max_hits_per_source,
                                    C.byref(self._c), blob))
        allh = gather_handles(bytes(blob), group)
        buf = (C.c_uint8 * len(allh)).from_buffer_copy(allh)
        check(L.mtsvgpu_comm_connect(self._c, buf))
        dist.barrier(group)  # every rank has mapped every buffer before the first batch stores into one

    def bin_reads(self, index, d_seqs_ptr, d_seq_off_ptr, n_reads, params):
        """mtsvgpu_bin_batch_chunked.  Returns (first_read, n_local_reads, d_pairs_ptr, d_off_ptr, n_pairs): the
        merged (tax_id, edit) lists of this rank's range, device pointers owned by the communicator."""
        L = _lib.load_library()
        ps = params.c_struct(2)
        first, nloc, nout = C.c_uint64(), C.c_uint64(), C.c_uint64()
        dp, do = C.c_void_p(), C.c_void_p()
        check(L.mtsvgpu_bin_batch_chunked(index._h, self._c, C.c_void_p(d_seqs_ptr), C.c_void_p(d_seq_off_ptr), n_reads,
                                          C.byref(ps), C.byref(first), C.byref(nloc), C.byref(dp), C.byref(do),
                                          C.byref(nout)))
        return first.value, nloc.value, dp.value, do.value, nout.value

    def bin_reads_tensors(self, index, d_reads, d_off, n_reads, params):
        """Same with torch tensors in and out: (first_read, pairs int32 [n, 2] = (tax_id, edit), offsets int64)."""
        import torch
        first, nloc, dp, do, nout = self.bin_reads(index, d_reads.data_ptr(), d_off.data_ptr(), n_reads, params)
        dev = torch.device("cuda", self.device)
        pairs = torch.as_tensor(_DevArray(dp, max(1, nout) * 8), device=dev).view(torch.int32).reshape(-1, 2)[:nout]
        offs = torch.as_tensor(_DevArray(do, (nloc + 1) * 8), device=dev).view(torch.int64)
        return first, pairs, offs

    def close(self):
        import torch.distributed as dist
        if self._c:
            dist.barrier(self.group)  # nobody may still be storing into a buffer that is about to go away
            _lib.load_library().mtsvgpu_comm_destroy(self._c)
            self._c = C.c_void_p()


def hybrid_groups(world, n_chunks):
    """Hybrid operation (SURVEY §8e row 3): `n_chunks` chunks on `world` GPUs, world = n_chunks x n_shards.  Rank r
    holds chunk r % n_chunks and works on read shard r // n_chunks; the ranks of one shard form one exchange group.
    Returns the list of rank lists, one per shard."""
    if n_chunks <= 0 or world % n_chunks:
        raise ValueError("world size %d is not a multiple of %d chunks" % (world, n_chunks))
    return [list(range(s * n_chunks, (s + 1) * n_chunks)) for s in range(world // n_chunks)]


class _DevArray:
    """Zero-copy view of a raw device pointer for torch.as_tensor (CUDA array interface v2)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 2}


def read_ranges(n_reads, world):
    """Contiguous ranges of reads owned by each rank: boundaries b[0..world]."""
    step = -(-n_reads // world) if world else 0
    return [min(n_reads, i * step) for i in range(world + 1)]


def _collapse_parts(fn, rec_bytes, device, stream, parts_hits, parts_counts, n_reads):
    """Runs the C collapse entry point `fn` (records of `rec_bytes` bytes).  Returns (uint8 tensor of the merged
    records, offsets int64 tensor [n_reads+1]), copies that own their memory."""
    import torch
    L = _lib.load_library()
    n = len(parts_hits)
    hp = (C.c_void_p * n)(*[C.c_void_p(t.data_ptr()) for t in parts_hits])
    cp = (C.c_void_p * n)(*[C.c_void_p(t.data_ptr()) for t in parts_counts])
    d_out, d_off, n_out = C.c_void_p(), C.c_void_p(), C.c_uint64()
    check(getattr(L, fn)(device, C.c_void_p(stream or 0), n, hp, cp, n_reads, C.byref(d_out), C.byref(d_off),
                         C.byref(n_out)))
    dev = torch.device("cuda", device)
    recs = torch.as_tensor(_DevArray(d_out.value, max(1, n_out.value) * rec_bytes), device=dev).clone()
    offs = torch.as_tensor(_DevArray(d_off.value, (n_reads + 1) * 8), device=dev).clone()
    L.mtsvgpu_device_free(d_out)
    L.mtsvgpu_device_free(d_off)
    return recs[: n_out.value * rec_bytes], offs.view(torch.int64)


def collapse_parts_device(device, stream, parts_hits, parts_counts, n_reads):
    """mtsv-collapse's mode TaxId on the device (src/collapse.rs:597-602): per read each TaxID once with its smallest
    edit, by ascending TaxID.  parts_hits / parts_counts: lists of torch CUDA tensors (uint8 bytes of mtsvgpu_hit[],
    int32 hits per read) for the same n_reads reads; stream: a CUDA stream handle or None.  Returns (pairs int32
    tensor [n_out, 2] = (tax_id, edit), offsets int64 tensor [n_reads+1])."""
    import torch
    pairs, offs = _collapse_parts("mtsvgpu_collapse_device", 8, device, stream, parts_hits, parts_counts, n_reads)
    return pairs.view(torch.int32).reshape(-1, 2), offs


def collapse_parts_device_taxid_gi(device, stream, parts_hits, parts_counts, n_reads):
    """mtsv-collapse's mode TaxIdGi on the device (src/collapse.rs:603-625): per read and (TaxID, GI) the hit with
    the smallest edit, ties to the smallest offset, listed by (TaxID, GI).  Same inputs as collapse_parts_device;
    returns (hits uint8 tensor of 24-byte mtsvgpu_hit records, offsets int64 tensor [n_reads+1])."""
    return _collapse_parts("mtsvgpu_collapse_device_taxid_gi", 24, device, stream, parts_hits, parts_counts, n_reads)
