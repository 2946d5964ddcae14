"""Device memory and device selection of the library: a failed allocation leaves nothing behind that fails a later
call, every entry point that takes a device number checks its range, and the memory of every path comes back."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from mtsv_tools_b200 import LibraryError, MGIndex, chunked, load_library, synth  # noqa: E402
from mtsv_tools_b200._lib import check  # noqa: E402
from mtsv_tools_b200.build_index import suffix_array  # noqa: E402
from mtsv_tools_b200.chunked import _DevArray  # noqa: E402
from mtsv_tools_b200.index import edit_distance  # noqa: E402

EINVAL, EFORMAT, ENOMEM = -1, -3, -6


@pytest.fixture(scope="module")
def ref(oracle):
    cat, off, gi, tax = synth.make_reference(6, 30000, seed=11, n_frac=0.002, shared_frac=0.1)
    return cat, off, gi, tax, oracle.Index.build((cat, off), gi, tax, 64, 32)


@pytest.fixture(scope="module")
def reads(ref):
    """4000 reads of 150 bases, on the host and on the device (one slice: no empty last slice)."""
    cat, off = ref[0], ref[1]
    host = synth.make_reads(cat, off, 4000, 150, seed=12)  # (bytes, offsets)
    rcat, roff = host
    d_seqs = torch.from_numpy(np.concatenate([rcat, np.zeros(1, np.uint8)])).cuda()
    d_off = torch.from_numpy(np.asarray(roff, np.uint64).astype(np.int64)).cuda()
    return host, d_seqs, d_off, len(roff) - 1


def _from_parts(oix, bwt=None, **kw):
    return MGIndex.from_parts(oix.text, oix.bins(), oix.bwt if bwt is None else bwt, oix.sa_sample,
                              oix.sa_sample_rate, **kw)


def _assign_device(g, d_seqs, d_off, n):
    dt, do, nt = g.assign_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), n)
    recs = torch.as_tensor(_DevArray(dt, max(nt, 1) * 8), device="cuda").cpu().numpy()[: nt * 8]
    offs = torch.as_tensor(_DevArray(do, (n + 1) * 8), device="cuda").cpu().numpy()
    return nt, recs.tobytes(), offs.tobytes()


def test_failed_allocation_does_not_fail_the_next_call(ref, reads):
    """A batch whose result offsets cannot be allocated fails with ENOMEM in its first reserve, before any read of
    the offsets; the next batch on the same thread and handle runs as if it had not happened."""
    _, d_seqs, d_off, n = reads
    with _from_parts(ref[4]) as g:
        first = _assign_device(g, d_seqs, d_off, n)
        assert first[0] > 0
        with pytest.raises(LibraryError) as ei:
            g.bin_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), 2 ** 40)
        assert ei.value.code == ENOMEM, str(ei.value)
        assert _assign_device(g, d_seqs, d_off, n) == first


def test_device_out_of_range_is_einval(ref, tmp_path):
    cat, off, gi, tax, oix = ref
    bad = torch.cuda.device_count()
    path = str(tmp_path / "ref.index")
    oix.write(path)
    parts = ([torch.zeros(24, dtype=torch.uint8, device="cuda")], [torch.zeros(1, dtype=torch.int32, device="cuda")])
    L = load_library()
    calls = {
        "index_open": lambda: MGIndex.from_file(path, device=bad),
        "index_from_parts": lambda: _from_parts(oix, device=bad),
        "index_build": lambda: MGIndex.build(cat, off, gi, tax, device=bad),
        "suffix_array": lambda: suffix_array(oix.text, device=bad),
        "edit_distance": lambda: edit_distance([b"ACGT"], [b"ACGA"], device=bad),
        "collapse_device": lambda: chunked.collapse_parts_device(bad, None, *parts, 1),
        "collapse_device_taxid_gi": lambda: chunked.collapse_parts_device_taxid_gi(bad, None, *parts, 1),
        "comm_create": lambda: check(L.mtsvgpu_comm_create(bad, 0, 1, 16, 16, C.byref(C.c_void_p()),
                                                           (C.c_uint8 * chunked.HANDLE_BYTES)())),
    }
    for name, call in calls.items():
        with pytest.raises(LibraryError) as ei:
            call()
        assert ei.value.code == EINVAL, (name, str(ei.value))


def _free_bytes():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def test_device_memory_comes_back(ref, reads):
    """Indexes that are opened, used and closed, an index rejected after its device allocations, and the collapse
    and edit-distance entry points: after a warm-up round, further rounds leave the free device memory where it
    was, to well below the footprint of one open index.  One index runs host-API batches of several slices with
    per-stage timing on, so that its streams and events (both lanes, the emit events, the profiling pool, the
    overlapped copy-out) are in use when it is closed."""
    cat, off, gi, tax, oix = ref
    host, d_seqs, d_off, n = reads
    # two '$' in the BWT: found by the re-layout kernel, after the index's arrays are on the device
    bwt2 = np.array(oix.bwt, np.uint8)
    bwt2[np.flatnonzero(bwt2 != ord("$"))[0]] = ord("$")
    with _from_parts(oix) as g:
        hits, hoff = g.bin_reads(host)
    parts = ([torch.from_numpy(np.frombuffer(hits.tobytes(), np.uint8).copy()).cuda()] * 2,
             [torch.from_numpy((hoff[1:] - hoff[:-1]).astype(np.int32)).cuda()] * 2)
    rcat, roff = host
    pats = [rcat[roff[i]:roff[i] + 100].tobytes() for i in range(500)]
    texts = [rcat[roff[i]:roff[i + 1]].tobytes() for i in range(500, 1000)]
    footprint = 0

    def one_round(base):
        nonlocal footprint
        with _from_parts(oix) as g:
            g.bin_reads(host)
            footprint = max(footprint, base - _free_bytes())
        with MGIndex.build(cat, off, gi, tax) as g:
            g.bin_reads_device(d_seqs.data_ptr(), d_off.data_ptr(), n)
            footprint = max(footprint, base - _free_bytes())
        with _from_parts(oix, batch_reads=500) as g:  # 8 slices, alternating between the two lanes
            g.set_profiling(True)
            for _ in range(2):  # the second call copies its results out slice by slice
                g.bin_reads_pinned(host)
            footprint = max(footprint, base - _free_bytes())
        with pytest.raises(LibraryError) as ei:
            _from_parts(oix, bwt=bwt2)
        assert ei.value.code == EFORMAT, str(ei.value)
        chunked.collapse_parts_device(0, None, *parts, n)
        chunked.collapse_parts_device_taxid_gi(0, None, *parts, n)
        edit_distance(pats, texts)

    one_round(_free_bytes())
    base = _free_bytes()
    footprint = 0
    for _ in range(3):
        one_round(base)
    drift = base - _free_bytes()
    assert footprint > 8 << 20, footprint
    assert drift < footprint // 8, (drift, footprint)
