"""mtsv_tools_b200 — B200 (sm_100a) implementation of mtsv-binner's read-assignment hot path.

The product is the C-ABI shared library ``libmtsv_b200.so`` (include/mtsv_b200.h); this package
is the thin Python host mirror of the reference's interface for that path:

* :class:`MGIndex`  — ``MGIndex`` + ``from_file`` (src/index.rs:60-68, src/io.rs:115-122)
* :func:`MGIndex.matching_tax_ids` — src/index.rs:258-432 (one strand of one read)
* :func:`MGIndex.bin_reads` — the per-read worker of run_fastx_pipeline (src/binner.rs:77-131), batched
* :func:`MGIndex.assign_reads` — the same batch reduced on the device to the default results format
* :func:`write_assignments` — src/binner.rs:310-379

There is no CPU fallback: importing works anywhere, computing requires the CUDA library and a GPU.
"""
from ._lib import LibraryError, build_library, load_library  # noqa: F401
from .index import Hit, MGIndex, Params  # noqa: F401
from .binner import format_assignments, write_assignments, results_lines, assignment_lines  # noqa: F401

__version__ = "0.1.0"
