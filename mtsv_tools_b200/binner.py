"""Results formatting of the binner (src/binner.rs:310-379)."""


def format_assignments(header, hits, long_info_output=False):
    """``write_assignments`` line for one read; '' when there are no hits (src/binner.rs:316-318).
    hits: iterable of objects/records with tax_id, gi, offset, edit."""
    best = {}
    for h in hits:
        tax, gi, off, edit = (int(h["tax_id"]), int(h["gi"]), int(h["offset"]), int(h["edit"])) \
            if not hasattr(h, "tax_id") else (int(h.tax_id), int(h.gi), int(h.offset), int(h.edit))
        key = (tax, gi, off) if long_info_output else tax
        if key not in best or edit < best[key]:
            best[key] = edit
    if not best:
        return ""
    if long_info_output:
        body = ",".join("%d-%d-%d=%d" % (k[0], k[1], k[2], best[k]) for k in sorted(best))
    else:
        body = ",".join("%d=%d" % (k, best[k]) for k in sorted(best))
    return "%s:%s\n" % (header, body)


def write_assignments(header, hits, writer, long_info_output=False):
    line = format_assignments(header, hits, long_info_output)
    if line:
        writer.write(line)


def results_lines(names, hits, hit_off, long_info_output=False):
    """Lines of a whole batch in read order (reads without hits produce no line)."""
    out = []
    for i, name in enumerate(names):
        a, b = int(hit_off[i]), int(hit_off[i + 1])
        if b > a:
            out.append(format_assignments(name, hits[a:b], long_info_output))
    return out


def assignment_lines(names, taxhits, off):
    """Default-format lines of a whole batch from the merged records of MGIndex.assign_reads* (each TaxID of a read
    once with its minimum edit, by ascending TaxID): the lines that results_lines(..., long_info_output=False) gives
    for the hits of the matching bin_reads* call."""
    out = []
    for i, name in enumerate(names):
        a, b = int(off[i]), int(off[i + 1])
        if b > a:
            body = ",".join("%d=%d" % (int(t["tax_id"]), int(t["edit"])) for t in taxhits[a:b])
            out.append("%s:%s\n" % (name, body))
    return out
