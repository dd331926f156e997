"""In-memory replacement of the per-locus `samtools faidx` subprocess (SURVEY.md 8f row 3).

The candidate stage of the reference spawns one `samtools faidx <fasta> <seqid>:<start>-<end>` process
per extend region (`dump_piece`, miR_PREFeR.py:1097-1108; also :1003, :2574-2597) and keeps
`"".join(stdout.split("\\n")[1:])`.  Once folding takes milliseconds that process storm is the next
wall-clock bottleneck.  `FastaIndex.fetch_region()` returns the same string from memory: host-only,
no GPU involved.  Semantics follow samtools' region rules: coordinates are 1-based and inclusive,
a region end beyond the contig is clipped, a start beyond the contig (or an unknown contig) gives
an empty sequence, letters are returned exactly as stored (case and IUPAC codes preserved), line
wrapping of the FASTA file is invisible, a region with a dangling dash ("seqid:3-") is empty (the
end parses as 0).  Pinned to the reference's own bundled samtools 0.1.18: tests/golden/faidx.json holds
its stdout and .fai for seeded FASTA files (tests/golden/make_golden_faidx.py; the binary only starts
against the no-op curses stub oracle/ncurses_stub.c because the image lacks libncurses.so.5).
"""
import os


class FastaIndex:
    def __init__(self, path):
        self.path = path
        self._seq = {}
        self._order = []
        name, chunks = None, []
        with open(path, "rb") as f:
            for raw in f:
                line = raw.rstrip(b"\r\n")
                if line.startswith(b">"):
                    if name is not None:
                        self._seq[name] = b"".join(chunks)
                    # samtools uses the first whitespace-delimited token of the header as the name
                    tok = line[1:].split(None, 1)
                    name = tok[0].decode("ascii") if tok else ""
                    if name not in self._seq:
                        self._order.append(name)
                    chunks = []
                elif name is not None:
                    chunks.append(line)
        if name is not None:
            self._seq[name] = b"".join(chunks)

    def names(self):
        return list(self._order)

    def length(self, seqid):
        return len(self._seq[seqid])

    def fetch(self, seqid, start, end):
        """Bases start..end (1-based, inclusive) of `seqid`; clipped like `samtools faidx`."""
        s = self._seq.get(seqid)
        if s is None:
            return ""
        start = max(int(start), 1)
        end = min(int(end), len(s))
        if start > end:
            return ""
        return s[start - 1:end].decode("ascii")

    def fetch_region(self, region):
        """`seqid:start-end`, `seqid:start` (to the end of the contig) or `seqid` -- the reference builds
        "seqid:start-(end-1)" from a half-open extend region (miR_PREFeR.py:1098)."""
        seqid, sep, span = region.rpartition(":")
        if not sep or seqid not in self._seq and region in self._seq:
            return self.fetch(region, 1, 1 << 62)      # a bare contig name (possibly containing ':')
        a, dash, b = span.replace(",", "").partition("-")
        try:
            start = int(a)
            end = (int(b) if b else 0) if dash else 1 << 62      # "seqid:3-": samtools 0.1.18 reads the missing end as 0
        except ValueError:
            return self.fetch(region, 1, 1 << 62)
        return self.fetch(seqid, start, end)

    def packed(self):
        """(names, bases, offsets): the contig names in file order, all their bases concatenated (bytes, exactly as
        stored) and uint64 offsets with contig k at bases[offsets[k]:offsets[k + 1]] -- the upload format of
        MirFold.upload_genome / mirfold_genome_upload.  fetch(names[k], s, e) == bases[offsets[k] + s - 1:...] after the
        same clipping."""
        import numpy as np
        names = list(self._order)
        off = np.zeros(len(names) + 1, np.uint64)
        if names:
            off[1:] = np.cumsum([len(self._seq[n]) for n in names], dtype=np.uint64)
        return names, b"".join(self._seq[n] for n in names), off

    def extend_region_sequence(self, seqid, extendregion):
        """Sequence of a half-open extend region [start, end) as dump_piece cuts it (:1097-1105)."""
        return self.fetch(seqid, extendregion[0], extendregion[1] - 1)

    def faidx_stdout(self, region, width=60):
        """What `samtools faidx fasta region` prints (header + lines of `width`), for callers that still
        parse the text like the reference does."""
        seq = self.fetch_region(region)
        lines = [">" + region] + [seq[k:k + width] for k in range(0, len(seq), width)]
        return "\n".join(lines) + "\n"


def write_fai(path):
    """Write the `.fai` index `samtools faidx fasta` would create (name, length, offset, bases per line,
    bytes per line), so that stages of the reference that only check for its existence keep working."""
    rows = []
    with open(path, "rb") as f:
        offset = 0
        name = None
        for raw in f:
            if raw.startswith(b">"):
                if name is not None:
                    rows.append((name, length, seq_off, lb, lw))
                tok = raw[1:].split(None, 1)
                name = tok[0].decode("ascii") if tok else ""
                length, seq_off, lb, lw = 0, offset + len(raw), 0, 0
            elif name is not None:
                body = raw.rstrip(b"\r\n")
                if lb == 0 and body:
                    lb, lw = len(body), len(raw)
                length += len(body)
            offset += len(raw)
        if name is not None:
            rows.append((name, length, seq_off, lb, lw))
    with open(path + ".fai", "w") as out:
        for r in rows:
            out.write("%s\t%d\t%d\t%d\t%d\n" % r)
    return path + ".fai"
