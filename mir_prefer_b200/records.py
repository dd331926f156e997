"""Locus records in, candidate structures out -- the fold stage without the FASTA/RNALfold text in
between (SURVEY.md 8f row 1).

In the reference the candidate stage writes every extend region as a two-line FASTA record
(`dump_piece`, miR_PREFeR.py:1070-1198), the fold stage pipes those files through RNALfold
(:3047-3119) and the predict stage parses the text back (:1541-1599).  Here the same record --
(seqid, region, strand, locus, 0/L/R tag, peaks, matures, genomic sequence) -- goes straight to
libmirfold and comes back as the tuples `get_structures_next_extendregion` would have produced.

What has to stay byte-compatible with the reference, and is pinned by tests:
  * the header line, because the parser reads `sp[2]` (locus, called "peak") and `sp[3]` (0/L/R)
    and because `write_fasta` / `write_rnalfold_text` must feed the unmodified reference stages;
  * `get_reverse_complement` (miR_PREFeR.py:232-239): the table only knows upper-case A T G C U
    (A->U, T->A, G->C, C->G, U->A); lower-case and IUPAC letters are reversed but NOT complemented;
  * an empty sequence still produces a record: RNALfold echoes the header and the blank line and
    prints nothing else (SURVEY A.6/A.7), the parser yields the record with no structures, so
    record count and order are those of the input.
"""
from collections import namedtuple

from . import structures as S

# region / locus are [start, end) in genome coordinates, exactly as dump_piece prints them;
# peaks = [(start, end, strand)], matures = [(start, end, strand, depth)];
# seq = the plus-strand genomic sequence of the region as `samtools faidx` returns it.
LocusRecord = namedtuple("LocusRecord", "seqid region strand locus tag peaks matures seq")

_COMPLEMENT = str.maketrans("ATGCU", "UACGA")


def get_complement(seq):
    """miR_PREFeR.py:232-235 -- upper-case ATGCU only, everything else is left as it is."""
    return seq.translate(_COMPLEMENT)


def get_reverse_complement(seq):
    """miR_PREFeR.py:238-239."""
    return get_complement(seq)[::-1]


def fold_sequence(rec):
    """The sequence line dump_piece writes for this record: minus-strand records are reverse
    complemented with the reference's table (:1131, :1177)."""
    return get_reverse_complement(rec.seq) if rec.strand == "-" else rec.seq


def header_line(rec):
    """`>SEQID:S-E STRAND LS-LE TAG s,e,strand;... [M:s-e/strand/depth]...` (:1124-1143, :1162-1179).
    Only the peaks of the record's own strand are listed when the region has peaks on both
    strands (:1158-1163, :1171-1176); pass them already filtered in that case."""
    peaks = ";".join("%s,%s,%s" % (p[0], p[1], p[2]) for p in rec.peaks)
    head = ">%s:%s-%s %s %s-%s %s %s" % (rec.seqid, rec.region[0], rec.region[1], rec.strand, rec.locus[0], rec.locus[1],
                                         rec.tag, peaks)
    for m in rec.matures:
        head += " M:%s-%s/%s/%s" % (m[0], m[1], m[2], m[3])
    return head


def parse_header(line):
    """Inverse of header_line (used to accept the reference's own FASTA shards as records)."""
    sp = line.strip().split()
    if len(sp) < 4 or not sp[0].startswith(">"):
        raise ValueError("not a candidate-region header: %r" % line)
    seqid, _, span = sp[0][1:].rpartition(":")
    rs, _, re_ = span.partition("-")
    ls, _, le = sp[2].partition("-")
    peaks, matures = [], []
    for tok in sp[4:]:
        if tok.startswith("M:"):
            pos, strand, depth = tok[2:].split("/")
            a, _, b = pos.partition("-")
            matures.append((int(a), int(b), strand, int(depth)))
        else:
            for p in tok.split(";"):
                a, b, strand = p.split(",")
                peaks.append((int(a), int(b), strand))
    return seqid, (int(rs), int(re_)), sp[1], (int(ls), int(le)), sp[3], peaks, matures


def records_from_fasta(text):
    """Records of a candidate FASTA shard written by the reference: two lines per record, the
    sequence line (possibly empty) already in fold orientation."""
    out = []
    lines = text.split("\n")
    for k, line in enumerate(lines):
        if line.startswith(">"):
            seq = lines[k + 1] if k + 1 < len(lines) and not lines[k + 1].startswith(">") else ""
            out.append(_Oriented(*(parse_header(line) + (seq,))))
    return out


class _Oriented(LocusRecord):
    """A record whose `seq` is already the line of the FASTA shard (fold orientation)."""
    __slots__ = ()


def _oriented_sequence(rec):
    return rec.seq if isinstance(rec, _Oriented) else fold_sequence(rec)


def write_fasta(records, path):
    """The candidate FASTA shard dump_piece would have written for these records."""
    with open(path, "w") as f:
        for rec in records:
            f.write(header_line(rec) + "\n")
            f.write(_oriented_sequence(rec) + "\n")


class RecordFold:
    """Folded records: structures for the predict stage and, on request, the RNALfold text."""

    def __init__(self, records, result, seq_of=None):
        self.records = records
        self.result = result
        self._seq_of = seq_of or _oriented_sequence   # genome records: extracted on the host (only the text needs it)

    def structures(self, minlen, minloop=3, native=True):
        """Generator of (which, peak, [(norm_energy, fold_start, ss, sstype)]) -- one per record,
        input order: what get_structures_next_extendregion(rnalfoldoutname, minlen) yields.
        native=True classifies with libmirfold's mirfold_classify(); False uses the Python rules."""
        per_unique = self.result.classify(minlen, minloop) if native else None
        for r, rec in enumerate(self.records):
            if native:
                found = list(per_unique[self.result.unique_index(r)])
            else:
                found = []
                for ss, e, start in self.result.hits(r):
                    if len(ss) >= minlen:
                        found.extend(S.classify(ss, e, start, minloop))
            yield (rec.tag, "%s-%s" % (rec.locus[0], rec.locus[1]), found)

    def rnalfold_text(self):
        data, offs = self.result.record_blocks()
        out = []
        for r, rec in enumerate(self.records):
            out.append(header_line(rec) + "\n")
            seq = self._seq_of(rec)
            if seq.split(None, 1)[:1] == []:      # blank line: echoed, not folded
                out.append(seq + "\n")
            else:
                b, e = self.result.block(r, offs)
                out.append(data[b:e].decode("ascii"))
        return "".join(out)

    def write_rnalfold_text(self, path):
        """Byte-identical to `RNALfold -L span < shard.fa`, for the unmodified reference predict stage."""
        with open(path, "w") as f:
            f.write(self.rnalfold_text())

    def close(self):
        self.result.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


_STRAND_CODE = {"+": 43, "-": 45}


def region_table(genome, records):
    """GENOME_REGION_DTYPE rows of the records' (seqid, region, strand) against `genome` (fold.Genome).  A seqid the
    genome does not have becomes contig -1 (an empty record); a strand other than '+' / '-' is rejected by the library."""
    import itertools
    import numpy as np
    from .fold import GENOME_REGION_DTYPE
    ids = genome.contig_ids
    flat = np.fromiter(itertools.chain.from_iterable((ids.get(r.seqid, -1), r.region[0], r.region[1], _STRAND_CODE.get(r.strand, 0))
                                                     for r in records), np.int32, count=4 * len(records))
    return flat.view(GENOME_REGION_DTYPE)


def _mature_table(records):
    """MATURE_DTYPE array of all records' matures, in record order, and the nseq+1 offsets."""
    import itertools
    import numpy as np
    from .fold import MATURE_DTYPE
    moff = np.zeros(len(records) + 1, np.uint64)
    moff[1:] = np.cumsum(np.fromiter((len(r.matures) for r in records), np.int64, count=len(records)), dtype=np.uint64)
    n = int(moff[-1])
    flat = np.fromiter(itertools.chain.from_iterable((m[0], m[1], ord(m[2]), m[3] if len(m) > 3 else 0) for r in records for m in r.matures),
                       np.int32, count=4 * n)
    return flat.view(MATURE_DTYPE), moff


def candidates_of_records(mf, records, span, minlen=55, minloop=3, min_mature_len=18, max_mature_len=24, genome=None):
    """Records -> (ss_records, DuplexTable) in ONE fused device pass (mirfold_fold_candidates): the fold, the candidate
    structures of get_structures_next_extendregion (miR_PREFeR.py:1566-1589) and get_maturestar_info (:1876-1999) for every
    (structure, mature) pair.  ss_records is what filter_next_loci consumes: (which, peak, structures) per record.
    genome (fold.Genome, from mf.upload_genome): every record is folded from its coordinates in the resident genome
    (mirfold_fold_candidates_regions) and its `seq` may be None; the result is the same."""
    import numpy as np
    from .predict import DuplexTable
    records = list(records)
    if genome is not None:
        matures, moff = _mature_table(records)
        cand = genome.fold_candidates(region_table(genome, records), span, matures, moff, minlen, minloop, min_mature_len,
                                      max_mature_len)
        ss_records = [(rec.tag, "%s-%s" % (rec.locus[0], rec.locus[1]), cand.structures(k)) for k, rec in enumerate(records)]
        return ss_records, DuplexTable.from_candidates(cand, records), cand
    seqs = [_oriented_sequence(r) for r in records]
    buf, off = mf.pack(seqs)
    matures, moff = [], [0]
    for r in records:
        matures.extend(r.matures)
        moff.append(len(matures))
    cand = mf.fold_candidates(buf, off, span, [[r.region[0], r.region[1]] for r in records], matures, np.array(moff, np.uint64),
                              minlen, minloop, min_mature_len, max_mature_len)
    ss_records = [(rec.tag, "%s-%s" % (rec.locus[0], rec.locus[1]), cand.structures(k)) for k, rec in enumerate(records)]
    return ss_records, DuplexTable.from_candidates(cand, records), cand


def candidate_precursors(cand, records, genome=None, only_passing=True):
    """The precursors hairpin_significance scores: (distinct precursor strings in order of first appearance, indices of the
    scored structures of cand, and for each of them the index of its precursor in the first list)."""
    import numpy as np
    st = cand.structs
    code0 = cand.verdicts["code"] == 0 if cand.nverdicts else np.zeros(0, bool)
    fs_all, ln_all = st["fold_start"].tolist(), st["len"].tolist()
    vb_all, vc_all = cand.verdict_begin.tolist(), cand.verdict_count.tolist()
    first, uniq, rows, which = {}, [], [], []
    for r in range(cand.nseq):
        b, c = int(cand.struct_begin[r]), int(cand.struct_count[r])
        seq = None
        for k in range(b, b + c):
            if only_passing and not code0[vb_all[k]:vb_all[k] + vc_all[k]].any():
                continue
            if seq is None:
                rec = records[r]
                seq = (genome.sequence(genome.contig_index(rec.seqid), rec.region[0], rec.region[1], rec.strand) if genome is not None
                       else _oriented_sequence(rec))
            p = seq[fs_all[k] - 1:fs_all[k] - 1 + ln_all[k]]
            if p not in first:
                first[p] = len(uniq)
                uniq.append(p)
            rows.append(k)
            which.append(first[p])
    return uniq, np.asarray(rows, np.int64), np.asarray(which, np.int64)


def hairpin_significance(mf, cand, records, n_shuffles, seed=0, mode="di", genome=None, only_passing=True, span=0):
    """MFE significance of the candidate precursors of `cand` (candidates_of_records' Candidates over `records`) against
    n_shuffles shuffles each (MirFold.shuffle_test; randfold's test).  The precursor of a structure is its record's folded
    sequence [fold_start - 1, fold_start - 1 + len); with genome= it is extracted on the host through Genome.sequence.
    only_passing=True scores only structures with at least one code-0 duplex verdict.  Identical precursors are folded
    once, so their rows are equal.  Returns one row per structure of cand, in cand's order: rec, struct (index within the
    record), fold_start, len, scored, then the SHUFFLE_DTYPE fields (zero counts and NaN statistics where not scored).
    Results depend on (seed, the distinct precursors in order of first appearance)."""
    import numpy as np
    from .fold import SHUFFLE_DTYPE
    dt = np.dtype([("rec", "<u4"), ("struct", "<u4"), ("fold_start", "<i4"), ("len", "<i4"), ("scored", "?")] + SHUFFLE_DTYPE.descr)
    out = np.zeros(cand.nstructs, dt)
    if cand.nstructs:   # structures of record r: structs[struct_begin[r] .. +struct_count[r])
        cnt = cand.struct_count.astype(np.int64)
        k = np.concatenate([np.arange(b, b + c, dtype=np.int64) for b, c in zip(cand.struct_begin.tolist(), cnt.tolist())])
        out["rec"][k] = np.repeat(np.arange(cand.nseq, dtype=np.int64), cnt)
        out["struct"][k] = k - np.repeat(cand.struct_begin.astype(np.int64), cnt)
    out["fold_start"], out["len"] = cand.structs["fold_start"], cand.structs["len"]
    for f in ("p_value", "mean", "sd", "z"):
        out[f] = np.nan
    uniq, rows, which = candidate_precursors(cand, list(records), genome, only_passing)
    if len(rows):
        res = mf.shuffle_test(uniq, n_shuffles, seed=seed, mode=mode, span=span)
        out["scored"][rows] = True
        for f in SHUFFLE_DTYPE.names:
            out[f][rows] = res[f][which]
    return out


def fold_records(mf, records, span, genome=None):
    """Fold LocusRecords on the device.  Identical oriented sequences (the reference writes
    duplicated records for both-strand L/R loci, SURVEY App. C) are folded once; record count and
    order are preserved because the predict stage pairs records positionally (:2364-2399).
    genome (fold.Genome): every record is folded from its coordinates (mirfold_fold_regions) and its `seq` may be None;
    records with the same (contig, clipped start, clipped end, strand) are folded once."""
    records = list(records)
    if genome is not None:
        return _fold_records_genome(records, span, genome)
    seqs = [_oriented_sequence(r) for r in records]
    first, uniq, index = {}, [], []
    for s in seqs:
        if s not in first:
            first[s] = len(uniq)
            uniq.append(s)
        index.append(first[s])
    return RecordFold(records, _Replicated(mf.fold(uniq, span), index))


def _fold_records_genome(records, span, genome):
    import numpy as np
    reg = region_table(genome, records)
    contig = reg["contig"].astype(np.int64)
    clen = np.where(contig >= 0, genome.lengths[np.maximum(contig, 0)] if len(genome.lengths) else 0, 0)
    s = np.maximum(reg["start"].astype(np.int64), 1)
    e = np.minimum(reg["end"].astype(np.int64) - 1, clen)
    empty = (contig < 0) | (s > e)
    key = np.stack([np.where(empty, -1, contig), np.where(empty, 0, s), np.where(empty, 0, e), reg["strand"]], axis=1)
    _, first, index = np.unique(key, axis=0, return_index=True, return_inverse=True)
    ureg = reg[first]                   # one representative record per distinct folded sequence
    res = genome.fold_regions(ureg, span)
    host = lambda: [genome.sequence(*(int(x) for x in r)) for r in ureg]   # noqa: E731 -- RNALfold text only
    seq_of = lambda rec: genome.sequence(genome.contig_index(rec.seqid), rec.region[0], rec.region[1], rec.strand)   # noqa: E731
    return RecordFold(records, _Replicated(res, index.reshape(-1).tolist(), host_seqs=host), seq_of)


class _Replicated:
    """View of a FoldResult through a record -> unique-sequence index."""

    def __init__(self, result, index, host_seqs=None):
        self._res, self._index = result, index
        self.stats = result.stats
        self._host_seqs = host_seqs     # genome results: the unique sequences, extracted on the host for record_blocks()

    def hits(self, r):
        return self._res.hits(self._index[r])

    def total(self, r):
        return self._res.total(self._index[r])

    def record_blocks(self):
        if self._host_seqs is not None:
            from .fold import MirFold
            self._res.set_inputs(*MirFold.pack(self._host_seqs()))
            self._host_seqs = None
        return self._res.record_blocks()

    def classify(self, minlen, minloop=3):
        return self._res.classify(minlen, minloop)

    def unique_index(self, r):
        return self._index[r]

    def block(self, r, offs):
        u = self._index[r]
        return int(offs[u]), int(offs[u + 1])

    def close(self):
        self._res.close()
