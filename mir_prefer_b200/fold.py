"""Host layer of the fold stage: the Python side of the drop-in boundary.

Mirrors the reference's fold-stage interface (/root/reference/miR_PREFeR.py):
  * fold_use_RNALfold(fastas, tmpdir, options, maxspan, chunksize)      MP:3047-3119
      -> MirFold.fold_fasta_files(): same inputs (FASTA shard paths, span), same outputs
         (one `<prefix>_rnalfoldoutput_<i>` text file per shard, byte-identical to RNALfold's).
  * `RNALfold -L <n>` stdin/stdout contract                              MP:3053, :3064
      -> MirFold.fold_text(): RNALfold-identical text for arbitrary RNALfold input text.
  * the hairpin lines parsed by get_structures_next_extendregion()       MP:1566-1573
      -> FoldResult.hits(r): (ss, energy_dcal, start) tuples without any text round trip.

All arithmetic happens in libmirfold.so on the GPU; this file only moves bytes.
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import MirfoldError

DEFAULT_PARAMSET = b"vienna-1.8.5-d1"
FLAG_WIDE = 1   # MIRFOLD_FLAG_WIDE: force the 32-bit fill kernel (results are identical)
FLAG_SERIAL = 2  # MIRFOLD_FLAG_SERIAL: one chunk at a time per device (disjoint per-stage device times)
DUPLEX_EXCEPTION = "EXCEPTION_UNBALANCED_STRUCTURE"   # verdict where the reference's get_maturestar_info raises
HIT_DTYPE = np.dtype([("start", "<i4"), ("len", "<i4"), ("mfe_dcal", "<i4"), ("reserved", "<i4"), ("ss_off", "<u8")])


class FoldResult:
    """Owns a mirfold_result.  Hit order inside a record is RNALfold's print order."""

    def __init__(self, lib, ptr, nseq, inputs=None, owner=None):
        self._lib = lib
        self._ptr = ptr
        self._inputs = inputs          # (uint8 buffer, uint64 offsets) the result was folded from
        self._owner = owner            # the MirFold it came from (the C library also lets a result outlive its context)
        r = ptr.contents
        self.nseq = int(r.nseq)
        self.nhits = int(r.nhits)
        self.ss_bytes = int(r.ss_bytes)
        self.stats = r.stats.as_dict()
        self.downloaded = bool(r.ss_arena) or self.nhits == 0
        self.hit_begin = self.hit_count = self.total_mfe_dcal = self.hit_table = self.arena = None
        if self.downloaded:
            if self.nseq:
                self.hit_begin = np.ctypeslib.as_array(r.hit_begin, shape=(self.nseq,))
                self.hit_count = np.ctypeslib.as_array(r.hit_count, shape=(self.nseq,))
                self.total_mfe_dcal = np.ctypeslib.as_array(r.total_mfe_dcal, shape=(self.nseq,))
            else:
                self.hit_begin, self.total_mfe_dcal = np.zeros(0, np.uint64), np.zeros(0, np.int32)
                self.hit_count = np.zeros(0, np.uint32)
            if self.nhits:
                raw = np.ctypeslib.as_array(C.cast(r.hits, C.POINTER(C.c_uint8)), shape=(self.nhits * C.sizeof(_lib.Hit),))
                self.hit_table = raw.view(HIT_DTYPE)
                self.arena = np.ctypeslib.as_array(C.cast(r.ss_arena, C.POINTER(C.c_uint8)), shape=(self.ss_bytes,))
            else:
                self.hit_table, self.arena = np.zeros(0, HIT_DTYPE), np.zeros(0, np.uint8)

    def hits(self, r):
        """[(dot_bracket, energy_dcal, start_1based)] of record r."""
        b = int(self.hit_begin[r])
        e = b + int(self.hit_count[r])
        out = []
        for h in self.hit_table[b:e]:
            o, n = int(h["ss_off"]), int(h["len"])
            out.append((self.arena[o:o + n].tobytes().decode("ascii"), int(h["mfe_dcal"]), int(h["start"])))
        return out

    def total(self, r):
        return int(self.total_mfe_dcal[r])

    def classify(self, minlen, minloop=3):
        """Candidate structures of every record, classified natively (mirfold_classify): a list per record of
        (norm_energy, fold_start, ss, sstype) -- the tuples get_structures_next_extendregion() builds
        (miR_PREFeR.py:1566-1589)."""
        return classify_result(self._lib, self._ptr, self.nseq, self.arena, minlen, minloop)

    def set_inputs(self, buf, off):
        """The packed sequences the result was folded from, for record_blocks() of a result that was folded from genome
        coordinates (Genome.fold_regions): the caller extracts them on the host when it wants the RNALfold text."""
        self._inputs = (np.ascontiguousarray(buf, np.uint8), np.ascontiguousarray(off, np.uint64))

    def record_blocks(self):
        """RNALfold's output of every record (hit lines, converted sequence, total line) as one bytes object
        plus nseq+1 offsets -- formatted natively by mirfold_format_records() (include/mirfold.h)."""
        if self._inputs is None or not self.downloaded:
            raise MirfoldError(-3, "record_blocks() needs a downloaded result of fold()/fold_packed()")
        buf, off = self._inputs
        text, rec_off = C.c_void_p(), C.POINTER(C.c_uint64)()
        rc = self._lib.mirfold_format_records(self._ptr, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              self.nseq, C.byref(text), C.byref(rec_off))
        if rc != 0:
            raise MirfoldError(rc, self._lib.mirfold_strerror(rc).decode())
        try:
            offs = np.ctypeslib.as_array(rec_off, shape=(self.nseq + 1,)).copy() if self.nseq else np.zeros(1, np.uint64)
            data = C.string_at(text, int(offs[-1]))
        finally:
            self._lib.mirfold_free_text(text, rec_off)
        return data, offs

    def close(self):
        if self._ptr is not None:
            self.hit_begin = self.hit_count = self.total_mfe_dcal = self.hit_table = self.arena = None
            self._lib.mirfold_free_result(self._ptr)
            self._ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


DUPLEX_QUERY_DTYPE = np.dtype([("ss_off", "<u8"), ("ss_len", "<i4"), ("fold_start", "<i4"), ("mature_start", "<i4"),
                               ("mature_end", "<i4"), ("region_start", "<i4"), ("region_end", "<i4"), ("strand", "<i4"),
                               ("reserved", "<i4")])
DUPLEX_VERDICT_DTYPE = np.dtype([(n, "<i4") for n in ("code", "star_start", "star_end", "fold_start", "fold_end", "star_ss_begin",
                                                     "star_ss_end", "mature_ss_begin", "mature_ss_end", "prime5", "total_dots",
                                                     "total_bps")])
STRUCT_DTYPE = np.dtype([("rec", "<u4"), ("fold_start", "<i4"), ("sstype", "<i4"), ("len", "<i4"), ("ss_off", "<u8"),
                         ("norm_energy", "<f8")])


def classify_result(lib, res_ptr, nseq, arena, minlen, minloop=3):
    """mirfold_classify() over a mirfold_result; `arena` is the result's ss_arena as a uint8 array."""
    out, n_out, rec_begin = C.POINTER(_lib.Structure)(), C.c_uint64(), C.POINTER(C.c_uint64)()
    rc = lib.mirfold_classify(res_ptr, int(minlen), int(minloop), C.byref(out), C.byref(n_out), C.byref(rec_begin))
    if rc != 0:
        raise MirfoldError(rc, "mirfold_classify: a hit without any base pair (the reference's filter_ss raises KeyError here)")
    try:
        n = int(n_out.value)
        rb = np.ctypeslib.as_array(rec_begin, shape=(nseq + 1,)).copy() if nseq else np.zeros(1, np.uint64)
        tab = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(max(n, 1) * C.sizeof(_lib.Structure),)).view(STRUCT_DTYPE)[:n].copy()
    finally:
        lib.mirfold_free_structures(out, rec_begin)
    raw = arena.tobytes() if n else b""
    ne, fs, ty, ln, so = (tab[k].tolist() for k in ("norm_energy", "fold_start", "sstype", "len", "ss_off"))
    per_rec = []
    for r in range(nseq):
        b, e = int(rb[r]), int(rb[r + 1])
        per_rec.append([(ne[k], fs[k], raw[so[k]:so[k] + ln[k]].decode("ascii"), ty[k]) for k in range(b, e)])
    return per_rec


def convert_sequence(tok):
    """RNALfold main(): upper-case, T->U (SURVEY A.6)."""
    return tok.upper().replace("T", "U")


def parse_rnalfold_input(text):
    """Split RNALfold stdin into ('echo', line) / ('seq', token) items exactly like RNALfold's main():
    lines starting with '>' or '*' and empty lines are echoed; '@' ends; the first whitespace-delimited
    token of any other line is a sequence."""
    items = []
    lines = text.split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    for line in lines:
        if line == "" or line[0] in ">*":
            items.append(("echo", line))
            continue
        if line == "@":
            break
        tok = line.split(None, 1)
        items.append(("seq", tok[0] if tok else ""))
    return items


def format_record(seq_token, hits, total_dcal):
    out = []
    for ss, e, start in hits:
        out.append("%s (%6.2f) %4d\n" % (ss, e / 100., start))
    out.append("%s\n (%6.2f)\n" % (convert_sequence(seq_token), total_dcal / 100.))
    return "".join(out)


class FoldChunk:
    """One chunk handed to a fold_stream() callback: numpy views that are only valid during the call."""

    def __init__(self, c):
        n, nh = int(c.n_records), int(c.nhits)
        self.device = int(c.device)
        self.records = np.ctypeslib.as_array(c.record, shape=(n,)) if n else np.zeros(0, np.uint32)
        self.hit_begin = np.ctypeslib.as_array(c.hit_begin, shape=(n,)) if n else np.zeros(0, np.uint64)
        self.hit_count = np.ctypeslib.as_array(c.hit_count, shape=(n,)) if n else np.zeros(0, np.uint32)
        self.total_mfe_dcal = np.ctypeslib.as_array(c.total_mfe_dcal, shape=(n,)) if n else np.zeros(0, np.int32)
        self.nhits, self.ss_bytes = nh, int(c.ss_bytes)
        if nh:
            raw = np.ctypeslib.as_array(C.cast(c.hits, C.POINTER(C.c_uint8)), shape=(nh * C.sizeof(_lib.Hit),))
            self.hit_table = raw.view(HIT_DTYPE)
            self.arena = np.ctypeslib.as_array(C.cast(c.ss_arena, C.POINTER(C.c_uint8)), shape=(self.ss_bytes,))
        else:
            self.hit_table, self.arena = np.zeros(0, HIT_DTYPE), np.zeros(0, np.uint8)

    def hits(self, k):
        """[(dot_bracket, energy_dcal, start_1based)] of the chunk's k-th record (input record self.records[k])."""
        b = int(self.hit_begin[k])
        out = []
        for h in self.hit_table[b:b + int(self.hit_count[k])]:
            o, n = int(h["ss_off"]), int(h["len"])
            out.append((self.arena[o:o + n].tobytes().decode("ascii"), int(h["mfe_dcal"]), int(h["start"])))
        return out


MATURE_DTYPE = np.dtype([("start", "<i4"), ("end", "<i4"), ("strand", "<i4"), ("depth", "<i4")])
REGION_DTYPE = np.dtype([("start", "<i4"), ("end", "<i4")])
# mirfold_genome_region: contig index (-1 = not in the FASTA), [start, end) as dump_piece prints it, strand ord('+') / ord('-')
GENOME_REGION_DTYPE = np.dtype([("contig", "<i4"), ("start", "<i4"), ("end", "<i4"), ("strand", "<i4")])


# mirfold_shuffle_stat plus the fields derived from it (shuffle_test)
SHUFFLE_MODES = {"mono": 1, "di": 2}   # MIRFOLD_SHUFFLE_MONO / MIRFOLD_SHUFFLE_DI
SHUFFLE_STAT_DTYPE = np.dtype([("native_dcal", "<i4"), ("n_le", "<u4"), ("sum_dcal", "<i8"), ("sumsq_dcal", "<i8")])
SHUFFLE_DTYPE = np.dtype(SHUFFLE_STAT_DTYPE.descr + [("p_value", "<f8"), ("mean", "<f8"), ("sd", "<f8"), ("z", "<f8")])


def shuffle_fields(stat, n_shuffles):
    """SHUFFLE_DTYPE rows from SHUFFLE_STAT_DTYPE rows of a test with K = n_shuffles shuffles: p = (n_le + 1) / (K + 1),
    mean and population sd of the shuffles' totals (dcal), z = (native - mean) / sd (NaN when sd == 0).  The variance is
    taken from the integer sums exactly (K * sumsq - sum^2 in Python integers), so sd is 0 exactly when all shuffles tie."""
    K = int(n_shuffles)
    out = np.zeros(len(stat), SHUFFLE_DTYPE)
    for f in SHUFFLE_STAT_DTYPE.names:
        out[f] = stat[f]
    out["p_value"] = (out["n_le"].astype(np.float64) + 1.0) / (K + 1)
    out["mean"] = out["sum_dcal"] / K
    var = [(K * q - s * s) / (K * K) for s, q in zip(stat["sum_dcal"].tolist(), stat["sumsq_dcal"].tolist())]
    out["sd"] = np.sqrt(np.asarray(var, np.float64)) if len(var) else 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        out["z"] = np.where(out["sd"] > 0, (out["native_dcal"] - out["mean"]) / out["sd"], np.nan)
    return out


def _mature_array(matures):
    """MATURE_DTYPE array of matures given as such an array or as (start, end, strand_char, depth) tuples."""
    if isinstance(matures, np.ndarray) and matures.dtype == MATURE_DTYPE:
        return np.ascontiguousarray(matures)
    mat = np.zeros(len(matures), MATURE_DTYPE)
    for k, m in enumerate(matures):
        mat[k] = (m[0], m[1], ord(m[2]) if isinstance(m[2], str) else int(m[2]), m[3] if len(m) > 3 else 0)
    return mat


def _stream(callback, call):
    """Run call(fn, stats) with fn a C trampoline handing FoldChunks to callback; an exception inside the callback
    aborts the fold (the library returns MIRFOLD_ERR_CALLBACK) and is re-raised here.  Returns (rc, stats dict)."""
    err = []

    def tramp(_user, cptr):
        try:
            callback(FoldChunk(cptr.contents))
            return 0
        except BaseException as e:   # noqa: BLE001 -- must not propagate through the C frames
            err.append(e)
            return 1

    fn = _lib.CHUNK_FN(tramp)
    st = _lib.Stats()
    rc = call(fn, st)
    if err:
        raise err[0]
    return rc, st.as_dict()


class Candidates:
    """Result of MirFold.fold_candidates(): per record the candidate structures the predict stage consumes and, for every
    (structure, size-admissible mature) pair, the get_maturestar_info() verdict -- computed on the device right after
    traceback (mirfold_fold_candidates).  Everything is copied out of the library's buffers at construction."""

    def __init__(self, lib, ptr, matures, mature_off):
        c = ptr.contents
        self.nseq, self.nstructs, self.nverdicts, self.nhits = int(c.nseq), int(c.nstructs), int(c.nverdicts), int(c.nhits)
        self.stats = c.stats.as_dict()
        ns, nv, n = self.nstructs, self.nverdicts, self.nseq
        self.struct_begin = np.ctypeslib.as_array(c.struct_begin, shape=(n,)).copy() if n else np.zeros(0, np.uint64)
        self.struct_count = np.ctypeslib.as_array(c.struct_count, shape=(n,)).copy() if n else np.zeros(0, np.uint32)
        self.structs = (np.ctypeslib.as_array(C.cast(c.structs, C.POINTER(C.c_uint8)), shape=(ns * C.sizeof(_lib.Structure),))
                        .view(STRUCT_DTYPE).copy() if ns else np.zeros(0, STRUCT_DTYPE))
        self.arena = C.string_at(c.ss_arena, int(c.ss_bytes)) if ns else b""
        self.verdict_begin = np.ctypeslib.as_array(c.verdict_begin, shape=(ns,)).copy() if ns else np.zeros(0, np.uint64)
        self.verdict_count = np.ctypeslib.as_array(c.verdict_count, shape=(ns,)).copy() if ns else np.zeros(0, np.uint32)
        self.verdicts = (np.ctypeslib.as_array(C.cast(c.verdicts, C.POINTER(C.c_uint8)), shape=(nv * C.sizeof(_lib.DuplexVerdict),))
                         .view(DUPLEX_VERDICT_DTYPE).copy() if nv else np.zeros(0, DUPLEX_VERDICT_DTYPE))
        self.verdict_mature = np.ctypeslib.as_array(c.verdict_mature, shape=(nv,)).copy() if nv else np.zeros(0, np.uint32)
        self._matures, self._mature_off = matures, mature_off
        self._names = {k: lib.mirfold_duplex_fail_name(k).decode() for k in list(range(12)) + [100]}
        lib.mirfold_free_candidates(ptr)

    def _ss(self, k):
        o, n = int(self.structs["ss_off"][k]), int(self.structs["len"][k])
        return self.arena[o:o + n].decode("ascii")

    def structures(self, r):
        """[(norm_energy, fold_start, ss, sstype)] of record r: get_structures_next_extendregion()'s third tuple field."""
        b = int(self.struct_begin[r])
        st = self.structs
        return [(float(st["norm_energy"][k]), int(st["fold_start"][k]), self._ss(k), int(st["sstype"][k]))
                for k in range(b, b + int(self.struct_count[r]))]

    def verdicts_of(self, r):
        """[(structure index within the record, mature tuple (start, end, strand, depth), verdict)] with the verdict in
        get_maturestar_info()'s own format (9-tuple or FAIL_* string; DUPLEX_EXCEPTION where the reference raises)."""
        out = []
        b = int(self.struct_begin[r])
        mb = int(self._mature_off[r])
        for k in range(b, b + int(self.struct_count[r])):
            ss = self._ss(k)
            vb = int(self.verdict_begin[k])
            for v in range(vb, vb + int(self.verdict_count[k])):
                m = self._matures[mb + int(self.verdict_mature[v])]
                out.append((k - b, (int(m["start"]), int(m["end"]), chr(int(m["strand"])), int(m["depth"])), self._verdict(ss, v)))
        return out

    def _verdict(self, ss, v):
        V = self.verdicts[v]
        c = int(V["code"])
        if c != 0:
            return self._names[c]
        return (int(V["star_start"]), int(V["star_end"]), int(V["fold_start"]), int(V["fold_end"]),
                ss[int(V["star_ss_begin"]):int(V["star_ss_end"])], bool(V["prime5"]),
                ss[int(V["mature_ss_begin"]):int(V["mature_ss_end"])], int(V["total_dots"]), int(V["total_bps"]))


class Batch:
    """Records sharded over the context's devices with their sequences resident in HBM (mirfold_batch_*)."""

    def __init__(self, owner, ptr, nseq, inputs):
        self._owner, self._ptr, self.nseq, self._inputs = owner, ptr, nseq, inputs

    def fold(self, download=False, flags=0):
        res = C.POINTER(_lib.Result)()
        rc = self._owner._lib.mirfold_batch_fold(self._owner._ctx, self._ptr, int(flags), 1 if download else 0, C.byref(res))
        if rc != 0:
            self._owner._raise(rc)
        return FoldResult(self._owner._lib, res, self.nseq, inputs=self._inputs if download else None, owner=self._owner)

    def close(self):
        if self._ptr:
            self._owner._lib.mirfold_batch_free(self._ptr)
            self._ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class Genome:
    """A FASTA resident in HBM on every device of its context (mirfold_genome_*): records are given as coordinates
    (GENOME_REGION_DTYPE rows) and the extend regions are cut, reverse-complemented and encoded on the device -- what
    dump_piece does with `samtools faidx` per record (miR_PREFeR.py:1097-1108, :1131, :1177), without the strings.
    Results equal those of the text entry points on FastaIndex.extend_region_sequence + records.fold_sequence."""

    def __init__(self, owner, ptr, index, names, off):
        self._owner, self._ptr, self.index = owner, ptr, index
        self.names = list(names)
        self.lengths = np.diff(off.astype(np.int64))
        self.contig_ids = {n: k for k, n in enumerate(self.names)}

    def contig_index(self, seqid):
        """Index of seqid in the upload, -1 for a seqid the FASTA does not have (an empty record, like samtools)."""
        return self.contig_ids.get(seqid, -1)

    def regions(self, seqids, starts, ends, strands):
        """GENOME_REGION_DTYPE array from per-record seqids, [start, end) and '+' / '-' strands."""
        reg = np.zeros(len(seqids), GENOME_REGION_DTYPE)
        reg["contig"] = [self.contig_ids.get(s, -1) for s in seqids]
        reg["start"], reg["end"] = starts, ends
        reg["strand"] = [ord(s) if isinstance(s, str) and len(s) == 1 else 0 for s in strands]
        return reg

    def sequence(self, contig, start, end, strand):
        """The folded sequence of one region, extracted on the host (FastaIndex + the reference's reverse complement)."""
        from .records import get_reverse_complement
        if contig < 0:
            return ""
        s = self.index.extend_region_sequence(self.names[contig], (int(start), int(end)))
        return get_reverse_complement(s) if strand in (45, "-") else s

    @staticmethod
    def _table(regions):
        if isinstance(regions, np.ndarray) and regions.dtype == GENOME_REGION_DTYPE:
            return np.ascontiguousarray(regions)
        ra = np.asarray(regions, np.int64).reshape(-1, 4)
        reg = np.zeros(len(ra), GENOME_REGION_DTYPE)
        for k, name in enumerate(GENOME_REGION_DTYPE.names):
            reg[name] = ra[:, k]
        return reg

    def _args(self, regions):
        if not self._ptr:
            raise MirfoldError(-3, "the genome was closed")
        reg = self._table(regions)
        return reg, (self._owner._ctx, self._ptr, reg.ctypes.data_as(C.c_void_p), len(reg))

    def fold_regions(self, regions, span, flags=0):
        """mirfold_fold_regions(): MirFold.fold_packed() of the regions' sequences.  record_blocks() of the result needs
        the sequences: FoldResult.set_inputs(*MirFold.pack([...Genome.sequence...]))."""
        reg, head = self._args(regions)
        res = C.POINTER(_lib.Result)()
        rc = self._owner._lib.mirfold_fold_regions(*head, int(span), int(flags), C.byref(res))
        if rc != 0:
            self._owner._raise(rc)
        return FoldResult(self._owner._lib, res, len(reg), owner=self._owner)

    def fold_regions_stream(self, regions, span, callback, flags=0):
        """mirfold_fold_regions_stream(): MirFold.fold_stream() of the regions' sequences.  Returns the stats dict."""
        reg, head = self._args(regions)
        rc, st = _stream(callback, lambda fn, st: self._owner._lib.mirfold_fold_regions_stream(
            *head, int(span), int(flags), fn, None, C.byref(st)))
        if rc != 0:
            self._owner._raise(rc)
        return st

    def fold_candidates(self, regions, span, matures, mature_off, minlen=55, minloop=3, min_mature_len=18, max_mature_len=24,
                        flags=0):
        """mirfold_fold_candidates_regions(): MirFold.fold_candidates() of the regions' sequences, with each record's
        (start, end) as its duplex region."""
        reg, head = self._args(regions)
        mat = _mature_array(matures)
        moff = np.ascontiguousarray(mature_off, np.uint64)
        res = C.POINTER(_lib.Candidates)()
        rc = self._owner._lib.mirfold_fold_candidates_regions(*head, int(span), int(flags), mat.ctypes.data_as(C.c_void_p),
                                                              moff.ctypes.data_as(C.POINTER(C.c_uint64)), int(minlen), int(minloop),
                                                              int(min_mature_len), int(max_mature_len), C.byref(res))
        if rc != 0:
            self._owner._raise(rc)
        return Candidates(self._owner._lib, res, mat, moff)

    def close(self):
        if self._ptr:
            self._owner._lib.mirfold_genome_free(self._ptr)
            self._ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def plan_shards(lengths, span, n_shards):
    """The library's own shard plan (mirfold_plan_shards: greedy LPT by DP cells -- what a context of n_shards devices
    does with these records).  Host-only.  Returns (shard_of[nseq] uint32, shard_cells[n_shards] uint64)."""
    lib = _lib.load()
    lengths = np.asarray(lengths, np.uint64)
    off = np.zeros(len(lengths) + 1, np.uint64)
    off[1:] = np.cumsum(lengths, dtype=np.uint64)
    shard_of = np.zeros(len(lengths), np.uint32)
    cells = np.zeros(n_shards, np.uint64)
    rc = lib.mirfold_plan_shards(off.ctypes.data_as(C.POINTER(C.c_uint64)), len(lengths), int(span), int(n_shards),
                                 shard_of.ctypes.data_as(C.POINTER(C.c_uint32)), cells.ctypes.data_as(C.POINTER(C.c_uint64)))
    if rc != 0:
        raise MirfoldError(rc, lib.mirfold_strerror(rc).decode())
    return shard_of, cells


def plan_fill_units(n, span):
    """How the band fill cuts a locus of n bases at this span into fill units (mirfold_plan_fill_units; host-only).
    Returns a dict: kernel (0 = generic, else the bucket stride), stride, tile_len, tile_step, n_units, dmax, band_cells."""
    lib = _lib.load()
    fp = _lib.FillPlan()
    rc = lib.mirfold_plan_fill_units(int(n), int(span), C.byref(fp))
    if rc != 0:
        raise MirfoldError(rc, lib.mirfold_strerror(rc).decode())
    return {k: int(getattr(fp, k)) for k, _ in _lib.FillPlan._fields_}


SEGMENT_DTYPE = np.dtype([("tile_first", np.int32), ("tile_last", np.int32), ("halo_tiles", np.int32), ("row_first", np.int32),
                          ("row_last", np.int32), ("reserved", np.int32), ("device_bytes", np.uint64)])


def plan_segments(n, span, budget_bytes):
    """How the fold runs a locus of n bases at this span with budget_bytes of device memory (mirfold_plan_segments;
    host-only): a structured array (SEGMENT_DTYPE) of segments in the order they run, 3' end first -- owned tiles
    tile_first..tile_last, halo_tiles more above them, owned rows row_first..row_last and device_bytes.  One segment when
    the locus fits the budget or is one fill unit."""
    lib = _lib.load()
    cnt = C.c_uint32(0)
    rc = lib.mirfold_plan_segments(int(n), int(span), int(budget_bytes), None, 0, C.byref(cnt))
    if rc != 0:
        raise MirfoldError(rc, lib.mirfold_strerror(rc).decode())
    out = np.zeros(cnt.value, SEGMENT_DTYPE)
    rc = lib.mirfold_plan_segments(int(n), int(span), int(budget_bytes), out.ctypes.data, cnt.value, C.byref(cnt))
    if rc != 0:
        raise MirfoldError(rc, lib.mirfold_strerror(rc).decode())
    return out


class MirFold:
    """A libmirfold context (one per process; `devices` = CUDA ordinals, default current device)."""

    def __init__(self, devices=None, param_set=DEFAULT_PARAMSET):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            rc = self._lib.mirfold_open(C.byref(self._ctx), arr, len(devices), param_set)
        else:
            rc = self._lib.mirfold_open(C.byref(self._ctx), None, 0, param_set)
        if rc != 0:
            raise MirfoldError(rc, self._lib.mirfold_strerror(rc).decode())

    def close(self):
        if self._ctx:
            self._lib.mirfold_close(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _raise(self, rc):
        raise MirfoldError(rc, "%s (%s)" % (self._lib.mirfold_strerror(rc).decode(),
                                            self._lib.mirfold_last_error(self._ctx).decode()))

    @staticmethod
    def pack(seqs):
        """list of str/bytes -> (uint8 buffer, uint64 offsets)."""
        bs = [s.encode("latin-1", "replace") if isinstance(s, str) else bytes(s) for s in seqs]
        off = np.zeros(len(bs) + 1, np.uint64)
        if bs:
            off[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
        buf = np.frombuffer(b"".join(bs), np.uint8) if bs else np.zeros(0, np.uint8)
        return buf, off

    def fold_packed(self, buf, off, span, flags=0):
        """buf: uint8 array of concatenated raw sequence tokens, off: uint64[nseq+1]."""
        buf = np.ascontiguousarray(buf, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        nseq = len(off) - 1
        res = C.POINTER(_lib.Result)()
        rc = self._lib.mirfold_fold(self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                    nseq, int(span), int(flags), C.byref(res))
        if rc != 0:
            self._raise(rc)
        return FoldResult(self._lib, res, nseq, inputs=(buf, off), owner=self)

    def fold_stream(self, buf, off, span, callback, flags=0):
        """mirfold_fold_stream(): fold like fold_packed() but hand the results to callback(FoldChunk) chunk by chunk
        while later chunks are still computing (the whole result never sits in host memory; replaces the
        reference's 2*CHECKPOINT_SIZE-line loop, miR_PREFeR.py:3022-3044).  Chunks arrive in completion order;
        FoldChunk.records names the input records.  Returns the call's stats dict."""
        buf = np.ascontiguousarray(buf, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        rc, st = _stream(callback, lambda fn, st: self._lib.mirfold_fold_stream(
            self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)), len(off) - 1, int(span),
            int(flags), fn, None, C.byref(st)))
        if rc != 0:
            self._raise(rc)
        return st

    def fold_candidates(self, buf, off, span, regions, matures, mature_off, minlen=55, minloop=3, min_mature_len=18,
                        max_mature_len=24, flags=0):
        """mirfold_fold_candidates(): fold + stage 1 (candidate structures) + stage 3 (duplex verdicts for every candidate
        structure x size-admissible mature of its record), all on the device; only the candidates are downloaded.
        regions: (nseq, 2) ints [start, end); matures: array of MATURE_DTYPE (or (start, end, strand_char, depth) tuples);
        mature_off: nseq+1 offsets into matures."""
        buf = np.ascontiguousarray(buf, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        nseq = len(off) - 1
        reg = np.zeros(nseq, REGION_DTYPE)
        if nseq:
            ra = np.asarray(regions, np.int64).reshape(nseq, 2)
            reg["start"], reg["end"] = ra[:, 0], ra[:, 1]
        mat = _mature_array(matures)
        moff = np.ascontiguousarray(mature_off, np.uint64)
        res = C.POINTER(_lib.Candidates)()
        rc = self._lib.mirfold_fold_candidates(self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                               nseq, int(span), int(flags), reg.ctypes.data_as(C.c_void_p),
                                               mat.ctypes.data_as(C.c_void_p), moff.ctypes.data_as(C.POINTER(C.c_uint64)),
                                               int(minlen), int(minloop), int(min_mature_len), int(max_mature_len), C.byref(res))
        if rc != 0:
            self._raise(rc)
        return Candidates(self._lib, res, mat, moff)

    def upload(self, buf, off, span):
        """mirfold_batch_upload(): shard the records over the context's devices and keep their sequences in HBM."""
        buf = np.ascontiguousarray(buf, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        ptr = C.c_void_p()
        rc = self._lib.mirfold_batch_upload(self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                            len(off) - 1, int(span), C.byref(ptr))
        if rc != 0:
            self._raise(rc)
        return Batch(self, ptr, len(off) - 1, (buf, off))

    def upload_genome(self, index):
        """mirfold_genome_upload(): keep the FASTA of `index` (a FastaIndex) in HBM on every device of this context.
        Returns a Genome (a context manager; close() frees the device copies)."""
        names, bases, off = index.packed()
        ptr = C.c_void_p()
        rc = self._lib.mirfold_genome_upload(self._ctx, bases, off.ctypes.data_as(C.POINTER(C.c_uint64)), len(names), C.byref(ptr))
        if rc != 0:
            self._raise(rc)
        return Genome(self, ptr, index, names, off)

    def fold(self, seqs, span, flags=0):
        buf, off = self.pack(seqs)
        return self.fold_packed(buf, off, span, flags)

    def fold_device(self, d_ptr, off, span, stream=None, flags=0):
        """Kernel-only path: raw sequences already in HBM at d_ptr (int), results stay on device."""
        off = np.ascontiguousarray(off, np.uint64)
        res = C.POINTER(_lib.Result)()
        rc = self._lib.mirfold_fold_device(self._ctx, C.c_void_p(d_ptr), None, off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                           len(off) - 1, int(span), int(flags), C.c_void_p(stream or 0), C.byref(res))
        if rc != 0:
            self._raise(rc)
        return FoldResult(self._lib, res, len(off) - 1, owner=self)

    @staticmethod
    def _shuffle_mode(mode):
        if mode not in SHUFFLE_MODES:
            raise MirfoldError(-3, "shuffle mode must be one of %s, not %r" % (sorted(SHUFFLE_MODES), mode))
        return SHUFFLE_MODES[mode]

    def shuffle_test(self, seqs, n_shuffles, seed=0, mode="di", span=0, flags=0, with_stats=False):
        """mirfold_shuffle_test(): the MFE of every sequence against n_shuffles shuffles of it (randfold's test), folded on
        the device.  mode "di" keeps dinucleotide counts (Altschul-Erickson), "mono" the base composition; span 0 folds
        globally (sequences up to 4096 nt).  Returns a SHUFFLE_DTYPE array, one row per sequence (energies in dcal), and
        with with_stats=True also the call's stats dict."""
        buf, off = self.pack(seqs)
        stat = np.zeros(len(off) - 1, SHUFFLE_STAT_DTYPE)
        st = _lib.Stats()
        rc = self._lib.mirfold_shuffle_test(self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                            len(off) - 1, int(span), int(flags), self._shuffle_mode(mode), int(n_shuffles),
                                            int(seed) & 0xFFFFFFFFFFFFFFFF, stat.ctypes.data_as(C.c_void_p), C.byref(st))
        if rc != 0:
            self._raise(rc)
        out = shuffle_fields(stat, n_shuffles)
        return (out, st.as_dict()) if with_stats else out

    def shuffle_sequences(self, seqs, replicate, seed=0, mode="di"):
        """mirfold_shuffle_sequences(): shuffle number `replicate` of every sequence exactly as shuffle_test folds it
        (upper-case, T -> U), generated by the device kernel.  Returns a list of str."""
        buf, off = self.pack(seqs)
        out = np.zeros(max(len(buf), 1), np.uint8)
        rc = self._lib.mirfold_shuffle_sequences(self._ctx, buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                 len(off) - 1, self._shuffle_mode(mode), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                 int(replicate), out.ctypes.data_as(C.c_void_p))
        if rc != 0:
            self._raise(rc)
        raw = out.tobytes()
        return [raw[int(off[r]):int(off[r + 1])].decode("latin-1") for r in range(len(off) - 1)]

    def int_peak2(self):
        """(add+min, DPX s32, VIADDMNMX.S16x2) min-plus terms/s on this context's device."""
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        rc = self._lib.mirfold_int_peak2(self._ctx, C.byref(a), C.byref(b), C.byref(c))
        if rc != 0:
            self._raise(rc)
        return a.value, b.value, c.value

    def int_peak(self):
        """Measured integer-issue roofline: (add+min terms/s, DPX terms/s) on this context's device."""
        a, b = C.c_double(), C.c_double()
        rc = self._lib.mirfold_int_peak(self._ctx, C.byref(a), C.byref(b))
        if rc != 0:
            self._raise(rc)
        return a.value, b.value

    def debug_matrices(self, seq, span, flags=0):
        """(c, fML, f3) of one sequence in the oracle's [i][d] layout (tests only)."""
        b = seq.encode() if isinstance(seq, str) else seq
        n = len(b)
        W = min(span, n) + 6
        c = np.empty((n + 2, W), np.int32)
        m = np.empty((n + 2, W), np.int32)
        f3 = np.empty(n + 4, np.int32)
        rc = self._lib.mirfold_debug_matrices(self._ctx, b, n, int(span), int(flags), c.ctypes.data_as(C.c_void_p),
                                              m.ctypes.data_as(C.c_void_p), f3.ctypes.data_as(C.c_void_p))
        if rc != 0:
            self._raise(rc)
        return c, m, f3

    # ---- stage 3: duplex checks on the device --------------------------------------------------
    def duplex(self, queries):
        """get_maturestar_info() for many (structure, mature) pairs at once (miR_PREFeR.py:1876-1999).
        queries: iterable of (ss, (m0, m1), foldstart, regionstart, regionend, strand) -- the reference's
        argument order minus the redundant foldend.  Returns, per query, exactly what the reference
        returns: the 9-tuple (star_start, star_end, fold_start, fold_end, star_ss, prime5, mature_ss,
        total_dots, total_bps) in genome coordinates, or the FAIL_* string; DUPLEX_EXCEPTION marks a pair on
        which the reference's function raises (unbalanced brackets inside the mature or its partner region)."""
        queries = list(queries)
        nq = len(queries)
        if nq == 0:
            return []
        # columns are built with numpy (a ctypes field store per value costs more than the kernel)
        offs, parts, pos = {}, [], 0
        ss_off = np.empty(nq, np.uint64)
        for k, q in enumerate(queries):
            ss = q[0]
            o = offs.get(ss)
            if o is None:
                o = offs[ss] = pos
                parts.append(ss)
                pos += len(ss) + 1
            ss_off[k] = o
        qarr = np.zeros(nq, DUPLEX_QUERY_DTYPE)
        qarr["ss_off"] = ss_off
        qarr["ss_len"] = [len(q[0]) for q in queries]
        qarr["fold_start"] = [q[2] for q in queries]
        qarr["mature_start"] = [q[1][0] for q in queries]
        qarr["mature_end"] = [q[1][1] for q in queries]
        qarr["region_start"] = [q[3] for q in queries]
        qarr["region_end"] = [q[4] for q in queries]
        qarr["strand"] = [ord(q[5]) for q in queries]
        arena = ("\0".join(parts) + "\0").encode("ascii")
        out = np.zeros(nq, DUPLEX_VERDICT_DTYPE)
        rc = self._lib.mirfold_duplex(self._ctx, arena, len(arena), qarr.ctypes.data_as(C.POINTER(_lib.DuplexQuery)), nq,
                                      out.ctypes.data_as(C.POINTER(_lib.DuplexVerdict)))
        if rc != 0:
            self._raise(rc)
        cols = {name: out[name].tolist() for name in DUPLEX_VERDICT_DTYPE.names}
        code = cols["code"]
        names = {}
        res = []
        for k, q in enumerate(queries):
            c = code[k]
            if c != 0:
                name = names.get(c)
                if name is None:
                    name = names[c] = self._lib.mirfold_duplex_fail_name(c).decode()
                res.append(name)   # code 100 = DUPLEX_EXCEPTION: the reference raises for this pair (see DuplexTable)
            else:
                ss = q[0]
                res.append((cols["star_start"][k], cols["star_end"][k], cols["fold_start"][k], cols["fold_end"][k],
                            ss[cols["star_ss_begin"][k]:cols["star_ss_end"][k]], bool(cols["prime5"][k]),
                            ss[cols["mature_ss_begin"][k]:cols["mature_ss_end"][k]], cols["total_dots"][k], cols["total_bps"][k]))
        return res

    # ---- RNALfold CLI contract -------------------------------------------------------------
    def fold_text_bytes(self, text, span, encoding=None):
        """RNALfold-identical stdout (bytes) for RNALfold-style stdin text (`RNALfold -L span`), in one native call
        (mirfold_fold_text: parse, fold, format).  `text` may be bytes; a str is encoded with `encoding` (default utf-8
        with surrogateescape, so header bytes that were decoded that way come back unchanged)."""
        if isinstance(text, str):
            text = text.encode(encoding) if encoding else text.encode("utf-8", "surrogateescape")
        out, n = C.c_void_p(), C.c_uint64()
        rc = self._lib.mirfold_fold_text(self._ctx, text, len(text), int(span), 0, C.byref(out), C.byref(n))
        if rc != 0:
            self._raise(rc)
        try:
            return C.string_at(out, n.value)
        finally:
            self._lib.mirfold_free_text(out, None)

    def fold_text_bytes_py(self, text, span, encoding=None):
        """The same through the Python parser and mirfold_format_records (kept as the readable statement of the I/O contract
        and as a cross-check of the native path)."""
        items = parse_rnalfold_input(text)
        seqs = [tok for kind, tok in items if kind == "seq"]
        out = []
        with self.fold(seqs, span) as res:
            data, offs = res.record_blocks()
            view = memoryview(data)
            r = 0
            for kind, tok in items:
                if kind == "echo":
                    out.append((tok.encode(encoding) if encoding else tok.encode("utf-8", "surrogateescape")) + b"\n")
                else:
                    out.append(view[int(offs[r]):int(offs[r + 1])])
                    r += 1
        return b"".join(out)

    def fold_text(self, text, span):
        """RNALfold-identical stdout for RNALfold-style stdin text (`RNALfold -L span`)."""
        return self.fold_text_bytes(text, span).decode("utf-8", "surrogateescape")

    def fold_fasta_files(self, fastas, outnames, span, batch_lines=200000):
        """fold_use_RNALfold() replacement (miR_PREFeR.py:3047-3119): fold every FASTA shard and write the
        RNALfold-format output files.  Like the reference's fold(), a shard is processed `batch_lines` input
        lines at a time (its 2*CHECKPOINT_SIZE, :3085-3098) and appended to `<outname>.tmp`, which is renamed
        when the shard is complete (:3098) -- a failing shard leaves no output file and no .tmp behind.
        Shards are read as bytes: header lines are echoed byte for byte, '\r' is not a line end."""
        for fa, outname in zip(fastas, outnames):
            tmp = outname + ".tmp"
            try:
                with open(fa, "rb") as fin, open(tmp, "wb") as fout:
                    while True:
                        lines = []
                        for line in fin:
                            lines.append(line)
                            if len(lines) >= batch_lines:
                                break
                        if not lines:
                            break
                        stop = any(ln.rstrip(b"\n") == b"@" for ln in lines)     # RNALfold stops reading at '@'
                        fout.write(self.fold_text_bytes(b"".join(lines), span))
                        if stop:
                            break
                os.rename(tmp, outname)   # atomic, like MP:3098
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        return list(outnames)
