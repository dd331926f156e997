/*
 * mirfold.h -- C ABI of libmirfold.so, the B200-native fold stage for miR-PREFeR.
 *
 * The reference has no FFI for this path; its boundary is a subprocess + text parser:
 *   caller   : subprocess.check_call("RNALfold -L <PRECURSOR_LEN>", stdin=<FASTA chunk>,
 *              stdout=<file>)                      /root/reference/miR_PREFeR.py:3053, :3064
 *   consumer : get_structures_next_extendregion()  /root/reference/miR_PREFeR.py:1541-1599
 *   duplex   : get_maturestar_info()               /root/reference/miR_PREFeR.py:1876-1999
 * Each entry point below names the reference interface it replaces.  Plain C types only
 * (pointers + sizes); no torch / C++ types cross this boundary.  Every function returns
 * MIRFOLD_OK (0) or a negative error code and never aborts the process.  The library has NO
 * CPU fallback: without a CUDA device mirfold_open() fails with MIRFOLD_ERR_NO_DEVICE.
 *
 * Ownership: inputs are borrowed for the duration of the call; results are owned by the
 * library until mirfold_free_result().  A context is single-caller (one host thread).
 * Results are deterministic and independent of device count and batch composition.
 * Lifetime: a result may outlive its context -- mirfold_close() with results still alive releases the
 * devices at once and the context's host bookkeeping when the last result is freed.
 */
#ifndef MIRFOLD_H
#define MIRFOLD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIRFOLD_OK 0
#define MIRFOLD_ERR_NO_DEVICE (-1)   /* no usable CUDA device / bad device id          */
#define MIRFOLD_ERR_CUDA (-2)        /* CUDA runtime error (see mirfold_last_error)     */
#define MIRFOLD_ERR_ARG (-3)         /* invalid argument                               */
#define MIRFOLD_ERR_PARAMSET (-4)    /* unknown energy parameter set                   */
#define MIRFOLD_ERR_BACKTRACK (-5)   /* traceback found no decomposition (the reference
                                        aborts with "backtrack failed ...")            */
#define MIRFOLD_ERR_NOMEM (-6)
#define MIRFOLD_ERR_CALLBACK (-7)    /* a mirfold_chunk_fn returned non-zero             */

/* The only parameter set with a runnable oracle: Turner 1999 as compiled into ViennaRNA
 * 1.8.5, dangles=1, 37 C, tetraloop bonus on (what `RNALfold -L n` uses by default). */
#define MIRFOLD_PARAMSET_DEFAULT "vienna-1.8.5-d1"

/* mirfold_fold flags.  The band fill normally runs a kernel that keeps its interior-loop window as
 * 16-bit values and transparently redoes any locus whose energies leave that range (below
 * -320 kcal/mol inside one window) with the 32-bit kernel; MIRFOLD_FLAG_WIDE forces the 32-bit kernel
 * for every locus.  Results are identical either way. */
#define MIRFOLD_FLAG_WIDE 1u
/* MIRFOLD_FLAG_SERIAL: run the chunks of a device one after the other on a single lane (no overlap of one chunk's
 * traceback / download with the next chunk's band fill).  Measurement aid: per-stage device times of
 * mirfold_stats are only disjoint in this mode.  Results are identical. */
#define MIRFOLD_FLAG_SERIAL 2u

typedef struct mirfold_ctx mirfold_ctx;

/* One printed RNALfold hairpin line: "<ss> (<mfe/100>) <start>".  Replaces one line of the
 * text that get_structures_next_extendregion() parses (miR_PREFeR.py:1566-1573). */
typedef struct mirfold_hit {
    int32_t start;     /* 1-based start printed by RNALfold                       */
    int32_t len;       /* strlen of the dot-bracket string                        */
    int32_t mfe_dcal;  /* energy in 0.01 kcal/mol (the printed %6.2f times 100)   */
    int32_t reserved;
    uint64_t ss_off;   /* offset of the NUL-terminated dot-bracket in ss_arena    */
} mirfold_hit;

typedef struct mirfold_stats {
    double ms_total;      /* host wall time of the call                                  */
    double ms_h2d;        /* device time: uploads                                        */
    double ms_fill;       /* device time of the c/fML band fill kernel(s) (CUDA events)  */
    double ms_f3;         /* f3 scan kernel                                              */
    double ms_trace;      /* emission plan + traceback + emission/pack kernels           */
    double ms_d2h;        /* result download                                             */
    double ms_device;     /* first kernel start -> last kernel end                       */
    uint64_t nt;          /* nucleotides folded                                          */
    uint64_t cells;       /* DP cells (i,j) visited, SURVEY.md 8(d) definition           */
    uint64_t tracebacks;  /* traceback calls                                             */
    uint64_t kernel_launches;
    uint64_t h2d_bytes, d2h_bytes;
    int32_t n_devices;
    int32_t n_chunks;
    uint64_t fill_units;  /* CTAs of the band fill: one per locus, one per tile of a longer locus (mirfold_plan_fill_units) */
} mirfold_stats;

/* Result of folding `nseq` records.  Hit order inside a record == RNALfold print order. */
typedef struct mirfold_result {
    uint32_t nseq;
    uint32_t reserved;
    uint64_t nhits;
    const uint64_t *hit_begin;   /* nseq entries: hits of record r are hits[hit_begin[r] .. hit_begin[r]+hit_count[r]) */
    const uint32_t *hit_count;   /* nseq entries.  Runs of different records are disjoint but NOT ordered by r: the
                                    table is left in the order the devices produced it (no per-hit host pass)    */
    const mirfold_hit *hits;     /* nhits entries                                                      */
    const char *ss_arena;        /* dot-bracket strings, NUL-terminated                                */
    uint64_t ss_bytes;
    const int32_t *total_mfe_dcal; /* nseq entries: the " (%6.2f)" total line of each record          */
    mirfold_stats stats;
} mirfold_result;

/* Replaces: locating/validating the RNALfold executable (check_RNALfold, miR_PREFeR.py:472-498).
 * device_ids == NULL or n_devices == 0 -> use the current CUDA device only. */
int mirfold_open(mirfold_ctx **ctx, const int *device_ids, int n_devices, const char *param_set);
void mirfold_close(mirfold_ctx *ctx);

/* Replaces: one `RNALfold -L span_L` subprocess run over a FASTA chunk (miR_PREFeR.py:3064)
 * plus the text parse of its hairpin lines (miR_PREFeR.py:1566-1573).
 *   seqs    : concatenated raw sequence tokens exactly as they appear on the FASTA sequence
 *             line (any case, DNA or RNA alphabet, IUPAC allowed; conversion to upper-case
 *             and T->U happens inside, like RNALfold's main()).
 *   seq_off : nseq+1 offsets into seqs.
 * With n_devices > 1 the records are sharded by DP work across the devices (no collectives)
 * and gathered back in input order. */
/* span_L is 5..4096 for every fold entry point.  A record may have up to 2^30 - 1 nt, whatever the device's memory: a
 * tiled record larger than the device budget is folded in segments (mirfold_plan_segments), with the same result.  At span_L > 800 a record longer
 * than 864 nt is filled as one unit (mirfold_plan_fill_units: kernel 0), which must hold fewer than 2^31 band cells,
 * (min(span_L, n-1) - 3) * stride < 2^31: records up to 2 691 072 nt at span_L = 801, 524 672 nt at 4096.  A batch
 * with a longer record is rejected as a whole with MIRFOLD_ERR_ARG before anything is allocated. */
int mirfold_fold(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq,
                 int span_L, uint32_t flags, mirfold_result **out);

/* Device-resident variant used for kernel-only timing: the same pipeline, but the raw
 * sequences/offsets already live in device memory of device 0 of the context and the
 * results stay in HBM (nothing is downloaded; *out carries only stats, nhits and nseq).
 * `stream` is a cudaStream_t passed as void* (NULL = the context's own stream). */
int mirfold_fold_device(mirfold_ctx *ctx, const void *d_seqs, const void *d_seq_off,
                        const uint64_t *h_seq_off, uint32_t nseq, int span_L, uint32_t flags,
                        void *stream, mirfold_result **out);

/* Debug/test hook: fill + f3 for ONE sequence and copy the band matrices back in the oracle's
 * [i][d] layout (row stride W = min(L,n)+6, rows 0..n+1, INF=1000000 where not computed).
 * c/m must hold (n+2)*W ints, f3 must hold n+4 ints. */
int mirfold_debug_matrices(mirfold_ctx *ctx, const char *seq, uint32_t n, int span_L, uint32_t flags,
                           int32_t *c, int32_t *m, int32_t *f3);

void mirfold_free_result(mirfold_result *res);

/* Replaces: the chunk loop of fold_use_RNALfold()/gen_next_chunk (miR_PREFeR.py:3022-3044, :3085-3098), which
 * folds a shard 2*CHECKPOINT_SIZE lines at a time and appends each chunk's text to the output file so that the
 * whole result never sits in memory.  Same fold as mirfold_fold(), but the results are handed to `fn` chunk by
 * chunk while later chunks are still computing; a chunk's buffers are only valid during the call.  Chunks are
 * delivered in the order the devices finish them (NOT input order; `record[k]` names the input record), one
 * callback at a time; every input record appears in exactly one chunk (records shorter than 5 nt, which have
 * no hits and a total of 0, arrive in a final chunk without hits).  A non-zero return value of `fn` aborts
 * the fold with MIRFOLD_ERR_CALLBACK.  ss_off of a chunk's hits is relative to the chunk's own ss_arena. */
typedef struct mirfold_chunk {
    uint32_t n_records;
    int32_t device;                /* CUDA ordinal that produced the chunk (-1 for the final hit-less chunk) */
    const uint32_t *record;        /* n_records input record indices                                         */
    const uint64_t *hit_begin;     /* n_records: hits of entry k are hits[hit_begin[k] .. +hit_count[k])      */
    const uint32_t *hit_count;
    const int32_t *total_mfe_dcal; /* n_records                                                              */
    uint64_t nhits;
    const mirfold_hit *hits;
    const char *ss_arena;
    uint64_t ss_bytes;
} mirfold_chunk;
typedef int (*mirfold_chunk_fn)(void *user, const mirfold_chunk *chunk);
int mirfold_fold_stream(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L,
                        uint32_t flags, mirfold_chunk_fn fn, void *user, mirfold_stats *stats /* may be NULL */);

/* Device-resident batches: the records are sharded over the context's devices (as mirfold_fold does) and their
 * raw sequences uploaded once; mirfold_batch_fold() then runs the whole pipeline on every device from HBM.
 * download = 0 leaves the results in HBM (*out carries stats, nhits and ss_bytes only) -- the kernel-only
 * measurement of bench.py on any number of devices; download = 1 returns the same result as mirfold_fold(). */
typedef struct mirfold_batch mirfold_batch;
int mirfold_batch_upload(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L,
                         mirfold_batch **out);
int mirfold_batch_fold(mirfold_ctx *ctx, mirfold_batch *batch, uint32_t flags, int download, mirfold_result **out);
void mirfold_batch_free(mirfold_batch *batch);

/* Genome-resident input.  Replaces what dump_piece does per record before the fold (miR_PREFeR.py:1097-1108, :1131, :1177):
 * ask `samtools faidx` for the bases of the extend region and reverse-complement minus-strand records.  The genome is
 * uploaded once; records are then given as coordinates and cut, oriented and encoded on the device.
 *   mirfold_genome_upload: contig c is seq[contig_off[c] .. contig_off[c+1]) (n_contigs+1 offsets, letters exactly as in
 *     the FASTA); one copy is kept on every device of ctx, and its bytes are taken off the lanes' memory budget while it
 *     lives (unless MIRFOLD_MEM_BUDGET_MB sets the budget).  mirfold_genome_free may be called before or after
 *     mirfold_close (the context's host bookkeeping lives until its last result and genome are freed).
 *   mirfold_genome_region: [start, end) is the extend region exactly as dump_piece prints it, strand '+' or '-', contig
 *     an index into the upload (-1: a seqid that is not in the FASTA, an empty record).  The folded bases are samtools
 *     0.1.18's `faidx seqid:start-(end-1)`: start clipped to >= 1, end-1 clipped to the contig length, empty if start >
 *     end-1.  A minus-strand record is reversed and complemented with the reference's get_complement table
 *     (miR_PREFeR.py:232-239): upper-case A T G C U only, so lower-case and IUPAC letters are reversed but not complemented.
 * mirfold_fold_regions / _stream / mirfold_fold_candidates_regions return byte for byte what mirfold_fold /
 * mirfold_fold_stream / mirfold_fold_candidates return on the host-extracted sequences; the duplex checks of the
 * candidates see the unclipped (start, end).  Only descriptors are uploaded per call (stats.h2d_bytes).  Each returns
 * MIRFOLD_ERR_ARG, and no result, for a contig index outside [-1, n_contigs), a strand other than '+' / '-', a genome of
 * another context or a closed context. */
typedef struct mirfold_genome mirfold_genome;
typedef struct mirfold_genome_region {
    int32_t contig;
    int32_t start, end;   /* [start, end), 1-based genome coordinates */
    int32_t strand;       /* '+' or '-' */
} mirfold_genome_region;
int mirfold_genome_upload(mirfold_ctx *ctx, const char *seq, const uint64_t *contig_off, uint32_t n_contigs,
                          mirfold_genome **out);
void mirfold_genome_free(mirfold_genome *genome);
int mirfold_fold_regions(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions, uint32_t nseq,
                         int span_L, uint32_t flags, mirfold_result **out);
int mirfold_fold_regions_stream(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions,
                                uint32_t nseq, int span_L, uint32_t flags, mirfold_chunk_fn fn, void *user,
                                mirfold_stats *stats /* may be NULL */);

/* Replaces: the split of the candidate FASTA into NUM_OF_CORE shards by locus count (miR_PREFeR.py:1329-1354)
 * that decides which RNALfold process folds which record (miR_PREFeR.py:3113-3118).  Here: greedy
 * longest-processing-time assignment by DP cells (SURVEY.md 8e), exactly the plan mirfold_fold() uses for a
 * context of n_shards devices.  Host-only (needs no device and no context).  shard_of[r] = shard of record r;
 * shard_cells[g] = DP cells assigned to shard g (either output may be NULL). */
int mirfold_plan_shards(const uint64_t *seq_off, uint32_t nseq, int span_L, int n_shards, uint32_t *shard_of,
                        uint64_t *shard_cells);

/* How the band fill cuts one locus of n bases at span span_L into fill units (one CTA each).  The reference has no
 * counterpart (RNALfold walks a locus row by row, Lfold.c:189-346); exported so that callers and tests can reason about
 * memory and work per locus.  Host-only.  A locus longer than the largest shared-memory bucket is filled as n_units
 * overlapping tiles of tile_len bases: tile t covers bases a_t+1 .. a_t+tile_len, a_t = min(t*tile_step, n-tile_len),
 * and owns rows a_t+1 .. a_t+tile_step (the last tile: all its remaining rows); every cell (i, j <= i+span) of an owned
 * row lies inside the tile.  kernel: 0 = generic global-memory kernel, else the shared-memory bucket's stride
 * (160 / 352 / 608 / 864).  band_cells = cells the band arrays hold (stride * diagonals * n_units).  MIRFOLD_ERR_ARG for an
 * untiled unit of 2^31 band cells or more, which the fold entry points reject (see mirfold_fold). */
typedef struct mirfold_fill_plan {
    int32_t kernel;
    int32_t stride;
    int32_t tile_len;    /* n when the locus is one unit */
    int32_t tile_step;   /* rows owned per tile; n when the locus is one unit */
    int32_t n_units;
    int32_t dmax;        /* widest diagonal of the band: min(span_L, n) capped at n-1 */
    uint64_t band_cells;
} mirfold_fill_plan;
int mirfold_plan_fill_units(uint32_t n, int span_L, mirfold_fill_plan *out);

/* How the fold runs one locus of n bases at span span_L when its device entry may use budget_bytes for it.  A tiled locus
 * (mirfold_plan_fill_units: n_units > 1) that needs more than the budget is folded in segments from its 3' end, so a
 * record's length is not bounded by device memory: a segment owns the tiles tile_first .. tile_last (rows row_first ..
 * row_last) and also fills the halo_tiles tiles above them, which own the rows up to row_last + min(span_L, n) + 1 that
 * its f3 and tracebacks read.  The sequence-sized arrays (about 16 bytes per nt) stay whole; device_bytes is what the
 * segment needs with them.  Segments take as many owned tiles as fit the budget, at least one.  A locus that fits, or is
 * one unit, is one segment.  The engine uses this plan with budget_bytes = a lane's share of the device entry's budget
 * (MIRFOLD_MEM_BUDGET_MB, or a share of free memory at mirfold_open) for every locus larger than the whole budget.
 * Host-only.  *n_segments = the number of segments; the first min(cap, *n_segments) are written to segs, in the order
 * they run.  MIRFOLD_ERR_ARG as mirfold_plan_fill_units, and for n >= 2^30. */
typedef struct mirfold_segment {
    int32_t tile_first, tile_last;   /* owned tiles */
    int32_t halo_tiles;              /* tiles tile_last+1 .. tile_last+halo_tiles, filled but not owned */
    int32_t row_first, row_last;     /* owned rows (1-based) */
    int32_t reserved;
    uint64_t device_bytes;
} mirfold_segment;
int mirfold_plan_segments(uint32_t n, int span_L, uint64_t budget_bytes, mirfold_segment *segs, uint32_t cap,
                          uint32_t *n_segments);

/* Replaces: what RNALfold's main() prints per record (RLF .rodata "%s (%6.2f) %4d\n" / "%s\n (%6.2f)\n",
 * SURVEY A.6) -- the text miR_PREFeR.py collects at :3085-3098 and parses at :1541-1599.  For every record r
 * of `res` (the result of mirfold_fold over the same seqs/seq_off) the block
 *     <ss> (<mfe>) <start>\n   per hit, in RNALfold's print order
 *     <sequence token upper-cased, T->U>\n (<total mfe>)\n
 * is written to one buffer; (*rec_off)[r] .. (*rec_off)[r+1] delimit record r's block (header echo lines are
 * the caller's).  Host-only, multi-threaded; both buffers are owned by the library until mirfold_free_text(). */
int mirfold_format_records(const mirfold_result *res, const char *seqs, const uint64_t *seq_off, uint32_t nseq,
                           char **text, uint64_t **rec_off);
void mirfold_free_text(char *text, uint64_t *rec_off);

/* Replaces: one whole `RNALfold -L span_L < text > out` run (miR_PREFeR.py:3053, :3064) -- RNALfold's main() in one call:
 * lines starting with '>' or '*' and empty lines are echoed, a line "@" ends the input, the first whitespace-delimited
 * token of any other line is folded and its record block printed (SURVEY A.6).  *out holds *out_len bytes, byte-identical
 * to RNALfold's stdout; release with mirfold_free_text(*out, NULL). */
int mirfold_fold_text(mirfold_ctx *ctx, const char *text, uint64_t len, int span_L, uint32_t flags, char **out,
                      uint64_t *out_len);

/* Replaces: the structure classification of get_structures_next_extendregion (miR_PREFeR.py:1566-1589) with
 * is_stem_loop (:1602), filter_ss (:1685) and has_one_good_bifurcation (:1611): for every hit of at least
 * `minlen` characters the candidate structures the predict stage consumes -- the whole hairpin (sstype 0) or
 * its outermost-stem pieces longer than 55 that are stem-loops (0) or have one good bifurcation (1).
 * Structures of record r are out[rec_begin[r] .. rec_begin[r+1]) in the reference's order.  The dot-bracket
 * string of a structure is ss_arena[ss_off .. ss_off+len) of `res` (NOT NUL-terminated for pieces).
 * norm_energy = printed energy / length of the whole hit, as in the reference.  Host-only, multi-threaded.
 * Returns MIRFOLD_ERR_ARG for input on which the reference's functions raise (a hit without any pair). */
typedef struct mirfold_structure {
    uint32_t rec;
    int32_t fold_start;   /* 1-based start of the structure in the record's sequence */
    int32_t sstype;       /* 0 stem-loop, 1 one good bifurcation */
    int32_t len;
    uint64_t ss_off;
    double norm_energy;
} mirfold_structure;
int mirfold_classify(const mirfold_result *res, int minlen, int minloop, mirfold_structure **out, uint64_t *n_out,
                     uint64_t **rec_begin);
void mirfold_free_structures(mirfold_structure *s, uint64_t *rec_begin);

/* Measurement aid (bench.py roofline denominator): sustained rate of independent min-plus terms
 * (one add + one min each) on device 0 of the context, terms per second, for plain add+min code and
 * for the DPX intrinsic __viaddmin_s32. */
int mirfold_int_peak(mirfold_ctx *ctx, double *addmin_terms_per_s, double *dpx_terms_per_s);
/* The same plus the packed 16-bit form the narrow fill kernel issues (VIADDMNMX.S16x2: two terms per instruction). */
int mirfold_int_peak2(mirfold_ctx *ctx, double *addmin_terms_per_s, double *dpx_terms_per_s, double *s16x2_terms_per_s);

const char *mirfold_strerror(int code);
/* Human-readable detail of the last error raised in this context (CUDA error string etc). */
const char *mirfold_last_error(const mirfold_ctx *ctx);
/* "mirfold <version> sm_100a <paramset>" */
const char *mirfold_version(void);

/* ---- stage 3: miRNA/miRNA* duplex checks fused on-device (miR_PREFeR.py:1876-1999) ---- */

/* One (structure, mature) query.  Coordinates follow get_maturestar_info()'s arguments. */
typedef struct mirfold_duplex_query {
    uint64_t ss_off;       /* dot-bracket string in the arena given to mirfold_duplex()   */
    int32_t ss_len;
    int32_t fold_start;    /* 1-based offset of ss[0] in the folded sequence ("foldstart") */
    int32_t mature_start;  /* genome coords [m0, m1) of the mature candidate               */
    int32_t mature_end;
    int32_t region_start;  /* extended region [rs, re)                                     */
    int32_t region_end;
    int32_t strand;        /* '+' or '-'                                                   */
    int32_t reserved;
} mirfold_duplex_query;

/* Verdict codes: 0 = pass; otherwise index into mirfold_duplex_fail_name(). */
typedef struct mirfold_duplex_verdict {
    int32_t code;
    int32_t star_start, star_end;   /* genome coords of the star                      */
    int32_t fold_start, fold_end;   /* genome coords of the folded region             */
    int32_t star_ss_begin, star_ss_end;     /* local slice [b,e) of ss = star_ss      */
    int32_t mature_ss_begin, mature_ss_end; /* local slice of ss = mature_ss          */
    int32_t prime5;                 /* 1 if the mature is on the 5' arm               */
    int32_t total_dots, total_bps;
} mirfold_duplex_verdict;

int mirfold_duplex(mirfold_ctx *ctx, const char *ss_arena, uint64_t ss_bytes,
                   const mirfold_duplex_query *queries, uint64_t nq,
                   mirfold_duplex_verdict *verdicts /* nq entries, caller-allocated */);
const char *mirfold_duplex_fail_name(int code);

/* ---- stages 1 + 3 fused on the device after traceback ----
 * Replaces, in one call: the fold (miR_PREFeR.py:3064), the candidate-structure pass of
 * get_structures_next_extendregion (:1566-1589) and get_maturestar_info (:1876-1999) for every (candidate structure x
 * size-admissible mature) pair of every record -- the superset of pairs check_loci (:2246-2262) can ask for.  The hit
 * text never leaves the device: only the candidate structures, their dot-bracket strings and the verdicts are
 * downloaded.  Records are what dump_piece writes (:1124-1143): the region [start, end) and the "M:s-e/strand/depth"
 * matures of the header line.
 *   regions[r]                      region of record r (genome coordinates)
 *   matures[mature_off[r] .. mature_off[r+1])   its matures, in header order
 * Output (owned by the library until mirfold_free_candidates):
 *   structures of record r: structs[struct_begin[r] .. +struct_count[r]) in the reference's order; ss_off indexes ss_arena
 *   (NUL-terminated strings); verdicts of structure s: verdicts[verdict_begin[s] .. +verdict_count[s]), one per mature
 *   with min_mature_len <= end-start <= max_mature_len in header order; verdict_mature[v] = index of that mature inside
 *   the record's mature list.  Returns MIRFOLD_ERR_ARG for input on which the reference's classifier raises. */
typedef struct mirfold_mature {
    int32_t start, end;   /* genome coordinates [start, end)                         */
    int32_t strand;       /* '+' or '-' (the strand get_maturestar_info is called with) */
    int32_t depth;        /* carried through for the caller                          */
} mirfold_mature;
typedef struct mirfold_region {
    int32_t start, end;   /* extended region [start, end) of the record              */
} mirfold_region;
typedef struct mirfold_candidates {
    uint32_t nseq;
    uint32_t reserved;
    uint64_t nstructs;
    const uint64_t *struct_begin;       /* nseq */
    const uint32_t *struct_count;       /* nseq */
    const mirfold_structure *structs;
    const char *ss_arena;
    uint64_t ss_bytes;
    uint64_t nverdicts;
    const uint64_t *verdict_begin;      /* nstructs */
    const uint32_t *verdict_count;      /* nstructs */
    const mirfold_duplex_verdict *verdicts;
    const uint32_t *verdict_mature;     /* nverdicts */
    uint64_t nhits;                     /* hairpins folded (not downloaded) */
    mirfold_stats stats;
} mirfold_candidates;
int mirfold_fold_candidates(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L,
                            uint32_t flags, const mirfold_region *regions, const mirfold_mature *matures,
                            const uint64_t *mature_off, int minlen, int minloop, int min_mature_len, int max_mature_len,
                            mirfold_candidates **out);
/* The same with the records given as regions of a resident genome (mirfold_genome_upload above); regions[r] also stands
 * for the mirfold_region of record r, unclipped. */
int mirfold_fold_candidates_regions(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions,
                                    uint32_t nseq, int span_L, uint32_t flags, const mirfold_mature *matures,
                                    const uint64_t *mature_off, int minlen, int minloop, int min_mature_len,
                                    int max_mature_len, mirfold_candidates **out);
void mirfold_free_candidates(mirfold_candidates *c);

/* ---- MFE significance against shuffled sequences (randfold's test, Bonnet et al. 2004) ----
 * For every record: its total MFE (the " (%6.2f)" total line) and that of n_shuffles shuffles of it, folded on the
 * device.  Shuffles act on the sequence as it is folded (upper-case, T -> U) and treat every distinct byte as a symbol:
 *   MIRFOLD_SHUFFLE_MONO  Fisher-Yates: keeps the multiset of symbols;
 *   MIRFOLD_SHUFFLE_DI    Altschul-Erickson (uShuffle, k = 2): keeps every dinucleotide count and the first and last
 *                         symbols, uniform over the sequences that do; at most 16 distinct symbols per record.
 * Replicate k of record r is a pure function of (seed, r, k) (splitmix64, csrc/shuffle_rng.cuh), so results do not
 * depend on the devices, chunks or rounds.  span_L = 0 folds every record globally (at a span of at least its length,
 * so native_dcal == mirfold_fold's total at span_L = n; records must then be at most 4096 nt); otherwise 5..4096.
 * Records shorter than 5 nt have native 0, every shuffle 0 and n_le = n_shuffles.  The fold stops after the f3 scan
 * (no traceback) and downloads 4 bytes per folded sequence; stats count every folded nt and cell, natives included.
 * Derived: p = (n_le + 1) / (n_shuffles + 1), mean = sum / K, sd^2 = sumsq / K - mean^2, z = (native - mean) / sd.
 * MIRFOLD_ERR_ARG, and no output, for n_shuffles = 0, an unknown mode, a closed context, a span outside the range
 * above or a record with more than 16 symbols in dinucleotide mode. */
#define MIRFOLD_SHUFFLE_MONO 1
#define MIRFOLD_SHUFFLE_DI 2
typedef struct mirfold_shuffle_stat {
    int32_t native_dcal;   /* total MFE of the unshuffled record (== mirfold_fold's total at this span) */
    uint32_t n_le;         /* shuffles whose total MFE <= native_dcal                                  */
    int64_t sum_dcal;      /* sum of the shuffles' totals                                              */
    int64_t sumsq_dcal;    /* sum of their squares                                                     */
} mirfold_shuffle_stat;
int mirfold_shuffle_test(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L /* 0 = global */,
                         uint32_t flags, int mode, uint32_t n_shuffles, uint64_t seed,
                         mirfold_shuffle_stat *out /* nseq, caller-allocated */, mirfold_stats *stats /* may be NULL */);
/* Inspection / test hook: replicate `replicate` of every record as mirfold_shuffle_test folds it, generated by the device
 * kernel on device 0 of ctx.  Record r's shuffle is written to out[seq_off[r] .. seq_off[r+1]) (converted letters). */
int mirfold_shuffle_sequences(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int mode,
                              uint64_t seed, uint32_t replicate, char *out /* seq_off[nseq] bytes */);

#ifdef __cplusplus
}
#endif
#endif /* MIRFOLD_H */
