// mirfold_internal.cuh -- shared device/host declarations of libmirfold (not part of the C ABI).
//
// Data layout in HBM (see DESIGN.md):
//   codes : per locus n+3 bytes, index 0..n+2; byte = S | (S1 << 4); S[0]=S[n+1]=S[n+2]=0
//   F     : per locus n+3 int32 at the same offsets (f3[0..n+2], f3[k>n-4]=0)
//   C, M  : diagonal-major band per locus, rectangular: diagonal d (=j-i, 4..dmax) holds cells
//           i=1..n-d at band_off + (d-4)*stride + (i-1), stride = n rounded up to the locus'
//           length bucket (a compile-time constant of the fill kernel, so that per-diagonal
//           offsets become instruction immediates).  dmax = min(L*, n-1).  All threads walking
//           one anti-diagonal touch consecutive addresses.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define MF_INF 1000000
#define MF_TURN 3
#define MF_MAXLOOP 30
#define MF_GEN_ITERS 14 /* generic interior-loop terms per lane in the skewed smem ring schedule */
#define MF_SKEW_A 11    /* ring row rotation per diagonal: bank class of (u,v) = (u - 11*(u+v)) mod 32 */
#define MF_MAX_SPAN 4096 /* hairpin-size table length; PRECURSOR_LEN is capped at 3000 (MP:168) */

/* ---- 16-bit pair ring of the narrow fill kernel (k_fill_s16) ------------------------------------
 * Two adjacent diagonals share one 32-bit shared-memory word per row (lo = even diagonal), so one LDS
 * + one VIADDMNMX.S16x2 evaluates two interior-loop terms.  Values are exact as long as every c of the
 * locus stays above MF16_GUARD; a locus that violates it is flagged and redone by the 32-bit kernel. */
#define MF16_NPS 17        /* pair slots: 16 read + 1 written per diagonal                         */
#define MF16_NQG 8         /* generic word-terms per lane                                           */
#define MF16_NQB 2         /* bulge word-terms per lane                                             */
#define MF16_NQ (MF16_NQG + MF16_NQB)
#define MF16_NMG 2         /* leading generic iterations that carry a half-word mask                */
#define MF16_NMK (MF16_NMG + MF16_NQB)
#define MF16_SKEW 17       /* row rotation per pair slot: bank class of a word-term = (x - 17 m) mod 32 */
#define MF16_INF 31000
#define MF16_INF2 0x79187918u
#define MF16_VALID 20000   /* anything >= this after the min is "no loop"                           */
#define MF16_GUARD (-32000)
#define MF16_DBIAS 128
/* 16-bit fML pairs of the DML strips (k_fill_s16): finite fML in (MF16M_GUARD, ~1300] for spans <= MF16_MAX_SPAN */
#define MF16M_INF 16383
#define MF16M_INF2 0x3FFF3FFFu
#define MF16M_VALID 2700    /* a sum of two finite fML is below this; anything with an INF operand is above */
#define MF16M_GUARD (-13600)
#define MF16_MAX_SPAN 1000  /* hairpin extrapolation keeps fML < 1350 up to this span */
#define MF_DYNW_MIN_SPAN 400  /* spans from here on: fML of ordinary sequence can pass MF16M_GUARD (measured: min fML -13340 at L=400, -16179 at L=500) */

struct DevParams {
    int hairpinE[MF_MAX_SPAN + 2];  // by loop size, incl. the lxc*log extrapolation (A.2)
    int bulge[31], internal_loop[31];
    int stack[64];
    int mismatchI[200], mismatchH[200];
    int dangle5[40], dangle3[40];  // clamped <= 0
    int MLintern[8];
    int int11[8 * 8 * 25], int21[8 * 8 * 125], int22[8 * 8 * 625];
    int ilc[16][32];               // generic kernel: interior-loop constants per (iteration, lane); INF = masked
    int gen_c[MF_GEN_ITERS][32];   // smem kernel: constant of the term lane l evaluates in iteration k (INF = none)
    int gen_us[MF_GEN_ITERS][32];  //              its u | (u+v) << 8 | valid << 16
    // narrow kernel, per parity of d: word-term descriptors m | xoff << 4 | ring << 10 | null << 11,
    // packed 16-bit constants (lo | hi << 16) and half-word keep masks of the masked iterations
    unsigned int s16_td[2][MF16_NQ][32];
    unsigned int s16_cst[2][MF16_NQ][32];
    unsigned int s16_mk[2][MF16_NMK][32];
    int MLclosing, TerminalAU;
    short tetra[4096];             // tetraloop bonus by 2-bit packed 6-mer
    unsigned char pair[64];        // BP_pair[S_i*8+S_j]
    unsigned char rtype[8];
    unsigned char uv[496][2];      // traceback (p,q) candidate order: u ascending, v ascending
};

struct LocusDesc {
    unsigned long long seq_off;   // into codes / F (elements)
    unsigned long long band_off;  // into C / M (elements)
    unsigned long long ring_off;  // into ring scratch (elements)
    unsigned long long raw_off;   // into the raw ASCII buffer; | MF_RAW_REVERSE: fold the reverse complement
    int n;
    int Ls;      // L* = min(L, n)
    int dmax;    // min(Ls, n-1)
    int rec;     // input record index
    int stride;  // band row stride (elements per diagonal)
    // Long loci are filled as overlapping tiles of TL bases by the shared-memory kernels (TL = MF_TILE_LEN,
    // or MF_TILE_LEN_BIG for wide spans: shape_locus() in host.cu; a tiled locus has stride == TL): tile t covers
    // bases a_t+1 .. a_t+TL, a_t = min(t*tile_step, n-TL), tile_step = TL - dmax.  Every cell value only depends
    // on the bases inside [i,j], so a tile's cells are the locus' cells; row i is read from its owner tile
    // min((i-1)/tile_step, tile_last), which holds all of (i, i+4..i+dmax).  Untiled: tile_last = 0.
    int tile_last;           // number of tiles - 1
    int tile_step;           // rows owned per tile
    unsigned int tile_rcp;   // ceil(2^32 / tile_step): __umulhi(i-1, tile_rcp) is (i-1)/tile_step or one more (tile_of_row)
};
// raw_off flag of a minus-strand genome region (mirfold_fold_regions): k_prepare reads the locus backwards and complements it
#define MF_RAW_REVERSE (1ULL << 63)
#define MF_TILE_LEN 608
#define MF_TILE_LEN_BIG 864   /* the largest shared-memory bucket: one 1024-thread CTA per SM (155 KB of rings) */

// owner tile of row i (1 <= i < 2^30) of a tiled locus: min((i-1)/tile_step, tile_last).  With x = i-1, S = tile_step and
// e = tile_rcp*S - 2^32 < S, __umulhi(x, tile_rcp) = floor(x/S + x*e/(S*2^32)); for x < 2^30 the second term is below 1/4,
// so the estimate is x/S or, when x mod S is near S-1, x/S + 1, and one compare corrects it.  Without the correction rows
// go wrong from x = 7 615 399 on (S = 580, L = 28).  tests/test_long_loci.py::test_owner_tile_is_exact checks a mirror of this expression
// for every S in [MF_TILE_MIN_STEP, MF_TILE_LEN_BIG] at the worst x < 2^30 of every residue class.
__device__ __forceinline__ int tile_of_row(int i, unsigned int tile_rcp, int tile_step, int tile_last)
{
    const unsigned int x = (unsigned int)(i - 1);
    unsigned int t = __umulhi(x, tile_rcp);
    t -= (t * (unsigned int)tile_step > x) ? 1u : 0u;
    return min((int)t, tile_last);
}

// element offset (relative to the locus' band_off) of row i's owner-tile origin, i.e. of cell
// (i, i+4); cell (i, i+d) sits (d-4)*stride further.  Any cell (i', j') with i <= i' and
// j' <= i+dmax may also be addressed relative to row i's tile (columns are local to the tile).
__device__ __forceinline__ unsigned long long band_row_base(const LocusDesc &L, int i)
{
    if (L.tile_last == 0) return (unsigned long long)(i - 1);
    const int t = tile_of_row(i, L.tile_rcp, L.tile_step, L.tile_last);
    const int a = min(t * L.tile_step, L.n - L.stride);   // tiled: stride == tile length
    return (unsigned long long)t * ((unsigned long long)(L.dmax - 3) * L.stride) + (unsigned long long)(i - 1 - a);
}

// offset of diagonal d inside a locus' band (elements)
__host__ __device__ __forceinline__ unsigned int band_doff(int stride, int d) { return (unsigned int)(d - 4) * (unsigned int)stride; }
__host__ __device__ __forceinline__ unsigned long long band_elems(int stride, int dmax)
{
    return dmax >= 4 ? (unsigned long long)(dmax - 3) * (unsigned long long)stride : 0ULL;
}
// length buckets of the shared-memory fill kernels; a stride that is none of them marks a unit of the generic kernel
__host__ __device__ __forceinline__ bool is_bucket_stride(int stride)
{
    return stride == 160 || stride == 352 || stride == MF_TILE_LEN || stride == MF_TILE_LEN_BIG;
}
__host__ __device__ __forceinline__ int band_stride_for(int n, bool big)
{
    if (n <= 160) return 160;
    if (n <= 352) return 352;
    if (n <= MF_TILE_LEN) return MF_TILE_LEN;
    if (big && n <= MF_TILE_LEN_BIG) return MF_TILE_LEN_BIG;
    const int s = (n + 31) & ~31;
    return is_bucket_stride(s) ? s + 32 : s;   // generic kernel
}

#define MF_RING_CM 64  /* generic kernel: Cm window ring in global memory (needs >= 33 diagonals) */
#define MF_RING_DML 16 /* DML ring (needs >= 9 diagonals)                                         */
#define MF_RING_PER_STRIDE (MF_RING_CM + MF_RING_DML)
// generic kernel scratch of an n-nt unit: sS[npad] | sS1[npad] | pair table[64] | typed-cell list[n] (int), 16 B slack.
// In dynamic shared memory while the launch's longest unit fits MF_GENERIC_SMEM_MAX (about 34 100 nt), else in the
// unit's ring region after its Cm ring (unit_ring_elems in host.cu reserves it for every generic unit)
#define MF_GENERIC_SMEM_MAX (200 * 1024)
__host__ __device__ __forceinline__ unsigned long long generic_scratch_bytes(int n)
{
    return 2ULL * (unsigned long long)((n + 3 + 15) & ~15) + 64 + 4ULL * (unsigned long long)n + 16;
}
// An untiled unit addresses its band with 32-bit offsets (d-4)*stride + i-1 (k_fill_generic, the f3 kernels, the
// traceback): its band must hold fewer than 2^31 cells.  Tiled units (stride <= 864) are far below.
#define MF_MAX_UNIT_BAND_CELLS (1ULL << 31)

// ---- kernel launchers (each defined next to its kernels) -------------------------------
struct FillLaunch {
    const LocusDesc *loci;
    int nloci;
    int max_n;
    const unsigned char *codes;
    int *C, *M, *ring;
    unsigned char *Ib;    // one byte per band cell: "some two-loop candidate reproduces c(i,j)" (traceback hint; all ones from the wide kernels)
    unsigned int *Mp;     // narrow kernel: fML as 16-bit row pairs (locus at band_off; layout by bucket, see dev_store_fml16)
    const DevParams *P;
    int bucket_first[6];  // fill units sorted by (bucket, descending n): [generic | 864 | 608 | 352 | 160 | end)
    int *flags;           // per locus: 1 = the 16-bit kernel left its range, redo with the 32-bit kernel
    int force_wide;       // skip the 16-bit kernel (MIRFOLD_FLAG_WIDE)
    int opts;             // experiment switches (env MIRFOLD_OPTS): bit 0 = no L1 prefetch in the 32-bit DML strips, bit 1 = 32-bit DML strips in the narrow kernels;
                          // bit 3 (set by the host for spans >= MF_DYNW_MIN_SPAN): launch the 608/864 instantiations that switch to int32 strips on out-of-range fML
};
cudaError_t launch_prepare(const char *raw, const LocusDesc *loci, int nloci, unsigned long long total_codes,
                           unsigned char *codes, int *F, cudaStream_t st);
cudaError_t launch_fill(const FillLaunch &a, cudaStream_t st, cudaStream_t side = nullptr, cudaEvent_t fork = nullptr,
                        cudaEvent_t join = nullptr);   // side != nullptr: small buckets run concurrently on it
cudaError_t fill_configure_device();
cudaError_t launch_f3(const LocusDesc *loci, int nloci, int n_long, int max_Ls, const unsigned char *codes, const int *C, int *F,
                      const DevParams *P, cudaStream_t st);   // first n_long loci: n > MF_TILE_LEN

struct TraceBuffers {
    const LocusDesc *loci;
    int nloci;
    const unsigned char *codes;
    const int *C, *M, *F;
    const unsigned char *Ib;       // traceback hint bytes of the fill (FillLaunch::Ib)
    const DevParams *P;
    // plan
    int *tb_count;                 // nloci
    unsigned long long *tb_base;   // nloci+1 (exclusive scan of tb_count)
    unsigned long long *list_off;  // nloci : offset of the locus' start list in tb_start_list
    int *tb_start_list;            // per locus up to n/2+2 starts
    // per traceback
    unsigned long long ntb;
    int slot_stride;               // bytes per structure slot
    char *slots;                   // ntb * slot_stride
    int *tb_len;                   // ntb
    int *tb_start;                 // ntb
    int *tb_locus;                 // ntb
    int *tb_flag;                  // ntb : printed?
    int *tb_energy;                // ntb
    int *stack_scratch;            // ntb * stack_cap * 2 ints
    int stack_cap;
    int code_win;                  // bytes of shared memory per traceback warp for the window's codes
    int *fail_flag;                // 1 int
};
cudaError_t launch_plan(const TraceBuffers &b, cudaStream_t st);
// segmented loci (host.cu, fold_segmented): f3 of a row range, the resumable plan, emission across segment edges
cudaError_t launch_f3_rows(const LocusDesc *locus, int Ls, int row_hi, int row_lo, const unsigned char *codes, const int *C, int *F,
                           const DevParams *P, cudaStream_t st);
cudaError_t launch_plan_seg(const int *F, int row_hi, int row_lo, int bottom, int *state, int *list, unsigned long long *tb_base,
                            int *tb_count, cudaStream_t st);
cudaError_t launch_emit_seg(const TraceBuffers &b, int n_carry, int shift, int last, const int *F, int n, int *abs_start, cudaStream_t st);
cudaError_t launch_traceback(const TraceBuffers &b, cudaStream_t st);
cudaError_t launch_emit(const TraceBuffers &b, cudaStream_t st);
struct mirfold_hit;
cudaError_t launch_pack(const TraceBuffers &b, const unsigned long long *ss_off, const unsigned long long *hit_idx,
                        char *arena, mirfold_hit *out_hits, unsigned long long arena_base, cudaStream_t st);
// fused stage 1 + 3 over a chunk's packed hits (candidates.cu)
struct mirfold_structure;
struct mirfold_mature;
struct mirfold_region;
struct mirfold_duplex_verdict;
struct CandLaunch {
    // the chunk as k_pack left it
    const LocusDesc *loci;
    int nloci;
    const mirfold_hit *hits;               // ss_off includes arena_base
    unsigned long long nhits;
    const char *arena;
    unsigned long long arena_base;
    const unsigned long long *bounds;      // nloci+1: first hit of every locus
    // the call's records
    const mirfold_region *regions;         // by record
    const mirfold_mature *matures;
    const unsigned long long *mature_off;  // by record, nseq+1
    int minlen, minloop, min_mature, max_mature;
    // classification
    unsigned long long *counts;            // nhits+1 (scan input)
    const unsigned long long *soff;        // nhits+1 (exclusive scan of counts)
    mirfold_structure *structs;            // chunk-relative ss_off
    unsigned long long nstructs;
    unsigned long long *nq, *sbytes;       // per structure (+1): verdicts / string bytes (scan inputs)
    const unsigned long long *voff, *aoff; // their exclusive scans
    unsigned long long *locus_sbegin;      // nloci+1: first structure of every locus
    // outputs
    mirfold_duplex_verdict *verdicts;
    unsigned int *verdict_mature;
    char *out_arena;
    unsigned long long out_base;           // added to the compact-arena offsets
    mirfold_structure *structs_out;
    int *fail_flag;
};
cudaError_t launch_cand_classify(const CandLaunch &a, int pass, cudaStream_t st);
cudaError_t launch_cand_finish(const CandLaunch &a, int max_len, cudaStream_t st);
cudaError_t run_int_peak(cudaStream_t st, int sm_count, double *addmin, double *dpx, double *s16x2);
// shuffled replicates of the significance test (shuffle.cu): item t writes replicate `rep` of input record `rec` (n bytes,
// converted letters) to out + dst, using scr + dst as n bytes of scratch
#define MF_SHUFFLE_MONO 1   /* == MIRFOLD_SHUFFLE_MONO */
#define MF_SHUFFLE_DI 2     /* == MIRFOLD_SHUFFLE_DI   */
struct ShuffleItem {
    unsigned int rec, rep;
    unsigned long long dst;
};
cudaError_t launch_shuffle(const char *in, const unsigned long long *in_off, const ShuffleItem *items, unsigned int nitems,
                           char *out, unsigned char *scr, unsigned long long seed, int mode, int *fail, cudaStream_t st);
struct mirfold_duplex_query;
struct mirfold_duplex_verdict;
cudaError_t launch_duplex(const char *arena, const mirfold_duplex_query *qs, unsigned long long nq,
                          mirfold_duplex_verdict *out, int maxlen, cudaStream_t st);
