/*
 * lfold_oracle.c -- CPU restatement of the reference fold stage's arithmetic.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (mir_prefer_b200/) may import, link
 * or execute this file; it exists so that tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline leg have a debuggable checker (it can expose the c / fML / f3 matrices, which
 * the reference binary cannot).
 *
 * What it restates: `RNALfold -L <span>` of ViennaRNA 1.8.5 with default flags (-d1, 37 C,
 * tetraloop bonus on), which is what miR-PREFeR's fold stage shells out to
 * (/root/reference/miR_PREFeR.py:3053, :3064).  ViennaRNA's source is NOT part of the reference
 * checkout -- only the binary dependency/Linux/x64/RNALfold (ViennaRNA 1.8.5, unstripped,
 * DWARF) -- so this file follows the behavioural spec in SURVEY.md Appendix A, whose items cite
 * the binary's DWARF line numbers ("RLF Lfold.c:NNN").  Sections below name the spec item.
 *
 * Parity pin: oracle/check_oracle.py runs this against the reference binary itself (sha256
 * golden pins of SURVEY.md App. C + randomized corpora); tests/golden holds RLF outputs.
 *
 * Design differs from the reference on purpose (this is a restatement, not a copy): full
 * band matrices indexed [i][d] instead of L+5 rolling rows, explicit accessor functions that
 * return INF outside the computed band, a sector stack on the heap.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../mir_prefer_b200/csrc/turner99_v185_tables.inc"

#define INF 1000000
#define TURN 3
#define MAXLOOP 30

/* ------------------------------------------------------------------ parameters (App. A.3, a10) */
typedef struct {
    int stack[8][8], hairpin[31], bulge[31], internal_loop[31];
    int mismatchI[8][5][5], mismatchH[8][5][5], dangle5[8][5], dangle3[8][5];
    int int11[8][8][5][5], int21[8][8][5][5][5], int22[8][8][5][5][5][5];
    int MLintern[8], MLbase, MLclosing, TerminalAU, ninio2, max_ninio;
    int tetra_energy[64];
    double lxc;
    int pair[8][8], rtype[8];
} params_t;

static params_t P0;
static int P_ready = 0;

/* scale_parameters at T=37: tables are taken as-is; dangles clamped to <= 0; MLintern[t] gets
 * TerminalAU for t>2 (RLF params.c:58-61, :88-95 per SURVEY A.3). */
static void params_init(void)
{
    if (P_ready) return;
    memcpy(P0.stack, T99_stack37, sizeof P0.stack);
    memcpy(P0.hairpin, T99_hairpin37, sizeof P0.hairpin);
    memcpy(P0.bulge, T99_bulge37, sizeof P0.bulge);
    memcpy(P0.internal_loop, T99_internal_loop37, sizeof P0.internal_loop);
    memcpy(P0.mismatchI, T99_mismatchI37, sizeof P0.mismatchI);
    memcpy(P0.mismatchH, T99_mismatchH37, sizeof P0.mismatchH);
    memcpy(P0.int11, T99_int11_37, sizeof P0.int11);
    memcpy(P0.int21, T99_int21_37, sizeof P0.int21);
    memcpy(P0.int22, T99_int22_37, sizeof P0.int22);
    memcpy(P0.pair, T99_BP_pair, sizeof P0.pair);
    memcpy(P0.rtype, T99_rtype, sizeof P0.rtype);
    for (int t = 0; t < 8; t++)
        for (int b = 0; b < 5; b++) {
            int d5 = T99_dangle5_37[t * 5 + b], d3 = T99_dangle3_37[t * 5 + b];
            P0.dangle5[t][b] = d5 > 0 ? 0 : d5;
            P0.dangle3[t][b] = d3 > 0 ? 0 : d3;
        }
    P0.TerminalAU = T99_TerminalAU;
    for (int t = 0; t < 8; t++) P0.MLintern[t] = T99_ML_intern37 + (t > 2 ? P0.TerminalAU : 0);
    P0.MLbase = 0;
    P0.MLclosing = T99_ML_closing37;
    P0.ninio2 = T99_F_ninio37[2];
    P0.max_ninio = T99_MAX_NINIO;
    P0.lxc = T99_lxc37;
    for (int k = 0; k < T99_N_TETRALOOPS; k++) P0.tetra_energy[k] = T99_TETRA_ENERGY37[k];
    P_ready = 1;
}

/* ------------------------------------------------------------------ fold state */
typedef struct {
    int n, Ls;      /* length, L* = min(L, n)                               (A: Lfold.c:149) */
    int W;          /* row width of band matrices = Ls + 6                                   */
    const char *seq; /* converted sequence, 0-based                                          */
    short *S, *S1;  /* 1-based codes                                                         */
    int *c, *m, *dml; /* [ (n+2) rows ][ W ]                                                 */
    int *f3;        /* n+3                                                                   */
    int mut;        /* TB_* tie-break mutations of traceback(); 0 = the reference's rules    */
    const params_t *P;  /* energy tables of this fold (&P0, or a copy with one entry changed) */
    const params_t *PL; /* tables of the two-loops the filter selects (P unless a filter-only entry changes) */
    int ln1, ln2, lpar, ls, ld; /* two-loop filter: n1, n2, parity of j-i, n1+n2, j-i; -1 = any; ln1 < -1: none */
    int ldelta;     /* added to every two-loop the filter selects                            */
    int hs, hdelta; /* added to every hairpin of size hs (after the log extrapolation)       */
} fold_t;

/* Energy perturbations (tests only): a fold in which one term class costs `delta` more.  A class whose raise changes the c
 * matrix is the unique minimiser of some cell, so a kernel that computes that class wrongly must differ from the oracle
 * in that cell.  PERT_NONE is the reference. */
enum {
    PERT_NONE, PERT_SHAPE, PERT_RING, PERT_HAIRPIN_SIZE, PERT_STACK, PERT_BULGE, PERT_INTERNAL, PERT_INT11, PERT_INT21,
    PERT_INT22, PERT_MISMATCH_I, PERT_MISMATCH_H, PERT_HAIRPIN, PERT_TETRA,
};

/* Tie-break mutants (tests only).  Each bit flips one "first match wins" rule of traceback(), so
 * that a test corpus can show it contains ties that rule has to break: a corpus on which a
 * mutant prints the same records as the unmodified oracle cannot tell a GPU traceback that
 * breaks that tie the other way from a correct one.  mut = 0 is the reference's traceback. */
enum {
    TB_F3_LAST = 1 << 0,        /* exterior scan: last k instead of first                       */
    TB_F3_ORDER = 1 << 1,       /* exterior scan, one k: (i+1,k) wins over (i,k)                */
    TB_HAIRPIN_LAST = 1 << 2,   /* pair: two-loop tried before hairpin                          */
    TB_LOOP_LAST = 1 << 3,      /* two-loop scan: last (p,q) instead of first                   */
    TB_ML_BEFORE_LOOP = 1 << 4, /* pair: multiloop closing tried before two-loop                */
    TB_MLC_LAST = 1 << 5,       /* multiloop closing: last split k instead of first             */
    TB_MLC_VARIANT = 1 << 6,    /* multiloop closing, one k: dangle variants in reverse order    */
    TB_FML_PEEL_5 = 1 << 7,     /* fML segment: peel the 5' base before the 3' base             */
    TB_FML_PAIR_ORDER = 1 << 8, /* fML segment: cij > ci1j1 > cij1 > ci1j instead of the reverse */
    TB_FML_SPLIT_LAST = 1 << 9, /* fML segment: last split k instead of first                   */
};

static inline int enc(char ch)
{   /* A.1: index in "_ACGUTXKI", indices >4 decremented; anything else 0 */
    switch (ch) {
    case 'A': return 1; case 'C': return 2; case 'G': return 3; case 'U': return 4;
    case 'T': return 4; case 'X': return 5; case 'K': return 6; case 'I': return 7;
    default: return 0;
    }
}
static const int ALIAS[8] = {0, 1, 2, 3, 4, 3, 2, 0};

static inline int ptype(const fold_t *f, int i, int j)
{   /* A.1: typed only for 4 <= j-i <= L*-1, j <= n */
    int d = j - i;
    if (i < 1 || j > f->n || d < TURN + 1 || d >= f->Ls) return 0;
    return P0.pair[f->S[i]][f->S[j]];
}
static inline int band_get(const fold_t *f, const int *a, int i, int j)
{
    int d = j - i;
    if (i < 1 || i > f->n || j > f->n || d < 0 || d >= f->W) return INF;
    return a[(size_t)i * f->W + d];
}
#define C_(i, j) band_get(f, f->c, (i), (j))
#define M_(i, j) band_get(f, f->m, (i), (j))
#define D_(i, j) band_get(f, f->dml, (i), (j))
static inline int F_(const fold_t *f, int i) { return (i >= 1 && i <= f->n + 2) ? f->f3[i] : 0; }
static inline int AU(const params_t *P, int t) { return t > 2 ? P->TerminalAU : 0; }

/* A.2 hairpin, size s = j-i-1 before any perturbation */
static int hairpin_tab(const params_t *P, const char *seq, const short *S1, int i, int j, int t)
{
    int s = j - i - 1;
    int e = s <= 30 ? P->hairpin[s] : P->hairpin[30] + (int)(P->lxc * log(s / 30.));
    if (s == 4) {
        char six[7];
        memcpy(six, seq + (i - 1), 6);
        six[6] = 0;
        const char *hit = strstr(T99_Tetraloops, six);
        if (hit) e += P->tetra_energy[(hit - T99_Tetraloops) / 7];
    }
    if (s == 3) e += AU(P, t);            /* no mismatch, Triloops empty */
    else e += P->mismatchH[t][S1[i + 1]][S1[j - 1]];
    return e;
}
static int hairpin_E(const fold_t *f, int i, int j)
{
    return hairpin_tab(f->P, f->seq, f->S1, i, j, ptype(f, i, j)) + (j - i - 1 == f->hs ? f->hdelta : 0);
}

/* A.2 two-loop closed by (i,j) [type t] and (p,q) [t2 = rtype of its type] */
static int loop_tab(const params_t *P, const short *S1, int i, int j, int p, int q, int t, int t2)
{
    int n1 = p - i - 1, n2 = j - q - 1;
    int nl = n1 > n2 ? n1 : n2, ns = n1 > n2 ? n2 : n1;
    if (nl == 0) return P->stack[t][t2];
    if (ns == 0) {
        int e = P->bulge[nl];
        return nl == 1 ? e + P->stack[t][t2] : e + AU(P, t) + AU(P, t2);
    }
    if (ns == 1 && nl == 1) return P->int11[t][t2][S1[i + 1]][S1[j - 1]];
    if (ns == 1 && nl == 2)
        return n1 == 1 ? P->int21[t][t2][S1[i + 1]][S1[q + 1]][S1[j - 1]]
                       : P->int21[t2][t][S1[q + 1]][S1[i + 1]][S1[p - 1]];
    if (n1 == 2 && n2 == 2) return P->int22[t][t2][S1[i + 1]][S1[p - 1]][S1[q + 1]][S1[j - 1]];
    int nin = (nl - ns) * P->ninio2;
    if (nin > P->max_ninio) nin = P->max_ninio;
    return P->internal_loop[n1 + n2] + nin + P->mismatchI[t][S1[i + 1]][S1[j - 1]] +
           P->mismatchI[t2][S1[q + 1]][S1[p - 1]];
}
static int loop_E(const fold_t *f, int i, int j, int p, int q, int t, int t2)
{
    int n1 = p - i - 1, n2 = j - q - 1, d = j - i;
    if (f->ln1 < -1 || (f->ln1 >= 0 && f->ln1 != n1) || (f->ln2 >= 0 && f->ln2 != n2) ||
        (f->lpar >= 0 && f->lpar != (d & 1)) || (f->ls >= 0 && f->ls != n1 + n2) || (f->ld >= 0 && f->ld != d))
        return loop_tab(f->P, f->S1, i, j, p, q, t, t2);
    return loop_tab(f->PL, f->S1, i, j, p, q, t, t2) + f->ldelta;
}

static inline int imin(int a, int b) { return a < b ? a : b; }

/* ------------------------------------------------------------------ A.3 fill */
static void fill_row(fold_t *f, int i)
{
    const params_t *P = f->P;
    const int n = f->n, Ls = f->Ls, W = f->W;
    const short *S1 = f->S1;
    int jmax = imin(n, i + Ls);
    for (int j = i + TURN + 1; j <= jmax; j++) {
        int t = ptype(f, i, j), cij = INF;
        if (t) {
            cij = hairpin_E(f, i, j);
            int pmax = imin(j - 2 - TURN, i + MAXLOOP + 1);
            for (int p = i + 1; p <= pmax; p++) {
                int minq = j - i + p - MAXLOOP - 2;
                if (minq < p + 1 + TURN) minq = p + 1 + TURN;
                for (int q = minq; q < j; q++) {
                    int t2 = ptype(f, p, q);
                    if (!t2) continue;
                    cij = imin(cij, loop_E(f, i, j, p, q, t, P->rtype[t2]) + C_(p, q));
                }
            }
            int tt = P->rtype[t];
            int d3 = P->dangle3[tt][S1[i + 1]], d5 = P->dangle5[tt][S1[j - 1]];
            int dec = D_(i + 1, j - 1);
            dec = imin(dec, D_(i + 2, j - 1) + d3 + P->MLbase);
            dec = imin(dec, D_(i + 1, j - 2) + d5 + P->MLbase);
            dec = imin(dec, D_(i + 2, j - 2) + d3 + d5 + 2 * P->MLbase);
            cij = imin(cij, P->MLclosing + P->MLintern[t] + dec);
        }
        f->c[(size_t)i * W + (j - i)] = cij;

        int mij = M_(i + 1, j) + P->MLbase;
        mij = imin(mij, M_(i, j - 1) + P->MLbase);
        mij = imin(mij, cij + P->MLintern[t]);
        int ta = ptype(f, i + 1, j);
        mij = imin(mij, C_(i + 1, j) + P->dangle5[ta][S1[i]] + P->MLintern[ta] + P->MLbase);
        int tb = ptype(f, i, j - 1);
        mij = imin(mij, C_(i, j - 1) + P->dangle3[tb][S1[j]] + P->MLintern[tb] + P->MLbase);
        int tc = ptype(f, i + 1, j - 1);
        mij = imin(mij, C_(i + 1, j - 1) + P->dangle5[tc][S1[i]] + P->dangle3[tc][S1[j]] +
                            P->MLintern[tc] + 2 * P->MLbase);
        int dec = INF;
        for (int k = i + 1 + TURN; k <= j - 2 - TURN; k++) dec = imin(dec, M_(i, k) + M_(k + 1, j));
        f->dml[(size_t)i * W + (j - i)] = dec;
        mij = imin(mij, dec);
        f->m[(size_t)i * W + (j - i)] = mij;
    }
}

static void f3_row(fold_t *f, int i)
{
    const params_t *P = f->P;
    const int n = f->n, Ls = f->Ls;
    const short *S1 = f->S1;
    int fi = F_(f, i + 1);
    for (int j = i + TURN + 1; j < n && j <= i + Ls; j++) {
        int t = ptype(f, i, j);
        if (t) {
            int e = C_(i, j) + AU(P, t);
            fi = imin(fi, e + F_(f, j + 1));
            fi = imin(fi, e + P->dangle3[t][S1[j + 1]] + F_(f, j + 2));
        }
        t = ptype(f, i + 1, j);
        if (t) {
            int e = C_(i + 1, j) + P->dangle5[t][S1[i]] + AU(P, t);
            fi = imin(fi, e + F_(f, j + 1));
            fi = imin(fi, e + P->dangle3[t][S1[j + 1]] + F_(f, j + 2));
        }
    }
    if (n <= i + Ls) {
        int t = ptype(f, i, n);
        if (t) fi = imin(fi, C_(i, n) + AU(P, t));
        t = ptype(f, i + 1, n);
        if (t) fi = imin(fi, C_(i + 1, n) + P->dangle5[t][S1[i]] + AU(P, t));
    }
    f->f3[i] = fi;
}

/* ------------------------------------------------------------------ A.4 traceback */
typedef struct { int i, j, ml; } sect_t;

/* two-loop (p,q) that reproduces c(i,j): p ascending, q descending, first match (last with TB_LOOP_LAST) */
static int two_loop_split(const fold_t *f, int i, int j, int cij, int t, int *pp, int *qq)
{
    const params_t *P = f->P;
    int found = 0;
    int pmax = imin(j - 2 - TURN, i + MAXLOOP + 1);
    for (int p = i + 1; p <= pmax; p++) {
        int minq = j - i + p - MAXLOOP - 2;
        if (minq < p + 1 + TURN) minq = p + 1 + TURN;
        for (int q = j - 1; q >= minq; q--) {
            int t2 = ptype(f, p, q);
            if (!t2) continue;
            if (cij == loop_E(f, i, j, p, q, t, P->rtype[t2]) + C_(p, q)) {
                *pp = p; *qq = q; found = 1;
                if (!(f->mut & TB_LOOP_LAST)) return 1;
            }
        }
    }
    return found;
}

/* multiloop closed by (i,j): split k ascending (descending with TB_MLC_LAST), four dangle variants per k */
static int ml_split(const fold_t *f, int i, int j, int cij, int t, int *kk, int *i1, int *j1)
{
    const params_t *P = f->P;
    int tt = P->rtype[t];
    int mm = P->MLclosing + P->MLintern[tt];
    int d5 = P->dangle5[tt][f->S1[j - 1]], d3 = P->dangle3[tt][f->S1[i + 1]];
    const int klo = i + 2 + TURN, khi = j - 3 - TURN;
    const int last = (f->mut & TB_MLC_LAST) != 0, rev = (f->mut & TB_MLC_VARIANT) != 0;
    for (int s = 0; s <= khi - klo; s++) {
        int k = last ? khi - s : klo + s;
        for (int o = 0; o < 4; o++) {
            int v = rev ? 3 - o : o, a = v & 1, b = v >> 1;   /* v: 0 (i+1,j-1), 1 (i+2,j-1), 2 (i+1,j-2), 3 (i+2,j-2) */
            int e = M_(i + 1 + a, k) + M_(k + 1, j - 1 - b) + mm + (a ? d3 : 0) + (b ? d5 : 0) + (a + b) * P->MLbase;
            if (cij == e) { *kk = k; *i1 = i + 1 + a; *j1 = j - 1 - b; return 1; }
        }
    }
    return 0;
}

/* returns malloc'ed finalised structure string, or NULL on "backtrack failed" */
static char *traceback(fold_t *f, int start, int md)
{
    const params_t *P = f->P;
    const int n = f->n;
    const short *S1 = f->S1;
    int ndash = imin(n - start, md) + 1;
    char *st = (char *)calloc((size_t)ndash + 4, 1);
    memset(st, '-', (size_t)ndash);
    int cap = 4 * (ndash + 8), sp = 0;
    sect_t *stk = (sect_t *)malloc(sizeof(sect_t) * (size_t)cap);
#define PUSH(a, b, c_) do { stk[sp].i = (a); stk[sp].j = (b); stk[sp].ml = (c_); sp++; } while (0)
    PUSH(start, imin(n, start + md + 1), 0);
    while (sp > 0) {
        sp--;
        int i = stk[sp].i, j = stk[sp].j, ml = stk[sp].ml;
        if (j < i + TURN + 1) continue;
        if (ml == 0) {
            int fij = F_(f, i);
            if (fij == F_(f, i + 1)) { PUSH(i + 1, j, 0); continue; }
            /* per k the later match wins: (i+1,k) then (i,k) (reversed by TB_F3_ORDER), no dangle then 3' dangle */
            int traced = 0, jj = 0, k, bt = 0, bjj = 0, bk = 0;
            for (k = i + TURN + 1; k <= j; k++) {
                jj = k + 1;
                traced = 0;
                for (int o = 0; o < 2; o++) {
                    int a = (o == 0) == !(f->mut & TB_F3_ORDER) ? i + 1 : i;
                    int t = ptype(f, a, k);
                    if (!t) continue;
                    int cc = C_(a, k) + (a > i ? P->dangle5[t][S1[i]] : 0) + AU(P, t);
                    if (fij == cc + F_(f, k + 1)) traced = a;
                    if (k < n && fij == F_(f, k + 2) + cc + P->dangle3[t][S1[k + 1]]) { traced = a; jj = k + 2; }
                }
                if (traced) {
                    bt = traced; bjj = jj; bk = k;
                    if (!(f->mut & TB_F3_LAST)) break;
                }
            }
            if (!bt) goto fail;
            traced = bt; jj = bjj; k = bk;
            if (j == n) PUSH(jj, j, 0);
            i = traced; j = k;
            st[i - start] = '('; st[j - start] = ')';
            if (jj == j + 2 && j < n) st[j + 1 - start] = '.';
        } else {
            int fij = M_(i, j);
            for (int o = 0; o < 2; o++) {   /* 3' base first (5' first with TB_FML_PEEL_5) */
                int five = (o == 0) == !!(f->mut & TB_FML_PEEL_5);
                if (M_(i + five, j - !five) + P->MLbase == fij) { PUSH(i + five, j - !five, 1); goto next; }
            }
            int t = ptype(f, i, j);
            int cij = C_(i, j) + P->MLintern[t];
            t = ptype(f, i + 1, j);
            int ci1j = C_(i + 1, j) + P->dangle5[t][S1[i]] + P->MLintern[t] + P->MLbase;
            t = ptype(f, i, j - 1);
            int cij1 = C_(i, j - 1) + P->dangle3[t][S1[j]] + P->MLintern[t] + P->MLbase;
            t = ptype(f, i + 1, j - 1);
            int ci1j1 = C_(i + 1, j - 1) + P->dangle5[t][S1[i]] + P->dangle3[t][S1[j]] + P->MLintern[t] + 2 * P->MLbase;
            if (fij == cij || fij == ci1j || fij == cij1 || fij == ci1j1) {
                /* first match of ci1j, cij1, ci1j1, cij (the reverse with TB_FML_PAIR_ORDER) */
                const int e[4] = {ci1j, cij1, ci1j1, cij}, di[4] = {1, 0, 1, 0}, dj[4] = {0, 1, 1, 0};
                for (int o = 0; o < 4; o++) {
                    int v = (f->mut & TB_FML_PAIR_ORDER) ? 3 - o : o;
                    if (fij == e[v]) { i += di[v]; j -= dj[v]; break; }
                }
                st[i - start] = '('; st[j - start] = ')';
            } else {
                int k, found = 0;
                for (k = i + 1 + TURN; k <= j - 2 - TURN; k++) {
                    int kk = (f->mut & TB_FML_SPLIT_LAST) ? i + j - 1 - k : k;   /* j-2-TURN .. i+1+TURN */
                    if (fij == M_(i, kk) + M_(kk + 1, j)) { k = kk; found = 1; break; }
                }
                if (!found) goto fail;
                PUSH(i, k, 1);
                PUSH(k + 1, j, 1);
                continue;
            }
        }
        /* "repeat": (i,j) is a known pair; walk the stem/interior loops down.  Hairpin, then two-loop, then
         * multiloop; TB_HAIRPIN_LAST and TB_ML_BEFORE_LOOP reorder these (0 hairpin, 1 two-loop, 2 multiloop). */
        for (;;) {
            int cij = C_(i, j), t = ptype(f, i, j);
            static const int ORDER[4][3] = {{0, 1, 2}, {1, 0, 2}, {0, 2, 1}, {2, 1, 0}};
            const int *ord = ORDER[((f->mut & TB_HAIRPIN_LAST) ? 1 : 0) + ((f->mut & TB_ML_BEFORE_LOOP) ? 2 : 0)];
            int step = -1, p = 0, q = 0, k = 0, i1 = 0, j1 = 0;
            for (int o = 0; o < 3 && step < 0; o++) {
                if (ord[o] == 0 && cij == hairpin_E(f, i, j)) step = 0;
                else if (ord[o] == 1 && two_loop_split(f, i, j, cij, t, &p, &q)) step = 1;
                else if (ord[o] == 2 && ml_split(f, i, j, cij, t, &k, &i1, &j1)) step = 2;
            }
            if (step < 0) goto fail;
            if (step == 0) break;
            if (step == 1) {
                st[p - start] = '('; st[q - start] = ')';
                i = p; j = q;
                continue;
            }
            PUSH(i1, k, 1);
            PUSH(k + 1, j1, 1);
            break;
        }
    next:
        if (sp + 4 > cap) { cap *= 2; stk = (sect_t *)realloc(stk, sizeof(sect_t) * (size_t)cap); }
    }
    free(stk);
    {
        int k = (int)strlen(st) - 1;
        for (; k > 0 && st[k] == '-'; k--) st[k] = 0;
        for (; k >= 0; k--) if (st[k] == '-') st[k] = '.';
    }
    return st;
fail:
    free(stk);
    free(st);
    return NULL;
#undef PUSH
}

/* ------------------------------------------------------------------ public result type */
typedef struct {
    int n_hits, cap_hits;
    int *start;       /* 1-based printed start                                   */
    int *energy;      /* dcal: F(start) - F(start+len)                            */
    char **ss;        /* finalised structures, print order                        */
    int total;        /* F(1), dcal                                               */
    int failed;       /* nonzero if a traceback failed (reference would abort)    */
    char *conv;       /* converted sequence (uppercase, T->U)                     */
    int n;
    /* optional matrix dumps (kept when keep_matrices) */
    int W, Ls;
    int *c, *m, *f3;
} lfold_result;

static void add_hit(lfold_result *r, const fold_t *f, char *ss, int start)
{
    if (r->n_hits == r->cap_hits) {
        r->cap_hits = r->cap_hits ? 2 * r->cap_hits : 32;
        r->start = (int *)realloc(r->start, sizeof(int) * (size_t)r->cap_hits);
        r->energy = (int *)realloc(r->energy, sizeof(int) * (size_t)r->cap_hits);
        r->ss = (char **)realloc(r->ss, sizeof(char *) * (size_t)r->cap_hits);
    }
    int len = (int)strlen(ss);
    r->start[r->n_hits] = start;
    r->energy[r->n_hits] = F_(f, start) - F_(f, start + len);
    r->ss[r->n_hits] = strdup(ss);
    r->n_hits++;
}

/* Fold one raw sequence token (A.6 conversion, A.3 fill, A.5 emission) with the tables, two-loop filter and hairpin
 * perturbation of `pert`; `mut`: TB_* bits of the tracebacks (0 = RNALfold's). */
static lfold_result *fold_core(const char *raw, int n, int L, int keep_matrices, int mut, const fold_t *pert)
{
    lfold_result *r = (lfold_result *)calloc(1, sizeof *r);
    r->n = n;
    r->conv = (char *)malloc((size_t)n + 1);
    for (int k = 0; k < n; k++) {
        char ch = raw[k];
        if (ch >= 'a' && ch <= 'z') ch = (char)(ch - 32);
        if (ch == 'T') ch = 'U';
        r->conv[k] = ch;
    }
    r->conv[n] = 0;
    fold_t F, *f = &F;
    f->n = n;
    f->Ls = L < n ? L : n;
    f->W = f->Ls + 6;
    f->seq = r->conv;
    f->S = (short *)calloc((size_t)n + 3, sizeof(short));
    f->S1 = (short *)calloc((size_t)n + 3, sizeof(short));
    for (int k = 1; k <= n; k++) { f->S[k] = (short)enc(r->conv[k - 1]); f->S1[k] = (short)ALIAS[f->S[k]]; }
    size_t cells = (size_t)(n + 2) * (size_t)f->W;
    f->c = (int *)malloc(sizeof(int) * cells);
    f->m = (int *)malloc(sizeof(int) * cells);
    f->dml = (int *)malloc(sizeof(int) * cells);
    for (size_t k = 0; k < cells; k++) f->c[k] = f->m[k] = f->dml[k] = INF;
    f->f3 = (int *)calloc((size_t)n + 4, sizeof(int));
    f->mut = mut;
    f->P = pert->P; f->PL = pert->PL;
    f->ln1 = pert->ln1; f->ln2 = pert->ln2; f->lpar = pert->lpar; f->ls = pert->ls; f->ld = pert->ld;
    f->ldelta = pert->ldelta;
    f->hs = pert->hs; f->hdelta = pert->hdelta;

    /* A.5 emission state machine, static state is per-call here (one Lfold() per process
     * call sequence in the reference keeps statics across records, but they are always
     * left at do_bt=0, prev=NULL when i==1 completes). */
    int do_bt = 0, prev_i = 0;
    char *prev = NULL;
    for (int i = n - TURN - 1; i >= 1 && !r->failed; i--) {
        fill_row(f, i);
        f3_row(f, i);
        if (F_(f, i) != F_(f, i + 1)) do_bt = 1;
        else if (do_bt) {
            char *ss = traceback(f, i + 1, f->Ls + 1);
            if (!ss) { r->failed = 1; break; }
            if (prev) {
                size_t ls = strlen(ss), lp = strlen(prev);
                int off = prev_i - i;
                if ((size_t)i + ls < (size_t)prev_i + lp || strncmp(ss + off, prev, lp) != 0)
                    add_hit(r, f, prev, prev_i);
                free(prev);
            }
            prev = ss; prev_i = i + 1; do_bt = 0;
        }
        if (i == 1) {
            if (prev) { add_hit(r, f, prev, prev_i); free(prev); prev = NULL; }
            else do_bt = 1;
            if (do_bt) {
                char *ss = traceback(f, 1, f->Ls);
                if (!ss) { r->failed = 1; break; }
                add_hit(r, f, ss, 1);
                free(ss);
            }
            do_bt = 0;
        }
    }
    free(prev);
    r->total = n >= 1 ? F_(f, 1) : 0;
    if (keep_matrices) { r->W = f->W; r->Ls = f->Ls; r->c = f->c; r->m = f->m; r->f3 = f->f3; }
    else { free(f->c); free(f->m); free(f->f3); }
    free(f->dml); free(f->S); free(f->S1);
    return r;
}

static void pert_none(fold_t *pf)
{
    params_init();
    memset(pf, 0, sizeof *pf);
    pf->P = pf->PL = &P0;
    pf->ln1 = -2;
    pf->hs = -1;
}

lfold_result *lfold_oracle_fold_mut(const char *raw, int n, int L, int keep_matrices, int mut)
{
    fold_t pf;
    pert_none(&pf);
    return fold_core(raw, n, L, keep_matrices, mut, &pf);
}

lfold_result *lfold_oracle_fold(const char *raw, int n, int L, int keep_matrices)
{
    return lfold_oracle_fold_mut(raw, n, L, keep_matrices, 0);
}

static int in_range(const int *x, int k, int lo, int hi)
{
    for (int a = 0; a < k; a++)
        if (x[a] < lo || x[a] > hi) return 0;
    return 1;
}

/* The fold of lfold_oracle_fold_mut with one term class raised by `delta` dcal (PERT_*, index x[]):
 *   SHAPE (n1, n2, parity)   every two-loop with n1 / n2 unpaired bases whose outer pair has j-i of that parity (stacks
 *                            and bulges included)
 *   RING (s, d)              every two-loop of n1+n2 = s closed by a pair with j-i = d
 *   HAIRPIN_SIZE (s)         every hairpin of s unpaired bases, after the lxc*log extrapolation of s > 30
 *   STACK (t, t2), BULGE (s), INTERNAL (s), INT11 (t, t2, x, y), INT22 (t, t2, a, b, c, d), MISMATCH_I (t, x, y),
 *   MISMATCH_H (t, x, y), HAIRPIN (s), TETRA (k)
 *                            that entry of the table, wherever it is read
 *   INT21 (n1, t, t2, x, y, z)   int21[t][t2][x][y][z], read by 1x2 loops of that n1 only (1: 5' side 1 nt, 2: 2 nt)
 * Returns NULL for an unknown kind or an index out of range. */
lfold_result *lfold_oracle_fold_pert(const char *raw, int n, int L, int keep_matrices, int mut, int kind, const int *x,
                                     int delta)
{
    fold_t pf;
    pert_none(&pf);
    params_t *Q = (params_t *)malloc(sizeof *Q);
    *Q = P0;
    int *e = NULL, ok = 1;
    switch (kind) {
    case PERT_NONE: break;
    case PERT_SHAPE:
        ok = in_range(x, 2, 0, MAXLOOP) && x[0] + x[1] <= MAXLOOP && in_range(x + 2, 1, 0, 1);
        pf.ln1 = x[0]; pf.ln2 = x[1]; pf.lpar = x[2]; pf.ls = pf.ld = -1; pf.ldelta = delta;
        break;
    case PERT_RING:
        ok = in_range(x, 1, 0, MAXLOOP) && x[1] >= 0;
        pf.ln1 = pf.ln2 = pf.lpar = -1; pf.ls = x[0]; pf.ld = x[1]; pf.ldelta = delta;
        break;
    case PERT_HAIRPIN_SIZE: ok = x[0] >= 3; pf.hs = x[0]; pf.hdelta = delta; break;
    case PERT_STACK: if ((ok = in_range(x, 2, 0, 7))) e = &Q->stack[x[0]][x[1]]; break;
    case PERT_BULGE: if ((ok = in_range(x, 1, 0, MAXLOOP))) e = &Q->bulge[x[0]]; break;
    case PERT_INTERNAL: if ((ok = in_range(x, 1, 0, MAXLOOP))) e = &Q->internal_loop[x[0]]; break;
    case PERT_HAIRPIN: if ((ok = in_range(x, 1, 0, MAXLOOP))) e = &Q->hairpin[x[0]]; break;
    case PERT_TETRA: if ((ok = in_range(x, 1, 0, T99_N_TETRALOOPS - 1))) e = &Q->tetra_energy[x[0]]; break;
    case PERT_INT11: if ((ok = in_range(x, 2, 0, 7) && in_range(x + 2, 2, 0, 4))) e = &Q->int11[x[0]][x[1]][x[2]][x[3]]; break;
    case PERT_INT22:
        if ((ok = in_range(x, 2, 0, 7) && in_range(x + 2, 4, 0, 4))) e = &Q->int22[x[0]][x[1]][x[2]][x[3]][x[4]][x[5]];
        break;
    case PERT_MISMATCH_I: if ((ok = in_range(x, 1, 0, 7) && in_range(x + 1, 2, 0, 4))) e = &Q->mismatchI[x[0]][x[1]][x[2]]; break;
    case PERT_MISMATCH_H: if ((ok = in_range(x, 1, 0, 7) && in_range(x + 1, 2, 0, 4))) e = &Q->mismatchH[x[0]][x[1]][x[2]]; break;
    case PERT_INT21:
        if ((ok = in_range(x, 1, 1, 2) && in_range(x + 1, 2, 0, 7) && in_range(x + 3, 3, 0, 4))) {
            e = &Q->int21[x[1]][x[2]][x[3]][x[4]][x[5]];
            pf.ln1 = x[0]; pf.ln2 = 3 - x[0]; pf.lpar = pf.ls = pf.ld = -1;
        }
        break;
    default: ok = 0;
    }
    lfold_result *r = NULL;
    if (ok) {
        if (e) *e += delta;
        if (kind == PERT_INT21) pf.PL = Q;
        else if (e) pf.P = pf.PL = Q;
        r = fold_core(raw, n, L, keep_matrices, mut, &pf);
    }
    free(Q);
    return r;
}

/* hairpin_E of the pair (i, j) (1-based) of a raw sequence, with the unmodified tables: the energy of a long hairpin,
 * whose fold would cost O(n^3) in the multiloop decomposition */
int lfold_oracle_hairpin_energy(const char *raw, int n, int i, int j)
{
    params_init();
    if (i < 1 || j > n || j - i - 1 < TURN) return INF;
    char *conv = (char *)malloc((size_t)n + 1);
    short *S = (short *)calloc((size_t)n + 3, sizeof(short)), *S1 = (short *)calloc((size_t)n + 3, sizeof(short));
    for (int k = 0; k < n; k++) {
        char ch = raw[k];
        if (ch >= 'a' && ch <= 'z') ch = (char)(ch - 32);
        conv[k] = ch == 'T' ? 'U' : ch;
        S[k + 1] = (short)enc(conv[k]);
        S1[k + 1] = (short)ALIAS[S[k + 1]];
    }
    conv[n] = 0;
    int t = P0.pair[S[i]][S[j]];
    int e = t ? hairpin_tab(&P0, conv, S1, i, j, t) : INF;
    free(conv); free(S); free(S1);
    return e;
}

void lfold_oracle_free(lfold_result *r)
{
    if (!r) return;
    for (int k = 0; k < r->n_hits; k++) free(r->ss[k]);
    free(r->ss); free(r->start); free(r->energy); free(r->conv);
    free(r->c); free(r->m); free(r->f3);
    free(r);
}

/* flat accessors for ctypes */
int lfold_oracle_nhits(const lfold_result *r) { return r->n_hits; }
int lfold_oracle_total(const lfold_result *r) { return r->total; }
int lfold_oracle_failed(const lfold_result *r) { return r->failed; }
int lfold_oracle_hit_start(const lfold_result *r, int k) { return r->start[k]; }
int lfold_oracle_hit_energy(const lfold_result *r, int k) { return r->energy[k]; }
const char *lfold_oracle_hit_ss(const lfold_result *r, int k) { return r->ss[k]; }
const char *lfold_oracle_conv(const lfold_result *r) { return r->conv; }
int lfold_oracle_W(const lfold_result *r) { return r->W; }
/* band matrices, [i][d] with row stride W (1-based i), INF where not computed */
const int *lfold_oracle_c(const lfold_result *r) { return r->c; }
const int *lfold_oracle_m(const lfold_result *r) { return r->m; }
const int *lfold_oracle_f3(const lfold_result *r) { return r->f3; }

/* ------------------------------------------------------------------ A.6 program I/O */
/* Reads multi-FASTA-ish text from `in`, writes RNALfold-identical text to `out`. */
int lfold_oracle_stream(FILE *in, FILE *out, int L)
{
    char *line = NULL;
    size_t cap = 0;
    ssize_t len;
    for (;;) {
        if ((len = getline(&line, &cap, in)) < 0) break;
        if (len && line[len - 1] == '\n') line[--len] = 0;
        while (line[0] == '*' || line[0] == 0 || line[0] == '>') {
            fprintf(out, "%s\n", line);
            if ((len = getline(&line, &cap, in)) < 0) goto done;
            if (len && line[len - 1] == '\n') line[--len] = 0;
        }
        if (strcmp(line, "@") == 0) break;
        /* first whitespace-delimited token */
        char *tok = line;
        while (*tok == ' ' || *tok == '\t' || *tok == '\r' || *tok == '\v' || *tok == '\f') tok++;
        int n = 0;
        while (tok[n] && tok[n] != ' ' && tok[n] != '\t' && tok[n] != '\r' && tok[n] != '\v' && tok[n] != '\f' && tok[n] != '\n') n++;
        lfold_result *r = lfold_oracle_fold(tok, n, L, 0);
        if (r->failed) { fprintf(stderr, "backtrack failed\n"); lfold_oracle_free(r); free(line); return 1; }
        for (int k = 0; k < r->n_hits; k++)
            fprintf(out, "%s (%6.2f) %4d\n", r->ss[k], r->energy[k] / 100., r->start[k]);
        fprintf(out, "%s\n (%6.2f)\n", r->conv, r->total / 100.);
        lfold_oracle_free(r);
    }
done:
    free(line);
    return 0;
}

#ifdef LFOLD_ORACLE_MAIN
int main(int argc, char **argv)
{
    int L = 150;  /* RNALfold default */
    for (int a = 1; a < argc; a++)
        if (!strcmp(argv[a], "-L") && a + 1 < argc) L = atoi(argv[++a]);
    return lfold_oracle_stream(stdin, stdout, L);
}
#endif
