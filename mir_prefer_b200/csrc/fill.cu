// fill.cu -- sequence encoding (K1), c/fML band fill (K2) and the f3 scan (K3) for sm_100a.
//
// Replaces the arithmetic of RNALfold's fill_arrays (SURVEY.md 8a rows a4-a7; behavioural spec
// Appendix A.1-A.3, "RLF Lfold.c:170-398").  One CTA owns one locus and walks the band by
// anti-diagonal d = j-i (all cells of a diagonal are independent).  Restructuring relative to the
// reference's row-by-row loop (results are bit-identical, the order of evaluation is not):
//   * DML(i,j) = min_k fML(i,k)+fML(k+1,j) only reads diagonals <= d-5, so it is produced in
//     strips of five diagonals ahead of the wavefront (phase A), one thread per row with the
//     five running minima in registers: one fML(i,k) load feeds five min-plus terms.  The band is
//     rectangular diagonal-major with a compile-time stride, so all operand addresses of the
//     unrolled loop are one pointer + immediates.
//   * the <=30-nt interior-loop search is a min-plus stencil over the previous 31 diagonals:
//     generic loops use Cm(p,q) = c(p,q)+mismatchI[rtype][..] (+INF if (p,q) cannot pair) and a
//     per-(u,v) constant, so no pair-type test is needed.  The 33-diagonal Cm window lives in a
//     shared-memory ring; a warp evaluates the 496 (u,v) terms of one typed cell in 16
//     fully-populated iterations (loop sizes s and 30-s share a warp; per-lane ring offsets and
//     constants are set up once per diagonal, the inner loop is LDS + VIADDMNMX) and finishes
//     with redux.sync.  Bulges reuse the ring through a byte ring of (AU - mismatch) deltas.
//   * the 7 table-driven two-loops (stack, 1-nt bulges, 1x1, 1x2, 2x1, 2x2), the hairpin and the
//     d1 multiloop closing are evaluated lane-per-cell for 32 typed cells at a time.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "mirfold_internal.cuh"
#include "fill_common.cuh"

// ------------------------------------------------------------------------------------ K1
__global__ void k_prepare(const char *__restrict__ raw, const LocusDesc *__restrict__ loci, int nloci,
                          unsigned char *__restrict__ codes, int *__restrict__ F)
{
    // one CTA per locus; RNALfold main(): toupper, T->U; encode_char + alias (A.1)
    // raw_off bit 63 (MF_RAW_REVERSE, uniform per CTA): a minus-strand genome region -- base k is raw[off + n - k]
    // through the reference's get_complement table (upper-case A T G C U only; miR_PREFeR.py:232-239), then as above
    const LocusDesc L = loci[blockIdx.x];
    const bool rev = (L.raw_off & MF_RAW_REVERSE) != 0;
    const char *src = raw + (L.raw_off & ~MF_RAW_REVERSE);
    unsigned char *dst = codes + L.seq_off;
    int *f = F + L.seq_off;
    for (int k = threadIdx.x; k < L.n + 3; k += blockDim.x) {
        int s = 0;
        if (k >= 1 && k <= L.n) {
            char ch;
            if (rev) {
                ch = src[L.n - k];
                ch = ch == 'A' ? 'U' : ch == 'T' ? 'A' : ch == 'G' ? 'C' : ch == 'C' ? 'G' : ch == 'U' ? 'A' : ch;
            } else ch = src[k - 1];
            if (ch >= 'a' && ch <= 'z') ch -= 32;
            switch (ch) {
            case 'A': s = 1; break;
            case 'C': s = 2; break;
            case 'G': s = 3; break;
            case 'U': case 'T': s = 4; break;
            case 'X': s = 5; break;
            case 'K': s = 6; break;
            case 'I': s = 7; break;
            default: s = 0;
            }
        }
        const int alias = (0x02343210 >> (4 * s)) & 7;  // {0,1,2,3,4,3,2,0}
        dst[k] = (unsigned char)(s | (alias << 4));
        f[k] = 0;
    }
}

cudaError_t launch_prepare(const char *raw, const LocusDesc *loci, int nloci, unsigned long long, unsigned char *codes,
                           int *F, cudaStream_t st)
{
    if (nloci == 0) return cudaSuccess;
    k_prepare<<<nloci, 128, 0, st>>>(raw, loci, nloci, codes, F);
    return cudaGetLastError();
}

// the seven table-driven two-loops of a typed cell + hairpin + d1 multiloop closing (A.2, A.3)
// Cb = band base of c; rD = DML ring [MF_RING_DML][NS]
template <class StrideT>
__device__ __forceinline__ int dev_cell_tail(const DevParams *__restrict__ P, const unsigned char *sS,
                                             const unsigned char *sS1, const unsigned char *sPair,
                                             const int *Cb, const int *rD, StrideT NS, int i,
                                             int d, int t, int si1, int sj1, int K)
{
    const int j = i + d;
    int best = MF_INF;
#pragma unroll
    for (int m = 0; m < 7; m++) {
        const int u = (m == 1 || m == 3 || m == 4) ? 1 : (m >= 5 ? 2 : 0);
        const int v = (m == 2 || m == 3 || m == 5) ? 1 : ((m == 4 || m == 6) ? 2 : 0);
        // m: 0 (0,0)  1 (1,0)  2 (0,1)  3 (1,1)  4 (1,2)  5 (2,1)  6 (2,2)
        if (u + v <= K) {
            const int p = i + 1 + u, q = j - 1 - v;
            const int t2 = sPair[sS[p] * 8 + sS[q]];
            if (t2) {
                const int e = dev_loop_energy(P, t, P->rtype[t2], u, v, si1, sj1, sS1[p - 1], sS1[q + 1]);
                best = min(best, e + Cb[(q - p - 4) * NS + (p - 1)]);
            }
        }
    }
    best = min(best, dev_hairpin(P, sS, sS1, i, j, t));
    const int tt = P->rtype[t];
    const int d3 = P->dangle3[tt * 5 + si1], d5 = P->dangle5[tt * 5 + sj1];
    int dec = MF_INF;
    if (d - 2 >= 4) dec = rD[((d - 2) & (MF_RING_DML - 1)) * NS + i];                          // DML(i+1,j-1)
    if (d - 3 >= 4) {
        dec = min(dec, rD[((d - 3) & (MF_RING_DML - 1)) * NS + i + 1] + d3);                   // DML(i+2,j-1)
        dec = min(dec, rD[((d - 3) & (MF_RING_DML - 1)) * NS + i] + d5);                       // DML(i+1,j-2)
    }
    if (d - 4 >= 4) dec = min(dec, rD[((d - 4) & (MF_RING_DML - 1)) * NS + i + 1] + d3 + d5);  // DML(i+2,j-2)
    return min(best, P->MLclosing + P->MLintern[t] + dec);
}

// fML(i,j) from its six boundary terms + DML (A.3)
template <class StrideT>
__device__ __forceinline__ int dev_fml(const DevParams *__restrict__ P, const unsigned char *sS, const unsigned char *sS1,
                                       const unsigned char *sPair, const int *Cb, const int *Mb,
                                       const int *rD, StrideT NS, int i, int d, int Ls)
{
    const int j = i + d;
    const int t = (d < Ls) ? sPair[sS[i] * 8 + sS[j]] : 0;
    int m = MF_INF;
    if (d - 1 >= 4) {
        const int *Mp = Mb + (d - 5) * NS, *Cp = Cb + (d - 5) * NS;
        m = min(Mp[i], Mp[i - 1]);                                  // fML(i+1,j), fML(i,j-1)
        const int ta = sPair[sS[i + 1] * 8 + sS[j]];                // (i+1, j)
        m = min(m, Cp[i] + P->dangle5[ta * 5 + sS1[i]] + P->MLintern[ta]);
        const int tb = sPair[sS[i] * 8 + sS[j - 1]];                // (i, j-1)
        m = min(m, Cp[i - 1] + P->dangle3[tb * 5 + sS1[j]] + P->MLintern[tb]);
    }
    m = min(m, Cb[(d - 4) * NS + i - 1] + P->MLintern[t]);
    if (d - 2 >= 4) {
        const int tc = sPair[sS[i + 1] * 8 + sS[j - 1]];            // (i+1, j-1)
        m = min(m, Cb[(d - 6) * NS + i] + P->dangle5[tc * 5 + sS1[i]] + P->dangle3[tc * 5 + sS1[j]] + P->MLintern[tc]);
    }
    return min(m, rD[(d & (MF_RING_DML - 1)) * NS + i - 1]);
}


// phase A: DML for the strip d..d1 from fML diagonals <= d-1.  One (row, part) per thread; `part`
// splits the e-range when the strip has fewer rows than the CTA has threads.
// STORE_INF: a (row, diagonal) without a valid split is written as MF_INF when the thread is its only writer, so the
// ring rows need no preset (k_fill_s16 switching to these strips mid-locus); the default leaves such cells untouched.
template <int NT, bool STORE_INF = false, class StrideT>
__device__ __forceinline__ void dev_phase_a(const int *Mb, int *rD, StrideT NS, int n, int d,
                                            int d1, int tid, bool prefetch = true)
{
    const int emax = d1 - 5;  // e ranges 4..emax for the widest diagonal of the strip
    if (emax < 4) return;
    const int R = n - d;
    const int Rpad = (R + 31) & ~31;
    int nparts = NT / Rpad;
    nparts = max(1, min(nparts, 8));
    const int span = emax - 3;
    const int per = (span + nparts - 1) / nparts;
    for (int base = 0; base < Rpad * nparts; base += NT) {
        const int idx = base + tid;
        const int part = idx / Rpad, i = idx - part * Rpad + 1;
        if (part >= nparts || i > R) continue;
        const int e0 = 4 + part * per, e1 = min(emax, e0 + per - 1);
        if (e0 > e1) continue;
        const int ns = min(d1 - d, n - d - i) + 1;          // valid strip diagonals for this row
        const int *pa = Mb + (e0 - 4) * NS + (i - 1);       // fML(i, i+e)
        const int *pb = Mb + (d - 5 - e0) * NS + (i + e0);  // fML(i+e+1, i+d)   (+ s*NS for d+s)
        int acc[5] = {MF_INF, MF_INF, MF_INF, MF_INF, MF_INF};
        const int emain = min(e1, d - 5);                   // all five diagonals accept e <= d-5
        int e = e0;
        for (; e + 3 <= emain; e += 4) {
            if (prefetch && e + 11 <= emain) {   // pull the two new cache lines of each step two batches ahead into L1
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    dev_prefetch_l1(pa + (8 + k) * NS);
                    dev_prefetch_l1(pb - (8 + k) * (NS - 1));
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int av = pa[k * NS];
#pragma unroll
                for (int s = 0; s < 5; s++)
                    if (s < ns) acc[s] = min(acc[s], av + pb[s * NS - k * (NS - 1)]);
            }
            pa += 4 * NS;
            pb -= 4 * (NS - 1);
        }
        for (; e <= emain; e++) {
            const int av = pa[0];
#pragma unroll
            for (int s = 0; s < 5; s++)
                if (s < ns) acc[s] = min(acc[s], av + pb[s * NS]);
            pa += NS;
            pb -= (NS - 1);
        }
        for (; e <= e1; e++) {   // tail: diagonal d+s accepts e <= d+s-5
            const int av = pa[0];
#pragma unroll
            for (int s = 1; s < 5; s++)
                if (s < ns && e <= d + s - 5) acc[s] = min(acc[s], av + pb[s * NS]);
            pa += NS;
            pb -= (NS - 1);
        }
#pragma unroll
        for (int s = 0; s < 5; s++)
            if (s < ns && (acc[s] < MF_INF || (STORE_INF && nparts == 1))) {
                int *dst = &rD[((d + s) & (MF_RING_DML - 1)) * NS + (i - 1)];
                if (nparts == 1) *dst = acc[s];
                else atomicMin(dst, acc[s]);
            }
    }
}


// phase A on 16-bit row pairs (narrow kernel).  Mp holds fML16 per diagonal as words of two rows: E[t] = rows
// (2t+1 | 2t+2) (lo | hi half).  Thread t owns the rows (i, i+1) = (2t+1, 2t+2): the left operand
// fML(i,i+e) | fML(i+1,i+1+e) is E[t] of diagonal e.  The right operand fML(i+e+1, .) | fML(i+e+2, .) is E[t + (e+1)/2]
// for odd e; for even e it is the odd-aligned pair rows (2u+2 | 2u+3), u = t + e/2.  Two layouts (template OC):
//   OC = true  : a second, odd-aligned copy O[u] of every diagonal is stored behind E (NS words per diagonal) -- one LDG;
//   OC = false : E only (NS/2 words per diagonal); the pair is spliced from E[u] and the neighbouring lane's E[u+1]
//                (SHFL + PRMT, one more halo lane).
// Measured (profiles/r02_v2_fml16_layout_ab.txt): the single copy cuts the kernel's DRAM traffic by a third (17.9 -> 11.6 GB
// per 20 k loci) and wins 6 % where the strips' working set overflows L2 (stride-608 tiles: long loci, L = 500), but the
// extra SHFL in the dependent chain costs 4.5 % where it already fits (stride <= 352), so the layout is a bucket property.
// One LDG + one VIADDMNMX.S16x2 covers two split terms.  Values are exact while every finite fML of the locus
// stays above MF16M_GUARD (fML16 INF = 16383: INF+INF and INF+finite stay above MF16M_VALID and
// never wrap); otherwise the locus is flagged for the 32-bit kernel.
// ---- OC = true: the round-1 functions, kept verbatim (the templated form below compiles to a 5 % slower stride-352 kernel
// for reasons that are ptxas' own: same-box A/B 139.6 vs 132.3 ms on 40 k arabidopsis loci) ----
template <class StrideT>
__device__ __forceinline__ void dev_store_fml16(unsigned int *Mp, StrideT NS, int d, int i, int m, int *sFlag)
{
    const int m16 = (m >= MF_INF / 2) ? MF16M_INF : max(m, -32768);
    if (m < MF16M_GUARD) *sFlag = 1;
    unsigned short *row = (unsigned short *)(Mp + (d - 4) * NS);
    // halfword index inside E: i-1; inside O (after NS/2 words = NS halfwords): i-2
    row[i - 1] = (unsigned short)m16;
    if (i >= 2) row[NS + i - 2] = (unsigned short)m16;
}

// non-systolic strips of the two-copy layout (MIRFOLD_OPTS bit 2; kept because removing this cold path costs the
// stride-352 kernel 3 % -- code placement, measured same-box)
template <int NT, class StrideT>
__device__ __forceinline__ void dev_phase_a16(const unsigned int *Mp, int *rD, StrideT NS, int n, int d, int d1,
                                              int tid, bool prefetch)
{
    const int emax = d1 - 5;  // e ranges 4..emax for the widest diagonal of the strip
    if (emax < 4) return;
    const int H = NS / 2;
    const int R = n - d, RP = (R + 1) >> 1;
    const int Rpad = (RP + 31) & ~31;
    int nparts = NT / Rpad;
    nparts = max(1, min(nparts, 8));
    const int span = emax - 3;
    const int per = ((span + nparts - 1) / nparts + 1) & ~1;      // even: every part starts at an even e
    for (int base = 0; base < Rpad * nparts; base += NT) {
        const int idx = base + tid;
        const int part = idx / Rpad, t = idx - part * Rpad, i = 2 * t + 1;   // rows i (lo half) and i+1 (hi half)
        if (part >= nparts || i > R) continue;
        const int e0 = 4 + part * per, e1 = min(emax, e0 + per - 1);
        if (e0 > e1) continue;
        const int ns = min(d1 - d, n - d - i) + 1;                  // valid strip diagonals for row i
        const int nsh = min(d1 - d, n - d - i - 1) + 1;             // ... and for row i+1 (0 if it has no cell on diagonal d)
        const unsigned int *pa = Mp + (e0 - 4) * NS + t;                      // E[t] of diagonal e
        const unsigned int *pb = Mp + (d - 5 - e0) * NS + H + t + (e0 >> 1);  // e even: O[t + e/2] of diagonal d-1-e   (+ s*NS for d+s)
        unsigned int acc[5] = {MF16M_INF2, MF16M_INF2, MF16M_INF2, MF16M_INF2, MF16M_INF2};
        const int emain = min(e1, d - 5);
        int e = e0;
        for (; e + 3 <= emain; e += 4) {
            if (prefetch && e + 11 <= emain) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    dev_prefetch_l1(pa + (8 + k) * NS);
                    dev_prefetch_l1(pb - (8 + k) * NS - (k & 1) * H + 4 + ((k + 1) >> 1));
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const unsigned int av = pa[k * NS];
                // step k: diagonal -k; odd k reads E (H words back) at word t + (e+k+1)/2
                const int bo = -k * NS - (k & 1) * H + ((k + 1) >> 1);
#pragma unroll
                for (int s = 0; s < 5; s++)
                    if (s < ns) acc[s] = __viaddmin_s16x2(av, pb[s * NS + bo], acc[s]);
            }
            pa += 4 * NS;
            pb += -4 * NS + 2;
        }
        for (; e <= e1; e++) {   // remainder and tail: diagonal d+s accepts e <= d+s-5
            const unsigned int av = Mp[(e - 4) * NS + t];
            const unsigned int *qb = Mp + (d - 5 - e) * NS + ((e & 1) ? t + ((e + 1) >> 1) : H + t + (e >> 1));
#pragma unroll
            for (int s = 0; s < 5; s++)
                if (s < ns && e <= d + s - 5) acc[s] = __viaddmin_s16x2(av, qb[s * NS], acc[s]);
        }
#pragma unroll
        for (int s = 0; s < 5; s++) {
            const int lo = (int)(short)(acc[s] & 0xffffu), hi = (int)acc[s] >> 16;
            int *dst = &rD[((d + s) & (MF_RING_DML - 1)) * NS + (i - 1)];
            if (s < ns && lo < MF16M_VALID) {
                if (nparts == 1) dst[0] = lo;
                else atomicMin(dst, lo);
            }
            if (s < nsh && hi < MF16M_VALID) {
                if (nparts == 1) dst[1] = hi;
                else atomicMin(dst + 1, hi);
            }
        }
    }
}

// Systolic variant of dev_phase_a16 (the default).  The right operand of thread t at split e and strip
// diagonal s is the word the next row pair t+1 used two splits earlier for diagonal s-2, so only
// s = 0 is loaded; s = 1 is spliced from the previous step's s = 0 words of this lane and lane+1, and
// s = 2..4 arrive by SHFL.DOWN from lane+1's registers of step e-2 (X*/Y* hold the words of the last
// even/odd step).  2 LDG + 4 SHFL + 1 PRMT + 5 VIADDMNMX.S16x2 per step instead of 6 LDG + 5:
// the strips are bound by L1-miss traffic, not by issue slots.  A warp covers 30 row pairs; lanes 30,
// 31 are the halo that feeds lanes 28, 29 and are recomputed by the next tile.
template <int NT, class StrideT>
__device__ __forceinline__ void dev_phase_a16_sys(const unsigned int *Mp, int *rD, StrideT NS, int n, int d, int d1, int tid)
{
    const int emax = d1 - 5;  // e ranges 4..emax for the widest diagonal of the strip
    if (emax < 4) return;
    constexpr int NW = NT / 32, TW = 30;
    const int H = NS / 2;
    const int R = n - d, RP = (R + 1) >> 1;
    const int ntiles = (RP + TW - 1) / TW;
    const int nparts = max(1, min(NW / ntiles, 8));
    const int span = emax - 3;
    const int per = ((span + nparts - 1) / nparts + 1) & ~1;      // even: every part starts at an even e
    const int lane = tid & 31, wid = tid >> 5;
    for (int unit = wid; unit < ntiles * nparts; unit += NW) {
        const int part = unit / ntiles, tile = unit - part * ntiles;
        const int e0 = 4 + part * per, e1 = min(emax, e0 + per - 1);
        if (e0 > e1) continue;
        const int t = tile * TW + lane, i = 2 * t + 1;              // rows i (lo half) and i+1 (hi half)
        const int ns = min(d1 - d, n - d - i) + 1;                  // valid strip diagonals for row i (<= 0: none)
        const int nsh = min(d1 - d, n - d - i - 1) + 1;             // ... and for row i+1
        const unsigned int *pa = Mp + (e0 - 4) * NS + t;                      // E[t] of diagonal e
        const unsigned int *pb = Mp + (d - 5 - e0) * NS + H + t + (e0 >> 1);  // e even: O[t + e/2] of diagonal d-1-e   (+ s*NS for d+s)
        unsigned int a0 = MF16M_INF2, a1 = MF16M_INF2, a2 = MF16M_INF2, a3 = MF16M_INF2, a4 = MF16M_INF2;
        const int emain = min(e1, d - 5);
        unsigned int X0 = 0, X1 = 0, X2 = 0, Y0 = 0, Y1 = 0, Y2 = 0;
        int e = e0;
        // every term of the main range is valid for every strip diagonal the row has, and halves / diagonals a
        // row does not have are simply not stored, so the accumulation is unconditional.
        // prologue: two steps with all five words loaded
        if (e <= emain) {
            const unsigned int av = pa[0];
            X0 = pb[0]; X1 = pb[NS]; X2 = pb[2 * NS];
            a0 = __viaddmin_s16x2(av, X0, a0); a1 = __viaddmin_s16x2(av, X1, a1); a2 = __viaddmin_s16x2(av, X2, a2);
            a3 = __viaddmin_s16x2(av, pb[3 * NS], a3); a4 = __viaddmin_s16x2(av, pb[4 * NS], a4);
            e++;
        }
        if (e <= emain) {
            const unsigned int av = pa[NS];
            const unsigned int *q = pb - NS - H + 1;
            Y0 = q[0]; Y1 = q[NS]; Y2 = q[2 * NS];
            a0 = __viaddmin_s16x2(av, Y0, a0); a1 = __viaddmin_s16x2(av, Y1, a1); a2 = __viaddmin_s16x2(av, Y2, a2);
            a3 = __viaddmin_s16x2(av, q[3 * NS], a3); a4 = __viaddmin_s16x2(av, q[4 * NS], a4);
            e++;
        }
        pa += 2 * NS;
        pb += -2 * NS + 1;
#define MF_SYS_COMPUTE(V0, V1, V2, P0, AV, N0)                                                     \
    {                                                                                              \
        const unsigned int av = (AV), n0 = (N0);                                                   \
        /* s = 1: rows (i, i+1) need the previous step's s = 0 words of rows (i+1, i+2) */         \
        const unsigned int n1 = __byte_perm(P0, __shfl_down_sync(0xffffffffu, P0, 1), 0x5432);     \
        const unsigned int b2 = __shfl_down_sync(0xffffffffu, V0, 1);                              \
        const unsigned int b3 = __shfl_down_sync(0xffffffffu, V1, 1);                              \
        const unsigned int b4 = __shfl_down_sync(0xffffffffu, V2, 1);                              \
        a0 = __viaddmin_s16x2(av, n0, a0); a1 = __viaddmin_s16x2(av, n1, a1);                      \
        a2 = __viaddmin_s16x2(av, b2, a2); a3 = __viaddmin_s16x2(av, b3, a3);                      \
        a4 = __viaddmin_s16x2(av, b4, a4);                                                         \
        V0 = n0; V1 = n1; V2 = b2;                                                                 \
    }
#define MF_SYS_STEP(V0, V1, V2, P0, AOFF, BOFF) MF_SYS_COMPUTE(V0, V1, V2, P0, pa[AOFF], pb[BOFF])
#ifndef MF_SYS_UNROLL
#define MF_SYS_UNROLL 2
#endif
#define MF_PRAGMA_(x) _Pragma(#x)
#define MF_UNROLL_(n) MF_PRAGMA_(unroll n)
        MF_UNROLL_(MF_SYS_UNROLL)
        for (; e + 1 <= emain; e += 2) {
            MF_SYS_STEP(X0, X1, X2, Y0, 0, 0)
            MF_SYS_STEP(Y0, Y1, Y2, X0, NS, -NS - H + 1)
            pa += 2 * NS;
            pb += -2 * NS + 1;
        }
        if (e <= emain) {
            MF_SYS_STEP(X0, X1, X2, Y0, 0, 0)
            e++;
        }
#undef MF_SYS_STEP
#undef MF_SYS_COMPUTE
        for (; e <= e1; e++) {   // tail: diagonal d+s accepts e <= d+s-5 (s >= 1 only), words loaded directly
            const unsigned int av = Mp[(e - 4) * NS + t];
            const unsigned int *qb = Mp + (d - 5 - e) * NS + ((e & 1) ? t + ((e + 1) >> 1) : H + t + (e >> 1));
            if (e <= d + 1 - 5) a1 = __viaddmin_s16x2(av, qb[NS], a1);
            if (e <= d + 2 - 5) a2 = __viaddmin_s16x2(av, qb[2 * NS], a2);
            if (e <= d + 3 - 5) a3 = __viaddmin_s16x2(av, qb[3 * NS], a3);
            a4 = __viaddmin_s16x2(av, qb[4 * NS], a4);
        }
        if (lane < TW) {
            const unsigned int acc[5] = {a0, a1, a2, a3, a4};
#pragma unroll
            for (int s = 0; s < 5; s++) {
                const int lo = (int)(short)(acc[s] & 0xffffu), hi = (int)acc[s] >> 16;
                int *dst = &rD[((d + s) & (MF_RING_DML - 1)) * NS + (i - 1)];
                if (nparts == 1) {   // the only writer of these cells: no preset needed (see the ring reset in k_fill_s16)
                    if (s < ns) dst[0] = lo < MF16M_VALID ? lo : MF_INF;
                    if (s < nsh) dst[1] = hi < MF16M_VALID ? hi : MF_INF;
                } else {
                    if (s < ns && lo < MF16M_VALID) atomicMin(dst, lo);
                    if (s < nsh && hi < MF16M_VALID) atomicMin(dst + 1, hi);
                }
            }
        }
    }
}


// ---- OC = false: single copy, spliced right operands ----
template <bool OC, class StrideT>
__device__ __forceinline__ void dev_store_fml16x(unsigned int *Mp, StrideT NS, int d, int i, int m, int *sFlag)
{
    const int m16 = (m >= MF_INF / 2) ? MF16M_INF : max(m, -32768);
    if (m < MF16M_GUARD) *sFlag = 1;
    unsigned short *row = (unsigned short *)(Mp + (d - 4) * (OC ? NS : NS / 2));
    // halfword index inside E: i-1; inside O (after NS/2 words = NS halfwords): i-2
    row[i - 1] = (unsigned short)m16;
    if (OC && i >= 2) row[NS + i - 2] = (unsigned short)m16;
}

// Systolic strips.  The right operand of thread t at split e and strip
// diagonal s is the word the next row pair t+1 used two splits earlier for diagonal s-2, so only
// s = 0 is loaded; s = 1 is spliced from the previous step's s = 0 words of this lane and lane+1, and
// s = 2..4 arrive by SHFL.DOWN from lane+1's registers of step e-2 (X*/Y* hold the words of the last
// even/odd step).  2 LDG + 4 SHFL + 1 PRMT + 5 VIADDMNMX.S16x2 per step instead of 6 LDG + 5:
// the strips are bound by L1-miss traffic, not by issue slots.  A warp covers 30 (OC) or 29 row pairs; the
// remaining lanes are the halo that feeds the last ones and are recomputed by the next tile.
template <int NT, bool OC, class StrideT>
__device__ __forceinline__ void dev_phase_a16_sysx(const unsigned int *Mp, int *rD, StrideT NS, int n, int d, int d1, int tid)
{
    const int emax = d1 - 5;  // e ranges 4..emax for the widest diagonal of the strip
    if (emax < 4) return;
    constexpr int NW = NT / 32, TW = OC ? 30 : 29;
    const int W = OC ? NS : NS / 2;                                  // words per diagonal
    const int OH = OC ? NS / 2 : 0;                                  // offset of the odd-aligned copy inside a diagonal
    const int R = n - d, RP = (R + 1) >> 1;
    const int ntiles = (RP + TW - 1) / TW;
    const int nparts = max(1, min(NW / ntiles, 8));
    const int span = emax - 3;
    const int per = ((span + nparts - 1) / nparts + 1) & ~1;      // even: every part starts at an even e
    const int lane = tid & 31, wid = tid >> 5;
    // rows (2u+2 | 2u+3): the stored copy, or spliced from the words u (this lane) and u+1 (lane+1)
#define MF_ODDPAIR(p_) (OC ? *(p_) : __byte_perm(*(p_), __shfl_down_sync(0xffffffffu, *(p_), 1), 0x5432))
    for (int unit = wid; unit < ntiles * nparts; unit += NW) {
        const int part = unit / ntiles, tile = unit - part * ntiles;
        const int e0 = 4 + part * per, e1 = min(emax, e0 + per - 1);
        if (e0 > e1) continue;
        const int t = tile * TW + lane, i = 2 * t + 1;              // rows i (lo half) and i+1 (hi half)
        const int ns = min(d1 - d, n - d - i) + 1;                  // valid strip diagonals for row i (<= 0: none)
        const int nsh = min(d1 - d, n - d - i - 1) + 1;             // ... and for row i+1
        const unsigned int *pa = Mp + (e0 - 4) * W + t;                        // left: E[t] of diagonal e
        const unsigned int *pb = Mp + (d - 5 - e0) * W + OH + t + (e0 >> 1);   // right, e even: pair u = t + e/2 of diagonal d-1-e   (+ s*W for d+s)
        unsigned int a0 = MF16M_INF2, a1 = MF16M_INF2, a2 = MF16M_INF2, a3 = MF16M_INF2, a4 = MF16M_INF2;
        const int emain = min(e1, d - 5);
        unsigned int X0 = 0, X1 = 0, X2 = 0, Y0 = 0, Y1 = 0, Y2 = 0;
        int e = e0;
        // every term of the main range is valid for every strip diagonal the row has, and halves / diagonals a
        // row does not have are simply not stored, so the accumulation is unconditional.
        // prologue: two steps with all five words loaded
        if (e <= emain) {
            const unsigned int av = pa[0];
            X0 = MF_ODDPAIR(pb); X1 = MF_ODDPAIR(pb + W); X2 = MF_ODDPAIR(pb + 2 * W);
            const unsigned int x3 = MF_ODDPAIR(pb + 3 * W), x4 = MF_ODDPAIR(pb + 4 * W);
            a0 = __viaddmin_s16x2(av, X0, a0); a1 = __viaddmin_s16x2(av, X1, a1); a2 = __viaddmin_s16x2(av, X2, a2);
            a3 = __viaddmin_s16x2(av, x3, a3); a4 = __viaddmin_s16x2(av, x4, a4);
            e++;
        }
        if (e <= emain) {
            const unsigned int av = pa[W];
            const unsigned int *q = pb - W - OH + 1;
            Y0 = q[0]; Y1 = q[W]; Y2 = q[2 * W];
            a0 = __viaddmin_s16x2(av, Y0, a0); a1 = __viaddmin_s16x2(av, Y1, a1); a2 = __viaddmin_s16x2(av, Y2, a2);
            a3 = __viaddmin_s16x2(av, q[3 * W], a3); a4 = __viaddmin_s16x2(av, q[4 * W], a4);
            e++;
        }
        pa += 2 * W;
        pb += -2 * W + 1;
#define MF_SYS_COMPUTE(V0, V1, V2, P0, AV, N0)                                                     \
    {                                                                                              \
        const unsigned int av = (AV), n0 = (N0);                                                   \
        /* s = 1: rows (i, i+1) need the previous step's s = 0 words of rows (i+1, i+2) */         \
        const unsigned int n1 = __byte_perm(P0, __shfl_down_sync(0xffffffffu, P0, 1), 0x5432);     \
        const unsigned int b2 = __shfl_down_sync(0xffffffffu, V0, 1);                              \
        const unsigned int b3 = __shfl_down_sync(0xffffffffu, V1, 1);                              \
        const unsigned int b4 = __shfl_down_sync(0xffffffffu, V2, 1);                              \
        a0 = __viaddmin_s16x2(av, n0, a0); a1 = __viaddmin_s16x2(av, n1, a1);                      \
        a2 = __viaddmin_s16x2(av, b2, a2); a3 = __viaddmin_s16x2(av, b3, a3);                      \
        a4 = __viaddmin_s16x2(av, b4, a4);                                                         \
        V0 = n0; V1 = n1; V2 = b2;                                                                 \
    }
#ifndef MF_SYS_UNROLL
#define MF_SYS_UNROLL 2
#endif
#define MF_PRAGMA_(x) _Pragma(#x)
#define MF_UNROLL_(n) MF_PRAGMA_(unroll n)
        MF_UNROLL_(MF_SYS_UNROLL)
        for (; e + 1 <= emain; e += 2) {
            MF_SYS_COMPUTE(X0, X1, X2, Y0, pa[0], MF_ODDPAIR(pb))          // even split
            MF_SYS_COMPUTE(Y0, Y1, Y2, X0, pa[W], pb[-W - OH + 1])         // odd split
            pa += 2 * W;
            pb += -2 * W + 1;
        }
        if (e <= emain) {
            MF_SYS_COMPUTE(X0, X1, X2, Y0, pa[0], MF_ODDPAIR(pb))
            e++;
        }
#undef MF_SYS_COMPUTE
        for (; e <= e1; e++) {   // tail: diagonal d+s accepts e <= d+s-5 (s >= 1 only), words loaded directly
            const unsigned int av = Mp[(e - 4) * W + t];
            const unsigned int *qe = Mp + (d - 5 - e) * W + t + ((e + 1) >> 1);   // E[t + ceil(e/2)] of diagonal d-1-e
            // right operand of strip diagonal s_: E word (odd e), else the odd-aligned pair (stored copy or two E words)
            auto right = [&](int s_) {
                if (e & 1) return qe[s_ * W];
                return OC ? qe[s_ * W + OH] : __byte_perm(qe[s_ * W], qe[s_ * W + 1], 0x5432);
            };
            if (e <= d + 1 - 5) a1 = __viaddmin_s16x2(av, right(1), a1);
            if (e <= d + 2 - 5) a2 = __viaddmin_s16x2(av, right(2), a2);
            if (e <= d + 3 - 5) a3 = __viaddmin_s16x2(av, right(3), a3);
            a4 = __viaddmin_s16x2(av, right(4), a4);
        }
#undef MF_ODDPAIR
        if (lane < TW) {
            const unsigned int acc[5] = {a0, a1, a2, a3, a4};
#pragma unroll
            for (int s = 0; s < 5; s++) {
                const int lo = (int)(short)(acc[s] & 0xffffu), hi = (int)acc[s] >> 16;
                int *dst = &rD[((d + s) & (MF_RING_DML - 1)) * NS + (i - 1)];
                if (nparts == 1) {   // the only writer of these cells: no preset needed (see the ring reset in k_fill_s16)
                    if (s < ns) dst[0] = lo < MF16M_VALID ? lo : MF_INF;
                    if (s < nsh) dst[1] = hi < MF16M_VALID ? hi : MF_INF;
                } else {
                    if (s < ns && lo < MF16M_VALID) atomicMin(dst, lo);
                    if (s < nsh && hi < MF16M_VALID) atomicMin(dst + 1, hi);
                }
            }
        }
    }
}


template <bool OC, class StrideT>
__device__ __forceinline__ void dev_store_fml16_sel(unsigned int *Mp, StrideT NS, int d, int i, int m, int *sFlag)
{
    if (OC) dev_store_fml16(Mp, NS, d, i, m, sFlag);
    else dev_store_fml16x<false>(Mp, NS, d, i, m, sFlag);
}
template <int NT, bool OC, class StrideT>
__device__ __forceinline__ void dev_phase_a16_sel(const unsigned int *Mp, int *rD, StrideT NS, int n, int d, int d1, int tid)
{
    if (OC) dev_phase_a16_sys<NT>(Mp, rD, NS, n, d, d1, tid);
    else dev_phase_a16_sysx<NT, false>(Mp, rD, NS, n, d, d1, tid);
}

// ------------------------------------------------------------------------------------ K2 (shared-memory rings)
// Ring geometry: 33 slots hold Cm of diagonals d-32..d, slot 33 is all-INF.  Rows are RS = NS+32
// words; diagonal d' is stored rotated by sk(d') = (11*d') & 31 words, which makes the bank of
// Cm(p,q) for the loop (u,v) of a cell equal to (u - 11*(u+v) + const) mod 32.  With that skew the
// 431 generic (u,v) terms split into 32 bank classes of <= 14 terms each: lane l owns class l and
// the warp needs 14 conflict-free LDS per typed cell (DevParams::gen_us / gen_c).
#define MF_SLOTS 33
template <int NS>
struct FillSmem {
    static constexpr int RS = NS + 32;
    static constexpr int cm_ints = (MF_SLOTS + 1) * RS;
    static constexpr int dl_bytes = MF_SLOTS * RS;
    static constexpr size_t bytes = (size_t)cm_ints * 4 + dl_bytes + 2 * (NS + 8) + 2 * 2 * NS + 64 + 16;
};
__device__ __forceinline__ int dev_skew(int dp) { return (MF_SKEW_A * dp) & 31; }

template <int NS, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_fill_smem(FillLaunch a)
{
    constexpr int RS = FillSmem<NS>::RS;
    constexpr int NW = NT / 32, NWM = NW / 4, NWC = NW - NWM;       // fML/list warps, c warps
    constexpr int CT = NWC * 32, MT = NWM * 32;
    constexpr int INFOFF = MF_SLOTS * RS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int *sCm = (int *)smem_raw;                                            // [34][RS]
    unsigned char *sDl = (unsigned char *)(sCm + FillSmem<NS>::cm_ints);   // [33][RS]  AU - mismatchI + 70
    unsigned char *sS = sDl + FillSmem<NS>::dl_bytes;                      // [NS+8]
    unsigned char *sS1 = sS + NS + 8;
    unsigned short *sList = (unsigned short *)(sS1 + NS + 8);              // [2][NS]
    unsigned char *sPair = (unsigned char *)(sList + 2 * NS);              // [64]
    __shared__ int sCount[3];

    if (a.flags && !a.flags[blockIdx.x]) return;   // only loci the 16-bit kernel flagged
    const LocusDesc L = a.loci[blockIdx.x];
    const int n = L.n, Ls = L.Ls, dmax = L.dmax;
    const DevParams *__restrict__ P = a.P;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // no traceback hint from this kernel: every cell says "scan the two-loop candidates"
    for (int k = tid; k < (dmax - 3) * (NS / 4); k += NT) ((unsigned int *)(a.Ib + L.band_off))[k] = 0x01010101u;

    for (int k = tid; k < NS + 8; k += NT) {
        const unsigned char b = (k < n + 3) ? a.codes[L.seq_off + k] : 0;
        sS[k] = b & 7;
        sS1[k] = b >> 4;
    }
    for (int k = tid; k < RS; k += NT) sCm[INFOFF + k] = MF_INF;
    if (tid < 64) sPair[tid] = P->pair[tid];
    if (tid < 3) sCount[tid] = 0;

    int *Cb = a.C + L.band_off;
    int *Mb = a.M + L.band_off;
    int *rD = a.ring + L.ring_off;   // [MF_RING_DML][NS]
    for (int k = tid; k < MF_RING_DML * NS; k += NT) rD[k] = MF_INF;
    __syncthreads();

    // per-lane constants of the generic pass
    int cst[MF_GEN_ITERS];
#pragma unroll
    for (int it = 0; it < MF_GEN_ITERS; it++) {
        const int c = P->gen_c[it][lane];
        cst[it] = (c < MF_INF) ? c : 0;
    }
    const int nlB = lane + 2;                                          // bulge size handled by this lane
    const int cstB = (nlB <= 30) ? P->bulge[nlB] - 70 : 0;

    // typed list of the first diagonal -> sList[0], sCount[4 % 3]
    if (dmax >= 4) {
        for (int i = tid + 1; i <= n - 4; i += NT) {
            const int t = (4 < Ls) ? sPair[sS[i] * 8 + sS[i + 4]] : 0;
            if (t) sList[atomicAdd(&sCount[1], 1)] = (unsigned short)i;
        }
    }
    __syncthreads();

    // iteration `it`: c warps fill c on diagonal it; fML warps fill fML on diagonal it-1 (which only
    // the next iteration and later DML strips read) and build the typed list of diagonal it+1.
    for (int it = 4; it <= dmax + 1; it++) {
        if (it >= 5 && (it - 5) % 5 == 0 && it - 1 <= dmax) {
            dev_phase_a<NT>(Mb, rD, NS, n, it - 1, min(it + 3, dmax), tid, !(a.opts & 1));   // DML strip [it-1, it+3]
            __syncthreads();
        }
        if (wid < NWC) {
            const int d = it;
            if (d <= dmax) {
                const int ntyped = sCount[d % 3];
                const unsigned short *list = sList + (d & 1) * NS;
                const int K = min(30, d - 6);
                const int bslot = (d - 2) % MF_SLOTS;
                const int drow = (d % MF_SLOTS) * RS + dev_skew(d);
                // INF for the untyped cells of this diagonal (ring + band)
                for (int i = tid + 1; i <= n - d; i += CT) {
                    const int t = (d < Ls) ? sPair[sS[i] * 8 + sS[i + d]] : 0;
                    if (!t) { sCm[drow + i - 1] = MF_INF; Cb[(d - 4) * NS + i - 1] = MF_INF; }
                }
                int off[MF_GEN_ITERS];
#pragma unroll
                for (int k = 0; k < MF_GEN_ITERS; k++) {
                    const int g = P->gen_us[k][lane];                  // u | s << 8 | valid << 16
                    const int u = g & 0xff, s = (g >> 8) & 0xff;
                    int slot = bslot - s;
                    if (slot < 0) slot += MF_SLOTS;
                    off[k] = ((g >> 16) && s <= K) ? slot * RS + dev_skew(d - 2 - s) + u : INFOFF;
                }
                int offB1, offB2, offD1, offD2;
                {
                    int slot = bslot - nlB;
                    if (slot < 0) slot += MF_SLOTS;
                    const bool ok = nlB <= K;                                   // K <= 30
                    const int row = slot * RS + dev_skew(d - 2 - nlB);
                    offB1 = ok ? row + nlB : INFOFF;                           // (u=nl, v=0): p = i+1+nl
                    offB2 = ok ? row : INFOFF;                                 // (u=0, v=nl): p = i+1
                    offD1 = ok ? row + nlB : 0;
                    offD2 = ok ? row : 0;
                }
                const int per = (ntyped + NWC - 1) / NWC;
                const int cend = min(ntyped, wid * per + per);
                for (int c0 = wid * per; c0 < cend; c0 += 32) {
                    const int cnt = min(32, cend - c0);
                    int myG = MF_INF, myB = MF_INF;
                    for (int k = 0; k < cnt; k++) {
                        const int i = list[c0 + k];
                        const int *w = sCm + i;
                        int g = MF_INF;
#pragma unroll
                        for (int q = 0; q < MF_GEN_ITERS; q++) g = min(g, w[off[q]] + cst[q]);
                        int bb = min(w[offB1] + (int)sDl[offD1 + i], w[offB2] + (int)sDl[offD2 + i]) + cstB;
                        g = warp_min(g);
                        bb = warp_min(bb);
                        if (lane == k) { myG = g; myB = bb; }
                    }
                    if (lane < cnt) {
                        const int i = list[c0 + lane], j = i + d;
                        const int t = sPair[sS[i] * 8 + sS[j]];
                        const int si1 = sS1[i + 1], sj1 = sS1[j - 1];
                        int best = myG + P->mismatchI[(t * 5 + si1) * 5 + sj1];
                        best = min(best, myB + (t > 2 ? P->TerminalAU : 0));
                        best = min(best, dev_cell_tail(P, sS, sS1, sPair, Cb, rD, NS, i, d, t, si1, sj1, K));
                        const int tt = P->rtype[t];
                        const int mm = P->mismatchI[(tt * 5 + sS1[j + 1]) * 5 + sS1[i - 1]];
                        Cb[(d - 4) * NS + i - 1] = best;
                        sCm[drow + i - 1] = best + mm;
                        sDl[drow + i - 1] = (unsigned char)((tt > 2 ? P->TerminalAU : 0) - mm + 70);
                    }
                }
            }
        } else {
            const int mt = tid - CT;
            const int dm = it - 1;
            if (dm >= 4) {
                for (int i = mt + 1; i <= n - dm; i += MT)
                    Mb[(dm - 4) * NS + i - 1] = dev_fml(P, sS, sS1, sPair, Cb, Mb, rD, NS, i, dm, Ls);
            }
            const int dn = it + 1;
            if (mt == 0) sCount[(it + 2) % 3] = 0;
            if (dn <= dmax) {
                unsigned short *list = sList + (dn & 1) * NS;
                for (int i = mt + 1; i <= n - dn; i += MT) {
                    const int t = (dn < Ls) ? sPair[sS[i] * 8 + sS[i + dn]] : 0;
                    if (t) list[atomicAdd(&sCount[dn % 3], 1)] = (unsigned short)i;
                }
            }
            if ((it + 1 - 5) % 5 == 0 && it <= dmax) {   // next iteration runs the DML strip [it, it+4]
                for (int s = 0; s < 5; s++)
                    for (int i = mt; i < n; i += MT) rD[((it + s) & (MF_RING_DML - 1)) * NS + i] = MF_INF;
            }
        }
        __syncthreads();
    }
}


// ------------------------------------------------------------------------------------ K2 (narrow: 16-bit pair ring)
// Same wavefront as k_fill_smem, but the interior-loop window is kept as 16-bit values with two
// adjacent diagonals per 32-bit word:  sG = c + mismatchI (generic loops), sB = c + AU (bulges).
// Pair pp = d'>>1 lives in slot pp % 17, rotated by (17 pp) & 31 words; lane l owns the word-terms of
// bank class l (DevParams::s16_*), so a typed cell costs 10 conflict-free LDS + 10 VIADDMNMX.S16x2 per
// lane (8 generic, 2 bulge), one packed combine and one redux.  Exact while c > MF16_GUARD; otherwise
// the locus is flagged for the 32-bit kernel.
#ifndef MF16_NWM_DELTA
#define MF16_NWM_DELTA 0
#endif
#ifndef MF16_NWM
#define MF16_NWM(NT) (((NT) / 32 * 3 + 4) / 8 - MF16_NWM_DELTA)   /* fML/list warps of the narrow kernel: 6 of 16, 4 of 10, 3 of 8 */
#endif
template <int NS>
struct Fill16Smem {
    static constexpr int RS = NS + 32;
    static constexpr int ring_words = (MF16_NPS + 1) * RS;   // + one all-INF row
    static constexpr int sched_words = 2 * MF16_NQ * 32 * 2 + 2 * MF16_NMK * 32;   // sOff, sCst (both parities), sMk
    static constexpr size_t bytes = (size_t)2 * ring_words * 4 + (size_t)5 * NS * 4 + 200 * 4 + (size_t)sched_words * 4 +
                                    2 * (NS + 8) + 64 + 16;
};

// Byte offset (from the start of sG) of the word-term `td` of lane `lane` for a cell on diagonal d.
// A lane without a term in this iteration reads the all-INF row at the bank its own class would use,
// which no other lane touches in the same instruction.
// Word offset of pair slot pp's row inside a ring: (pp % 17) * RS + ((17 pp) & 31).  The modulo is not cheap and every ring
// access of the thread-per-cell phases needs it for two or three diagonals, so the kernel keeps the values of the live pairs in
// a 32-entry shared table (entry pp & 31; one thread adds the next pair per diagonal) -- fML -20 %, word-term offsets -60 %
// instructions (profiles/r02_v6_rowtab_ab.txt).
struct RingRows {
    const int *tab;
    int RS;
    __device__ __forceinline__ int operator()(int pp) const
    {
#ifdef MF_NO_ROWTAB
        return (pp % MF16_NPS) * RS + ((MF16_SKEW * pp) & 31);
#else
        return tab[pp & 31];
#endif
    }
    static __device__ __forceinline__ int direct(int pp, int RS_) { return (pp % MF16_NPS) * RS_ + ((MF16_SKEW * pp) & 31); }
};

__device__ __forceinline__ unsigned dev_term_off16(unsigned td, int lane, int d, RingRows rr, int RS, int RW)
{
    const int ppb = (d - 2) >> 1;
    if (td >> 11) return (unsigned)(MF16_NPS * RS + ((lane + MF16_SKEW * ppb) & 31)) * 4u;
    const int m = td & 15, xo = (td >> 4) & 63, pp = ppb - m;
    const int row = pp < 0 ? MF16_NPS * RS : rr(pp);   // pp < 0: all-INF row (d < 34 only)
    return (unsigned)(((td >> 10) & 1) * RW + row + xo) * 4u;
}
__device__ __forceinline__ void dev_ring16_put(unsigned int *ring, RingRows rr, int d, int x, int v)
{
    unsigned short *w = (unsigned short *)(ring + rr(d >> 1) + x);
    w[d & 1] = (unsigned short)v;
}


// 16-bit ring read: value of diagonal dd at row index x (= p-1)
__device__ __forceinline__ int dev_ring16_get(const unsigned int *ring, RingRows rr, int dd, int x)
{
    const short *w = (const short *)(ring + rr(dd >> 1) + x);
    return w[dd & 1];
}

// The seven table-driven two-loops + hairpin + d1 multiloop closing of a typed cell, narrow kernel:
// branch-free (all lookups of the seven loops are independent and overlap) and with c(p,q) read from
// the shared-memory bulge ring (c + AU) instead of the band.
template <class StrideT>
__device__ __forceinline__ int dev_cell_tail16(const DevParams *__restrict__ P, const unsigned char *sS,
                                               const unsigned char *sS1, const unsigned char *sPair,
                                               const unsigned int *sB, RingRows RS, const int *rD, StrideT NS, int i,
                                               int d, int t, int si1, int sj1, int K, int &two_loop_min)
{
    const int j = i + d;
    const int AUp = P->TerminalAU;
    int best = MF_INF;
#pragma unroll
    for (int m = 0; m < 7; m++) {
        const int u = (m == 1 || m == 3 || m == 4) ? 1 : (m >= 5 ? 2 : 0);
        const int v = (m == 2 || m == 3 || m == 5) ? 1 : ((m == 4 || m == 6) ? 2 : 0);
        // m: 0 (0,0)  1 (1,0)  2 (0,1)  3 (1,1)  4 (1,2)  5 (2,1)  6 (2,2)
        const bool ok = (u + v <= K);
        const int p = ok ? i + 1 + u : i + 1, q = ok ? j - 1 - v : j - 1;   // clamped: always a legal address
        const int t2 = sPair[sS[p] * 8 + sS[q]];
        const int r2 = dev_rtype(t2);
        const int c2 = dev_ring16_get(sB, RS, ok ? d - 2 - u - v : d - 2, p - 1) - (t2 > 2 ? AUp : 0);
        const int sp1 = sS1[p - 1], sq1 = sS1[q + 1];
        int e;
        if (m == 0) e = P->stack[t * 8 + r2];
        else if (m == 1 || m == 2) e = P->bulge[1] + P->stack[t * 8 + r2];
        else if (m == 3) e = P->int11[((t * 8 + r2) * 5 + si1) * 5 + sj1];
        else if (m == 4) e = P->int21[(((t * 8 + r2) * 5 + si1) * 5 + sq1) * 5 + sj1];           // n1 = 1, n2 = 2
        else if (m == 5) e = P->int21[(((r2 * 8 + t) * 5 + sq1) * 5 + si1) * 5 + sp1];           // n1 = 2, n2 = 1
        else e = P->int22[((((t * 8 + r2) * 5 + si1) * 5 + sp1) * 5 + sq1) * 5 + sj1];
        if (ok && t2) best = min(best, e + c2);
    }
    two_loop_min = best;
    best = min(best, dev_hairpin(P, sS, sS1, i, j, t));
    const int tt = dev_rtype(t);
    const int d3 = P->dangle3[tt * 5 + si1], d5 = P->dangle5[tt * 5 + sj1];
    int dec = MF_INF;
    if (d - 2 >= 4) dec = rD[((d - 2) & (MF_RING_DML - 1)) * NS + i];                          // DML(i+1,j-1)
    if (d - 3 >= 4) {
        dec = min(dec, rD[((d - 3) & (MF_RING_DML - 1)) * NS + i + 1] + d3);                   // DML(i+2,j-1)
        dec = min(dec, rD[((d - 3) & (MF_RING_DML - 1)) * NS + i] + d5);                       // DML(i+1,j-2)
    }
    if (d - 4 >= 4) dec = min(dec, rD[((d - 4) & (MF_RING_DML - 1)) * NS + i + 1] + d3 + d5);  // DML(i+2,j-2)
    return min(best, P->MLclosing + P->MLintern[t] + dec);
}

// fML(i,j) for the narrow kernel: c of the three newest diagonals comes from the shared-memory bulge
// ring (c + AU, exact inside the guarded range) and fML of diagonal d-1 from a shared row buffer, so
// the only global read is DML(i,j).
template <class StrideT>
__device__ __forceinline__ int dev_fml16(const DevParams *__restrict__ P, const unsigned char *sS, const unsigned char *sS1,
                                         const unsigned char *sPair, const unsigned int *sB, RingRows RS, const int *Mprev,
                                         const int *rD, StrideT NS, int i, int d, int Ls)
{
    const int j = i + d;
    const int AUp = P->TerminalAU;
    const int t = (d < Ls) ? sPair[sS[i] * 8 + sS[j]] : 0;
    int m = MF_INF;
    if (d - 1 >= 4) {
        m = min(Mprev[i], Mprev[i - 1]);                            // fML(i+1,j), fML(i,j-1)
        const int ta = sPair[sS[i + 1] * 8 + sS[j]];                // (i+1, j)
        if (ta) m = min(m, dev_ring16_get(sB, RS, d - 1, i) - (ta > 2 ? AUp : 0) + P->dangle5[ta * 5 + sS1[i]] + P->MLintern[ta]);
        const int tb = sPair[sS[i] * 8 + sS[j - 1]];                // (i, j-1)
        if (tb) m = min(m, dev_ring16_get(sB, RS, d - 1, i - 1) - (tb > 2 ? AUp : 0) + P->dangle3[tb * 5 + sS1[j]] + P->MLintern[tb]);
    }
    if (t) m = min(m, dev_ring16_get(sB, RS, d, i - 1) - (t > 2 ? AUp : 0) + P->MLintern[t]);
    if (d - 2 >= 4) {
        const int tc = sPair[sS[i + 1] * 8 + sS[j - 1]];            // (i+1, j-1)
        if (tc) m = min(m, dev_ring16_get(sB, RS, d - 2, i) - (tc > 2 ? AUp : 0) + P->dangle5[tc * 5 + sS1[i]] +
                               P->dangle3[tc * 5 + sS1[j]] + P->MLintern[tc]);
    }
    return min(m, rD[(d & (MF_RING_DML - 1)) * NS + i - 1]);
}

#ifdef MF_TIMELINE   /* per-warp cycle accounting of one CTA (debug builds only: make TIMELINE=1) */
#define TL_DECL long long tl_acc[6] = {0, 0, 0, 0, 0, 0}; long long tl_t = clock64();
/* the clock read is predicated on a shared-memory word loaded at this point, so it cannot be scheduled across a barrier */
#define TL_MARK(k) { long long t_ = tl_t; if (*(volatile int *)&sFlag != 0x7fffffff) t_ = clock64(); tl_acc[k] += t_ - tl_t; tl_t = t_; }
#define TL_DUMP if (blockIdx.x == 3 && lane == 0) printf("TL n=%d warp %2d  dml %8lld  work1 %8lld  bar1 %8lld  work2 %8lld  sync %8lld  dmlsync %8lld\n", n, wid, tl_acc[0], tl_acc[1], tl_acc[2], tl_acc[3], tl_acc[4], tl_acc[5]);
#else
#define TL_DECL
#define TL_MARK(k)
#define TL_DUMP
#endif
template <int NS, int NT, int NWM, int MINB, bool DYNW>
__global__ void __launch_bounds__(NT, MINB) k_fill_s16(FillLaunch a)
{
    constexpr int RS = Fill16Smem<NS>::RS, RW = Fill16Smem<NS>::ring_words;
    constexpr int NW = NT / 32, NWC = NW - NWM;
    constexpr int CT = NWC * 32, MT = NWM * 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned int *sG = (unsigned int *)smem_raw;              // [18][RS]
    unsigned int *sB = sG + RW;                               // [18][RS]
    unsigned int *sList = sB + RW;                            // [2][NS]  i*4 | (AU - mismatchI + bias) << 16
    int *sMy = (int *)(sList + 2 * NS);                       // [NS] interior-loop minimum of the listed cell
    int *sMrow = sMy + NS;                                    // [2][NS] fML of the last two diagonals (by parity)
    int *sMM = sMrow + 2 * NS;                                // mismatchI[200]
    unsigned int *sOff = (unsigned int *)(sMM + 200);         // [2][NQ][32] word-term byte offsets of diagonal d (by parity of d)
    unsigned int *sCst = sOff + 2 * MF16_NQ * 32;             // [2][NQ][32] packed constants (by parity)
    unsigned int *sMk = sCst + 2 * MF16_NQ * 32;              // [2][NMK][32] half-word keep masks (by parity)
    unsigned char *sS = (unsigned char *)(sMk + 2 * MF16_NMK * 32);   // [NS+8]
    unsigned char *sS1 = sS + NS + 8;
    unsigned char *sPair = sS1 + NS + 8;                      // [64]
    int *sWideM = (int *)(sPair + 64);                        // [1] DYNW buckets: some fML left the 16-bit strips' range
    __shared__ int sCount[3];
    __shared__ int sFlag;
    __shared__ int sRowP[32];                                 // ring row (words) of pair slot pp at [pp & 31]
    const RingRows rr{sRowP, RS};

    // DYNW (launched for spans >= MF_DYNW_MIN_SPAN, launch_fill_bucket): windows long enough for fML to drop below
    // MF16M_GUARD on ordinary sequence (-136 kcal/mol: about half of all 500-nt windows at GC 0.40) do not hand the unit
    // to the 32-bit kernel: from the first out-of-range fML on, the DML strips -- the only consumer of the 16-bit fML
    // copy -- read the int32 band instead, and the interior-loop rings stay 16-bit.  Only c below MF16_GUARD (-320
    // kcal/mol) still flags the unit.  The switch costs the stride-864 kernel 4 % where it never fires (L = 300: 172.4 ->
    // 180.9 ms on the long-locus law), hence two instantiations.
    const LocusDesc L = a.loci[blockIdx.x];
    const int n = L.n, Ls = L.Ls, dmax = L.dmax;
    const DevParams *__restrict__ P = a.P;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int AUp = P->TerminalAU;
    if (tid < 32) sRowP[tid] = RingRows::direct(tid, RS);

    for (int k = tid; k < NS + 8; k += NT) {
        const unsigned char b = (k < n + 3) ? a.codes[L.seq_off + k] : 0;
        sS[k] = b & 7;
        sS1[k] = b >> 4;
    }
    for (int k = tid; k < 2 * RW; k += NT) sG[k] = MF16_INF2;
    for (int k = tid; k < 200; k += NT) sMM[k] = P->mismatchI[k];
    if (tid < 64) sPair[tid] = P->pair[tid];
    if (tid < 3) sCount[tid] = 0;
    if (tid == 0) sFlag = 0;
    if (DYNW && tid == 0) *sWideM = 0;
    for (int k = tid; k < 2 * MF16_NQ * 32; k += NT) sCst[k] = (&P->s16_cst[0][0][0])[k];
    for (int k = tid; k < 2 * MF16_NMK * 32; k += NT) sMk[k] = (&P->s16_mk[0][0][0])[k];

    int *Cb = a.C + L.band_off;
    int *Mb = a.M + L.band_off;
    unsigned char *Ib = a.Ib + L.band_off;     // one byte per band cell, written for every typed cell (the only ones a traceback asks about)
    constexpr bool OC = NS <= 352;           // fML16 layout of this bucket (see dev_store_fml16)
#ifdef MF_NO_BULK_ROWS
    constexpr bool BULK = false;
#else
    // int32 fML rows leave the SM as one cp.async.bulk per diagonal from the shared row buffer instead of one STG per cell.
    // Same-box A/B (profiles/r02_v2_fml16_layout_ab.txt): neutral to slightly faster for the stride-608 bucket, 1.3 % slower
    // for stride 352 (the single issuing thread's proxy fence + wait sit on the fML warps' critical path), so by bucket.
    constexpr bool BULK = NS > 352;
#endif
    unsigned int *Mp = a.Mp + L.band_off;    // the single-copy layout uses the first half of the locus' words
    int *rD = a.ring + L.ring_off;   // [MF_RING_DML][NS]
    for (int k = tid; k < MF_RING_DML * NS; k += NT) rD[k] = MF_INF;
    __syncthreads();

    // word-term offsets of the first diagonal (the row table is ready now)
    for (int k = tid; k < MF16_NQ * 32; k += NT) sOff[k] = dev_term_off16((&P->s16_td[0][0][0])[k], k & 31, 4, rr, RS, RW);
    // typed list / untyped INF of the first diagonal
    if (dmax >= 4) {
        for (int i = tid + 1; i <= n - 4; i += NT) {
            const int t = (4 < Ls) ? sPair[sS[i] * 8 + sS[i + 4]] : 0;
            if (t) {
                const int dl = (t > 2 ? AUp : 0) - sMM[(t * 5 + sS1[i + 1]) * 5 + sS1[i + 3]] + MF16_DBIAS;
                sList[atomicAdd(&sCount[1], 1)] = (unsigned)(i * 4) | ((unsigned)dl << 16);
            } else Cb[i - 1] = MF_INF;   // ring halves already hold INF
        }
    }
    __syncthreads();

    const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem_raw);

    TL_DECL
    for (int it = 4; it <= dmax + 1; it++) {
        bool newest_row_stored = false;
        if (it >= 5 && (it - 5) % 5 == 0 && it - 1 <= dmax) {
            // DML strip [it-1, it+3]
            if (DYNW && *(volatile int *)sWideM) {   // uniform: written before the barrier that ended the last iteration
                if (BULK) {   // the int32 fML row of diagonal it-2 is still only in the shared row buffer
                    if (tid == CT && it - 2 >= 4) {
                        dev_bulk_store_row(Mb + (it - 6) * NS, sMrow + (it & 1) * NS, (unsigned)(((n - it + 2) * 4 + 15) & ~15));
                        dev_bulk_wait_all();
                    }
                    newest_row_stored = true;
                    __syncthreads();
                }
                dev_phase_a<NT, true>(Mb, rD, NS, n, it - 1, min(it + 3, dmax), tid, !(a.opts & 1));
            } else if (a.opts & 2) dev_phase_a<NT>(Mb, rD, NS, n, it - 1, min(it + 3, dmax), tid, !(a.opts & 1));
            else if (OC && (a.opts & 4)) dev_phase_a16<NT>(Mp, rD, NS, n, it - 1, min(it + 3, dmax), tid, !(a.opts & 1));
            else dev_phase_a16_sel<NT, OC>(Mp, rD, NS, n, it - 1, min(it + 3, dmax), tid);
            TL_MARK(0)
            __syncthreads();
            TL_MARK(5)
        }
        if (wid < NWC) {
            const int d = it;
            if (d <= dmax) {
                const int par = d & 1;
                const int ntyped = sCount[d % 3];
                const unsigned int *list = sList + par * NS;
                const int K = min(30, d - 6);
#ifndef MF_NO_TAIL_PREFETCH
                // phase 2 of this thread's cell reads DML(d-2..d-4) from the global ring: start pulling those
                // lines into L1 now, the interior-loop phase hides the L2 latency
                if (tid < ntyped && d >= 8) {
                    const int i = (int)(list[tid] & 0xffffu) >> 2;
                    dev_prefetch_l1(&rD[((d - 2) & (MF_RING_DML - 1)) * NS + i]);
                    dev_prefetch_l1(&rD[((d - 3) & (MF_RING_DML - 1)) * NS + i]);
                    dev_prefetch_l1(&rD[((d - 4) & (MF_RING_DML - 1)) * NS + i + 1]);
                }
#endif
                // per-lane word-term addresses (bytes, shared window) and packed constants
                unsigned off[MF16_NQ], cst[MF16_NQ], mk[MF16_NMK];
#pragma unroll
                for (int q = 0; q < MF16_NQ; q++) {
                    off[q] = smem_base + sOff[(par * MF16_NQ + q) * 32 + lane];
                    asm("" : "+r"(off[q]));   // keep the byte address as one register (no re-association in the cell loop)
                    cst[q] = sCst[(par * MF16_NQ + q) * 32 + lane];
                }
#pragma unroll
                for (int q = 0; q < MF16_NMK; q++) mk[q] = sMk[(par * MF16_NMK + q) * 32 + lane];

                // phase 1: one typed cell per warp pass -> interior-loop minimum in sMy
                const int per = (ntyped + NWC - 1) / NWC;
                const int cend = min(ntyped, wid * per + per);
                for (int c = wid * per; c < cend; c++) {
                    const unsigned e = list[c];
                    const unsigned i4 = e & 0xffffu;
                    unsigned accG = MF16_INF2, accB = MF16_INF2;
#pragma unroll
                    for (int q = 0; q < MF16_NQG; q++) {
                        unsigned w = dev_lds(off[q] + i4);
                        if (q < MF16_NMG) w = (w & mk[q]) | (~mk[q] & MF16_INF2);
                        accG = __viaddmin_s16x2(w, cst[q], accG);
                    }
#pragma unroll
                    for (int q = 0; q < MF16_NQB; q++) {
                        unsigned w = dev_lds(off[MF16_NQG + q] + i4);
                        w = (w & mk[MF16_NMG + q]) | (~mk[MF16_NMG + q] & MF16_INF2);
                        accB = __viaddmin_s16x2(w, cst[MF16_NQG + q], accB);
                    }
                    const unsigned dl2 = __byte_perm(e, 0, 0x3232);              // (dl, dl)
                    const unsigned acc = __viaddmin_s16x2(accB, dl2, accG);      // relative to the outer mismatch
                    int v = min((int)(short)(acc & 0xffffu), (int)acc >> 16);
                    v = warp_min(v);
                    if (lane == 0) sMy[c] = v;
                }
                TL_MARK(1)
                asm volatile("bar.sync 1, %0;" ::"n"(CT) : "memory");   // c warps only
                TL_MARK(2)
                // phase 2: one typed cell per thread -- small loops, hairpin, multiloop closing, stores
                for (int c = tid; c < ntyped; c += CT) {
                    const int i = (int)(list[c] & 0xffffu) >> 2, j = i + d;
                    const int my = sMy[c];
                    const int t = sPair[sS[i] * 8 + sS[j]];
                    const int si1 = sS1[i + 1], sj1 = sS1[j - 1];
                    const int wide_loops = (my < MF16_VALID) ? my + sMM[(t * 5 + si1) * 5 + sj1] : MF_INF;
                    int small_loops;
                    const int best = min(wide_loops, dev_cell_tail16(P, sS, sS1, sPair, sB, rr, rD, NS, i, d, t, si1, sj1, K, small_loops));
                    const int tt = dev_rtype(t);
                    const int mm = sMM[(tt * 5 + sS1[j + 1]) * 5 + sS1[i - 1]];
                    Cb[(d - 4) * NS + i - 1] = best;
                    // traceback hint: some two-loop (p,q) reproduces c(i,j).  Where the bit stays 0 the traceback skips its
                    // 496-candidate scan and goes straight to the multiloop decomposition (58 % of its scan rounds end there)
                    Ib[(d - 4) * NS + i - 1] = (unsigned char)(min(wide_loops, small_loops) == best);
                    if (best < MF16_GUARD) sFlag = 1;
                    dev_ring16_put(sG, rr, d, i - 1, max(best + mm, -32768));
                    dev_ring16_put(sB, rr, d, i - 1, max(best + (tt > 2 ? AUp : 0), -32768));
                }
            } else asm volatile("bar.sync 1, %0;" ::"n"(CT) : "memory");
        } else {
            const int mt = tid - CT;
            const int dm = it - 1;
            // the int32 fML row of diagonal it-2 (complete since the last barrier) leaves through the TMA engine
            if (BULK && mt == 0 && dm - 1 >= 4 && !newest_row_stored)
                dev_bulk_store_row(Mb + (dm - 5) * NS, sMrow + ((dm - 1) & 1) * NS, (unsigned)(((n - dm + 1) * 4 + 15) & ~15));
            if (dm >= 4) {
                const int *Mprev = sMrow + ((dm - 1) & 1) * NS;
                int *Mcur = sMrow + (dm & 1) * NS;
                for (int i = mt + 1; i <= n - dm; i += MT) {
                    const int m = dev_fml16(P, sS, sS1, sPair, sB, rr, Mprev, rD, NS, i, dm, Ls);
                    if (!BULK) Mb[(dm - 4) * NS + i - 1] = m;
                    Mcur[i - 1] = m;
                    dev_store_fml16_sel<OC>(Mp, NS, dm, i, m, DYNW ? sWideM : &sFlag);   // 16-bit copy (copies) for the DML strips
                }
            }
            TL_MARK(1)
            const int dn = it + 1;
            if (mt == 0) sCount[(it + 2) % 3] = 0;
            if (dn <= dmax) {
                unsigned int *list = sList + (dn & 1) * NS;
                for (int i = mt + 1; i <= n - dn; i += MT) {
                    const int t = (dn < Ls) ? sPair[sS[i] * 8 + sS[i + dn]] : 0;
                    if (t) {
                        const int dl = (t > 2 ? AUp : 0) - sMM[(t * 5 + sS1[i + 1]) * 5 + sS1[i + dn - 1]] + MF16_DBIAS;
                        list[atomicAdd(&sCount[dn % 3], 1)] = (unsigned)(i * 4) | ((unsigned)dl << 16);
                    } else {
                        dev_ring16_put(sG, rr, dn, i - 1, MF16_INF);
                        dev_ring16_put(sB, rr, dn, i - 1, MF16_INF);
                        Cb[(dn - 4) * NS + i - 1] = MF_INF;
                    }
                }
                for (int k = mt; k < MF16_NQ * 32; k += MT)
                    sOff[(dn & 1) * MF16_NQ * 32 + k] = dev_term_off16((&P->s16_td[dn & 1][0][0])[k], k & 31, dn, rr, RS, RW);
            }
            if (mt == MT - 1) sRowP[((it + 3) >> 1) & 31] = RingRows::direct((it + 3) >> 1, RS);   // first used for diagonal it+2
            if ((it + 1 - 5) % 5 == 0 && it <= dmax) {   // next iteration runs the DML strip [it, it+4]
                // a strip whose rows are not split over several warps (nparts == 1) overwrites every cell it owns; only the
                // atomicMin accumulation of split rows needs the ring rows preset
                constexpr int TWs = OC ? 30 : 29;
                const int ntiles = (((n - it + 1) >> 1) + TWs - 1) / TWs;
                if (NW / ntiles > 1)
                    for (int s = 0; s < 5; s++)
                        for (int i = mt; i < n; i += MT) rD[((it + s) & (MF_RING_DML - 1)) * NS + i] = MF_INF;
            }
        }
        TL_MARK(3)
        if (BULK && tid == CT) dev_bulk_wait_read();   // the row buffer of diagonal it-2 is rewritten in the next iteration
        __syncthreads();
        TL_MARK(4)
    }
    TL_DUMP
    if (BULK && tid == CT && dmax >= 4) {      // last row: diagonal dmax, filled in the final iteration
        dev_bulk_store_row(Mb + (dmax - 4) * NS, sMrow + (dmax & 1) * NS, (unsigned)(((n - dmax) * 4 + 15) & ~15));
        dev_bulk_wait_all();
    }
    if (tid == 0 && sFlag) a.flags[blockIdx.x] = 1;
}

// ------------------------------------------------------------------------------------ K2 (generic: any n)
// Same algorithm with the Cm window in a global-memory ring (for loci longer than the largest
// shared-memory bucket).  Scratch sS[npad] | sS1[npad] | pairtab[64] | list[n] (int), generic_scratch_bytes():
// dynamic shared memory, or (GSCR) global memory after the unit's Cm ring when the launch's longest unit does not fit
template <int NT, bool GSCR>
__global__ void __launch_bounds__(NT) k_fill_generic(FillLaunch a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const LocusDesc L = a.loci[blockIdx.x];
    const int n = L.n, Ls = L.Ls, dmax = L.dmax, NS = L.stride;
    const DevParams *__restrict__ P = a.P;
    const int npad = (n + 3 + 15) & ~15;
    int *rD = a.ring + L.ring_off;                              // [MF_RING_DML][NS]
    int *rCm = rD + (unsigned long long)MF_RING_DML * NS;       // [MF_RING_CM][NS]
    unsigned char *sS = GSCR ? (unsigned char *)(rCm + (unsigned long long)MF_RING_CM * NS) : smem_raw;
    unsigned char *sS1 = sS + npad;
    unsigned char *sPair = sS1 + npad;
    int *sList = (int *)(sPair + 64);
    __shared__ int sCount;

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    constexpr int NW = NT / 32;

    for (int k = tid; k < n + 3; k += NT) {
        const unsigned char b = a.codes[L.seq_off + k];
        sS[k] = b & 7;
        sS1[k] = b >> 4;
    }
    if (tid < 64) sPair[tid] = P->pair[tid];

    int *Cb = a.C + L.band_off;
    int *Mb = a.M + L.band_off;
    for (long long k = tid; k < (long long)(dmax - 3) * (NS / 4); k += NT) ((unsigned int *)(a.Ib + L.band_off))[k] = 0x01010101u;   // no traceback hint
    for (int k = tid; k < MF_RING_DML * NS; k += NT) rD[k] = MF_INF;
    __syncthreads();

    for (int d = 4; d <= dmax; d++) {
        if ((d - 4) % 5 == 0) {
            dev_phase_a<NT>(Mb, rD, NS, n, d, min(d + 4, dmax), tid);
            __syncthreads();
        }
        const int ncell = n - d;
        int *Cd = Cb + (d - 4) * NS;
        int *CmD = rCm + (d & (MF_RING_CM - 1)) * NS;
        if (tid == 0) sCount = 0;
        __syncthreads();
        for (int i = tid + 1; i <= ncell; i += NT) {
            const int t = (d < Ls) ? sPair[sS[i] * 8 + sS[i + d]] : 0;
            if (t) sList[atomicAdd(&sCount, 1)] = i;
            else { Cd[i - 1] = MF_INF; CmD[i - 1] = MF_INF; }
        }
        __syncthreads();
        const int ntyped = sCount;
        const int K = min(30, d - 6);
        for (int c = wid; c < ntyped; c += NW) {
            const int i = sList[c], j = i + d;
            const int t = sPair[sS[i] * 8 + sS[j]];
            const int si1 = sS1[i + 1], sj1 = sS1[j - 1];
            int best = MF_INF;
#pragma unroll 4
            for (int it = 0; it < 16; it++) {
                int s, u;
                if (it < 15) { if (lane <= it) { s = it; u = lane; } else { s = 30 - it; u = lane - it - 1; } }
                else { s = 15; u = lane; }
                const int cst = P->ilc[it][lane];
                if (s <= K && cst < MF_INF)
                    best = min(best, rCm[((d - 2 - s) & (MF_RING_CM - 1)) * NS + (i + u)] + cst);
            }
            best += P->mismatchI[(t * 5 + si1) * 5 + sj1];
            // bulges of size >= 2 (58 terms): lanes 0..28 take (nl,0) and (0,nl)
            {
                const int nl = lane + 2;
                if (nl <= K) {
                    const int q1 = j - 1, p1 = i + 1 + nl, p2 = i + 1, q2 = j - 1 - nl;
                    const int ta = sPair[sS[p1] * 8 + sS[q1]], tb = sPair[sS[p2] * 8 + sS[q2]];
                    const int au = (t > 2 ? P->TerminalAU : 0), bl = P->bulge[nl];
                    if (ta) best = min(best, Cb[(q1 - p1 - 4) * NS + p1 - 1] + bl + au + (ta > 2 ? P->TerminalAU : 0));
                    if (tb) best = min(best, Cb[(q2 - p2 - 4) * NS + p2 - 1] + bl + au + (tb > 2 ? P->TerminalAU : 0));
                }
            }
            best = warp_min(best);
            if (lane == 0) {
                best = min(best, dev_cell_tail(P, sS, sS1, sPair, Cb, rD, NS, i, d, t, si1, sj1, K));
                const int tt = P->rtype[t];
                Cd[i - 1] = best;
                CmD[i - 1] = best + P->mismatchI[(tt * 5 + sS1[j + 1]) * 5 + sS1[i - 1]];
            }
        }
        __syncthreads();
        for (int i = tid + 1; i <= ncell; i += NT)
            Mb[(d - 4) * NS + i - 1] = dev_fml(P, sS, sS1, sPair, Cb, Mb, rD, NS, i, d, Ls);
        if (d + 1 <= dmax && (d + 1 - 4) % 5 == 0) {
            for (int s = 0; s < 5; s++)
                for (int i = tid; i < n; i += NT) rD[((d + 1 + s) & (MF_RING_DML - 1)) * NS + i] = MF_INF;
        }
        __syncthreads();
    }
}

#ifndef MF_B608_NT
#define MF_B608_NT 512
#endif
#ifndef MF_B864_NT
#define MF_B864_NT 1024    /* stride-864 bucket: 155 KB of shared memory, so one CTA per SM -- it has to bring all 32 warps itself */
#endif
#ifndef MF_B352_NT
#define MF_B352_NT 320     /* threads and CTAs/SM of the stride-352 bucket: 10 warps, 72 registers, no spills (70.5 -> 66.4 ms on 20 k loci of ~306 nt) */
#define MF_B352_MINB 3
#endif
template <int NS, int NT, int MINB>
static cudaError_t configure_fill_bucket()
{
    cudaError_t e = cudaFuncSetAttribute(k_fill_smem<NS, NT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FillSmem<NS>::bytes);
    if (e != cudaSuccess) return e;
    if (NS > 352) {
        e = cudaFuncSetAttribute(k_fill_s16<NS, NT, MF16_NWM(NT), MINB, (NS > 352)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Fill16Smem<NS>::bytes);
        if (e != cudaSuccess) return e;
    }
    return cudaFuncSetAttribute(k_fill_s16<NS, NT, MF16_NWM(NT), MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Fill16Smem<NS>::bytes);
}
// function attributes are per device: called once per device of a context (mirfold_open)
cudaError_t fill_configure_device()
{
    cudaError_t e;
    if ((e = configure_fill_bucket<MF_TILE_LEN_BIG, MF_B864_NT, 1>()) != cudaSuccess) return e;
    if ((e = configure_fill_bucket<608, MF_B608_NT, 2>()) != cudaSuccess) return e;
    if ((e = configure_fill_bucket<352, MF_B352_NT, MF_B352_MINB>()) != cudaSuccess) return e;
    if ((e = configure_fill_bucket<160, 256, 4>()) != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_fill_generic<512, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MF_GENERIC_SMEM_MAX);
}

template <int NS, int NT, int MINB>
static cudaError_t launch_fill_bucket(const FillLaunch &a, int first, int count, cudaStream_t st)
{
    if (count <= 0) return cudaSuccess;
    const size_t smem = FillSmem<NS>::bytes, smem16 = Fill16Smem<NS>::bytes;
    FillLaunch b = a;
    b.loci = a.loci + first;
    b.nloci = count;
    if (a.force_wide) b.flags = nullptr;
    else {
        b.flags = a.flags + first;
        cudaError_t e;
        // wide spans: the instantiation that survives out-of-range fML (FillLaunch::opts bit 3, set by the host from the span)
        if (NS > 352 && (a.opts & 8)) k_fill_s16<NS, NT, MF16_NWM(NT), MINB, (NS > 352)><<<count, NT, smem16, st>>>(b);
        else k_fill_s16<NS, NT, MF16_NWM(NT), MINB, false><<<count, NT, smem16, st>>>(b);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    k_fill_smem<NS, NT, MINB><<<count, NT, smem, st>>>(b);   // 32-bit kernel: all loci if forced, else only flagged ones
    return cudaGetLastError();
}

// Loci arrive sorted by descending DP cells == descending n (for a fixed span), so each stride
// bucket is a contiguous range [bucket_first[k], bucket_first[k+1]).
cudaError_t launch_fill(const FillLaunch &a, cudaStream_t st, cudaStream_t side, cudaEvent_t fork, cudaEvent_t join)
{
    if (a.nloci == 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    // The buckets touch disjoint fill units: the smaller ones run on a side stream so that their CTAs fill
    // the SMs the last wave of the big bucket leaves idle.
    const bool fork_small = side != nullptr && (a.bucket_first[5] - a.bucket_first[3]) > 0 && (a.bucket_first[3] - a.bucket_first[0]) > 0;
    cudaStream_t st2 = fork_small ? side : st;
    if (fork_small) {
        if ((e = cudaEventRecord(fork, st)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(side, fork, 0)) != cudaSuccess) return e;
    }
    // generic (units no shared-memory bucket holds)
    const int ng = a.bucket_first[1] - a.bucket_first[0];
    if (ng > 0) {
        constexpr int NT = 512;
        const size_t smem = generic_scratch_bytes(a.max_n);
        FillLaunch b = a;
        b.loci = a.loci + a.bucket_first[0];
        b.nloci = ng;
        if (smem <= MF_GENERIC_SMEM_MAX) k_fill_generic<NT, false><<<ng, NT, smem, st>>>(b);
        else k_fill_generic<NT, true><<<ng, NT, 0, st>>>(b);   // a unit of more than about 34 100 nt
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if ((e = launch_fill_bucket<MF_TILE_LEN_BIG, MF_B864_NT, 1>(a, a.bucket_first[1], a.bucket_first[2] - a.bucket_first[1], st)) != cudaSuccess) return e;
    if ((e = launch_fill_bucket<608, MF_B608_NT, 2>(a, a.bucket_first[2], a.bucket_first[3] - a.bucket_first[2], st)) != cudaSuccess) return e;
    if ((e = launch_fill_bucket<352, MF_B352_NT, MF_B352_MINB>(a, a.bucket_first[3], a.bucket_first[4] - a.bucket_first[3], st2)) != cudaSuccess) return e;
    if ((e = launch_fill_bucket<160, 256, 4>(a, a.bucket_first[4], a.bucket_first[5] - a.bucket_first[4], st2)) != cudaSuccess) return e;
    if (fork_small) {
        if ((e = cudaEventRecord(join, side)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(st, join, 0)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------ K3
// f3 scan (A.3, "RLF Lfold.c:355-398").  One warp per locus; rows are taken in blocks of 32 from the
// 3' end.  f3(i) = min(f3(i+1), min_j term(i,j)) where term(i,j) reads f3(j+1), f3(j+2) with
// j >= i+4, so for a block [ilo, ihi] every term with span d >= 31 only reads rows above the block:
//   phase P: lane = row, loop over d = 31..L* -- all loads of the diagonal-major band are coalesced
//            (32 consecutive rows of one diagonal = 128 B) and f3/code operands slide in registers;
//   phase S: rows sequential, lane = d (4..30) with the f3 window f3(i+1..i+32) kept in registers
//            and shifted by one lane per row; lane 31 takes the j == n boundary term.
__device__ __forceinline__ int dev_f3_term(const unsigned char *sPair, const int *sD3, const int *sD5, int AUp,
                                           int si, int s1i, int si1, int sj, int s1j1, int d, int Ls,
                                           int cA, int cB, int f1, int f2)
{
    int best = MF_INF;
    int t = (d < Ls) ? sPair[si * 8 + sj] : 0;
    if (t) {
        const int e = cA + (t > 2 ? AUp : 0);
        best = min(e + f1, e + sD3[t * 5 + s1j1] + f2);
    }
    t = (d - 1 >= 4) ? sPair[si1 * 8 + sj] : 0;
    if (t) {
        const int e = cB + sD5[t * 5 + s1i] + (t > 2 ? AUp : 0);
        best = min(best, min(e + f1, e + sD3[t * 5 + s1j1] + f2));
    }
    return best;
}

#ifndef MF_F3_MINB
#define MF_F3_MINB 12   /* 40 registers: more resident warps = more band lines in flight (4.2 -> 3.75 ms) */
#endif
__global__ void __launch_bounds__(128, MF_F3_MINB) k_f3(const LocusDesc *__restrict__ loci, int nloci,
                                            const unsigned char *__restrict__ codes, const int *__restrict__ Call,
                                            int *__restrict__ Fall, const DevParams *__restrict__ P)
{
    __shared__ unsigned char sPair[64];
    __shared__ int sD3[40], sD5[40];
    if (threadIdx.x < 64) sPair[threadIdx.x] = P->pair[threadIdx.x];
    if (threadIdx.x < 40) { sD3[threadIdx.x] = P->dangle3[threadIdx.x]; sD5[threadIdx.x] = P->dangle5[threadIdx.x]; }
    __syncthreads();
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= nloci) return;
    const LocusDesc L = loci[w];
    const int n = L.n, Ls = L.Ls, NS = L.stride;
    const unsigned char *__restrict__ cd = codes + L.seq_off;
    const int *__restrict__ C = Call + L.band_off;
    int *F = Fall + L.seq_off;
    const int AUp = P->TerminalAU;
    constexpr int DS = 31;   // first span of phase P
    for (int ihi = n - 4; ihi >= 1; ihi -= 32) {
        const int ilo = max(1, ihi - 31);
        // ---- phase P
        int gout = MF_INF;
        {
            const int i = ilo + lane;
            if (i <= ihi) {
                const int dend = min(Ls, n - 1 - i);
                if (dend >= DS) {
                    const int ci = cd[i], si = ci & 7, s1i = ci >> 4, si1 = cd[i + 1] & 7;
                    int j = i + DS;
                    int cj = cd[j], f1 = F[j + 1];
                    const int *pa = C + band_row_base(L, i) + (DS - 4) * NS;   // C(i, i+d), in row i's owner tile
#ifndef MF_F3_UNROLL
#define MF_F3_UNROLL 4
#endif
                    MF_UNROLL_(MF_F3_UNROLL)
                    for (int d = DS; d <= dend; d++, j++, pa += NS) {
                        const int cj1 = cd[j + 1], f2 = F[j + 2];
                        const int cA = pa[0], cB = pa[1 - NS];      // C(i+1, j) sits one diagonal down, one row up
                        gout = min(gout, dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, cj & 7, cj1 >> 4, d, Ls, cA, cB, f1, f2));
                        cj = cj1; f1 = f2;
                    }
                }
            }
        }
        // ---- phase S
        int Fw;
        {
            const int k = ihi + 1 + lane;
            Fw = (k <= n + 2) ? F[k] : 0;
        }
        for (int i = ihi; i >= ilo; i--) {
            const int d = lane, j = i + d;
            const int *Ci = C + band_row_base(L, i);   // row i of its owner tile; (i+1, j) is one diagonal down, one row up
            const int f2 = __shfl_down_sync(0xffffffffu, Fw, 1);
            const int ci = cd[i], si = ci & 7, s1i = ci >> 4, si1 = cd[i + 1] & 7;
            int best = MF_INF;
            if (d >= 4 && d < DS && d <= Ls && j <= n - 1) {
                const int cA = Ci[(d - 4) * NS];
                const int cB = (d >= 5) ? Ci[(d - 5) * NS + 1] : MF_INF;
                best = dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, cd[j] & 7, cd[j + 1] >> 4, d, Ls, cA, cB, Fw, f2);
            }
            if (lane == 31 && n <= i + Ls) {   // j == n: no f3 / dangle3 terms
                const int dn = n - i, sj = cd[n] & 7;
                int t = (dn < Ls) ? sPair[si * 8 + sj] : 0;
                if (t) best = min(best, Ci[(dn - 4) * NS] + (t > 2 ? AUp : 0));
                t = (dn - 1 >= 4) ? sPair[si1 * 8 + sj] : 0;
                if (t) best = min(best, Ci[(dn - 5) * NS + 1] + sD5[t * 5 + s1i] + (t > 2 ? AUp : 0));
            }
            best = warp_min(best);
            const int g = __shfl_sync(0xffffffffu, gout, i - ilo);
            const int fnext = __shfl_sync(0xffffffffu, Fw, 0);   // f3(i+1)
            const int fi = min(fnext, min(best, g));
            if (lane == 0) F[i] = fi;
            Fw = __shfl_up_sync(0xffffffffu, Fw, 1);
            if (lane == 0) Fw = fi;
        }
        __syncwarp();
    }
}

// f3 for long loci: one CTA of NW warps per locus.  Same two phases as k_f3; the block's f3 / code
// window is staged in shared memory and phase P's span range [31, L*] is cut into NW contiguous
// slices (one per warp, lane = row), so the sequential chain over 32-row blocks only carries
// ~L*/NW band loads per block instead of L*.
template <int NW>
__global__ void __launch_bounds__(NW * 32) k_f3_cta(const LocusDesc *__restrict__ loci, int nloci,
                                                    const unsigned char *__restrict__ codes, const int *__restrict__ Call,
                                                    int *__restrict__ Fall, const DevParams *__restrict__ P, int win)
{
    __shared__ unsigned char sPair[64];
    __shared__ int sD3[40], sD5[40];
    __shared__ int sG[NW][32];
    extern __shared__ __align__(16) unsigned char f3_dyn[];
    int *sF = (int *)f3_dyn;                              // f3(ilo + k), k < win
    unsigned char *sC = (unsigned char *)(sF + win);      // codes(ilo + k)
    constexpr int NT = NW * 32;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid < 64) sPair[tid] = P->pair[tid];
    if (tid < 40) { sD3[tid] = P->dangle3[tid]; sD5[tid] = P->dangle5[tid]; }
    const LocusDesc L = loci[blockIdx.x];
    const int n = L.n, Ls = L.Ls, NS = L.stride;
    const unsigned char *__restrict__ cd = codes + L.seq_off;
    const int *__restrict__ C = Call + L.band_off;
    int *F = Fall + L.seq_off;
    const int AUp = P->TerminalAU;
    constexpr int DS = 31;
    const int slice = (max(Ls - DS + 1, 0) + NW - 1) / NW;
    for (int ihi = n - 4; ihi >= 1; ihi -= 32) {
        const int ilo = max(1, ihi - 31);
        __syncthreads();   // previous block's f3 stores (warp 0) are visible; sF/sC/sG free again
        for (int k = tid; k < win; k += NT) {
            const int pos = ilo + k;
            sF[k] = (pos <= n + 2) ? F[pos] : 0;
            sC[k] = (pos <= n + 2) ? cd[pos] : 0;
        }
        __syncthreads();
        // ---- phase P: warp w takes spans [d0, d1]
        int gout = MF_INF;
        {
            const int i = ilo + lane;
            if (i <= ihi && slice > 0) {
                const int dend = min(Ls, n - 1 - i);
                const int d0 = DS + w * slice, d1 = min(dend, d0 + slice - 1);
                if (d0 <= d1) {
                    const int ci = sC[lane], si = ci & 7, s1i = ci >> 4, si1 = sC[lane + 1] & 7;
                    const int *pa = C + band_row_base(L, i) + (d0 - 4) * NS;
                    int jl = lane + d0;   // j - ilo
#pragma unroll 4
                    for (int d = d0; d <= d1; d++, jl++, pa += NS) {
                        const int cA = pa[0], cB = pa[1 - NS];
                        gout = min(gout, dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, sC[jl] & 7, sC[jl + 1] >> 4, d, Ls, cA, cB,
                                                     sF[jl + 1], sF[jl + 2]));
                    }
                }
            }
        }
        sG[w][lane] = gout;
        __syncthreads();
        if (w == 0) {
#pragma unroll
            for (int k = 1; k < NW; k++) gout = min(gout, sG[k][lane]);
            // ---- phase S (as k_f3)
            int Fw = sF[ihi + 1 - ilo + lane];
            for (int i = ihi; i >= ilo; i--) {
                const int d = lane, j = i + d;
                const int *Ci = C + band_row_base(L, i);
                const int f2 = __shfl_down_sync(0xffffffffu, Fw, 1);
                const int ci = sC[i - ilo], si = ci & 7, s1i = ci >> 4, si1 = sC[i + 1 - ilo] & 7;
                int best = MF_INF;
                if (d >= 4 && d < DS && d <= Ls && j <= n - 1) {
                    const int cA = Ci[(d - 4) * NS];
                    const int cB = (d >= 5) ? Ci[(d - 5) * NS + 1] : MF_INF;
                    best = dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, sC[j - ilo] & 7, sC[j + 1 - ilo] >> 4, d, Ls, cA, cB, Fw, f2);
                }
                if (lane == 31 && n <= i + Ls) {   // j == n: no f3 / dangle3 terms
                    const int dn = n - i, sj = cd[n] & 7;
                    int t = (dn < Ls) ? sPair[si * 8 + sj] : 0;
                    if (t) best = min(best, Ci[(dn - 4) * NS] + (t > 2 ? AUp : 0));
                    t = (dn - 1 >= 4) ? sPair[si1 * 8 + sj] : 0;
                    if (t) best = min(best, Ci[(dn - 5) * NS + 1] + sD5[t * 5 + s1i] + (t > 2 ? AUp : 0));
                }
                best = warp_min(best);
                const int g = __shfl_sync(0xffffffffu, gout, i - ilo);
                const int fnext = __shfl_sync(0xffffffffu, Fw, 0);   // f3(i+1)
                const int fi = min(fnext, min(best, g));
                if (lane == 0) F[i] = fi;
                Fw = __shfl_up_sync(0xffffffffu, Fw, 1);
                if (lane == 0) Fw = fi;
            }
        }
    }
}

// k_f3_cta over rows row_hi down to row_lo of one segment of a segmented locus (host.cu, fold_segmented), below rows whose
// f3 earlier segments left in F.  The descriptor is the locus' suffix from the segment's first tile on, so every band offset
// is relative to the segment's buffer.  A copy of k_f3_cta rather than a shared body: k_f3_cta keeps its exact code.
template <int NW>
__global__ void __launch_bounds__(NW * 32) k_f3_seg(const LocusDesc *__restrict__ loci, const unsigned char *__restrict__ codes,
                                                    const int *__restrict__ Call, int *__restrict__ Fall,
                                                    const DevParams *__restrict__ P, int win, int row_hi, int row_lo)
{
    __shared__ unsigned char sPair[64];
    __shared__ int sD3[40], sD5[40];
    __shared__ int sG[NW][32];
    extern __shared__ __align__(16) unsigned char f3_dyn[];
    int *sF = (int *)f3_dyn;                              // f3(ilo + k), k < win
    unsigned char *sC = (unsigned char *)(sF + win);      // codes(ilo + k)
    constexpr int NT = NW * 32;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid < 64) sPair[tid] = P->pair[tid];
    if (tid < 40) { sD3[tid] = P->dangle3[tid]; sD5[tid] = P->dangle5[tid]; }
    const LocusDesc L = loci[blockIdx.x];
    const int n = L.n, Ls = L.Ls, NS = L.stride;
    const unsigned char *__restrict__ cd = codes + L.seq_off;
    const int *__restrict__ C = Call + L.band_off;
    int *F = Fall + L.seq_off;
    const int AUp = P->TerminalAU;
    constexpr int DS = 31;
    const int slice = (max(Ls - DS + 1, 0) + NW - 1) / NW;
    for (int ihi = row_hi; ihi >= row_lo; ihi -= 32) {
        const int ilo = max(row_lo, ihi - 31);
        __syncthreads();   // previous block's f3 stores (warp 0) are visible; sF/sC/sG free again
        for (int k = tid; k < win; k += NT) {
            const int pos = ilo + k;
            sF[k] = (pos <= n + 2) ? F[pos] : 0;
            sC[k] = (pos <= n + 2) ? cd[pos] : 0;
        }
        __syncthreads();
        // ---- phase P: warp w takes spans [d0, d1]
        int gout = MF_INF;
        {
            const int i = ilo + lane;
            if (i <= ihi && slice > 0) {
                const int dend = min(Ls, n - 1 - i);
                const int d0 = DS + w * slice, d1 = min(dend, d0 + slice - 1);
                if (d0 <= d1) {
                    const int ci = sC[lane], si = ci & 7, s1i = ci >> 4, si1 = sC[lane + 1] & 7;
                    const int *pa = C + band_row_base(L, i) + (d0 - 4) * NS;
                    int jl = lane + d0;   // j - ilo
#pragma unroll 4
                    for (int d = d0; d <= d1; d++, jl++, pa += NS) {
                        const int cA = pa[0], cB = pa[1 - NS];
                        gout = min(gout, dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, sC[jl] & 7, sC[jl + 1] >> 4, d, Ls, cA, cB,
                                                     sF[jl + 1], sF[jl + 2]));
                    }
                }
            }
        }
        sG[w][lane] = gout;
        __syncthreads();
        if (w == 0) {
#pragma unroll
            for (int k = 1; k < NW; k++) gout = min(gout, sG[k][lane]);
            // ---- phase S (as k_f3)
            int Fw = sF[ihi + 1 - ilo + lane];
            for (int i = ihi; i >= ilo; i--) {
                const int d = lane, j = i + d;
                const int *Ci = C + band_row_base(L, i);
                const int f2 = __shfl_down_sync(0xffffffffu, Fw, 1);
                const int ci = sC[i - ilo], si = ci & 7, s1i = ci >> 4, si1 = sC[i + 1 - ilo] & 7;
                int best = MF_INF;
                if (d >= 4 && d < DS && d <= Ls && j <= n - 1) {
                    const int cA = Ci[(d - 4) * NS];
                    const int cB = (d >= 5) ? Ci[(d - 5) * NS + 1] : MF_INF;
                    best = dev_f3_term(sPair, sD3, sD5, AUp, si, s1i, si1, sC[j - ilo] & 7, sC[j + 1 - ilo] >> 4, d, Ls, cA, cB, Fw, f2);
                }
                if (lane == 31 && n <= i + Ls) {   // j == n: no f3 / dangle3 terms
                    const int dn = n - i, sj = cd[n] & 7;
                    int t = (dn < Ls) ? sPair[si * 8 + sj] : 0;
                    if (t) best = min(best, Ci[(dn - 4) * NS] + (t > 2 ? AUp : 0));
                    t = (dn - 1 >= 4) ? sPair[si1 * 8 + sj] : 0;
                    if (t) best = min(best, Ci[(dn - 5) * NS + 1] + sD5[t * 5 + s1i] + (t > 2 ? AUp : 0));
                }
                best = warp_min(best);
                const int g = __shfl_sync(0xffffffffu, gout, i - ilo);
                const int fnext = __shfl_sync(0xffffffffu, Fw, 0);   // f3(i+1)
                const int fi = min(fnext, min(best, g));
                if (lane == 0) F[i] = fi;
                Fw = __shfl_up_sync(0xffffffffu, Fw, 1);
                if (lane == 0) Fw = fi;
            }
        }
    }
}

// loci are sorted by descending length: the first n_long (n > MF_TILE_LEN) get a CTA each
cudaError_t launch_f3(const LocusDesc *loci, int nloci, int n_long, int max_Ls, const unsigned char *codes, const int *C, int *F,
                      const DevParams *P, cudaStream_t st)
{
    if (nloci == 0) return cudaSuccess;
    if (n_long > 0) {
        constexpr int NW = 8;
        const int win = (std::max(max_Ls, 32) + 40 + 3) & ~3;   // phase S touches up to 64 entries past ilo
        k_f3_cta<NW><<<n_long, NW * 32, (size_t)win * 5, st>>>(loci, n_long, codes, C, F, P, win);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    const int rest = nloci - n_long;
    if (rest > 0) {
        const int warps_per_block = 4;
        k_f3<<<(rest + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(loci + n_long, rest, codes, C, F, P);
    }
    return cudaGetLastError();
}

cudaError_t launch_f3_rows(const LocusDesc *locus, int Ls, int row_hi, int row_lo, const unsigned char *codes, const int *C, int *F,
                           const DevParams *P, cudaStream_t st)
{
    if (row_hi < row_lo) return cudaSuccess;
    constexpr int NW = 8;
    const int win = (std::max(Ls, 32) + 40 + 3) & ~3;
    k_f3_seg<NW><<<1, NW * 32, (size_t)win * 5, st>>>(locus, codes, C, F, P, win, row_hi, row_lo);
    return cudaGetLastError();
}
