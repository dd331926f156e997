// trace.cu -- emission plan, order-exact traceback and hairpin emission (K4) for sm_100a.
//
// Replaces RNALfold's emission state machine and backtrack() (SURVEY.md 8a rows a8-a9; spec
// Appendix A.4-A.5, "RLF Lfold.c:402-435, 459-771").  The reference interleaves tracebacks with
// the row loop; here the band is complete first, which makes every traceback independent:
//   k_plan      : the state machine depends on f3 only -> list of traceback starts per locus
//   k_traceback : one warp per traceback; every "first match wins" scan of the reference is a
//                 lane-parallel test in reference order + ballot/ffs (lowest lane = first match)
//   k_emit      : the shifted-strncmp containment test between consecutive tracebacks decides
//                 which structures RNALfold would have printed; energy = f3[start]-f3[start+len]
//   k_pack      : compacts printed structures into the result arena (offsets from a device scan)
#include "../../include/mirfold.h"
#include "mirfold_internal.cuh"

#define FULL 0xffffffffu
#ifndef TB_UNR
#define TB_UNR 1   /* 32-candidate chunks evaluated per round of a first-match scan */
#endif

// ------------------------------------------------------------------------------------ plan
__global__ void k_plan(TraceBuffers b)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= b.nloci) return;
    const LocusDesc L = b.loci[l];
    const int *F = b.F + L.seq_off;
    int *list = b.tb_start_list + b.list_off[l];
    int cnt = 0, do_bt = 0, have_prev = 0;
    int fnext = F[L.n - 3];
    for (int i = L.n - 4; i >= 1; i--) {
        const int fi = F[i];
        if (fi != fnext) do_bt = 1;
        else if (do_bt) { list[cnt++] = i + 1; have_prev = 1; do_bt = 0; }
        if (i == 1) {
            if (!have_prev) do_bt = 1;
            if (do_bt) list[cnt++] = 1;   // final backtrack(1, L*)
        }
        fnext = fi;
    }
    b.tb_count[l] = cnt;
}

cudaError_t launch_plan(const TraceBuffers &b, cudaStream_t st)
{
    if (b.nloci == 0) return cudaSuccess;
    k_plan<<<(b.nloci + 127) / 128, 128, 0, st>>>(b);
    return cudaGetLastError();
}

// k_plan over rows row_hi .. row_lo of one segment of a segmented locus (host.cu, fold_segmented), resumed from the state
// the segment above left in state[0..2] (fnext, do_bt, have_prev; all 0 at the top: f3(n-3) == 0) and left there for the
// segment below.  The row loop produces the starts i + 1 of rows row_lo .. row_hi, so every start lies in the segment's
// owned rows or the first row above them, whose traceback the segment's halo holds.  F and the starts are relative to the
// segment's suffix descriptor; `bottom`: the segment holds row 1 of the locus (the final backtrack(1, L*)).
__global__ void k_plan_seg(const int *__restrict__ F, int row_hi, int row_lo, int bottom, int *state, int *list,
                           unsigned long long *tb_base, int *tb_count)
{
    int cnt = 0, fnext = state[0], do_bt = state[1], have_prev = state[2];
    for (int i = row_hi; i >= row_lo; i--) {
        const int fi = F[i];
        if (fi != fnext) do_bt = 1;
        else if (do_bt) { list[cnt++] = i + 1; have_prev = 1; do_bt = 0; }
        if (bottom && i == 1) {
            if (!have_prev) do_bt = 1;
            if (do_bt) list[cnt++] = 1;
        }
        fnext = fi;
    }
    state[0] = fnext; state[1] = do_bt; state[2] = have_prev;
    tb_base[0] = 0; tb_base[1] = (unsigned long long)cnt;
    tb_count[0] = cnt;
}

cudaError_t launch_plan_seg(const int *F, int row_hi, int row_lo, int bottom, int *state, int *list, unsigned long long *tb_base,
                            int *tb_count, cudaStream_t st)
{
    k_plan_seg<<<1, 1, 0, st>>>(F, row_hi, row_lo, bottom, state, list, tb_base, tb_count);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ traceback
// band offset of cell (i, i+d) of a tiled long locus (LocusDesc::tile_*, see band_row_base)
__device__ __noinline__ unsigned long long tb_tiled_off(int i, int d, unsigned int tile_rcp, int tile_last, int tile_step, int n, int dmax)
{
    const int t = tile_of_row(i, tile_rcp, tile_step, tile_last);
    const int TL = tile_step + dmax;   // tile length == the locus' band stride (608 or 864)
    const int a = min(t * tile_step, n - TL);   // tile t's first row - 1: a <= t * tile_step <= i - 1
    // tile t, diagonal d >= 4, local row i-1-a >= 0: every term is non-negative
    return ((unsigned long long)t * (unsigned)(dmax - 3) + (unsigned)(d - 4)) * (unsigned)TL + (unsigned)(i - 1 - a);
}

struct Fold {
    const DevParams *__restrict__ P;
    const unsigned char *__restrict__ cd;  // codes, 1-based
    const int *__restrict__ C;
    const int *__restrict__ M;
    const int *__restrict__ F;
    const unsigned char *__restrict__ Ib;  // hint bytes, same cell addressing as C
    const unsigned char *pairT;   // shared-memory copies of DevParams::pair / rtype (block-wide)
    const unsigned char *rtypeT;
    int AUp;                      // TerminalAU
    int n, Ls, NS;
    // tiled long loci (LocusDesc::tile_*): row i lives in tile min((i-1)/tile_step, tile_last)
    int tile_last, tile_step, dmax;
    unsigned int tile_rcp;
    __device__ __forceinline__ int S(int k) const { return cd[k] & 7; }
    __device__ __forceinline__ int S1(int k) const { return cd[k] >> 4; }
    __device__ __forceinline__ int type(int i, int j) const
    {
        const int d = j - i;
        if (i < 1 || j > n || d < 4 || d >= Ls) return 0;
        return pairT[S(i) * 8 + S(j)];
    }
    // unchecked variants for callers that know 1 <= i, j <= n and 4 <= j-i < Ls (inner cells of a pair)
    __device__ __forceinline__ int type_nc(int i, int j) const { return pairT[S(i) * 8 + S(j)]; }
    __device__ __forceinline__ int c_nc(int i, int j) const
    {
        const int d = j - i;
        unsigned long long off = (unsigned)((d - 4) * NS + (i - 1));
        if (tile_last) off = tb_tiled_off(i, d, tile_rcp, tile_last, tile_step, n, dmax);
        return C[off];
    }
    // fill's hint for the pair (i,j): false = no two-loop (p,q) reproduces c(i,j), the candidate scan cannot succeed
    __device__ __forceinline__ bool two_loop_possible(int i, int j) const
    {
        const int d = j - i;
        unsigned long long off = (unsigned)((d - 4) * NS + (i - 1));
        if (tile_last) off = tb_tiled_off(i, d, tile_rcp, tile_last, tile_step, n, dmax);
        return Ib[off] != 0;
    }
    __device__ __forceinline__ int band(const int *__restrict__ A, int i, int j) const
    {
        const int d = j - i;
        if (i < 1 || j > n || d < 4 || d > Ls) return MF_INF;
        unsigned long long off = (unsigned)((d - 4) * NS + (i - 1));
        if (tile_last) off = tb_tiled_off(i, d, tile_rcp, tile_last, tile_step, n, dmax);   // warp-uniform branch, out of line: not if-converted into the common path
        return A[off];
    }
    __device__ __forceinline__ int c(int i, int j) const { return band(C, i, j); }
    __device__ __forceinline__ int m(int i, int j) const { return band(M, i, j); }
    __device__ __forceinline__ int f(int i) const { return (i >= 1 && i <= n + 2) ? F[i] : 0; }
    __device__ __forceinline__ int AU(int t) const { return t > 2 ? AUp : 0; }
};

__device__ int tb_loop_energy(const Fold &f, int i, int j, int p, int q, int t, int t2)
{
    const DevParams *__restrict__ P = f.P;
    const int n1 = p - i - 1, n2 = j - q - 1;
    const int nl = max(n1, n2), ns = min(n1, n2);
    if (nl == 0) return P->stack[t * 8 + t2];
    if (ns == 0) {
        int e = P->bulge[nl];
        if (nl == 1) return e + P->stack[t * 8 + t2];
        return e + f.AU(t) + f.AU(t2);
    }
    const int si1 = f.S1(i + 1), sj1 = f.S1(j - 1), sp1 = f.S1(p - 1), sq1 = f.S1(q + 1);
    if (ns == 1 && nl == 1) return P->int11[((t * 8 + t2) * 5 + si1) * 5 + sj1];
    if (ns == 1 && nl == 2) {
        if (n1 == 1) return P->int21[(((t * 8 + t2) * 5 + si1) * 5 + sq1) * 5 + sj1];
        return P->int21[(((t2 * 8 + t) * 5 + sq1) * 5 + si1) * 5 + sp1];
    }
    if (n1 == 2 && n2 == 2) return P->int22[((((t * 8 + t2) * 5 + si1) * 5 + sp1) * 5 + sq1) * 5 + sj1];
    return P->internal_loop[n1 + n2] + min(300, (nl - ns) * 50) + P->mismatchI[(t * 5 + si1) * 5 + sj1] +
           P->mismatchI[(t2 * 5 + sq1) * 5 + sp1];
}

__device__ int tb_hairpin(const Fold &f, int i, int j, int t)
{
    const DevParams *__restrict__ P = f.P;
    const int s = j - i - 1;
    int e = P->hairpinE[s];
    if (s == 4) {
        int code = 0, ok = 1;
        for (int k = 0; k < 6; k++) {
            const int b = f.S(i + k);
            ok &= (b >= 1 && b <= 4);
            code |= ((b - 1) & 3) << (2 * k);
        }
        if (ok) e += P->tetra[code];
    }
    if (s == 3) e += f.AU(t);
    else e += P->mismatchH[(t * 5 + f.S1(i + 1)) * 5 + f.S1(j - 1)];
    return e;
}

// one warp per traceback
#ifndef TB_MINB
#define TB_MINB 12
#endif
__global__ void __launch_bounds__(128, TB_MINB) k_traceback(TraceBuffers b)
{
    __shared__ unsigned char sPairT[64], sRtypeT[8], sUV[496 * 2];
    if (threadIdx.x < 64) sPairT[threadIdx.x] = b.P->pair[threadIdx.x];
    if (threadIdx.x < 8) sRtypeT[threadIdx.x] = b.P->rtype[threadIdx.x];
    for (int k = threadIdx.x; k < 496 * 2; k += 128) sUV[k] = (&b.P->uv[0][0])[k];
    __syncthreads();
    const unsigned long long g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= b.ntb) return;
    // locate the locus: largest l with tb_base[l] <= g
    int lo = 0, hi = b.nloci;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (b.tb_base[mid] <= g) lo = mid; else hi = mid;
    }
    const int l = lo;
    const LocusDesc L = b.loci[l];
    const int kidx = (int)(g - b.tb_base[l]);
    const int start = b.tb_start_list[b.list_off[l] + kidx];
    Fold f;
    f.P = b.P; f.C = b.C + L.band_off; f.M = b.M + L.band_off; f.F = b.F + L.seq_off;
    f.Ib = b.Ib + L.band_off;
    f.pairT = sPairT; f.rtypeT = sRtypeT; f.AUp = b.P->TerminalAU;
    f.n = L.n; f.Ls = L.Ls; f.NS = L.stride;
    f.tile_last = L.tile_last; f.tile_step = L.tile_step; f.dmax = L.dmax; f.tile_rcp = L.tile_rcp;
    const DevParams *__restrict__ P = b.P;
    const int n = L.n;
    const int md = (start == 1) ? L.Ls : L.Ls + 1;   // final backtrack(1, L*) vs backtrack(i+1, L*+1)
    {   // stage the codes of the window [start-1, min(n, start+md+1)+2] in shared memory (every S/S1 lookup hits it)
        extern __shared__ unsigned char s_codes[];
        unsigned char *w = s_codes + (threadIdx.x >> 5) * b.code_win;
        const unsigned char *src = b.codes + L.seq_off;
        const int lo = start - 1, hi = min(n + 2, start + md + 3);
        for (int k = lo + lane; k <= hi; k += 32) w[k - lo] = src[k];
        f.cd = w - lo;
        __syncwarp();
    }

    char *st = b.slots + g * (unsigned long long)b.slot_stride;
    const int ndash = min(n - start, md) + 1;
    for (int k = lane; k < b.slot_stride; k += 32) st[k] = k < ndash ? '-' : 0;
    __syncwarp();

    int *stk = b.stack_scratch + g * (unsigned long long)b.stack_cap * 2ULL;
    int sp = 0;
    bool failed = false;
#define PUSH(a_, b_, ml_)                                                      \
    do {                                                                       \
        if (sp < b.stack_cap) {                                                \
            if (lane == 0) { stk[2 * sp] = (a_); stk[2 * sp + 1] = ((b_) << 1) | (ml_); } \
            sp++;                                                              \
        } else failed = true;                                                  \
    } while (0)
    PUSH(start, min(n, start + md + 1), 0);
    __syncwarp();

    while (sp > 0 && !failed) {
        sp--;
        __syncwarp();
        int i = stk[2 * sp];
        int j = stk[2 * sp + 1];
        const int ml = j & 1;
        j >>= 1;
        if (j < i + 4) continue;
        if (ml == 0) {
            // leading unpaired bases: the reference pushes (i+1, j, 0) and pops it again, one base per round
            // (Lfold.c:501-506); the run of equal f3 values is skipped in one lane-parallel step instead
            int fij = f.f(i);
            bool dropped = false;
            for (;;) {
                const unsigned eq = __ballot_sync(FULL, f.f(i + 1 + lane) == fij);
                const int run = (eq == FULL) ? 32 : __ffs(~eq) - 1;
                if (run == 0) break;
                i += run;
                if (j < i + 4) { dropped = true; break; }   // the popped entry would be discarded (Lfold.c:499)
                // fij is unchanged: f3(i) == f3(i - run) along the run
            }
            if (dropped) continue;
            int traced = 0, jj = 0, kk = 0;
            // candidates k = i+4 .. j in reference order; TB_UNR chunks of 32 per round so that the band / f3
            // loads of a round are all in flight together (the scan is latency-bound, not issue-bound)
            for (int kb = i + 4; kb <= j && !traced; kb += 32 * TB_UNR) {
                int tr[TB_UNR], myjj[TB_UNR];
#pragma unroll
                for (int r = 0; r < TB_UNR; r++) {
                    const int k = kb + 32 * r + lane;
                    tr[r] = 0; myjj[r] = k + 1;
                    if (k <= j) {
                        int t = f.type(i + 1, k);
                        if (t) {
                            const int cc = f.c(i + 1, k) + P->dangle5[t * 5 + f.S1(i)] + f.AU(t);
                            if (fij == cc + f.f(k + 1)) tr[r] = i + 1;
                            if (k < n && fij == f.f(k + 2) + cc + P->dangle3[t * 5 + f.S1(k + 1)]) { tr[r] = i + 1; myjj[r] = k + 2; }
                        }
                        t = f.type(i, k);
                        if (t) {
                            const int cc = f.c(i, k) + f.AU(t);
                            if (fij == cc + f.f(k + 1)) tr[r] = i;
                            if (k < n && fij == f.f(k + 2) + cc + P->dangle3[t * 5 + f.S1(k + 1)]) { tr[r] = i; myjj[r] = k + 2; }
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < TB_UNR; r++) {
                    const unsigned hit = __ballot_sync(FULL, tr[r] != 0);
                    if (hit && !traced) {
                        const int src = __ffs(hit) - 1;
                        traced = __shfl_sync(FULL, tr[r], src);
                        jj = __shfl_sync(FULL, myjj[r], src);
                        kk = kb + 32 * r + src;
                    }
                }
            }
            if (!traced) { failed = true; break; }
            if (j == n) PUSH(jj, j, 0);
            i = traced; j = kk;
            if (lane == 0) {
                st[i - start] = '('; st[j - start] = ')';
                if (jj == j + 2 && j < n) st[j + 1 - start] = '.';
            }
        } else {
            // unpaired bases of a multiloop segment: the reference peels one base per push/pop round, 3' side
            // first, then 5' side (Lfold.c:555-566).  Same order here, but a whole run per step and no stack traffic.
            int fij = 0;
            bool dropped = false;
            for (;;) {
                if (j < i + 4) { dropped = true; break; }   // the popped entry would be discarded (Lfold.c:499)
                fij = f.m(i, j);
                const unsigned eq3 = __ballot_sync(FULL, f.m(i, j - 1 - lane) == fij);
                if (eq3 & 1u) { j -= (eq3 == FULL) ? 32 : __ffs(~eq3) - 1; continue; }
                // 5' side: lane l stands for the state after l peels; it stops at the first l whose 5' test fails or
                // (l >= 1) whose 3' test succeeds -- the outer loop then re-evaluates at that position
                const bool c5 = f.m(i + 1 + lane, j) == fij;
                const bool c3 = lane >= 1 && f.m(i + lane, j - 1) == fij;
                const unsigned go = __ballot_sync(FULL, c5 && !c3);
                const int run = (go == FULL) ? 32 : __ffs(~go) - 1;
                if (run == 0) break;
                i += run;
            }
            if (dropped) continue;
            int t = f.type(i, j);
            const int cij = f.c(i, j) + P->MLintern[t];
            t = f.type(i + 1, j);
            const int ci1j = f.c(i + 1, j) + P->dangle5[t * 5 + f.S1(i)] + P->MLintern[t];
            t = f.type(i, j - 1);
            const int cij1 = f.c(i, j - 1) + P->dangle3[t * 5 + f.S1(j)] + P->MLintern[t];
            t = f.type(i + 1, j - 1);
            const int ci1j1 = f.c(i + 1, j - 1) + P->dangle5[t * 5 + f.S1(i)] + P->dangle3[t * 5 + f.S1(j)] + P->MLintern[t];
            if (fij == cij || fij == ci1j || fij == cij1 || fij == ci1j1) {
                if (fij == ci1j) i++;
                else if (fij == cij1) j--;
                else if (fij == ci1j1) { i++; j--; }
                if (lane == 0) { st[i - start] = '('; st[j - start] = ')'; }
            } else {
                int ksplit = -1;
                for (int kb = i + 4; kb <= j - 5 && ksplit < 0; kb += 32 * TB_UNR) {
                    bool ok[TB_UNR];
#pragma unroll
                    for (int r = 0; r < TB_UNR; r++) {
                        const int k = kb + 32 * r + lane;
                        ok[r] = (k <= j - 5) && (fij == f.m(i, k) + f.m(k + 1, j));
                    }
#pragma unroll
                    for (int r = 0; r < TB_UNR; r++) {
                        const unsigned hit = __ballot_sync(FULL, ok[r]);
                        if (hit && ksplit < 0) ksplit = kb + 32 * r + __ffs(hit) - 1;
                    }
                }
                if (ksplit < 0) { failed = true; break; }
                PUSH(i, ksplit, 1);
                PUSH(ksplit + 1, j, 1);
                continue;
            }
        }
        // "repeat": (i,j) pairs; follow stacks / interior loops until a hairpin or multiloop
        for (;;) {
            // Speculative helix run: lane l looks at the pair (i+l, j-l).  A pair is left by the stack
            // (p,q) = (i+1,j-1) -- the first candidate in reference order -- iff it is not closed by a
            // hairpin and c == stack + c(i+1,j-1); the run ends at the first lane for which that fails,
            // so a whole helix costs one round trip to the band instead of one per base pair.
            const int pi = i + lane, pj = j - lane, dl = pj - pi;
            int tl = 0, cl = MF_INF, hl = 0;
            if (dl >= 4) {   // (i,j) is a pair inside the band, so every (i+l, j-l) with span >= 4 is addressable
                tl = f.type_nc(pi, pj);
                if (tl) { cl = f.c_nc(pi, pj); hl = tb_hairpin(f, pi, pj, tl); }
            }
            const int tn = __shfl_down_sync(FULL, tl, 1), cn = __shfl_down_sync(FULL, cl, 1);
            const bool cont = tl && tn && lane < 31 && cl != hl && dl >= 6 && cl == P->stack[tl * 8 + f.rtypeT[tn]] + cn;
            const int r = __ffs(~__ballot_sync(FULL, cont)) - 1;   // 0..31: first pair of the run that is not left by a stack
            if (lane >= 1 && lane <= r) { st[pi - start] = '('; st[pj - start] = ')'; }
            i += r; j -= r;
            if (r == 31) continue;                                 // lane 31 cannot look ahead: speculate again from there
            const int cij = __shfl_sync(FULL, cl, r), t = __shfl_sync(FULL, tl, r);
            if (cij == __shfl_sync(FULL, hl, r)) break;            // hairpin
            const int d = j - i;
            const int K = min(30, d - 6);
            int np = 0, nq = 0;
            bool found = false;
            if (K >= 0 && f.two_loop_possible(i, j)) {
                for (int cb = 0; cb < 496 && !found; cb += 32 * TB_UNR) {
                    bool ok[TB_UNR];
                    int p[TB_UNR], q[TB_UNR];
#pragma unroll
                    for (int rr = 0; rr < TB_UNR; rr++) {
                        const int m = cb + 32 * rr + lane;
                        ok[rr] = false; p[rr] = 0; q[rr] = 0;
                        if (m < 496) {
                            const int u = sUV[2 * m], v = sUV[2 * m + 1];
                            if (u + v <= K) {   // span of (p,q) = d-2-u-v >= 4: inside the band
                                p[rr] = i + 1 + u; q[rr] = j - 1 - v;
                                const int t2 = f.type_nc(p[rr], q[rr]);
                                if (t2) ok[rr] = (cij == tb_loop_energy(f, i, j, p[rr], q[rr], t, f.rtypeT[t2]) + f.c_nc(p[rr], q[rr]));
                            }
                        }
                    }
#pragma unroll
                    for (int rr = 0; rr < TB_UNR; rr++) {
                        const unsigned hit = __ballot_sync(FULL, ok[rr]);
                        if (hit && !found) {
                            const int src = __ffs(hit) - 1;
                            np = __shfl_sync(FULL, p[rr], src);
                            nq = __shfl_sync(FULL, q[rr], src);
                            found = true;
                        }
                    }
                    // rows u > K contribute nothing; entries are u-major, so stop once u exceeds K
                    if (sUV[2 * min(cb + 32 * TB_UNR, 495)] > K) break;
                }
            }
            if (found) {
                i = np; j = nq;
                if (lane == 0) { st[i - start] = '('; st[j - start] = ')'; }
                continue;
            }
            // multiloop decomposition
            const int tt = f.rtypeT[t];
            const int mm = P->MLclosing + P->MLintern[tt];
            const int d5 = P->dangle5[tt * 5 + f.S1(j - 1)], d3 = P->dangle3[tt * 5 + f.S1(i + 1)];
            int ksplit = -1, which = 0;
            for (int kb = i + 5; kb <= j - 6 && ksplit < 0; kb += 32 * TB_UNR) {
                int w[TB_UNR];
#pragma unroll
                for (int rr = 0; rr < TB_UNR; rr++) {
                    const int k = kb + 32 * rr + lane;
                    w[rr] = 0;
                    if (k <= j - 6) {
                        const int a1 = f.m(i + 1, k), a2 = f.m(i + 2, k), b1 = f.m(k + 1, j - 1), b2 = f.m(k + 1, j - 2);
                        if (cij == a1 + b1 + mm) w[rr] = 1;
                        else if (cij == a2 + b1 + mm + d3) w[rr] = 2;
                        else if (cij == a1 + b2 + mm + d5) w[rr] = 3;
                        else if (cij == a2 + b2 + mm + d3 + d5) w[rr] = 4;
                    }
                }
#pragma unroll
                for (int rr = 0; rr < TB_UNR; rr++) {
                    const unsigned hit = __ballot_sync(FULL, w[rr] != 0);
                    if (hit && ksplit < 0) {
                        const int src = __ffs(hit) - 1;
                        ksplit = kb + 32 * rr + src;
                        which = __shfl_sync(FULL, w[rr], src);
                    }
                }
            }
            if (ksplit < 0) { failed = true; break; }
            const int i1 = (which == 2 || which == 4) ? i + 2 : i + 1;
            const int j1 = (which == 3 || which == 4) ? j - 2 : j - 1;
            PUSH(i1, ksplit, 1);
            PUSH(ksplit + 1, j1, 1);
            break;
        }
    }
#undef PUSH
    __syncwarp();
    if (failed) {
        if (lane == 0) { atomicExch(b.fail_flag, 1); b.tb_len[g] = 0; b.tb_start[g] = start; b.tb_locus[g] = l; }
        return;
    }
    // finalise (Lfold.c:765-768): C string ends at first NUL; strip trailing '-'; '-' -> '.'
    int len0 = b.slot_stride;
    for (int kb = 0; kb < b.slot_stride; kb += 32) {
        const int k = kb + lane;
        const unsigned z = __ballot_sync(FULL, k < b.slot_stride && st[k] == 0);
        if (z) { len0 = kb + __ffs(z) - 1; break; }
    }
    int last = 0;  // last index with a non-dash char (index 0 is never stripped)
    for (int kb = 0; kb < len0; kb += 32) {
        const int k = kb + lane;
        const unsigned nz = __ballot_sync(FULL, k < len0 && st[k] != '-');
        if (nz) last = max(last, kb + 31 - __clz(nz));
    }
    const int len = last + 1;
    for (int k = lane; k < b.slot_stride; k += 32) {
        if (k < len) { if (st[k] == '-') st[k] = '.'; }
        else st[k] = 0;
    }
    if (lane == 0) { b.tb_len[g] = len; b.tb_start[g] = start; b.tb_locus[g] = l; }
}

cudaError_t launch_traceback(const TraceBuffers &b, cudaStream_t st)
{
    if (b.ntb == 0) return cudaSuccess;
    const unsigned long long blocks = (b.ntb + 3) / 4;
    k_traceback<<<(unsigned)blocks, 128, 4 * (size_t)b.code_win, st>>>(b);   // code_win <= 4112: below the 48 KB default
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ emit
// one warp per traceback: decide whether RNALfold prints it (A.5)
__global__ void __launch_bounds__(128) k_emit(TraceBuffers b)
{
    const unsigned long long g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= b.ntb) return;
    const int l = b.tb_locus[g];
    const LocusDesc L = b.loci[l];
    const int kidx = (int)(g - b.tb_base[l]), cnt = b.tb_count[l];
    const int start = b.tb_start[g], len = b.tb_len[g];
    const int *F = b.F + L.seq_off;
    bool printed;
    const bool last_is_final = (b.tb_start[b.tb_base[l] + cnt - 1] == 1);
    const int last_regular = last_is_final ? cnt - 2 : cnt - 1;
    if (kidx >= last_regular) printed = true;   // last "prev" at i==1, and the final backtrack(1,L*)
    else {
        // next traceback (ss) against this one (prev): prev_i = start, i = start_next - 1
        const unsigned long long gn = g + 1;
        const int i = b.tb_start[gn] - 1, ls = b.tb_len[gn];
        const char *ss = b.slots + gn * (unsigned long long)b.slot_stride;
        const char *prev = b.slots + g * (unsigned long long)b.slot_stride;
        if (i + ls < start + len) printed = true;
        else {
            const int off = start - i;
            bool diff = false;
            for (int kb = 0; kb < len && !diff; kb += 32) {
                const int k = kb + lane;
                const bool dneq = (k < len) && (ss[off + k] != prev[k]);
                diff = __any_sync(FULL, dneq);
            }
            printed = diff;
        }
    }
    if (lane == 0) {
        b.tb_flag[g] = printed ? 1 : 0;
        const int a = F[start];
        const int e2 = (start + len <= L.n + 2) ? F[start + len] : 0;
        b.tb_energy[g] = a - e2;
    }
}

cudaError_t launch_emit(const TraceBuffers &b, cudaStream_t st)
{
    if (b.ntb == 0) return cudaSuccess;
    const unsigned long long blocks = (b.ntb + 3) / 4;
    k_emit<<<(unsigned)blocks, 128, 0, st>>>(b);
    return cudaGetLastError();
}

// k_emit over one segment of a segmented locus.  Its tracebacks are, in print order, the one carried over from the segment
// above (n_carry = 1: entry 0, start already absolute, traced there) and the segment's own (starts relative to the
// segment's suffix, which begins after base `shift`).  Every entry is decided against the next one; the last entry of a
// segment that is not the last waits for the first traceback of the segment below (the host carries it over and it is
// not printed here).  In the last segment the final entries are printed as k_emit prints them.  Writes the absolute start
// of every entry to abs_start (k_pack's tb_start); F is the whole locus' f3, n its length.
__global__ void __launch_bounds__(128) k_emit_seg(TraceBuffers b, int n_carry, int shift, int last, const int *__restrict__ F, int n,
                                                  int *__restrict__ abs_start)
{
    const unsigned long long g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= b.ntb) return;
    const unsigned long long ntb = b.ntb;
    auto start_of = [&](unsigned long long k) { return b.tb_start[k] + (k < (unsigned long long)n_carry ? 0 : shift); };
    const int start = start_of(g), len = b.tb_len[g];
    bool printed;
    const int last_regular = (int)ntb - ((start_of(ntb - 1) == 1) ? 2 : 1);
    if (last && (long long)g >= last_regular) printed = true;   // last "prev" at i==1, and the final backtrack(1,L*)
    else if (g + 1 == ntb) printed = false;                       // carried: decided in the segment below
    else {
        const unsigned long long gn = g + 1;
        const int i = start_of(gn) - 1, ls = b.tb_len[gn];
        const char *ss = b.slots + gn * (unsigned long long)b.slot_stride;
        const char *prev = b.slots + g * (unsigned long long)b.slot_stride;
        if (i + ls < start + len) printed = true;
        else {
            const int off = start - i;
            bool diff = false;
            for (int kb = 0; kb < len && !diff; kb += 32) {
                const int k = kb + lane;
                const bool dneq = (k < len) && (ss[off + k] != prev[k]);
                diff = __any_sync(FULL, dneq);
            }
            printed = diff;
        }
    }
    if (lane == 0) {
        b.tb_flag[g] = printed ? 1 : 0;
        const int e2 = (start + len <= n + 2) ? F[start + len] : 0;
        b.tb_energy[g] = F[start] - e2;
        abs_start[g] = start;
    }
}

cudaError_t launch_emit_seg(const TraceBuffers &b, int n_carry, int shift, int last, const int *F, int n, int *abs_start, cudaStream_t st)
{
    if (b.ntb == 0) return cudaSuccess;
    const unsigned long long blocks = (b.ntb + 3) / 4;
    k_emit_seg<<<(unsigned)blocks, 128, 0, st>>>(b, n_carry, shift, last, F, n, abs_start);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ pack
__global__ void __launch_bounds__(128) k_pack(TraceBuffers b, const unsigned long long *__restrict__ ss_off,
                                              const unsigned long long *__restrict__ hit_idx, char *__restrict__ arena,
                                              mirfold_hit *__restrict__ out_hits, unsigned long long arena_base)
{
    const unsigned long long g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= b.ntb || !b.tb_flag[g]) return;
    const int len = b.tb_len[g];
    const char *src = b.slots + g * (unsigned long long)b.slot_stride;
    char *dst = arena + ss_off[g];
    for (int k = lane; k <= len; k += 32) dst[k] = k < len ? src[k] : 0;
    if (lane == 0) {
        // the finished public record (include/mirfold.h): the host only copies the table
        mirfold_hit h;
        h.start = b.tb_start[g]; h.len = len; h.mfe_dcal = b.tb_energy[g]; h.reserved = 0;
        h.ss_off = arena_base + ss_off[g];
        out_hits[hit_idx[g]] = h;
    }
}

cudaError_t launch_pack(const TraceBuffers &b, const unsigned long long *ss_off, const unsigned long long *hit_idx,
                        char *arena, mirfold_hit *out_hits, unsigned long long arena_base, cudaStream_t st)
{
    if (b.ntb == 0) return cudaSuccess;
    const unsigned long long blocks = (b.ntb + 3) / 4;
    k_pack<<<(unsigned)blocks, 128, 0, st>>>(b, ss_off, hit_idx, arena, out_hits, arena_base);
    return cudaGetLastError();
}
