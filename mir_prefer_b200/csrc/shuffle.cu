// shuffle.cu -- shuffled copies of records for the MFE significance test (mirfold_shuffle_test, randfold's test:
// Bonnet et al. 2004).  One thread per (record, replicate); a shuffle costs O(n) against the O(n * L) fold it feeds.
//
// Shuffles act on the sequence as it is folded (upper-case, T -> U: RNALfold's conversion, which k_prepare applies
// again harmlessly); every distinct byte is a symbol, so N and IUPAC letters move like any base.
//   * mononucleotide: Fisher-Yates over the positions (i = n-1 .. 1 swaps i with a draw in [0, i]).
//   * dinucleotide: Altschul-Erickson by the random-arborescence construction (Kandel et al. 1996; uShuffle, k = 2).
//     The multigraph has one edge s[t] -> s[t+1] per position.  Every symbol but the last one gets a "last out-edge" so
//     that these edges form a tree directed at the last symbol, drawn uniformly over the edge instances' arborescences;
//     every symbol's other out-edges are put in Fisher-Yates order, and the walk from the first symbol that takes each
//     symbol's out-edges in that order (its last edge last) spells the shuffle.  It keeps every dinucleotide count and
//     the first and last symbols, and is uniform over the sequences that do.  The tree is drawn with Wilson's
//     loop-erased random walk, which has the same distribution as drawing every symbol's last edge independently and
//     retrying until they form a tree, but does not need ~prod(out-degree) retries on block-structured sequences such
//     as A^200 C^200 G^200 U^200.
// Random draws come from shuffle_rng.cuh in this order: Wilson's walks from symbols 0, 1, ... (symbols numbered by
// first occurrence), then each symbol's Fisher-Yates in symbol order.
#include "mirfold_internal.cuh"
#include "shuffle_rng.cuh"

__device__ __forceinline__ unsigned char fold_letter(char c)
{
    if (c >= 'a' && c <= 'z') c -= 32;
    return (unsigned char)(c == 'T' ? 'U' : c);
}

__device__ void shuffle_mono(const char *src, int n, unsigned char *dst, uint64_t st)
{
    for (int t = 0; t < n; t++) dst[t] = fold_letter(src[t]);
    for (int i = n - 1; i >= 1; i--) {
        const int j = (int)mf_shuf_below(st, (uint32_t)i + 1);
        const unsigned char x = dst[i];
        dst[i] = dst[j];
        dst[j] = x;
    }
}

// scr: n bytes of edge lists; returns false for more than MF_SHUF_MAX_SYMBOLS distinct symbols
__device__ bool shuffle_di(const char *src, int n, unsigned char *dst, unsigned char *scr, uint64_t st)
{
    unsigned char sym[MF_SHUF_MAX_SYMBOLS];
    int ns = 0;
    for (int t = 0; t < n; t++) {   // symbol index of every position, kept in dst until the walk
        const unsigned char c = fold_letter(src[t]);
        int u = 0;
        while (u < ns && sym[u] != c) u++;
        if (u == ns) {
            if (ns == MF_SHUF_MAX_SYMBOLS) return false;
            sym[ns++] = c;
        }
        dst[t] = (unsigned char)u;
    }
    if (n <= 2) {   // one Eulerian path
        for (int t = 0; t < n; t++) dst[t] = sym[dst[t]];
        return true;
    }
    int deg[MF_SHUF_MAX_SYMBOLS], beg[MF_SHUF_MAX_SYMBOLS], pos[MF_SHUF_MAX_SYMBOLS], nxt[MF_SHUF_MAX_SYMBOLS];
    bool tree[MF_SHUF_MAX_SYMBOLS];
    for (int u = 0; u < ns; u++) { deg[u] = 0; pos[u] = 0; tree[u] = false; }
    for (int t = 0; t + 1 < n; t++) deg[dst[t]]++;
    for (int u = 0, acc = 0; u < ns; u++) { beg[u] = acc; acc += deg[u]; }
    for (int t = 0; t + 1 < n; t++) { const int u = dst[t]; scr[beg[u] + pos[u]++] = dst[t + 1]; }   // in order of occurrence
    const int first = dst[0], last = dst[n - 1];
    tree[last] = true;
    for (int u = 0; u < ns; u++) {   // Wilson: every symbol but the last has an out-edge, so each walk reaches the tree
        int x = u;
        while (!tree[x]) { nxt[x] = (int)mf_shuf_below(st, (uint32_t)deg[x]); x = scr[beg[x] + nxt[x]]; }
        x = u;
        while (!tree[x]) { tree[x] = true; x = scr[beg[x] + nxt[x]]; }
    }
    for (int u = 0; u < ns; u++) {
        unsigned char *e = scr + beg[u];
        int m = deg[u];
        if (u != last) {   // the tree edge goes last
            const unsigned char x = e[nxt[u]];
            e[nxt[u]] = e[m - 1];
            e[m - 1] = x;
            m--;
        }
        for (int i = m - 1; i >= 1; i--) {
            const int j = (int)mf_shuf_below(st, (uint32_t)i + 1);
            const unsigned char x = e[i];
            e[i] = e[j];
            e[j] = x;
        }
        pos[u] = 0;
    }
    int cur = first;
    dst[0] = sym[first];
    for (int t = 1; t < n; t++) {
        cur = scr[beg[cur] + pos[cur]++];
        dst[t] = sym[cur];
    }
    return true;
}

__global__ void k_shuffle(const char *__restrict__ in, const unsigned long long *__restrict__ in_off,
                          const ShuffleItem *__restrict__ items, unsigned int nitems, char *__restrict__ out,
                          unsigned char *__restrict__ scr, unsigned long long seed, int mode, int *__restrict__ fail)
{
    const unsigned int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nitems) return;
    const ShuffleItem it = items[t];
    const unsigned long long b = in_off[it.rec];
    const int n = (int)(in_off[it.rec + 1] - b);
    const uint64_t st = mf_shuf_state(seed, it.rec, it.rep);
    unsigned char *dst = (unsigned char *)out + it.dst;
    if (mode == MF_SHUFFLE_MONO) shuffle_mono(in + b, n, dst, st);
    else if (!shuffle_di(in + b, n, dst, scr + it.dst, st)) atomicExch(fail, 1);
}

cudaError_t launch_shuffle(const char *in, const unsigned long long *in_off, const ShuffleItem *items, unsigned int nitems,
                           char *out, unsigned char *scr, unsigned long long seed, int mode, int *fail, cudaStream_t st)
{
    if (nitems == 0) return cudaSuccess;
    k_shuffle<<<(nitems + 127) / 128, 128, 0, st>>>(in, in_off, items, nitems, out, scr, seed, mode, fail);
    return cudaGetLastError();
}
