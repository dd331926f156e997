// host.cu -- libmirfold host runtime: contexts, memory pools, the two-lane chunk pipeline, multi-GPU
// sharding and the fold entry points of the C ABI declared in include/mirfold.h.
//
// Replaces fold_use_RNALfold()/fold() (/root/reference/miR_PREFeR.py:3047-3119): where the reference
// forks one RNALfold process per FASTA shard and folds it 2*CHECKPOINT_SIZE lines at a time, this
// runtime shards records over GPUs by DP work (no collectives: loci are independent), cuts every
// shard into chunks and keeps two chunks in flight per device on two "lanes" (complete buffer sets):
// while one lane runs f3 / traceback / pack / download of chunk k on a high-priority stream, the other
// lane's band fill of chunk k+1 already occupies the SMs the last wave of chunk k left idle.  Results
// are downloaded straight into buffers shared by all devices of the call (no merge pass) or handed
// to a callback chunk by chunk (mirfold_fold_stream).  There is no CPU fallback.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "../../include/mirfold.h"
#include "mirfold_internal.cuh"
#include "shuffle_rng.cuh"

#define MIRFOLD_VERSION "0.2.0"

void build_params(DevParams &P);   // params.cu

namespace {

struct DBuf {  // grow-only device buffer
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

struct HBuf {  // grow-only pinned host buffer
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

struct Locus {
    uint32_t rec;
    int n;
    uint64_t cells;
};

// host-side description of one chunk on a lane
struct Prep {
    size_t cb = 0, ce = 0;   // [cb, ce) into the device's locus list
    int nl = 0, nu = 0, max_n = 0, max_Ls = 0, n_long = 0;
    int bucket_first[6] = {0, 0, 0, 0, 0, 0};
    unsigned long long seq_acc = 0, band_acc = 0, raw_acc = 0, list_acc = 0, ring_acc = 0;
};

struct OverflowChunk {   // a chunk that did not fit the shared result buffers (capacity is an estimate)
    HBuf hits, arena;
    ~OverflowChunk() { hits.release(); arena.release(); }
    uint64_t nhits = 0, abytes = 0;
    std::vector<uint32_t> recs, count;
    std::vector<uint64_t> begin;
};

// Lane::ev: the events a chunk (or a segment) records, in stream order; side fork / join are launch_fill's
enum { EV_H2D, EV_KERNELS, EV_FILL, EV_FILL_END, EV_F3_END, EV_PACK_END, EV_D2H_END, EV_SIDE_FORK, EV_SIDE_JOIN, EV_COUNT };
// Lane::h_small: what a lane downloads before a host sync -- tracebacks (plan), printed bytes and hits (emission), the fail
// flag (an int) and, for SINK_CAND, the candidate structures, their verdicts and string bytes
enum { HS_NTB, HS_ABYTES, HS_NHITS, HS_FAIL, HS_NSTRUCTS, HS_NVERDICTS, HS_SBYTES };

// A lane = one complete set of pipeline buffers and streams; a device alternates chunks between two lanes.
struct Lane {
    cudaStream_t s_lo = nullptr;   // uploads, encode, band fill
    cudaStream_t s_hi = nullptr;   // f3, plan, traceback, pack, downloads (high priority: gets freed SM slots first)
    cudaStream_t side = nullptr;   // small fill buckets run here, concurrently with the big one
    DBuf units, raw, loci, codes, F, C, M, Mp, Ib, ring, fillflags, tbcount, tbbase, listoff, startlist, scan_in, scan_out, scan_tmp;
    DBuf slots, tblen, tbstart, tblocus, tbflag, tbenergy, stackscr, fail, ssoff, hitidx;
    DBuf segstate;   // segmented loci: the emission plan's state carried from segment to segment (k_plan_seg)
    DBuf o_hits, o_arena, bounds, totals;
    DBuf c_counts, c_soff, c_structs, c_nq, c_sbytes, c_voff, c_aoff, c_lsb, c_verd, c_vmat, c_arena, c_sout;   // fused stage 1 + 3
    HBuf hc_structs, hc_arena, hc_verd, hc_vmat, hc_voff, hc_lsb;
    uint64_t c_ns = 0, c_nv = 0, c_nb = 0;
    HBuf h_raw, h_loci, h_units, h_listoff, h_small, h_hits, h_arena;
    HBuf h_out;   // the chunk's per-locus tables: nl + 1 first-hit bounds (u64), then nl totals (int)
    cudaEvent_t ev[EV_COUNT] = {};
    // chunk in flight
    bool pending = false;
    Prep prep;
    TraceBuffers tb{};
    uint64_t nhits = 0, abytes = 0, hit_base = 0, arena_base = 0;
    std::unique_ptr<OverflowChunk> ovf;
    std::vector<uint32_t> s_rec, s_count;   // stream sink: per-record tables handed to the callback
    std::vector<uint64_t> s_begin;
    std::vector<int32_t> s_total;
    cudaError_t create(int prio_hi)
    {
        cudaError_t e = cudaStreamCreateWithFlags(&s_lo, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s_hi, cudaStreamNonBlocking, prio_hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking);
        for (auto &x : ev) if (e == cudaSuccess) e = cudaEventCreate(&x);
        return e;
    }
    void release()
    {
        DBuf *all[] = {&units, &raw, &loci, &codes, &F, &C, &M, &Mp, &Ib, &ring, &fillflags, &tbcount, &tbbase, &listoff, &startlist, &scan_in,
                       &scan_out, &scan_tmp, &slots, &tblen, &tbstart, &tblocus, &tbflag, &tbenergy, &stackscr, &fail,
                       &ssoff, &hitidx, &o_hits, &o_arena, &bounds, &totals, &c_counts, &c_soff, &c_structs, &c_nq, &c_sbytes,
                       &c_voff, &c_aoff, &c_lsb, &c_verd, &c_vmat, &c_arena, &c_sout, &segstate};
        for (DBuf *b : all) b->release();
        HBuf *hall[] = {&h_raw, &h_loci, &h_units, &h_listoff, &h_small, &h_out, &h_hits, &h_arena, &hc_structs, &hc_arena, &hc_verd,
                        &hc_vmat, &hc_voff, &hc_lsb};
        for (HBuf *b : hall) b->release();
        for (auto &e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        if (s_lo) cudaStreamDestroy(s_lo);
        if (s_hi) cudaStreamDestroy(s_hi);
        if (side) cudaStreamDestroy(side);
        s_lo = s_hi = side = nullptr;
    }
};

struct Device {
    int id = 0;
    DevParams *dP = nullptr;
    size_t mem_budget = 0;
    Lane lane[2];
    cudaEvent_t ev_first = nullptr, ev_last = nullptr;
    DBuf duplex_arena, duplex_q, duplex_v;   // mirfold_duplex scratch
    DBuf cand_regions, cand_matures, cand_moff;   // the call's records (mirfold_fold_candidates)
    DBuf shuf_in, shuf_off, shuf_items, shuf_raw, shuf_scr, shuf_fail;   // mirfold_shuffle_test: records, one round's replicates
    void release()
    {
        lane[0].release(); lane[1].release();
        duplex_arena.release(); duplex_q.release(); duplex_v.release();
        cand_regions.release(); cand_matures.release(); cand_moff.release();
        shuf_in.release(); shuf_off.release(); shuf_items.release(); shuf_raw.release(); shuf_scr.release(); shuf_fail.release();
        if (ev_first) cudaEventDestroy(ev_first);
        if (ev_last) cudaEventDestroy(ev_last);
        ev_first = ev_last = nullptr;
        if (dP) cudaFree(dP);
        dP = nullptr;
    }
};

}  // namespace

struct mirfold_ctx {
    std::vector<Device> devs;
    std::string last_error;
    std::vector<HBuf> arena_pool;  // pinned arenas returned by mirfold_free_result
    std::vector<HBuf> hits_pool;   // pinned hit tables returned by mirfold_free_result
    std::mutex pool_mu;
    int live_results = 0;          // results not yet freed (guarded by pool_mu)
    int live_genomes = 0;          // genomes not yet freed (guarded by pool_mu)
    bool closed = false;           // mirfold_close() was called; the last mirfold_free_result / mirfold_genome_free deletes the context
    double arena_per_nt = 30.0;    // capacity estimates of the shared result buffers, raised when a call overflows them
    double hits_per_nt = 0.20;
};

struct mirfold_batch {
    mirfold_ctx *ctx = nullptr;
    uint32_t nseq = 0;
    int span_L = 0;
    std::vector<uint64_t> h_off;                   // copy of the caller's offsets
    std::vector<std::vector<uint32_t>> shard;      // per device, descending DP cells
    std::vector<uint64_t> raw_off;                 // per record: offset inside its device's buffer
    std::vector<void *> d_raw;                     // per device
};

// A genome resident in HBM: one copy of the bases per distinct CUDA ordinal of the context.  The handle keeps its
// context's host bookkeeping alive (live_genomes) and knows its own ordinals, so it may be freed before or after
// mirfold_close().
struct mirfold_genome {
    mirfold_ctx *ctx = nullptr;
    std::vector<uint64_t> contig_off;    // n_contigs + 1, from 0
    std::vector<int> ordinal;            // distinct CUDA ordinals ...
    std::vector<void *> replica;         // ... and the copy of the bases on each
    std::vector<void *> d_raw;           // per device entry of the context (entries of one ordinal share its replica)
    std::vector<size_t> budget_taken;    // per device entry: bytes taken off Device::mem_budget while the genome lives
};

namespace {

struct ResultOwner {  // lives right behind the public struct
    mirfold_result pub;
    mirfold_ctx *ctx;
    std::vector<uint64_t> hit_begin;
    std::vector<uint32_t> hit_count;
    std::vector<int32_t> totals;
    HBuf hits, arena;   // pinned, written directly by the devices' downloads
};

// result buffers shared by all devices of one mirfold_fold call
struct SharedOut {
    HBuf hits, arena;
    uint64_t hits_cap = 0, arena_cap = 0;     // records / bytes
    uint64_t hits_used = 0, arena_used = 0;
    std::mutex mu;
    std::vector<std::unique_ptr<OverflowChunk>> overflow;
    uint64_t *hit_begin = nullptr;
    uint32_t *hit_count = nullptr;
    int32_t *totals = nullptr;
    bool reserve(uint64_t nh, uint64_t ab, uint64_t &hb, uint64_t &abase)
    {
        std::lock_guard<std::mutex> lk(mu);
        if (hits_used + nh > hits_cap || arena_used + ab > arena_cap) return false;
        hb = hits_used; abase = arena_used;
        hits_used += nh; arena_used += ab;
        return true;
    }
};

// SINK_TOTALS: the totals-only pass of mirfold_shuffle_test -- prepare, fill and f3, then only F[seq_off + 1] per locus
// (4 bytes) leaves the device; no emission plan, traceback or pack
enum { SINK_NONE = 0, SINK_SHARED = 1, SINK_STREAM = 2, SINK_CAND = 3, SINK_TOTALS = 4 };

// fused stage 1 + 3: what the chunks of all devices append to (small: a few percent of the hit text)
struct CandCollector {
    std::mutex mu;
    std::vector<mirfold_structure> structs;
    std::vector<char> arena;
    std::vector<mirfold_duplex_verdict> verdicts;
    std::vector<uint32_t> verdict_mature, struct_count, verdict_count;
    std::vector<uint64_t> struct_begin, verdict_begin;
};
struct CandArgs {
    const mirfold_region *regions = nullptr;
    const mirfold_mature *matures = nullptr;
    const uint64_t *mature_off = nullptr;
    uint32_t nseq = 0;
    int minlen = 55, minloop = 3, min_mature = 18, max_mature = 24;
};

struct Job {   // one fold call; shared read-only by the device threads (sinks are synchronised)
    const char *seqs = nullptr;
    const uint64_t *h_off = nullptr;
    int L = 0;
    bool force_wide = false;
    bool serial = false;               // MIRFOLD_FLAG_SERIAL: one lane
    int sink = SINK_NONE;
    SharedOut *shared = nullptr;
    mirfold_chunk_fn fn = nullptr;
    void *user = nullptr;
    std::mutex *cb_mu = nullptr;
    std::atomic<int> *cb_abort = nullptr;
    const CandArgs *cand = nullptr;
    CandCollector *collect = nullptr;
    int32_t *totals = nullptr;         // SINK_TOTALS: per record of the call
};

struct DevOut {
    mirfold_stats st{};
    uint64_t nhits = 0, arena_bytes = 0;
    int err = MIRFOLD_OK;
    std::string errmsg;
};

// host-side phase log (MIRFOLD_HOST_TIMING=1): where the wall time outside the kernels goes
struct HostTimer {
    std::chrono::steady_clock::time_point t;
    bool on;
    HostTimer() : t(std::chrono::steady_clock::now()) { static const bool e = getenv("MIRFOLD_HOST_TIMING") != nullptr; on = e; }
    void mark(const char *what)
    {
        if (!on) return;
        const auto n = std::chrono::steady_clock::now();
        fprintf(stderr, "[mirfold host] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};

int env_opts()
{
    static const int v = getenv("MIRFOLD_OPTS") ? atoi(getenv("MIRFOLD_OPTS")) : 0;
    return v;
}

uint64_t cells_of(int64_t n, int L)
{   // SURVEY 8(d): sum_{i=1}^{n-4} (min(n, i+L*) - i - 3); rows with i+L* <= n contribute L*-3, the rest n-i-3
    if (n < 5) return 0;
    const int64_t Ls = std::min<int64_t>(L, n);
    const int64_t full = std::max<int64_t>(0, std::min(n - 4, n - Ls));
    const int64_t m = n - 4 - full;
    return (uint64_t)(full * (Ls - 3) + m * (m + 1) / 2);
}

// ---- shard plan (SURVEY 8e): records in descending DP cells (== descending length for a fixed span, ties by
// record index), greedy longest-processing-time assignment.  Every shard list stays in that order, which is
// also the order the device's CTA scheduler wants (largest first).
void plan_shards(const uint64_t *off, uint32_t nseq, int L, int G, std::vector<std::vector<uint32_t>> &shard, std::vector<uint64_t> &load)
{
    shard.assign((size_t)G, {});
    load.assign((size_t)G, 0);
    if (nseq == 0) return;
    std::vector<uint32_t> order(nseq);
    uint64_t maxn = 0;
    for (uint32_t r = 0; r < nseq; r++) maxn = std::max(maxn, off[r + 1] - off[r]);
    if (maxn <= 4ull * nseq + 65536) {   // counting sort by length, stable in the record index
        std::vector<uint32_t> cnt((size_t)maxn + 2, 0);
        for (uint32_t r = 0; r < nseq; r++) cnt[(size_t)(maxn - (off[r + 1] - off[r])) + 1]++;
        for (size_t k = 1; k < cnt.size(); k++) cnt[k] += cnt[k - 1];
        for (uint32_t r = 0; r < nseq; r++) order[cnt[(size_t)(maxn - (off[r + 1] - off[r]))]++] = r;
    } else {
        for (uint32_t r = 0; r < nseq; r++) order[r] = r;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return off[a + 1] - off[a] > off[b + 1] - off[b]; });
    }
    if (G == 1) {
        for (uint32_t r : order) load[0] += cells_of((int64_t)(off[r + 1] - off[r]), L) + 1;
        shard[0].swap(order);
        return;
    }
    for (auto &s : shard) s.reserve(nseq / G + 16);
    for (uint32_t r : order) {
        int g = 0;
        for (int k = 1; k < G; k++) if (load[k] < load[g]) g = k;
        shard[g].push_back(r);
        load[g] += cells_of((int64_t)(off[r + 1] - off[r]), L) + 1;
    }
}

#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            out.err = e_ == cudaErrorMemoryAllocation ? MIRFOLD_ERR_NOMEM : MIRFOLD_ERR_CUDA;    \
            out.errmsg = std::string(#call) + ": " + cudaGetErrorString(e_);                     \
            cudaGetLastError();                                                                  \
            return false;                                                                        \
        }                                                                                        \
    } while (0)

__global__ void k_widen_counts(const int *__restrict__ in, unsigned long long *__restrict__ out, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= n) out[k] = k < n ? (unsigned long long)in[k] : 0ULL;
}
__global__ void k_emit_sizes(const int *__restrict__ flag, const int *__restrict__ len,
                             unsigned long long *__restrict__ bytes, unsigned long long *__restrict__ ones,
                             unsigned long long ntb)
{
    const unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= ntb) {
        const bool f = k < ntb && flag[k];
        bytes[k] = f ? (unsigned long long)len[k] + 1ULL : 0ULL;
        ones[k] = f ? 1ULL : 0ULL;
    }
}
// per-locus first-hit index = hitidx[tb_base[l]] and total line F[seq_off + 1]
__global__ void k_gather_bounds(const unsigned long long *tb_base, const unsigned long long *hitidx, const LocusDesc *loci,
                                const int *F, unsigned long long *out, int *totals, int nl)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= nl) out[k] = hitidx[tb_base[k]];
    if (k < nl) totals[k] = F[loci[k].seq_off + 1];
}
__global__ void k_gather_totals(const LocusDesc *loci, const int *F, int *totals, int nl)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nl) totals[k] = F[loci[k].seq_off + 1];
}

cudaError_t exclusive_scan(Lane &Ln, const unsigned long long *in, unsigned long long *out, size_t n, cudaStream_t st)
{
    size_t tmp = 0;
    cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, n, st);
    if (e != cudaSuccess) return e;
    e = Ln.scan_tmp.ensure(tmp);
    if (e != cudaSuccess) return e;
    return cub::DeviceScan::ExclusiveSum(Ln.scan_tmp.p, tmp, in, out, n, st);
}

// the band fill of the nu units in Ln.units (sorted into buckets as bucket_first says) on the lane's buffers, at span L
FillLaunch fill_launch(const Lane &Ln, const DevParams *dP, int nu, int max_n, const int bucket_first[6], bool force_wide, int L)
{
    FillLaunch fa{Ln.units.as<LocusDesc>(), nu, max_n, Ln.codes.as<unsigned char>(), Ln.C.as<int>(), Ln.M.as<int>(), Ln.ring.as<int>(),
                  Ln.Ib.as<unsigned char>(), Ln.Mp.as<unsigned int>(), dP, {0, 0, 0, 0, 0, 0}, Ln.fillflags.as<int>(), force_wide ? 1 : 0,
                  env_opts() | (L >= MF_DYNW_MIN_SPAN ? 8 : 0)};
    for (int b = 0; b < 6; b++) fa.bucket_first[b] = bucket_first[b];
    return fa;
}

// Band shape of one locus: stride bucket or, for a longer locus with a span that leaves at least
// MF_TILE_MIN_STEP owned rows per tile, overlapping tiles for the shared-memory kernels.  A tile owns TL - dmax of
// its TL rows, so spans from big_tile_min_span() on use the 864 bucket: at L = 500 a 608-nt tile owns 108 rows (the
// locus' cells are computed 3.3 times over), an 864-nt tile 364 (1.7 times); at L = 300 it is 1.49 against 1.27.  Loci
// of 609..864 nt are then one untiled unit of that bucket.  The 864 kernel is one CTA per SM and 13 % (L = 300) to
// 35 % (L = 500) slower per executed cell than the 608 kernel (two CTAs per SM hide each other's barriers), so narrower
// spans keep the 608-nt tiles.  Measured same-box (profiles/r02_v7_bigtile_ab.txt): long loci -6.6 % at L = 300, -29 % at L = 500.
// Returns the band elements (per int32 array) the locus occupies.
#define MF_TILE_MIN_STEP 64
#ifndef MF_BIG_TILE_MIN_SPAN
#define MF_BIG_TILE_MIN_SPAN 300
#endif
static int big_tile_min_span()
{
    static const int v = [] { const char *e = getenv("MIRFOLD_BIG_TILE_MIN_SPAN"); return e ? atoi(e) : MF_BIG_TILE_MIN_SPAN; }();   // A/B runs; a huge value disables the 864 bucket
    return v;
}
unsigned long long shape_locus(LocusDesc &d, int n, int L)
{
    d.n = n; d.Ls = std::min(L, n); d.dmax = std::min(d.Ls, n - 1);
    d.tile_last = 0; d.tile_step = 1 << 30; d.tile_rcp = 0;
    static const bool no_tiles = getenv("MIRFOLD_NO_TILES") != nullptr;   // A/B runs: long loci through k_fill_generic
    const bool big = n > MF_TILE_LEN && d.dmax >= big_tile_min_span() && !no_tiles &&
                     (n <= MF_TILE_LEN_BIG || MF_TILE_LEN_BIG - d.dmax >= MF_TILE_MIN_STEP);
    d.stride = band_stride_for(n, big);
    const int TL = big ? MF_TILE_LEN_BIG : MF_TILE_LEN;
    if (n > TL && d.dmax >= 4 && TL - d.dmax >= MF_TILE_MIN_STEP && !no_tiles) {
        const int S = TL - d.dmax;
        d.stride = TL;
        d.tile_step = S;
        d.tile_last = (n - TL + S - 1) / S;
        d.tile_rcp = (unsigned int)((0x100000000ULL + (unsigned long long)S - 1) / (unsigned long long)S);
        return (unsigned long long)(d.tile_last + 1) * band_elems(TL, d.dmax);
    }
    return band_elems(d.stride, d.dmax);
}
// ring scratch of one fill unit: the DML ring; a generic unit adds its Cm ring and room for the kernel's scratch, which
// k_fill_generic keeps there when it does not fit shared memory (rounded to 128 B so that the next unit's rings stay aligned)
unsigned long long unit_ring_elems(int stride)
{
    if (is_bucket_stride(stride)) return (unsigned long long)stride * MF_RING_DML;
    return (unsigned long long)stride * MF_RING_PER_STRIDE + (generic_scratch_bytes(stride) + 127) / 128 * 32;
}
// an untiled unit of 2^31 band cells or more overflows the kernels' 32-bit band offsets (MF_MAX_UNIT_BAND_CELLS)
static bool band_offsets_fit(const LocusDesc &d)
{
    return d.tile_last > 0 || band_elems(d.stride, d.dmax) < MF_MAX_UNIT_BAND_CELLS;
}
static int unit_bucket(const LocusDesc &u)   // index into FillLaunch::bucket_first
{
    return !is_bucket_stride(u.stride) ? 0 : u.stride == MF_TILE_LEN_BIG ? 1 : u.stride == MF_TILE_LEN ? 2 : u.stride == 352 ? 3 : 4;
}
// fill unit of tile t of a tiled locus: TL bases from a_t + 1, band at the locus' band_off + t tiles
LocusDesc tile_unit(const LocusDesc &d, int t)
{
    LocusDesc u = d;
    const int TL = d.stride;
    const int a = std::min(t * d.tile_step, d.n - TL);
    u.n = TL; u.Ls = std::min(d.Ls, TL); u.dmax = d.dmax;
    u.seq_off = d.seq_off + (unsigned long long)a;
    u.band_off = d.band_off + (unsigned long long)t * band_elems(TL, d.dmax);
    u.tile_last = 0;
    return u;
}
// Fill units of a chunk: one per untiled locus, one per tile otherwise, sorted by (bucket, descending n)
// so that the stride buckets are contiguous.  Assigns ring offsets; returns ring elements.
unsigned long long build_fill_units(const LocusDesc *loci, int nl, std::vector<LocusDesc> &units, int bucket_first[6], int &max_n)
{
    units.clear();
    max_n = 0;
    for (int k = 0; k < nl; k++) {
        const LocusDesc &d = loci[k];
        if (d.dmax < 4) continue;   // n < 5 never reaches here; keeps the kernels' assumptions explicit
        if (d.tile_last == 0) { units.push_back(d); continue; }
        for (int t = 0; t <= d.tile_last; t++) units.push_back(tile_unit(d, t));
    }
    std::stable_sort(units.begin(), units.end(), [](const LocusDesc &a, const LocusDesc &b) {
        const int ba = unit_bucket(a), bb = unit_bucket(b);
        return ba != bb ? ba < bb : a.n > b.n;
    });
    unsigned long long ring_acc = 0;
    int k = 0;
    const int nu = (int)units.size();
    bucket_first[0] = 0;
    for (int b = 0; b < 5; b++) {
        while (k < nu && unit_bucket(units[k]) <= b) k++;
        bucket_first[b + 1] = k;
    }
    for (auto &u : units) {
        u.ring_off = ring_acc;
        ring_acc += unit_ring_elems(u.stride);
        max_n = std::max(max_n, u.n);
    }
    return ring_acc;
}

// estimated device bytes of one traceback (slot, stack, per-traceback ints)
static size_t traceback_bytes(int n, int L)
{
    return (size_t)((std::min(L, n) + 8) & ~3) + (size_t)(std::min(L, n) / 4 + 16) * 8 + 64;
}
// device bytes one locus needs on a lane: band (C, M, Mp), ring, descriptors, sequence-sized arrays and an
// estimate of the per-traceback buffers (slots, stacks, per-traceback ints: about one traceback per 8 nt)
size_t locus_bytes(int n, int L)
{
    LocusDesc d{};
    const unsigned long long be = shape_locus(d, n, L);
    return (size_t)be * 13 + (size_t)(d.tile_last + 1) * unit_ring_elems(d.stride) * 4 +
           (size_t)(d.tile_last + 2) * sizeof(LocusDesc) + (size_t)n * 16 + (size_t)(n / 8 + 2) * traceback_bytes(n, L) + 4096;
}

// ---- segmented loci.  A tiled locus larger than the device budget is folded in segments from its 3' end: a segment owns
// the tiles [t0, t1] and also holds `halo` tiles above t1, those owning rows up to (its last owned row + L* + 1) -- what f3
// (row i reads only row i's owner tile) and a traceback from a start in its owned rows or the row above them can read.
// The sequence-sized arrays (codes, F, raw) stay whole; band, rings and traceback scratch are per segment.
struct SegPlan {
    int t0, t1, halo;      // owned tiles [t0, t1], tiles t1+1 .. t1+halo above
    int row_lo, row_hi;    // owned rows
    size_t bytes;          // device bytes while the segment runs (the locus' sequence-sized arrays included)
};
static int64_t tile_last_row(const LocusDesc &d, int t) { return t == d.tile_last ? d.n : (int64_t)(t + 1) * d.tile_step; }
static size_t segment_bytes(const LocusDesc &d, int L, int t0, int t1, int halo)
{
    const size_t tiles = (size_t)(t1 + halo - t0 + 1);
    const int64_t rows = tile_last_row(d, t1) - (int64_t)t0 * d.tile_step;
    return tiles * band_elems(d.stride, d.dmax) * 13 + tiles * unit_ring_elems(d.stride) * 4 + (tiles + 2) * sizeof(LocusDesc) +
           (size_t)d.n * 16 + (size_t)(rows / 8 + 2) * traceback_bytes(d.n, L) + 4096;
}
// Segments in the order they run (3' end first).  A locus that fits `budget` (or is one unit) is one segment; otherwise each
// segment takes as many owned tiles as fit, at least one.
void plan_segments(int n, int L, size_t budget, std::vector<SegPlan> &out)
{
    out.clear();
    LocusDesc d{};
    shape_locus(d, n, L);
    const size_t whole = locus_bytes(n, L);
    if (d.tile_last == 0 || whole <= budget) { out.push_back(SegPlan{0, d.tile_last, 0, 1, n, whole}); return; }
    for (int t1 = d.tile_last; t1 >= 0;) {
        const int64_t hi = tile_last_row(d, t1), reach = std::min<int64_t>(n, hi + d.Ls + 1);
        const int halo = (int)std::min<int64_t>((reach - 1) / d.tile_step, d.tile_last) - t1;
        int t0 = t1;
        while (t0 > 0 && segment_bytes(d, L, t0 - 1, t1, halo) <= budget) t0--;
        out.push_back(SegPlan{t0, t1, halo, t0 * d.tile_step + 1, (int)hi, segment_bytes(d, L, t0, t1, halo)});
        t1 = t0 - 1;
    }
}

// ------------------------------------------------------------------------------------------------------------
// One device's share of a fold call.
struct DevicePipeline {
    Device &D;
    const Job &J;
    const char *d_raw;            // != nullptr: raw sequences already on this device
    const uint64_t *raw_off;      // ... at these per-record offsets
    DevOut &out;
    std::vector<Locus> loci;      // descending DP cells
    struct Chunk { size_t begin, end; bool segmented; };
    std::vector<Chunk> chunks;
    int nlanes_ = 1;
    HostTimer ht;

    DevicePipeline(Device &D_, const Job &J_, const char *d_raw_, const uint64_t *raw_off_, DevOut &out_)
        : D(D_), J(J_), d_raw(d_raw_), raw_off(raw_off_), out(out_) {}

    bool run(const std::vector<uint32_t> &recs)
    {
        out.st = mirfold_stats{};
        out.st.n_devices = 1;
        CK(cudaSetDevice(D.id));
        const auto t0 = std::chrono::steady_clock::now();
        loci.reserve(recs.size());
        uint64_t total_cells = 0;
        for (uint32_t r : recs) {
            const uint64_t len = J.h_off[r + 1] - J.h_off[r];
            out.st.nt += len;
            if (len >= 5) {
                Locus l{r, (int)len, cells_of((int64_t)len, J.L)};
                loci.push_back(l);
                total_cells += l.cells;
            }
        }
        out.st.cells = total_cells;
        if (J.sink == SINK_CAND) {
            const CandArgs &c = *J.cand;
            const uint64_t nm = c.mature_off[c.nseq];
            CK(D.cand_regions.ensure(sizeof(mirfold_region) * (size_t)c.nseq + 16));
            CK(D.cand_matures.ensure(sizeof(mirfold_mature) * (size_t)nm + 16));
            CK(D.cand_moff.ensure(8 * ((size_t)c.nseq + 1)));
            CK(cudaMemcpy(D.cand_regions.p, c.regions, sizeof(mirfold_region) * (size_t)c.nseq, cudaMemcpyHostToDevice));
            if (nm) CK(cudaMemcpy(D.cand_matures.p, c.matures, sizeof(mirfold_mature) * (size_t)nm, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(D.cand_moff.p, c.mature_off, 8 * ((size_t)c.nseq + 1), cudaMemcpyHostToDevice));
            out.st.h2d_bytes += sizeof(mirfold_region) * (uint64_t)c.nseq + sizeof(mirfold_mature) * nm + 8 * ((uint64_t)c.nseq + 1);
        }
        plan_chunks(total_cells);
        out.st.n_chunks = (int32_t)chunks.size();
        ht.mark("plan chunks");
        const int nlanes = nlanes_ = (J.serial || chunks.size() < 2) ? 1 : 2;
        bool ok = true;
        if (!chunks.empty()) {
            CK(cudaEventRecord(D.ev_first, D.lane[0].s_lo));
            ok = chunks[0].segmented || front(D.lane[0], 0);
            for (size_t k = 0; ok && k < chunks.size(); k++) {
                Lane &Ln = D.lane[k % nlanes];
                const bool pre = k + 1 < chunks.size() && !chunks[k + 1].segmented;   // a segmented chunk has no front
                if (chunks[k].segmented) ok = fold_segmented(Ln, k) && (!pre || front(D.lane[(k + 1) % nlanes], k + 1));
                else {
                    if (nlanes == 2 && pre) ok = front(D.lane[(k + 1) % 2], k + 1);   // its fill overlaps everything below
                    ok = ok && middle(Ln) && back(Ln, k + 1 == chunks.size());
                    if (nlanes == 1 && ok && pre) ok = front(Ln, k + 1);
                }
                if (J.cb_abort && J.cb_abort->load()) { out.err = MIRFOLD_ERR_CALLBACK; out.errmsg = "chunk callback returned non-zero"; ok = false; }
            }
            for (int l = 0; ok && l < nlanes; l++) ok = retire(D.lane[l]);
        }
        if (!ok) {   // nothing may stay in flight into buffers the caller is about to drop
            cudaDeviceSynchronize();
            cudaGetLastError();
            D.lane[0].pending = D.lane[1].pending = false;
            D.lane[0].ovf.reset(); D.lane[1].ovf.reset();
            return false;
        }
        if (!chunks.empty()) {
            float ms = 0;
            cudaEventElapsedTime(&ms, D.ev_first, D.ev_last);
            out.st.ms_device = ms;
        }
        out.st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        return true;
    }

    // chunks of about equal device bytes, each within a lane's budget.  A chunk boundary costs about 1.2 ms of device time
    // (launch train, two host syncs, wave tails the other lane only partly fills: 25 k loci in 1 / 2 / 4 / 9 chunks = 106.0 /
    // 108.3 / 108.0 / 111.5 ms end to end; 200 k loci in 7 / 16 / 37 chunks = 855.0 / 849.2 / 855.4) while a download runs at 55 GB/s, so a shard is only cut further than memory
    // demands when it is long enough for the last chunk's download (the only one not overlapped) to matter
    void plan_chunks(uint64_t total_cells)
    {
        if (loci.empty()) return;
        static const double cells_per_chunk = getenv("MIRFOLD_CHUNK_CELLS") ? atof(getenv("MIRFOLD_CHUNK_CELLS")) : 6.0e8;
        std::vector<size_t> lb(loci.size());
        size_t total = 0;
        int last_n = -1; size_t last_b = 0;
        for (size_t k = 0; k < loci.size(); k++) {
            if (loci[k].n != last_n) { last_n = loci[k].n; last_b = locus_bytes(last_n, J.L); }
            lb[k] = last_b; total += last_b;
        }
        const size_t lane_budget = lane_bytes();
        size_t nch = (total + lane_budget - 1) / lane_budget;
        if (J.sink != SINK_NONE || nch > 1) nch = std::max<size_t>(nch, std::min<size_t>(64, (size_t)(total_cells / cells_per_chunk)));
        nch = std::max<size_t>(nch, 1);
        const size_t target = std::min(lane_budget, total / nch + 1);
        size_t b = 0, acc = 0;
        for (size_t k = 0; k < loci.size(); k++) {
            if (k > b && acc + lb[k] > target) { chunks.push_back({b, k, false}); b = k; acc = 0; }
            acc += lb[k];
        }
        chunks.push_back({b, loci.size(), false});
        // The download of a device's LAST chunk is the only one nothing overlaps (154 MB per device take 11.6 ms when eight GPUs
        // write into host memory at once): cut the last chunk 80 : 20 so that only the small tail's download is exposed.
        if (J.sink != SINK_NONE && J.sink != SINK_TOTALS) {
            const Chunk last = chunks.back();
            uint64_t cells = 0;
            for (size_t k = last.begin; k < last.end; k++) cells += loci[k].cells;
            if (cells > 100000000ull && last.end - last.begin >= 64) {
                uint64_t acc2 = 0;
                size_t cut = last.begin;
                while (cut < last.end && acc2 < cells - cells / 5) acc2 += loci[cut++].cells;
                if (cut > last.begin && cut < last.end) {
                    chunks.back().end = cut;
                    chunks.push_back({cut, last.end, false});
                }
            }
        }
        // a tiled locus over the device's whole budget (always a chunk of its own: it exceeds the target) runs in segments
        for (Chunk &c : chunks)
            if (c.end == c.begin + 1 && lb[c.begin] > D.mem_budget) {
                LocusDesc d{};
                shape_locus(d, loci[c.begin].n, J.L);
                c.segmented = d.tile_last > 0;
            }
    }

    size_t lane_bytes() const { return std::max<size_t>(D.mem_budget / (J.serial ? 1 : 2), 1); }

    // ---- front: descriptors, upload, encode, band fill, f3, emission plan (everything up to the first host sync)
    bool front(Lane &Ln, size_t ci)
    {
        if (!retire(Ln)) return false;
        Prep &P = Ln.prep;
        P = Prep{};
        P.cb = chunks[ci].begin; P.ce = chunks[ci].end;
        const int nl = P.nl = (int)(P.ce - P.cb);
        CK(Ln.h_loci.ensure(sizeof(LocusDesc) * nl));
        CK(Ln.h_listoff.ensure(sizeof(unsigned long long) * nl));
        LocusDesc *hl = Ln.h_loci.as<LocusDesc>();
        unsigned long long *hlo = Ln.h_listoff.as<unsigned long long>();
        for (int k = 0; k < nl; k++) {
            const Locus &l = loci[P.cb + k];
            LocusDesc &d = hl[k];
            d = LocusDesc{};
            const unsigned long long be = shape_locus(d, l.n, J.L);
            d.rec = (int)l.rec;
            d.seq_off = P.seq_acc; d.band_off = P.band_acc; d.ring_off = 0;
            d.raw_off = d_raw ? raw_off[l.rec] : P.raw_acc;
            hlo[k] = P.list_acc;
            P.seq_acc += (unsigned long long)l.n + 3;
            P.band_acc += be;
            P.raw_acc += (unsigned long long)l.n;
            P.list_acc += (unsigned long long)l.n / 2 + 2;
            P.max_Ls = std::max(P.max_Ls, d.Ls);
        }
        while (P.n_long < nl && hl[P.n_long].n > MF_TILE_LEN) P.n_long++;   // sorted by descending cells == descending n
        std::vector<LocusDesc> units;
        P.ring_acc = build_fill_units(hl, nl, units, P.bucket_first, P.max_n);
        const int nu = P.nu = (int)units.size();
        CK(Ln.h_units.ensure(sizeof(LocusDesc) * (size_t)nu + 64));
        memcpy(Ln.h_units.p, units.data(), sizeof(LocusDesc) * (size_t)nu);
        out.st.fill_units += (uint64_t)nu;
        // ---- buffers (grow-only; cudaFree of an outgrown buffer synchronises the device, which also orders it after its last use)
        CK(Ln.loci.ensure(sizeof(LocusDesc) * nl));
        CK(Ln.listoff.ensure(sizeof(unsigned long long) * nl));
        CK(Ln.codes.ensure(P.seq_acc));
        CK(Ln.F.ensure(P.seq_acc * 4));
        CK(Ln.C.ensure(P.band_acc * 4));
        CK(Ln.M.ensure(P.band_acc * 4));
        CK(Ln.Ib.ensure(P.band_acc + 256));
        if (!J.force_wide) CK(Ln.Mp.ensure(P.band_acc * 4 + 4096));   // fML16 row pairs: NS (two copies) or NS/2 words per diagonal, by bucket
        CK(Ln.ring.ensure(P.ring_acc * 4));
        CK(Ln.tbcount.ensure((size_t)nl * 4));
        CK(Ln.tbbase.ensure((size_t)(nl + 1) * 8));
        CK(Ln.scan_in.ensure((size_t)(nl + 1) * 8));
        CK(Ln.startlist.ensure(P.list_acc * 4));
        CK(Ln.fail.ensure(4));
        CK(Ln.fillflags.ensure((size_t)nu * 4 + 4));
        CK(Ln.units.ensure(sizeof(LocusDesc) * (size_t)nu + 64));
        CK(Ln.h_small.ensure(256));
        // ---- upload
        cudaStream_t lo = Ln.s_lo, hi = Ln.s_hi;
        CK(cudaEventRecord(Ln.ev[EV_H2D], lo));
        const char *raw_dev = d_raw;
        if (!d_raw) {
            CK(Ln.h_raw.ensure(P.raw_acc));
            char *hr = Ln.h_raw.as<char>();
            for (int k = 0; k < nl; k++) memcpy(hr + hl[k].raw_off, J.seqs + J.h_off[loci[P.cb + k].rec], (size_t)hl[k].n);
            CK(Ln.raw.ensure(P.raw_acc));
            CK(cudaMemcpyAsync(Ln.raw.p, hr, P.raw_acc, cudaMemcpyHostToDevice, lo));
            out.st.h2d_bytes += P.raw_acc;
            raw_dev = Ln.raw.as<char>();
        }
        CK(cudaMemcpyAsync(Ln.loci.p, hl, sizeof(LocusDesc) * nl, cudaMemcpyHostToDevice, lo));
        CK(cudaMemcpyAsync(Ln.listoff.p, hlo, sizeof(unsigned long long) * nl, cudaMemcpyHostToDevice, lo));
        CK(cudaMemcpyAsync(Ln.units.p, Ln.h_units.p, sizeof(LocusDesc) * (size_t)nu, cudaMemcpyHostToDevice, lo));
        out.st.h2d_bytes += (sizeof(LocusDesc) + 8) * (uint64_t)nl + sizeof(LocusDesc) * (uint64_t)nu;
        CK(cudaMemsetAsync(Ln.fail.p, 0, 4, lo));
        CK(cudaMemsetAsync(Ln.fillflags.p, 0, (size_t)nu * 4 + 4, lo));
        CK(cudaEventRecord(Ln.ev[EV_KERNELS], lo));
        // The two lanes' fills normally share the SMs and finish together, which is what hides wave tails -- but it also means the
        // small last chunk (plan_chunks cuts it 80 : 20) would be done before the previous chunk's download even starts.  Its fill
        // therefore waits for the previous chunk's fill to END: it then runs next to that chunk's traceback and under its download.
        if (J.sink != SINK_NONE && J.sink != SINK_TOTALS && nlanes_ == 2 && ci > 0 && ci + 1 == chunks.size())
            CK(cudaStreamWaitEvent(lo, D.lane[(ci + 1) % 2].ev[EV_FILL_END], 0));
        // ---- K1, K2 on the low-priority stream
        const LocusDesc *dl = Ln.loci.as<LocusDesc>();
        CK(launch_prepare(raw_dev, dl, nl, P.seq_acc, Ln.codes.as<unsigned char>(), Ln.F.as<int>(), lo));
        CK(cudaEventRecord(Ln.ev[EV_FILL], lo));
        static const bool no_side = getenv("MIRFOLD_NO_SIDE_STREAM") != nullptr;   // A/B runs
        CK(launch_fill(fill_launch(Ln, D.dP, nu, P.max_n, P.bucket_first, J.force_wide, J.L), lo, no_side ? nullptr : Ln.side,
                       Ln.ev[EV_SIDE_FORK], Ln.ev[EV_SIDE_JOIN]));
        CK(cudaEventRecord(Ln.ev[EV_FILL_END], lo));
        // ---- K3 + emission plan on the high-priority stream
        CK(cudaStreamWaitEvent(hi, Ln.ev[EV_FILL_END], 0));
        CK(launch_f3(dl, nl, P.n_long, P.max_Ls, Ln.codes.as<unsigned char>(), Ln.C.as<int>(), Ln.F.as<int>(), D.dP, hi));
        {   // kernels launched so far: k_prepare, the fill kernels (16-bit + 32-bit redo per non-empty bucket, generic), k_f3 / k_f3_cta
            int nfill = P.bucket_first[1] > P.bucket_first[0] ? 1 : 0;
            for (int b = 1; b < 5; b++) if (P.bucket_first[b + 1] > P.bucket_first[b]) nfill += J.force_wide ? 1 : 2;
            out.st.kernel_launches += 1 + nfill + (P.n_long > 0 ? 1 : 0) + (P.n_long < nl ? 1 : 0);
        }
        CK(cudaEventRecord(Ln.ev[EV_F3_END], hi));
        if (J.sink == SINK_TOTALS) return front_totals(Ln, ci + 1 == chunks.size());
        TraceBuffers &tb = Ln.tb;
        tb = trace_buffers(Ln, dl, nl);
        CK(launch_plan(tb, hi));
        k_widen_counts<<<(nl + 1 + 255) / 256, 256, 0, hi>>>(tb.tb_count, Ln.scan_in.as<unsigned long long>(), nl);
        CK(cudaGetLastError());
        CK(exclusive_scan(Ln, Ln.scan_in.as<unsigned long long>(), tb.tb_base, (size_t)nl + 1, hi));
        CK(cudaMemcpyAsync(Ln.h_small.p, tb.tb_base + nl, 8, cudaMemcpyDeviceToHost, hi));
        out.st.kernel_launches += 4;   // k_plan, k_widen_counts, cub scan (init + scan)
        Ln.pending = true;
        ht.mark("front (descriptors, uploads, K1-K3 enqueue)");
        return true;
    }

    // ---- SINK_TOTALS: the chunk ends after f3 with the download of its total lines (retire publishes them)
    bool front_totals(Lane &Ln, bool last_chunk)
    {
        cudaStream_t hi = Ln.s_hi;
        const int nl = Ln.prep.nl;
        CK(Ln.totals.ensure((size_t)nl * 4 + 4));
        CK(Ln.h_out.ensure((size_t)(nl + 1) * 8 + (size_t)nl * 4 + 64));
        k_gather_totals<<<(nl + 255) / 256, 256, 0, hi>>>(Ln.loci.as<LocusDesc>(), Ln.F.as<int>(), Ln.totals.as<int>(), nl);
        CK(cudaGetLastError());
        CK(cudaEventRecord(Ln.ev[EV_PACK_END], hi));
        if (last_chunk) CK(cudaEventRecord(D.ev_last, hi));
        CK(cudaMemcpyAsync(Ln.h_out.as<unsigned long long>() + nl + 1, Ln.totals.p, (size_t)nl * 4, cudaMemcpyDeviceToHost, hi));
        CK(cudaEventRecord(Ln.ev[EV_D2H_END], hi));
        CK(cudaStreamWaitEvent(Ln.s_lo, Ln.ev[EV_D2H_END], 0));   // the lane's next upload waits for this chunk to leave the device
        out.st.kernel_launches += 1;
        out.st.d2h_bytes += (uint64_t)nl * 4;
        Ln.pending = true;
        ht.mark("front (descriptors, uploads, K1-K3, totals enqueue)");
        return true;
    }

    // ---- middle: tracebacks, emission decisions, output sizes (second host sync)
    bool middle(Lane &Ln)
    {
        if (J.sink == SINK_TOTALS) return true;
        cudaStream_t hi = Ln.s_hi;
        TraceBuffers &tb = Ln.tb;
        CK(cudaStreamSynchronize(hi));
        const unsigned long long ntb = Ln.h_small.as<unsigned long long>()[HS_NTB];
        out.st.tracebacks += ntb;
        ht.mark("plan sync");
        if (!trace_scratch(Ln, tb, ntb, Ln.prep.max_Ls)) return false;
        CK(launch_traceback(tb, hi));
        CK(launch_emit(tb, hi));
        if (ntb) out.st.kernel_launches += 2;
        if (!emission_sizes(Ln, tb, hi)) return false;
        ht.mark("traceback sync");
        return true;
    }

    // the plan's buffers of the lane for nl descriptors at dl; per-traceback scratch comes from trace_scratch
    TraceBuffers trace_buffers(Lane &Ln, const LocusDesc *dl, int nl) const
    {
        TraceBuffers tb{};
        tb.loci = dl; tb.nloci = nl; tb.codes = Ln.codes.as<unsigned char>();
        tb.C = Ln.C.as<int>(); tb.M = Ln.M.as<int>(); tb.F = Ln.F.as<int>(); tb.Ib = Ln.Ib.as<unsigned char>(); tb.P = D.dP;
        tb.tb_count = Ln.tbcount.as<int>(); tb.tb_base = Ln.tbbase.as<unsigned long long>();
        tb.list_off = Ln.listoff.as<unsigned long long>(); tb.tb_start_list = Ln.startlist.as<int>();
        tb.fail_flag = Ln.fail.as<int>();
        return tb;
    }

    // scratch of ntb tracebacks of at most max_Ls nt: slots, per-traceback ints, stacks and the emission scans
    bool trace_scratch(Lane &Ln, TraceBuffers &tb, unsigned long long ntb, int max_Ls)
    {
        tb.ntb = ntb;
        tb.slot_stride = (max_Ls + 4 + 3) & ~3;
        tb.stack_cap = max_Ls / 4 + 16;
        tb.code_win = (max_Ls + 8 + 15) & ~15;
        CK(Ln.slots.ensure((size_t)ntb * tb.slot_stride + 16));
        CK(Ln.tblen.ensure((size_t)ntb * 4 + 16)); CK(Ln.tbstart.ensure((size_t)ntb * 4 + 16));
        CK(Ln.tblocus.ensure((size_t)ntb * 4 + 16)); CK(Ln.tbflag.ensure((size_t)ntb * 4 + 16));
        CK(Ln.tbenergy.ensure((size_t)ntb * 4 + 16));
        CK(Ln.stackscr.ensure((size_t)ntb * tb.stack_cap * 8 + 16));
        CK(Ln.ssoff.ensure((size_t)(ntb + 1) * 8)); CK(Ln.hitidx.ensure((size_t)(ntb + 1) * 8));
        CK(Ln.scan_in.ensure((size_t)(ntb + 1) * 8 + (size_t)(tb.nloci + 1) * 8));
        CK(Ln.scan_out.ensure((size_t)(ntb + 1) * 8));
        tb.slots = Ln.slots.as<char>(); tb.tb_len = Ln.tblen.as<int>(); tb.tb_start = Ln.tbstart.as<int>();
        tb.tb_locus = Ln.tblocus.as<int>(); tb.tb_flag = Ln.tbflag.as<int>(); tb.tb_energy = Ln.tbenergy.as<int>();
        tb.stack_scratch = Ln.stackscr.as<int>();
        return true;
    }

    // after the emission decisions: the printed bytes (ssoff) and hit indices (hitidx) of the tb.ntb tracebacks, their
    // totals into Ln.abytes / Ln.nhits, and the fail flag (host sync)
    bool emission_sizes(Lane &Ln, const TraceBuffers &tb, cudaStream_t st)
    {
        const unsigned long long ntb = tb.ntb;
        unsigned long long *hs = Ln.h_small.as<unsigned long long>();
        if (ntb) {
            k_emit_sizes<<<(unsigned)((ntb + 1 + 255) / 256), 256, 0, st>>>(tb.tb_flag, tb.tb_len, Ln.scan_in.as<unsigned long long>(),
                                                                             Ln.scan_out.as<unsigned long long>(), ntb);
            CK(cudaGetLastError());
            CK(exclusive_scan(Ln, Ln.scan_in.as<unsigned long long>(), Ln.ssoff.as<unsigned long long>(), (size_t)ntb + 1, st));
            CK(exclusive_scan(Ln, Ln.scan_out.as<unsigned long long>(), Ln.hitidx.as<unsigned long long>(), (size_t)ntb + 1, st));
            CK(cudaMemcpyAsync(&hs[HS_ABYTES], Ln.ssoff.as<unsigned long long>() + ntb, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(&hs[HS_NHITS], Ln.hitidx.as<unsigned long long>() + ntb, 8, cudaMemcpyDeviceToHost, st));
            out.st.kernel_launches += 5;   // k_emit_sizes, two cub scans (init + scan each)
        }
        CK(cudaMemcpyAsync(&hs[HS_FAIL], Ln.fail.p, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (*(int *)&hs[HS_FAIL]) { out.err = MIRFOLD_ERR_BACKTRACK; out.errmsg = "traceback found no decomposition"; return false; }
        Ln.abytes = ntb ? hs[HS_ABYTES] : 0;
        Ln.nhits = ntb ? hs[HS_NHITS] : 0;
        return true;
    }

    // where the lane's Ln.nhits hits and Ln.abytes string bytes go on the host: a reservation in the shared result buffers,
    // else an overflow chunk of their own (Ln.ovf); the stream sink's buffers; nowhere for the other sinks
    bool pick_destination(Lane &Ln, mirfold_hit *&dst_hits, char *&dst_arena)
    {
        const uint64_t nhits = Ln.nhits, abytes = Ln.abytes;
        dst_hits = nullptr;
        dst_arena = nullptr;
        Ln.hit_base = Ln.arena_base = 0;
        if (J.sink == SINK_SHARED) {
            if (J.shared->reserve(nhits, abytes, Ln.hit_base, Ln.arena_base)) {
                dst_hits = J.shared->hits.as<mirfold_hit>() + Ln.hit_base;
                dst_arena = J.shared->arena.as<char>() + Ln.arena_base;
            } else {
                Ln.ovf.reset(new OverflowChunk());
                CK(Ln.ovf->hits.ensure(nhits * sizeof(mirfold_hit) + 16));
                CK(Ln.ovf->arena.ensure(abytes + 16));
                Ln.ovf->nhits = nhits; Ln.ovf->abytes = abytes;
                dst_hits = Ln.ovf->hits.as<mirfold_hit>();
                dst_arena = Ln.ovf->arena.as<char>();
            }
        } else if (J.sink == SINK_STREAM) {
            CK(Ln.h_hits.ensure(nhits * sizeof(mirfold_hit) + 16));
            CK(Ln.h_arena.ensure(abytes + 16));
            dst_hits = Ln.h_hits.as<mirfold_hit>();
            dst_arena = Ln.h_arena.as<char>();
        }
        return true;
    }

    // Ln.bounds / Ln.totals of the chunk: every locus' first hit and total, or all zero when the chunk has no traceback
    // (hitidx was never scanned)
    bool gather_bounds(Lane &Ln)
    {
        cudaStream_t hi = Ln.s_hi;
        const TraceBuffers &tb = Ln.tb;
        const int nl = Ln.prep.nl;
        if (tb.ntb) {
            k_gather_bounds<<<(nl + 1 + 255) / 256, 256, 0, hi>>>(tb.tb_base, Ln.hitidx.as<unsigned long long>(), tb.loci, tb.F,
                                                                  Ln.bounds.as<unsigned long long>(), Ln.totals.as<int>(), nl);
            CK(cudaGetLastError());
            out.st.kernel_launches += 1;
        } else {
            CK(cudaMemsetAsync(Ln.bounds.p, 0, (size_t)(nl + 1) * 8, hi));
            CK(cudaMemsetAsync(Ln.totals.p, 0, (size_t)nl * 4, hi));
        }
        return true;
    }

    // ---- back: pack the printed structures and start the download into the sink (asynchronous; see retire)
    bool back(Lane &Ln, bool last_chunk)
    {
        if (J.sink == SINK_TOTALS) return true;
        cudaStream_t hi = Ln.s_hi;
        TraceBuffers &tb = Ln.tb;
        const Prep &P = Ln.prep;
        const int nl = P.nl;
        const uint64_t nhits = Ln.nhits, abytes = Ln.abytes;
        mirfold_hit *dst_hits;
        char *dst_arena;
        if (!pick_destination(Ln, dst_hits, dst_arena)) return false;
        CK(Ln.o_hits.ensure(nhits * sizeof(mirfold_hit) + 16));
        CK(Ln.o_arena.ensure(abytes + 16));
        CK(Ln.bounds.ensure((size_t)(nl + 1) * 8));
        CK(Ln.totals.ensure((size_t)nl * 4 + 4));
        CK(launch_pack(tb, Ln.ssoff.as<unsigned long long>(), Ln.hitidx.as<unsigned long long>(), Ln.o_arena.as<char>(),
                       Ln.o_hits.as<mirfold_hit>(), Ln.arena_base, hi));
        out.st.kernel_launches += 1;
        if (J.sink == SINK_CAND) {
            if (!back_candidates(Ln, last_chunk)) return false;
        } else {
            CK(cudaEventRecord(Ln.ev[EV_PACK_END], hi));
            if (last_chunk) CK(cudaEventRecord(D.ev_last, hi));
            if (J.sink != SINK_NONE) {
                if (!gather_bounds(Ln)) return false;
                CK(Ln.h_out.ensure((size_t)(nl + 1) * 8 + (size_t)nl * 4 + 64));
                unsigned long long *h_bounds = Ln.h_out.as<unsigned long long>();
                if (nhits) CK(cudaMemcpyAsync(dst_hits, Ln.o_hits.p, nhits * sizeof(mirfold_hit), cudaMemcpyDeviceToHost, hi));
                if (abytes) CK(cudaMemcpyAsync(dst_arena, Ln.o_arena.p, abytes, cudaMemcpyDeviceToHost, hi));
                CK(cudaMemcpyAsync(h_bounds, Ln.bounds.p, (size_t)(nl + 1) * 8, cudaMemcpyDeviceToHost, hi));
                CK(cudaMemcpyAsync(h_bounds + nl + 1, Ln.totals.p, (size_t)nl * 4, cudaMemcpyDeviceToHost, hi));
                out.st.d2h_bytes += nhits * sizeof(mirfold_hit) + (uint64_t)(nl + 1) * 8 + (uint64_t)nl * 4 + abytes + 32;
            } else out.st.d2h_bytes += 32;
        }
        CK(cudaEventRecord(Ln.ev[EV_D2H_END], hi));
        // the lane's next chunk (uploads on s_lo) may only start once this one has left the device
        CK(cudaStreamWaitEvent(Ln.s_lo, Ln.ev[EV_D2H_END], 0));
        out.nhits += nhits;
        out.arena_bytes += abytes;
        ht.mark("back (pack + download enqueue)");
        return true;
    }

    // ---- fused stages 1 + 3 on the chunk's packed hits (still in HBM): classify, duplex verdicts, compact download
    bool back_candidates(Lane &Ln, bool last_chunk, bool bounds_ready = false)
    {
        cudaStream_t hi = Ln.s_hi;
        TraceBuffers &tb = Ln.tb;
        const Prep &P = Ln.prep;
        const int nl = P.nl;
        const uint64_t nhits = Ln.nhits;
        const CandArgs &ca = *J.cand;
        unsigned long long *hs = Ln.h_small.as<unsigned long long>();
        if (!bounds_ready && !gather_bounds(Ln)) return false;   // bounds_ready: a segmented locus' staged bounds were uploaded
        CK(Ln.c_counts.ensure((nhits + 2) * 8)); CK(Ln.c_soff.ensure((nhits + 2) * 8));
        CK(Ln.c_lsb.ensure((size_t)(nl + 1) * 8));
        CandLaunch c{};
        c.loci = tb.loci; c.nloci = nl; c.hits = Ln.o_hits.as<mirfold_hit>(); c.nhits = nhits;
        c.arena = Ln.o_arena.as<char>(); c.arena_base = Ln.arena_base; c.bounds = Ln.bounds.as<unsigned long long>();
        c.regions = D.cand_regions.as<mirfold_region>(); c.matures = D.cand_matures.as<mirfold_mature>();
        c.mature_off = D.cand_moff.as<unsigned long long>();
        c.minlen = ca.minlen; c.minloop = ca.minloop; c.min_mature = ca.min_mature; c.max_mature = ca.max_mature;
        c.counts = Ln.c_counts.as<unsigned long long>(); c.soff = Ln.c_soff.as<unsigned long long>();
        c.locus_sbegin = Ln.c_lsb.as<unsigned long long>();
        c.fail_flag = Ln.fail.as<int>();
        CK(launch_cand_classify(c, 0, hi));
        CK(exclusive_scan(Ln, c.counts, Ln.c_soff.as<unsigned long long>(), (size_t)nhits + 1, hi));
        CK(cudaMemcpyAsync(&hs[HS_NSTRUCTS], Ln.c_soff.as<unsigned long long>() + nhits, 8, cudaMemcpyDeviceToHost, hi));
        CK(cudaMemcpyAsync(&hs[HS_FAIL], Ln.fail.p, 4, cudaMemcpyDeviceToHost, hi));
        CK(cudaStreamSynchronize(hi));
        if (*(int *)&hs[HS_FAIL]) { out.err = MIRFOLD_ERR_ARG; out.errmsg = "a hit on which the reference's classifier raises (no pair / unbalanced)"; return false; }
        const uint64_t ns = Ln.c_ns = hs[HS_NSTRUCTS];
        CK(Ln.c_structs.ensure(ns * sizeof(mirfold_structure) + 16)); CK(Ln.c_sout.ensure(ns * sizeof(mirfold_structure) + 16));
        CK(Ln.c_nq.ensure((ns + 2) * 8)); CK(Ln.c_sbytes.ensure((ns + 2) * 8));
        CK(Ln.c_voff.ensure((ns + 2) * 8)); CK(Ln.c_aoff.ensure((ns + 2) * 8));
        CK(cudaMemsetAsync(Ln.c_nq.p, 0, (ns + 1) * 8, hi)); CK(cudaMemsetAsync(Ln.c_sbytes.p, 0, (ns + 1) * 8, hi));
        c.structs = Ln.c_structs.as<mirfold_structure>(); c.nstructs = ns;
        c.nq = Ln.c_nq.as<unsigned long long>(); c.sbytes = Ln.c_sbytes.as<unsigned long long>();
        CK(launch_cand_classify(c, 1, hi));
        CK(exclusive_scan(Ln, c.nq, Ln.c_voff.as<unsigned long long>(), (size_t)ns + 1, hi));
        CK(exclusive_scan(Ln, c.sbytes, Ln.c_aoff.as<unsigned long long>(), (size_t)ns + 1, hi));
        CK(cudaMemcpyAsync(&hs[HS_NVERDICTS], Ln.c_voff.as<unsigned long long>() + ns, 8, cudaMemcpyDeviceToHost, hi));
        CK(cudaMemcpyAsync(&hs[HS_SBYTES], Ln.c_aoff.as<unsigned long long>() + ns, 8, cudaMemcpyDeviceToHost, hi));
        CK(cudaStreamSynchronize(hi));
        const uint64_t nv = Ln.c_nv = hs[HS_NVERDICTS], nb = Ln.c_nb = hs[HS_SBYTES];
        CK(Ln.c_verd.ensure(nv * sizeof(mirfold_duplex_verdict) + 16)); CK(Ln.c_vmat.ensure(nv * 4 + 16)); CK(Ln.c_arena.ensure(nb + 16));
        c.voff = Ln.c_voff.as<unsigned long long>(); c.aoff = Ln.c_aoff.as<unsigned long long>();
        c.verdicts = Ln.c_verd.as<mirfold_duplex_verdict>(); c.verdict_mature = Ln.c_vmat.as<unsigned int>();
        c.out_arena = Ln.c_arena.as<char>(); c.out_base = 0; c.structs_out = Ln.c_sout.as<mirfold_structure>();
        CK(launch_cand_finish(c, P.max_Ls + 4, hi));
        out.st.kernel_launches += 10;   // 2 x classify, locus bounds, 3 x cub scan (2 kernels each), duplex, strings
        CK(cudaEventRecord(Ln.ev[EV_PACK_END], hi));
        if (last_chunk) CK(cudaEventRecord(D.ev_last, hi));
        CK(Ln.hc_structs.ensure(ns * sizeof(mirfold_structure) + 16)); CK(Ln.hc_arena.ensure(nb + 16));
        CK(Ln.hc_verd.ensure(nv * sizeof(mirfold_duplex_verdict) + 16)); CK(Ln.hc_vmat.ensure(nv * 4 + 16));
        CK(Ln.hc_voff.ensure((ns + 1) * 8)); CK(Ln.hc_lsb.ensure((size_t)(nl + 1) * 8));
        if (ns) CK(cudaMemcpyAsync(Ln.hc_structs.p, Ln.c_sout.p, ns * sizeof(mirfold_structure), cudaMemcpyDeviceToHost, hi));
        if (nb) CK(cudaMemcpyAsync(Ln.hc_arena.p, Ln.c_arena.p, nb, cudaMemcpyDeviceToHost, hi));
        if (nv) CK(cudaMemcpyAsync(Ln.hc_verd.p, Ln.c_verd.p, nv * sizeof(mirfold_duplex_verdict), cudaMemcpyDeviceToHost, hi));
        if (nv) CK(cudaMemcpyAsync(Ln.hc_vmat.p, Ln.c_vmat.p, nv * 4, cudaMemcpyDeviceToHost, hi));
        CK(cudaMemcpyAsync(Ln.hc_voff.p, Ln.c_voff.p, (ns + 1) * 8, cudaMemcpyDeviceToHost, hi));
        CK(cudaMemcpyAsync(Ln.hc_lsb.p, Ln.c_lsb.p, (size_t)(nl + 1) * 8, cudaMemcpyDeviceToHost, hi));
        out.st.d2h_bytes += ns * sizeof(mirfold_structure) + nb + nv * (sizeof(mirfold_duplex_verdict) + 4) + (ns + 1) * 8 + (uint64_t)(nl + 1) * 8 + 64;
        return true;
    }

    // ---- a segmented locus (plan_segments): every segment fills its tiles, runs f3 over its owned rows, the emission plan
    // from the state the segment above left, the tracebacks from its starts and the emission decisions, then packs and
    // downloads its hits.  Each segment is addressed as the locus' suffix from its first tile's origin on (the same tiles,
    // rows and f3 shifted by that origin), so the band buffer starts at the segment's first tile.  The last traceback of a
    // segment is decided against the first one of the next: its slot, start and length are carried over, not traced again.
    // The record's hits are staged on the host and published as one record once its last segment is done.
    bool fold_segmented(Lane &Ln, size_t ci)
    {
        if (!retire(Ln)) return false;
        cudaStream_t st = Ln.s_lo;
        const Locus &l = loci[chunks[ci].begin];
        const int n = l.n;
        const bool last_chunk = ci + 1 == chunks.size();
        Prep &P = Ln.prep;
        P = Prep{};
        P.cb = chunks[ci].begin; P.ce = chunks[ci].end; P.nl = 1;
        LocusDesc d{};
        shape_locus(d, n, J.L);
        d.rec = (int)l.rec;
        d.raw_off = d_raw ? raw_off[l.rec] : 0;
        P.max_Ls = d.Ls;
        const int S = d.tile_step, TL = d.stride;
        std::vector<SegPlan> segs;
        plan_segments(n, J.L, lane_bytes(), segs);
        // whole-locus arrays: raw, codes, F; descriptors [0] = the locus, [1] = the running segment's suffix
        CK(Ln.h_loci.ensure(2 * sizeof(LocusDesc)));
        CK(Ln.loci.ensure(2 * sizeof(LocusDesc)));
        CK(Ln.codes.ensure((size_t)n + 3));
        CK(Ln.F.ensure(((size_t)n + 3) * 4));
        CK(Ln.segstate.ensure(16));
        CK(Ln.fail.ensure(4));
        CK(Ln.listoff.ensure(8));
        CK(Ln.tbbase.ensure(16));
        CK(Ln.tbcount.ensure(4));
        CK(Ln.h_small.ensure(256));
        LocusDesc *hl = Ln.h_loci.as<LocusDesc>();
        hl[0] = d;
        const LocusDesc *dl = Ln.loci.as<LocusDesc>();
        CK(cudaEventRecord(Ln.ev[EV_H2D], st));
        const char *raw_dev = d_raw;
        if (!d_raw) {
            CK(Ln.raw.ensure((size_t)n));
            CK(cudaMemcpyAsync(Ln.raw.p, J.seqs + J.h_off[l.rec], (size_t)n, cudaMemcpyHostToDevice, st));
            out.st.h2d_bytes += (uint64_t)n;
            raw_dev = Ln.raw.as<char>();
        }
        CK(cudaMemcpyAsync(Ln.loci.p, hl, sizeof(LocusDesc), cudaMemcpyHostToDevice, st));
        CK(cudaMemsetAsync(Ln.segstate.p, 0, 16, st));   // fnext = f3(n-3) = 0, do_bt = have_prev = 0
        CK(cudaMemsetAsync(Ln.fail.p, 0, 4, st));
        CK(cudaMemsetAsync(Ln.listoff.p, 0, 8, st));
        CK(cudaEventRecord(Ln.ev[EV_KERNELS], st));
        CK(launch_prepare(raw_dev, dl, 1, (unsigned long long)n + 3, Ln.codes.as<unsigned char>(), Ln.F.as<int>(), st));
        out.st.kernel_launches += 1;
        std::vector<mirfold_hit> hits;   // the record's hits in print order; ss_off into `arena`
        std::vector<char> arena;
        std::vector<char> carry_slot;    // the last traceback of the segment above: slot, length, absolute start
        int carry_len = 0, carry_start = 0;
        bool carry = false;
        unsigned long long *hs = Ln.h_small.as<unsigned long long>();
        for (size_t sg = 0; sg < segs.size(); sg++) {
            const SegPlan &g = segs[sg];
            const bool last = sg + 1 == segs.size();
            const int t_hi = g.t1 + g.halo, ntiles = t_hi - g.t0 + 1;
            const int a = std::min(g.t0 * S, n - TL);   // the first tile's origin: suffix row k is locus row a + k
            LocusDesc ds = d;
            ds.n = n - a; ds.seq_off = d.seq_off + (unsigned long long)a; ds.band_off = 0; ds.tile_last = d.tile_last - g.t0;
            hl[1] = ds;
            // ---- fill of the segment's tiles (one bucket), f3 over its owned rows
            const size_t be = (size_t)ntiles * band_elems(TL, d.dmax);
            CK(Ln.h_units.ensure(sizeof(LocusDesc) * (size_t)ntiles + 64));
            LocusDesc *hu = Ln.h_units.as<LocusDesc>();
            for (int t = g.t0; t <= t_hi; t++) {
                LocusDesc u = tile_unit(d, t);
                u.band_off = (unsigned long long)(t - g.t0) * band_elems(TL, d.dmax);
                u.ring_off = (unsigned long long)(t - g.t0) * unit_ring_elems(TL);
                hu[t - g.t0] = u;
            }
            CK(Ln.C.ensure(be * 4));
            CK(Ln.M.ensure(be * 4));
            CK(Ln.Ib.ensure(be + 256));
            if (!J.force_wide) CK(Ln.Mp.ensure(be * 4 + 4096));
            CK(Ln.ring.ensure((size_t)ntiles * unit_ring_elems(TL) * 4));
            CK(Ln.units.ensure(sizeof(LocusDesc) * (size_t)ntiles + 64));
            CK(Ln.fillflags.ensure((size_t)ntiles * 4 + 4));
            CK(cudaMemcpyAsync(Ln.units.p, hu, sizeof(LocusDesc) * (size_t)ntiles, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(Ln.loci.as<LocusDesc>() + 1, &hl[1], sizeof(LocusDesc), cudaMemcpyHostToDevice, st));
            CK(cudaMemsetAsync(Ln.fillflags.p, 0, (size_t)ntiles * 4 + 4, st));
            out.st.h2d_bytes += sizeof(LocusDesc) * (uint64_t)(ntiles + 1);
            out.st.fill_units += (uint64_t)ntiles;
            CK(cudaEventRecord(Ln.ev[EV_FILL], st));
            const int bucket = unit_bucket(hu[0]);
            int bucket_first[6];
            for (int b = 0; b < 6; b++) bucket_first[b] = b <= bucket ? 0 : ntiles;
            CK(launch_fill(fill_launch(Ln, D.dP, ntiles, TL, bucket_first, J.force_wide, J.L), st));
            CK(cudaEventRecord(Ln.ev[EV_FILL_END], st));
            const int row_lo = g.row_lo - a, row_hi = std::min(g.row_hi, n - 4) - a;   // owned rows with an f3 / plan step
            CK(launch_f3_rows(dl + 1, d.Ls, row_hi, row_lo, Ln.codes.as<unsigned char>(), Ln.C.as<int>(), Ln.F.as<int>(), D.dP, st));
            CK(cudaEventRecord(Ln.ev[EV_F3_END], st));
            out.st.kernel_launches += (J.force_wide ? 1 : 2) + (row_hi >= row_lo ? 1 : 0);
            if (J.sink == SINK_TOTALS) {
                CK(cudaEventRecord(Ln.ev[EV_PACK_END], st));
                CK(cudaEventRecord(Ln.ev[EV_D2H_END], st));
                CK(cudaStreamSynchronize(st));
                add_stage_times(Ln, sg == 0);
                continue;
            }
            // ---- emission plan over the owned rows, resumed from the segment above
            const int *Fs = Ln.F.as<int>() + ds.seq_off;
            CK(Ln.startlist.ensure(((size_t)(g.row_hi - g.row_lo + 1) / 2 + 4) * 4));
            CK(launch_plan_seg(Fs, row_hi, row_lo, g.row_lo == 1 ? 1 : 0, Ln.segstate.as<int>(), Ln.startlist.as<int>(),
                               Ln.tbbase.as<unsigned long long>(), Ln.tbcount.as<int>(), st));
            CK(cudaMemcpyAsync(&hs[HS_NTB], Ln.tbbase.as<unsigned long long>() + 1, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const int nc = carry ? 1 : 0;
            const unsigned long long m = hs[HS_NTB], ntb = m + (unsigned long long)nc;
            out.st.tracebacks += m;
            // ---- tracebacks of the segment's starts behind the carried entry 0
            TraceBuffers tb = trace_buffers(Ln, dl + 1, 1);
            if (!trace_scratch(Ln, tb, ntb, d.Ls)) return false;
            const int slot_stride = tb.slot_stride;
            if (carry) {
                CK(cudaMemcpyAsync(tb.slots, carry_slot.data(), (size_t)slot_stride, cudaMemcpyHostToDevice, st));
                CK(cudaMemcpyAsync(tb.tb_len, &carry_len, 4, cudaMemcpyHostToDevice, st));
                CK(cudaMemcpyAsync(tb.tb_start, &carry_start, 4, cudaMemcpyHostToDevice, st));
            }
            TraceBuffers tv = tb;   // the segment's own tracebacks: entries nc .. ntb-1
            tv.ntb = m;
            tv.slots += (size_t)nc * slot_stride; tv.tb_len += nc; tv.tb_start += nc; tv.tb_locus += nc; tv.tb_flag += nc; tv.tb_energy += nc;
            tv.stack_scratch += (size_t)nc * tb.stack_cap * 2;
            CK(launch_traceback(tv, st));
            int *abs_start = Ln.tblocus.as<int>();
            CK(launch_emit_seg(tb, nc, a, last ? 1 : 0, Ln.F.as<int>() + d.seq_off, n, abs_start, st));
            if (!emission_sizes(Ln, tb, st)) return false;
            const uint64_t nhits = Ln.nhits, abytes = Ln.abytes;
            // ---- pack and download the printed hits; carry the undecided last traceback to the next segment
            CK(Ln.o_hits.ensure(nhits * sizeof(mirfold_hit) + 16));
            CK(Ln.o_arena.ensure(abytes + 16));
            CK(Ln.h_hits.ensure(nhits * sizeof(mirfold_hit) + 16));
            CK(Ln.h_arena.ensure(abytes + 16));
            TraceBuffers tp = tb;
            tp.tb_start = abs_start;
            CK(launch_pack(tp, Ln.ssoff.as<unsigned long long>(), Ln.hitidx.as<unsigned long long>(), Ln.o_arena.as<char>(),
                           Ln.o_hits.as<mirfold_hit>(), (unsigned long long)arena.size(), st));
            CK(cudaEventRecord(Ln.ev[EV_PACK_END], st));
            if (nhits) CK(cudaMemcpyAsync(Ln.h_hits.p, Ln.o_hits.p, nhits * sizeof(mirfold_hit), cudaMemcpyDeviceToHost, st));
            if (abytes) CK(cudaMemcpyAsync(Ln.h_arena.p, Ln.o_arena.p, abytes, cudaMemcpyDeviceToHost, st));
            carry = !last && ntb > 0;
            if (carry) {
                carry_slot.resize((size_t)slot_stride);
                CK(cudaMemcpyAsync(carry_slot.data(), tb.slots + (ntb - 1) * slot_stride, (size_t)slot_stride, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(&carry_len, tb.tb_len + (ntb - 1), 4, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(&carry_start, abs_start + (ntb - 1), 4, cudaMemcpyDeviceToHost, st));
            }
            CK(cudaEventRecord(Ln.ev[EV_D2H_END], st));
            CK(cudaStreamSynchronize(st));
            out.st.kernel_launches += 1 + (m ? 1 : 0) + (ntb ? 2 : 0);   // k_plan_seg, k_traceback, k_emit_seg, k_pack
            out.st.d2h_bytes += nhits * sizeof(mirfold_hit) + abytes + 32;
            hits.insert(hits.end(), Ln.h_hits.as<mirfold_hit>(), Ln.h_hits.as<mirfold_hit>() + nhits);
            arena.insert(arena.end(), Ln.h_arena.as<char>(), Ln.h_arena.as<char>() + abytes);
            add_stage_times(Ln, sg == 0);
        }
        int total = 0;
        CK(cudaMemcpyAsync(&total, Ln.F.as<int>() + d.seq_off + 1, 4, cudaMemcpyDeviceToHost, st));
        if (last_chunk) CK(cudaEventRecord(D.ev_last, st));
        CK(cudaStreamSynchronize(st));
        out.st.d2h_bytes += 4;
        ht.mark("segmented locus");
        return publish_segmented(Ln, hits, arena, total, last_chunk);
    }

    // the segmented record's staged hits (ss_off relative to its own arena) into the call's sink, as a chunk of one record
    bool publish_segmented(Lane &Ln, const std::vector<mirfold_hit> &hits, const std::vector<char> &arena, int total, bool last_chunk)
    {
        const uint64_t nh = hits.size(), ab = arena.size();
        out.nhits += nh;
        out.arena_bytes += ab;
        Ln.nhits = nh; Ln.abytes = ab;
        if (J.sink == SINK_CAND) {   // stages 1 + 3 on the record's hits, uploaded again as a chunk of one locus
            cudaStream_t hi = Ln.s_hi;
            const unsigned long long bounds[2] = {0, nh};
            CK(Ln.o_hits.ensure(nh * sizeof(mirfold_hit) + 16));
            CK(Ln.o_arena.ensure(ab + 16));
            CK(Ln.bounds.ensure(16));
            CK(Ln.totals.ensure(8));
            if (nh) CK(cudaMemcpyAsync(Ln.o_hits.p, hits.data(), nh * sizeof(mirfold_hit), cudaMemcpyHostToDevice, hi));
            if (ab) CK(cudaMemcpyAsync(Ln.o_arena.p, arena.data(), ab, cudaMemcpyHostToDevice, hi));
            CK(cudaMemcpyAsync(Ln.bounds.p, bounds, 16, cudaMemcpyHostToDevice, hi));
            CK(cudaMemcpyAsync(Ln.totals.p, &total, 4, cudaMemcpyHostToDevice, hi));
            out.st.h2d_bytes += nh * sizeof(mirfold_hit) + ab + 20;
            Ln.tb = TraceBuffers{};
            Ln.tb.loci = Ln.loci.as<LocusDesc>(); Ln.tb.nloci = 1;
            Ln.arena_base = 0;
            if (!back_candidates(Ln, last_chunk, true)) return false;
            CK(cudaEventRecord(Ln.ev[EV_D2H_END], hi));
            CK(cudaEventSynchronize(Ln.ev[EV_D2H_END]));
            retire_candidates(Ln);
            return true;
        }
        // the segment loop is done with Ln.h_hits / h_arena: the stream sink's destination may be those
        mirfold_hit *dst_hits;
        char *dst_arena;
        if (!pick_destination(Ln, dst_hits, dst_arena)) return false;
        if (dst_hits) {
            for (uint64_t k = 0; k < nh; k++) { dst_hits[k] = hits[k]; dst_hits[k].ss_off += Ln.arena_base; }   // as k_pack adds it
            if (ab) memcpy(dst_arena, arena.data(), ab);
        }
        CK(Ln.h_out.ensure(2 * 8 + 4 + 64));
        unsigned long long *h_bounds = Ln.h_out.as<unsigned long long>();
        h_bounds[0] = 0; h_bounds[1] = nh;
        *(int *)(h_bounds + 2) = total;
        publish(Ln);
        return true;
    }

    void retire_candidates(Lane &Ln)
    {
        const Prep &P = Ln.prep;
        const int nl = P.nl;
        CandCollector &C = *J.collect;
        const uint64_t ns = Ln.c_ns, nv = Ln.c_nv, nb = Ln.c_nb;
        const unsigned long long *lsb = Ln.hc_lsb.as<unsigned long long>(), *voff = Ln.hc_voff.as<unsigned long long>();
        std::lock_guard<std::mutex> lk(C.mu);
        const uint64_t bs = C.structs.size(), bv = C.verdicts.size(), ba = C.arena.size();
        C.structs.insert(C.structs.end(), Ln.hc_structs.as<mirfold_structure>(), Ln.hc_structs.as<mirfold_structure>() + ns);
        for (uint64_t k = bs; k < bs + ns; k++) C.structs[k].ss_off += ba;
        C.arena.insert(C.arena.end(), Ln.hc_arena.as<char>(), Ln.hc_arena.as<char>() + nb);
        C.verdicts.insert(C.verdicts.end(), Ln.hc_verd.as<mirfold_duplex_verdict>(), Ln.hc_verd.as<mirfold_duplex_verdict>() + nv);
        C.verdict_mature.insert(C.verdict_mature.end(), Ln.hc_vmat.as<uint32_t>(), Ln.hc_vmat.as<uint32_t>() + nv);
        for (uint64_t k = 0; k < ns; k++) { C.verdict_begin.push_back(bv + voff[k]); C.verdict_count.push_back((uint32_t)(voff[k + 1] - voff[k])); }
        for (int k = 0; k < nl; k++) {
            const uint32_t r = loci[P.cb + k].rec;
            C.struct_begin[r] = bs + lsb[k];
            C.struct_count[r] = (uint32_t)(lsb[k + 1] - lsb[k]);
        }
    }

    // stage times of the chunk or segment whose events the lane last recorded (all complete); h2d: its uploads too
    void add_stage_times(const Lane &Ln, bool h2d)
    {
        float ms = 0;
        if (h2d) { cudaEventElapsedTime(&ms, Ln.ev[EV_H2D], Ln.ev[EV_KERNELS]); out.st.ms_h2d += ms; }
        cudaEventElapsedTime(&ms, Ln.ev[EV_FILL], Ln.ev[EV_FILL_END]); out.st.ms_fill += ms;
        cudaEventElapsedTime(&ms, Ln.ev[EV_FILL_END], Ln.ev[EV_F3_END]); out.st.ms_f3 += ms;
        cudaEventElapsedTime(&ms, Ln.ev[EV_F3_END], Ln.ev[EV_PACK_END]); out.st.ms_trace += ms;
        cudaEventElapsedTime(&ms, Ln.ev[EV_PACK_END], Ln.ev[EV_D2H_END]); out.st.ms_d2h += ms;
    }

    // the chunk's per-record tables (first-hit bounds and totals in Ln.h_out) into the sink; its hits are already where
    // pick_destination put them
    void publish(Lane &Ln)
    {
        if (J.sink == SINK_NONE) return;
        const Prep &P = Ln.prep;
        const int nl = P.nl;
        const unsigned long long *h_bounds = Ln.h_out.as<unsigned long long>();
        const int *h_total = (const int *)(h_bounds + nl + 1);
        if (J.sink == SINK_TOTALS) {
            for (int k = 0; k < nl; k++) J.totals[loci[P.cb + k].rec] = h_total[k];
        } else if (J.sink == SINK_SHARED) {
            SharedOut &S = *J.shared;
            if (!Ln.ovf) {
                for (int k = 0; k < nl; k++) {
                    const uint32_t r = loci[P.cb + k].rec;
                    S.hit_begin[r] = Ln.hit_base + h_bounds[k];
                    S.hit_count[r] = (uint32_t)(h_bounds[k + 1] - h_bounds[k]);
                    S.totals[r] = h_total[k];
                }
            } else {
                OverflowChunk &O = *Ln.ovf;
                O.recs.resize(nl); O.begin.resize(nl); O.count.resize(nl);
                for (int k = 0; k < nl; k++) {
                    const uint32_t r = loci[P.cb + k].rec;
                    O.recs[k] = r; O.begin[k] = h_bounds[k]; O.count[k] = (uint32_t)(h_bounds[k + 1] - h_bounds[k]);
                    S.totals[r] = h_total[k];
                }
                std::lock_guard<std::mutex> lk(S.mu);
                S.overflow.push_back(std::move(Ln.ovf));
            }
        } else if (J.sink == SINK_STREAM) {
            Ln.s_rec.resize(nl); Ln.s_begin.resize(nl); Ln.s_count.resize(nl); Ln.s_total.resize(nl);
            for (int k = 0; k < nl; k++) {
                Ln.s_rec[k] = loci[P.cb + k].rec;
                Ln.s_begin[k] = h_bounds[k];
                Ln.s_count[k] = (uint32_t)(h_bounds[k + 1] - h_bounds[k]);
                Ln.s_total[k] = h_total[k];
            }
            mirfold_chunk c{};
            c.n_records = (uint32_t)nl; c.device = D.id;
            c.record = Ln.s_rec.data(); c.hit_begin = Ln.s_begin.data(); c.hit_count = Ln.s_count.data();
            c.total_mfe_dcal = Ln.s_total.data();
            c.nhits = Ln.nhits; c.hits = Ln.h_hits.as<mirfold_hit>();
            c.ss_arena = Ln.h_arena.as<char>(); c.ss_bytes = Ln.abytes;
            std::lock_guard<std::mutex> lk(*J.cb_mu);
            if (!J.cb_abort->load() && J.fn(J.user, &c) != 0) J.cb_abort->store(1);
        }
    }

    // ---- retire: wait for the lane's download, collect stage times, publish the chunk's per-record tables
    bool retire(Lane &Ln)
    {
        if (!Ln.pending) return true;
        Ln.pending = false;
        CK(cudaEventSynchronize(Ln.ev[EV_D2H_END]));
        add_stage_times(Ln, true);
        static const bool trace_events = getenv("MIRFOLD_TRACE_EVENTS") != nullptr;
        if (trace_events) {   // device timeline of the chunk relative to the call's first event (ms)
            float t[EV_D2H_END + 1];
            for (int k = 0; k <= EV_D2H_END; k++) cudaEventElapsedTime(&t[k], D.ev_first, Ln.ev[k]);
            fprintf(stderr, "[mirfold events] dev %d lane %d loci %6d  h2d %.2f-%.2f  fill %.2f-%.2f  f3 -%.2f  pack -%.2f  d2h -%.2f\n", D.id,
                    (int)(&Ln - D.lane), Ln.prep.nl, t[0], t[1], t[2], t[3], t[4], t[5], t[6]);
        }
        if (J.sink == SINK_CAND) retire_candidates(Ln);
        else publish(Ln);
        ht.mark("retire (download wait + record tables)");
        return true;
    }
};
#undef CK

bool run_device(Device &D, const Job &J, const std::vector<uint32_t> &recs, const char *d_raw, const uint64_t *raw_off, DevOut &out)
{
    DevicePipeline p(D, J, d_raw, raw_off, out);
    return p.run(recs);
}

HBuf pool_take(mirfold_ctx *ctx, std::vector<HBuf> &pool, size_t bytes)
{   // smallest pooled buffer that is large enough, else the largest one (it will be re-grown by the caller)
    std::lock_guard<std::mutex> lk(ctx->pool_mu);
    int best = -1;
    for (int k = 0; k < (int)pool.size(); k++)
        if (pool[k].cap >= bytes && (best < 0 || pool[k].cap < pool[best].cap)) best = k;
    HBuf b;
    if (best >= 0) { b = pool[best]; pool.erase(pool.begin() + best); }
    return b;
}
void pool_give(mirfold_ctx *ctx, std::vector<HBuf> &pool, HBuf &b)
{   // caller holds ctx->pool_mu
    if (!b.p) return;
    if (ctx->closed) { b.release(); return; }
    if (pool.size() >= 4) {
        int small = 0;
        for (int k = 1; k < (int)pool.size(); k++) if (pool[k].cap < pool[small].cap) small = k;
        if (pool[small].cap < b.cap) std::swap(pool[small], b);
        b.release();
        return;
    }
    pool.push_back(b);
    b = HBuf();
}

void add_stats(mirfold_stats &a, const mirfold_stats &b)
{
    a.ms_h2d = std::max(a.ms_h2d, b.ms_h2d); a.ms_fill = std::max(a.ms_fill, b.ms_fill);
    a.ms_f3 = std::max(a.ms_f3, b.ms_f3); a.ms_trace = std::max(a.ms_trace, b.ms_trace);
    a.ms_d2h = std::max(a.ms_d2h, b.ms_d2h); a.ms_device = std::max(a.ms_device, b.ms_device);
    a.nt += b.nt; a.cells += b.cells; a.tracebacks += b.tracebacks; a.kernel_launches += b.kernel_launches;
    a.h2d_bytes += b.h2d_bytes; a.d2h_bytes += b.d2h_bytes; a.n_chunks += b.n_chunks; a.fill_units += b.fill_units;
}

// span_L > 0: also every record the engine would fill as one unit of 2^31 band cells or more (band_offsets_fit), so
// that such a batch is refused before anything is allocated.  Those need n * (min(span_L, n) - 3) >= 2^31, so n > 2^19.
int validate_offsets(mirfold_ctx *ctx, const uint64_t *seq_off, uint32_t nseq, int span_L)
{
    for (uint32_t r = 0; r < nseq; r++) {
        if (seq_off[r + 1] < seq_off[r]) { ctx->last_error = "seq_off is not non-decreasing"; return MIRFOLD_ERR_ARG; }
        const uint64_t len = seq_off[r + 1] - seq_off[r];
        if (len > (uint64_t)0x3fffffff) { ctx->last_error = "a sequence is longer than 2^30 - 1 nt"; return MIRFOLD_ERR_ARG; }
        if (span_L > 0 && len > (1u << 19)) {
            LocusDesc d{};
            shape_locus(d, (int)len, span_L);
            if (!band_offsets_fit(d)) {
                char msg[160];
                snprintf(msg, sizeof msg, "record %u: %llu nt at span %d is one fill unit of %llu band cells (at most 2^31 - 1)", r,
                         (unsigned long long)len, span_L, band_elems(d.stride, d.dmax));
                ctx->last_error = msg;
                return MIRFOLD_ERR_ARG;
            }
        }
    }
    return MIRFOLD_OK;
}

// the common engine behind mirfold_fold / mirfold_fold_stream / mirfold_fold_device / mirfold_batch_fold
struct FoldArgs {
    const char *seqs = nullptr;
    const uint64_t *seq_off = nullptr;
    uint32_t nseq = 0;
    int span_L = 0;
    uint32_t flags = 0;
    int sink = SINK_SHARED;
    mirfold_chunk_fn fn = nullptr;
    void *user = nullptr;
    // device-resident input: per device a buffer and per record its offset; `shard` then comes from the batch
    const std::vector<void *> *d_raw = nullptr;
    const uint64_t *raw_off = nullptr;
    const std::vector<std::vector<uint32_t>> *shard = nullptr;
    int n_devices = 0;   // 0 = all devices of the context
    const CandArgs *cand = nullptr;      // SINK_CAND
    CandCollector *collect = nullptr;
    uint64_t *nhits_out = nullptr;
    int32_t *totals = nullptr;           // SINK_TOTALS: nseq entries, records shorter than 5 nt are left as they are
};

int fold_engine(mirfold_ctx *ctx, const FoldArgs &A, mirfold_result **out, mirfold_stats *stats_out)
{
    static const bool env_wide = getenv("MIRFOLD_FORCE_WIDE") != nullptr;   // A/B runs of bench.py
    static const bool env_serial = getenv("MIRFOLD_SERIAL") != nullptr;
    if (!ctx || !A.seq_off || (!A.seqs && !A.d_raw && A.nseq)) return MIRFOLD_ERR_ARG;
    if (ctx->closed) return MIRFOLD_ERR_ARG;
    if (A.span_L < 5 || A.span_L > MF_MAX_SPAN) { ctx->last_error = "span_L out of range [5, 4096]"; return MIRFOLD_ERR_ARG; }
    if (out) *out = nullptr;
    int rc = validate_offsets(ctx, A.seq_off, A.nseq, A.span_L);
    if (rc != MIRFOLD_OK) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    HostTimer ht;
    const int G = A.n_devices > 0 ? A.n_devices : (int)ctx->devs.size();
    const uint32_t nseq = A.nseq;
    std::vector<std::vector<uint32_t>> shard_local;
    std::vector<uint64_t> load;
    if (!A.shard) plan_shards(A.seq_off, nseq, A.span_L, G, shard_local, load);
    const std::vector<std::vector<uint32_t>> &shard = A.shard ? *A.shard : shard_local;
    ht.mark("shard plan");

    Job J;
    J.seqs = A.seqs; J.h_off = A.seq_off; J.L = A.span_L;
    J.force_wide = (A.flags & MIRFOLD_FLAG_WIDE) != 0 || env_wide || A.span_L > MF16_MAX_SPAN;
    J.serial = (A.flags & MIRFOLD_FLAG_SERIAL) != 0 || env_serial;
    J.sink = A.sink;
    std::mutex cb_mu;
    std::atomic<int> cb_abort{0};
    J.fn = A.fn; J.user = A.user; J.cb_mu = &cb_mu; J.cb_abort = &cb_abort;
    J.cand = A.cand; J.collect = A.collect; J.totals = A.totals;

    std::unique_ptr<ResultOwner> R;
    SharedOut S;
    const uint64_t nt_total = nseq ? A.seq_off[nseq] - A.seq_off[0] : 0;
    if (A.sink == SINK_SHARED || A.sink == SINK_NONE) {
        R.reset(new ResultOwner());
        R->ctx = ctx;
        R->hit_begin.assign((size_t)nseq + 1, 0);
        R->hit_count.assign((size_t)nseq + 1, 0);
        R->totals.assign((size_t)nseq + 1, 0);
    }
    if (A.sink == SINK_SHARED) {
        // capacity is an estimate (a chunk that does not fit takes the overflow path below); MIRFOLD_RESULT_CAP_SCALE
        // shrinks it so that tests can reach that path
        const char *cs = getenv("MIRFOLD_RESULT_CAP_SCALE");
        const double scale = cs ? atof(cs) : 1.25;
        S.hits_cap = (uint64_t)(ctx->hits_per_nt * scale * (double)nt_total) + (cs ? 1 : 4096);
        S.arena_cap = (uint64_t)(ctx->arena_per_nt * scale * (double)nt_total) + (cs ? 1 : 65536);
        S.hits = pool_take(ctx, ctx->hits_pool, S.hits_cap * sizeof(mirfold_hit));
        S.arena = pool_take(ctx, ctx->arena_pool, S.arena_cap);
        cudaSetDevice(ctx->devs[0].id);
        if (S.hits.ensure(S.hits_cap * sizeof(mirfold_hit)) != cudaSuccess || S.arena.ensure(S.arena_cap) != cudaSuccess) {
            cudaGetLastError();
            S.hits.release(); S.arena.release();
            ctx->last_error = "pinned result buffers";
            return MIRFOLD_ERR_NOMEM;
        }
        if (!cs) { S.hits_cap = S.hits.cap / sizeof(mirfold_hit); S.arena_cap = S.arena.cap; }
        S.hit_begin = R->hit_begin.data(); S.hit_count = R->hit_count.data(); S.totals = R->totals.data();
        J.shared = &S;
    }
    ht.mark("result buffers");

    std::vector<DevOut> parts(G);
    auto dev_raw = [&](int g) { return A.d_raw ? (const char *)(*A.d_raw)[g] : nullptr; };
    if (G == 1) run_device(ctx->devs[0], J, shard[0], dev_raw(0), A.raw_off, parts[0]);
    else {
        std::vector<std::thread> th;
        for (int g = 0; g < G; g++)
            th.emplace_back([&, g] { run_device(ctx->devs[g], J, shard[g], dev_raw(g), A.raw_off, parts[g]); });
        for (auto &t : th) t.join();
    }
    for (int g = 0; g < G; g++)
        if (parts[g].err != MIRFOLD_OK) {
            ctx->last_error = parts[g].errmsg;
            std::lock_guard<std::mutex> lk(ctx->pool_mu);
            pool_give(ctx, ctx->hits_pool, S.hits);
            pool_give(ctx, ctx->arena_pool, S.arena);
            return parts[g].err;
        }
    ht.mark("devices");
    mirfold_stats st{};
    uint64_t nhits = 0, abytes = 0;
    for (int g = 0; g < G; g++) { add_stats(st, parts[g].st); nhits += parts[g].nhits; abytes += parts[g].arena_bytes; }
    st.n_devices = G;

    if (A.sink == SINK_CAND || A.sink == SINK_TOTALS) {
        st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (stats_out) *stats_out = st;
        if (A.nhits_out) *A.nhits_out = nhits;
        return MIRFOLD_OK;
    }
    if (A.sink == SINK_STREAM) {
        // records without a DP band (shorter than 5 nt) were never part of a device chunk
        std::vector<uint32_t> rec;
        for (uint32_t r = 0; r < nseq; r++) if (A.seq_off[r + 1] - A.seq_off[r] < 5) rec.push_back(r);
        if (!rec.empty()) {
            std::vector<uint64_t> hb(rec.size(), 0);
            std::vector<uint32_t> hc(rec.size(), 0);
            std::vector<int32_t> tot(rec.size(), 0);
            mirfold_chunk c{};
            c.n_records = (uint32_t)rec.size(); c.device = -1;
            c.record = rec.data(); c.hit_begin = hb.data(); c.hit_count = hc.data(); c.total_mfe_dcal = tot.data();
            if (A.fn(A.user, &c) != 0) { ctx->last_error = "chunk callback returned non-zero"; return MIRFOLD_ERR_CALLBACK; }
        }
        st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (stats_out) *stats_out = st;
        return MIRFOLD_OK;
    }

    if (A.sink == SINK_SHARED) {
        if (!S.overflow.empty()) {
            // the capacity estimate was too small: one exact-size copy, and a better estimate for the next call
            uint64_t th = S.hits_used, ta = S.arena_used;
            for (auto &o : S.overflow) { th += o->nhits; ta += o->abytes; }
            HBuf nh, na;
            if (nh.ensure(th * sizeof(mirfold_hit) + 16) != cudaSuccess || na.ensure(ta + 16) != cudaSuccess) {
                cudaGetLastError();
                nh.release(); na.release(); S.hits.release(); S.arena.release();
                return MIRFOLD_ERR_NOMEM;
            }
            memcpy(nh.p, S.hits.p, S.hits_used * sizeof(mirfold_hit));
            memcpy(na.p, S.arena.p, S.arena_used);
            uint64_t hb = S.hits_used, ab = S.arena_used;
            for (auto &o : S.overflow) {
                mirfold_hit *dst = nh.as<mirfold_hit>() + hb;
                memcpy(dst, o->hits.p, o->nhits * sizeof(mirfold_hit));
                for (uint64_t h = 0; h < o->nhits; h++) dst[h].ss_off += ab;
                memcpy(na.as<char>() + ab, o->arena.p, o->abytes);
                for (size_t k = 0; k < o->recs.size(); k++) { S.hit_begin[o->recs[k]] = hb + o->begin[k]; S.hit_count[o->recs[k]] = o->count[k]; }
                hb += o->nhits; ab += o->abytes;
                o->hits.release(); o->arena.release();
            }
            S.hits.release(); S.arena.release();
            S.hits = nh; S.arena = na;
            S.hits_used = th; S.arena_used = ta;
        }
        if (nt_total && !getenv("MIRFOLD_RESULT_CAP_SCALE")) {
            ctx->hits_per_nt = std::max(ctx->hits_per_nt, (double)S.hits_used / (double)nt_total);
            ctx->arena_per_nt = std::max(ctx->arena_per_nt, (double)S.arena_used / (double)nt_total);
        }
        R->hits = S.hits; S.hits = HBuf();
        R->arena = S.arena; S.arena = HBuf();
        R->pub.hits = R->hits.as<mirfold_hit>();
        R->pub.ss_arena = R->arena.as<char>();
        if (R->arena.cap > abytes) R->arena.as<char>()[abytes] = 0;
    } else {
        R->pub.hits = nullptr;
        R->pub.ss_arena = nullptr;
    }
    ht.mark("publish");
    st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    R->pub.nseq = nseq;
    R->pub.nhits = nhits;
    R->pub.ss_bytes = abytes;
    R->pub.hit_begin = R->hit_begin.data();
    R->pub.hit_count = R->hit_count.data();
    R->pub.total_mfe_dcal = R->totals.data();
    R->pub.stats = st;
    if (stats_out) *stats_out = st;
    {
        std::lock_guard<std::mutex> lk(ctx->pool_mu);
        ctx->live_results++;
    }
    *out = &R.release()->pub;
    return MIRFOLD_OK;
}

}  // namespace

// ====================================================================================== C ABI
extern "C" {

const char *mirfold_version(void) { return "mirfold " MIRFOLD_VERSION " sm_100a " MIRFOLD_PARAMSET_DEFAULT; }

const char *mirfold_strerror(int code)
{
    switch (code) {
    case MIRFOLD_OK: return "ok";
    case MIRFOLD_ERR_NO_DEVICE: return "no usable CUDA device (libmirfold has no CPU fallback)";
    case MIRFOLD_ERR_CUDA: return "CUDA runtime error";
    case MIRFOLD_ERR_ARG: return "invalid argument";
    case MIRFOLD_ERR_PARAMSET: return "unknown energy parameter set";
    case MIRFOLD_ERR_BACKTRACK: return "backtrack failed";
    case MIRFOLD_ERR_NOMEM: return "out of memory";
    case MIRFOLD_ERR_CALLBACK: return "chunk callback returned non-zero";
    default: return "unknown error";
    }
}

const char *mirfold_last_error(const mirfold_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }

int mirfold_open(mirfold_ctx **pctx, const int *device_ids, int n_devices, const char *param_set)
{
    if (!pctx) return MIRFOLD_ERR_ARG;
    *pctx = nullptr;
    if (param_set && strcmp(param_set, MIRFOLD_PARAMSET_DEFAULT) != 0) return MIRFOLD_ERR_PARAMSET;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return MIRFOLD_ERR_NO_DEVICE; }
    std::vector<int> ids;
    if (!device_ids || n_devices <= 0) {
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) return MIRFOLD_ERR_NO_DEVICE;
        ids.push_back(cur);
    } else {
        for (int k = 0; k < n_devices; k++) {
            if (device_ids[k] < 0 || device_ids[k] >= ndev) return MIRFOLD_ERR_NO_DEVICE;
            ids.push_back(device_ids[k]);
        }
    }
    mirfold_ctx *ctx = new mirfold_ctx();
    DevParams *hp = new DevParams();
    build_params(*hp);
    int rc = MIRFOLD_OK;
    ctx->devs.resize(ids.size());
    size_t made = 0;
    for (size_t k = 0; k < ids.size() && rc == MIRFOLD_OK; k++) {
        Device &D = ctx->devs[k];
        D.id = ids[k];
        made = k + 1;
        // the same ordinal may be listed more than once (each entry is an independent pipeline sharing the GPU):
        // the memory budget is split between the entries
        int share = 0;
        for (int id : ids) share += id == D.id;
        int prio_lo = 0, prio_hi = 0;
        cudaError_t e = cudaSetDevice(D.id);
        if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        for (int l = 0; l < 2; l++) if (e == cudaSuccess) e = D.lane[l].create(prio_hi);
        if (e == cudaSuccess) e = cudaEventCreate(&D.ev_first);
        if (e == cudaSuccess) e = cudaEventCreate(&D.ev_last);
        if (e == cudaSuccess) e = cudaMalloc(&D.dP, sizeof(DevParams));
        if (e == cudaSuccess) e = cudaMemcpy(D.dP, hp, sizeof(DevParams), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = fill_configure_device();
        size_t fr = 0, tot = 0;
        if (e == cudaSuccess) e = cudaMemGetInfo(&fr, &tot);
        if (e != cudaSuccess) { ctx->last_error = cudaGetErrorString(e); cudaGetLastError(); rc = MIRFOLD_ERR_CUDA; break; }
        const char *env = getenv("MIRFOLD_MEM_BUDGET_MB");
        D.mem_budget = env ? (size_t)atoll(env) << 20 : std::min<size_t>((size_t)(fr * 0.60), (size_t)96 << 30) / (size_t)share;
    }
    delete hp;
    if (rc != MIRFOLD_OK) {
        for (size_t k = 0; k < made; k++) { cudaSetDevice(ctx->devs[k].id); ctx->devs[k].release(); }
        delete ctx;
        return rc;
    }
    *pctx = ctx;
    return MIRFOLD_OK;
}

void mirfold_close(mirfold_ctx *ctx)
{
    if (!ctx) return;
    bool del;
    {
        std::lock_guard<std::mutex> lk(ctx->pool_mu);
        if (ctx->closed) return;
        ctx->closed = true;
        for (auto &D : ctx->devs) { cudaSetDevice(D.id); cudaDeviceSynchronize(); D.release(); }
        ctx->devs.clear();
        for (auto &b : ctx->arena_pool) b.release();
        for (auto &b : ctx->hits_pool) b.release();
        ctx->arena_pool.clear(); ctx->hits_pool.clear();
        del = ctx->live_results == 0 && ctx->live_genomes == 0;
    }
    if (del) delete ctx;   // otherwise the last mirfold_free_result() / mirfold_genome_free() deletes it
}

int mirfold_fold(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L, uint32_t flags,
                 mirfold_result **out)
{
    if (!out) return MIRFOLD_ERR_ARG;
    FoldArgs A;
    A.seqs = seqs; A.seq_off = seq_off; A.nseq = nseq; A.span_L = span_L; A.flags = flags; A.sink = SINK_SHARED;
    return fold_engine(ctx, A, out, nullptr);
}

int mirfold_fold_stream(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L, uint32_t flags,
                        mirfold_chunk_fn fn, void *user, mirfold_stats *stats)
{
    if (!fn) return MIRFOLD_ERR_ARG;
    FoldArgs A;
    A.seqs = seqs; A.seq_off = seq_off; A.nseq = nseq; A.span_L = span_L; A.flags = flags; A.sink = SINK_STREAM;
    A.fn = fn; A.user = user;
    return fold_engine(ctx, A, nullptr, stats);
}

int mirfold_fold_device(mirfold_ctx *ctx, const void *d_seqs, const void *d_seq_off, const uint64_t *h_seq_off,
                        uint32_t nseq, int span_L, uint32_t flags, void *stream, mirfold_result **out)
{
    (void)d_seq_off;
    if (!d_seqs || !out || !ctx || ctx->closed) return MIRFOLD_ERR_ARG;
    cudaSetDevice(ctx->devs[0].id);
    if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) { cudaGetLastError(); return MIRFOLD_ERR_CUDA; }   // the caller's producer
    std::vector<void *> d_raw(1, const_cast<void *>(d_seqs));
    FoldArgs A;
    A.seq_off = h_seq_off; A.nseq = nseq; A.span_L = span_L; A.flags = flags; A.sink = SINK_NONE;
    A.d_raw = &d_raw; A.raw_off = h_seq_off; A.n_devices = 1;
    return fold_engine(ctx, A, out, nullptr);
}

int mirfold_batch_upload(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L, mirfold_batch **out)
{
    if (!ctx || !out || !seq_off || (!seqs && nseq) || ctx->closed) return MIRFOLD_ERR_ARG;
    *out = nullptr;
    if (span_L < 5 || span_L > MF_MAX_SPAN) { ctx->last_error = "span_L out of range [5, 4096]"; return MIRFOLD_ERR_ARG; }
    int rc = validate_offsets(ctx, seq_off, nseq, span_L);
    if (rc != MIRFOLD_OK) return rc;
    std::unique_ptr<mirfold_batch> B(new mirfold_batch());
    B->ctx = ctx; B->nseq = nseq; B->span_L = span_L;
    B->h_off.assign(seq_off, seq_off + (size_t)nseq + 1);
    const int G = (int)ctx->devs.size();
    std::vector<uint64_t> load;
    plan_shards(seq_off, nseq, span_L, G, B->shard, load);
    B->raw_off.assign((size_t)nseq + 1, 0);
    B->d_raw.assign((size_t)G, nullptr);
    for (int g = 0; g < G; g++) {
        uint64_t bytes = 0;
        for (uint32_t r : B->shard[g]) { B->raw_off[r] = bytes; bytes += seq_off[r + 1] - seq_off[r]; }
        std::vector<char> stage((size_t)bytes + 1);
        for (uint32_t r : B->shard[g]) memcpy(stage.data() + B->raw_off[r], seqs + seq_off[r], (size_t)(seq_off[r + 1] - seq_off[r]));
        cudaError_t e = cudaSetDevice(ctx->devs[g].id);
        if (e == cudaSuccess) e = cudaMalloc(&B->d_raw[g], (size_t)bytes + 16);
        if (e == cudaSuccess) e = cudaMemcpy(B->d_raw[g], stage.data(), (size_t)bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            ctx->last_error = cudaGetErrorString(e);
            cudaGetLastError();
            mirfold_batch_free(B.release());
            return e == cudaErrorMemoryAllocation ? MIRFOLD_ERR_NOMEM : MIRFOLD_ERR_CUDA;
        }
    }
    *out = B.release();
    return MIRFOLD_OK;
}

int mirfold_batch_fold(mirfold_ctx *ctx, mirfold_batch *B, uint32_t flags, int download, mirfold_result **out)
{
    if (!ctx || !B || B->ctx != ctx || !out) return MIRFOLD_ERR_ARG;
    FoldArgs A;
    A.seq_off = B->h_off.data(); A.nseq = B->nseq; A.span_L = B->span_L; A.flags = flags;
    A.sink = download ? SINK_SHARED : SINK_NONE;
    A.d_raw = &B->d_raw; A.raw_off = B->raw_off.data(); A.shard = &B->shard;
    return fold_engine(ctx, A, out, nullptr);
}

void mirfold_batch_free(mirfold_batch *B)
{
    if (!B) return;
    if (B->ctx && !B->ctx->closed)
        for (size_t g = 0; g < B->d_raw.size() && g < B->ctx->devs.size(); g++)
            if (B->d_raw[g]) { cudaSetDevice(B->ctx->devs[g].id); cudaFree(B->d_raw[g]); }
    delete B;
}

namespace {
struct CandOwner {
    mirfold_candidates pub;
    CandCollector c;
};

// mirfold_fold_candidates / mirfold_fold_candidates_regions: A carries the input (host text or genome regions)
int fold_candidates_engine(mirfold_ctx *ctx, FoldArgs &A, const mirfold_region *regions, const mirfold_mature *matures,
                           const uint64_t *mature_off, int minlen, int minloop, int min_mature_len, int max_mature_len,
                           mirfold_candidates **out)
{
    const uint32_t nseq = A.nseq;
    for (uint32_t r = 0; r < nseq; r++) if (mature_off[r + 1] < mature_off[r]) { ctx->last_error = "mature_off is not non-decreasing"; return MIRFOLD_ERR_ARG; }
    std::unique_ptr<CandOwner> O(new CandOwner());
    O->c.struct_begin.assign((size_t)nseq + 1, 0);
    O->c.struct_count.assign((size_t)nseq + 1, 0);
    CandArgs ca;
    ca.regions = regions; ca.matures = matures; ca.mature_off = mature_off; ca.nseq = nseq;
    ca.minlen = minlen; ca.minloop = minloop; ca.min_mature = min_mature_len; ca.max_mature = max_mature_len;
    A.sink = SINK_CAND;
    A.cand = &ca; A.collect = &O->c;
    uint64_t nhits = 0;
    A.nhits_out = &nhits;
    mirfold_stats st{};
    const int rc = fold_engine(ctx, A, nullptr, &st);
    if (rc != MIRFOLD_OK) return rc;
    CandCollector &c = O->c;
    mirfold_candidates &p = O->pub;
    p = mirfold_candidates{};
    p.nseq = nseq;
    p.nstructs = c.structs.size();
    p.struct_begin = c.struct_begin.data(); p.struct_count = c.struct_count.data();
    p.structs = c.structs.data();
    c.arena.push_back(0);
    p.ss_arena = c.arena.data(); p.ss_bytes = c.arena.size() - 1;
    p.nverdicts = c.verdicts.size();
    p.verdict_begin = c.verdict_begin.data(); p.verdict_count = c.verdict_count.data();
    p.verdicts = c.verdicts.data(); p.verdict_mature = c.verdict_mature.data();
    p.nhits = nhits;
    p.stats = st;
    *out = &O.release()->pub;
    return MIRFOLD_OK;
}

// Genome regions -> the engine's inputs, in one pass: a synthetic seq_off from the clipped lengths (shard plan, chunking
// and every per-record table work from it unchanged) and per record raw_off = contig start + start - 1 into the device
// replica, | MF_RAW_REVERSE on the minus strand.  Clipping is samtools faidx's on "seqid:start-(end-1)" (FastaIndex.fetch).
struct RegionInput {
    std::vector<uint64_t> seq_off, raw_off;
    std::vector<mirfold_region> cand;   // the unclipped (start, end): the region the duplex checks see
};
int region_input(mirfold_ctx *ctx, const mirfold_genome *g, const mirfold_genome_region *reg, uint32_t nseq, bool cand, RegionInput &I)
{
    if (!ctx || !g || (!reg && nseq) || ctx->closed) return MIRFOLD_ERR_ARG;
    if (g->ctx != ctx) { ctx->last_error = "the genome belongs to another context"; return MIRFOLD_ERR_ARG; }
    const int64_t nc = (int64_t)g->contig_off.size() - 1;
    I.seq_off.resize((size_t)nseq + 1);
    I.raw_off.resize((size_t)nseq + 1);
    if (cand) I.cand.resize((size_t)nseq + 1);
    I.seq_off[0] = 0;
    uint64_t acc = 0;
    char msg[128];
    for (uint32_t r = 0; r < nseq; r++) {
        const mirfold_genome_region &x = reg[r];
        if (x.strand != '+' && x.strand != '-') {
            snprintf(msg, sizeof msg, "region %u: strand %d is neither '+' nor '-'", r, x.strand);
            ctx->last_error = msg;
            return MIRFOLD_ERR_ARG;
        }
        if (x.contig < -1 || x.contig >= nc) {
            snprintf(msg, sizeof msg, "region %u: contig %d out of range [-1, %lld)", r, x.contig, (long long)nc);
            ctx->last_error = msg;
            return MIRFOLD_ERR_ARG;
        }
        uint64_t len = 0, raw = 0;
        if (x.contig >= 0) {
            const uint64_t base = g->contig_off[x.contig], clen = g->contig_off[x.contig + 1] - base;
            const int64_t s = std::max<int64_t>(x.start, 1), e = std::min<int64_t>((int64_t)x.end - 1, (int64_t)clen);
            if (s <= e) { len = (uint64_t)(e - s + 1); raw = base + (uint64_t)(s - 1); }
        }
        I.raw_off[r] = raw | (x.strand == '-' ? MF_RAW_REVERSE : 0ULL);
        acc += len;
        I.seq_off[r + 1] = acc;
        if (cand) I.cand[r] = mirfold_region{x.start, x.end};
    }
    return MIRFOLD_OK;
}
}  // namespace

int mirfold_fold_candidates(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L, uint32_t flags,
                            const mirfold_region *regions, const mirfold_mature *matures, const uint64_t *mature_off, int minlen,
                            int minloop, int min_mature_len, int max_mature_len, mirfold_candidates **out)
{
    if (!ctx || !out || !seq_off || (!regions && nseq) || !mature_off || (!matures && mature_off[nseq])) return MIRFOLD_ERR_ARG;
    *out = nullptr;
    FoldArgs A;
    A.seqs = seqs; A.seq_off = seq_off; A.nseq = nseq; A.span_L = span_L; A.flags = flags;
    return fold_candidates_engine(ctx, A, regions, matures, mature_off, minlen, minloop, min_mature_len, max_mature_len, out);
}

int mirfold_genome_upload(mirfold_ctx *ctx, const char *seq, const uint64_t *contig_off, uint32_t n_contigs, mirfold_genome **out)
{
    if (!ctx || !out || !contig_off || ctx->closed) return MIRFOLD_ERR_ARG;
    *out = nullptr;
    for (uint32_t c = 0; c < n_contigs; c++)
        if (contig_off[c + 1] < contig_off[c]) { ctx->last_error = "contig_off is not non-decreasing"; return MIRFOLD_ERR_ARG; }
    const uint64_t bytes = contig_off[n_contigs] - contig_off[0];
    if (!seq && bytes) return MIRFOLD_ERR_ARG;
    std::unique_ptr<mirfold_genome> G(new mirfold_genome());
    G->ctx = ctx;
    G->contig_off.resize((size_t)n_contigs + 1);
    for (uint32_t c = 0; c <= n_contigs; c++) G->contig_off[c] = contig_off[c] - contig_off[0];
    const size_t nd = ctx->devs.size();
    G->d_raw.assign(nd, nullptr);
    G->budget_taken.assign(nd, 0);
    cudaError_t e = cudaSuccess;
    for (size_t k = 0; k < nd && e == cudaSuccess; k++) {
        Device &D = ctx->devs[k];
        const size_t j = std::find(G->ordinal.begin(), G->ordinal.end(), D.id) - G->ordinal.begin();
        if (j == G->ordinal.size()) {
            void *p = nullptr;
            e = cudaSetDevice(D.id);
            if (e == cudaSuccess) e = cudaMalloc(&p, (size_t)bytes + 16);
            if (e != cudaSuccess) break;
            G->ordinal.push_back(D.id);
            G->replica.push_back(p);
            if (bytes) e = cudaMemcpyAsync(p, seq + contig_off[0], (size_t)bytes, cudaMemcpyHostToDevice, D.lane[0].s_lo);
            if (e == cudaSuccess) e = cudaStreamSynchronize(D.lane[0].s_lo);
        }
        G->d_raw[k] = G->replica[j];
    }
    if (e != cudaSuccess) {
        ctx->last_error = std::string("genome upload: ") + cudaGetErrorString(e);
        cudaGetLastError();
        for (size_t j = 0; j < G->ordinal.size(); j++) { cudaSetDevice(G->ordinal[j]); cudaFree(G->replica[j]); }
        return e == cudaErrorMemoryAllocation ? MIRFOLD_ERR_NOMEM : MIRFOLD_ERR_CUDA;
    }
    // the lanes' budget was set from free HBM at mirfold_open; the replica now occupies part of it (split between the entries
    // of one ordinal like the budget itself).  An explicit MIRFOLD_MEM_BUDGET_MB is taken as given.
    std::lock_guard<std::mutex> lk(ctx->pool_mu);
    if (!getenv("MIRFOLD_MEM_BUDGET_MB"))
        for (size_t k = 0; k < nd; k++) {
            Device &D = ctx->devs[k];
            size_t share = 0;
            for (const Device &o : ctx->devs) share += o.id == D.id;
            const size_t keep = std::min(D.mem_budget, (size_t)256 << 20);
            G->budget_taken[k] = std::min((size_t)bytes / share, D.mem_budget - keep);
            D.mem_budget -= G->budget_taken[k];
        }
    ctx->live_genomes++;
    *out = G.release();
    return MIRFOLD_OK;
}

void mirfold_genome_free(mirfold_genome *g)
{
    if (!g) return;
    for (size_t j = 0; j < g->ordinal.size(); j++) { cudaSetDevice(g->ordinal[j]); cudaFree(g->replica[j]); }
    mirfold_ctx *ctx = g->ctx;
    bool del;
    {
        std::lock_guard<std::mutex> lk(ctx->pool_mu);
        if (!ctx->closed)
            for (size_t k = 0; k < ctx->devs.size() && k < g->budget_taken.size(); k++) ctx->devs[k].mem_budget += g->budget_taken[k];
        ctx->live_genomes--;
        del = ctx->closed && ctx->live_results == 0 && ctx->live_genomes == 0;
    }
    delete g;
    if (del) delete ctx;
}

int mirfold_fold_regions(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions, uint32_t nseq,
                         int span_L, uint32_t flags, mirfold_result **out)
{
    if (!out) return MIRFOLD_ERR_ARG;
    *out = nullptr;
    RegionInput I;
    const int rc = region_input(ctx, genome, regions, nseq, false, I);
    if (rc != MIRFOLD_OK) return rc;
    FoldArgs A;
    A.seq_off = I.seq_off.data(); A.nseq = nseq; A.span_L = span_L; A.flags = flags; A.sink = SINK_SHARED;
    A.d_raw = &genome->d_raw; A.raw_off = I.raw_off.data();
    return fold_engine(ctx, A, out, nullptr);
}

int mirfold_fold_regions_stream(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions, uint32_t nseq,
                                int span_L, uint32_t flags, mirfold_chunk_fn fn, void *user, mirfold_stats *stats)
{
    if (!fn) return MIRFOLD_ERR_ARG;
    RegionInput I;
    const int rc = region_input(ctx, genome, regions, nseq, false, I);
    if (rc != MIRFOLD_OK) return rc;
    FoldArgs A;
    A.seq_off = I.seq_off.data(); A.nseq = nseq; A.span_L = span_L; A.flags = flags; A.sink = SINK_STREAM;
    A.fn = fn; A.user = user;
    A.d_raw = &genome->d_raw; A.raw_off = I.raw_off.data();
    return fold_engine(ctx, A, nullptr, stats);
}

int mirfold_fold_candidates_regions(mirfold_ctx *ctx, const mirfold_genome *genome, const mirfold_genome_region *regions, uint32_t nseq,
                                    int span_L, uint32_t flags, const mirfold_mature *matures, const uint64_t *mature_off, int minlen,
                                    int minloop, int min_mature_len, int max_mature_len, mirfold_candidates **out)
{
    if (!out || !mature_off || (!matures && mature_off[nseq])) return MIRFOLD_ERR_ARG;
    *out = nullptr;
    RegionInput I;
    const int rc = region_input(ctx, genome, regions, nseq, true, I);
    if (rc != MIRFOLD_OK) return rc;
    FoldArgs A;
    A.seq_off = I.seq_off.data(); A.nseq = nseq; A.span_L = span_L; A.flags = flags;
    A.d_raw = &genome->d_raw; A.raw_off = I.raw_off.data();
    return fold_candidates_engine(ctx, A, I.cand.data(), matures, mature_off, minlen, minloop, min_mature_len, max_mature_len, out);
}

void mirfold_free_candidates(mirfold_candidates *c)
{
    if (c) delete reinterpret_cast<CandOwner *>(c);
}

}  // extern "C"

namespace {
// ---- MFE significance against shuffles (mirfold_shuffle_test / mirfold_shuffle_sequences)
int shuffle_args(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int mode)
{
    if (!ctx || ctx->closed || !seq_off || (!seqs && nseq)) return MIRFOLD_ERR_ARG;
    if (mode != MIRFOLD_SHUFFLE_MONO && mode != MIRFOLD_SHUFFLE_DI) { ctx->last_error = "unknown shuffle mode"; return MIRFOLD_ERR_ARG; }
    const int rc = validate_offsets(ctx, seq_off, nseq, 0);   // the span is checked by mirfold_shuffle_test
    if (rc != MIRFOLD_OK) return rc;
    if (mode == MIRFOLD_SHUFFLE_DI)
        for (uint32_t r = 0; r < nseq; r++) {
            bool seen[256] = {};
            int ns = 0;
            for (uint64_t t = seq_off[r]; t < seq_off[r + 1]; t++) {
                unsigned char c = (unsigned char)seqs[t];
                if (c >= 'a' && c <= 'z') c -= 32;
                if (c == 'T') c = 'U';
                if (!seen[c]) { seen[c] = true; ns++; }
            }
            if (ns > MF_SHUF_MAX_SYMBOLS) {
                char msg[128];
                snprintf(msg, sizeof msg, "record %u has %d distinct symbols; dinucleotide shuffles allow %d", r, ns, MF_SHUF_MAX_SYMBOLS);
                ctx->last_error = msg;
                return MIRFOLD_ERR_ARG;
            }
        }
    return MIRFOLD_OK;
}

// the records, rebased to offset 0 (off), onto device D
cudaError_t shuffle_upload(Device &D, const char *seqs, const std::vector<uint64_t> &off)
{
    const size_t nseq = off.size() - 1, bytes = (size_t)off.back();
    cudaError_t e = cudaSetDevice(D.id);
    if (e == cudaSuccess) e = D.shuf_in.ensure(bytes + 16);
    if (e == cudaSuccess) e = D.shuf_off.ensure(8 * (nseq + 1));
    if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(D.shuf_in.p, seqs, bytes, cudaMemcpyHostToDevice, D.lane[0].s_lo);
    if (e == cudaSuccess) e = cudaMemcpyAsync(D.shuf_off.p, off.data(), 8 * (nseq + 1), cudaMemcpyHostToDevice, D.lane[0].s_lo);
    if (e == cudaSuccess) e = cudaStreamSynchronize(D.lane[0].s_lo);
    return e;
}

// the round's replicates into D.shuf_raw (bytes in all); *bad = a record with too many symbols (checked on the host before)
cudaError_t shuffle_generate(Device &D, const std::vector<ShuffleItem> &items, uint64_t bytes, uint64_t seed, int mode, int *bad)
{
    cudaStream_t st = D.lane[0].s_lo;
    cudaError_t e = cudaSetDevice(D.id);
    if (e == cudaSuccess) e = D.shuf_items.ensure(sizeof(ShuffleItem) * items.size() + 16);
    if (e == cudaSuccess) e = D.shuf_raw.ensure(bytes + 16);
    if (e == cudaSuccess) e = D.shuf_scr.ensure(bytes + 16);
    if (e == cudaSuccess) e = D.shuf_fail.ensure(4);
    if (e == cudaSuccess) e = cudaMemsetAsync(D.shuf_fail.p, 0, 4, st);
    if (e == cudaSuccess && !items.empty())
        e = cudaMemcpyAsync(D.shuf_items.p, items.data(), sizeof(ShuffleItem) * items.size(), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        e = launch_shuffle(D.shuf_in.as<char>(), D.shuf_off.as<unsigned long long>(), D.shuf_items.as<ShuffleItem>(), (unsigned)items.size(),
                           D.shuf_raw.as<char>(), D.shuf_scr.as<unsigned char>(), seed, mode, D.shuf_fail.as<int>(), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bad, D.shuf_fail.p, 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e;
}

void add_stats_sequential(mirfold_stats &a, const mirfold_stats &b)   // engine calls that ran one after the other
{
    a.ms_h2d += b.ms_h2d; a.ms_fill += b.ms_fill; a.ms_f3 += b.ms_f3; a.ms_trace += b.ms_trace; a.ms_d2h += b.ms_d2h;
    a.ms_device += b.ms_device;
    a.nt += b.nt; a.cells += b.cells; a.tracebacks += b.tracebacks; a.kernel_launches += b.kernel_launches;
    a.h2d_bytes += b.h2d_bytes; a.d2h_bytes += b.d2h_bytes; a.n_chunks += b.n_chunks; a.fill_units += b.fill_units;
}

int cuda_fail(mirfold_ctx *ctx, cudaError_t e, const char *what)
{
    ctx->last_error = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? MIRFOLD_ERR_NOMEM : MIRFOLD_ERR_CUDA;
}
}  // namespace

extern "C" {

// Rounds: the (record, replicate) pairs of records of at least 5 nt, replicate-major, are cut into rounds of at most
// MIRFOLD_SHUFFLE_ROUND_NT nucleotides (default 2^27; a single longer pair is a round of its own).  Every device generates
// the whole round into its own raw buffer (cheaper than moving it), and the round is folded as a device-resident batch
// through the engine (LPT shards, chunks and lanes unchanged) with the totals-only sink.  The natives are folded once the
// same way.  The tally is integer arithmetic on the host, so it is exact and independent of the order of the rounds.
int mirfold_shuffle_test(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int span_L, uint32_t flags,
                         int mode, uint32_t n_shuffles, uint64_t seed, mirfold_shuffle_stat *out, mirfold_stats *stats)
{
    if (!out || n_shuffles == 0) return MIRFOLD_ERR_ARG;
    int rc = shuffle_args(ctx, seqs, seq_off, nseq, mode);
    if (rc != MIRFOLD_OK) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<uint64_t> off((size_t)nseq + 1);
    uint64_t max_n = 0;
    for (uint32_t r = 0; r <= nseq; r++) off[r] = seq_off[r] - seq_off[0];
    for (uint32_t r = 0; r < nseq; r++) max_n = std::max(max_n, off[r + 1] - off[r]);
    int L = span_L;
    if (span_L == 0) {   // global: L* = min(L, n) = n for every record
        if (max_n > MF_MAX_SPAN) { ctx->last_error = "span_L = 0 (global) needs records of at most 4096 nt"; return MIRFOLD_ERR_ARG; }
        L = (int)std::max<uint64_t>(max_n, 5);
    } else if (span_L < 5 || span_L > MF_MAX_SPAN) { ctx->last_error = "span_L out of range [5, 4096] (or 0)"; return MIRFOLD_ERR_ARG; }
    if ((rc = validate_offsets(ctx, seq_off, nseq, L)) != MIRFOLD_OK) return rc;
    const char *base = nseq ? seqs + seq_off[0] : seqs;
    mirfold_stats st{};
    for (Device &D : ctx->devs) {
        const cudaError_t e = shuffle_upload(D, base, off);
        if (e != cudaSuccess) return cuda_fail(ctx, e, "shuffle upload");
        st.h2d_bytes += off.back() + 8 * ((uint64_t)nseq + 1);
    }
    std::vector<void *> d_in, d_round;
    for (Device &D : ctx->devs) d_in.push_back(D.shuf_in.p);
    // natives
    std::vector<int32_t> native((size_t)nseq + 1, 0);
    {
        FoldArgs A;
        A.seq_off = off.data(); A.nseq = nseq; A.span_L = L; A.flags = flags; A.sink = SINK_TOTALS;
        A.d_raw = &d_in; A.raw_off = off.data(); A.totals = native.data();
        mirfold_stats s{};
        rc = fold_engine(ctx, A, nullptr, &s);
        if (rc != MIRFOLD_OK) return rc;
        add_stats_sequential(st, s);
    }
    std::vector<mirfold_shuffle_stat> res((size_t)nseq);
    std::vector<uint32_t> recs;
    for (uint32_t r = 0; r < nseq; r++) {
        res[r] = mirfold_shuffle_stat{native[r], 0, 0, 0};
        if (off[r + 1] - off[r] >= 5) recs.push_back(r);
        else res[r].n_le = n_shuffles;   // nothing to fold: every shuffle totals 0 == native
    }
    const char *env = getenv("MIRFOLD_SHUFFLE_ROUND_NT");
    const uint64_t round_nt = std::max<uint64_t>(env ? strtoull(env, nullptr, 10) : (1ull << 27), 1);
    std::vector<ShuffleItem> items;
    std::vector<uint64_t> roff;
    std::vector<int32_t> tot;
    size_t cursor = 0;
    const size_t npairs = recs.size() * (size_t)n_shuffles;
    while (cursor < npairs) {
        items.clear(); roff.assign(1, 0);
        for (; cursor < npairs; cursor++) {
            const uint32_t r = recs[cursor % recs.size()];
            const uint64_t n = off[r + 1] - off[r];
            if (!items.empty() && roff.back() + n > round_nt) break;
            items.push_back(ShuffleItem{r, (uint32_t)(cursor / recs.size()), roff.back()});
            roff.push_back(roff.back() + n);
        }
        d_round.clear();
        for (Device &D : ctx->devs) {
            int bad = 0;
            const cudaError_t e = shuffle_generate(D, items, roff.back(), seed, mode, &bad);
            if (e != cudaSuccess) return cuda_fail(ctx, e, "shuffle kernel");
            if (bad) { ctx->last_error = "a record has too many distinct symbols"; return MIRFOLD_ERR_ARG; }
            d_round.push_back(D.shuf_raw.p);
            st.h2d_bytes += sizeof(ShuffleItem) * items.size();
            st.kernel_launches += 1;
        }
        tot.assign(items.size(), 0);
        FoldArgs A;
        A.seq_off = roff.data(); A.nseq = (uint32_t)items.size(); A.span_L = L; A.flags = flags; A.sink = SINK_TOTALS;
        A.d_raw = &d_round; A.raw_off = roff.data(); A.totals = tot.data();
        mirfold_stats s{};
        rc = fold_engine(ctx, A, nullptr, &s);
        if (rc != MIRFOLD_OK) return rc;
        add_stats_sequential(st, s);
        for (size_t i = 0; i < items.size(); i++) {
            mirfold_shuffle_stat &o = res[items[i].rec];
            const int64_t t = tot[i];
            o.n_le += t <= (int64_t)o.native_dcal;
            o.sum_dcal += t;
            o.sumsq_dcal += t * t;
        }
    }
    if (nseq) memcpy(out, res.data(), sizeof(mirfold_shuffle_stat) * nseq);
    st.n_devices = (int32_t)ctx->devs.size();
    st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = st;
    return MIRFOLD_OK;
}

int mirfold_shuffle_sequences(mirfold_ctx *ctx, const char *seqs, const uint64_t *seq_off, uint32_t nseq, int mode, uint64_t seed,
                              uint32_t replicate, char *out)
{
    if (!out) return MIRFOLD_ERR_ARG;
    const int rc = shuffle_args(ctx, seqs, seq_off, nseq, mode);
    if (rc != MIRFOLD_OK) return rc;
    std::vector<uint64_t> off((size_t)nseq + 1);
    for (uint32_t r = 0; r <= nseq; r++) off[r] = seq_off[r] - seq_off[0];
    std::vector<ShuffleItem> items((size_t)nseq);
    for (uint32_t r = 0; r < nseq; r++) items[r] = ShuffleItem{r, replicate, off[r]};
    Device &D = ctx->devs[0];
    int bad = 0;
    cudaError_t e = shuffle_upload(D, nseq ? seqs + seq_off[0] : seqs, off);
    if (e == cudaSuccess) e = shuffle_generate(D, items, off.back(), seed, mode, &bad);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "shuffle kernel");
    if (bad) { ctx->last_error = "a record has too many distinct symbols"; return MIRFOLD_ERR_ARG; }
    if (off.back()) {
        e = cudaMemcpyAsync(out + seq_off[0], D.shuf_raw.p, (size_t)off.back(), cudaMemcpyDeviceToHost, D.lane[0].s_lo);
        if (e == cudaSuccess) e = cudaStreamSynchronize(D.lane[0].s_lo);
        if (e != cudaSuccess) return cuda_fail(ctx, e, "shuffle download");
    }
    return MIRFOLD_OK;
}

int mirfold_plan_shards(const uint64_t *seq_off, uint32_t nseq, int span_L, int n_shards, uint32_t *shard_of, uint64_t *shard_cells)
{
    if (!seq_off || n_shards < 1 || span_L < 5) return MIRFOLD_ERR_ARG;
    for (uint32_t r = 0; r < nseq; r++) if (seq_off[r + 1] < seq_off[r]) return MIRFOLD_ERR_ARG;
    std::vector<std::vector<uint32_t>> shard;
    std::vector<uint64_t> load;
    plan_shards(seq_off, nseq, span_L, n_shards, shard, load);
    for (int g = 0; g < n_shards; g++) {
        if (shard_of) for (uint32_t r : shard[g]) shard_of[r] = (uint32_t)g;
        if (shard_cells) shard_cells[g] = load[g] - shard[g].size();   // the plan weighs every record cells + 1
    }
    return MIRFOLD_OK;
}

int mirfold_plan_fill_units(uint32_t n, int span_L, mirfold_fill_plan *out)
{
    if (!out || n < 1 || n > 0x7fffffffu || span_L < 5) return MIRFOLD_ERR_ARG;
    LocusDesc d{};
    const unsigned long long be = shape_locus(d, (int)n, span_L);
    if (!band_offsets_fit(d)) return MIRFOLD_ERR_ARG;
    out->kernel = is_bucket_stride(d.stride) ? d.stride : 0;
    out->stride = d.stride;
    out->tile_len = d.tile_last ? d.stride : (int)n;
    out->tile_step = d.tile_last ? d.tile_step : (int)n;
    out->n_units = d.dmax >= 4 ? d.tile_last + 1 : 0;   // n < 5: nothing to fill
    out->dmax = d.dmax;
    out->band_cells = be;
    return MIRFOLD_OK;
}

int mirfold_plan_segments(uint32_t n, int span_L, uint64_t budget_bytes, mirfold_segment *segs, uint32_t cap, uint32_t *n_segments)
{
    if (!n_segments || n < 1 || n > 0x3fffffffu || span_L < 5 || span_L > MF_MAX_SPAN || (!segs && cap)) return MIRFOLD_ERR_ARG;
    LocusDesc d{};
    shape_locus(d, (int)n, span_L);
    if (!band_offsets_fit(d)) return MIRFOLD_ERR_ARG;
    std::vector<SegPlan> plan;
    plan_segments((int)n, span_L, (size_t)budget_bytes, plan);
    *n_segments = (uint32_t)plan.size();
    for (uint32_t k = 0; k < cap && k < plan.size(); k++) {
        const SegPlan &g = plan[k];
        segs[k] = mirfold_segment{g.t0, g.t1, g.halo, g.row_lo, g.row_hi, 0, (uint64_t)g.bytes};
    }
    return MIRFOLD_OK;
}

void mirfold_free_result(mirfold_result *res)
{
    if (!res) return;
    ResultOwner *R = reinterpret_cast<ResultOwner *>(res);
    mirfold_ctx *ctx = R->ctx;
    bool del = false;
    {
        std::lock_guard<std::mutex> lk(ctx->pool_mu);
        pool_give(ctx, ctx->arena_pool, R->arena);
        pool_give(ctx, ctx->hits_pool, R->hits);
        ctx->live_results--;
        del = ctx->closed && ctx->live_results == 0 && ctx->live_genomes == 0;
    }
    R->arena.release();
    R->hits.release();
    delete R;
    if (del) delete ctx;
}

int mirfold_debug_matrices(mirfold_ctx *ctx, const char *seq, uint32_t n, int span_L, uint32_t flags, int32_t *c, int32_t *m,
                           int32_t *f3)
{
    if (!ctx || ctx->closed || !seq || n < 5 || !c || !m || !f3) return MIRFOLD_ERR_ARG;
    Device &D = ctx->devs[0];
    Lane &Ln = D.lane[0];
#define CK(call)                                                                  \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) { ctx->last_error = cudaGetErrorString(e_); cudaGetLastError(); return MIRFOLD_ERR_CUDA; } \
    } while (0)
    CK(cudaSetDevice(D.id));
    cudaStream_t st = Ln.s_lo;
    LocusDesc d{};
    const unsigned long long cells = shape_locus(d, (int)n, span_L);
    if (!band_offsets_fit(d)) { ctx->last_error = "one fill unit of 2^31 band cells or more"; return MIRFOLD_ERR_ARG; }
    std::vector<LocusDesc> units;
    int bucket_first[6], max_n = 0;
    const unsigned long long ring_elems = build_fill_units(&d, 1, units, bucket_first, max_n);
    const int nu = (int)units.size();
    CK(Ln.raw.ensure(n)); CK(Ln.loci.ensure(sizeof d)); CK(Ln.codes.ensure(n + 3)); CK(Ln.F.ensure((n + 3) * 4));
    CK(Ln.C.ensure(cells * 4)); CK(Ln.M.ensure(cells * 4)); CK(Ln.Mp.ensure(cells * 4 + 4096)); CK(Ln.Ib.ensure(cells + 256));
    CK(Ln.ring.ensure((size_t)ring_elems * 4));
    CK(Ln.units.ensure(sizeof(LocusDesc) * (size_t)nu + 64));
    CK(cudaMemcpyAsync(Ln.raw.p, seq, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(Ln.loci.p, &d, sizeof d, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(Ln.units.p, units.data(), sizeof(LocusDesc) * (size_t)nu, cudaMemcpyHostToDevice, st));
    const LocusDesc *dl = Ln.loci.as<LocusDesc>();
    CK(launch_prepare(Ln.raw.as<char>(), dl, 1, n + 3, Ln.codes.as<unsigned char>(), Ln.F.as<int>(), st));
    CK(Ln.fillflags.ensure((size_t)nu * 4 + 4));
    CK(cudaMemsetAsync(Ln.fillflags.p, 0, (size_t)nu * 4 + 4, st));
    CK(launch_fill(fill_launch(Ln, D.dP, nu, max_n, bucket_first, (flags & MIRFOLD_FLAG_WIDE) || span_L > MF16_MAX_SPAN, span_L), st));
    CK(launch_f3(dl, 1, d.n > MF_TILE_LEN ? 1 : 0, d.Ls, Ln.codes.as<unsigned char>(), Ln.C.as<int>(), Ln.F.as<int>(), D.dP, st));
    std::vector<int> hc(cells), hm(cells), hf(n + 3);
    CK(cudaMemcpyAsync(hc.data(), Ln.C.p, cells * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hm.data(), Ln.M.p, cells * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hf.data(), Ln.F.p, (n + 3) * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const int W = d.Ls + 6;
    for (size_t k = 0; k < (size_t)(n + 2) * W; k++) c[k] = m[k] = MF_INF;
    for (int dd = 4; dd <= d.dmax; dd++)
        for (int i = 1; i <= (int)n - dd; i++) {
            // owner tile of row i (same mapping as band_row_base on the device)
            unsigned long long base = (unsigned long long)(i - 1);
            if (d.tile_last) {
                const int t = std::min((i - 1) / d.tile_step, d.tile_last);
                const int a = std::min(t * d.tile_step, (int)n - d.stride);
                base = (unsigned long long)t * band_elems(d.stride, d.dmax) + (unsigned long long)(i - 1 - a);
            }
            c[(size_t)i * W + dd] = hc[base + band_doff(d.stride, dd)];
            m[(size_t)i * W + dd] = hm[base + band_doff(d.stride, dd)];
        }
    for (uint32_t k = 0; k < n + 3; k++) f3[k] = hf[k];
    f3[n + 3] = 0;
    return MIRFOLD_OK;
}

int mirfold_int_peak(mirfold_ctx *ctx, double *addmin_terms_per_s, double *dpx_terms_per_s)
{
    if (!ctx || ctx->closed || !addmin_terms_per_s || !dpx_terms_per_s) return MIRFOLD_ERR_ARG;
    Device &D = ctx->devs[0];
    cudaSetDevice(D.id);
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, D.id);
    cudaError_t e = run_int_peak(D.lane[0].s_lo, sms, addmin_terms_per_s, dpx_terms_per_s, nullptr);
    if (e != cudaSuccess) { ctx->last_error = cudaGetErrorString(e); return MIRFOLD_ERR_CUDA; }
    return MIRFOLD_OK;
}

int mirfold_int_peak2(mirfold_ctx *ctx, double *addmin_terms_per_s, double *dpx_terms_per_s, double *s16x2_terms_per_s)
{
    if (!ctx || ctx->closed || !addmin_terms_per_s || !dpx_terms_per_s || !s16x2_terms_per_s) return MIRFOLD_ERR_ARG;
    Device &D = ctx->devs[0];
    cudaSetDevice(D.id);
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, D.id);
    cudaError_t e = run_int_peak(D.lane[0].s_lo, sms, addmin_terms_per_s, dpx_terms_per_s, s16x2_terms_per_s);
    if (e != cudaSuccess) { ctx->last_error = cudaGetErrorString(e); return MIRFOLD_ERR_CUDA; }
    return MIRFOLD_OK;
}

int mirfold_duplex(mirfold_ctx *ctx, const char *ss_arena, uint64_t ss_bytes, const mirfold_duplex_query *queries,
                   uint64_t nq, mirfold_duplex_verdict *verdicts)
{
    if (!ctx || ctx->closed || (!ss_arena && ss_bytes) || (!queries && nq) || (!verdicts && nq)) return MIRFOLD_ERR_ARG;
    if (nq == 0) return MIRFOLD_OK;
    int maxlen = 1;
    for (uint64_t k = 0; k < nq; k++) {
        if (queries[k].ss_len < 0 || queries[k].ss_off + (uint64_t)queries[k].ss_len > ss_bytes) {
            ctx->last_error = "mirfold_duplex: query structure outside the arena";
            return MIRFOLD_ERR_ARG;
        }
        maxlen = std::max(maxlen, queries[k].ss_len);
    }
    if (maxlen > 32000) { ctx->last_error = "mirfold_duplex: structure longer than 32000"; return MIRFOLD_ERR_ARG; }
    Device &D = ctx->devs[0];
    cudaStream_t st = D.lane[0].s_hi;
    CK(cudaSetDevice(D.id));
    CK(D.duplex_arena.ensure(ss_bytes + 16));
    CK(D.duplex_q.ensure(nq * sizeof(mirfold_duplex_query)));
    CK(D.duplex_v.ensure(nq * sizeof(mirfold_duplex_verdict)));
    CK(cudaMemcpyAsync(D.duplex_arena.p, ss_arena, ss_bytes, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(D.duplex_q.p, queries, nq * sizeof(mirfold_duplex_query), cudaMemcpyHostToDevice, st));
    CK(launch_duplex(D.duplex_arena.as<char>(), D.duplex_q.as<mirfold_duplex_query>(), nq, D.duplex_v.as<mirfold_duplex_verdict>(),
                     (maxlen + 7) & ~7, st));
    CK(cudaMemcpyAsync(verdicts, D.duplex_v.p, nq * sizeof(mirfold_duplex_verdict), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return MIRFOLD_OK;
}
#undef CK

}  // extern "C"
