// Balanced assignment (the reference's `auction_lap_half`, balancekmeans/__init__.py:12-140) as
// HBM-streaming sm_100a kernels.
//
// Data in HBM
//   S      [K][ld] fp16, worker(cluster)-major score matrix = (-dist).half().T  (:29,:40); ld is a
//          multiple of 128 and columns >= N hold -inf.  Written once by the score pass, read once
//          per pass here.  Never modified.
//   cost   [ld] fp16 (:55), owner [ld] int16 = the winner recorded in `index` (:122), -1 = job had
//          no bidder in the previous round (= `jobs_without_bidder`, :96).
//   `value` (:119-123) and `bids` (:49,:82-89) are never materialised: value[w][j] is recomputed as
//          owner[j]==w ? S[w][j] : S[w][j]-cost[j] (one fp16 rounding, like the reference) while S
//          streams through shared memory, and bids are reduced to (highest bid, first highest
//          bidder) per job on the fly.
//
// A ROUND of the reference finds each worker's threshold T_w, the (N/K+1)-th largest value (:66), and then bids.
// Here that is a chain of kernels; a device-side state machine decides what the round needs, and a kernel whose turn
// it is not returns at once.
//   window sampling  (auction_sample_kernel, K CTAs) a strided 8192-job sample of each worker's current values
//            brackets the threshold's rank (+-4.5 sigma of the order statistic, capped by the previous threshold:
//            costs only grow, so thresholds only sink); 256 one-key bins are laid over that bracket (split in two
//            runs around the widest sampled hole if it is wider than 256 keys, coarser bins if even that does not
//            fit) plus "above" / "gap" counters.
//   HIST pass  (auction_hist_kernel, G CTAs) the exact 16-bit radix select over that window.  Warps stream row
//            segments straight from global memory (16-byte loads, four in flight per lane): per 8 jobs 1 LDG.128
//            + 1 LDS.128 + 4 HSUB2 + 4 HSET2 + 4 LOP3.  The ~1.5 % survivors (values at or above the window's low
//            edge) are histogrammed in 16-bit packed shared-memory counters and appended to the survivor list of
//            their (4096-job sub-range, worker).  The histograms are dumped per CTA (or, in the step-by-step flow,
//            merged with atomics into the reduce block).
//   merge + resolve  (auction_merge_resolve_kernel, one CTA per worker) sums the worker's dumps, turns them into an
//            exact threshold (hit -> exact; miss -> slide / refine / coarse restart; a coarse bin is refined from
//            the survivor lists) and prefix-sums the per-CTA tie counts so the canonical tie rule is global.
//   bid-list replay  (auction_bidlist_kernel, G CTAs) the bidding round from the survivor lists, without reading S
//            again: bids ((v - T_w) + eps, :76), ties at T_w taken lowest job index first up to the worker's quota,
//            retain hack (:86-87) and counter>1000 fallback (:88-89) per job, column max with first-argmax (:104),
//            cost / owner update (:118-123).
//   S-scanning fallback  (auction_pass_kernel, after a survivor-list overflow) the same bidding round from tiles of
//            all K workers x 128 (K<=128) or 64 jobs, bulk-copied into shared memory through a 3-deep ring.
// In the single-GPU driver the last CTA of the bidding kernel runs the resolve step (termination, frozen detection,
// next state).  With the jobs sharded over GPUs the same kernels run on every rank's shard, and the sums over ranks
// happen either inside the kernels over peer memory (rqk_auction_peer_round) or through NCCL between step functions.
//
// Exact fast-forward.  With N % K != 0 the reference cannot terminate before its counter>1000
// fallback and runs 1002 rounds (SURVEY.md F4).  But once a round's fresh bids all land on jobs
// the bidder already owns and every owned job keeps a bid ("frozen"), nothing but `cost` can ever
// change again: owned values are S (constant), all other values are S-cost with cost
// non-decreasing, so every worker's top-N/K set stays its owned set.  Hence
//   * frozen at counter c < 100: each remaining retain round adds exactly eps to the cost of every
//     owned job -> apply (99-c) fp16 adds per job and jump to counter = 100;
//   * frozen at 100 <= counter <= 1000 without termination: the run ends at counter 1001 with the
//     owners unchanged and the never-bid jobs dumped on worker 0 -> emit that, rounds = 1002.
// tests/ check this against the oracle, which simulates every one of the 1002 rounds.
#include "common.cuh"

namespace rqk {

constexpr int AUC_W = 256;         // histogram bins per worker
constexpr int AUC_HALF = AUC_W / 2;
constexpr int AUC_NBUF = 3;        // tile buffers of the BID kernel
constexpr int AUC_BPL = AUC_W / 32; // bins per lane in the resolve kernel
constexpr int AUC_NW = 16;         // warps per CTA
constexpr int AUC_THREADS = AUC_NW * 32;
constexpr int AUC_BASE_CTAS = 296; // 2 per SM
constexpr int AUC_MAX_CTAS = 1024; // tie-prefix kernel limit
constexpr int AUC_MAX_JOBS_PER_CTA = 65024;   // 16-bit per-CTA counters
constexpr int AUC_MIN_TILES_PER_CTA = 2;
constexpr int AUC_COLD_SHIFT = 8;  // 256 bins x 256 keys cover all 65536 fp16 keys
constexpr int AUC_MIN_KEY = 0x0400; // key of the most negative finite half: fine windows never reach -inf
constexpr int AUC_SUB = 4096;      // jobs whose cost / owner are staged in shared memory at a time
constexpr int AUC_QCAP = 256;      // per-warp survivor queue of the HIST kernel (one row segment; = AUC_SEG_CAP)
constexpr int AUC_SAMPLE_MAX = 8192; // window-sampling jobs per worker (all ranks together)
constexpr int AUC_SEG_CAP = 256;   // survivor-list entries per (sub-range, worker); ~60 expected
constexpr int AUC_KH = 128;        // workers per histogram half of the HIST kernel
constexpr int AUC_SAMPLE_THREADS = 512; // threads of a window-sampling CTA (2 CTAs per SM: K = 256 in one wave)

enum { MODE_HIST = 0, MODE_BID = 1, MODE_DONE = 2 };

// Programmatic dependent launch (the single-GPU driver launches its round kernels with
// cudaLaunchAttributeProgrammaticStreamSerialization): a kernel lets its successor be scheduled as soon as all of
// its own CTAs have started, and the successor runs whatever does not depend on earlier kernels (shared-memory
// set-up, parameter loads) before it waits for them to complete.  Both instructions are no-ops in a normal launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

struct AuctionState {
    int mode;
    int counter;        // the reference's `counter`
    int rounds;         // topk evaluations the reference would have executed
    int done;
    int ff_pending;     // eps-adds owed to every owned job's cost (retain fast-forward)
    int frozen_exit;    // 1 if finished through the frozen shortcut
    int passes;         // passes over S actually executed
    int cold_passes;    // of which histogram-only
    int window_misses;
    unsigned int eps_bits;
    unsigned int smax_bits, smin_bits;
    int need_sample;    // windows are cold: estimate them from a sample before the next pass
    int error;
    int use_list;       // the coming BID pass reads the survivor lists of the HIST pass instead of S
    int force_scan;     // debugging / tests: never use the lists
    int list_passes;    // BID passes served from the lists
    int sink[4];        // statistics: worker-rounds whose threshold sank by < 64, < 128, < 250, >= 250 keys
    int branch[4];      // statistics (directly after sink[]): worker-passes that ended in a refine inside a coarse bin /
                        // in the gap of a split window / in a slide after a miss / in a coarse restart
    int pad_[4];
};

struct AuctionPtrs {
    AuctionState* st;
    __half* cost;
    short* owner;
    __half* sown;             // [ld] S[owner[j]][j]: the owner's own value of job j (valid where owner >= 0)
    // "reduce block": contiguous int32 [K*W + 2K + 2]; the only per-pass data ranks must sum when the
    // jobs are sharded over GPUs (hist_g | above_g | gap_g | n_with | n_viol)
    unsigned int* hist_g;     // [K][W]
    unsigned int* above_g;    // [K] values above the window
    unsigned int* gap_g;      // [K] values between the two halves of a split window
    unsigned int* n_with;     // [1] jobs with a bidder in the last BID pass
    unsigned int* n_viol;     // [1] frozen-condition violations in the last BID pass
    unsigned int* tie_total;  // [K] local number of values equal to the threshold (for the cross-rank prefix)
    int* win_base;            // [K] key of bin 0
    int* win_hbase;           // [K] fine windows may be split in two runs of one-key bins: [base, base+nlo) and
    int* win_nlo;             // [K] [hbase, hbase+128-nlo); contiguous = (base, base+64, 64)
    int* win_shift;           // [K] log2 keys per bin
    int* tkey;                // [K] resolved threshold key, -1 = unresolved
    int* take;                // [K] ties at the threshold that still get a bid
    int* tprev;               // [K] threshold of the previous round (-1 = none): thresholds only sink within an auction
    int* miss_run;            // [K] consecutive window slides
    unsigned int* tieprefix;  // [G][K]
    unsigned short* hist_cta; // [G][K][W] per-CTA histograms (16-bit: a CTA owns < 65536 jobs)
    // survivor lists of the last HIST pass: every (worker, job) whose value reached the worker's window, i.e. a
    // superset of the coming round's bidders.  One segment per (4096-job sub-range, worker), unordered.
    unsigned int* seg_list;   // [G*spc][K][AUC_SEG_CAP]  (job - sub-range start) << 16 | value key
    unsigned int* seg_cnt;    // [G*spc][K]  entries the HIST pass wanted to write (> AUC_SEG_CAP: overflow)
    int* list_ok;             // [1] cleared by a HIST CTA whose segment overflowed
    unsigned int* rank_off;   // [K] ties at the threshold held by lower ranks (peer-memory sharding; else 0)
    unsigned int* ticket;     // [1] CTAs finished in the running pass kernel (fused resolve)
    int* res_pass;            // [K] value of AuctionState.passes when the worker's threshold was resolved
    // single-GPU driver: the HIST pass only dumps per CTA; auction_merge_resolve_kernel (one CTA per worker) sums them
    unsigned int* above_cta;  // [G][K]
    unsigned int* gap_cta;    // [G][K]
    int* unres_g;             // [4] workers the running merge-resolve pass left unresolved / window misses among them /
                              //     arrival ticket of auction_peer_publish_kernel
};

static inline int auction_tile_cols(int K) { return K <= 128 ? 128 : 64; }

static inline int auction_grid(long long N, int K) {
    long long tiles = ceil_div<long long>(N, auction_tile_cols(K));
    long long g = ceil_div<long long>(tiles, AUC_MIN_TILES_PER_CTA);
    // RQK_AUCTION_GRID: fewer, longer CTA ranges (tests: several 4096-job sub-ranges per CTA at small N)
    const char* e = getenv("RQK_AUCTION_GRID");
    const int cap = (e && atoi(e) >= 1 && atoi(e) <= AUC_BASE_CTAS) ? atoi(e) : AUC_BASE_CTAS;
    if (g > cap) g = cap;
    long long g16 = ceil_div<long long>(N, AUC_MAX_JOBS_PER_CTA);
    if (g < g16) g = g16;
    if (g < 1) g = 1;
    return (int)g;
}

// sub-ranges per CTA (upper bound): CTA b owns tiles [T*b/G, T*(b+1)/G)
static inline int auction_spc(long long N, int K) {
    const int J = auction_tile_cols(K), G = auction_grid(N, K);
    const long long tiles = ceil_div<long long>(N, J);
    const long long len = ceil_div<long long>(tiles, G) * J;
    return (int)ceil_div<long long>(len, AUC_SUB);
}

static inline size_t auction_ws_layout(long long N, long long ld, int K, AuctionPtrs* p, char* base,
                                       size_t* reduce_off = nullptr, size_t* tie_total_off = nullptr) {
    int G = auction_grid(N, K);
    size_t off = 0;
    auto take_ = [&](size_t bytes) { size_t o = off; off += align256(bytes); return o; };
    size_t o_st = take_(sizeof(AuctionState));
    size_t o_cost = take_((size_t)ld * 2);
    size_t o_own = take_((size_t)ld * 2);
    size_t o_sown = take_((size_t)ld * 2);
    size_t o_hist = take_(((size_t)K * AUC_W + 2 * K + 2) * 4);
    size_t o_tt = take_((size_t)K * 4);
    size_t o_wb = take_((size_t)K * 4);
    size_t o_whb = take_((size_t)K * 4);
    size_t o_wnl = take_((size_t)K * 4);
    size_t o_ws = take_((size_t)K * 4);
    size_t o_tk = take_((size_t)K * 4);
    size_t o_take = take_((size_t)K * 4);
    size_t o_tprev = take_((size_t)K * 4);
    size_t o_mr = take_((size_t)K * 4);
    size_t o_tp = take_((size_t)G * K * 4);
    size_t o_hc = take_((size_t)G * K * AUC_W * 2);
    const size_t nseg = (size_t)G * auction_spc(N, K);
    size_t o_sl = take_(nseg * K * AUC_SEG_CAP * 4);
    size_t o_sc = take_(nseg * K * 4);
    size_t o_lo = take_(4);
    size_t o_ro = take_((size_t)K * 4);
    size_t o_tk2 = take_(4);
    size_t o_rp = take_((size_t)K * 4);
    size_t o_ac = take_((size_t)G * K * 4);
    size_t o_gc = take_((size_t)G * K * 4);
    size_t o_ug = take_(16);
    if (reduce_off) *reduce_off = o_hist;
    if (tie_total_off) *tie_total_off = o_tt;
    if (p) {
        p->st = (AuctionState*)(base + o_st);
        p->cost = (__half*)(base + o_cost);
        p->owner = (short*)(base + o_own);
        p->sown = (__half*)(base + o_sown);
        p->hist_g = (unsigned int*)(base + o_hist);
        p->above_g = p->hist_g + (size_t)K * AUC_W;
        p->gap_g = p->above_g + K;
        p->n_with = p->gap_g + K;
        p->n_viol = p->n_with + 1;
        p->tie_total = (unsigned int*)(base + o_tt);
        p->win_base = (int*)(base + o_wb);
        p->win_hbase = (int*)(base + o_whb);
        p->win_nlo = (int*)(base + o_wnl);
        p->win_shift = (int*)(base + o_ws);
        p->tkey = (int*)(base + o_tk);
        p->take = (int*)(base + o_take);
        p->tprev = (int*)(base + o_tprev);
        p->miss_run = (int*)(base + o_mr);
        p->tieprefix = (unsigned int*)(base + o_tp);
        p->hist_cta = (unsigned short*)(base + o_hc);
        p->seg_list = (unsigned int*)(base + o_sl);
        p->seg_cnt = (unsigned int*)(base + o_sc);
        p->list_ok = (int*)(base + o_lo);
        p->rank_off = (unsigned int*)(base + o_ro);
        p->ticket = (unsigned int*)(base + o_tk2);
        p->res_pass = (int*)(base + o_rp);
        p->above_cta = (unsigned int*)(base + o_ac);
        p->gap_cta = (unsigned int*)(base + o_gc);
        p->unres_g = (int*)(base + o_ug);
    }
    return off;
}

// ------------------------------------------------------------------------------------------
// init: cost = 0, owner = -1, eps from the fp16 extrema (:33-34), cold windows
// ------------------------------------------------------------------------------------------
__global__ void auction_init_kernel(AuctionPtrs p, long long ld, int K, const unsigned int* minmax_keys, int force_scan) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long j = i; j < ld; j += stride) {
        p.cost[j] = __ushort_as_half(0);
        p.owner[j] = -1;
    }
    for (long long j = i; j < (long long)K * AUC_W + 2 * K + 2; j += stride) p.hist_g[j] = 0;
    for (long long j = i; j < K; j += stride) {
        p.win_base[j] = 0;
        p.win_hbase[j] = AUC_HALF;
        p.win_nlo[j] = AUC_HALF;
        p.win_shift[j] = AUC_COLD_SHIFT;
        p.tkey[j] = -1;
        p.take[j] = 0;
        p.tprev[j] = -1;
        p.miss_run[j] = 0;
        p.rank_off[j] = 0;
        p.res_pass[j] = -1;
    }
    if (i == 0) {
        AuctionState s;
        memset(&s, 0, sizeof(s));
        s.mode = MODE_HIST;
        s.need_sample = 1;
        s.force_scan = force_scan;
        *p.list_ok = 1;
        *p.ticket = 0;
        p.unres_g[0] = 0;
        p.unres_g[1] = 0;
        p.unres_g[2] = 0;
        unsigned int smax = key2h(minmax_keys[0]), smin = key2h(minmax_keys[1]);
        // eps = (max - min) / 50 in fp16 (two roundings), floored at half(1e-4)  (:33-34)
        __half range = __hsub(bits2h(smax), bits2h(smin));
        __half e = __float2half_rn(__half2float(range) / 50.0f);
        __half fl = __float2half_rn(1e-4f);
        if (__half2float(fl) > __half2float(e)) e = fl;
        s.eps_bits = h2bits(e);
        s.smax_bits = smax;
        s.smin_bits = smin;
        *p.st = s;
    }
}


// ------------------------------------------------------------------------------------------
// Jobs sharded over GPUs, exchange through peer memory (NVLink / NVSwitch P2P) instead of NCCL.
// Every rank owns one "exchange block" in symmetric memory (allocated and mapped into every peer by
// the host: torch symmetric memory); kernels read the other ranks' blocks directly and synchronise
// with monotonically increasing sequence flags, so that the collective a round needs (sum of the
// threshold histograms, rank-major tie counts, the two bid counters, the window samples) is part of
// the round's kernels instead of a library call between two kernels.
//   flags  int32 [3 kinds][8 ranks]   flags[kind][r] = last sequence number rank r has published
//   tail   int32 [2 parities][2]      jobs with a bidder, frozen-state violations of the local BID round
//   hist   int32 [2 parities][RB]     local histogram rows [K][256], above [K], gap [K] (RB >= K*256 + 2K)
//   sample uint16[2 parities][K][cnt] local window samples
// Blocks are double-buffered by the parity of the sequence number: a rank can only be two exchanges
// ahead of a peer that still reads its block, never in the same parity.
// ------------------------------------------------------------------------------------------
constexpr int PEER_MAX = 8;
constexpr int PEER_FLAGS_BYTES = 256;
constexpr int PEER_TAIL_BYTES = 256;
struct PeerCtx {
    unsigned char* buf[PEER_MAX];
    int world, rank;
};
__host__ __device__ inline size_t peer_rb_words(int K) { return ((size_t)K * AUC_W + 2 * K + 2 + 63) / 64 * 64; }
__host__ __device__ inline size_t peer_sample_off(int K) { return PEER_FLAGS_BYTES + PEER_TAIL_BYTES + 2 * peer_rb_words(K) * 4; }
__host__ __device__ inline size_t peer_bytes(int K) { return peer_sample_off(K) + 2 * (size_t)K * AUC_SAMPLE_MAX * 2; }
__device__ __forceinline__ int* peer_flags(const PeerCtx& c, int r) { return reinterpret_cast<int*>(c.buf[r]); }
__device__ __forceinline__ int* peer_tail(const PeerCtx& c, int r, int par) {
    return reinterpret_cast<int*>(c.buf[r] + PEER_FLAGS_BYTES) + 2 * par;
}
__device__ __forceinline__ unsigned int* peer_hist(const PeerCtx& c, int r, int K, int par) {
    return reinterpret_cast<unsigned int*>(c.buf[r] + PEER_FLAGS_BYTES + PEER_TAIL_BYTES) + (size_t)par * peer_rb_words(K);
}
__device__ __forceinline__ const unsigned short* peer_sample(const PeerCtx& c, int r, int K, int par) {
    return reinterpret_cast<const unsigned short*>(c.buf[r] + peer_sample_off(K)) + (size_t)par * K * AUC_SAMPLE_MAX;
}
// All threads of the CTA call this after their stores to the local exchange block.  Returns false on a timeout
// (a peer that never arrives: 4 s), which the caller turns into an error state instead of a hang.
// `signal` = false: wait only (another CTA of the grid publishes this rank's arrival).
__device__ bool peer_barrier(const PeerCtx& c, int kind, int seq, bool signal) {
    __shared__ int s_ok;
    __threadfence_system();
    __syncthreads();
    const int t = threadIdx.x;
    if (t == 0) s_ok = 1;
    __syncthreads();
    if (t < c.world && t != c.rank) {
        if (signal) {
            int* dst = peer_flags(c, t) + kind * PEER_MAX + c.rank;
            asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(dst), "r"(seq) : "memory");
        }
        const int* src = peer_flags(c, c.rank) + kind * PEER_MAX + t;
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        int v;
        do {
            asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
            if (v >= seq) break;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 4000000000ull) { s_ok = 0; break; }
            __nanosleep(200);
        } while (true);
    }
    __syncthreads();
    return s_ok != 0;
}

// ------------------------------------------------------------------------------------------
// resolve: merged histograms -> thresholds / next windows / state machine.  One CTA.
// ------------------------------------------------------------------------------------------
// Outcome of a bidding round from its two global counters: all jobs have a bidder (:113-114), or the state is
// frozen (file header) - at counter 100..1000 the run is decided, below 99 the retain phase is fast-forwarded.
struct BidOutcome { bool finished, jump; };
__device__ __forceinline__ BidOutcome bid_outcome(int counter, unsigned long long n_with, unsigned long long n_viol, long long N) {
    BidOutcome o{false, false};
    if (n_with == (unsigned long long)N) {
        o.finished = true;
    } else if (n_viol == 0 && counter >= 1) {
        if (counter >= 100 && counter <= 1000) o.finished = true;
        else if (counter < 99) o.jump = true;
    }
    return o;
}

// Threshold of ONE worker from its merged window histogram (one warp; lane l holds bins [8l, 8l+8) in h, lsum = their
// sum).  Either resolves the worker (tkey / take / res_pass), or re-aims its window (refine inside a coarse bin, the
// gap of a split window, a slide after a miss) and counts it in *unresolved (and *miss).
__device__ __forceinline__ void resolve_one_worker(const AuctionPtrs& p, int w, const unsigned int (&h)[AUC_BPL],
                                                   unsigned int lsum, unsigned long long ab, unsigned long long gap,
                                                   int base, int shift, int hbase, int nlo, long long need, long long jpw,
                                                   int passes, int* sink, int* unresolved, int* miss) {
    const int lane = threadIdx.x & 31;
    // suffix sums over lanes (bins above mine)
    unsigned int suf = lsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned int o = __shfl_down_sync(0xffffffffu, suf, d);
        if (lane + d < 32) suf += o;
    }
                // strictly above my bins (the gap of a split window sits between bins nlo-1 and nlo)
    unsigned long long cum_excl = ab + (suf - lsum) + ((AUC_BPL * lane + AUC_BPL - 1) < nlo ? gap : 0ull);
    const unsigned long long total = ab + __shfl_sync(0xffffffffu, suf, 0) + gap;
    unsigned int hsum = 0;                                    // my bins of the upper run
#pragma unroll
    for (int i = 0; i < AUC_BPL; ++i) hsum += (AUC_BPL * lane + i >= nlo) ? h[i] : 0u;
#pragma unroll
    for (int d = 16; d; d >>= 1) hsum += __shfl_xor_sync(0xffffffffu, hsum, d);
    const unsigned long long c_hi = ab + hsum;               // everything >= hbase
    const bool in_gap = gap > 0 && c_hi < (unsigned long long)need && c_hi + gap >= (unsigned long long)need;
    int found_bin = -1;
    unsigned long long g_above = 0;
    if (!in_gap && ab < (unsigned long long)need && total >= (unsigned long long)need) {
        unsigned long long c = cum_excl;
#pragma unroll
        for (int i = AUC_BPL - 1; i >= 0; --i) {
            if (i != AUC_BPL - 1 && AUC_BPL * lane + i == nlo - 1) c += gap;   // stepping over the gap inside my bins
            if (found_bin < 0 && c < (unsigned long long)need && c + h[i] >= (unsigned long long)need) {
                found_bin = lane * AUC_BPL + i;
                g_above = c;
            }
            c += h[i];
        }
    }
    unsigned int who = __ballot_sync(0xffffffffu, found_bin >= 0);
    if (who) {
        int src = __ffs(who) - 1;
        found_bin = __shfl_sync(0xffffffffu, found_bin, src);
        g_above = __shfl_sync(0xffffffffu, g_above, src);
        if (lane == 0) {
            p.miss_run[w] = 0;
            if (shift == 0) {
                const int tk_new = found_bin >= nlo ? hbase + found_bin - nlo : base + found_bin;
                const int tp = p.tprev[w];
                if (tp >= 0) {
                    const int d = tp - tk_new;
                    atomicAdd(&sink[d < 64 ? 0 : d < 128 ? 1 : d < 250 ? 2 : 3], 1);
                }
                p.tkey[w] = found_bin >= nlo ? hbase + found_bin - nlo : base + found_bin;
                p.take[w] = (int)(jpw - (long long)g_above);
                p.res_pass[w] = passes;
            } else {   // refine inside the bin that holds the threshold
                atomicAdd(&sink[4], 1);
                int nshift = shift >= 8 ? shift - 8 : 0;
                const int nb2 = base + (found_bin << shift);
                p.win_base[w] = nb2;
                p.win_hbase[w] = nb2 + AUC_HALF;
                p.win_nlo[w] = AUC_HALF;
                p.win_shift[w] = nshift;
                p.tkey[w] = -1;
                atomicAdd(unresolved, 1);
            }
        }
    } else if (lane == 0 && in_gap) {
        // the threshold lies between the two halves of a split window: histogram just that range
        atomicAdd(&sink[5], 1);
        int nb2 = base + nlo, span = hbase - nb2, nshift = 0;
        while ((span >> nshift) > AUC_W) ++nshift;
        p.win_base[w] = nb2;
        p.win_hbase[w] = nb2 + AUC_HALF;
        p.win_nlo[w] = AUC_HALF;
        p.win_shift[w] = nshift;
        p.tkey[w] = -1;
        atomicAdd(unresolved, 1);
        atomicAdd(miss, 1);
    } else if (lane == 0) {
        // the window missed the threshold: slide one window up / down, restart coarse if that
        // keeps failing (or if the window was a refinement, which cannot miss by construction)
        const int run = p.miss_run[w];
        const bool is_above = ab >= (unsigned long long)need;
        int nb = is_above ? (shift == 0 ? hbase + (AUC_W - nlo) : base + (AUC_W << shift)) : base - (AUC_W << shift);
        atomicAdd(&sink[(shift != 0 || run >= 2 || nb < AUC_MIN_KEY || nb > 65536 - AUC_W) ? 7 : 6], 1);
        if (shift != 0 || run >= 2 || nb < AUC_MIN_KEY || nb > 65536 - AUC_W) {
            p.win_base[w] = 0;
            p.win_hbase[w] = AUC_HALF;
            p.win_nlo[w] = AUC_HALF;
            p.win_shift[w] = AUC_COLD_SHIFT;
            p.miss_run[w] = 0;
        } else {
            p.win_base[w] = nb;
            p.win_hbase[w] = nb + AUC_HALF;
            p.win_nlo[w] = AUC_HALF;
            p.miss_run[w] = run + 1;
        }
        p.tkey[w] = -1;
        atomicAdd(unresolved, 1);
        if (shift == 0) atomicAdd(miss, 1);
    }
}

// `expect`: -1, or the mode whose pass must have just run (MODE_HIST / MODE_BID) for the call to act.
__device__ __noinline__ void auction_resolve_body(AuctionPtrs p, long long N, int K, long long jpw, int expect) {
    __shared__ int s_unresolved, s_miss;
    __shared__ AuctionState s;
    __shared__ unsigned long long s_nwith_g, s_nviol_g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NT = blockDim.x, NWARPS = NT >> 5;
    if (tid == 0) { s = *p.st; s_unresolved = 0; s_miss = 0; s_nwith_g = *p.n_with; s_nviol_g = *p.n_viol; }
    __syncthreads();
    if (s.mode == MODE_DONE || (expect >= 0 && s.mode != expect)) return;
    const bool was_bid = (s.mode == MODE_BID);

    // ---- 1. outcome of the bidding round that just ran ----
    bool finished = false, jump = false;
    if (was_bid) {
        const BidOutcome o = bid_outcome(s.counter, s_nwith_g, s_nviol_g, N);
        finished = o.finished;
        jump = o.jump;
    }
    if (finished) {
        __syncthreads();
        if (tid == 0) {
            bool normal = (s_nwith_g == (unsigned long long)N);
            s.rounds = normal ? s.counter + 1 : 1002;
            s.frozen_exit = normal ? 0 : 1;
            s.mode = MODE_DONE;
            s.done = 1;
            s.passes += 1;
            if (s.use_list) s.list_passes += 1;
            *p.st = s;
        }
        return;
    }

    // ---- 2. thresholds from the histogram (of the values the next selection sees) ----
    // A BID pass leaves no histogram: the next pass is a HIST pass over the new state with windows
    // placed by the sample kernel.
    const long long need = jpw + 1;
    if (was_bid) {
        for (int w = tid; w < K; w += NT) {
            p.tprev[w] = p.tkey[w];
            p.win_base[w] = 0;
            p.win_hbase[w] = AUC_HALF;
            p.win_nlo[w] = AUC_HALF;
            p.win_shift[w] = AUC_COLD_SHIFT;
            p.tkey[w] = -1;
            p.miss_run[w] = 0;
        }
        if (tid == 0) s_unresolved = 1;
    } else if (!jump) {
        // the next worker's bins are loaded while the current worker is resolved (one CTA: latency is all there is)
        unsigned int hn[AUC_BPL];
#pragma unroll
        for (int i = 0; i < AUC_BPL; ++i) hn[i] = (warp < K) ? __ldcg(p.hist_g + warp * AUC_W + lane * AUC_BPL + i) : 0u;
        for (int w = warp; w < K; w += NWARPS) {
            const bool settled = p.tkey[w] >= 0;      // resolved by an earlier pass of this round: not streamed again
            const int base = p.win_base[w], shift = p.win_shift[w];
            const int hbase = p.win_hbase[w], nlo = (shift == 0) ? p.win_nlo[w] : 0;
            const unsigned long long gap = (shift == 0) ? p.gap_g[w] : 0ull;
            unsigned int h[AUC_BPL];
            unsigned int lsum = 0;
#pragma unroll
            for (int i = 0; i < AUC_BPL; ++i) { h[i] = hn[i]; lsum += h[i]; }
            if (w + NWARPS < K) {
#pragma unroll
                for (int i = 0; i < AUC_BPL; ++i) hn[i] = __ldcg(p.hist_g + (w + NWARPS) * AUC_W + lane * AUC_BPL + i);
            }
            if (settled) continue;
            resolve_one_worker(p, w, h, lsum, p.above_g[w], gap, base, shift, hbase, nlo, need, jpw, s.passes, s.sink,
                               &s_unresolved, &s_miss);
        }
    }
    __syncthreads();
    // ---- 3. zero the reduce block for the next pass ----
    // (after a BID pass only its counters: the histogram part was zeroed by the HIST resolve before it, or never
    // written at all when the HIST passes dump per CTA for auction_merge_resolve_kernel)
    for (int i = tid + (was_bid ? K * AUC_W : 0); i < K * AUC_W + 2 * K + 2; i += NT) p.hist_g[i] = 0;
    __syncthreads();
    if (tid == 0) {
        s.passes += 1;
        if (!was_bid) s.cold_passes += 1;
        s.window_misses += s_miss;
        if (was_bid) s.counter += 1;                                     // :125
        s.ff_pending = 0;
        s.need_sample = was_bid ? 1 : 0;
        if (was_bid && s.use_list) s.list_passes += 1;
        // survivor lists of this round's HIST passes (a worker's segments come from the pass that resolved it):
        // complete unless a segment overflowed in any of them
        if (!was_bid) s.use_list = (*p.list_ok != 0 && !s.force_scan) ? 1 : 0;
        else *p.list_ok = 1;
        if (jump) {
            // frozen at counter c (already incremented to c+1): rounds c+1..99 add eps each
            s.ff_pending = 100 - s.counter;
            s.counter = 100;
            s.mode = MODE_HIST;
        } else {
            s.mode = (s_unresolved == 0) ? MODE_BID : MODE_HIST;
        }
        *p.st = s;
    }
}


__global__ void __launch_bounds__(1024, 1)
auction_resolve_kernel(AuctionPtrs p, long long N, int K, long long jpw, int expect) {
    auction_resolve_body(p, N, K, jpw, expect);
}

// Single-GPU runs fold the resolve step into the pass kernel itself: the CTA that finishes last (a ticket
// counter) sees every other CTA's histogram merges / bid counts and runs the resolve body, which saves a
// kernel boundary per pass.  Sharded runs cannot (the merged histograms must be summed over ranks first).
__device__ __forceinline__ bool auction_last_cta(unsigned int* ticket) {
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1) ? 1 : 0;
        if (s_last) *ticket = 0;
    }
    __syncthreads();
    if (s_last) __threadfence();
    return s_last != 0;
}

// ------------------------------------------------------------------------------------------
// the streaming pass
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ __half2 u2h2(unsigned u) { return *reinterpret_cast<__half2*>(&u); }
__device__ __forceinline__ unsigned h22u(__half2 h) { return *reinterpret_cast<unsigned*>(&h); }

struct PassSmem {
    __half* tile0;             // [NBUF][K][J]
    unsigned int* hist;        // [K][W/2] two 16-bit counters per word
    unsigned int* above;       // [K]
    unsigned int* tie_seen;    // [K]
    int* r_take;               // [K]
    int* r_base;               // [K]
    int* r_hbase;              // [K]
    int* r_nlo;                // [K]
    unsigned int* gap;         // [K]
    unsigned int* r_T2;        // [K] threshold as a duplicated half2
    unsigned int* r_lo2;       // [K] sweep filter as a duplicated half2 (window low value; T for coarse rows)
    unsigned char* r_shift;    // [K]
    unsigned char* row_flag;   // [K] an owner entry ties with the threshold in this tile
    unsigned int* colmax;      // [J] (bid << 16) | (0xffff - worker)
    unsigned short* colcost;   // [J]
    short* colown;             // [J]
    unsigned char* colviol;    // [J]
};

__device__ __forceinline__ void hist_add(unsigned int* hist, int w, int bin, unsigned int n = 1) {
    atomicAdd(&hist[(w * AUC_W + bin) >> 1], n << ((bin & 1) * 16));
}

// Window geometry.  shift > 0: 128 contiguous bins of 2^shift keys from `base`.  shift == 0: one-key bins,
// bins 0..nlo-1 = [base, base+nlo), bins nlo..127 = [hbase, hbase+128-nlo), hbase >= base+nlo; keys in
// between are counted in `gap`, keys above in `above`, keys below `base` are ignored.  Worker w's histogram is row
// `hrow` of sm.hist.
__device__ __forceinline__ void window_count(const PassSmem& sm, int w, int hrow, int key) {
    const int base = sm.r_base[w];
    const int shift = sm.r_shift[w];
    if (key < base) return;
    if (shift == 0) {
        const int hb = sm.r_hbase[w], nlo = sm.r_nlo[w];
        if (key >= hb) {
            if (key - hb >= AUC_W - nlo) atomicAdd(&sm.above[w], 1u);
            else hist_add(sm.hist, hrow, nlo + key - hb);
        } else if (key >= base + nlo) {
            atomicAdd(&sm.gap[w], 1u);
        } else {
            hist_add(sm.hist, hrow, key - base);
        }
    } else {
        const int bin = (key - base) >> shift;
        if (bin >= AUC_W) atomicAdd(&sm.above[w], 1u);
        else hist_add(sm.hist, hrow, bin);
    }
}

// ---- mbarrier + bulk-copy (UBLKCP) tile loads: one 16-byte-aligned row per instruction ----
__device__ __forceinline__ unsigned s_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mb_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(s_addr(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(s_addr(dst)), "l"(src), "r"(bytes), "r"(s_addr(bar)) : "memory");
}

// The BID pass.  Per tile (all K workers x J jobs in shared memory, bulk-copied, double buffered): the sweep
// filters S - cost against each worker's threshold T_w (one HSUB2 + one HSET2 per two elements); the ~1 %
// survivors, kept as register bitmasks, become bids; column maximum; cost / owner update.
template <int J>
__global__ void __launch_bounds__(AUC_THREADS, (J == 128 ? 2 : 1))
auction_pass_kernel(const __half* __restrict__ S, long long ld, long long N, int K, long long jpw, AuctionPtrs p,
                    long long n_global, int fused) {
    constexpr int CPL = J / 32;           // columns per lane
    constexpr int NH2 = CPL / 2;          // half2 words per lane
    constexpr int MAXR = 256 / AUC_NW * (J == 128 ? 1 : 2) / 2;   // rows per warp: 8 (K<=128) / 16 (K<=256)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_launch_dependents();
    pdl_wait();
    const AuctionState st = *p.st;
    if (st.mode != MODE_BID || st.use_list) return;    // HIST passes run in auction_hist_kernel, list rounds in auction_bidlist_kernel
    const bool do_bid = true;
    const int ff = 0;
    const int counter = st.counter;
    const __half eps = bits2h(st.eps_bits);
    const unsigned int eps_bits = st.eps_bits;
    const bool retain = do_bid && counter >= 1 && counter < 100;   // :86 (index is set from round 1 on)
    const bool fallback = do_bid && counter > 1000;                // :88

    // ---- shared memory carve-up ----
    PassSmem sm;
    {
        unsigned char* q = smem_raw;
        sm.tile0 = (__half*)q;               q += (size_t)AUC_NBUF * K * J * 2;
        sm.tie_seen = (unsigned int*)q;      q += (size_t)K * 4;
        sm.r_take = (int*)q;                 q += (size_t)K * 4;
        sm.r_T2 = (unsigned int*)q;          q += (size_t)K * 4;
        sm.r_lo2 = (unsigned int*)q;         q += (size_t)K * 4;
        sm.colmax = (unsigned int*)q;        q += (size_t)J * 4;
        sm.colcost = (unsigned short*)q;     q += (size_t)J * 2;
        sm.colown = (short*)q;               q += (size_t)J * 2;
        sm.r_shift = (unsigned char*)q;      q += (size_t)K;
        sm.row_flag = (unsigned char*)q;     q += (size_t)K;
        sm.colviol = (unsigned char*)q;      q += (size_t)J;
    }
    __shared__ unsigned int s_nwith, s_nviol;
    __shared__ __align__(8) unsigned long long tile_bar[AUC_NBUF];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int lt = (1u << lane) - 1u;
    const int G = gridDim.x, b = blockIdx.x;
    const long long tiles_total = (N + J - 1) / J;
    const long long t_begin = tiles_total * b / G, t_end = tiles_total * (b + 1) / G;

    for (int i = tid; i < K; i += AUC_THREADS) {
        sm.tie_seen[i] = p.tieprefix[(size_t)b * K + i];
        const int tk = p.tkey[i];
        const unsigned int Tb = key2h((unsigned)(tk < 0 ? 0 : tk));
        sm.r_T2[i] = Tb | (Tb << 16);
        sm.r_take[i] = p.take[i];
        sm.r_lo2[i] = Tb | (Tb << 16);                     // the sweep finds bidders: v >= T_w
        sm.row_flag[i] = 0;
    }
    for (int i = tid; i < J; i += AUC_THREADS) { sm.colmax[i] = 0; sm.colviol[i] = 0; }
    if (tid == 0) {
        s_nwith = 0; s_nviol = 0;
        for (int i = 0; i < AUC_NBUF; ++i) mb_init(&tile_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // per-row sweep filter in registers (the rows of a warp are w = warp + 16 i)
    unsigned int f2r[MAXR];
#pragma unroll
    for (int i = 0; i < MAXR; ++i) {
        const int w = warp + AUC_NW * i;
        f2r[i] = (w < K) ? sm.r_lo2[w] : 0x7c007c00u;
    }

    auto issue_tile = [&](long long t, int buf) {
        if (tid == 0) mb_expect_tx(&tile_bar[buf], (unsigned)(K * J * 2));
        if (tid < K)
            bulk_g2s(sm.tile0 + (size_t)buf * K * J + (size_t)tid * J, S + (size_t)tid * ld + t * J, J * 2, &tile_bar[buf]);
    };
    // AUC_NBUF-deep ring: tiles t+1 .. t+NBUF-1 are in flight while tile t is processed
    for (int i = 0; i < AUC_NBUF - 1; ++i)
        if (t_begin + i < t_end) issue_tile(t_begin + i, i);

    for (long long t = t_begin; t < t_end; ++t) {
        const int it = (int)(t - t_begin);
        const int buf = it % AUC_NBUF;
        const __half* tile = sm.tile0 + (size_t)buf * K * J;
        const long long col0 = t * J;
        const int ncols = (int)((N - col0) < J ? (N - col0) : J);   // valid columns of this tile
        // ---- stage per-column state ----
        if (tid < J) {
            long long col = col0 + tid;
            unsigned short c = 0;
            short o = -1;
            if (tid < ncols) {
                __half ch = p.cost[col];
                o = p.owner[col];
                if (ff > 0 && o >= 0) {   // retain fast-forward: (99-c) rounds of cost += eps
                    for (int r = 0; r < ff; ++r) ch = __hadd(ch, eps);
                    p.cost[col] = ch;
                }
                c = __half_as_ushort(ch);
            }
            sm.colcost[tid] = c;
            sm.colown[tid] = o;
        }
        // prefetch into the buffer whose last readers finished before the barrier that closed the
        // previous iteration
        if (t + AUC_NBUF - 1 < t_end) issue_tile(t + AUC_NBUF - 1, (it + AUC_NBUF - 1) % AUC_NBUF);
        mb_wait(&tile_bar[buf], (unsigned)(it / AUC_NBUF) & 1u);
        __syncthreads();                                                     // S0: tile + column state visible

        __half2 c2[NH2];
#pragma unroll
        for (int h = 0; h < NH2; ++h) c2[h] = u2h2(reinterpret_cast<const unsigned*>(sm.colcost)[lane * NH2 + h]);

        unsigned int flagmask = 0;                                           // bit i: row warp+16i has an owner tie
        if (do_bid) {
            // ---------------- owner entries: one per job, handled by the job's column thread ----------------
            if (tid < ncols) {
                const int o = sm.colown[tid];
                unsigned int init = 0;
                if (o >= 0) {
                    const __half s = tile[(size_t)o * J + tid];              // owner's value is S itself (:123)
                    const __half T = bits2h(sm.r_T2[o] & 0xffffu);
                    unsigned int bid = 0;
                    if (__hgt(s, T)) bid = h2bits(__hadd(__hsub(s, T), eps));
                    else if (__heq(s, T)) sm.row_flag[o] = 1;                // tie: the row's warp ranks it exactly
                    if (retain) bid = eps_bits;                              // :87
                    if (bid) init = (bid << 16) | (0xffffu - (unsigned)o);
                } else if (fallback) {
                    init = (eps_bits << 16) | 0xffffu;                       // :89 worker 0 takes never-bid jobs
                }
                if (init) atomicMax(&sm.colmax[tid], init);
            }
            __syncthreads();                                                 // S1: row flags visible
            const int wf = warp + AUC_NW * lane;
            flagmask = __ballot_sync(0xffffffffu, lane < MAXR && wf < K && sm.row_flag[wf] != 0);
        }

        // ---------------- the sweep: half2 filter; survivors recorded as register bitmasks ----------------
        // acc[h] bit i      : column 2h   of row warp+16i survives
        // acc[h] bit 16 + i : column 2h+1 of row warp+16i survives        (rej[h]: same layout, rejected ties)
        unsigned int acc[NH2], rej[NH2];
#pragma unroll
        for (int h = 0; h < NH2; ++h) { acc[h] = 0; rej[h] = 0; }
        const unsigned* tile_u = reinterpret_cast<const unsigned*>(tile) + lane * NH2;
#pragma unroll
        for (int i = 0; i < MAXR; ++i) {
            const int w = warp + AUC_NW * i;
            if (w >= K) break;
            const __half2 f2 = u2h2(f2r[i]);
            const unsigned* row = tile_u + (size_t)w * (J / 2);
            const bool flagged = (flagmask >> i) & 1u;
            const unsigned int rowbits = (1u << i) | (1u << (16 + i));
            __half2 v2[NH2];
            if (!flagged) {
#pragma unroll
                for (int h = 0; h < NH2; ++h) {
                    v2[h] = __hsub2(u2h2(row[h]), c2[h]);                    // ownership ignored: the owner's S is only larger
                    acc[h] |= __hge2_mask(v2[h], f2) & rowbits;
                }
            } else {
#pragma unroll
                for (int h = 0; h < NH2; ++h) {                              // exact values incl. owner entries
                    unsigned int cr = h22u(c2[h]);
                    if (sm.colown[lane * CPL + 2 * h] == w) cr &= 0xffff0000u;
                    if (sm.colown[lane * CPL + 2 * h + 1] == w) cr &= 0x0000ffffu;
                    v2[h] = __hsub2(u2h2(row[h]), u2h2(cr));
                    acc[h] |= __hge2_mask(v2[h], f2) & rowbits;
                }
            }
            if (do_bid) {                                                    // f2 == T_w in a BID pass
                unsigned int anye = 0, em[NH2];
#pragma unroll
                for (int h = 0; h < NH2; ++h) { em[h] = __heq2_mask(v2[h], f2); anye |= em[h]; }
                const unsigned int seen0 = sm.tie_seen[w];
                const long long quota0 = sm.r_take[w];
                if ((long long)seen0 >= quota0) {
                    // the worker's quota of ties was used up by lower job indices: every tie here is rejected
                    // (owner entries and padding columns are skipped in stage A anyway)
#pragma unroll
                    for (int h = 0; h < NH2; ++h) rej[h] |= em[h] & rowbits;
                } else if (__any_sync(0xffffffffu, anye != 0)) {
                    // canonical tie rule: lowest job index first, globally (tieprefix + tiles so far).
                    // In unflagged rows owner entries cannot tie (the column thread would have flagged the row).
                    bool eq[CPL];
                    unsigned int before = 0, total = 0, mine = 0;
#pragma unroll
                    for (int e = 0; e < CPL; ++e) {
                        const int cidx = lane * CPL + e;
                        eq[e] = ((em[e >> 1] >> ((e & 1) * 16)) & 1u) != 0 && cidx < ncols &&
                                (flagged || sm.colown[cidx] != w);
                        unsigned int mm = __ballot_sync(0xffffffffu, eq[e]);
                        before += __popc(mm & lt);
                        total += __popc(mm);
                    }
                    const unsigned int seen = sm.tie_seen[w];
                    const long long quota = sm.r_take[w];
#pragma unroll
                    for (int e = 0; e < CPL; ++e) {
                        if (eq[e]) {
                            if (!((long long)(seen + before + mine) < quota)) rej[e >> 1] |= 1u << ((e & 1) * 16 + i);
                            mine++;
                        }
                    }
                    __syncwarp();
                    if (lane == 0) sm.tie_seen[w] = seen + total;
                    __syncwarp();
                }
            }
        }

        if (do_bid) {
            // ---------------- stage A: survivors -> bids ----------------
#pragma unroll
            for (int h = 0; h < NH2; ++h) {
                unsigned int a = acc[h];
                while (a) {
                    const int bpos = __ffs(a) - 1;
                    a &= a - 1;
                    const int i = bpos & 15;
                    const int w = warp + AUC_NW * i, col = lane * CPL + 2 * h + (bpos >> 4);
                    if (col >= ncols) continue;
                    const int o = sm.colown[col];
                    const bool own = (o == w);
                    const bool flagged_row = (flagmask >> i) & 1u;
                    if (own && !flagged_row) continue;                       // the column thread did it
                    const __half sv = tile[(size_t)w * J + col];
                    const __half v = own ? sv : __hsub(sv, __ushort_as_half(sm.colcost[col]));
                    const __half T = bits2h(sm.r_T2[w] & 0xffffu);
                    const bool rejected = (rej[h] >> bpos) & 1u;
                    if (!(__hgt(v, T) || (__heq(v, T) && !rejected))) continue;
                    if (fallback && w == 0 && o < 0) continue;               // :89 overrides worker 0's own bid
                    unsigned int bid = h2bits(__hadd(__hsub(v, T), eps));    // :76, two roundings
                    if (retain && own) bid = eps_bits;                       // :87
                    if (!own) sm.colviol[col] = 1;                           // fresh bid on a job the bidder does not own
                    atomicMax(&sm.colmax[col], (bid << 16) | (0xffffu - (unsigned)w));   // :104
                }
            }
            __syncthreads();                                                 // S3: all bids in colmax

            // ---------------- highest bid per job, cost/owner update (:104, :118-123) ----------------
            if (tid < J) {
                const unsigned int pk = sm.colmax[tid];
                bool has = false, vv = false;
                if (tid < ncols) {
                    const long long col = col0 + tid;
                    const short old_owner = sm.colown[tid];
                    vv = sm.colviol[tid] != 0;
                    if (pk) {
                        has = true;
                        const short wnr = (short)(0xffffu - (pk & 0xffffu));
                        p.cost[col] = __hadd(__ushort_as_half(sm.colcost[tid]), bits2h(pk >> 16));
                        p.owner[col] = wnr;
                        p.sown[col] = tile[(size_t)wnr * J + tid];
                    } else {
                        p.owner[col] = -1;
                        if (old_owner >= 0) vv = true;                       // an owned job lost its bidder
                    }
                }
                sm.colmax[tid] = 0;
                sm.colviol[tid] = 0;
                unsigned int mh = __ballot_sync(0xffffffffu, has);
                unsigned int mv = __ballot_sync(0xffffffffu, vv);
                if (lane == 0) {
                    if (mh) atomicAdd(&s_nwith, __popc(mh));
                    if (mv) atomicAdd(&s_nviol, __popc(mv));
                }
            }
            for (int i = tid; i < K; i += AUC_THREADS) sm.row_flag[i] = 0;
        }
        __syncthreads();                                                     // S4: tile buffer + column state free
    }

    if (tid == 0) {
        if (s_nwith) atomicAdd(p.n_with, s_nwith);
        if (s_nviol) atomicAdd(p.n_viol, s_nviol);
    }
    if (fused && auction_last_cta(p.ticket)) auction_resolve_body(p, n_global, K, n_global / K, MODE_BID);
}

// ------------------------------------------------------------------------------------------
// HIST pass as a tile-free streaming kernel.  A HIST pass needs no column maximum, so nothing forces
// the K rows of a job through shared memory together: every warp streams row segments straight from
// global memory with 16-byte loads, four in flight per lane, which hides HBM latency far better than a
// double-buffered tile.  Per 8 jobs of a row: 1 LDG.128, 1 LDS.128 (costs), 4 HSUB2, 4 HSET2, 4 LOP3.
// Survivors are recorded as register bitmasks and histogrammed afterwards.
// CTA b owns exactly the job range CTA b of the tiled BID kernel owns (the per-CTA dumps feed its tie prefix).
// ------------------------------------------------------------------------------------------
constexpr int HS_SUB = AUC_SUB;   // jobs staged (cost, owner) per sub-range
__device__ __forceinline__ uint4 ldg_stream128(const void* ptr) {
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(ptr));
    return r;
}

// Shared-memory layout with compile-time offsets: with run-time offsets the compiler re-derives the array bases inside
// the hot loops (64 registers per thread leave no room to keep them).  The histogram holds one half of the workers
// (AUC_KH rows, 64 KB, so that two CTAs fit on an SM); the per-worker arrays hold all K <= 256.
struct HistSmem {
    static constexpr int KMAX = 256;
    static constexpr int HIST = 0;                                    // [AUC_KH][W/2] two 16-bit counters per word
    static constexpr int COST = HIST + AUC_KH * AUC_W * 2;            // [HS_SUB] fp16
    static constexpr int OWN = COST + HS_SUB * 2;                     // [HS_SUB] int16
    static constexpr int HQ = OWN + HS_SUB * 2;                       // [NW][QCAP] survivor queue
    static constexpr int ABOVE = HQ + AUC_NW * AUC_QCAP * 2;          // [KMAX] u32 ...
    static constexpr int GAP = ABOVE + KMAX * 4;
    static constexpr int RBASE = GAP + KMAX * 4;
    static constexpr int RHBASE = RBASE + KMAX * 4;
    static constexpr int RNLO = RHBASE + KMAX * 4;
    static constexpr int RLO2 = RNLO + KMAX * 4;
    static constexpr int SEGCNT = RLO2 + KMAX * 4;
    static constexpr int ACT = SEGCNT + KMAX * 4;                     // [KMAX] u16 unresolved workers, ascending
    static constexpr int RSHIFT = ACT + KMAX * 2;                     // [KMAX] u8 (0xff: resolved by an earlier pass)
    static constexpr int TOTAL = (RSHIFT + KMAX + 15) / 16 * 16;
};

// K > AUC_KH: the CTA runs its job range once per half of the workers, [0, 128) then [128, K), with the histogram
// cleared in between.  That keeps the K = 128 register and shared-memory budget (2 CTAs per SM) for every K; the
// cost / owner staging is repeated per half (6 bytes per job against 256 bytes of S per job and half).
__global__ void __launch_bounds__(AUC_THREADS, 2)
auction_hist_kernel(const __half* __restrict__ S, long long ld, long long N, int K, int J, int spc, AuctionPtrs p,
                    long long n_global, int fused) {
    using L = HistSmem;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_launch_dependents();
    // nothing below depends on earlier kernels until pdl_wait(): the histogram is cleared while they finish
    auto clear_hist = [&] {
        for (int i = threadIdx.x; i < AUC_KH * AUC_W * 2 / 16; i += AUC_THREADS)
            reinterpret_cast<uint4*>(smem_raw + L::HIST)[i] = make_uint4(0u, 0u, 0u, 0u);
    };
    clear_hist();
    pdl_wait();
    const AuctionState st = *p.st;
    if (st.mode != MODE_HIST) return;
    const int ff = st.ff_pending;
    const __half eps = bits2h(st.eps_bits);

    PassSmem sm;
    sm.hist = reinterpret_cast<unsigned int*>(smem_raw + L::HIST);
    sm.above = reinterpret_cast<unsigned int*>(smem_raw + L::ABOVE);
    sm.gap = reinterpret_cast<unsigned int*>(smem_raw + L::GAP);
    sm.r_base = reinterpret_cast<int*>(smem_raw + L::RBASE);
    sm.r_hbase = reinterpret_cast<int*>(smem_raw + L::RHBASE);
    sm.r_nlo = reinterpret_cast<int*>(smem_raw + L::RNLO);
    sm.r_lo2 = reinterpret_cast<unsigned int*>(smem_raw + L::RLO2);
    sm.r_shift = smem_raw + L::RSHIFT;
    unsigned short* const cost_s = reinterpret_cast<unsigned short*>(smem_raw + L::COST);
    short* const own_s = reinterpret_cast<short*>(smem_raw + L::OWN);
    unsigned int* const seg_cnt_s = reinterpret_cast<unsigned int*>(smem_raw + L::SEGCNT);
    unsigned short* const act = reinterpret_cast<unsigned short*>(smem_raw + L::ACT);
    __shared__ int s_act_off[3], s_any_cold[2], s_wcnt[AUC_NW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int lt = (1u << lane) - 1u;
    unsigned short* const wq = reinterpret_cast<unsigned short*>(smem_raw + L::HQ) + warp * AUC_QCAP;
    const int G = gridDim.x, b = blockIdx.x;
    const long long tiles_total = (N + J - 1) / J;
    const long long c_begin = (tiles_total * b / G) * J;
    long long c_end = (tiles_total * (b + 1) / G) * J;
    if (c_end > N) c_end = N;

    // Rows (workers) of this pass.  A worker whose threshold an earlier pass of the SAME round resolved keeps what
    // that pass produced (threshold, survivor lists, per-CTA dump) and is skipped: after a window miss only the
    // workers that missed are streamed again, spread over the warps (act[] = the unresolved workers, ascending; those
    // of half h are act[s_act_off[h] .. s_act_off[h + 1])).
    if (tid < 2) s_any_cold[tid] = 0;
    for (int i = tid; i < K; i += AUC_THREADS) {
        sm.above[i] = 0;
        sm.gap[i] = 0;
        const int base = p.win_base[i];
        sm.r_base[i] = base;
        sm.r_hbase[i] = p.win_hbase[i];
        sm.r_nlo[i] = p.win_nlo[i];
        sm.r_shift[i] = (p.tkey[i] >= 0) ? (unsigned char)0xff : (unsigned char)p.win_shift[i];   // 0xff: resolved
        const unsigned int lob = base > 0 ? key2h((unsigned)base) : 0x7c00u;   // cold rows: direct path below
        sm.r_lo2[i] = lob | (lob << 16);
    }
    __syncthreads();
    {   // ordered compaction (K <= 256 < AUC_THREADS: one round)
        const bool a = tid < K && sm.r_shift[tid] != 0xff;
        const unsigned int m = __ballot_sync(0xffffffffu, a);
        if (lane == 0) s_wcnt[warp] = __popc(m);
        __syncthreads();
        int off = 0;
        for (int q = 0; q < warp; ++q) off += s_wcnt[q];
        if (a) {
            act[off + __popc(m & lt)] = (unsigned short)tid;
            if (sm.r_base[tid] <= 0) s_any_cold[tid / AUC_KH] = 1;
        }
        if (tid == 0) {
            int t = 0;
            for (int q = 0; q < AUC_NW; ++q) {
                if (q == AUC_KH / 32) s_act_off[1] = t;
                t += s_wcnt[q];
            }
            s_act_off[0] = 0;
            s_act_off[2] = t;
        }
        __syncthreads();
    }

    int ffh = ff;                                            // the retain fast-forward goes to the first half streamed
    for (int h0 = 0; h0 < K; h0 += AUC_KH) {
        const unsigned short* const acth = act + s_act_off[h0 / AUC_KH];
        const int nact = s_act_off[h0 / AUC_KH + 1] - s_act_off[h0 / AUC_KH];
        if (nact == 0) continue;                                 // every worker of the half was resolved by an earlier pass
        const int any_cold = s_any_cold[h0 / AUC_KH];            // cold rows take the unpipelined path
        if (h0 > 0) {
            __syncthreads();                                     // the previous half's histogram has been published
            clear_hist();
            __syncthreads();
        }

        int seg = b * spc;
        for (long long sub = c_begin; sub < c_end; sub += HS_SUB, ++seg) {
            const int sublen = (int)((c_end - sub) < HS_SUB ? (c_end - sub) : HS_SUB);
            unsigned int* seg_lists = p.seg_list + (size_t)seg * K * AUC_SEG_CAP;
            if (tid < K) seg_cnt_s[tid] = 0;
            // ---- stage costs / owners of the sub-range (retain fast-forward applied here, once) ----
            unsigned short so_r[HS_SUB / AUC_THREADS];   // the owner's own value of my jobs (kept by the BID kernels)
#pragma unroll
            for (int it = 0; it < HS_SUB / AUC_THREADS; ++it) {
                const int i = tid + it * AUC_THREADS;
                unsigned short c = 0;
                short o = -1;
                so_r[it] = 0;
                if (i < sublen) {
                    __half ch = p.cost[sub + i];
                    o = p.owner[sub + i];
                    so_r[it] = __half_as_ushort(p.sown[sub + i]);
                    if (ffh > 0 && o >= 0) {
                        for (int r = 0; r < ffh; ++r) ch = __hadd(ch, eps);
                        p.cost[sub + i] = ch;
                    }
                    c = __half_as_ushort(ch);
                }
                cost_s[i] = c;
                own_s[i] = o;
            }
            __syncthreads();
            // ---- owner entries (value = S): one per job, counted in the owner's half ----
#pragma unroll
            for (int it = 0; it < HS_SUB / AUC_THREADS; ++it) {
                const int i = tid + it * AUC_THREADS;
                const int o = (i < sublen) ? own_s[i] : -1;
                if (o >= h0 && o < h0 + AUC_KH && sm.r_base[o] > 0 && sm.r_shift[o] != 0xff) {
                    const int key = (int)h2key((unsigned)so_r[it]);
                    window_count(sm, o, o - h0, key);
                    if (key >= sm.r_base[o]) {
                        const unsigned int slot = atomicAdd(&seg_cnt_s[o], 1u);
                        if (slot < AUC_SEG_CAP) seg_lists[(size_t)o * AUC_SEG_CAP + slot] = ((unsigned)i << 16) | (unsigned)key;
                    }
                }
            }
            // One survivor per lane: exact value -> key -> survivor list + window histogram.  Called with all 32 lanes.
            auto emit = [&](int w, const __half* srow, bool live, int cc, int wbase, int whb, int wnlo, int wshift) {
                live = live && own_s[cc] != w;                                   // owner entry: counted above
                int key = 0;
                if (live) key = (int)h2key(h2bits(__hsub(srow[cc], __ushort_as_half(cost_s[cc]))));
                const unsigned int m = __ballot_sync(0xffffffffu, live);
                if (m) {
                    unsigned int slot0 = 0;
                    if (lane == 0) slot0 = atomicAdd(&seg_cnt_s[w], (unsigned)__popc(m));
                    slot0 = __shfl_sync(0xffffffffu, slot0, 0);
                    const unsigned int slot = slot0 + __popc(m & lt);
                    if (live && slot < AUC_SEG_CAP) seg_lists[(size_t)w * AUC_SEG_CAP + slot] = ((unsigned)cc << 16) | (unsigned)key;
                }
                if (live) {
                    int bin;
                    if (wshift == 0) bin = key >= whb ? (key - whb >= AUC_W - wnlo ? AUC_W : wnlo + key - whb)
                                                      : (key >= wbase + wnlo ? -1 : key - wbase);
                    else { bin = (key - wbase) >> wshift; bin = bin > AUC_W ? AUC_W : bin; }
                    if (bin >= AUC_W) atomicAdd(&sm.above[w], 1u);
                    else if (bin < 0) atomicAdd(&sm.gap[w], 1u);
                    else hist_add(sm.hist, w - h0, bin);
                }
            };
            if (!any_cold) {
                // Fast path (every active row has a fine window).  Software-pipelined: the next step's four 16-byte loads
                // are in flight while this step is filtered, across row boundaries too.  Survivors are not
                // handled by the lane that found them (a divergent loop, ~5 of 32 lanes busy) but pushed as
                // job offsets into a per-warp queue and handled 32 at a time when the queue fills / the row ends.
                int qn = 0;
                const int nfull = sublen >> 10, nsteps = (sublen + 1023) >> 10;
                auto load_step = [&](int w, int st, uint4 (&sv)[4]) {
                    const uint4* rp = reinterpret_cast<const uint4*>(S + (size_t)w * ld + sub) + (st << 7) + lane;
                    if (st < nfull) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) sv[q] = ldg_stream128(rp + q * 32);
                    } else {   // tail step; columns >= N of S hold -inf and their staged cost is 0: they never survive
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            sv[q] = make_uint4(0xfc00fc00u, 0xfc00fc00u, 0xfc00fc00u, 0xfc00fc00u);
                            if ((st << 10) + q * 256 + lane * 8 < sublen) sv[q] = ldg_stream128(rp + q * 32);
                        }
                    }
                };
                auto flush = [&](int w) {
                    const __half* srow = S + (size_t)w * ld + sub;
                    const int wbase = sm.r_base[w], whb = sm.r_hbase[w], wnlo = sm.r_nlo[w], wshift = sm.r_shift[w];
                    unsigned int* lw = seg_lists + (size_t)w * AUC_SEG_CAP;
                    __syncwarp();
                    for (int i0 = 0; i0 < qn; i0 += 32) {
                        const int i = i0 + lane;
                        bool live = i < qn;
                        const int cc = live ? (int)wq[i] : 0;
                        live = live && own_s[cc] != w;                               // owner entry: counted above
                        int key = 0;
                        if (live) key = (int)h2key(h2bits(__hsub(srow[cc], __ushort_as_half(cost_s[cc]))));
                        const unsigned int m = __ballot_sync(0xffffffffu, live);
                        if (m) {
                            unsigned int slot0 = 0;
                            if (lane == 0) slot0 = atomicAdd(&seg_cnt_s[w], (unsigned)__popc(m));
                            slot0 = __shfl_sync(0xffffffffu, slot0, 0);
                            const unsigned int slot = slot0 + __popc(m & lt);
                            if (live && slot < AUC_SEG_CAP) lw[slot] = ((unsigned)cc << 16) | (unsigned)key;
                        }
                        if (live) {
                            if (wshift == 0) {
                                if (key >= whb) {
                                    if (key - whb >= AUC_W - wnlo) atomicAdd(&sm.above[w], 1u);
                                    else hist_add(sm.hist, w - h0, wnlo + key - whb);
                                } else if (key >= wbase + wnlo) {
                                    atomicAdd(&sm.gap[w], 1u);
                                } else {
                                    hist_add(sm.hist, w - h0, key - wbase);
                                }
                            } else {
                                const int bin = (key - wbase) >> wshift;
                                if (bin >= AUC_W) atomicAdd(&sm.above[w], 1u);
                                else hist_add(sm.hist, w - h0, bin);
                            }
                        }
                    }
                    qn = 0;
                    __syncwarp();
                };
                uint4 bufA[4], bufB[4];
                int a = warp, st = 0;                                  // position in the active-row list, step in the row
                int w = a < nact ? (int)acth[a] : 0;
                if (a < nact) load_step(w, 0, bufA);
                auto body = [&](uint4 (&cur)[4], uint4 (&nxt)[4]) {
                    int an = a, wn = w, sn = st + 1;
                    if (sn == nsteps) { an = a + AUC_NW; sn = 0; wn = an < nact ? (int)acth[an] : 0; }
                    if (an < nact) load_step(wn, sn, nxt);
                    // ---- filter: v = S - cost against the window's low edge ----
                    const __half2 f2 = u2h2(sm.r_lo2[w]);
                    const uint4* cp = reinterpret_cast<const uint4*>(cost_s) + (st << 7) + lane;
                    unsigned int acc = 0;   // low half bit 4q+h: job 2h of load q survives; high half: job 2h+1
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint4 cv = cp[q * 32];
                        const unsigned int sw[4] = {cur[q].x, cur[q].y, cur[q].z, cur[q].w};
                        const unsigned int cw[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            const __half2 v2 = __hsub2(u2h2(sw[h]), u2h2(cw[h]));
                            acc |= __hge2_mask(v2, f2) & ((1u << (4 * q + h)) | (1u << (16 + 4 * q + h)));
                        }
                    }
                    // ---- push the survivors' job offsets ----
                    const int mine = __popc(acc);
                    int incl = mine;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const int o = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += o;
                    }
                    const int total = __shfl_sync(0xffffffffu, incl, 31);
                    if (total) {
                        const int cbase = (st << 10) + lane * 8;
                        if (qn + total > AUC_QCAP) flush(w);
                        if (total <= AUC_QCAP) {
                            int pos = qn + incl - mine;
                            while (acc) {
                                const int bpos = __ffs(acc) - 1;
                                acc &= acc - 1;
                                const int pq = bpos & 15;
                                wq[pos++] = (unsigned short)(cbase + ((pq >> 2) << 8) + ((pq & 3) << 1) + (bpos >> 4));
                            }
                            qn += total;
                        } else {
                            // more than a queue's worth in one step (only with very wide windows): 4 per lane per round
                            while (__any_sync(0xffffffffu, acc != 0)) {
                                const int pc = __popc(acc);
                                const int take = pc < 4 ? pc : 4;
                                int in2 = take;
#pragma unroll
                                for (int d = 1; d < 32; d <<= 1) {
                                    const int o = __shfl_up_sync(0xffffffffu, in2, d);
                                    if (lane >= d) in2 += o;
                                }
                                int pos = in2 - take;
                                for (int r = 0; r < take; ++r) {
                                    const int bpos = __ffs(acc) - 1;
                                    acc &= acc - 1;
                                    const int pq = bpos & 15;
                                    wq[pos++] = (unsigned short)(cbase + ((pq >> 2) << 8) + ((pq & 3) << 1) + (bpos >> 4));
                                }
                                qn = __shfl_sync(0xffffffffu, in2, 31);
                                flush(w);
                            }
                        }
                    }
                    if (sn == 0 && qn) flush(w);                                     // the queue is per row
                    a = an;
                    w = wn;
                    st = sn;
                };
                while (a < nact) {
                    body(bufA, bufB);
#pragma unroll
                    for (int q = 0; q < 4; ++q) bufA[q] = bufB[q];
                }
            } else {
                for (int a = warp; a < nact; a += AUC_NW) {
                    const int w = acth[a];
                    const __half* srow = S + (size_t)w * ld + sub;
                    const int wbase = sm.r_base[w];
                    if (wbase > 0) {
                        const int whb = sm.r_hbase[w], wnlo = sm.r_nlo[w], wshift = sm.r_shift[w];
                        const __half lo = bits2h(key2h((unsigned)wbase));
                        for (int c0 = 0; c0 < sublen; c0 += 32) {
                            const int cc = c0 + lane;
                            bool live = cc < sublen;
                            if (live) live = __hge(__hsub(srow[cc], __ushort_as_half(cost_s[cc])), lo);
                            if (__any_sync(0xffffffffu, live)) emit(w, srow, live, live ? cc : 0, wbase, whb, wnlo, wshift);
                        }
                    } else {
                        // cold row (all 65536 keys in 256 coarse bins): exact values, every element
                        const int shift = sm.r_shift[w];
                        for (int c0 = 0; c0 < sublen; c0 += 32) {
                            const int cc = c0 + lane;
                            const bool valid = cc < sublen;
                            __half v = __ushort_as_half(0xfc00);
                            if (valid) {
                                const __half sx = srow[cc];
                                v = (own_s[cc] == w) ? sx : __hsub(sx, __ushort_as_half(cost_s[cc]));
                            }
                            const int bin = (int)h2key(h2bits(v)) >> shift;
                            const bool hb = valid && bin < AUC_W;
                            const bool ab = valid && bin >= AUC_W;
                            unsigned int na = __popc(__ballot_sync(0xffffffffu, ab));
                            if (lane == 0 && na) atomicAdd(&sm.above[w], na);
                            unsigned int actm = __ballot_sync(0xffffffffu, hb);
                            if (actm) {
                                int lead = __ffs(actm) - 1;
                                int lbin = __shfl_sync(0xffffffffu, bin, lead);
                                unsigned int same = __ballot_sync(0xffffffffu, hb && bin == lbin);
                                if (same == actm) {
                                    if (lane == lead) hist_add(sm.hist, w - h0, lbin, __popc(actm));
                                } else if (hb) {
                                    hist_add(sm.hist, w - h0, bin);
                                }
                            }
                        }
                    }
                }
            }
            __syncthreads();
            if (tid >= h0 && tid < h0 + AUC_KH && tid < K && sm.r_shift[tid] != 0xff) {
                const unsigned int c = seg_cnt_s[tid];
                p.seg_cnt[(size_t)seg * K + tid] = c;
                if (c > AUC_SEG_CAP) *p.list_ok = 0;
            }
        }

        // ---- publish the half's histogram rows (active rows only) ----
        // fused (single-GPU driver): plain stores into the per-CTA dump; auction_merge_resolve_kernel (one CTA per worker,
        // next in the chain) sums them over the CTAs, resolves the worker's threshold and takes the tie prefix - no global
        // atomics here, no serial resolve in a last CTA.  Step-by-step / sharded flows: the per-CTA dump (for the tie
        // prefix) and a merge of the non-empty bins into the reduce block.
        unsigned int* dump = reinterpret_cast<unsigned int*>(p.hist_cta + ((size_t)b * K + h0) * AUC_W);
        for (int a = tid >> 7; a < nact; a += AUC_THREADS >> 7) {                // AUC_W / 2 = 128 words per row
            const int i = ((int)acth[a] - h0) * (AUC_W / 2) + (tid & 127);
            const unsigned int h = sm.hist[i];
            dump[i] = h;
            if (!fused) {
                const int ig = h0 * (AUC_W / 2) + i;
                if (h & 0xffffu) atomicAdd(&p.hist_g[2 * ig], h & 0xffffu);
                if (h >> 16) atomicAdd(&p.hist_g[2 * ig + 1], h >> 16);
            }
        }
        ffh = 0;
    }

    const int nact_all = s_act_off[2];
    for (int a = tid; a < nact_all; a += AUC_THREADS) {
        const int i = act[a];
        if (fused) {
            p.above_cta[(size_t)b * K + i] = sm.above[i];
            p.gap_cta[(size_t)b * K + i] = sm.gap[i];
        } else {
            if (sm.above[i]) atomicAdd(&p.above_g[i], sm.above[i]);
            if (sm.gap[i]) atomicAdd(&p.gap_g[i], sm.gap[i]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// BID pass from the survivor lists.  The HIST pass that resolved the thresholds already computed
// S - cost for every entry and kept those at or above each worker's window (a superset of the
// bidders, ~1.5 % of the matrix), so the bidding round does not have to read S again: CTA b replays
// its own segments (L2-resident, written microseconds ago), then updates cost / owner of its jobs.
// Same arithmetic as auction_pass_kernel; ties at the threshold are ranked by job index only in the
// one segment per worker that straddles the worker's quota.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(AUC_THREADS, 2)
auction_bidlist_kernel(const __half* __restrict__ S, long long ld, long long N, int K, int J, int spc, AuctionPtrs p,
                       long long n_global, int fused) {
    pdl_launch_dependents();
    pdl_wait();
    const AuctionState st = *p.st;
    if (st.mode != MODE_BID || !st.use_list) return;
    constexpr int NCH = AUC_SEG_CAP / 32;
    __shared__ __align__(16) unsigned int colmax[AUC_SUB];
    __shared__ __align__(16) short own_s[AUC_SUB];
    __shared__ __align__(16) unsigned char colviol[AUC_SUB];
    __shared__ unsigned int tie_seen[256];
    __shared__ int r_take[256], r_tk[256];
    __shared__ unsigned int s_nwith, s_nviol;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int counter = st.counter;
    const __half eps = bits2h(st.eps_bits);
    const unsigned int eps_bits = st.eps_bits;
    const bool retain = counter >= 1 && counter < 100;      // :86
    const bool fallback = counter > 1000;                    // :88
    const int G = gridDim.x, b = blockIdx.x;
    const long long tiles_total = (N + J - 1) / J;
    const long long c_begin = (tiles_total * b / G) * J;
    long long c_end = (tiles_total * (b + 1) / G) * J;
    if (c_end > N) c_end = N;

    for (int i = tid; i < K; i += AUC_THREADS) {
        tie_seen[i] = p.tieprefix[(size_t)b * K + i];
        r_tk[i] = p.tkey[i];
        r_take[i] = p.take[i];
    }
    if (tid == 0) { s_nwith = 0; s_nviol = 0; }

    int seg = b * spc;
    for (long long sub = c_begin; sub < c_end; sub += AUC_SUB, ++seg) {
        const int sublen = (int)((c_end - sub) < AUC_SUB ? (c_end - sub) : AUC_SUB);
        // ---- stage cost / owner; bids that do not depend on S (retain hack :87, fallback :89) ----
        // A thread owns 8 consecutive jobs (AUC_SUB = 8 * AUC_THREADS): one 16-byte access per array.  cost / owner /
        // sown hold ld >= N entries (columns >= N: cost 0, owner -1, never touched), so whole groups are in bounds.
        static_assert(AUC_SUB == 8 * AUC_THREADS, "one 8-job group per thread");
        const int j0 = tid * 8;
        const bool grp = j0 < sublen;                            // sublen is a multiple of 8 except at the matrix end
        uint4 c8 = make_uint4(0u, 0u, 0u, 0u), o8 = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        if (grp) {
            c8 = *reinterpret_cast<const uint4*>(p.cost + sub + j0);
            o8 = *reinterpret_cast<const uint4*>(p.owner + sub + j0);
        }
        {
            const unsigned int ow[4] = {o8.x, o8.y, o8.z, o8.w};
            unsigned int init[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int o = (int)(short)((ow[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
                unsigned int v = 0;
                if (j0 + e < sublen) {
                    if (o >= 0) { if (retain) v = (eps_bits << 16) | (0xffffu - (unsigned)o); }
                    else if (fallback) v = (eps_bits << 16) | 0xffffu;
                }
                init[e] = v;
            }
            *reinterpret_cast<uint4*>(own_s + j0) = o8;
            *reinterpret_cast<uint4*>(colmax + j0) = make_uint4(init[0], init[1], init[2], init[3]);
            *reinterpret_cast<uint4*>(colmax + j0 + 4) = make_uint4(init[4], init[5], init[6], init[7]);
            *reinterpret_cast<uint2*>(colviol + j0) = make_uint2(0u, 0u);
        }
        __syncthreads();
        // ---- segments: a warp per worker ----
        // lengths of this warp's segments with one load; the first 64 entries of the next segment are fetched
        // while the current one is replayed (a segment holds ~60)
        const int nrows = (K - warp + AUC_NW - 1) / AUC_NW;
        unsigned int E_l = (lane < nrows) ? __ldcg(p.seg_cnt + (size_t)seg * K + warp + AUC_NW * lane) : 0u;
        if (E_l > AUC_SEG_CAP) E_l = AUC_SEG_CAP;            // cannot happen when use_list is set
        unsigned int pre0 = 0, pre1 = 0;
        {
            const unsigned int E0 = __shfl_sync(0xffffffffu, E_l, 0);
            const unsigned int* L0 = p.seg_list + ((size_t)seg * K + warp) * AUC_SEG_CAP;
            if ((unsigned)lane < E0) pre0 = __ldcg(L0 + lane);
            if ((unsigned)lane + 32 < E0) pre1 = __ldcg(L0 + 32 + lane);
        }
        for (int r = 0; r < nrows; ++r) {
            const int w = warp + AUC_NW * r;
            const unsigned int E = __shfl_sync(0xffffffffu, E_l, r);
            const unsigned int* L = p.seg_list + ((size_t)seg * K + w) * AUC_SEG_CAP;
            const int tk = r_tk[w];
            const __half T = bits2h(key2h((unsigned)tk));
            unsigned int ent[NCH], tmask[NCH];
            unsigned int n_ties = 0;
            ent[0] = pre0;
            ent[1] = pre1;
#pragma unroll
            for (int c = 2; c < NCH; ++c) {
                ent[c] = 0u;                                   // key 0 is below every threshold: never a bidder
                if ((unsigned)(c * 32) < E) {                  // warp-uniform: a segment holds ~60 entries, rarely > 64
                    const unsigned int idx = c * 32 + lane;
                    if (idx < E) ent[c] = __ldcg(L + idx);
                }
            }
            pre0 = 0; pre1 = 0;
            if (r + 1 < nrows) {
                const unsigned int En = __shfl_sync(0xffffffffu, E_l, r + 1);
                const unsigned int* Ln = L + (size_t)AUC_NW * AUC_SEG_CAP;
                if ((unsigned)lane < En) pre0 = __ldcg(Ln + lane);
                if ((unsigned)lane + 32 < En) pre1 = __ldcg(Ln + 32 + lane);
            }
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                tmask[c] = 0u;
                if ((unsigned)(c * 32) < E) {
                    const unsigned int idx = c * 32 + lane;
                    tmask[c] = __ballot_sync(0xffffffffu, idx < E && (int)(ent[c] & 0xffffu) == tk);
                    n_ties += __popc(tmask[c]);
                }
            }
            const unsigned int seen0 = tie_seen[w];
            const long long quota = r_take[w];
            const bool all_rej = (long long)seen0 >= quota;
            const bool all_acc = (long long)seen0 + n_ties <= quota;
            unsigned int rank[NCH];
#pragma unroll
            for (int c = 0; c < NCH; ++c) rank[c] = 0;
            if (n_ties && !all_rej && !all_acc) {
                // the segment straddles the quota: rank its ties by job index (lowest first)
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    unsigned int m = tmask[c];
                    while (m) {
                        const int src = __ffs(m) - 1;
                        m &= m - 1;
                        const unsigned int jsrc = __shfl_sync(0xffffffffu, ent[c], src) >> 16;
#pragma unroll
                        for (int c2 = 0; c2 < NCH; ++c2) rank[c2] += ((ent[c2] >> 16) > jsrc) ? 1u : 0u;
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                if ((unsigned)(c * 32) >= E) break;
                const unsigned int idx = c * 32 + lane;
                if (idx >= E) continue;
                const int key = (int)(ent[c] & 0xffffu);
                const int cc = (int)(ent[c] >> 16);
                bool bidder = key > tk;
                if (key == tk) bidder = all_acc || (!all_rej && (long long)seen0 + rank[c] < quota);
                if (!bidder) continue;
                const int o = own_s[cc];
                const bool own = (o == w);
                if (fallback && w == 0 && o < 0) continue;                       // :89 overrides worker 0's own bid
                const __half v = bits2h(key2h((unsigned)key));
                unsigned int bid = h2bits(__hadd(__hsub(v, T), eps));            // :76, two roundings
                if (retain && own) bid = eps_bits;                               // :87
                if (!own) colviol[cc] = 1;
                atomicMax(&colmax[cc], (bid << 16) | (0xffffu - (unsigned)w));   // :104
            }
            if (lane == 0) tie_seen[w] = seen0 + n_ties;
        }
        __syncthreads();
        // ---- highest bid per job, cost / owner update (:104, :118-123): the thread's 8 jobs again ----
        {
            const uint4 pa = *reinterpret_cast<const uint4*>(colmax + j0), pb = *reinterpret_cast<const uint4*>(colmax + j0 + 4);
            const uint2 vi = *reinterpret_cast<const uint2*>(colviol + j0);
            const unsigned int pk[8] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w};
            const unsigned int cw[4] = {c8.x, c8.y, c8.z, c8.w}, ow[4] = {o8.x, o8.y, o8.z, o8.w};
            unsigned short sv[8];
            unsigned int changed = 0;                                            // bit e: job e has a new owner
#pragma unroll
            for (int e = 0; e < 8; ++e) {                                        // new owners' own values: loads first
                sv[e] = 0;
                const int old_owner = (int)(short)((ow[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
                if (pk[e]) {
                    const int wnr = (int)(0xffffu - (pk[e] & 0xffffu));
                    if (wnr != old_owner) {
                        changed |= 1u << e;
                        sv[e] = __half_as_ushort(S[(size_t)wnr * ld + sub + j0 + e]);
                    }
                }
            }
            unsigned int nc[4], no[4];
            int n_has = 0, n_vv = 0;
            bool cost_dirty = false, own_dirty = false;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int sh = (e & 1) * 16;
                unsigned int c = (cw[e >> 1] >> sh) & 0xffffu, o = (ow[e >> 1] >> sh) & 0xffffu;
                const int old_owner = (int)(short)o;
                bool vv = ((e < 4 ? vi.x >> (8 * e) : vi.y >> (8 * (e - 4))) & 0xffu) != 0;
                if (pk[e]) {
                    ++n_has;
                    c = h2bits(__hadd(__ushort_as_half((unsigned short)c), bits2h(pk[e] >> 16)));
                    cost_dirty = true;
                    if ((changed >> e) & 1u) { o = 0xffffu - (pk[e] & 0xffffu); own_dirty = true; }
                } else if (old_owner >= 0) {                                     // an owned job lost its bidder
                    o = 0xffffu;
                    own_dirty = true;
                    vv = true;
                }
                n_vv += vv ? 1 : 0;
                if (e & 1) { nc[e >> 1] |= c << 16; no[e >> 1] |= o << 16; }
                else { nc[e >> 1] = c; no[e >> 1] = o; }
            }
            if (grp) {
                if (cost_dirty) *reinterpret_cast<uint4*>(p.cost + sub + j0) = make_uint4(nc[0], nc[1], nc[2], nc[3]);
                if (own_dirty) *reinterpret_cast<uint4*>(p.owner + sub + j0) = make_uint4(no[0], no[1], no[2], no[3]);
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if ((changed >> e) & 1u) p.sown[sub + j0 + e] = __ushort_as_half(sv[e]);
            }
            n_has = __reduce_add_sync(0xffffffffu, n_has);
            n_vv = __reduce_add_sync(0xffffffffu, n_vv);
            if (lane == 0) {
                if (n_has) atomicAdd(&s_nwith, (unsigned)n_has);
                if (n_vv) atomicAdd(&s_nviol, (unsigned)n_vv);
            }
        }
        __syncthreads();
    }
    if (tid == 0) {
        if (s_nwith) atomicAdd(p.n_with, s_nwith);
        if (s_nviol) atomicAdd(p.n_viol, s_nviol);
    }
    if (fused && auction_last_cta(p.ticket)) auction_resolve_body(p, n_global, K, n_global / K, MODE_BID);
}

static inline size_t auction_pass_smem(int K, int J) {
    return (size_t)AUC_NBUF * K * J * 2 + (size_t)K * 16 + (size_t)J * 4 +
           (size_t)J * 4 + (size_t)K * 2 + (size_t)J + 64;
}

// ------------------------------------------------------------------------------------------
// sampled windows: instead of a coarse 3-pass radix descent from cold, estimate each worker's
// threshold from a strided sample of its current values and open a fine window around the
// estimate (+-4.5 sigma of the order statistic).  A wrong guess only costs a slide / coarse restart.
// Grid = K CTAs x AUC_SAMPLE_THREADS threads, 8192 samples (4096 left twice as many window misses at K = 256 on clustered data).
// ------------------------------------------------------------------------------------------
constexpr int AUC_SAMPLE = AUC_SAMPLE_MAX;
// Warp-parallel descending scan of a 256-bin histogram: the highest bin b with base + sum(hist[b..255]) >= need,
// and base + sum(hist[b+1..255]).  Called by one full warp; results written by lane 0 (and returned to all lanes).
__device__ __forceinline__ void sample_select_bin(const unsigned int* hist, int base, int need, int* out_bin, int* out_above) {
    const int lane = threadIdx.x & 31;
    int h[8], lsum = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { h[i] = (int)hist[lane * 8 + i]; lsum += h[i]; }
    int suf = lsum;                                   // inclusive suffix sum over lanes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_down_sync(0xffffffffu, suf, d);
        if (lane + d < 32) suf += o;
    }
    int c = base + suf - lsum, bin = -1, above = 0;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        if (bin < 0 && c + h[i] >= need) { bin = lane * 8 + i; above = c; }
        c += h[i];
    }
    const unsigned int who = __ballot_sync(0xffffffffu, bin >= 0);
    int rb = 0, ra = base + __shfl_sync(0xffffffffu, suf, 0);   // not found: bin 0, everything above (as the serial scan)
    if (who) {
        const int src = 31 - __clz(who);
        rb = __shfl_sync(0xffffffffu, bin, src);
        ra = __shfl_sync(0xffffffffu, above, src);
    }
    if (lane == 0) { *out_bin = rb; *out_above = ra; }
    *out_bin = rb;
    *out_above = ra;
}



// Sharded jobs: every rank samples AUC_SAMPLE / world jobs of its shard (collect_out != null: write the keys
// and return), the host all-gathers them, and every rank places identical windows from the union
// (ext_keys != null: [ext_n / ext_cnt][K][ext_cnt] keys = every rank's gathered sample, N = global job count).
// peers.world > 0: the parts are the ranks' exchange blocks instead (parity of peer_seq), after a flag barrier.
__global__ void __launch_bounds__(AUC_SAMPLE_THREADS, 2)
auction_sample_kernel(const __half* __restrict__ S, long long ld, long long N, int K, long long jpw, AuctionPtrs p,
                      unsigned short* __restrict__ collect_out, int collect_n,
                      const unsigned short* __restrict__ ext_keys, int ext_n, int ext_cnt, PeerCtx peers, int peer_seq) {
    pdl_launch_dependents();
    pdl_wait();
    const AuctionState st = *p.st;
    if (st.mode != MODE_HIST || !st.need_sample) return;
    __shared__ unsigned short keys[AUC_SAMPLE];
    const int w = blockIdx.x, tid = threadIdx.x;
    if (peers.world > 0) {
        // every rank's samples are in its exchange block once the kernel before this one has completed (which the
        // wait above guarantees): CTA 0 publishes this rank's arrival, every CTA waits for all ranks
        if (!peer_barrier(peers, 0, peer_seq, blockIdx.x == 0)) {
            if (tid == 0) { p.st->error = 1; p.st->mode = MODE_DONE; p.st->done = 1; }
            return;
        }
    }
    long long ns = N < AUC_SAMPLE ? N : AUC_SAMPLE;
    if (collect_out) ns = collect_n < ns ? collect_n : ns;
    if (ext_keys || peers.world > 0) ns = ext_n;
    const __half eps = bits2h(st.eps_bits);
    {
        // a thread takes AUC_SAMPLE / AUC_SAMPLE_THREADS = 16 samples in two batches of 8: each batch issues all its
        // loads first (one latency, not 8) within the 64 registers of two CTAs per SM
        constexpr int PER = 8;
        static_assert(AUC_SAMPLE % (PER * AUC_SAMPLE_THREADS) == 0, "whole batches");
        const long long nchunks = (ns + 15) / 16, cstride = N / (nchunks > 0 ? nchunks : 1);
        for (int q0 = 0; q0 < AUC_SAMPLE / AUC_SAMPLE_THREADS; q0 += PER) {
            __half c_r[PER], s_r[PER];
            short o_r[PER];
            unsigned short k_r[PER];
#pragma unroll
            for (int q = 0; q < PER; ++q) {
                const int i = tid + (q0 + q) * AUC_SAMPLE_THREADS;
                k_r[q] = 0;                                                    // padding sorts last
                c_r[q] = s_r[q] = __ushort_as_half(0);
                o_r[q] = -1;
                if (ext_keys || peers.world > 0) {
                    if (i < ns) {
                        if (peers.world > 0)      // part r = rank r's sample block, read through its peer mapping
                            k_r[q] = __ldcv(peer_sample(peers, i / ext_cnt, K, peer_seq & 1) + (size_t)w * ext_cnt + (i % ext_cnt));
                        else
                            k_r[q] = ext_keys[((size_t)(i / ext_cnt) * K + w) * ext_cnt + (i % ext_cnt)];   // [part][K][ext_cnt]
                    }
                } else if (i < ns) {
                    // 16 consecutive jobs = one 32-byte sector of the row; chunks evenly strided over the jobs
                    long long col = cstride * (i >> 4) + (i & 15);
                    if (col >= N) col = N - 1;
                    c_r[q] = p.cost[col];
                    o_r[q] = p.owner[col];
                    s_r[q] = S[(size_t)w * ld + col];
                }
            }
#pragma unroll
            for (int q = 0; q < PER; ++q) {
                const int i = tid + (q0 + q) * AUC_SAMPLE_THREADS;
                unsigned short key = k_r[q];
                if (!ext_keys && peers.world == 0 && i < ns) {
                    __half c = c_r[q];
                    if (st.ff_pending > 0 && o_r[q] >= 0)
                        for (int r = 0; r < st.ff_pending; ++r) c = __hadd(c, eps);
                    const __half v = (o_r[q] == w) ? s_r[q] : __hsub(s_r[q], c);
                    key = (unsigned short)h2key(h2bits(v));
                }
                keys[i] = key;
                if (collect_out && i < collect_n) collect_out[(size_t)w * collect_n + i] = key;
            }
        }
    }
    if (collect_out) return;
    __syncthreads();
    // Only ranks r_hi .. r_lo of the descending order are needed (a few dozen for K >= 64): find the key at
    // rank r_lo by a two-level radix select, collect everything >= it and rank that short list by counting.
    // Full bitonic sort as the fallback (small K, or many duplicates).
    __shared__ unsigned int shist[256];
    __shared__ unsigned short top[1024], sorted[1024];
    __shared__ int s_b1, s_above1, s_vlo, s_cnt;
    bool need_full_sort = true;
    {
        const double r = (double)(jpw + 1) * (double)ns / (double)N - 0.5;
        const double sg = sqrt(r > 1.0 ? r : 1.0);
        long long r_lo = (long long)ceil(r + 4.5 * sg + 2.0);
        if (r_lo > ns - 1) r_lo = ns - 1;
        const int need_n = (int)r_lo + 1;
        if (need_n <= 512) {
            if (tid < 256) shist[tid] = 0;
            if (tid == 0) s_cnt = 0;
            __syncthreads();
            for (int i = tid; i < AUC_SAMPLE; i += AUC_SAMPLE_THREADS) atomicAdd(&shist[keys[i] >> 8], 1u);
            __syncthreads();
            if (tid < 32) sample_select_bin(shist, 0, need_n, &s_b1, &s_above1);
            __syncthreads();
            const int b1 = s_b1;
            if (tid < 256) shist[tid] = 0;
            __syncthreads();
            for (int i = tid; i < AUC_SAMPLE; i += AUC_SAMPLE_THREADS)
                if ((keys[i] >> 8) == b1) atomicAdd(&shist[keys[i] & 255], 1u);
            __syncthreads();
            if (tid < 32) {
                int bsel, dummy;
                sample_select_bin(shist, s_above1, need_n, &bsel, &dummy);
                if (tid == 0) s_vlo = (b1 << 8) | bsel;
            }
            __syncthreads();
            const int vlo = s_vlo;
            for (int i = tid; i < AUC_SAMPLE; i += AUC_SAMPLE_THREADS) {
                const unsigned short kk = keys[i];
                if ((int)kk >= vlo) {
                    const int slot = atomicAdd(&s_cnt, 1);
                    if (slot < 1024) top[slot] = kk;
                }
            }
            __syncthreads();
            const int cnt = s_cnt;
            if (cnt <= 1024) {
                need_full_sort = false;
                for (int i = tid; i < cnt; i += AUC_SAMPLE_THREADS) {
                    const unsigned short kk = top[i];
                    int rank = 0;
                    for (int j = 0; j < cnt; ++j) {
                        const unsigned short kj = top[j];
                        rank += (kj > kk) || (kj == kk && j < i);
                    }
                    sorted[rank] = kk;
                }
                __syncthreads();
                for (int i = tid; i < cnt; i += AUC_SAMPLE_THREADS) keys[i] = sorted[i];   // ranks 0 .. cnt-1 (>= r_lo) are exact
                __syncthreads();
            }
        }
    }
    if (need_full_sort) {
        // bitonic sort, descending
        for (int k = 2; k <= AUC_SAMPLE; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < AUC_SAMPLE; i += AUC_SAMPLE_THREADS) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const unsigned short a = keys[i], b2 = keys[ixj];
                        const bool desc = (i & k) == 0;
                        if (desc ? (a < b2) : (a > b2)) { keys[i] = b2; keys[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        }
    }
    if (tid == 0) {
        // rank (0-based, descending) of the (jpw+1)-th largest of N inside the sample, +- its spread
        const double r = (double)(jpw + 1) * (double)ns / (double)N - 0.5;
        const double sg = sqrt(r > 1.0 ? r : 1.0);
        long long r_hi = (long long)floor(r - 4.5 * sg - 2.0), r_lo = (long long)ceil(r + 4.5 * sg + 2.0);
        if (r_hi < 0) r_hi = 0;
        if (r_lo > ns - 1) r_lo = ns - 1;
        int lo = (int)keys[r_lo] - 1, hi = (int)keys[r_hi] + 1;
        if (r_hi == 0) hi += 32;                                            // the sample's maximum is no bound
        // costs only grow, so a worker's threshold never rises from one round to the next (up to a rare
        // tie corner case, which the slide-up path catches): the window need not reach above the last one
        const int tp = p.tprev[w];
        if (tp >= 0 && hi > tp + 2) hi = tp + 2;
        if (lo < AUC_MIN_KEY) lo = AUC_MIN_KEY;
        if (hi < lo + 8) hi = lo + 8;
        if (hi > 65535) hi = 65535;
        int span = hi - lo + 1, shift = 0, hb = lo + AUC_HALF, nlo = AUC_HALF;
        if (span > AUC_W) {
            // the candidates usually form two clumps (the worker's owned jobs at their full score, everything
            // else one or more cost steps lower): cut the window at the widest hole between consecutive
            // sampled candidates and spend the 128 one-key bins on the two sides; keys inside the hole are
            // counted in `gap`.  If the two sides do not fit: coarser bins and a refine pass.
            long long cut = -1;
            int hole = 0;
            for (long long q = r_hi; q < r_lo; ++q) {
                const int d = (int)keys[q] - (int)keys[q + 1];
                if (d > hole) { hole = d; cut = q; }
            }
            bool ok = false;
            if (cut >= 0) {
                const int up_lo = keys[cut], dn_hi = keys[cut + 1];       // hole = (dn_hi, up_lo)
                const int need_up = hi - up_lo + 1, need_dn = dn_hi - lo + 1;
                if (need_up + need_dn <= AUC_W && need_up >= 1 && need_dn >= 1) {
                    int spare = AUC_W - need_up - need_dn;
                    const int room = up_lo - dn_hi - 1;                    // keys strictly inside the hole
                    if (spare > room) spare = room;
                    const int ext_dn = spare / 2, ext_up = spare - ext_dn; // margins into the hole
                    nlo = need_dn + ext_dn;
                    hb = up_lo - ext_up;
                    ok = true;
                }
            }
            if (!ok) {
                while ((span >> shift) > AUC_W) ++shift;
                hb = lo + AUC_HALF;
                nlo = AUC_HALF;
            }
        }
        if (shift == 0 && nlo == AUC_HALF && hb == lo + AUC_HALF && lo > 65536 - AUC_W) { lo = 65536 - AUC_W; hb = lo + AUC_HALF; }
        p.win_base[w] = lo;
        p.win_hbase[w] = hb;
        p.win_nlo[w] = nlo;
        p.win_shift[w] = shift;
    }
}

// ------------------------------------------------------------------------------------------
// Sharded jobs, whole-round protocol (rqk_auction_peer_round): seven launches per round, chained with programmatic
// dependent launch, three flag barriers that sit INSIDE kernels which have work of their own:
//   1. auction_peer_bid_collect_kernel      (K CTAs)  counters of the previous round's bids exchanged and resolved
//                                                     (every CTA derives the next state from the summed counters, the
//                                                     LAST CTA applies it), then the local window samples
//   2. auction_sample_kernel                (K CTAs)  sample barrier, windows from the union of all ranks' samples
//   3. auction_hist_kernel                  (G CTAs)  dumps its histograms per CTA, as in the single-GPU driver
//   4. auction_peer_publish_kernel          (K CTAs)  CTA w sums worker w's dumps into this rank's exchange block; the
//                                                     last CTA signals the peers (histogram barrier)
//   5. auction_peer_resolve_workers_kernel  (K CTAs)  CTA w waits for the peers, sums worker w's row over the ranks,
//                                                     resolves it and takes its rank-major tie prefix
//   6. auction_bidlist_kernel               (G CTAs)  bid-list replay
//   7. auction_pass_kernel                  (G CTAs)  S-scanning fallback (returns at once unless a list overflowed)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024, 1)
auction_peer_bid_collect_kernel(const __half* __restrict__ S, long long ld, long long N, int K, long long n_global,
                                AuctionPtrs p, int count, PeerCtx peers, int seq_bid, int seq_sample) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ AuctionState st;
    __shared__ unsigned int s_sum[2];
    const int tid = threadIdx.x, w = blockIdx.x;
    if (tid == 0) st = *p.st;          // nobody writes the state before the LAST CTA of this grid has read it
    __syncthreads();
    if (st.mode == MODE_DONE) return;
    const bool was_bid = st.mode == MODE_BID;
    bool do_sample = st.mode == MODE_HIST && st.need_sample != 0;
    if (was_bid) {
        const int par = seq_bid & 1;
        if (w == 0 && tid == 0) {
            int* mine = peer_tail(peers, peers.rank, par);
            mine[0] = (int)*p.n_with;
            mine[1] = (int)*p.n_viol;
        }
        if (!peer_barrier(peers, 2, seq_bid, w == 0)) {
            if (tid == 0) { p.st->error = 1; p.st->mode = MODE_DONE; p.st->done = 1; }
            return;
        }
        if (tid < 32) {                                        // one lane per rank: the peer loads overlap
            unsigned int a = 0, b = 0;
            if (tid < peers.world) {
                const int* t = peer_tail(peers, tid, par);
                a = (unsigned int)__ldcv(t);
                b = (unsigned int)__ldcv(t + 1);
            }
#pragma unroll
            for (int d = 16; d; d >>= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, d);
                b += __shfl_xor_sync(0xffffffffu, b, d);
            }
            if (tid == 0) { s_sum[0] = a; s_sum[1] = b; }
        }
        __syncthreads();
        const BidOutcome o = bid_outcome(st.counter, s_sum[0], s_sum[1], n_global);
        __syncthreads();
        if (tid == 0 && !o.finished) {                         // the state auction_resolve_body will write
            st.counter += 1;
            st.ff_pending = 0;
            if (o.jump) { st.ff_pending = 100 - st.counter; st.counter = 100; }
            st.mode = MODE_HIST;
            st.need_sample = 1;
        }
        __syncthreads();
        do_sample = !o.finished;
    }
    if (do_sample) {
        // `count` evenly strided local jobs of worker w -> own exchange block (16 consecutive jobs = one sector)
        unsigned short* out = reinterpret_cast<unsigned short*>(peers.buf[peers.rank] + peer_sample_off(K)) +
                              (size_t)(seq_sample & 1) * K * AUC_SAMPLE_MAX + (size_t)w * count;
        long long ns = N < count ? N : count;
        const __half eps = bits2h(st.eps_bits);
        const long long nchunks = (ns + 15) / 16, cstride = N / (nchunks > 0 ? nchunks : 1);
        for (int i = tid; i < count; i += 1024) {
            unsigned short key = 0;                            // padding sorts last
            if (i < ns) {
                long long col = cstride * (i >> 4) + (i & 15);
                if (col >= N) col = N - 1;
                __half c = p.cost[col];
                const short o = p.owner[col];
                const __half sv = S[(size_t)w * ld + col];
                if (st.ff_pending > 0 && o >= 0)
                    for (int r = 0; r < st.ff_pending; ++r) c = __hadd(c, eps);
                key = (unsigned short)h2key(h2bits((o == w) ? sv : __hsub(sv, c)));
            }
            out[i] = key;
        }
    }
    if (was_bid && auction_last_cta(p.ticket)) {
        // every CTA has taken its snapshot of the state and CTA 0 has published the local counters: apply the round
        if (tid == 0) { *p.n_with = s_sum[0]; *p.n_viol = s_sum[1]; }
        __syncthreads();
        auction_resolve_body(p, n_global, K, n_global / K, MODE_BID);
    }
}

// Step-by-step flow (rqk_auction_resolve), after a resolve that leaves every worker resolved: per-CTA exclusive
// prefix of the number of values equal to the threshold (bin tkey-base of the per-CTA dumps).  Grid = K CTAs.
__global__ void __launch_bounds__(AUC_MAX_CTAS, 1)
auction_tieprefix_kernel(AuctionPtrs p, int K, int G) {
    pdl_launch_dependents();
    pdl_wait();
    if (p.st->mode != MODE_BID) return;
    const int w = blockIdx.x, tid = threadIdx.x;
    __shared__ unsigned int cnt[AUC_MAX_CTAS];
    const int base = p.win_base[w], hbase = p.win_hbase[w];
    const int tk = p.tkey[w];
    const int nlo = p.win_nlo[w];
    const int bin = tk >= hbase ? nlo + tk - hbase : tk - base;   // shift is 0 when resolved
    unsigned int c = 0;
    if (tid < G) c = p.hist_cta[((size_t)tid * K + w) * AUC_W + bin];
    cnt[tid] = c;
    __syncthreads();
    for (int d = 1; d < AUC_MAX_CTAS; d <<= 1) {   // Hillis-Steele inclusive scan
        unsigned int v = (tid >= d) ? cnt[tid - d] : 0;
        __syncthreads();
        cnt[tid] += v;
        __syncthreads();
    }
    if (tid < G) p.tieprefix[(size_t)tid * K + w] = cnt[tid] - c + p.rank_off[w];
    if (tid == AUC_MAX_CTAS - 1) p.tie_total[w] = cnt[AUC_MAX_CTAS - 1];
}

// ---- pieces shared by the per-worker merge kernels (one CTA of AUC_MAX_CTAS threads per worker) ----
struct MergeSmem {
    unsigned int part[8][AUC_W];
    unsigned int hist[AUC_W];
    unsigned int cnt[AUC_MAX_CTAS];
    unsigned int ab[AUC_MAX_CTAS / 32], gp[AUC_MAX_CTAS / 32];
};

// hist[0..255] = worker w's window histogram summed over the G per-CTA dumps of the HIST pass (16-bit pairs -> 32-bit
// bins); returns the summed above / gap counts to every thread.  Ends with a __syncthreads.
__device__ __forceinline__ void merge_worker_dumps(const AuctionPtrs& p, int K, int G, int w, MergeSmem& m,
                                                   unsigned int* above, unsigned int* gap) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int* d32 = reinterpret_cast<const unsigned int*>(p.hist_cta);
    const int word = tid & 127, grp = tid >> 7;              // 8 groups of 128 threads, group q takes CTAs q, q+8, ..
    unsigned int lo = 0, hi = 0;
#pragma unroll 8
    for (int g = grp; g < G; g += 8) {                       // ~37 independent loads per thread: keep 8 in flight
        const unsigned int h = __ldcg(d32 + ((size_t)g * K + w) * (AUC_W / 2) + word);
        lo += h & 0xffffu;
        hi += h >> 16;
    }
    m.part[grp][2 * word] = lo;
    m.part[grp][2 * word + 1] = hi;
    unsigned int ab = 0, gp = 0;
    if (tid < G) { ab = __ldcg(p.above_cta + (size_t)tid * K + w); gp = __ldcg(p.gap_cta + (size_t)tid * K + w); }
    ab = __reduce_add_sync(0xffffffffu, ab);
    gp = __reduce_add_sync(0xffffffffu, gp);
    if (lane == 0) { m.ab[warp] = ab; m.gp[warp] = gp; }
    __syncthreads();
    if (tid < AUC_W) {
        unsigned int t = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += m.part[q][tid];
        m.hist[tid] = t;
    }
    unsigned int abt = 0, gpt = 0;
    for (int q = 0; q < AUC_MAX_CTAS / 32; ++q) { abt += m.ab[q]; gpt += m.gp[q]; }
    *above = abt;
    *gap = gpt;
    __syncthreads();
}

// m.cnt[b] = number of values equal to worker w's threshold in CTA b's job range (0 for b >= G): exclusive prefix over
// the CTAs, offset by the ties lower ranks hold, -> tieprefix / tie_total.  All threads of the CTA; contains __syncthreads.
__device__ __forceinline__ void tie_scan_store(const AuctionPtrs& p, int K, int G, int w, MergeSmem& m, unsigned int rank_off) {
    const int tid = threadIdx.x;
    __syncthreads();
    const unsigned int c = m.cnt[tid];
    for (int d = 1; d < AUC_MAX_CTAS; d <<= 1) {                  // Hillis-Steele inclusive scan
        unsigned int v = (tid >= d) ? m.cnt[tid - d] : 0;
        __syncthreads();
        m.cnt[tid] += v;
        __syncthreads();
    }
    if (tid < G) p.tieprefix[(size_t)tid * K + w] = m.cnt[tid] - c + rank_off;
    if (tid == AUC_MAX_CTAS - 1) p.tie_total[w] = m.cnt[AUC_MAX_CTAS - 1];
}

// The per-CTA tie counts from the per-CTA dumps of the HIST pass (bin of the resolved threshold).
__device__ __forceinline__ void tie_prefix_worker(const AuctionPtrs& p, int K, int G, int w, MergeSmem& m, unsigned int rank_off) {
    const int tid = threadIdx.x;
    const int tk = p.tkey[w];
    const int base = p.win_base[w], hbase = p.win_hbase[w], nlo = p.win_nlo[w];
    const int bin = tk >= hbase ? nlo + tk - hbase : tk - base;   // shift is 0 when resolved
    unsigned int c = 0;
    if (tid < G) c = p.hist_cta[((size_t)tid * K + w) * AUC_W + bin];
    m.cnt[tid] = c;
    tie_scan_store(p, K, G, w, m, rank_off);
}

// One sweep over worker w's survivor lists (nseg segments of <= AUC_SEG_CAP entries) by all warps of the CTA.  A warp
// takes 8 consecutive segments at a time: their lengths with one load, then chunk c of all eight in flight together -
// the sweep is a chain of L2 round trips, so what counts is how few of them there are (at 10 M rows a worker has
// 2664 segments).  MODE 0: fh[key - lo] += 1 for lo <= key < lo + range;  MODE 1: cnt_cta[seg / spc] += #(key == lo).
// Returns (to lane 0 of each warp, OR it over the warps) whether a segment had overflowed.
template <int MODE>
__device__ __forceinline__ bool sweep_worker_lists(const AuctionPtrs& p, int K, int w, int nseg, int spc, int lo, int range,
                                                   unsigned int* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NWARP = blockDim.x >> 5;
    bool over = false;
    for (int s0 = warp * 8; s0 < nseg; s0 += NWARP * 8) {
        unsigned int cnt_l = 0;
        if (lane < 8 && s0 + lane < nseg) cnt_l = __ldcg(p.seg_cnt + (size_t)(s0 + lane) * K + w);
        unsigned int cnt[8], mx = 0, nt[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            cnt[u] = __shfl_sync(0xffffffffu, cnt_l, u);
            if (cnt[u] > AUC_SEG_CAP) { over = true; cnt[u] = 0; }
            mx = cnt[u] > mx ? cnt[u] : mx;
            nt[u] = 0;
        }
        for (unsigned int c = 0; c * 32 < mx; ++c) {
            const unsigned int i = c * 32 + lane;
            unsigned int e[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                e[u] = (i < cnt[u]) ? __ldcg(p.seg_list + ((size_t)(s0 + u) * K + w) * AUC_SEG_CAP + i) : 0xffffffffu;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (e[u] == 0xffffffffu) continue;               // (a job offset is < 4096: never a real entry)
                const int key = (int)(e[u] & 0xffffu);
                if (MODE == 0) { if (key >= lo && key < lo + range) atomicAdd(&out[key - lo], 1u); }
                else nt[u] += (key == lo) ? 1u : 0u;
            }
        }
        if (MODE == 1) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const unsigned int n = __reduce_add_sync(0xffffffffu, nt[u]);
                if (lane == 0 && n) atomicAdd(&out[(s0 + u) / spc], n);
            }
        }
    }
    return over;
}

// Refine from the survivor lists.  The worker's window had coarse bins (2^shift0 keys each, from `base0`) and the
// resolve step has just found the bin that holds the threshold and aimed a one-key window [nb2, nb2 + range) at it
// for another HIST pass over the worker's row (likewise for the gap of a split window).  But the pass that has just
// run already pushed EVERY value >= base0 of this worker into its survivor lists (job, exact key), so the one-key
// histogram of that range - and the per-CTA tie counts at the threshold - can be taken from the lists (L2-resident,
// ~2 % of the row) right here, and the extra pass over S never happens.  Returns false (nothing changed: the next
// HIST pass refines as before) if a list overflowed.  All threads of the CTA; m.part is reused as scratch.
__device__ __forceinline__ bool refine_from_lists(const AuctionPtrs& p, int K, int G, int spc, int w, MergeSmem& m,
                                                  unsigned long long above_bin, int nb2, int range, long long jpw, int passes) {
    __shared__ int s_over, s_T;
    __shared__ unsigned int s_above_T;
    const int tid = threadIdx.x, lane = tid & 31;
    unsigned int* fh = &m.part[0][0];                          // [range <= 8 * 256] one-key histogram of [nb2, nb2 + range)
    const int nseg = G * spc;
    for (int i = tid; i < range; i += AUC_MAX_CTAS) fh[i] = 0;
    if (tid == 0) { s_over = 0; s_T = -1; }
    m.cnt[tid] = 0;
    __syncthreads();
    if (sweep_worker_lists<0>(p, K, w, nseg, spc, nb2, range, fh) && lane == 0) s_over = 1;
    __syncthreads();
    if (s_over) return false;
    if (tid == 0) {
        const unsigned long long need = (unsigned long long)(jpw + 1);
        unsigned long long c = above_bin;
        for (int k = range - 1; k >= 0; --k) {
            if (c < need && c + fh[k] >= need) { s_T = nb2 + k; s_above_T = (unsigned int)c; break; }
            c += fh[k];
        }
    }
    __syncthreads();
    const int T = s_T;
    if (T < 0) return false;                                   // cannot happen with complete lists
    sweep_worker_lists<1>(p, K, w, nseg, spc, T, 1, m.cnt);
    if (tid == 0) {
        const int tp = p.tprev[w];
        if (tp >= 0) {
            const int d = tp - T;
            atomicAdd(&p.st->sink[d < 64 ? 0 : d < 128 ? 1 : d < 250 ? 2 : 3], 1);
        }
        p.tkey[w] = T;
        p.take[w] = (int)(jpw - (long long)s_above_T);
        p.res_pass[w] = passes;
        p.miss_run[w] = 0;
    }
    tie_scan_store(p, K, G, w, m, p.rank_off[w]);
    return true;
}

// State transition after a HIST pass whose workers were resolved one per CTA (part 4 of auction_resolve_body); run
// by thread 0 of the CTA that finished last.
__device__ __forceinline__ void merge_state_transition(const AuctionPtrs& p) {
    AuctionState s = *p.st;
    const int unresolved = __ldcg(&p.unres_g[0]), miss = __ldcg(&p.unres_g[1]);
    p.unres_g[0] = 0;
    p.unres_g[1] = 0;
    s.passes += 1;
    s.cold_passes += 1;
    s.window_misses += miss;
    s.ff_pending = 0;
    s.need_sample = 0;
    s.use_list = (*p.list_ok != 0 && !s.force_scan) ? 1 : 0;
    s.mode = (unresolved == 0) ? MODE_BID : MODE_HIST;
    *p.st = s;
}

// One warp: worker w's threshold from the histogram in m.hist (see resolve_one_worker).
__device__ __forceinline__ void resolve_worker_from_smem(const AuctionPtrs& p, int w, const MergeSmem& m, unsigned long long abt,
                                                         unsigned long long gpt, long long jpw, int passes, int* flags) {
    const int lane = threadIdx.x & 31;
    const int base = p.win_base[w], shift = p.win_shift[w];
    const int hbase = p.win_hbase[w], nlo = (shift == 0) ? p.win_nlo[w] : 0;
    const unsigned long long gap = (shift == 0) ? gpt : 0ull;
    unsigned int h[AUC_BPL];
    unsigned int lsum = 0;
#pragma unroll
    for (int i = 0; i < AUC_BPL; ++i) { h[i] = m.hist[lane * AUC_BPL + i]; lsum += h[i]; }
    resolve_one_worker(p, w, h, lsum, abt, gap, base, shift, hbase, nlo, jpw + 1, jpw, passes, p.st->sink, &flags[0], &flags[1]);
}

// Single-GPU driver, after a HIST pass that only dumped per CTA: CTA w sums worker w's window histogram over the G
// dumps, resolves the worker's threshold (what the last CTA of the HIST kernel used to do for all K workers one after
// the other), takes the tie prefix if the worker was resolved, and the CTA that finishes last makes the state
// transition of the resolve step.  Workers settled by an earlier pass of the round keep what that pass left
// (threshold, dump, tie prefix).
__global__ void __launch_bounds__(AUC_MAX_CTAS, 1)
auction_merge_resolve_kernel(AuctionPtrs p, int K, int G, long long jpw, int spc, int list_refine) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ MergeSmem m;
    __shared__ int s_flag[2], s_mode, s_passes, s_scan;
    const int w = blockIdx.x, tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { s_mode = p.st->mode; s_passes = p.st->passes; s_scan = p.st->force_scan; s_flag[0] = 0; s_flag[1] = 0; }
    __syncthreads();
    if (s_mode != MODE_HIST) return;                         // no HIST pass has just run (done, or a no-op round)
    if (s_scan) list_refine = 0;                             // the S-scanning route stays independent of the lists
    const bool settled = p.tkey[w] >= 0;
    if (!settled) {
        unsigned int abt, gpt;
        merge_worker_dumps(p, K, G, w, m, &abt, &gpt);
        const int base0 = p.win_base[w], shift0 = p.win_shift[w];   // the window the pass ran with
        const int hbase0 = p.win_hbase[w], nlo0 = p.win_nlo[w];
        __syncthreads();
        if (warp == 0) resolve_worker_from_smem(p, w, m, abt, gpt, jpw, s_passes, s_flag);
        __syncthreads();
        if (p.tkey[w] >= 0) {
            tie_prefix_worker(p, K, G, w, m, p.rank_off[w]);
        } else if (list_refine && base0 > 0 && shift0 >= 1 && shift0 <= 8 && p.win_shift[w] == 0 && p.win_base[w] >= base0) {
            // resolved to a coarse bin of a sampled window: finish from the survivor lists instead of another pass
            const int nb2 = p.win_base[w], bin = (nb2 - base0) >> shift0;
            unsigned long long above_bin = abt;
            for (int i = bin + 1; i < AUC_W; ++i) above_bin += m.hist[i];
            __syncthreads();                                   // m.hist / m.part are about to be reused
            if (refine_from_lists(p, K, G, spc, w, m, above_bin, nb2, 1 << shift0, jpw, s_passes) && tid == 0) {
                s_flag[0] = 0;
                atomicAdd(&p.st->branch[0], -1);               // statistics: this refine did not cost a pass
            }
        } else if (list_refine && base0 > 0 && shift0 == 0 && hbase0 > base0 + nlo0 && p.win_base[w] == base0 + nlo0 &&
                   hbase0 - (base0 + nlo0) <= 8 * AUC_W) {
            // the threshold fell into the gap of a split window (keys [base0 + nlo0, hbase0), up to 2048 of them):
            // those values are in the survivor lists as well
            unsigned long long above_gap = abt;
            for (int i = nlo0; i < AUC_W; ++i) above_gap += m.hist[i];
            __syncthreads();
            if (refine_from_lists(p, K, G, spc, w, m, above_gap, base0 + nlo0, hbase0 - (base0 + nlo0), jpw, s_passes) && tid == 0) {
                s_flag[0] = 0;
                atomicAdd(&p.st->branch[1], -1);
            }
        }
        __syncthreads();
        if (tid == 0) {
            if (s_flag[0]) atomicAdd(&p.unres_g[0], 1);
            if (s_flag[1]) atomicAdd(&p.unres_g[1], 1);
        }
    }
    if (auction_last_cta(p.ticket) && tid == 0) merge_state_transition(p);
}

// Sharded jobs, whole-round protocol, after a HIST pass that only dumped per CTA.  Two kernels of K CTAs:
//  publish   CTA w sums worker w's dumps and writes the LOCAL histogram row (+ above / gap) into this rank's exchange
//            block with plain stores; the CTA that finishes last signals every peer (flag kind 1).  Never waits.
//  resolve   CTA w waits for the peers' signals, sums worker w's row over the ranks (all peers' loads in flight
//            together: one NVLink round trip of 1 KB per peer), resolves the threshold - every rank computes the same -
//            and takes the tie prefix over its own CTAs, offset by the ties lower ranks hold at the resolved bin (their
//            local rows are in shared memory already).  Last CTA: state transition.
// Rows of settled workers are neither written nor read; rows are rewritten in full every pass, so nothing is cleared.
__global__ void __launch_bounds__(AUC_MAX_CTAS, 1)
auction_peer_publish_kernel(AuctionPtrs p, int K, int G, PeerCtx peers, int seq) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ MergeSmem m;
    __shared__ int s_mode;
    const int w = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_mode = p.st->mode;
    __syncthreads();
    if (s_mode != MODE_HIST) return;
    if (p.tkey[w] < 0) {
        unsigned int abt, gpt;
        merge_worker_dumps(p, K, G, w, m, &abt, &gpt);
        unsigned int* mine = peer_hist(peers, peers.rank, K, seq & 1);
        if (tid < AUC_W) mine[(size_t)w * AUC_W + tid] = m.hist[tid];
        if (tid == 0) { mine[(size_t)K * AUC_W + w] = abt; mine[(size_t)K * AUC_W + K + w] = gpt; }
    }
    __threadfence_system();
    __syncthreads();
    if (tid == 0) {
        const int t = atomicAdd(&p.unres_g[2], 1);
        s_mode = (t == (int)gridDim.x - 1) ? 1 : 0;
        if (s_mode) p.unres_g[2] = 0;
    }
    __syncthreads();
    if (s_mode && tid < peers.world && tid != peers.rank) {     // every local row is in place: tell the peers
        __threadfence_system();
        int* dst = peer_flags(peers, tid) + 1 * PEER_MAX + peers.rank;
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(dst), "r"(seq) : "memory");
    }
}

__global__ void __launch_bounds__(AUC_MAX_CTAS, 1)
auction_peer_resolve_workers_kernel(AuctionPtrs p, int K, int G, long long jpw, PeerCtx peers, int seq) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ MergeSmem m;
    __shared__ unsigned int s_rows[PEER_MAX][AUC_W];          // the ranks' local rows of worker w
    __shared__ unsigned int s_abgp[2][PEER_MAX];
    __shared__ int s_flag[2], s_mode, s_passes;
    const int w = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, par = seq & 1;
    if (tid == 0) { s_mode = p.st->mode; s_passes = p.st->passes; s_flag[0] = 0; s_flag[1] = 0; }
    __syncthreads();
    if (s_mode != MODE_HIST) return;
    const bool settled = p.tkey[w] >= 0;
    if (!settled) {
        if (!peer_barrier(peers, 1, seq, false)) {              // wait only: auction_peer_publish_kernel has signalled
            if (tid == 0) { p.st->error = 1; p.st->mode = MODE_DONE; p.st->done = 1; }
            return;
        }
        // the ranks' rows: thread (r, i) loads bin i of rank r - 8 x 256 loads, all in flight together
        for (int i = tid; i < PEER_MAX * AUC_W; i += AUC_MAX_CTAS) {
            const int r = i / AUC_W, b = i % AUC_W;
            unsigned int v = 0;
            if (r < peers.world) {
                const unsigned int* src = peer_hist(peers, r, K, par) + (size_t)w * AUC_W + b;
                v = (r == peers.rank) ? __ldcg(src) : __ldcv(src);
            }
            s_rows[r][b] = v;
        }
        if (tid < 2 * PEER_MAX) {
            const int r = tid % PEER_MAX, which = tid / PEER_MAX;
            unsigned int v = 0;
            if (r < peers.world) {
                const unsigned int* src = peer_hist(peers, r, K, par) + (size_t)K * AUC_W + (size_t)which * K + w;
                v = (r == peers.rank) ? __ldcg(src) : __ldcv(src);
            }
            s_abgp[which][r] = v;
        }
        __syncthreads();
        if (tid < AUC_W) {
            unsigned int t = 0;
#pragma unroll
            for (int r = 0; r < PEER_MAX; ++r) t += s_rows[r][tid];
            m.hist[tid] = t;
        }
        __syncthreads();
        if (warp == 0) {
            unsigned long long abt = 0, gpt = 0;
#pragma unroll
            for (int r = 0; r < PEER_MAX; ++r) { abt += s_abgp[0][r]; gpt += s_abgp[1][r]; }
            resolve_worker_from_smem(p, w, m, abt, gpt, jpw, s_passes, s_flag);
        }
        __syncthreads();
        const int tk = p.tkey[w];
        if (tk >= 0) {
            const int base = p.win_base[w], hbase = p.win_hbase[w], nlo = p.win_nlo[w];
            const int bin = tk >= hbase ? nlo + tk - hbase : tk - base;
            unsigned int off = 0;
            for (int r = 0; r < peers.rank; ++r) off += s_rows[r][bin];   // rank-major: lower ranks' ties come first
            if (tid == 0) p.rank_off[w] = off;
            tie_prefix_worker(p, K, G, w, m, off);
        }
        if (tid == 0) {
            if (s_flag[0]) atomicAdd(&p.unres_g[0], 1);
            if (s_flag[1]) atomicAdd(&p.unres_g[1], 1);
        }
    }
    if (auction_last_cta(p.ticket) && tid == 0) merge_state_transition(p);
}

// sharded jobs: ranks are ordered, so a rank's CTAs come after all ties of lower ranks
__global__ void auction_tie_offset_kernel(AuctionPtrs p, int K, int G, const int* __restrict__ totals, int rank) {
    if (p.st->mode != MODE_BID) return;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < G * K) {
        unsigned int off = 0;
        for (int r = 0; r < rank; ++r) off += (unsigned int)totals[r * K + i % K];
        p.tieprefix[i] += off;
    }
}

__global__ void auction_finalize_kernel(AuctionPtrs p, long long N, int* __restrict__ assign) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        short o = p.owner[i];
        assign[i] = o >= 0 ? (int)o : 0;   // never-bid jobs land on worker 0 (:88-89 with a flat index < N)
    }
}

}  // namespace rqk

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
namespace rqk {
struct AuctionArgs {
    AuctionPtrs p;
    int G, J;
    size_t smem;
};
static int auction_prepare(int64_t n, int64_t ld, int32_t k, void* workspace, size_t workspace_bytes, AuctionArgs* a,
                           const char* who) {
    if (!workspace) return fail(RQK_ERR_ARG, "%s: null workspace", who);
    if (k < 1 || k > 256) return fail(RQK_ERR_UNSUPPORTED, "%s: k=%lld outside [1,256]", who, k);
    if (n < 1) return fail(RQK_ERR_ARG, "%s: n=%lld < 1", who, n);
    if (ld % 128 != 0 || ld < n) return fail(RQK_ERR_ARG, "%s: ld=%lld must be a multiple of 128 and >= n", who, ld);
    size_t need = auction_ws_layout(n, ld, k, &a->p, (char*)workspace);
    if (workspace_bytes < need) return fail(RQK_ERR_WORKSPACE, "%s: workspace %lld < %lld bytes", who, (long long)workspace_bytes, (long long)need);
    a->G = auction_grid(n, k);
    if (a->G > AUC_MAX_CTAS) return fail(RQK_ERR_UNSUPPORTED, "%s: n=%lld jobs per GPU exceed the 66 M limit of this build", who, n);
    a->J = auction_tile_cols(k);
    a->smem = auction_pass_smem(k, a->J);
    return 0;
}

// Enqueues the kernels of one pass; the device-side state machine makes those whose turn it is not return at
// once.  which: bit 0 window sampling, bit 1 HIST, bit 2 BID (list replay + S scan), bit 3 merge + resolve (between
// HIST and BID; fused only).  fused: HIST dumps per CTA and the last CTA of a bidding kernel runs the resolve step.
template <typename... KArgs, typename... Args>
static cudaError_t launch_round_kernel(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem,
                                       cudaStream_t stream, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// RQK_AUCTION_NO_LIST_REFINE=1 (tests, timing): coarse windows are always refined by another HIST pass
static bool auction_list_refine_ok() {
    static const bool ok = [] { const char* e = getenv("RQK_AUCTION_NO_LIST_REFINE"); return !(e && e[0] == '1'); }();
    return ok;
}

static bool auction_pdl_ok() {
    static const bool ok = [] { const char* e = getenv("RQK_NO_PDL"); return !(e && e[0] == '1'); }();
    return ok;
}

static int auction_launch(const AuctionArgs& a, const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global,
                          int which, int fused, cudaStream_t stream, bool chain = false) {
    // the single-GPU driver (fused resolve) and the whole-round sharded protocol (`chain`) chain their round kernels
    // with programmatic dependent launch
    const bool pdl = (fused != 0 || chain) && auction_pdl_ok();
    auto kern = (a.J == 128) ? auction_pass_kernel<128> : auction_pass_kernel<64>;
    // the attribute is per device (and this process may drive several): cache what has been set per device ordinal
    int devi = 0;
    RQK_CUDA_OK(cudaGetDevice(&devi));
    devi &= RQK_MAX_DEVICES - 1;
    static size_t smem_set[RQK_MAX_DEVICES][2] = {};
    size_t& cur = smem_set[devi][a.J == 128 ? 0 : 1];
    if (a.smem > cur) {
        RQK_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a.smem));
        cur = a.smem;
    }
    const int spc = auction_spc(n, k);
    if (which & 1)
        RQK_CUDA_OK(launch_round_kernel(auction_sample_kernel, (unsigned)k, (unsigned)AUC_SAMPLE_THREADS, 0, stream, pdl, (const __half*)scores_t,
                                        (long long)ld, (long long)n, (int)k, (long long)(n_global / k), a.p,
                                        (unsigned short*)nullptr, 0, (const unsigned short*)nullptr, 0, 1, PeerCtx{}, 0));
    if (which & 2) {
        static bool hs_set[RQK_MAX_DEVICES] = {};
        const size_t hs = HistSmem::TOTAL;
        if (!hs_set[devi]) {
            RQK_CUDA_OK(cudaFuncSetAttribute(auction_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hs));
            hs_set[devi] = true;
        }
        RQK_CUDA_OK(launch_round_kernel(auction_hist_kernel, (unsigned)a.G, (unsigned)AUC_THREADS, hs, stream, pdl,
                                        (const __half*)scores_t, (long long)ld, (long long)n, (int)k, a.J, spc, a.p,
                                        (long long)n_global, fused));
    }
    if (which & 8)      // HIST only dumped: merge + resolve + tie prefix, one CTA per worker
        RQK_CUDA_OK(launch_round_kernel(auction_merge_resolve_kernel, (unsigned)k, (unsigned)AUC_MAX_CTAS, 0, stream, pdl,
                                        a.p, (int)k, a.G, (long long)(n_global / k), spc, auction_list_refine_ok() ? 1 : 0));
    if (which & 4) {
        RQK_CUDA_OK(launch_round_kernel(auction_bidlist_kernel, (unsigned)a.G, (unsigned)AUC_THREADS, 0, stream, pdl,
                                        (const __half*)scores_t, (long long)ld, (long long)n, (int)k, a.J, spc, a.p,
                                        (long long)n_global, fused));
        RQK_CUDA_OK(launch_round_kernel(kern, (unsigned)a.G, (unsigned)AUC_THREADS, a.smem, stream, pdl,
                                        (const __half*)scores_t, (long long)ld, (long long)n, (int)k, (long long)(n_global / k),
                                        a.p, (long long)n_global, fused));
    }
    RQK_LAUNCH_OK();
    return 0;
}
}  // namespace rqk

extern "C" {

struct rqk_auction_layout {
    int64_t total_bytes;        // workspace size
    int64_t reduce_offset;      // byte offset of the int32 reduce block (sum over ranks after every pass)
    int64_t reduce_count;       // its length in int32 elements: k*256 + 2k + 2
    int64_t tie_total_offset;   // byte offset of int32[k]: local ties at the threshold (allgather after resolve)
};

struct rqk_auction_info {
    int32_t done;
    int32_t rounds;         // what the reference's loop would have executed (1002 in the fallback regime)
    int32_t passes;         // passes over the score matrix actually made
    int32_t cold_passes;    // of which histogram-only (cold start / window miss / after fast-forward)
    int32_t window_misses;
    int32_t frozen_exit;    // 1 = ended through the frozen-state shortcut
    int32_t counter;        // reference `counter` at exit
    uint16_t eps_bits;
    uint16_t list_passes;
};

int rqk_auction_layout_query(int64_t n, int32_t k, rqk_auction_layout* out) {
    using namespace rqk;
    if (!out || n < 1 || k < 1 || k > 256) return fail(RQK_ERR_ARG, "rqk_auction_layout_query: bad argument%s");
    long long ld = round_up<long long>(n, 128);
    size_t ro = 0, to = 0;
    out->total_bytes = (int64_t)auction_ws_layout(n, ld, k, nullptr, nullptr, &ro, &to);
    out->reduce_offset = (int64_t)ro;
    out->reduce_count = (int64_t)k * AUC_W + 2 * k + 2;
    out->tie_total_offset = (int64_t)to;
    return 0;
}

size_t rqk_auction_workspace_bytes(int64_t n, int32_t k) {
    long long ld = rqk::round_up<long long>(n, 128);
    return rqk::auction_ws_layout(n, ld, k, nullptr, nullptr);
}

// minmax_keys: device uint32[2] = {max key, min key} over ALL ranks' score entries.
int rqk_auction_init(int64_t n, int64_t ld, int32_t k, const void* minmax_keys, void* workspace,
                     size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_init");
    if (rc) return rc;
    if (!minmax_keys) return fail(RQK_ERR_ARG, "rqk_auction_init: null minmax_keys%s");
    cudaStream_t stream = (cudaStream_t)stream_;
    RQK_CUDA_OK(cudaMemsetAsync(a.p.tieprefix, 0, (size_t)a.G * k * 4, stream));
    const char* ns = getenv("RQK_AUCTION_NO_LIST");      // tests: force the S-scanning BID kernel
    auction_init_kernel<<<148, 256, 0, stream>>>(a.p, ld, k, (const unsigned int*)minmax_keys, (ns && ns[0] == '1') ? 1 : 0);
    RQK_LAUNCH_OK();
    return 0;
}

// One pass over this rank's [k][ld] score shard (n local jobs).  jobs_per_worker = n_global / k.
// The device-side state machine decides what the pass is: three kernels are enqueued and two of them
// return at once - window sampling (only when windows are cold and the jobs are not sharded), the
// streaming HIST kernel, the tiled BID kernel.  `which` (0 = all) restricts the launch to a subset
// (bit 0 sample, bit 1 HIST, bit 2 BID, bit 3 merge + resolve with bit 4) so that a caller can time one kernel alone.
int rqk_auction_pass(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, int32_t which,
                     void* workspace, size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_pass");
    if (rc) return rc;
    if (!scores_t) return fail(RQK_ERR_ARG, "rqk_auction_pass: null scores%s");
    if (n_global < k) return fail(RQK_ERR_ARG, "rqk_auction_pass: n_global=%s%lld < k=%lld (argmin path, reference :24-26)", "", n_global, k);
    if (which == 0) which = 7;
    if (n_global != n) which &= ~1;   // sharded jobs: rqk_auction_sample_collect / _window (ranks must agree on the windows)
    // bit 4: the kernels of the single-GPU driver's flow (HIST dumps per CTA, bit 3 = merge + resolve + tie prefix, the
    // bidding kernel's last CTA resolves) - timing and tests of exactly what rqk_auction chains; unsharded jobs only
    const int fused = (which & 16) && n_global == n ? 1 : 0;
    if ((which & 8) && !fused) return fail(RQK_ERR_ARG, "rqk_auction_pass: bit 3 (merge + resolve) needs bit 4 and unsharded jobs%s");
    return auction_launch(a, scores_t, ld, n, k, n_global, which & 15, fused, (cudaStream_t)stream_);
}

// Sharded window sampling, step 1: keys of `count` (<= 8192) evenly strided local jobs per worker -> out [k][count]
// (uint16 fp16 keys).  Writes nothing unless the state machine wants a sample (then `out` is untouched and the
// window step ignores it), so the host may call both steps unconditionally before every pass.
int rqk_auction_sample_collect(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, void* out,
                               int32_t count, void* workspace, size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_sample_collect");
    if (rc) return rc;
    if (!scores_t || !out || count < 1 || count > AUC_SAMPLE) return fail(RQK_ERR_ARG, "rqk_auction_sample_collect: bad argument%s");
    auction_sample_kernel<<<k, AUC_SAMPLE_THREADS, 0, (cudaStream_t)stream_>>>((const __half*)scores_t, ld, n, k, n_global / k, a.p,
                                                                  (unsigned short*)out, count, nullptr, 0, 1, PeerCtx{}, 0);
    RQK_LAUNCH_OK();
    return 0;
}

// Sharded window sampling, step 2: keys [parts][k][count] = the all-gathered samples of every rank, exactly as an
// all-gather of step 1's outputs lays them out (parts * count <= 8192).
int rqk_auction_sample_window(int64_t n, int64_t ld, int32_t k, int64_t n_global, const void* keys, int32_t count,
                              int32_t parts, void* workspace, size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_sample_window");
    if (rc) return rc;
    if (!keys || count < 1 || parts < 1 || (int64_t)count * parts > AUC_SAMPLE)
        return fail(RQK_ERR_ARG, "rqk_auction_sample_window: bad argument%s");
    auction_sample_kernel<<<k, AUC_SAMPLE_THREADS, 0, (cudaStream_t)stream_>>>(nullptr, ld, n_global, k, n_global / k, a.p, nullptr, 0,
                                                                  (const unsigned short*)keys, count * parts, count, PeerCtx{}, 0);
    RQK_LAUNCH_OK();
    return 0;
}

// Thresholds from the (already rank-summed) reduce block + local tie prefix.
// expect: -1, or 0 (HIST) / 1 (BID): act only if that is the pass that just ran, so that a caller can enqueue
// "HIST, resolve(0), BID, resolve(1)" per round without knowing whether the HIST pass resolved every threshold.
int rqk_auction_resolve(int64_t n, int64_t ld, int32_t k, int64_t n_global, int32_t expect, void* workspace,
                        size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_resolve");
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (expect < -1 || expect > 1) return fail(RQK_ERR_ARG, "rqk_auction_resolve: expect must be -1, 0 or 1%s");
    auction_resolve_kernel<<<1, 1024, 0, stream>>>(a.p, n_global, k, n_global / k, expect);
    auction_tieprefix_kernel<<<k, AUC_MAX_CTAS, 0, stream>>>(a.p, k, a.G);
    RQK_LAUNCH_OK();
    return 0;
}

// ---- peer-memory sharding (DESIGN.md section 4): the exchange is inside the kernels ----
// peers: HOST array of `world` device pointers, peers[r] = rank r's exchange block (rqk_auction_peer_bytes(k_max)
// bytes of symmetric memory, zeroed once before first use) as mapped into THIS process.  Its flags are never reset:
// sequence numbers only grow, over all auctions that share the block.
size_t rqk_auction_peer_bytes(int32_t k) { return rqk::peer_bytes(k); }

static int peer_ctx(const void* const* peers, int32_t world, int32_t rank, rqk::PeerCtx* c, const char* who) {
    using namespace rqk;
    if (!peers || world < 1 || world > PEER_MAX || rank < 0 || rank >= world)
        return fail(RQK_ERR_ARG, "%s: bad peer arguments (world 1..8)", who);
    for (int r = 0; r < PEER_MAX; ++r) c->buf[r] = r < world ? (unsigned char*)peers[r] : nullptr;
    for (int r = 0; r < world; ++r)
        if (!c->buf[r]) return fail(RQK_ERR_ARG, "%s: null peer pointer", who);
    c->world = world;
    c->rank = rank;
    return 0;
}

// One whole ROUND of a sharded job in one call: seven launches chained with programmatic dependent launch (see
// "whole-round protocol" above).  Sequence numbers: seq0 = the bid-counter exchange of the PREVIOUS round (its
// resolve runs at the head of this call), seq0+1 the window samples, seq0+2 the threshold histograms; this round's
// bid counters are exchanged under seq0+3 by the next call (the caller advances its counter by 3 per call and
// keeps calling until the state reports done).
int rqk_auction_peer_round(const void* scores_t, int64_t ld, int64_t n, int32_t k, int64_t n_global, int32_t count,
                           const void* const* peers, int32_t world, int32_t rank, int32_t seq0, void* workspace,
                           size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_peer_round");
    if (rc) return rc;
    PeerCtx c;
    if ((rc = peer_ctx(peers, world, rank, &c, "rqk_auction_peer_round"))) return rc;
    if (!scores_t || count < 1 || (int64_t)count * world > AUC_SAMPLE) return fail(RQK_ERR_ARG, "rqk_auction_peer_round: bad argument%s");
    if (n_global < k) return fail(RQK_ERR_ARG, "rqk_auction_peer_round: n_global=%s%lld < k=%lld", "", n_global, k);
    cudaStream_t stream = (cudaStream_t)stream_;
    const bool pdl = auction_pdl_ok();
    RQK_CUDA_OK(launch_round_kernel(auction_peer_bid_collect_kernel, (unsigned)k, 1024u, 0, stream, pdl, (const __half*)scores_t,
                                    (long long)ld, (long long)n, (int)k, (long long)n_global, a.p, (int)count, c, (int)seq0,
                                    (int)(seq0 + 1)));
    RQK_CUDA_OK(launch_round_kernel(auction_sample_kernel, (unsigned)k, (unsigned)AUC_SAMPLE_THREADS, 0, stream, pdl, (const __half*)nullptr, (long long)ld,
                                    (long long)n_global, (int)k, (long long)(n_global / k), a.p, (unsigned short*)nullptr, 0,
                                    (const unsigned short*)nullptr, (int)(count * world), (int)count, c, (int)(seq0 + 1)));
    // HIST dumps per CTA (as in the single-GPU driver); the per-worker publish / resolve kernels exchange the rows
    if ((rc = auction_launch(a, scores_t, ld, n, k, n_global, 2, 1, stream, true))) return rc;
    RQK_CUDA_OK(launch_round_kernel(auction_peer_publish_kernel, (unsigned)k, (unsigned)AUC_MAX_CTAS, 0, stream, pdl, a.p, (int)k,
                                    a.G, c, (int)(seq0 + 2)));
    RQK_CUDA_OK(launch_round_kernel(auction_peer_resolve_workers_kernel, (unsigned)k, (unsigned)AUC_MAX_CTAS, 0, stream, pdl, a.p,
                                    (int)k, a.G, (long long)(n_global / k), c, (int)(seq0 + 2)));
    if ((rc = auction_launch(a, scores_t, ld, n, k, n_global, 4, 0, stream, true))) return rc;
    RQK_LAUNCH_OK();
    return 0;
}

// totals: device int32[world][k] = every rank's tie_total (an all-gather of it); this rank's CTAs come after all
// ties of the ranks below it.
int rqk_auction_tie_offset(int64_t n, int64_t ld, int32_t k, const int32_t* totals, int32_t rank, void* workspace,
                           size_t workspace_bytes, void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_tie_offset");
    if (rc) return rc;
    if (!totals || rank < 0) return fail(RQK_ERR_ARG, "rqk_auction_tie_offset: bad argument%s");
    if (rank == 0) return 0;
    auction_tie_offset_kernel<<<ceil_div(a.G * k, 256), 256, 0, (cudaStream_t)stream_>>>(a.p, k, a.G, totals, rank);
    RQK_LAUNCH_OK();
    return 0;
}

// Copies the state machine's status to the host.  Synchronises `stream`.
int rqk_auction_poll(int64_t n, int64_t ld, int32_t k, void* workspace, size_t workspace_bytes, rqk_auction_info* info,
                     void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_poll");
    if (rc) return rc;
    if (!info) return fail(RQK_ERR_ARG, "rqk_auction_poll: null info%s");
    AuctionState host;
    cudaStream_t stream = (cudaStream_t)stream_;
    RQK_CUDA_OK(cudaMemcpyAsync(&host, a.p.st, sizeof(host), cudaMemcpyDeviceToHost, stream));
    RQK_CUDA_OK(cudaStreamSynchronize(stream));
    if (host.error)
        return fail(RQK_ERR_INTERNAL, "auction: device-side error %s%lld (1 = a peer rank did not arrive within 4 s)", "", (long long)host.error);
    info->done = host.done;
    info->rounds = host.rounds;
    info->passes = host.passes;
    info->cold_passes = host.cold_passes;
    info->window_misses = host.window_misses;
    info->frozen_exit = host.frozen_exit;
    info->counter = host.counter;
    info->eps_bits = (uint16_t)host.eps_bits;
    info->list_passes = (uint16_t)(host.list_passes > 65535 ? 65535 : host.list_passes);
    return 0;
}

int rqk_auction_finalize(int64_t n, int64_t ld, int32_t k, void* workspace, size_t workspace_bytes, int32_t* assign,
                         void* stream_) {
    using namespace rqk;
    AuctionArgs a;
    int rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction_finalize");
    if (rc) return rc;
    if (!assign) return fail(RQK_ERR_ARG, "rqk_auction_finalize: null assign%s");
    auction_finalize_kernel<<<(unsigned)ceil_div<long long>(n, 256), 256, 0, (cudaStream_t)stream_>>>(a.p, n, assign);
    RQK_LAUNCH_OK();
    return 0;
}

// Single-GPU driver of the pieces above.
// scores_t: device [k][ld] fp16 (ld = multiple of 128 >= n, columns >= n hold -inf); minmax_keys: device
// uint32[2] = {max key, min key} of the valid entries (monotone fp16 keys, see common.cuh).
// assign: device int32[n].  Synchronises `stream` (returns host scalars in *info).
int rqk_auction(const void* scores_t, int64_t ld, int64_t n, int32_t k, const void* minmax_keys,
                int32_t* assign, void* workspace, size_t workspace_bytes, rqk_auction_info* info,
                void* stream_) {
    using namespace rqk;
    if (n < k) return fail(RQK_ERR_ARG, "rqk_auction: n=%s%lld < k=%lld (use the argmin path, reference :24-26)", "", n, k);
    int rc = rqk_auction_init(n, ld, k, minmax_keys, workspace, workspace_bytes, stream_);
    if (rc) return rc;
    rqk_auction_info st;
    memset(&st, 0, sizeof(st));
    AuctionArgs a;
    if ((rc = auction_prepare(n, ld, k, workspace, workspace_bytes, &a, "rqk_auction"))) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    // A round = sample, HIST (+ resolve in its last CTA), tie prefix, BID (+ resolve).  The host never waits for
    // the round it just enqueued: the state is copied to a pinned two-slot mailbox after every batch and the
    // host looks at the copy of the batch BEFORE the one it enqueued last, so the GPU always has work queued
    // (passes enqueued after the auction finished return at once).  The mailbox (pinned host memory, 2 x 128 B
    // per host thread) is the one allocation this library makes.
    // per host thread AND per device: an event belongs to the device that was current when it was created
    static thread_local AuctionState* mailbox_d[RQK_MAX_DEVICES] = {};
    static thread_local cudaEvent_t ev_d[RQK_MAX_DEVICES][2];
    int devi = 0;
    RQK_CUDA_OK(cudaGetDevice(&devi));
    devi &= RQK_MAX_DEVICES - 1;
    if (!mailbox_d[devi]) {
        RQK_CUDA_OK(cudaHostAlloc((void**)&mailbox_d[devi], 2 * sizeof(AuctionState), cudaHostAllocPortable));
        RQK_CUDA_OK(cudaEventCreateWithFlags(&ev_d[devi][0], cudaEventDisableTiming));
        RQK_CUDA_OK(cudaEventCreateWithFlags(&ev_d[devi][1], cudaEventDisableTiming));
    }
    AuctionState* mailbox = mailbox_d[devi];
    cudaEvent_t* ev = ev_d[devi];
    const int rounds_per_batch = 2;
    const AuctionState* fin = nullptr;
    // hard stop: the reference itself cannot exceed 1002 rounds; each round is a handful of passes at most
    for (int b = 0; b < 4000 && !fin; ++b) {
        for (int q = 0; q < rounds_per_batch; ++q)
            if ((rc = auction_launch(a, scores_t, ld, n, k, n, 1 | 2 | 4 | 8, 1, stream))) return rc;
        RQK_CUDA_OK(cudaMemcpyAsync(&mailbox[b & 1], a.p.st, sizeof(AuctionState), cudaMemcpyDeviceToHost, stream));
        RQK_CUDA_OK(cudaEventRecord(ev[b & 1], stream));
        if (b >= 1) {
            RQK_CUDA_OK(cudaEventSynchronize(ev[(b - 1) & 1]));
            if (mailbox[(b - 1) & 1].done) fin = &mailbox[(b - 1) & 1];
        }
    }
    // drain the trailing (no-op) batch so that no mailbox copy is in flight when this thread's next auction starts
    RQK_CUDA_OK(cudaStreamSynchronize(stream));
    if (fin) {
        st.done = fin->done; st.rounds = fin->rounds; st.passes = fin->passes; st.cold_passes = fin->cold_passes;
        st.window_misses = fin->window_misses; st.frozen_exit = fin->frozen_exit; st.counter = fin->counter;
        st.eps_bits = (uint16_t)fin->eps_bits;
        st.list_passes = (uint16_t)(fin->list_passes > 65535 ? 65535 : fin->list_passes);
    }
    if (fin) {
        static const bool dbg = [] { const char* e = getenv("RQK_AUCTION_DEBUG"); return e && e[0] == '1'; }();
        if (dbg)
            fprintf(stderr, "rqk_auction n=%lld k=%d: rounds %d passes %d (HIST %d, from lists %d) window misses %d | worker-passes: "
                    "refine in coarse bin %d, in gap %d, slide %d, coarse restart %d | sink <64 %d <128 %d <250 %d >=250 %d\n",
                    (long long)n, (int)k, fin->rounds, fin->passes, fin->cold_passes, fin->list_passes, fin->window_misses,
                    fin->branch[0], fin->branch[1], fin->branch[2], fin->branch[3], fin->sink[0], fin->sink[1], fin->sink[2],
                    fin->sink[3]);
    }
    if (!st.done) return fail(RQK_ERR_INTERNAL, "rqk_auction: did not terminate%s");
    if ((rc = rqk_auction_finalize(n, ld, k, workspace, workspace_bytes, assign, stream_))) return rc;
    if (info) *info = st;
    return 0;
}

}  // extern "C"
