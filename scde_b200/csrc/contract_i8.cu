// contract_i8.cu -- the bootstrap joint posterior (src/jpmatLogBoot.cpp:216-275, :460-499) on the 5th-generation tensor
// cores: tcgen05.mma.kind::i8 with 32-bit integer accumulators in tensor memory.
//
// Per gene the reference computes  T[b, k] = sum_c W[c, b] * lp[c, x[g, c], k]  (W = how often boot b drew cell c) and
// then jp[g, :] = (1/B) sum_b softmax_k T[b, :].  boot_contract.cu evaluates that sum on the FP64 pipe (DMMA), where it
// is bound by the 37 TFLOP/s FP64 rate.  Here the table is held in FIXED POINT instead: in the zero-base form every
// table value D = lp(x) - lp(0) (or lp(x) itself) lies in [-751, 751] -- log of a normalised double -- or is the
// reference's "log 0" sentinel (-DBL_MAX/n/1.1, :127,204).  D is rounded to a multiple of 2^-29 and split into five
// signed radix-256 digits (int8 planes 0..4, value = 2^-29 * sum_p 256^p d_p).  W is a small non-negative integer
// (<= 127 is checked).  Every product and every sum is then EXACT in int32 (|sum| <= 128 * draws), the planes are
// recombined in int64 and converted to FP64 once per (boot, grid point), so the only error is the table rounding:
// |T error| <= draws * 2^-30 in the worst case and about sqrt(2 * draws) * 2^-29 / sqrt(12) typically (5e-8 at 5000
// cells per group) -- inside the 1e-6 tolerance on log-posteriors, and independent of the summation order, so the
// result is deterministic by construction.
//
// The sentinel is not summed at all.  A grid point of (gene, boot) is "log 0" exactly when some drawn row is "log 0"
// there; the non-sentinel points of a row form one interval [klo, khi] (common.cuh), so it is enough to intersect the
// intervals of the drawn rows: sentinel_range_kernel does that per (gene, boot) with packed 16-bit max / min, and the
// epilogue writes the sentinel outside the intersection.  (gene, boot) pairs with an EMPTY intersection -- where the
// reference's soft-max would compare multiples of the sentinel -- and irregular rows raise flag 4: the caller reruns on
// the FP64 kernel, which adds the sentinels as the reference does.
//
// Kernel: persistent, one CTA per SM, three warp roles, no CTA-wide barrier in the steady state (the pipeline skeleton
// below, which bound_i8_kernel shares).
//   * work item = (gene, piece): one 512-byte piece of the gene's table rows = 102 grid points x 5 planes.  The item
//     accumulates D[boot (128 lanes, 104 real)][plane * 102 + i] in all 512 tensor-memory columns of the SM.
//   * producers (4 warps): gather the list entries' pieces (512 contiguous, 512-byte-aligned bytes per entry) and W rows
//     (128 bytes) with 16-byte cp.async straight into the canonical 128-byte-swizzle layout of an MN-major operand;
//     completion is signalled by cp.async.mbarrier.arrive; a 10-stage ring of 32 entries (20 KB per stage) keeps up to
//     200 KB in flight per SM.  The loop is branch-free per stage: constant offsets, slot / phase counters instead of
//     divisions, list entries fetched 8-16 stages ahead.
//   * MMA (1 thread): per stage two tcgen05.mma (M = 128 boots, N = 256, K = 32 entries), then tcgen05.commit onto the
//     stage's "empty" barrier; after the last stage a commit onto the accumulator barrier.
//   * epilogue (8 warps, two per 32-lane quarter of tensor memory): tcgen05.ld the five planes of 8 grid points at a
//     time, recombine into one 64-bit integer per (boot, grid point) and store it; softmax_i8_warp_kernel finishes the gene
//     (conversion, zero-count base Z[b, k], sentinel ranges, soft-max, average).  Producers keep prefetching the next
//     item meanwhile.
// Roofline: HBM gather bandwidth (512 bytes per visited (gene, cell) pair and piece; tools/gather_bench.cu measures
// 6.8 TB/s for this access pattern with 128 KB in flight per SM); the tensor pipe needs 2 x 128 cycles per 32 entries.
#include "common.cuh"
#include "ptx_sm100.cuh"
#include "fastmath.cuh"
#include <cfloat>
#include <cmath>
#include <cstdlib>

namespace scde {
namespace {

using namespace ptx;

constexpr int Q_ES = 32;                         // list entries per stage = K of one tcgen05.mma.kind::i8
constexpr int Q_NS = 10;                         // ring depth (largest; the kernel takes the depth as a template parameter)
constexpr int Q_A_BYTES = Q_ES * Q_WB;           // W tile of a stage: 4096
constexpr int Q_B_BYTES = Q_ES * Q_PIECE;        // table tile of a stage: 16384
constexpr int Q_STAGE_BYTES = Q_A_BYTES + Q_B_BYTES;  // 20480, a multiple of the 1024-byte swizzle atom
// Warp roles of both tcgen05 kernels: the producer warps, the epilogue warps, then the MMA warp, which also allocates the
// tensor memory.  ONE producer group: every producer warp touches every stage, so the ring itself bounds the producers'
// lead.  (Two groups taking alternate stages were no faster and deadlocked: a group with no stage of its own in a run of
// short items ran ahead until a parity wait on "empty" was satisfied by a phase two uses back -- DESIGN.md 4.3.)
// Eight epilogue warps: a warp may only read the tensor-memory lanes 32 (warp id mod 4) .. + 31, so two warps share each
// quarter.  (With four warps the contraction's epilogue of an item took longer than the ring can cover, and the tensor
// memory is not free for the next item before it ends.)
constexpr int Q_PRODUCER_WARPS = 4;              // one per 8-entry k-group of a stage
constexpr int Q_EPILOGUE_WARPS = 8;
constexpr int Q_MMA_WARP = Q_PRODUCER_WARPS + Q_EPILOGUE_WARPS;
constexpr int Q_THREADS = (Q_MMA_WARP + 1) * 32;
constexpr int Q_EPI_ROUNDS = (Q_PW + 7) / 8;  // rounds of 8 grid points per piece
constexpr int Q_TMEM_COLS = 512;
constexpr long long Q_WATCHDOG_CYCLES = 4000000000ll;  // a barrier wait longer than ~2 s aborts the kernel (err = 2)
static_assert(Q_NV * Q_PW <= Q_TMEM_COLS && Q_NV * Q_PW <= Q_PIECE, "a piece is one pass of tensor memory");
static_assert((Q_PW & 1) == 0, "the epilogue reads pairs of columns");

// The gene lists of a launch and the draw set of every gene, as both tcgen05 kernels read them
struct ListParams {
    const int32_t *row, *cell, *len, *order;  // GeneLists, order from the launch's first gene
    int64_t ld;
    const int32_t *gene_set;  // draw set of every gene (NULL: one set): its W rows start gene_set[gene] * set_w8 bytes
    int64_t set_w8;           // after each side's W8
};

// ---- the pipeline skeleton of both tcgen05 kernels --------------------------------------------------------------------
// The producer warps gather the Q_ES list entries of a stage into a ring slot with cp.async and arrive on the slot's
// "full" barrier.  The MMA thread waits on "full", issues the stage's MMAs into the item's accumulator buffer and commits
// onto the slot's "empty" barrier; after the item's last stage it commits onto the buffer's "full" barrier (or arrives on
// it: an empty list), and the epilogue warps read the buffer and arrive on its "empty" barrier.  Waiting for the n-th
// completion (n >= 1) of a barrier is a wait on parity (n - 1) & 1.
template <int NSB, int NACC>  // NSB >= the ring depth
struct PipeBars {
    uint64_t full[NSB], empty[NSB];
    uint64_t acc_full[NACC], acc_empty[NACC];
    uint32_t tmem_base;
    volatile int abort;
    __device__ __forceinline__ void init(int ns) {  // thread 0, before the init fence
        for (int s = 0; s < ns; ++s) {
            mbar_init(&full[s], Q_PRODUCER_WARPS * 32);  // one cp.async completion arrival per producer thread
            mbar_init(&empty[s], 1);                     // one tcgen05.commit
        }
        for (int b = 0; b < NACC; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], Q_EPILOGUE_WARPS * 32);
        }
        abort = 0;
    }
};

// the producer and MMA roles wait spinning; false when the kernel aborts
__device__ __forceinline__ bool wait_spin(volatile int &abort, uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return true;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (abort) return false;
        if (clock64() - t0 > Q_WATCHDOG_CYCLES) {  // never in a correct run: leave instead of hanging the GPU
            abort = 1;
            return false;
        }
    }
    return true;
}
// the epilogues' wait: an item takes microseconds, so sleep between polls; false when the kernel aborts
template <int SLEEP_NS>
__device__ __forceinline__ bool wait_sleep(volatile int &abort, uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(SLEEP_NS);
        if (abort) return false;
    }
    return true;
}

// A role's position in the ring of NS stages of STAGE bytes: the slot, and how often it has been filled before.  The
// producers' and the MMA thread's cursors run across items and visit the same slots in the same order.
template <int NS, int STAGE>
struct Ring {
    uint32_t stage0;
    int slot = 0;
    uint32_t fill = 0;
    __device__ __forceinline__ uint32_t stage() const { return stage0 + (uint32_t)slot * STAGE; }
    __device__ __forceinline__ void advance() {
        if (++slot == NS) {
            slot = 0;
            ++fill;
        }
    }
};

// The CTA's items blockIdx.x, + gridDim.x, .. < n_items.  gene_of(item) = the item's gene; its list length and (W_SET)
// the byte offset of its draw set's W rows are loaded one item ahead.  body(item, gene, stages, wset) returns false to
// stop (abort).
template <bool W_SET, class GeneOf, class Body>
__device__ __forceinline__ void walk_items(const ListParams &l, int n_items, GeneOf gene_of, Body body) {
    int64_t gene_n = 0, wset_n = 0;
    int len_n = 0;
    auto fetch = [&](int item) {
        gene_n = gene_of(item);
        len_n = l.len[gene_n];
        if (W_SET && l.gene_set) wset_n = l.gene_set[gene_n] * l.set_w8;
    };
    int item = blockIdx.x;
    if (item < n_items) fetch(item);
    for (; item < n_items; item += gridDim.x) {
        const int64_t gene = gene_n, wset = wset_n;
        const int nst = (len_n + Q_ES - 1) / Q_ES;
        if (item + (int)gridDim.x < n_items) fetch(item + gridDim.x);
        if (!body(item, gene, nst, wset)) return;
    }
}

template <int DOFF, int SOFF>
__device__ __forceinline__ void cp_async16_at(uint32_t dst_smem, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0+%2], [%1+%3], 16;" ::"r"(dst_smem), "l"(src), "n"(DOFF), "n"(SOFF) : "memory");
}
template <int DOFF, int SOFF>
__device__ __forceinline__ void cp_async16_hint_at(uint32_t dst_smem, const void *src, uint64_t policy) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0+%2], [%1+%3], 16, %4;" ::"r"(dst_smem), "l"(src), "n"(DOFF), "n"(SOFF),
                 "l"(policy)
                 : "memory");
}

// ---- producers: warp kg gathers entries 8 kg .. 8 kg + 7 (one k-group of the MMA) of every stage ----------------------
// Canonical 128-byte-swizzle layout of an MN-major operand: the bytes of one entry are split into runs of 128 (8 pieces
// of 16 bytes); run r of entry kk of k-group kg sits at [r][kg][kk][128 B] and its piece j at 16 * (j ^ kk).  Lane
// (l3 = lane >> 3, l7 = lane & 7) copies piece l7 of every run of entries l3 and l3 + 4: a warp instruction moves four
// 128-byte runs of global memory into four 128-byte lines of shared memory -- coalesced on both sides, no bank conflicts.
//
// List entries: lane (l3, l7) holds entries l3 and l3 + 4 of the warp's stage 8 t + l7 -- one load instruction fetches
// the entries of eight stages, issued one block (8 stages) before its first use, the first two blocks at the start of the
// item; the identity of the NEXT item (gene, list length) is loaded one item ahead.  An earlier version with a shorter
// look-ahead spent 17 % of the producers' cycles waiting on these loads and 55 % issuing ~180 dependent instructions per
// stage (profiles/r01v); this loop issues about 45.
//
// copy(dst0, dst1, row0, row1, cell0, cell1) issues the cp.async of one stage for this lane's entries l3 and l3 + 4 (their
// table rows and raw cell words); dst0 / dst1 = their piece l7 in the stage's first 128-byte-swizzled tile.
template <int NS, int STAGE, int NSB, int NACC, class Copy>
__device__ __forceinline__ bool gather_item(const ListParams &l, PipeBars<NSB, NACC> &b, Ring<NS, STAGE> &ring, int64_t gene,
                                            int nst, int kg, int lane, Copy copy) {
    const int l7 = lane & 7, l3 = lane >> 3;
    // entry kk = l3 (and l3 + 4): line kk of this warp's k-group, piece l7 at 16 * (l7 ^ kk)
    const uint32_t d0 = (uint32_t)kg * 1024u + (uint32_t)l3 * 128u + (uint32_t)((l7 ^ l3) << 4);
    const uint32_t d1 = (uint32_t)kg * 1024u + (uint32_t)(l3 + 4) * 128u + (uint32_t)((l7 ^ (l3 + 4)) << 4);
    const int32_t *lrow = l.row + gene * l.ld + kg * 8 + l3;
    const int32_t *lcell = l.cell + gene * l.ld + kg * 8 + l3;
    int32_t r0a = 0, r1a = 0, c0a = 0, c1a = 0, r0b = 0, r1b = 0, c0b = 0, c1b = 0;
    auto load_block = [&](int t, int32_t &r0, int32_t &r1, int32_t &c0, int32_t &c1) {
        const int s = 8 * t + l7;
        r0 = r1 = c0 = c1 = 0;
        if (s < nst) {
            r0 = __ldg(lrow + s * Q_ES);
            r1 = __ldg(lrow + s * Q_ES + 4);
            c0 = __ldg(lcell + s * Q_ES);
            c1 = __ldg(lcell + s * Q_ES + 4);
        }
    };
    load_block(0, r0a, r1a, c0a, c1a);
    load_block(1, r0b, r1b, c0b, c1b);
    for (int t = 0; 8 * t < nst; ++t) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (8 * t + u < nst) {  // warp-uniform
                const int from = (lane & 24) | u;
                const int32_t row0 = __shfl_sync(0xffffffffu, r0a, from), row1 = __shfl_sync(0xffffffffu, r1a, from);
                const int32_t cel0 = __shfl_sync(0xffffffffu, c0a, from), cel1 = __shfl_sync(0xffffffffu, c1a, from);
                // acquire the slot: the MMAs of its previous fill have read it
                if (ring.fill > 0 && !wait_spin(b.abort, &b.empty[ring.slot], (ring.fill - 1) & 1u)) return false;
                const uint32_t sA = ring.stage();
                copy(sA + d0, sA + d1, row0, row1, cel0, cel1);
                cp_async_mbar_arrive_noinc(&b.full[ring.slot]);
                ring.advance();
            }
        }
        r0a = r0b;
        r1a = r1b;
        c0a = c0b;
        c1a = c1b;
        load_block(t + 2, r0b, r1b, c0b, c1b);
    }
    return true;
}

// The producer role: make_copy(item, wset) returns the copy of one stage of the item (see gather_item)
template <int NS, int STAGE, int NSB, int NACC, class GeneOf, class MakeCopy>
__device__ __forceinline__ void run_producer(const ListParams &l, PipeBars<NSB, NACC> &b, uint32_t stage0, int n_items, int kg,
                                             int lane, GeneOf gene_of, MakeCopy make_copy) {
    Ring<NS, STAGE> ring{stage0};
    walk_items<true>(l, n_items, gene_of, [&](int item, int64_t gene, int nst, int64_t wset) {
        return gather_item(l, b, ring, gene, nst, kg, lane, make_copy(item, wset));
    });
}

// The MMA role (one thread): item n goes to accumulator buffer n mod NACC, of Q_TMEM_COLS / NACC columns.
// issue(stage, acc, accumulate) issues the MMAs of one stage into the buffer at tensor-memory address acc.  dbg (or NULL):
// [2] += cycles spent waiting for the epilogue to release a buffer.
template <int NS, int STAGE, int NSB, int NACC, class GeneOf, class Issue>
__device__ __forceinline__ void run_mma(const ListParams &l, PipeBars<NSB, NACC> &b, uint32_t stage0, uint32_t tmem, int n_items,
                                        GeneOf gene_of, unsigned long long *dbg, Issue issue) {
    Ring<NS, STAGE> ring{stage0};
    uint32_t n_done = 0;
    walk_items<false>(l, n_items, gene_of, [&](int, int64_t, int nst, int64_t) {
        const int buf = (int)(n_done % NACC);
        const uint32_t use = n_done / NACC;
        ++n_done;
        if (use > 0) {  // the epilogue has read this buffer's previous item
            const long long t0 = dbg ? clock64() : 0;
            if (!wait_spin(b.abort, &b.acc_empty[buf], (use - 1) & 1u)) return false;
            tc_fence_after_sync();
            if (dbg) atomicAdd(dbg + 2, (unsigned long long)(clock64() - t0));
        }
        const uint32_t acc = tmem + (uint32_t)(buf * (Q_TMEM_COLS / NACC));
        for (int s = 0; s < nst; ++s) {
            if (!wait_spin(b.abort, &b.full[ring.slot], ring.fill & 1u)) return false;
            fence_proxy_async_smem();
            tc_fence_after_sync();
            issue(ring.stage(), acc, s > 0);
            umma_commit(&b.empty[ring.slot]);  // frees the slot once these MMAs have read it
            ring.advance();
        }
        if (nst > 0)
            umma_commit(&b.acc_full[buf]);
        else
            mbar_arrive(&b.acc_full[buf]);  // an empty list: the sums are 0, nothing to wait for
        return true;
    });
}

// The kernel frame: a ring of NS stages from the first 1024-byte boundary of the dynamic shared memory (the swizzle pattern
// is a function of the shared-memory address bits), the kernel's Smem (whose member `pipe` is its PipeBars) smem_off bytes
// after the ring's start, all 512 tensor-memory columns, and the three roles: producer(sm, stage0, kg, lane) on the
// producer warps, epilogue(sm, stage0, tmem, ewarp, lane) on the epilogue warps (ewarp & 3 = the warp's tensor-memory
// quarter), mma(sm, stage0, tmem) on lane 0 of the MMA warp.  init(sm): thread 0 initialises the kernel's other barriers.
extern __shared__ __align__(1024) unsigned char q_smem_raw[];
template <int NS, class Smem, class Init, class Producer, class Epilogue, class Mma>
__device__ __forceinline__ void run_pipeline(uint32_t smem_off, int32_t *err, Init init, Producer producer, Epilogue epilogue,
                                             Mma mma) {
    const uint32_t raw = smem_u32(q_smem_raw);
    const uint32_t stage0 = (raw + 1023u) & ~1023u;
    Smem &sm = *reinterpret_cast<Smem *>(q_smem_raw + (stage0 - raw) + smem_off);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        sm.pipe.init(NS);
        init(sm);
        mbar_fence_init();
    }
    if (warp == Q_MMA_WARP) tmem_alloc(&sm.pipe.tmem_base, Q_TMEM_COLS);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = sm.pipe.tmem_base;
    if (warp < Q_PRODUCER_WARPS)
        producer(sm, stage0, warp, lane);
    else if (warp < Q_MMA_WARP)
        epilogue(sm, stage0, tmem, warp - Q_PRODUCER_WARPS, lane);
    else if (lane == 0)
        mma(sm, stage0, tmem);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    if (sm.pipe.abort && err && threadIdx.x == 0) atomicExch(err, 2);
    if (warp == Q_MMA_WARP) tmem_dealloc(tmem, Q_TMEM_COLS);
}

// ---- contract_i8_kernel -------------------------------------------------------------------------------------------------
struct I8Smem {
    PipeBars<Q_NS, 1> pipe;
};
constexpr int Q_XBUF_BYTES = Q_EPILOGUE_WARPS * 2048;  // per epilogue warp: one [32 boots][8 grid points] tile of 64-bit sums
constexpr size_t q_smem_bytes(int ns) { return 1024 /* alignment slack */ + (size_t)ns * Q_STAGE_BYTES + Q_XBUF_BYTES + sizeof(I8Smem); }

struct I8Params {
    ListParams lists;
    const int8_t *qtable;  // [rows][ldq]: row = [piece][plane][102] (+ 2)
    int64_t ldq;
    const int8_t *W8[2];   // side s: its pass's W rows [n_w_rows][128] (of the first draw set); [1]: twin launches only
    long long *T[2];       // side s: [n_pos][104][416]: 2^29 * T[boot, grid] as exact integers (without Z, without sentinels)
    int n_boot;            // real boots of side 0's pass: rows beyond are not stored
    int n_pos;             // genes in this launch: positions [0, n_pos) of `order`
    int n_pieces;          // pieces per gene
    int32_t *err;          // device flag: 2 = watchdog abort
    unsigned long long *dbg;  // optional diagnostics: [0] += cycles between "accumulators ready" and "tensor memory released",
                              // [1] += items, [2] += cycles the MMA thread waited for the release (epilogue warp 0 / MMA thread)
    int twin;            // 1: two sides, items come in pairs (2 i, 2 i + 1) = the same (gene, piece) for side 0 and side 1, so
                         // that two neighbouring CTAs gather the same table rows at the same time and the second read is an L2 hit
    int piece_major;     // item order: 0 = (gene, piece) with the piece fastest, 1 = (piece, gene) with the gene fastest
    int cold_evict_first;  // HINT kernels: rows without the hot bit are loaded evict_first (else without a hint)
    const int32_t *items;  // pruned launch: the codes (item numbers of the order above) of the live items, *n_live of
    const int32_t *n_live; // them, written on the device by prune_compact_kernel; NULL = every item
};

// item -> (gene position, piece).  Gene-major order: the pieces of one gene go to neighbouring CTAs of the same round, so
// the W rows and list entries they share are L2 hits for three of the four.  Piece-major order: all CTAs work on the same
// 512-byte piece of the table rows at the same time -- four times as many genes in flight per piece, and a quarter of
// the table as the working set of a phase, so the rows of small counts (shared by thousands of genes) are L2 hits more
// often; the lists and W rows are re-read once per phase (8 + 128 B per entry against the piece's 512 B).
struct Item {
    int pos, piece;
};
__device__ __forceinline__ int item_code(const I8Params &p, int item) {
    item >>= p.twin;  // twin launch: bit 0 of the item selects the side
    return p.items ? __ldg(p.items + item) : item;
}
__device__ __forceinline__ Item decode_item(const I8Params &p, int item) {
    Item it;
    item = item_code(p, item);
    if (p.piece_major) {
        it.piece = item / p.n_pos;
        it.pos = item - it.piece * p.n_pos;
    } else {
        it.pos = item / p.n_pieces;
        it.piece = item - it.pos * p.n_pieces;
    }
    return it;
}
__device__ __forceinline__ int64_t item_gene(const I8Params &p, int item) {
    item = item_code(p, item);
    const int pos = p.piece_major ? item % p.n_pos : item / p.n_pieces;
    return p.lists.order ? p.lists.order[pos] : pos;
}

// A stage: the W tile (Q_A_BYTES), then the table tile of the item's piece, four 128-byte runs per entry.
// HINT: list entries carry LIST_HOT_BIT in `cell` when the row is one of the first few of its cell (a small count: such a
// row is shared by thousands of genes); its pieces are loaded with the L2 evict_last policy, the others evict_first (or
// unhinted), so that the stream of rows that are used once does not push the shared ones out of the L2.
template <bool HINT, int NS>
__device__ __forceinline__ void contract_producer(const I8Params &p, I8Smem &sm, uint32_t stage0, int n_items, int kg, int lane) {
    uint64_t pol_hot = 0, pol_cold = 0;
    if (HINT) {
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_hot));
        if (p.cold_evict_first)
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_cold));
        else
            asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol_cold));
    }
    const int l7 = lane & 7;
    run_producer<NS, Q_STAGE_BYTES>(
        p.lists, sm.pipe, stage0, n_items, kg, lane, [&](int item) { return item_gene(p, item); },
        [&](int item, int64_t wset) {
            const int8_t *qbase = p.qtable + (int64_t)decode_item(p, item).piece * Q_PIECE + l7 * 16;
            const int8_t *wbase = ((p.twin && (item & 1)) ? p.W8[1] : p.W8[0]) + l7 * 16 + wset;
            return [=, &p](uint32_t dst0, uint32_t dst1, int32_t row0, int32_t row1, int32_t cel0, int32_t cel1) {
                const int8_t *src0 = qbase + (int64_t)row0 * p.ldq;
                const int8_t *src1 = qbase + (int64_t)row1 * p.ldq;
                const int8_t *w0 = wbase + (int64_t)(cel0 & ~LIST_HOT_BIT) * Q_WB;
                const int8_t *w1 = wbase + (int64_t)(cel1 & ~LIST_HOT_BIT) * Q_WB;
                if (HINT) {
                    const uint64_t pol0 = (cel0 & LIST_HOT_BIT) ? pol_hot : pol_cold;
                    const uint64_t pol1 = (cel1 & LIST_HOT_BIT) ? pol_hot : pol_cold;
                    cp_async16_hint_at<Q_A_BYTES, 0>(dst0, src0, pol0);
                    cp_async16_hint_at<Q_A_BYTES, 0>(dst1, src1, pol1);
                    cp_async16_hint_at<Q_A_BYTES + 4096, 128>(dst0, src0, pol0);
                    cp_async16_hint_at<Q_A_BYTES + 4096, 128>(dst1, src1, pol1);
                    cp_async16_hint_at<Q_A_BYTES + 8192, 256>(dst0, src0, pol0);
                    cp_async16_hint_at<Q_A_BYTES + 8192, 256>(dst1, src1, pol1);
                    cp_async16_hint_at<Q_A_BYTES + 12288, 384>(dst0, src0, pol0);
                    cp_async16_hint_at<Q_A_BYTES + 12288, 384>(dst1, src1, pol1);
                    cp_async16_hint_at<0, 0>(dst0, w0, pol_hot);
                    cp_async16_hint_at<0, 0>(dst1, w1, pol_hot);
                } else {
                    cp_async16_at<Q_A_BYTES, 0>(dst0, src0);
                    cp_async16_at<Q_A_BYTES, 0>(dst1, src1);
                    cp_async16_at<Q_A_BYTES + 4096, 128>(dst0, src0);
                    cp_async16_at<Q_A_BYTES + 4096, 128>(dst1, src1);
                    cp_async16_at<Q_A_BYTES + 8192, 256>(dst0, src0);
                    cp_async16_at<Q_A_BYTES + 8192, 256>(dst1, src1);
                    cp_async16_at<Q_A_BYTES + 12288, 384>(dst0, src0);
                    cp_async16_at<Q_A_BYTES + 12288, 384>(dst1, src1);
                    cp_async16_at<0, 0>(dst0, w0);
                    cp_async16_at<0, 0>(dst1, w1);
                }
            };
        });
}

// ---- epilogue: warps e = 0..7; warp e reads tensor-memory lanes 32 (e & 3) .. + 31 and the rounds of half e >> 2 --------
// The tensor memory is not free for the next item's MMAs before the epilogue ends (all 512 columns belong to one item), so
// the epilogue does the minimum: tcgen05.ld 8 grid points x 5 planes, recombine the plane sums into ONE 64-bit integer
// per (boot, grid point) and store it with streaming stores -- no loads, no floating point.  |sum_p| <= 128 * draws < 2^23
// (draws <= 65000 is checked by the launcher), so a = s0 + 256 s1 and b = s2 + 256 s3 fit 32 bits and the value is
// a + 2^16 b + 2^32 s4.  Conversion to FP64, the zero-count base Z and the sentinel ranges are applied by
// softmax_i8_warp_kernel when it reads T.  (An epilogue that did all of that took 16 800 cycles per item -- 8.9 us, of which
// the ring hides 3 -- and cost a quarter of the kernel: SCDE_B200_EPI_TIMING, profiles/r01x.)
__device__ __forceinline__ void contract_epilogue(const I8Params &p, I8Smem &sm, uint32_t xbuf, uint32_t tmem, int n_items,
                                                  int ewarp, int lane) {
    const int qd = ewarp & 3, half = ewarp >> 2;
    const uint32_t tlane = tmem + ((uint32_t)(qd * 32) << 16);
    // A thread holds 8 grid points of ONE boot (64 bytes of a T row; rows are 3328 bytes apart): stored directly, a warp
    // store touches 32 lines.  The round's [32 boots][8 points] tile is turned through shared memory instead, so that a
    // store instruction writes the complete 64-byte runs of 8 boots (8 lines, every sector full).  Tile layout: 16-byte
    // chunk j of boot l at unit (l + 8 j) mod 32 of row j -- conflict-free both ways.
    const uint32_t xw = xbuf + (uint32_t)ewarp * 2048u;
    const int rb = lane >> 2, rc = lane & 3;  // read side: boot rb + 8 i of the warp, chunk rc
    const int r_begin = half ? (Q_EPI_ROUNDS + 1) / 2 : 0, r_end = half ? Q_EPI_ROUNDS : (Q_EPI_ROUNDS + 1) / 2;
    uint32_t n_done = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n_done) {
        const Item it = decode_item(p, item);
        const int64_t gene = p.lists.order ? p.lists.order[it.pos] : it.pos;
        const bool empty_list = p.lists.len[gene] <= 0;
        if (!wait_sleep<200>(sm.pipe.abort, &sm.pipe.acc_full[0], n_done & 1u)) return;
        tc_fence_after_sync();
        const long long t_ready = p.dbg ? clock64() : 0;
        long long *Tbase = ((p.twin && (item & 1)) ? p.T[1] : p.T[0]) + ((int64_t)it.pos * WP_TILED + qd * 32) * KP_TILED + it.piece * Q_PW;
        for (int rd = r_begin; rd < r_end; ++rd) {
            const int i0 = rd * 8;
            const int n = Q_PW - i0 < 8 ? Q_PW - i0 : 8;  // 8, or 6 in the last round
            uint32_t r[Q_NV][8];
#pragma unroll
            for (int pl = 0; pl < Q_NV; ++pl)
#pragma unroll
                for (int j = 0; j < 8; ++j) r[pl][j] = 0u;
            if (!empty_list) {
                // eight columns per load (the columns past a plane's 102 points belong to the next plane or are the
                // piece's two spare columns: read, not used)
#pragma unroll
                for (int pl = 0; pl < Q_NV; ++pl) tmem_ld_32x32b_x8(tlane + (uint32_t)(pl * Q_PW + i0), r[pl]);
                tmem_wait_ld();
            }
            long long out[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int32_t a = (int32_t)r[0][j] + ((int32_t)r[1][j] << 8);
                const int32_t c = (int32_t)r[2][j] + ((int32_t)r[3][j] << 8);
                out[j] = (long long)a + ((long long)c << 16) + ((long long)(int32_t)r[4][j] << 32);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(xw + 512u * j + (uint32_t)(((lane + 8 * j) & 31) << 4)),
                             "l"(out[2 * j]), "l"(out[2 * j + 1])
                             : "memory");
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int bw = rb + 8 * i;  // boot within the warp's 32
                long long v0, v1;
                asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(v0), "=l"(v1)
                             : "r"(xw + 512u * rc + (uint32_t)(((bw + 8 * rc) & 31) << 4)) : "memory");
                // streaming stores: T is read back once, by the soft-max kernel, long after it has left the L2 -- it
                // should not push table rows out (an evict-first hint on the table loads, on the other hand, cost
                // 4 %: the rows of small counts are shared by thousands of genes and live in the L2)
                if (qd * 32 + bw < p.n_boot && 2 * rc < n)
                    __stcs(reinterpret_cast<longlong2 *>(Tbase + (int64_t)bw * KP_TILED + i0 + 2 * rc), make_longlong2(v0, v1));
            }
            __syncwarp();
        }
        tc_fence_before_sync();
        mbar_arrive(&sm.pipe.acc_empty[0]);
        if (p.dbg && ewarp == 0 && lane == 0) {
            atomicAdd(p.dbg, (unsigned long long)(clock64() - t_ready));
            atomicAdd(p.dbg + 1, 1ull);
        }
    }
}

template <bool HINT, int NS>
__global__ void __launch_bounds__(Q_THREADS, 1) contract_i8_kernel(const I8Params p) {
    static_assert(NS >= 2 && NS <= Q_NS, "ring depth");
    const int n_items = (p.items ? *p.n_live : p.n_pos * p.n_pieces) << p.twin;
    run_pipeline<NS, I8Smem>(
        NS * Q_STAGE_BYTES + Q_XBUF_BYTES, p.err, [](I8Smem &) {},
        [&](I8Smem &sm, uint32_t stage0, int kg, int lane) { contract_producer<HINT, NS>(p, sm, stage0, n_items, kg, lane); },
        [&](I8Smem &sm, uint32_t stage0, uint32_t tmem, int ewarp, int lane) {
            contract_epilogue(p, sm, stage0 + NS * Q_STAGE_BYTES, tmem, n_items, ewarp, lane);
        },
        [&](I8Smem &sm, uint32_t stage0, uint32_t tmem) {
            const uint32_t idesc = umma_idesc_s8_mn(128, 256);
            run_mma<NS, Q_STAGE_BYTES>(p.lists, sm.pipe, stage0, tmem, n_items, [&](int item) { return item_gene(p, item); }, p.dbg,
                                       [&](uint32_t sA, uint32_t acc, bool accumulate) {
                                           const uint32_t sB = sA + Q_A_BYTES;
                                           const uint64_t da = umma_desc_sw128(sA, 4096u, 1024u);
                                           umma_s8(acc, da, umma_desc_sw128(sB, 4096u, 1024u), idesc, accumulate);  // runs 0, 1
                                           umma_s8(acc + 256u, da, umma_desc_sw128(sB + 2u * 4096u, 4096u, 1024u), idesc,
                                                   accumulate);  // runs 2, 3
                                       });
        });
}

// ------------------------------------------------------------------------------------------------
// Sentinel range of every (gene, boot): [max klo, min khi] over the list entries the boot drew.  One warp per gene, lane l
// owns boots 4 l .. 4 l + 3 (one 32-bit word of the entry's W row); klo / khi are kept as packed 16-bit pairs and
// combined with __vmaxu2 / __vminu2 under a mask made of the non-zero multiplicities.  Entries whose row has no sentinel
// (the common case) are skipped after one uniform load.  flag |= 4 when a drawn row is irregular or an intersection is
// empty.
__global__ void __launch_bounds__(256) sentinel_range_kernel(const int32_t *__restrict__ lst_row, const int32_t *__restrict__ lst_cell,
                                                             const int32_t *__restrict__ lst_len, const int32_t *__restrict__ order,
                                                             int64_t ld_lst, const uint32_t *__restrict__ row_range,
                                                             const int8_t *__restrict__ W8, const int32_t *__restrict__ gene_set,
                                                             int64_t set_w8, int n_pos, int K, int n_boot,
                                                             uint32_t *__restrict__ SR, int32_t *__restrict__ flag) {
    const int pos = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pos >= n_pos) return;
    const int lane = threadIdx.x & 31;
    const int64_t gene = order ? order[pos] : pos;
    if (gene_set) W8 += gene_set[gene] * set_w8;  // the W rows of the gene's draw set
    const int len = lst_len[gene];
    const int32_t *lr = lst_row + gene * ld_lst, *lc = lst_cell + gene * ld_lst;
    const uint32_t full = (uint32_t)(K - 1) << 16;
    uint32_t lo01 = 0u, lo23 = 0u, hi01 = 0xFFFFFFFFu, hi23 = 0xFFFFFFFFu;
    const uint32_t v01 = (4 * lane < n_boot ? 0xFFFFu : 0u) | (4 * lane + 1 < n_boot ? 0xFFFF0000u : 0u);
    const uint32_t v23 = (4 * lane + 2 < n_boot ? 0xFFFFu : 0u) | (4 * lane + 3 < n_boot ? 0xFFFF0000u : 0u);
    bool irregular = false;
    // the (row -> range) lookups of the next 32 entries are in flight while the current ones are combined
    auto fetch = [&](int e0, uint32_t &rr, int32_t &cell) {
        const int e = e0 + lane;
        rr = full;
        cell = 0;
        if (e < len) {
            rr = __ldg(row_range + lr[e]);
            cell = lc[e] & ~LIST_HOT_BIT;
        }
    };
    uint32_t rr_n = full;
    int32_t cell_n = 0;
    if (len > 0) fetch(0, rr_n, cell_n);
    for (int e0 = 0; e0 < len; e0 += 32) {
        const uint32_t rr = rr_n;
        const int32_t cell = cell_n;
        if (e0 + 32 < len) fetch(e0 + 32, rr_n, cell_n);
        // An entry whose klo is not above the smallest lower bound any boot holds so far, and whose khi is not below the
        // largest upper bound, cannot change any boot's range whatever its multiplicities are: it is skipped without
        // touching its W row.  The bounds tighten within the first few dozen entries (every boot draws 63 % of the
        // cells), after which almost every entry is skipped.  (Boots beyond n_boot hold no bounds: masked out.)
        const uint32_t lmin2 = __vminu2(lo01 | ~v01, lo23 | ~v23), hmax2 = __vmaxu2(hi01 & v01, hi23 & v23);
        const uint32_t gmin = __reduce_min_sync(0xffffffffu, min(lmin2 & 0xFFFFu, lmin2 >> 16));
        const uint32_t gmax = __reduce_max_sync(0xffffffffu, max(hmax2 & 0xFFFFu, hmax2 >> 16));
        unsigned need = __ballot_sync(0xffffffffu, rr != full && (rr == Q_RANGE_IRREGULAR || (rr & 0xFFFFu) > gmin ||
                                                                  (rr >> 16) < gmax));
        while (need) {  // four entries per round: their W words are loaded before any is used (the loop is latency-bound)
            uint32_t r[4], w[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                r[u] = full;
                w[u] = 0u;
                if (need) {
                    const int src = __ffs(need) - 1;
                    need &= need - 1;
                    r[u] = __shfl_sync(0xffffffffu, rr, src);
                    const int32_t c = __shfl_sync(0xffffffffu, cell, src);
                    w[u] = __ldg(reinterpret_cast<const uint32_t *>(W8 + (int64_t)c * Q_WB + 4 * lane));
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (r[u] == Q_RANGE_IRREGULAR) {
                    irregular = true;
                    continue;
                }
                const uint32_t m = __vcmpne4(w[u], 0u);  // 0xFF per boot that drew this cell
                const uint32_t m01 = __byte_perm(m, 0u, 0x1100), m23 = __byte_perm(m, 0u, 0x3322);
                const uint32_t klo2 = (r[u] & 0xFFFFu) * 0x10001u, khi2 = (r[u] >> 16) * 0x10001u;
                lo01 = __vmaxu2(lo01, klo2 & m01);
                lo23 = __vmaxu2(lo23, klo2 & m23);
                hi01 = __vminu2(hi01, khi2 | ~m01);
                hi23 = __vminu2(hi23, khi2 | ~m23);
            }
        }
    }
    uint32_t out[4];
    bool bad = irregular;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t lo = ((j < 2 ? lo01 : lo23) >> (16 * (j & 1))) & 0xFFFFu;
        uint32_t hi = ((j < 2 ? hi01 : hi23) >> (16 * (j & 1))) & 0xFFFFu;
        if (hi > (uint32_t)(K - 1)) hi = (uint32_t)(K - 1);
        if (4 * lane + j < n_boot && lo > hi) bad = true;
        // points beyond khi: only real grid points matter, padding columns are never read by the soft-max
        out[j] = lo | (hi == (uint32_t)(K - 1) ? 0xFFFF0000u : hi << 16);
    }
    *reinterpret_cast<uint4 *>(SR + (int64_t)pos * Q_WB + 4 * lane) = make_uint4(out[0], out[1], out[2], out[3]);
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flag, 4);
}

// ------------------------------------------------------------------------------------------------
// softmax_i8_warp_kernel + softmax_i8_reduce_kernel: jp[gene, k] (+)= sum_b softmax_k(T[b, :])[k] / scale from the integer
// T tiles of contract_i8_kernel (src/jpmatLogBoot.cpp:264-269).  T[b, k] = 2^-29 * integer + Z[b, k], "log 0" (excluded
// from the soft-max) outside the (gene, boot) sentinel range.  A CTA owns one group of 13 boots; the eight groups' partial
// sums are added in group order by the reduce kernel: the result is deterministic.
constexpr int SP_GROUPS = 8, SP_ROWS = WP_TILED / SP_GROUPS;
static_assert(SP_GROUPS * SP_ROWS == WP_TILED && SP_ROWS * 32 == KP_TILED, "13 warps x 32 lanes = the 416 grid slots");
// softmax_i8_warp_kernel: a warp per gene.  A CTA owns one group of 13 boots, whose Z rows it keeps in shared memory
// (43 KB); each of its warps walks genes on its own and, for a gene, the 13 boots in ascending order: T row (the next
// boot's row is already in flight), soft-max pieces by shuffles (exp_nonpos, skipped warp-wide where a 32-point stretch
// lies > 746 nats below the row maximum: a joint posterior is sharply peaked), and the normalised row is added to 13
// accumulators per lane in ascending boot order.
// SETS (several draw sets, DESIGN.md "Draw sets"): each gene reads the Z rows of its own set, gene_set[gene] * set_z doubles
// after Z, from global memory (L2) instead of shared memory -- the same values in the same order, so the same result.
// live (pruned launches, else NULL): bit p of live[pos] = piece p of the gene was contracted.  The points of the other
// pieces are neither loaded (their T tiles were not written) nor candidates: bound_i8_kernel proved them more than
// 746 nats below the row maximum for every boot, where exp_nonpos is exactly 0 -- m, sum, amask and acc are unchanged.
constexpr int SW_WARPS = 8;
// LIVE: the instance of pruned launches (live != NULL); the other one is the kernel as it was before pruning.
template <bool SETS, bool LIVE>
__global__ void __launch_bounds__(SW_WARPS * 32, 2)
softmax_i8_warp_kernel(const long long *__restrict__ T, const double *__restrict__ Z, const uint32_t *__restrict__ SR, int K,
                       int n_boot_pass, double scale, double *__restrict__ part, int n_pos, const int32_t *__restrict__ order,
                       const int32_t *__restrict__ gene_set, int64_t set_z, const uint8_t *__restrict__ live) {
    constexpr int NJ = KP_TILED / 32;
    extern __shared__ double s_z[];  // [SP_ROWS][KP_TILED] (one set only)
    const int group = blockIdx.x % SP_GROUPS, batch = blockIdx.x / SP_GROUPS, n_batch = gridDim.x / SP_GROUPS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b0 = group * SP_ROWS;
    const int nb = min(SP_ROWS, n_boot_pass - b0);  // boots of this group (<= 0: none)
    if (!SETS) {
        for (int i = threadIdx.x; i < SP_ROWS * KP_TILED; i += SW_WARPS * 32)
            s_z[i] = (Z && i / KP_TILED < nb) ? Z[(int64_t)b0 * KP_TILED + i] : 0.0;
        __syncthreads();
    }
    const double q = 1.0 / (double)(1ll << Q_FRAC);
    for (int pos = batch * SW_WARPS + warp; pos < n_pos; pos += n_batch * SW_WARPS) {
        double acc[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[j] = 0.0;
        const long long *rows = T + ((int64_t)pos * WP_TILED + b0) * KP_TILED + lane;
        // the group's 13 range words, one per lane
        const uint32_t sr_l = (SR && lane < SP_ROWS) ? SR[(int64_t)pos * Q_WB + b0 + lane] : 0xFFFF0000u;
        const double *zg = s_z;
        if (SETS) zg = Z + gene_set[order ? order[pos] : pos] * set_z + (int64_t)b0 * KP_TILED;
        uint32_t lm = (1u << NJ) - 1u;  // bit j: stretch j of this lane lies in a contracted piece
        if (LIVE) {
            const uint32_t pm = live[pos];
            lm = 0u;
#pragma unroll
            for (int j = 0; j < NJ; ++j) lm |= ((pm >> ((lane + 32 * j) / Q_PW)) & 1u) << j;
        }
        long long nxt[NJ];
        if (nb > 0) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) nxt[j] = (lm >> j) & 1u ? __ldcs(rows + 32 * j) : 0ll;
        }
        for (int bi = 0; bi < nb; ++bi) {
            long long cur[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) cur[j] = nxt[j];
            if (bi + 1 < nb) {
                const long long *r2 = rows + (int64_t)(bi + 1) * KP_TILED;
#pragma unroll
                for (int j = 0; j < NJ; ++j) nxt[j] = (lm >> j) & 1u ? __ldcs(r2 + 32 * j) : 0ll;
            }
            const uint32_t sr = __shfl_sync(0xffffffffu, sr_l, bi);
            const int klo = (int)(sr & 0xFFFFu), span = min((int)(sr >> 16), K - 1) - klo;  // admissible: klo .. klo + span
            const double *zr = zg + bi * KP_TILED + lane;
            double v[NJ], m = -INFINITY;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int k = lane + 32 * j;
                // some drawn row is "log 0" outside the range: the reference's T is a multiple of the sentinel there
                const double t = fma((double)cur[j], q, zr[32 * j]);
                v[j] = (unsigned)(k - klo) <= (unsigned)span && span >= 0 && ((lm >> j) & 1u) ? t : -INFINITY;
                m = v[j] > m ? v[j] : m;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double mo = __shfl_xor_sync(0xffffffffu, m, o);
                m = mo > m ? mo : m;
            }
            double sum = 0.0;
            uint32_t amask = 0u;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const double d = v[j] - m;
                v[j] = 0.0;
                if (__any_sync(0xffffffffu, d > -746.0)) {
                    v[j] = d > -INFINITY ? exp_nonpos(d) : 0.0;
                    amask |= 1u << j;
                }
                sum += v[j];
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const double inv = 1.0 / (sum * scale);
#pragma unroll
            for (int j = 0; j < NJ; ++j)
                if (amask & (1u << j)) acc[j] = __dadd_rn(acc[j], __dmul_rn(v[j], inv));
        }
        double *dst = part + ((int64_t)group * n_pos + pos) * KP_TILED + lane;
#pragma unroll
        for (int j = 0; j < NJ; ++j) dst[32 * j] = acc[j];
    }
}

__global__ void softmax_i8_reduce_kernel(const double *__restrict__ part, const int32_t *__restrict__ order, int K, int n_pos,
                                         double *__restrict__ jp, int64_t ld_jp, int accumulate) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n_pos * KP_TILED) return;
    const int pos = (int)(idx / KP_TILED), k = (int)(idx - (int64_t)pos * KP_TILED);
    if (k >= K) return;
    double r = 0.0;
#pragma unroll
    for (int g = 0; g < SP_GROUPS; ++g) r += part[((int64_t)g * n_pos + pos) * KP_TILED + k];
    const int64_t gene = order ? order[pos] : pos;
    double *out = jp + gene * ld_jp + k;
    *out = accumulate ? *out + r : r;
}

// the integer T tiles as the FP64 values the reference would hold (tests: scde_b200_probe_contract_i8), in place
__global__ void finalize_t_kernel(long long *__restrict__ T, const uint32_t *__restrict__ SR, double sentinel, int64_t n) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const int k = (int)(idx % KP_TILED);
    const int64_t row = idx / KP_TILED;
    const int b = (int)(row % WP_TILED);
    const int64_t pos = row / WP_TILED;
    const uint32_t sr = SR ? SR[pos * Q_WB + b] : 0xFFFF0000u;
    double t = (double)T[idx] * (1.0 / (double)(1ll << Q_FRAC));
    if (k < (int)(sr & 0xFFFFu) || k > (int)(sr >> 16)) t = sentinel;
    reinterpret_cast<double *>(T)[idx] = t;
}

// ------------------------------------------------------------------------------------------------
// Pruning (DESIGN.md 4.3).  For a (gene, boot) with sentinel range [klo, khi] and S = the bound pass's sums over the drawn
// rows (units of 2^-5 nat, rounded outwards row by row, so exact bounds on the integer T):
//   LB = max over the samples k_c in [klo, khi] of Z(k_c) + S_lb[c] / 32  <=  T(k_c)  <=  the row maximum m,
//   UB_p = max over the blocks meeting [klo, khi] and piece p of max Z over the block + S_ub[u] / 32  >=  every admissible
//          T of piece p.
// Piece p is dead when UB_p < LB - 747 for every real boot: its points lie more than 746 nats below m (one nat covers the
// FP64 rounding of fma(T, 2^-29, Z) and of these sums), where the soft-max adds exactly 0.

// zb[row][slot] (row = (set, pass, boot), the rows of Z): max of Z over UB block `slot`, Z at LB sample slot - Q_UB_N
__global__ void z_bounds_kernel(const double *__restrict__ Z, int64_t n_rows, int K, double *__restrict__ zb) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * Q_BSLOTS) return;
    const int64_t row = idx / Q_BSLOTS;
    const int s = (int)(idx - row * Q_BSLOTS);
    const double *z = Z + row * KP_TILED;
    double v = -INFINITY;
    if (s < Q_UB_N) {
        for (int k = s * Q_UB_PTS; k < (s + 1) * Q_UB_PTS && k < K; ++k) v = fmax(v, Z ? z[k] : 0.0);
    } else if (s < Q_UB_N + Q_LB_N) {
        const int k = Q_LB_STEP * (s - Q_UB_N) + Q_LB_OFF;
        if (k < K) v = Z ? z[k] : 0.0;
    }
    zb[idx] = v;
}

// ---- bound_i8_kernel: the bound sums and the decision in one pass -------------------------------------------------------
// live[pos] = the pieces of gene order[pos] that are not dead for every real boot of the launch's sides.  Persistent, one
// CTA per SM, item = one gene with both sides of a two-sided launch, the contraction's pipeline skeleton in a geometry of
// its own:
//   * producers: a stage is 32 list entries -- each side's 128-byte W rows and, gathered ONCE for both sides, the
//     128-byte bound rows.  B_RING = 192 KB of 8 or 12 KB stages are in flight per SM; the contraction's ring, whose
//     20 KB stages a bound stage filled only 8 KB of, held 80.
//   * MMA (1 thread): per stage and side one tcgen05.mma (M = 128 boots, N = 128 bound columns, K = 32 entries) into the
//     side's accumulator of the gene's buffer.  The 512 tensor-memory columns hold 4 buffers (one side) or 2 (two), so
//     the MMAs of the next genes run while the epilogue reads this one.
//   * epilogue (8 warps): a thread owns one boot (tensor-memory lane) of its warp's quarter.  The warps of half 1 form LB
//     from the sample slots, those of half 0 UB_p from the block slots -- both digits of a slot in one thread -- with the
//     arithmetic of the formulas above; LB reaches the UB thread of its boot through shared memory.  The dead pieces are
//     ANDed over the sides and the warp's boots, and each warp ORs its live pieces into live[pos] (zeroed before the
//     launch).  The sums never leave the SM.
constexpr int B_TILE = Q_ES * Q_WB;  // one operand tile of a stage: 32 entries x 128 bytes = 4096
constexpr int B_RING = 192 * 1024;
template <int SIDES>
struct BoundGeom {
    static constexpr int STAGE = (SIDES + 1) * B_TILE;            // the sides' W tiles, then the bound-row tile
    static constexpr int NS = B_RING / STAGE;                     // 24 or 16 stages
    static constexpr int NACC = Q_TMEM_COLS / (SIDES * Q_BW);     // accumulator buffers: 4 or 2
};
template <int SIDES>
struct BoundSmem {
    PipeBars<BoundGeom<SIDES>::NS, BoundGeom<SIDES>::NACC> pipe;
    uint64_t lb_full, lb_empty;  // the LB exchange: written by half 1, read by half 0
    double lb[SIDES][Q_WB];
};
template <int SIDES>
constexpr size_t bound_smem_bytes() { return 1024 /* alignment slack */ + (size_t)B_RING + sizeof(BoundSmem<SIDES>); }

struct BoundParams {
    ListParams lists;
    const int8_t *qbound;  // the table's bound rows [rows][Q_BW]
    int64_t set_zb;           // doubles of zb per draw set
    const int8_t *W8[2];      // side s: its pass's W rows [n_w_rows][128] (of the first draw set)
    const uint32_t *SR[2];    // side s: sentinel ranges [n_pos][128], or NULL (no row holds a sentinel)
    const double *zb[2];      // side s: its pass's Z extrema [104][Q_BSLOTS] (of the first draw set)
    int n_boot[2];            // side s: real boots
    int n_pos, K, n_pieces;
    uint32_t *live;           // live[pos] (bytes), written as words by atomicOr
    double *lb_out, *ub_out;  // side 0's LB [n_pos][104] and UB [n_pos][104][4] (scde_b200_probe_prune_i8), or NULL
};

__device__ __forceinline__ int64_t bound_gene(const BoundParams &p, int pos) { return p.lists.order ? p.lists.order[pos] : pos; }

// A stage: the sides' W tiles, then the bound-row tile
template <int SIDES>
__device__ __forceinline__ void bound_producer(const BoundParams &p, BoundSmem<SIDES> &sm, uint32_t stage0, int kg, int lane) {
    using G = BoundGeom<SIDES>;
    const int l7 = lane & 7;
    run_producer<G::NS, G::STAGE>(
        p.lists, sm.pipe, stage0, p.n_pos, kg, lane, [&](int pos) { return bound_gene(p, pos); },
        [&](int, int64_t wset) {
            const int8_t *qbase = p.qbound + l7 * 16;
            const int8_t *wb0 = p.W8[0] + wset + l7 * 16;
            const int8_t *wb1 = p.W8[SIDES - 1] + wset + l7 * 16;
            return [=](uint32_t dst0, uint32_t dst1, int32_t row0, int32_t row1, int32_t cel0, int32_t cel1) {
                const int64_t c0 = cel0 & ~LIST_HOT_BIT, c1 = cel1 & ~LIST_HOT_BIT;
                cp_async16_at<SIDES * B_TILE, 0>(dst0, qbase + (int64_t)row0 * Q_BW);
                cp_async16_at<SIDES * B_TILE, 0>(dst1, qbase + (int64_t)row1 * Q_BW);
                cp_async16_at<0, 0>(dst0, wb0 + c0 * Q_WB);
                cp_async16_at<0, 0>(dst1, wb0 + c1 * Q_WB);
                if (SIDES > 1) {
                    cp_async16_at<B_TILE, 0>(dst0, wb1 + c0 * Q_WB);
                    cp_async16_at<B_TILE, 0>(dst1, wb1 + c1 * Q_WB);
                }
            };
        });
}

template <int SIDES>
__device__ __forceinline__ void bound_epilogue(const BoundParams &p, BoundSmem<SIDES> &sm, uint32_t tmem, int ewarp, int lane) {
    using G = BoundGeom<SIDES>;
    const int qd = ewarp & 3, half = ewarp >> 2;
    const int boot = qd * 32 + lane;
    const uint32_t tq = tmem + ((uint32_t)(qd * 32) << 16);
    const uint32_t all = (1u << p.n_pieces) - 1u;
    uint32_t n_done = 0;
    for (int pos = blockIdx.x; pos < p.n_pos; pos += gridDim.x, ++n_done) {
        const int64_t gene = bound_gene(p, pos);
        const bool empty_list = p.lists.len[gene] <= 0;
        const int64_t zoff = p.lists.gene_set ? p.lists.gene_set[gene] * p.set_zb : 0;
        int klo[SIDES], khi[SIDES];
        const double *zr[SIDES];
#pragma unroll
        for (int side = 0; side < SIDES; ++side) {
            const uint32_t sr = p.SR[side] ? p.SR[side][(int64_t)pos * Q_WB + boot] : 0xFFFF0000u;
            klo[side] = (int)(sr & 0xFFFFu);
            khi[side] = min((int)(sr >> 16), p.K - 1);
            zr[side] = p.zb[side] + zoff + (int64_t)(boot < p.n_boot[side] ? boot : 0) * Q_BSLOTS;  // past the boots: not used
        }
        const int buf = (int)(n_done % G::NACC);
        if (!wait_sleep<100>(sm.pipe.abort, &sm.pipe.acc_full[buf], (n_done / G::NACC) & 1u)) return;
        tc_fence_after_sync();
        // slot i of the bound row: digits in columns i and Q_BSLOTS + i, read 8 slots at a time
        auto load8 = [&](int side, int j, uint32_t (&lo)[8], uint32_t (&hi)[8]) {
#pragma unroll
            for (int i = 0; i < 8; ++i) lo[i] = hi[i] = 0u;
            if (!empty_list) {
                const uint32_t col = tq + (uint32_t)(buf * SIDES * Q_BW + side * Q_BW + 8 * j);
                tmem_ld_32x32b_x8(col, lo);
                tmem_ld_32x32b_x8(col + Q_BSLOTS, hi);
                tmem_wait_ld();
            }
        };
        if (half) {  // LB: the sample slots Q_UB_N .. Q_UB_N + Q_LB_N - 1 (chunks 3 .. 7)
            double lb[SIDES];
#pragma unroll
            for (int side = 0; side < SIDES; ++side) {
                lb[side] = -INFINITY;
#pragma unroll
                for (int j = Q_UB_N / 8; j < (Q_UB_N + Q_LB_N + 7) / 8; ++j) {
                    uint32_t lo[8], hi[8];
                    load8(side, j, lo, hi);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int slot = 8 * j + i;
                        if (slot < Q_UB_N || slot >= Q_UB_N + Q_LB_N) continue;
                        const int k = Q_LB_STEP * (slot - Q_UB_N) + Q_LB_OFF;
                        if (k >= klo[side] && k <= khi[side])
                            lb[side] = fmax(lb[side], zr[side][slot] + ((double)(int32_t)lo[i] + 256.0 * (int32_t)hi[i]) * (1.0 / 32.0));
                    }
                }
            }
            tc_fence_before_sync();
            mbar_arrive(&sm.pipe.acc_empty[buf]);
            // half 0 has read the previous LB
            if (n_done > 0 && !wait_sleep<100>(sm.pipe.abort, &sm.lb_empty, (n_done - 1) & 1u)) return;
#pragma unroll
            for (int side = 0; side < SIDES; ++side) sm.lb[side][boot] = lb[side];
            mbar_arrive(&sm.lb_full);
        } else {  // UB: the block slots 0 .. Q_UB_N - 1 (chunks 0 .. 3)
            double ub[SIDES][4];
#pragma unroll
            for (int side = 0; side < SIDES; ++side) {
#pragma unroll
                for (int pc = 0; pc < 4; ++pc) ub[side][pc] = -INFINITY;
#pragma unroll
                for (int j = 0; j < (Q_UB_N + 7) / 8; ++j) {
                    uint32_t lo[8], hi[8];
                    load8(side, j, lo, hi);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int u = 8 * j + i;
                        if (u >= Q_UB_N) continue;
                        const int bl = max(u * Q_UB_PTS, klo[side]), bh = min(u * Q_UB_PTS + Q_UB_PTS - 1, khi[side]);
                        if (bl > bh) continue;
                        const double v = zr[side][u] + ((double)(int32_t)lo[i] + 256.0 * (int32_t)hi[i]) * (1.0 / 32.0);
#pragma unroll
                        for (int pc = 0; pc < 4; ++pc)
                            if (max(bl, pc * Q_PW) <= min(bh, pc * Q_PW + Q_PW - 1)) ub[side][pc] = fmax(ub[side][pc], v);
                    }
                }
            }
            tc_fence_before_sync();
            mbar_arrive(&sm.pipe.acc_empty[buf]);
            if (!wait_sleep<100>(sm.pipe.abort, &sm.lb_full, n_done & 1u)) return;
            double lb[SIDES];
#pragma unroll
            for (int side = 0; side < SIDES; ++side) lb[side] = sm.lb[side][boot];
            mbar_arrive(&sm.lb_empty);
            uint32_t dead = all;
#pragma unroll
            for (int side = 0; side < SIDES; ++side) {
                if (boot >= p.n_boot[side]) continue;  // a ragged pass: boots past its own count are not real
                if (side == 0 && p.lb_out) {           // scde_b200_probe_prune_i8
                    p.lb_out[(int64_t)pos * WP_TILED + boot] = lb[0];
                    for (int pc = 0; pc < 4; ++pc) p.ub_out[((int64_t)pos * WP_TILED + boot) * 4 + pc] = ub[0][pc];
                }
                const double thr = lb[side] - 747.0;  // lb = -inf (no sample inside the range): nothing is dead
                uint32_t d = 0u;
#pragma unroll
                for (int pc = 0; pc < 4; ++pc) d |= ub[side][pc] < thr ? 1u << pc : 0u;
                dead &= d;
            }
            dead = __reduce_and_sync(0xffffffffu, dead);
            const uint32_t lv = ~dead & all;
            if (lane == 0 && lv) atomicOr(p.live + (pos >> 2), lv << (8 * (pos & 3)));
        }
    }
}

template <int SIDES>
__global__ void __launch_bounds__(Q_THREADS, 1) bound_i8_kernel(const BoundParams p, int32_t *err) {
    using G = BoundGeom<SIDES>;
    run_pipeline<G::NS, BoundSmem<SIDES>>(
        B_RING, err,
        [](BoundSmem<SIDES> &sm) {
            mbar_init(&sm.lb_full, Q_EPILOGUE_WARPS / 2 * 32);
            mbar_init(&sm.lb_empty, Q_EPILOGUE_WARPS / 2 * 32);
        },
        [&](BoundSmem<SIDES> &sm, uint32_t stage0, int kg, int lane) { bound_producer<SIDES>(p, sm, stage0, kg, lane); },
        [&](BoundSmem<SIDES> &sm, uint32_t, uint32_t tmem, int ewarp, int lane) { bound_epilogue<SIDES>(p, sm, tmem, ewarp, lane); },
        [&](BoundSmem<SIDES> &sm, uint32_t stage0, uint32_t tmem) {
            const uint32_t idesc = umma_idesc_s8_mn(128, Q_BW);
            run_mma<G::NS, G::STAGE>(p.lists, sm.pipe, stage0, tmem, p.n_pos, [&](int pos) { return bound_gene(p, pos); }, nullptr,
                                     [&](uint32_t sA, uint32_t acc, bool accumulate) {
                                         const uint64_t db = umma_desc_sw128(sA + SIDES * B_TILE, 4096u, 1024u);
#pragma unroll
                                         for (int side = 0; side < SIDES; ++side)
                                             umma_s8(acc + (uint32_t)(side * Q_BW), umma_desc_sw128(sA + side * B_TILE, 4096u, 1024u),
                                                     db, idesc, accumulate);
                                     });
        });
}

// items[0 .. *n_live) = the live items' codes in launch order (piece-major or gene-major, as decode_item reads them); one
// CTA, four items per thread and round.  stats (may be NULL): [0] += items, [1] += live items, [2] += list entries over
// the items (what the unpruned launch would gather, in entry-pieces), [3] += the same over the live items.
constexpr int PC_THREADS = 1024;
__global__ void __launch_bounds__(PC_THREADS) prune_compact_kernel(const uint8_t *__restrict__ live, int n_pos, int n_pieces,
                                                                   int piece_major, const int32_t *__restrict__ order,
                                                                   const int32_t *__restrict__ lst_len, int32_t *__restrict__ items,
                                                                   int32_t *__restrict__ n_live, unsigned long long *stats) {
    __shared__ int wsum[PC_THREADS / 32];
    unsigned long long work = 0, live_work = 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = n_pos * n_pieces;
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += 4 * PC_THREADS) {
        uint32_t f = 0u;
        int c = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int i = i0 + 4 * threadIdx.x + e;
            if (i < n) {
                const int piece = piece_major ? i / n_pos : i % n_pieces;
                const int pos = piece_major ? i - piece * n_pos : i / n_pieces;
                const unsigned long long len = stats ? (unsigned long long)max(lst_len[order ? order[pos] : pos], 0) : 0ull;
                work += len;
                if ((live[pos] >> piece) & 1u) {
                    f |= 1u << e;
                    ++c;
                    live_work += len;
                }
            }
        }
        int x = c;  // inclusive scan over the warp
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        int off = base + (warp ? wsum[warp - 1] : 0) + x - c;
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if ((f >> e) & 1u) items[off++] = i0 + 4 * threadIdx.x + e;
        base += wsum[PC_THREADS / 32 - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *n_live = base;
        if (stats) {
            atomicAdd(stats, (unsigned long long)n);
            atomicAdd(stats + 1, (unsigned long long)base);
        }
    }
    if (stats) {
        work = __reduce_add_sync(0xffffffffu, (unsigned)work) + 0ull;  // < 2^32: a warp sees <= 4096 items of <= 65536 entries
        live_work = __reduce_add_sync(0xffffffffu, (unsigned)live_work) + 0ull;
        if (lane == 0) {
            atomicAdd(stats + 2, work);
            atomicAdd(stats + 3, live_work);
        }
    }
}

// exp_nonpos at -745, -746, -747 as softmax_i8_warp_kernel evaluates it (scde_b200_probe_prune_i8): the soft-max weight of a
// point more than 746 nats below its row maximum must be exactly 0 for pruning to leave the result unchanged
__global__ void exp_probe_kernel(double *out) {
    const int i = threadIdx.x;
    if (i < 3) out[i] = exp_nonpos(-745.0 - i);
}

// ------------------------------------------------------------------------------------------------
// fixed-point planes and non-sentinel range of every row of an FP64 table (the general row kernel writes FP64 only; the
// constant-theta fast kernel emits both itself, lp_table.cu): one warp per row
__global__ void __launch_bounds__(256) quantize_rows_kernel(const double *__restrict__ table, int ld_table, int K, int64_t n_rows,
                                                            int8_t *__restrict__ qtable, int64_t ldq,
                                                            uint32_t *__restrict__ row_range, int8_t *__restrict__ qbound) {
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    const double *src = table + row * ld_table;
    int8_t *dst = qtable + row * ldq;
    for (int64_t j = lane; j < ldq / 4; j += 32) reinterpret_cast<uint32_t *>(dst)[j] = 0u;
    __syncwarp();
    int n_ok = 0, kmin = 0x7fffffff, kmax = -1;
    for (int k = lane; k < K; k += 32) {
        const double v = src[k];
        if (!(v > -1.0e290)) continue;  // the "log 0" sentinel (or a difference to it): digits stay zero
        ++n_ok;
        kmin = min(kmin, k);
        kmax = max(kmax, k);
        long long x = __double2ll_rn(fmin(fmax(v, -1000.0), 1000.0) * (double)(1ll << Q_FRAC));
        const int pc = k / Q_PW, i = k - pc * Q_PW;
#pragma unroll
        for (int pl = 0; pl < Q_NV; ++pl) {
            const int d = (int)(int8_t)(x & 0xFF);
            dst[pc * Q_PIECE + pl * Q_PW + i] = (int8_t)d;
            x = (x - d) >> 8;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_ok += __shfl_xor_sync(0xffffffffu, n_ok, o);
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    uint32_t rr;
    if (n_ok == 0)
        rr = Q_RANGE_IRREGULAR;  // a row of sentinels only: let the FP64 kernel deal with it
    else if (kmax - kmin + 1 != n_ok)
        rr = Q_RANGE_IRREGULAR;
    else
        rr = (uint32_t)kmin | ((uint32_t)kmax << 16);
    if (lane == 0) row_range[row] = rr;
    if (qbound) {
        __syncwarp();  // the planes the other lanes wrote
        q_bound_row(dst, K, rr, qbound + row * Q_BW, lane, 32);
    }
}

// W (FP64 multiplicities, pass-major [pass][n_w_rows][108]) -> int8 rows of 128 bytes; flag |= 1 when a count > 127
__global__ void w_to_i8_kernel(const double *__restrict__ W, int64_t n_rows_total, int8_t *__restrict__ W8,
                               int32_t *__restrict__ flag) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows_total * Q_WB) return;
    const int64_t row = idx / Q_WB;
    const int col = (int)(idx - row * Q_WB);
    int v = 0;
    if (col < WP_TILED) {
        const double w = W[row * WS_TILED + col];
        if (w > 127.0) {
            atomicOr(flag, 1);
            v = 127;
        } else {
            v = (int)w;
        }
    }
    W8[idx] = (int8_t)v;
}

}  // namespace

cudaError_t launch_quantize_rows(const double *table, int ld_table, int K, int64_t n_rows, int8_t *qtable,
                                 uint32_t *row_range, int8_t *qbound, cudaStream_t st) {
    if (n_rows <= 0) return cudaSuccess;
    if (K > ld_table || K > Q_MAX_K) return cudaErrorInvalidValue;
    quantize_rows_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, st>>>(table, ld_table, K, n_rows, qtable, q_row_bytes(K),
                                                                        row_range, qbound);
    return cudaGetLastError();
}

cudaError_t launch_w_to_i8(const double *W, int n_w_rows, int n_boot, int8_t *W8, int32_t *flag, cudaStream_t st) {
    const int passes = (n_boot + WP_TILED - 1) / WP_TILED;
    const int64_t rows = (int64_t)(passes > 0 ? passes : 1) * n_w_rows;
    const int64_t n = rows * Q_WB;
    w_to_i8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, rows, W8, flag);
    return cudaGetLastError();
}

bool contract_i8_supported(int K, int ld_table, int ld_lst, int n_draws) {
    return K >= 1 && K <= Q_MAX_K && ld_table == KP_TILED && (ld_lst % Q_ES) == 0 && n_draws <= 65000;
}

size_t contract_i8_range_words(int n_genes) { return (size_t)(n_genes > 0 ? n_genes : 1) * Q_WB; }

// boots of a side's pass
static int side_boots(const ContractI8Args &a, const I8Side &s) {
    return (a.n_boot - s.pass * WP_TILED) < WP_TILED ? (a.n_boot - s.pass * WP_TILED) : WP_TILED;
}

// the lists of genes order[g0 ..] and the draw sets, as the kernels of a launch at g0 read them
static ListParams list_params(const ContractI8Args &a, int g0) {
    return ListParams{a.lists.row, a.lists.cell,  a.lists.len, a.lists.order ? a.lists.order + g0 : nullptr,
                      a.lists.ld,  a.gene_set,    a.set_w8};
}

// one launch of a pipeline kernel, one CTA of Q_THREADS per SM; function attributes are per device: set on every launch
// (a process may hold contexts on several GPUs)
template <class... Args>
static cudaError_t launch_pipeline(void (*kernel)(Args...), int grid, size_t smem, cudaStream_t st, Args... args) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, Q_THREADS, smem, st>>>(args...);
    return cudaGetLastError();
}

cudaError_t launch_sentinel_ranges(const ContractI8Args &a, int g0, int n_pos, const I8Side &s, cudaStream_t st) {
    if (n_pos <= 0 || !a.row_range) return cudaSuccess;
    if (!s.SR) return cudaErrorInvalidValue;
    const ListParams l = list_params(a, g0);
    sentinel_range_kernel<<<(unsigned)((n_pos + 7) / 8), 256, 0, st>>>(l.row, l.cell, l.len, l.order, l.ld, a.row_range, s.W8,
                                                                       l.gene_set, l.set_w8, n_pos, a.K, side_boots(a, s),
                                                                       s.SR, a.err);
    return cudaGetLastError();
}

cudaError_t launch_contract_i8_pass(const ContractI8Args &a, int g0, int n_pos, const I8Side *s, int n_sides, int n_sm,
                                    cudaStream_t st) {
    if (n_pos <= 0) return cudaSuccess;
    if (n_sides < 1 || n_sides > 2) return cudaErrorInvalidValue;
    I8Params p{};
    p.lists = list_params(a, g0);
    p.qtable = a.qtable;
    p.ldq = a.ldq;
    for (int i = 0; i < n_sides; ++i) {
        p.W8[i] = s[i].W8;
        p.T[i] = reinterpret_cast<long long *>(s[i].T);
    }
    p.n_boot = side_boots(a, s[0]);
    p.n_pos = n_pos;
    p.n_pieces = q_pieces(a.K);
    p.err = a.err;
    p.dbg = a.dbg;
    p.twin = n_sides > 1 ? 1 : 0;
    p.piece_major = a.item_order == 1;
    p.cold_evict_first = a.cold_evict_first;
    p.items = a.items;
    p.n_live = a.items ? a.n_live : nullptr;
    const int n_items = (n_pos * p.n_pieces) << p.twin;
    int grid = n_sm < n_items ? n_sm : n_items;
    if (p.twin) grid &= ~1;  // an even stride keeps every CTA on one side and the pairs (2 i, 2 i + 1) together
    if (a.hot_rank >= 0) return launch_pipeline(contract_i8_kernel<true, Q_NS>, grid, q_smem_bytes(Q_NS), st, p);
    // the shallow ring leaves 69 KB of shared memory and a third of the register file to a co-resident kernel
    if (a.ring_stages == 7) return launch_pipeline(contract_i8_kernel<false, 7>, grid, q_smem_bytes(7), st, p);
    if (a.ring_stages == 8) return launch_pipeline(contract_i8_kernel<false, 8>, grid, q_smem_bytes(8), st, p);
    return launch_pipeline(contract_i8_kernel<false, Q_NS>, grid, q_smem_bytes(Q_NS), st, p);
}

size_t prune_zb_doubles(int n_sets, int n_boot) {
    const int passes = (n_boot + WP_TILED - 1) / WP_TILED;
    return (size_t)(n_sets > 0 ? n_sets : 1) * (passes > 0 ? passes : 1) * WP_TILED * Q_BSLOTS;
}

cudaError_t launch_z_bounds(const ContractI8Args &a, const double *Z, int n_sets, double *zb, cudaStream_t st) {
    const int64_t rows = (int64_t)prune_zb_doubles(n_sets, a.n_boot) / Q_BSLOTS;
    z_bounds_kernel<<<(unsigned)((rows * Q_BSLOTS + 255) / 256), 256, 0, st>>>(Z, rows, a.K, zb);
    return cudaGetLastError();
}

cudaError_t launch_prune_items(const ContractI8Args &a, int g0, int n_pos, const I8Side *s, int n_sides, int n_sm, uint8_t *live,
                               int32_t *items, int32_t *n_live, unsigned long long *stats, cudaStream_t st,
                               double *lb_out, double *ub_out) {
    if (n_pos <= 0) return cudaSuccess;
    if (!a.qbound || n_sides < 1 || n_sides > 2) return cudaErrorInvalidValue;
    BoundParams p{};
    p.lists = list_params(a, g0);
    p.qbound = a.qbound;
    p.set_zb = (int64_t)prune_zb_doubles(1, a.n_boot);
    for (int i = 0; i < n_sides; ++i) {
        p.W8[i] = s[i].W8;
        p.SR[i] = a.row_range ? s[i].SR : nullptr;
        p.zb[i] = s[i].zb + (size_t)s[i].pass * WP_TILED * Q_BSLOTS;
        p.n_boot[i] = side_boots(a, s[i]);
    }
    p.n_pos = n_pos;
    p.K = a.K;
    p.n_pieces = q_pieces(a.K);
    p.live = reinterpret_cast<uint32_t *>(live);
    p.lb_out = lb_out;
    p.ub_out = ub_out;
    cudaError_t e = cudaMemsetAsync(live, 0, prune_live_bytes(n_pos), st);
    if (e != cudaSuccess) return e;
    const int grid = n_sm < n_pos ? n_sm : n_pos;
    e = n_sides > 1 ? launch_pipeline(bound_i8_kernel<2>, grid, bound_smem_bytes<2>(), st, p, a.err)
                    : launch_pipeline(bound_i8_kernel<1>, grid, bound_smem_bytes<1>(), st, p, a.err);
    if (e != cudaSuccess) return e;
    prune_compact_kernel<<<1, PC_THREADS, 0, st>>>(live, n_pos, q_pieces(a.K), a.item_order == 1, p.lists.order, a.lists.len,
                                                   items, n_live, stats);
    return cudaGetLastError();
}

size_t prune_live_bytes(int n_pos) { return (size_t)((n_pos > 0 ? n_pos : 1) + 3) & ~(size_t)3; }

cudaError_t launch_exp_probe(double *out_host, cudaStream_t st) {
    double *d = nullptr;
    cudaError_t e = cudaMallocAsync(&d, 3 * sizeof(double), st);
    if (e != cudaSuccess) return e;
    exp_probe_kernel<<<1, 32, 0, st>>>(d);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_host, d, 3 * sizeof(double), cudaMemcpyDeviceToHost, st);
    const cudaError_t f = cudaFreeAsync(d, st);
    return e != cudaSuccess ? e : f;
}

size_t softmax_i8_scratch_doubles(int n_pos) { return (size_t)SP_GROUPS * (n_pos > 0 ? n_pos : 1) * KP_TILED; }

cudaError_t launch_softmax_i8(const ContractI8Args &a, int g0, int n_pos, const I8Side &s, double *part_scratch, int n_sm,
                              cudaStream_t st, const uint8_t *live) {
    if (n_pos <= 0) return cudaSuccess;
    if (a.row_range && !s.SR) return cudaErrorInvalidValue;
    const bool sets = a.gene_set && s.Z;
    const size_t smem = sets ? 0 : sizeof(double) * SP_ROWS * KP_TILED;
    auto kernel = sets ? (live ? softmax_i8_warp_kernel<true, true> : softmax_i8_warp_kernel<true, false>)
                       : (live ? softmax_i8_warp_kernel<false, true> : softmax_i8_warp_kernel<false, false>);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int wb = n_sm * 2 / SP_GROUPS;  // two CTAs of eight warps per SM
    if (wb * SW_WARPS > n_pos) wb = (n_pos + SW_WARPS - 1) / SW_WARPS;
    if (wb < 1) wb = 1;
    kernel<<<wb * SP_GROUPS, SW_WARPS * 32, smem, st>>>(reinterpret_cast<const long long *>(s.T), s.Z,
                                                        a.row_range ? s.SR : nullptr, a.K, side_boots(a, s), a.scale,
                                                        part_scratch, n_pos, a.lists.order ? a.lists.order + g0 : nullptr,
                                                        a.gene_set, a.set_z, live);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int64_t n = (int64_t)n_pos * KP_TILED;
    softmax_i8_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(part_scratch, a.lists.order ? a.lists.order + g0 : nullptr,
                                                                          a.K, n_pos, s.jp, a.ld_jp, s.pass > 0);
    return cudaGetLastError();
}

cudaError_t launch_finalize_t(const ContractI8Args &a, int n_pos, const I8Side &s, cudaStream_t st) {
    if (n_pos <= 0) return cudaSuccess;
    const int64_t n = (int64_t)n_pos * WP_TILED * KP_TILED;
    finalize_t_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(reinterpret_cast<long long *>(s.T),
                                                                   a.row_range ? s.SR : nullptr, a.sentinel, n);
    return cudaGetLastError();
}

}  // namespace scde
