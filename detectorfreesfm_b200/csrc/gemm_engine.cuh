// Shifted-row implicit-GEMM engine on tcgen05 tensor cores (sm_100a).
//
//   acc[p, n] = sum_t sum_c  A_t[p + shift_t, c] * Wt[n, t*cpad + c]          (fp32 accumulate in TMEM)
//
// One kernel serves every dense contraction of both hot paths:
//   * 3x3 / 5x5 / 1x1 convolutions on "flat halo" NHWC activations (a conv tap is a pure row shift, see DESIGN.md),
//   * stride-2 convolutions (taps read the four parity planes written by the previous layer's epilogue),
//   * linear layers (one tap, shift 0; a concat of two inputs is two taps),
//   * the LxS similarity GEMM of the dual-softmax matcher.
// Operands are "split-fp16": every fp32 value x is stored as two fp16 planes (hi, lo) with hi+lo ~= x to 22 bits, and a
// K-step issues hi*hi + hi*lo + lo*hi (3 tcgen05.mma, kind::f16) -- fp32-grade results at tensor-core rate (kSplit=true),
// or a single hi*hi pass (kSplit=false).
//
// CTA = 128 x BN output tile, 192 threads: warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM allocator),
// warps 2..5 = epilogue (TMEM -> registers -> global).  A/B tiles are [rows][64 halves] with the 128-byte TMA swizzle.
#pragma once
#include "tc_common.cuh"

namespace dfsfm {

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr int kMaxTaps = 26;
constexpr int kMaxAMaps = 5;
constexpr int kGemmThreads = 192;   // engine 1: 2 role warps + 4 epilogue warps
constexpr int kGemm2EpiWarps = 8;  // engine 2: two warps per TMEM lane quadrant, each takes half of the tile's columns
constexpr int kGemm2Threads = 64 + 32 * kGemm2EpiWarps;

// Engine-2 extras handed to an epilogue warp: its staging buffer (Epi::kEpiStageBytes, null on engine 1), the buffer of the
// warp that owns the other half of the same rows' columns, and the named barrier the two share.
struct EpiCtx {
    uint8_t* stg;
    uint8_t* stg_partner;
    int bar_id;
};

struct TmapPack {
    CUtensorMap a[kMaxAMaps];  // activation planes: dims {C, rows, 2 (hi/lo)}, box {64, 128, 1}
    CUtensorMap b;             // weights: dims {Ktot, Nrows, 2 (hi/lo)}, box {64, BN, 1}
};

struct GemmCore {
    int M;         // rows of the flat index space
    int num_taps;  // <= kMaxTaps
    int kchunks;   // 64-wide K chunks per tap = ceil(cpad / 64)
    int k16_last;  // valid 16-wide K steps in the last chunk of a tap (1..4)
    int cpad;      // K elements per tap in the weight matrix
    int b_row0;    // first weight row (output channel) of this launch
    int bo_mode;   // tap groups only: 1 = put (address >> 7) & 7 into the descriptor's base-offset field for row-shifted starts
    int seg_mp0;   // engine 2: row-pair tiles (256 rows) >= seg_mp0 read their weight tile seg_b_rows rows further down (0: off) --
    int seg_b_rows;  //   the two images of a pair carry different per-call "weights" (the attention state folded into merge)
    int8_t tap_map[kMaxTaps];  // which activation map a tap reads
    int tap_shift[kMaxTaps];   // row shift of a tap
    unsigned long long* tl;    // engine 2, debugging: when set, [CTA][16] globaltimer stamps of this launch (dfsfm_debug_timeline)
};

__device__ __forceinline__ void tl_stamp(const GemmCore& core, int ev) {
    if (core.tl != nullptr && blockIdx.x < 148) {  // the host buffer holds 148 CTAs per launch
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        core.tl[blockIdx.x * 16 + ev] = t;
    }
}

template <int BN, bool kSplit>
struct GemmCfg {
    static constexpr int kABytes = kBM * 128;  // one plane of an A tile
    static constexpr int kBBytes = BN * 128;   // one plane of a B tile
    static constexpr int kPlanes = kSplit ? 2 : 1;
    static constexpr int kStageBytes = kPlanes * (kABytes + kBBytes);
    static constexpr int kBudget = 200 * 1024;
    static constexpr int kStagesRaw = kBudget / kStageBytes;
    static constexpr int kStages = kStagesRaw > 6 ? 6 : kStagesRaw;
    static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
    // Two accumulators in TMEM: the main one takes hi*hi, the correction one (kCorrOff columns further) takes
    // hi*lo + lo*hi.  Tensor-core fp32 accumulation truncates, so keeping the 2^-11-sized terms out of the large
    // accumulator cuts both the number of truncating adds into it (3x) and the rounding bias; they are summed
    // in the epilogue with round-to-nearest.
    static constexpr int kAccCols = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    static constexpr int kCorrOff = kSplit ? kAccCols : 0;
    static constexpr int kTmemCols = kSplit ? 2 * kAccCols : kAccCols;
    static_assert(kStages >= 2, "tile too large");
    static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "invalid UMMA N");
};

// Epi must provide:  struct Params;  static __device__ void run(const Params&, uint32_t tmem_warp, int row0_warp, int lane, int n0)
template <int BN, bool kSplit, class Epi>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ TmapPack maps, const GemmCore core, const typename Epi::Params ep) {
    using Cfg = GemmCfg<BN, kSplit>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
    uint64_t* empty_bar = full_bar + Cfg::kStages;
    uint64_t* tmem_full_bar = empty_bar + Cfg::kStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * kBM;
    const int n0 = blockIdx.y * BN;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < kMaxAMaps; ++i) tma_prefetch_desc(&maps.a[i]);
        tma_prefetch_desc(&maps.b);
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full_bar, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n_iters = core.num_taps * core.kchunks;

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t phase = 0;
            for (int it = 0; it < n_iters; ++it) {
                const int t = it / core.kchunks;
                const int c = it - t * core.kchunks;
                mbar_wait(&empty_bar[s], phase ^ 1);
                mbar_arrive_expect_tx(&full_bar[s], Cfg::kStageBytes);
                uint8_t* st = smem + s * Cfg::kStageBytes;
                const CUtensorMap* am = &maps.a[core.tap_map[t]];
                const int row = m0 + core.tap_shift[t];
                const int kb = t * core.cpad + c * kBK;
                tma_load_3d(st, am, &full_bar[s], c * kBK, row, 0);
                if (kSplit) tma_load_3d(st + Cfg::kABytes, am, &full_bar[s], c * kBK, row, 1);
                uint8_t* sb = st + Cfg::kPlanes * Cfg::kABytes;
                tma_load_3d(sb, &maps.b, &full_bar[s], kb, core.b_row0 + n0, 0);
                if (kSplit) tma_load_3d(sb + Cfg::kBBytes, &maps.b, &full_bar[s], kb, core.b_row0 + n0, 1);
                if (++s == Cfg::kStages) { s = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_f16(kBM, BN);
            int s = 0;
            uint32_t phase = 0;
            uint32_t acc = 0;
            const uint32_t tmem_corr = tmem_base + Cfg::kCorrOff;
            for (int it = 0; it < n_iters; ++it) {
                const int c = it % core.kchunks;
                mbar_wait(&full_bar[s], phase);
                tc_fence_after();
                const uint32_t a_hi = smem_u32(smem + s * Cfg::kStageBytes);
                const uint32_t b_hi = a_hi + Cfg::kPlanes * Cfg::kABytes;
                const int nk = (c == core.kchunks - 1) ? core.k16_last : 4;
                for (int k = 0; k < nk; ++k) {
                    const uint64_t da = make_smem_desc_sw128(a_hi + k * 32);
                    const uint64_t db = make_smem_desc_sw128(b_hi + k * 32);
                    umma_f16(tmem_base, da, db, idesc, acc);
                    if (kSplit) {
                        const uint64_t dal = make_smem_desc_sw128(a_hi + Cfg::kABytes + k * 32);
                        const uint64_t dbl = make_smem_desc_sw128(b_hi + Cfg::kBBytes + k * 32);
                        umma_f16(tmem_corr, da, dbl, idesc, acc);
                        umma_f16(tmem_corr, dal, db, idesc, 1);
                    }
                    acc = 1;
                }
                umma_commit(&empty_bar[s]);
                if (++s == Cfg::kStages) { s = 0; phase ^= 1; }
            }
            umma_commit(tmem_full_bar);
        }
        __syncwarp();
    } else {
        const int quad = warp & 3;  // TMEM lane quadrant this warp may read
        mbar_wait(tmem_full_bar, 0);
        tc_fence_after();
        Epi::template run<BN, Cfg::kCorrOff>(ep, tmem_base + (static_cast<uint32_t>(quad * 32) << 16), m0 + quad * 32, lane, n0, 0, BN,
                                             static_cast<int>(blockIdx.y), EpiCtx{nullptr, nullptr, 0});
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

// ================================================================================================ engine v2
// Persistent CTA-pair engine: a cluster of two CTAs (cta_group::2) owns a 256-row x BN output tile per step -- each CTA
// stages its own 128 activation rows and HALF of the weight tile, the leader CTA issues M=256 tcgen05.mma for both, so the
// shared-memory traffic per MMA drops from (A + B) to (A + B/2) per SM.  Clusters loop over tiles (static round-robin);
// the TMA producer runs ahead across tile boundaries and, when TMEM has room for two accumulator sets (BN <= 128 with
// split operands), the epilogue of tile i overlaps the MMAs of tile i+1.
// G = taps per group: G consecutive taps whose row shifts are consecutive (the dx = -1,0,1 taps of one kernel row) share ONE
// activation slab of 128 + 8 rows per stage -- the tap's operand is the slab advanced by i rows (128 bytes) -- so the
// activation traffic (L2 -> SM and TMA writes into shared memory) drops by G.
constexpr int kSlabRows = kBM + 8;
template <int BN, bool kSplit, bool kSepCorr = true, int G = 1, int kEpiStageBytes = 0>
struct Gemm2Cfg {
    static constexpr int kABytes = (G == 1 ? kBM : kSlabRows) * 128;
    static constexpr int kBTapBytes = (BN / 2) * 128;  // this CTA's half of one tap's weight tile
    static constexpr int kBBytes = G * kBTapBytes;
    static constexpr int kPlanes = kSplit ? 2 : 1;
    static constexpr int kStageBytes = kPlanes * (kABytes + kBBytes);
    // per-warp epilogue staging (Epi::kEpiStageBytes: the warp's 32-row block is transposed through shared memory so that global
    // loads / stores of the epilogue are row-contiguous); it comes out of the operand-stage budget only when it has to
    static constexpr int kEpiSmem = kEpiStageBytes * kGemm2EpiWarps;
    static constexpr int kBarBytes = 768;  // pipeline barriers, TMEM slot, cluster-launch-control answers + their barriers
    static constexpr int kBudgetMax = 227 * 1024 - 1024 - kBarBytes - kEpiSmem;
    static constexpr int kBudget = kBudgetMax < 204 * 1024 ? kBudgetMax : 204 * 1024;
    static constexpr int kStagesRaw = kBudget / kStageBytes;
    static constexpr int kStages = kStagesRaw > 6 ? 6 : kStagesRaw;
    static constexpr int kEpiOff = kStages * kStageBytes + kBarBytes;  // after the barriers
    static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + kBarBytes + kEpiSmem;
    static constexpr int kAccCols = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    // kSepCorr: hi*lo + lo*hi go to their own accumulator (long-K convolutions).  Short-K linears fold them into the main
    // accumulator (truncation bias ~ -5.5e-9*K*3 relative: harmless at K <= 512), which leaves TMEM room for a second
    // accumulator set even at BN = 256, so the epilogue of a tile overlaps the MMAs of the next.
    static constexpr int kCorrOff = (kSplit && kSepCorr) ? kAccCols : 0;
    static constexpr int kSetCols = (kSplit && kSepCorr) ? 2 * kAccCols : kAccCols;
    static constexpr int kAccStages = (512 / kSetCols) >= 2 ? 2 : 1;
    static constexpr int kTmemCols = kSetCols * kAccStages;
    static_assert(kStages >= 2, "tile too large");
    static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256 && (BN / 2) % 8 == 0, "invalid UMMA N for a CTA pair");
};

// Tile order of a cluster.  Static: tile = cluster + k * clusters with min(tiles, SM pairs) clusters in the grid.  Stealing: the grid has
// ONE cluster per tile; while a cluster works on a tile its producer asks the hardware to cancel a cluster of the grid that has not been
// launched yet (cluster launch control) and the whole cluster takes that tile next, until nothing is left to cancel.  Clusters that start
// late -- SMs held by another stream's kernel (several pair workers per GPU), or by the tail of the previous kernel of this stream under
// programmatic dependent launch -- then simply take fewer tiles instead of stretching the launch by their static share.
// The answers go through a ring of kClcSlots slots without "empty" barriers: the producer of a cluster is never more than kStages
// K-chunks ahead of the MMA thread and that at most two accumulator sets ahead of the slowest epilogue warp, far fewer than 16 tiles.
constexpr int kClcSlots = 16;
struct TileSched {
    uint64_t* bars;  // [kClcSlots], this CTA's
    uint4* resp;     // [kClcSlots]
    int num_tiles, num_clusters;
    bool steal;
    int j, tile;
    __device__ __forceinline__ int first() {
        j = 0;
        tile = blockIdx.x >> 1;
        return tile;
    }
    // the producer thread of each CTA, at the start of its tile j: arm the slot; CTA 0 also sends the request whose answer is tile j + 1
    __device__ __forceinline__ void request(uint32_t rank) {
        if (steal) {
            const int q = j & (kClcSlots - 1);
            mbar_arrive_expect_tx(&bars[q], 16);
            if (rank == 0) clc_try_cancel_multicast(&resp[q], &bars[q]);
        }
    }
    __device__ __forceinline__ int next() {
        if (steal) {
            const int q = j & (kClcSlots - 1);
            mbar_wait(&bars[q], (j / kClcSlots) & 1);
            const int x = clc_decode(&resp[q]);
            fence_proxy_async();  // this generic read before the slot's next asynchronous write
            tile = x < 0 ? -1 : (x >> 1);
        } else {
            tile += num_clusters;
            if (tile >= num_tiles) tile = -1;
        }
        ++j;
        return tile;
    }
};

struct EpiNoState {};
template <class Epi, bool = Epi::kHasState>
struct EpiStateOf { using type = EpiNoState; };
template <class Epi>
struct EpiStateOf<Epi, true> { using type = typename Epi::State; };

template <int BN, bool kSplit, class Epi, int G = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemm2Threads, 1)
gemm_tc2_kernel(const __grid_constant__ TmapPack maps, const GemmCore core, const typename Epi::Params ep, const int num_tiles,
                const int n_tiles, const int steal) {
    using Cfg = Gemm2Cfg<BN, kSplit, Epi::kSeparateCorr, G, Epi::kEpiStageBytes>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
    uint64_t* empty_bar = full_bar + Cfg::kStages;
    uint64_t* tmem_full_bar = empty_bar + Cfg::kStages;
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    uint64_t* clc_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes + 256);
    uint4* clc_resp = reinterpret_cast<uint4*>(clc_bar + kClcSlots);
    static_assert(256 + kClcSlots * (8 + 16) <= Cfg::kBarBytes && (2 * 6 + 4) * 8 + 4 <= 256, "barrier region");

    // Programmatic dependent launch: let the next kernel of the stream start its prologue on SMs we leave idle ...
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (threadIdx.x == 0) tl_stamp(core, 0);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1;
    const int num_clusters = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < kMaxAMaps; ++i) tma_prefetch_desc(&maps.a[i]);
        tma_prefetch_desc(&maps.b);
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1);
            mbar_init(&tmem_empty_bar[a], 2 * kGemm2EpiWarps);  // every epilogue warp of both CTAs arrives on the leader's barrier
        }
        for (int q = 0; q < kClcSlots; ++q) mbar_init(&clc_bar[q], 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_2sm<Cfg::kTmemCols>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) tl_stamp(core, 1);
    // ... and wait here, with barriers initialised and TMEM allocated, until the previous kernel's results are visible.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (threadIdx.x == 0) tl_stamp(core, 2);
    const int n_iters = (core.num_taps / G) * core.kchunks;
    TileSched ts;
    ts.bars = clc_bar;
    ts.resp = clc_resp;
    ts.num_tiles = num_tiles;
    ts.num_clusters = num_clusters;
    ts.steal = steal != 0;

    if (warp == 0) {
        if (elect_one()) {
            int s = 0;
            uint32_t phase = 0;
            for (int tile = ts.first(); tile >= 0; tile = ts.next()) {
                ts.request(rank);
                const int mp = tile / n_tiles, nt = tile - mp * n_tiles;
                const int m0 = (mp * 2 + static_cast<int>(rank)) * kBM;
                const int nrow = core.b_row0 + nt * BN + static_cast<int>(rank) * (BN / 2) + ((core.seg_mp0 > 0 && mp >= core.seg_mp0) ? core.seg_b_rows : 0);
                for (int it = 0; it < n_iters; ++it) {
                    const int t = (it / core.kchunks) * G;  // first tap of the group
                    const int c = it % core.kchunks;
                    mbar_wait(&empty_bar[s], phase ^ 1);
                    if (rank == 0) mbar_arrive_expect_tx(&full_bar[s], 2 * Cfg::kStageBytes);
                    uint8_t* st = smem + s * Cfg::kStageBytes;
                    const CUtensorMap* am = &maps.a[core.tap_map[t]];
                    const int row = m0 + core.tap_shift[t];
                    tma_load_3d_2sm(st, am, &full_bar[s], c * kBK, row, 0);  // G == 1: 128 rows; else the (128+8)-row slab
                    if (kSplit) tma_load_3d_2sm(st + Cfg::kABytes, am, &full_bar[s], c * kBK, row, 1);
                    uint8_t* sb = st + Cfg::kPlanes * Cfg::kABytes;
#pragma unroll
                    for (int i = 0; i < G; ++i) {
                        const int kb = (t + i) * core.cpad + c * kBK;
                        tma_load_3d_2sm(sb + i * Cfg::kBTapBytes, &maps.b, &full_bar[s], kb, nrow, 0);
                        if (kSplit) tma_load_3d_2sm(sb + Cfg::kBBytes + i * Cfg::kBTapBytes, &maps.b, &full_bar[s], kb, nrow, 1);
                    }
                    if (++s == Cfg::kStages) { s = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (rank == 0 && elect_one()) {
            constexpr uint32_t idesc = make_idesc_f16(2 * kBM, BN);
            int s = 0;
            uint32_t phase = 0;
            int a = 0;
            uint32_t aphase = 0;
            for (int tile = ts.first(); tile >= 0; tile = ts.next()) {
                mbar_wait(&tmem_empty_bar[a], aphase ^ 1);
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + a * Cfg::kSetCols;
                const uint32_t tmem_corr = tmem_acc + Cfg::kCorrOff;
                uint32_t acc = 0;
                for (int it = 0; it < n_iters; ++it) {
                    const int c = it % core.kchunks;
                    mbar_wait(&full_bar[s], phase);
                    tc_fence_after();
                    if (it == 0 && ts.j == 0) tl_stamp(core, 3);
                    const uint32_t a_hi = smem_u32(smem + s * Cfg::kStageBytes);
                    const uint32_t b_hi = a_hi + Cfg::kPlanes * Cfg::kABytes;
                    const int nk = (c == core.kchunks - 1) ? core.k16_last : 4;
                    // One descriptor per operand plane and stage; every MMA's descriptors are that plus a small constant in the 16-byte
                    // address field (K step k: +32 B; tap i of a slab: +i rows = +128 B inside the swizzle atom; lo plane; tap's weight
                    // tile).  The issuing thread is on the critical path of a 128-column tile (64 clocks per MMA at the peak rate): built
                    // from scratch per MMA the descriptors cost ~17 dependent uniform-datapath instructions each.
                    const uint64_t da0 = make_smem_desc_sw128(a_hi), db0 = make_smem_desc_sw128(b_hi);
                    auto issue = [&](int i, int k) {
                        const uint64_t bo = (G > 1 && core.bo_mode) ? (static_cast<uint64_t>(i) << 49) : 0;  // debug hook only (dfsfm_debug_gemm2)
                        const uint64_t da = (da0 + static_cast<uint64_t>(i * 8 + k * 2)) | bo;
                        const uint64_t db = db0 + static_cast<uint64_t>(i * (Cfg::kBTapBytes >> 4) + k * 2);
                        umma_f16_2sm(tmem_acc, da, db, idesc, acc);
                        if (kSplit) {
                            umma_f16_2sm(tmem_corr, da, db + (Cfg::kBBytes >> 4), idesc, Epi::kSeparateCorr ? acc : 1u);
                            umma_f16_2sm(tmem_corr, da + (Cfg::kABytes >> 4), db, idesc, 1);
                        }
                        acc = 1;
                    };
                    if (nk == 4) {
#pragma unroll
                        for (int i = 0; i < G; ++i) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) issue(i, k);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < G; ++i) {
                            for (int k = 0; k < nk; ++k) issue(i, k);
                        }
                    }
                    umma_commit_2sm(&empty_bar[s]);
                    if (++s == Cfg::kStages) { s = 0; phase ^= 1; }
                }
                umma_commit_2sm(&tmem_full_bar[a]);
                tl_stamp(core, ts.j == 0 ? 4 : 5);  // MMAs of the first / of the latest tile issued
                if (++a == Cfg::kAccStages) { a = 0; aphase ^= 1; }
            }
        }
        __syncwarp();
    } else {
        const int quad = warp & 3;            // TMEM lane quadrant this warp may read
        const int half = (warp - 2) >> 2;     // which half of the tile's columns this warp handles
        constexpr int kHalfCols = ((BN / 2 + 31) / 32) * 32;
        const int cb = half * kHalfCols, ce = half == 0 ? kHalfCols : BN;
        int a = 0;
        uint32_t aphase = 0;
        EpiCtx ctx;
        ctx.stg = Epi::kEpiStageBytes ? smem + Cfg::kEpiOff + (warp - 2) * Epi::kEpiStageBytes : nullptr;
        ctx.stg_partner = Epi::kEpiStageBytes ? smem + Cfg::kEpiOff + ((warp - 2) ^ 4) * Epi::kEpiStageBytes : nullptr;
        ctx.bar_id = 1 + quad;
        // stateful epilogues (KvEpi) carry per-thread accumulators across the tiles of this persistent CTA
        typename EpiStateOf<Epi>::type est;
        if constexpr (Epi::kHasState) Epi::init(est);
        for (int tile = ts.first(); tile >= 0; tile = ts.next()) {
            const int mp = tile / n_tiles, nt = tile - mp * n_tiles;
            const int m0 = (mp * 2 + static_cast<int>(rank)) * kBM;
            mbar_wait(&tmem_full_bar[a], aphase);
            tc_fence_after();
            if (warp == 2 && lane == 0) tl_stamp(core, ts.j == 0 ? 6 : 8);  // accumulator of the first / latest tile complete
            if constexpr (Epi::kHasState)
                Epi::template run_state<BN>(ep, est, tmem_base + a * Cfg::kSetCols + (static_cast<uint32_t>(quad * 32) << 16), m0 + quad * 32, lane, nt,
                                            half, quad, ctx, smem + Cfg::kEpiOff);
            else
                Epi::template run<BN, Cfg::kCorrOff>(ep, tmem_base + a * Cfg::kSetCols + (static_cast<uint32_t>(quad * 32) << 16), m0 + quad * 32, lane,
                                                     nt * BN, cb, ce, nt * 2 + half, ctx);
            tc_fence_before();
            __syncwarp();
            if (warp == 2 && lane == 0) tl_stamp(core, ts.j == 0 ? 7 : 9);  // epilogue of the first / latest tile done (this warp)
            if (lane == 0) mbar_arrive_remote(&tmem_empty_bar[a], 0);
            if (++a == Cfg::kAccStages) { a = 0; aphase ^= 1; }
        }
        if constexpr (Epi::kHasState) Epi::finish(ep, est, lane, half, quad, smem + Cfg::kEpiOff);
    }
    tc_fence_before();
    if (threadIdx.x == 0) tl_stamp(core, 10);
    cluster_sync_all();
    if (threadIdx.x == 0) tl_stamp(core, 11);
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------------ epilogues
__device__ __forceinline__ float fast_ex2(float x) {  // 2^x, MUFU.EX2 (2 ulp), flushes denormal results to zero
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float ex2_denorm(float x) {  // 2^x keeping subnormal results (thr = 0 must see every conf > 0)
    float y;
    asm("ex2.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// 32 accumulator columns of this thread's row: main (+ correction accumulator, added with round-to-nearest).
template <int kCorr>
__device__ __forceinline__ void load_acc32(uint32_t taddr, float* v) {
    tmem_ld32(taddr, v);
    if (kCorr > 0) {
        float w[32];
        tmem_ld32(taddr + kCorr, w);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += w[j];
    } else {
        tmem_ld_wait();
    }
}

// Geometry of a "flat halo" index space: image n, row y, col x  <->  p = n*Hp*Wp + y*Wp + x with Hp = H+1, Wp = W+1.
// Column x == W and row y == H are zero halo cells shared by neighbouring rows / images: they are zeroed when the
// buffer is allocated and never written afterwards, so a conv tap (dy,dx) is the row shift dy*Wp + dx.
struct FlatGeom {
    int Hp, Wp, H, W;  // Hp == 0: dense rows (no halo)
};

enum OutMode : int {
    OUT_FLAT = 0,    // same flat geometry as the input index space
    OUT_PARITY = 1,  // four half-resolution parity planes (feeds a stride-2 conv)
    OUT_DENSE = 2,   // dense token rows n*H*W + y*W + x
    OUT_WINDOW = 3,  // a (wh x ww) window at (y0,x0) re-packed into its own flat-halo geometry (ohp x owp per image)
    OUT_WINDOW_DENSE = 4,  // the window re-packed into dense rows n*wh*ww + y*ww + x
    OUT_UNPARITY = 5,      // the input geometry is parity plane (upy,upx): pixel (y,x) lands at (2y+upy, 2x+upx) of a flat geometry (ohp x owp)
};

struct ConvEpiParams {
    int M, N;           // valid rows, output channels to write (padded channel count of the output buffer)
    FlatGeom g;
    const float* bias;  // [>= N] (BatchNorm folded), may be null
    int relu;
    const __half* res_hi;  // optional residual in the input flat geometry
    const __half* res_lo;
    int res_ld;
    const float* addend;  // optional fp32 addend [.][N]
    int addend_mode;      // 0: row (y*W + x), added to the fp32 output only, after activation (position encoding next to raw planes);
                          // 1: row n_img (one vector per image / window), added before the activation to every output
    int out_mode;
    __half* out_hi;
    __half* out_lo;
    int out_ld;
    long long plane_stride;  // OUT_PARITY: elements between consecutive parity planes
    float* out_f32;          // optional fp32 copy (same row mapping as out_hi)
    float* out_f32_1;        // OUT_DENSE: image 1's fp32 rows go here (from row 0) instead of after image 0 in out_f32; may be null
    int out_f32_ld;
    int wy0, wx0, wh, ww;    // OUT_WINDOW / OUT_WINDOW_DENSE
    int ohp, owp;            // OUT_WINDOW / OUT_UNPARITY: rows / pitch of the output geometry
    int upy, upx;            // OUT_UNPARITY
};

struct ConvEpi {
    using Params = ConvEpiParams;
    static constexpr bool kHasState = false;
    static constexpr bool kSeparateCorr = true;
    static constexpr int kEpiStageBytes = 0;
    template <int BN, int kCorr>
    static __device__ __forceinline__ void run(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, int ce, int part_idx, const EpiCtx& ctx) {
        const int row = row0 + lane;
        bool valid = row < p.M;
        int n_img = 0, y = 0, x = 0;
        if (p.g.Hp > 0) {
            const int per = p.g.Hp * p.g.Wp;
            n_img = row / per;
            const int r = row - n_img * per;
            y = r / p.g.Wp;
            x = r - y * p.g.Wp;
            valid = valid && (y < p.g.H) && (x < p.g.W);
        }
        long long orow = row;   // output row index
        long long obase = 0;    // extra element offset (parity plane)
        float* out_f32 = p.out_f32;
        if (p.out_mode == OUT_PARITY) {
            const int Hp2 = p.g.H / 2 + 1, Wp2 = p.g.W / 2 + 1;
            obase = static_cast<long long>((y & 1) * 2 + (x & 1)) * p.plane_stride;
            orow = static_cast<long long>(n_img) * Hp2 * Wp2 + (y >> 1) * Wp2 + (x >> 1);
        } else if (p.out_mode == OUT_DENSE) {
            if (n_img == 1 && p.out_f32_1) {
                out_f32 = p.out_f32_1;
                orow = y * p.g.W + x;
            } else {
                orow = static_cast<long long>(n_img) * p.g.H * p.g.W + y * p.g.W + x;
            }
        } else if (p.out_mode == OUT_WINDOW) {
            valid = valid && y >= p.wy0 && y < p.wy0 + p.wh && x >= p.wx0 && x < p.wx0 + p.ww;
            orow = static_cast<long long>(n_img) * p.ohp * p.owp + (y - p.wy0) * p.owp + (x - p.wx0);
        } else if (p.out_mode == OUT_WINDOW_DENSE) {
            valid = valid && y >= p.wy0 && y < p.wy0 + p.wh && x >= p.wx0 && x < p.wx0 + p.ww;
            orow = static_cast<long long>(n_img) * p.wh * p.ww + (y - p.wy0) * p.ww + (x - p.wx0);
        } else if (p.out_mode == OUT_UNPARITY) {
            orow = static_cast<long long>(n_img) * p.ohp * p.owp + (2 * y + p.upy) * p.owp + (2 * x + p.upx);
        }
#pragma unroll 1
        for (int c0 = cb; c0 < ce; c0 += 32) {
            float v[32];
            load_acc32<kCorr>(tmem_warp + c0, v);  // warp-collective: every lane executes it
            const int nb = n0 + c0;
            if (!valid || nb >= p.N) continue;
            const int ncnt = p.N - nb;  // columns to write in this chunk (a multiple of 8; may exceed 32)
            if (p.bias) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (j < ncnt) {
                        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + nb + j));
                        v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
                    }
                }
            }
            if (p.res_hi) {
                const __half* rh = p.res_hi + static_cast<long long>(row) * p.res_ld + nb;
                const __half* rl = p.res_lo + static_cast<long long>(row) * p.res_ld + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    if (j < ncnt) {
                        const uint4 uh = *reinterpret_cast<const uint4*>(rh + j);
                        const uint4 ul = *reinterpret_cast<const uint4*>(rl + j);
                        const __half2* hh = reinterpret_cast<const __half2*>(&uh);
                        const __half2* hl = reinterpret_cast<const __half2*>(&ul);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float2 a = __half22float2(hh[q]);
                            const float2 b = __half22float2(hl[q]);
                            v[j + 2 * q] += a.x + b.x;
                            v[j + 2 * q + 1] += a.y + b.y;
                        }
                    }
                }
            }
            if (p.addend && p.addend_mode == 1) {
                const float* ad = p.addend + static_cast<long long>(n_img) * p.N + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (j < ncnt) {
                        const float4 a4 = __ldg(reinterpret_cast<const float4*>(ad + j));
                        v[j] += a4.x; v[j + 1] += a4.y; v[j + 2] += a4.z; v[j + 3] += a4.w;
                    }
                }
            }
            if (p.relu == 1) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            } else if (p.relu == 2) {  // LeakyReLU(0.01) of the FPN fine branch (resnet_fpn.py:63,70)
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] : 0.01f * v[j];
            }
            if (p.out_hi) {
                __half* oh = p.out_hi + obase + orow * p.out_ld + nb;
                __half* ol = p.out_lo ? p.out_lo + obase + orow * p.out_ld + nb : nullptr;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    if (j < ncnt) {
                        uint4 uh, ul;
                        __half* hh = reinterpret_cast<__half*>(&uh);
                        __half* hl = reinterpret_cast<__half*>(&ul);
#pragma unroll
                        for (int q = 0; q < 8; ++q) split_f16(v[j + q], hh[q], hl[q]);
                        *reinterpret_cast<uint4*>(oh + j) = uh;
                        if (ol) *reinterpret_cast<uint4*>(ol + j) = ul;
                    }
                }
            }
            if (p.addend && p.addend_mode == 0) {
                const float* ad = p.addend + static_cast<long long>(y * p.g.W + x) * p.N + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (j < ncnt) {
                        const float4 a4 = __ldg(reinterpret_cast<const float4*>(ad + j));
                        v[j] += a4.x; v[j + 1] += a4.y; v[j + 2] += a4.z; v[j + 3] += a4.w;
                    }
                }
            }
            if (out_f32) {
                float* of = out_f32 + orow * p.out_f32_ld + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (j < ncnt) *reinterpret_cast<float4*>(of + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
        }
    }
};


// ---------------------------------------------------------------------------- transformer linear epilogues
enum LinMode : int {
    LIN_F32_ELU = 0,   // fp32 out; elu(x)+1 on output columns < elu_cols (q/k feature map of linear attention)
    LIN_RELU_HL = 1,   // relu -> split-fp16 planes
    LIN_LN = 2,        // LayerNorm over the full row (BN == d_model) [+ residual] -> fp32 and/or split-fp16 planes
    LIN_QZ = 3,        // q projection of linear attention: Q = elu(q)+1, z = 1/(Q . Ksum_head + eps) per 32-wide head, out = Q*z -> planes
};

struct LinEpiParams {
    int M, N;
    int mode;
    int elu_cols;
    const float* gamma;  // LIN_LN
    const float* beta;
    const float* resid;  // LIN_LN: optional fp32 residual x (out = x + LN(acc)) ...
    int resid_ld;
    const __half* res_hi;  // ... or the residual as split-fp16 planes (x = hi + lo; engine 2 only), row pitch res_ld
    const __half* res_lo;
    int res_ld;
    float* out_f32;
    int out_f32_ld;
    int out_col0;        // column offset added to n for the fp32 output
    const float* ksum;   // LIN_QZ: [segments][N] sum over the source tokens of elu(k)+1 (linear_attention.py:43)
    int seg_row0;        // LIN_QZ: rows >= seg_row0 belong to segment 1 (ksum + N); 0 = single segment
    float qz_scale[2];   // LIN_QZ: per segment, the source length v_length (linear_attention.py:39,45): Q*Z*len is O(1) -- without it the
                         //   values (~1/len) would sink into the fp16 subnormals of the split planes
    __half* out_hi;
    __half* out_lo;
    int out_ld;
#ifdef DFSFM_LIN_DEBUG
    int dbg;             // tuning builds only (-DDFSFM_LIN_DEBUG, env DFSFM_LIN_DBG): 1 no global stores, 4 no LN statistics pass, 8 no column blocks
#endif
};
#ifdef DFSFM_LIN_DEBUG
#define DFSFM_DBG(p, bit) ((p).dbg & (bit))
#else
#define DFSFM_DBG(p, bit) false
#endif

struct LinEpi {
    using Params = LinEpiParams;
    static constexpr bool kHasState = false;
    static constexpr bool kSeparateCorr = false;
    static constexpr int kEpiStageBytes = 4096;  // engine 2: one 32 x 32 fp32 block per epilogue warp
    template <int BN, int kCorr>
    static __device__ __forceinline__ void run(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, int ce, int part_idx,
                                               const EpiCtx& ctx) {
        if constexpr (kCorr == 0) {  // engine 2 (engine 1 keeps a separate correction accumulator and has no staging buffers)
            if (DFSFM_DBG(p, 8)) return;
            // generic fallback (the engines launch the LinEpiS specialisations instead, see launch_gemm_counted)
            if (p.mode == LIN_LN) {
                if (p.resid != nullptr) run_ln_staged<BN, 1>(p, tmem_warp, row0, lane, n0, cb, ctx);
                else if (p.res_hi != nullptr) run_ln_staged<BN, 2>(p, tmem_warp, row0, lane, n0, cb, ctx);
                else run_ln_staged<BN, 0>(p, tmem_warp, row0, lane, n0, cb, ctx);
            } else if (p.mode == LIN_RELU_HL) {
                run_plain_staged<LIN_RELU_HL>(p, tmem_warp, row0, lane, n0, cb, ce, ctx);
            } else {
                run_plain_staged<LIN_F32_ELU>(p, tmem_warp, row0, lane, n0, cb, ce, ctx);
            }
            return;
        }
        const int row = row0 + lane;
        const bool valid = row < p.M;
        float mean = 0.f, rstd = 0.f;
        if (p.mode == LIN_LN) {
            // one statistics pass over this thread's TMEM row (BN == N == d_model): shifted sums about the first element
            float s1 = 0.f, s2 = 0.f, pivot = 0.f;
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                float v[32];
                load_acc32<kCorr>(tmem_warp + c0, v);
                if (c0 == 0) pivot = v[0];
#pragma unroll
                for (int j = 0; j < 32; ++j) { const float d = v[j] - pivot; s1 += d; s2 = fmaf(d, d, s2); }
            }
            const float inv_n = 1.f / static_cast<float>(BN);
            const float md = s1 * inv_n;
            mean = pivot + md;
            rstd = rsqrtf(fmaxf(s2 * inv_n - md * md, 0.f) + 1e-5f);
        }
#pragma unroll 1
        for (int c0 = cb; c0 < ce; c0 += 32) {
            float v[32];
            load_acc32<kCorr>(tmem_warp + c0, v);
            const int nb = n0 + c0;
            if (!valid || nb >= p.N) continue;
            if (p.mode == LIN_F32_ELU) {
                if (nb < p.elu_cols) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] + 1.f : fast_ex2(v[j] * 1.4426950408889634f);  // elu(x) + 1 == exp(x), x <= 0
                }
            } else if (p.mode == LIN_RELU_HL) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            } else {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.gamma + nb + j));
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.beta + nb + j));
                    v[j] = (v[j] - mean) * rstd * g4.x + b4.x;
                    v[j + 1] = (v[j + 1] - mean) * rstd * g4.y + b4.y;
                    v[j + 2] = (v[j + 2] - mean) * rstd * g4.z + b4.z;
                    v[j + 3] = (v[j + 3] - mean) * rstd * g4.w + b4.w;
                }
                if (p.resid) {
                    const float* rr = p.resid + static_cast<long long>(row) * p.resid_ld + nb;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 r4 = *reinterpret_cast<const float4*>(rr + j);
                        v[j] += r4.x; v[j + 1] += r4.y; v[j + 2] += r4.z; v[j + 3] += r4.w;
                    }
                }
            }
            if (p.out_f32) {
                float* of = p.out_f32 + static_cast<long long>(row) * p.out_f32_ld + p.out_col0 + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(of + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            }
            if (p.out_hi) {
                __half* oh = p.out_hi + static_cast<long long>(row) * p.out_ld + nb;
                __half* ol = p.out_lo + static_cast<long long>(row) * p.out_ld + nb;
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    uint4 uh, ul;
                    __half* hh = reinterpret_cast<__half*>(&uh);
                    __half* hl = reinterpret_cast<__half*>(&ul);
#pragma unroll
                    for (int q = 0; q < 8; ++q) split_f16(v[j + q], hh[q], hl[q]);
                    *reinterpret_cast<uint4*>(oh + j) = uh;
                    *reinterpret_cast<uint4*>(ol + j) = ul;
                }
            }
        }
    }

    // Engine-2 paths.  A thread owns one accumulator ROW (a TMEM lane), so writing results straight from registers makes every
    // warp-wide store touch 32 different cache lines (one per row): the L1 tag stage then costs 32 cycles per instruction and
    // the short-K linears become epilogue-bound.  Here each 32 x 32 block is transposed through a 4 KB swizzled staging
    // buffer (16-byte chunk index XOR row % 8: conflict-free both ways); afterwards lane l owns columns 4*(l%8)..+3 of rows
    // 4*i + l/8, i = 0..7, so a warp-wide access covers four full 128-byte rows -- residual loads and all stores coalesce.
    // The epilogue is instruction-issue bound (two warps per scheduler), hence the packed conversions and folded FMAs.
    struct Blk {  // per-lane geometry of the transposed ("coalesced") domain
        int ch, rsub;
    };
    static __device__ __forceinline__ void stage_rows(uint8_t* stg, int lane, const float* v) {
        uint8_t* st_row = stg + lane * 128;
        const int sw = lane & 7;
#pragma unroll
        for (int q = 0; q < 8; ++q) *reinterpret_cast<float4*>(st_row + ((q ^ sw) << 4)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
    static __device__ __forceinline__ float4 unstage(const uint8_t* stg, int rl, int ch) {
        return *reinterpret_cast<const float4*>(stg + rl * 128 + ((ch ^ (rl & 7)) << 4));
    }
    static __device__ __forceinline__ void store_out(const Params& p, int r, int col, const float4& w) {
        if (DFSFM_DBG(p, 1)) return;
        if (p.out_f32) *reinterpret_cast<float4*>(p.out_f32 + static_cast<long long>(r) * p.out_f32_ld + p.out_col0 + col) = w;
        if (p.out_hi) {
            uint2 uh, ul;
            split_f16x2(w.x, w.y, uh.x, ul.x);
            split_f16x2(w.z, w.w, uh.y, ul.y);
            const long long o = static_cast<long long>(r) * p.out_ld + col;
            *reinterpret_cast<uint2*>(p.out_hi + o) = uh;
            *reinterpret_cast<uint2*>(p.out_lo + o) = ul;
        }
    }

    // LIN_F32_ELU / LIN_RELU_HL: block by block.  Loops stay rolled: the epilogue warps walk this code once per tile, and
    // straight-line code of tens of KB turns instruction fetch into the bottleneck.
    template <int kMode>
    static __device__ __forceinline__ void run_plain_staged(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, int ce,
                                                            const EpiCtx& ctx) {
        const int ch = lane & 7, rsub = lane >> 3;
#pragma unroll 1
        for (int c0 = cb; c0 < ce; c0 += 32) {
            const int nb = n0 + c0;
            if (nb >= p.N) break;  // warp-uniform
            const int col = nb + 4 * ch;
            float v[32];
            load_acc32<0>(tmem_warp + c0, v);
            if (kMode == LIN_QZ) {
                // this thread holds one head (32 columns) of its row: the normaliser Z of linear_attention.py:43 is row-local.
                // The message is then msg = (Q*Z) . KV, folded with the merge projection into one GEMM against G = len * KV . Wm^T.
                const int sg = (p.seg_row0 > 0 && row0 + lane >= p.seg_row0) ? 1 : 0;
                const float* ks = p.ksum + sg * p.N + nb;
                float dot = 0.f;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 k4 = __ldg(reinterpret_cast<const float4*>(ks + j));
                    v[j] = v[j] > 0.f ? v[j] + 1.f : fast_ex2(v[j] * 1.4426950408889634f);
                    v[j + 1] = v[j + 1] > 0.f ? v[j + 1] + 1.f : fast_ex2(v[j + 1] * 1.4426950408889634f);
                    v[j + 2] = v[j + 2] > 0.f ? v[j + 2] + 1.f : fast_ex2(v[j + 2] * 1.4426950408889634f);
                    v[j + 3] = v[j + 3] > 0.f ? v[j + 3] + 1.f : fast_ex2(v[j + 3] * 1.4426950408889634f);
                    dot = fmaf(v[j], k4.x, dot); dot = fmaf(v[j + 1], k4.y, dot); dot = fmaf(v[j + 2], k4.z, dot); dot = fmaf(v[j + 3], k4.w, dot);
                }
                const float z = p.qz_scale[sg] / (dot + 1e-6f);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] *= z;
            }
            stage_rows(ctx.stg, lane, v);
            __syncwarp();
            const bool elu = kMode == LIN_F32_ELU && nb < p.elu_cols;
#pragma unroll 2
            for (int i = 0; i < 8; ++i) {
                const int rl = 4 * i + rsub;
                const int r = row0 + rl;
                float4 w = unstage(ctx.stg, rl, ch);
                if (r >= p.M) continue;
                if (kMode == LIN_RELU_HL) {
                    w.x = fmaxf(w.x, 0.f); w.y = fmaxf(w.y, 0.f); w.z = fmaxf(w.z, 0.f); w.w = fmaxf(w.w, 0.f);
                } else if (elu) {
                    w.x = w.x > 0.f ? w.x + 1.f : fast_ex2(w.x * 1.4426950408889634f);  // elu(x) + 1 == exp(x), x <= 0
                    w.y = w.y > 0.f ? w.y + 1.f : fast_ex2(w.y * 1.4426950408889634f);
                    w.z = w.z > 0.f ? w.z + 1.f : fast_ex2(w.z * 1.4426950408889634f);
                    w.w = w.w > 0.f ? w.w + 1.f : fast_ex2(w.w * 1.4426950408889634f);
                }
                store_out(p, r, col, w);
            }
            __syncwarp();
        }
    }

    // LIN_LN (BN == N == d_model; this warp owns BN/2 columns of 32 rows, its partner warp the other half).  One TMEM pass: the
    // half-row stays in registers, the two warps exchange (mean, sum of squared deviations) of their halves through shared
    // memory, then each normalises, transposes and writes its own columns.  TMEM reads run at 64 B/clk/SM, so reading the
    // tile once instead of three times (statistics by both warps + output) is worth ~2 us per tile.
    // residual of row r, 4 columns at col, in the transposed domain: fp32 bits, or {hi.x, hi.y, lo.x, lo.y} of the split planes
    template <int kRes>
    static __device__ __forceinline__ uint4 load_resid(const Params& p, int r, int col) {
        uint4 q = make_uint4(0u, 0u, 0u, 0u);
        if (r < p.M) {
            if (kRes == 1) {
                q = *reinterpret_cast<const uint4*>(p.resid + static_cast<long long>(r) * p.resid_ld + col);
            } else if (kRes == 2) {
                const long long o = static_cast<long long>(r) * p.res_ld + col;
                const uint2 h = *reinterpret_cast<const uint2*>(p.res_hi + o);
                const uint2 l = *reinterpret_cast<const uint2*>(p.res_lo + o);
                q = make_uint4(h.x, h.y, l.x, l.y);
            }
        }
        return q;
    }
    // transposed phase of one LN block: rows 4i + rsub, i = 0..7.  q[] holds the residual of four rows: on entry rows 0..3 of this
    // block; an entry is reloaded as soon as it has been consumed -- with row i + 4 of this block, then with rows 0..3 of the
    // next block (col_next >= 0) -- so a residual load has four rows' worth of work to hide behind.
    template <int kRes>  // 0: none, 1: fp32 residual, 2: split-fp16 residual
    static __device__ __forceinline__ void ln_block_out(const Params& p, const EpiCtx& ctx, int row0, int rsub, int ch, int col, int col_next,
                                                        uint4 (&q)[4]) {
        constexpr bool has_res = kRes != 0;
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.gamma + col));
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.beta + col));
#pragma unroll 1
        for (int g = 0; g < 2; ++g) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int rl = 4 * (4 * g + k) + rsub;
                const int r = row0 + rl;
                float4 w = unstage(ctx.stg, rl, ch);
                w.x = fmaf(w.x, g4.x, b4.x); w.y = fmaf(w.y, g4.y, b4.y); w.z = fmaf(w.z, g4.z, b4.z); w.w = fmaf(w.w, g4.w, b4.w);
                if (has_res) {
                    const uint4 qc = q[k];
                    if (g == 0) q[k] = load_resid<kRes>(p, r + 16, col);
                    else if (col_next >= 0) q[k] = load_resid<kRes>(p, r - 16, col_next);
                    if (kRes == 1) {
                        w.x += __uint_as_float(qc.x); w.y += __uint_as_float(qc.y); w.z += __uint_as_float(qc.z); w.w += __uint_as_float(qc.w);
                    } else {
                        add_f16x2(w.x, w.y, qc.z); add_f16x2(w.z, w.w, qc.w);
                        add_f16x2(w.x, w.y, qc.x); add_f16x2(w.z, w.w, qc.y);
                    }
                }
                if (r < p.M) store_out(p, r, col, w);
            }
        }
    }
    template <int BN, int kRes>
    static __device__ __forceinline__ void run_ln_staged(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, const EpiCtx& ctx) {
        constexpr int NB = BN / 64;       // 32-column blocks per warp
        constexpr int NV = 32 * NB;       // columns per warp
        constexpr bool has_res = kRes != 0;
        const int ch = lane & 7, rsub = lane >> 3;
        float v[NV];
#pragma unroll
        for (int b = 0; b < NB; ++b) tmem_ld32(tmem_warp + cb + 32 * b, v + 32 * b);
        uint4 q[4];
        if (has_res) {  // residual of the first four rows of block 0: in flight behind the TMEM read and the statistics
#pragma unroll
            for (int k = 0; k < 4; ++k) q[k] = load_resid<kRes>(p, row0 + 4 * k + rsub, n0 + cb + 4 * ch);
        }
        tmem_ld_wait();
        float scale = 1.f, shift = 0.f;
        if (!DFSFM_DBG(p, 4)) {
            // half-row statistics about the first element (no cancellation), then Chan's combination of the two halves
            const float pivot = v[0];
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int j = 0; j < NV; ++j) { const float d = v[j] - pivot; s1 += d; s2 = fmaf(d, d, s2); }
            const float inv_h = 1.f / static_cast<float>(NV);
            const float m_own = pivot + s1 * inv_h;
            const float q_own = fmaxf(s2 - s1 * s1 * inv_h, 0.f);
            *reinterpret_cast<float2*>(ctx.stg + lane * 8) = make_float2(m_own, q_own);
            named_bar_sync(ctx.bar_id, 64);
            const float2 o = *reinterpret_cast<const float2*>(ctx.stg_partner + lane * 8);
            named_bar_sync(ctx.bar_id, 64);  // the partner has read our slot: the staging buffer may be overwritten
            const float mean = 0.5f * (m_own + o.x);
            const float dm = m_own - o.x;
            const float var = (q_own + o.y + 0.5f * static_cast<float>(NV) * dm * dm) * (1.f / static_cast<float>(BN));
            scale = rsqrtf(var + 1e-5f);
            shift = -mean * scale;
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            float* vb = v + 32 * b;
#pragma unroll
            for (int j = 0; j < 32; ++j) vb[j] = fmaf(vb[j], scale, shift);
            stage_rows(ctx.stg, lane, vb);
            __syncwarp();
            const int col = n0 + cb + 32 * b + 4 * ch;
            ln_block_out<kRes>(p, ctx, row0, rsub, ch, col, b + 1 < NB ? col + 32 : -1, q);
            __syncwarp();
        }
    }
};

// Engine-2 specialisations: one kernel per (mode, residual flavour).  The epilogue warps walk their code once per tile, so the
// instruction footprint matters (a kernel holding every variant measured 2x slower epilogues than one holding just its own).
template <int kMode, int kRes>
struct LinEpiS {
    using Params = LinEpiParams;
    static constexpr bool kHasState = false;
    static constexpr bool kSeparateCorr = false;
    static constexpr int kEpiStageBytes = LinEpi::kEpiStageBytes;
    template <int BN, int kCorr>
    static __device__ __forceinline__ void run(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, int ce, int part_idx,
                                               const EpiCtx& ctx) {
        static_assert(kCorr == 0, "engine 2 only");
        if (DFSFM_DBG(p, 8)) return;
        if (kMode == LIN_LN) LinEpi::run_ln_staged<BN, kRes>(p, tmem_warp, row0, lane, n0, cb, ctx);
        else LinEpi::run_plain_staged<kMode>(p, tmem_warp, row0, lane, n0, cb, ce, ctx);
    }
};

// ------------------------------------------------------------------- k/v projection + linear-attention state (engine 2 only)
// The source tokens' k, v projection with the state reduction of linear_attention.py:40-42 folded into the epilogue:
//     KV[h][d][v] = sum_s (elu(k[s,h,d]) + 1) * v[s,h,v],      Ksum[h][d] = sum_s (elu(k[s,h,d]) + 1)
// k and v never reach HBM.  The weight rows are packed so that one 256-column tile holds [K of heads 4t..4t+3 | V of the same heads]
// (packing.py "kvp"): the warp that owns columns [0,128) of a lane quadrant holds four 32x32 K blocks, its partner warp the matching V
// blocks.  Per head both blocks go through the per-warp staging buffers and the 64 threads of the pair accumulate the 32x32 outer-
// product sum over their 32 rows in registers (thread = (d, 16 of the v)); the accumulators live across all tiles of the persistent
// CTA and are combined over the four lane quadrants through shared memory in a fixed order when the CTA is done with a
// (segment, column-tile) -- deterministic.  A second tiny kernel (kv_state_final_kernel) adds the per-CTA partials.
struct KvEpiParams {
    int M;
    int seg_row0;      // rows >= seg_row0 (a multiple of 256) belong to segment 1; 0 = one segment
    int row_begin[2];  // valid rows of a segment: [row_begin, row_end) in launch-relative rows (padding rows contribute nothing)
    int row_end[2];
    float* part;       // [2 segments][2 column tiles][gridDim.x CTAs][4 heads * 32 * 33]
    unsigned* flags;   // [2][2][gridDim.x]: == epoch when the slot was written by this launch
    unsigned epoch;
};
constexpr int kKvPartFloats = 4 * 32 * 33;

struct KvEpi {
    using Params = KvEpiParams;
    static constexpr bool kHasState = true;
    static constexpr bool kSeparateCorr = false;
    static constexpr int kEpiStageBytes = 4096;
    // Register tile of a thread: 4 d x 4 v of each head's 32 x 32 outer-product sum (lane = (dq, vq): d = 4*dq + i, v = 16*half + 4*vq + j).
    // Per staged row a thread then loads ONE 16-byte K unit and ONE 16-byte V unit for 16 FMAs -- a 128-bit shared load costs four
    // wavefronts per warp whatever the addresses, so the (1 d x 16 v) tile of the first version (five loads per 16 FMAs, 17 wavefronts
    // per row) made the epilogue LSU-bound at ~15 us per tile (profiles/r02_timeline_fused.log); this layout needs 8.
    // Tried and measured slower: the same reduction as a warp-level tensor-core product (mma.sync m16n8k8 tf32, split hi + lo, conflict-free
    // fragment loads; commit 'KvEpi: the K^T V state reduction on warp-level tf32 tensor-core MMAs', parity green) -- 16 us per tile instead
    // of 8.9: the legacy HMMA.1688.TF32 path of sm_100 issues at ~20 clocks per instruction per SM here, far below the FFMA rate it replaces.
    struct State {
        float acc[4][16];
        float ks[4][4];
        int seg, nt;
    };
    static __device__ __forceinline__ void reset(State& st) {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
#pragma unroll
            for (int j = 0; j < 4; ++j) st.ks[h][j] = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) st.acc[h][j] = 0.f;
        }
    }
    static __device__ __forceinline__ void init(State& st) {
        reset(st);
        st.seg = -1;
        st.nt = -1;
    }
    // combine the four quadrant pairs of this CTA in quadrant order and write the partial of (st.seg, st.nt)
    static __device__ __forceinline__ void flush(const Params& p, State& st, int lane, int half, int quad, uint8_t* epi_smem) {
        float* red = reinterpret_cast<float*>(epi_smem);  // 16.5 KB of the 32 KB staging area
        const int dq = lane >> 2, vq = lane & 3;
        named_bar_sync(5, 32 * kGemm2EpiWarps);
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            if (quad == q) {
#pragma unroll
                for (int h = 0; h < 4; ++h) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float* r = red + (h * 32 + dq * 4 + i) * 33;
#pragma unroll
                        for (int j = 0; j < 4; ++j) r[half * 16 + vq * 4 + j] = (q == 0 ? 0.f : r[half * 16 + vq * 4 + j]) + st.acc[h][4 * i + j];
                        if (half == 0 && vq == 0) r[32] = (q == 0 ? 0.f : r[32]) + st.ks[h][i];
                    }
                }
            }
            named_bar_sync(5, 32 * kGemm2EpiWarps);
        }
        const long long slot = (static_cast<long long>(st.seg * 2 + st.nt) * gridDim.x + blockIdx.x);
        float* o = p.part + slot * kKvPartFloats;
        const int t = (half * 4 + quad) * 32 + lane;
        for (int i = t; i < kKvPartFloats; i += 32 * kGemm2EpiWarps) o[i] = red[i];
        if (t == 0) p.flags[slot] = p.epoch;
        named_bar_sync(5, 32 * kGemm2EpiWarps);
        reset(st);
    }
    template <int BN>
    static __device__ __forceinline__ void run_state(const Params& p, State& st, uint32_t tmem_warp, int row0, int lane, int nt, int half, int quad,
                                                     const EpiCtx& ctx, uint8_t* epi_smem) {
        static_assert(BN == 256, "KvEpi tiles are [4 K heads | 4 V heads]");
        const int seg = (p.seg_row0 > 0 && row0 >= p.seg_row0) ? 1 : 0;
        if (st.seg != seg || st.nt != nt) {  // uniform over the CTA's epilogue warps (same tile sequence)
            if (st.seg >= 0) flush(p, st, lane, half, quad, epi_smem);
            st.seg = seg;
            st.nt = nt;
        }
        const int row = row0 + lane;
        const bool valid = row >= p.row_begin[seg] && row < p.row_end[seg];
        const uint8_t* kst = half == 0 ? ctx.stg : ctx.stg_partner;
        const uint8_t* vst = half == 0 ? ctx.stg_partner : ctx.stg;
        const int dq = lane >> 2, vch = half * 4 + (lane & 3);
#pragma unroll
        for (int h = 0; h < 4; ++h) {  // unrolled: the per-head accumulators must stay in registers
            float v[32];
            load_acc32<0>(tmem_warp + half * 128 + h * 32, v);
            if (half == 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float e = v[j] > 0.f ? v[j] + 1.f : fast_ex2(v[j] * 1.4426950408889634f);  // elu(x) + 1
                    v[j] = valid ? e : 0.f;
                }
            }
            LinEpi::stage_rows(ctx.stg, lane, v);
            named_bar_sync(ctx.bar_id, 64);
            float a[16], k0 = st.ks[h][0], k1 = st.ks[h][1], k2 = st.ks[h][2], k3 = st.ks[h][3];
#pragma unroll
            for (int j = 0; j < 16; ++j) a[j] = st.acc[h][j];
#pragma unroll 8
            for (int r = 0; r < 32; ++r) {
                const float4 k = LinEpi::unstage(kst, r, dq);
                const float4 w = LinEpi::unstage(vst, r, vch);
                k0 += k.x; k1 += k.y; k2 += k.z; k3 += k.w;
                a[0] = fmaf(k.x, w.x, a[0]);   a[1] = fmaf(k.x, w.y, a[1]);   a[2] = fmaf(k.x, w.z, a[2]);   a[3] = fmaf(k.x, w.w, a[3]);
                a[4] = fmaf(k.y, w.x, a[4]);   a[5] = fmaf(k.y, w.y, a[5]);   a[6] = fmaf(k.y, w.z, a[6]);   a[7] = fmaf(k.y, w.w, a[7]);
                a[8] = fmaf(k.z, w.x, a[8]);   a[9] = fmaf(k.z, w.y, a[9]);   a[10] = fmaf(k.z, w.z, a[10]); a[11] = fmaf(k.z, w.w, a[11]);
                a[12] = fmaf(k.w, w.x, a[12]); a[13] = fmaf(k.w, w.y, a[13]); a[14] = fmaf(k.w, w.z, a[14]); a[15] = fmaf(k.w, w.w, a[15]);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) st.acc[h][j] = a[j];
            st.ks[h][0] = k0; st.ks[h][1] = k1; st.ks[h][2] = k2; st.ks[h][3] = k3;
            named_bar_sync(ctx.bar_id, 64);  // both warps are done reading the staged blocks
        }
    }
    static __device__ __forceinline__ void finish(const Params& p, State& st, int lane, int half, int quad, uint8_t* epi_smem) {
        if (st.seg >= 0) flush(p, st, lane, half, quad, epi_smem);
    }
};

// ------------------------------------------------------------------- dual-softmax similarity epilogues
// t[i,j] = acc[i,j] * c2 with c2 = log2(e) / (d_model * temperature): the similarity in the log2 domain, so that every
// exponential is one ex2.  SIM_STATS: per-row (max, sum 2^(t-max)) over this warp's columns -> part[part_idx][row].
// SIM_CONF: conf = softmax_row * softmax_col = 2^(2t - lse_row - lse_col) with lse = max + log2(sum) from the merged
// statistics; every entry above thr competes for its row's and its column's best (64-bit atomicMax on (conf bits, ~index)).
enum SimMode : int { SIM_STATS = 0, SIM_CONF = 1 };

struct SimEpiParams {
    int M, N;       // rows (tokens of A), columns (tokens of B)
    int mode;
    float c2;       // log2(e) / (d_model * temperature)
    float2* part;   // SIM_STATS: [partial tiles][M] (max, sum) in the log2 domain
    const float* row_lse;  // SIM_CONF: [M] log2-sum-exp2 of the row
    const float* col_lse;  // SIM_CONF: [N]
    float thr;
    float lthr;     // SIM_CONF: screening bound, a margin below log2(thr) (-inf when thr < 0: every entry is a candidate)
    unsigned long long* row_best;  // [M]
    unsigned long long* col_best;  // [N]
    float* conf_out;               // optional dense [M][N] (debug / small problems)
};

__device__ __forceinline__ unsigned long long pack_best(float conf, int idx) {
    return (static_cast<unsigned long long>(__float_as_uint(conf)) << 32) | static_cast<unsigned int>(0x7fffffff - idx);
}

struct SimEpi {
    using Params = SimEpiParams;
    static constexpr bool kHasState = false;
    static constexpr bool kSeparateCorr = false;
    static constexpr int kEpiStageBytes = 0;
    template <int BN, int kCorr>
    static __device__ __forceinline__ void run(const Params& p, uint32_t tmem_warp, int row0, int lane, int n0, int cb, int ce, int part_idx, const EpiCtx& ctx) {
        const int row = row0 + lane;
        const bool valid = row < p.M;
        if (p.mode == SIM_STATS) {
            float m = -INFINITY, s = 0.f;
#pragma unroll 1
            for (int c0 = cb; c0 < ce; c0 += 32) {
                float v[32];
                load_acc32<kCorr>(tmem_warp + c0, v);
                const int nb = n0 + c0;
                if (nb >= p.N) continue;
                if (nb + 32 <= p.N) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] *= p.c2;
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = (nb + j < p.N) ? v[j] * p.c2 : -INFINITY;
                }
                float m0 = fmaxf(v[0], v[1]), m1 = fmaxf(v[2], v[3]), m2 = fmaxf(v[4], v[5]), m3 = fmaxf(v[6], v[7]);
#pragma unroll
                for (int j = 8; j < 32; j += 4) {
                    m0 = fmaxf(m0, v[j]); m1 = fmaxf(m1, v[j + 1]); m2 = fmaxf(m2, v[j + 2]); m3 = fmaxf(m3, v[j + 3]);
                }
                const float cm = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
                if (cm > m) { s *= fast_ex2(m - cm); m = cm; }
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    s0 += fast_ex2(v[j] - m); s1 += fast_ex2(v[j + 1] - m); s2 += fast_ex2(v[j + 2] - m); s3 += fast_ex2(v[j + 3] - m);
                }
                s += (s0 + s1) + (s2 + s3);
            }
            if (valid) p.part[static_cast<long long>(part_idx) * p.M + row] = make_float2(m, s);
        } else {
            const float a_row = valid ? p.row_lse[row] : 0.f;
            const float c22 = 2.f * p.c2;
            // screening bound in the log2 domain: conf > thr  =>  2t - lse_row - lse_col > lthr (lthr sits a margin below log2(thr),
            // so rounding differences between the screening and the exact expression below cannot lose a candidate)
            const float row_bound = valid ? p.lthr + a_row : INFINITY;
            float best = -1.f;
            int best_j = 0;
#pragma unroll 1
            for (int c0 = cb; c0 < ce; c0 += 32) {
                float v[32];
                load_acc32<kCorr>(tmem_warp + c0, v);
                const int nb = n0 + c0;
                if (nb >= p.N) continue;
                // lane j holds the column term of column nb + j; +inf for columns past N makes their confidence 0.  (Warp-uniform 16-byte
                // loads of the 32 terms per thread instead of the shuffles measured SLOWER: 12.4 vs 11.0 ms per 28 pairs.)
                const float b_col = (nb + lane < p.N) ? __ldg(p.col_lse + nb + lane) : INFINITY;
                float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    m0 = fmaxf(m0, fmaf(v[j], c22, -__shfl_sync(0xffffffffu, b_col, j)));
                    m1 = fmaxf(m1, fmaf(v[j + 1], c22, -__shfl_sync(0xffffffffu, b_col, j + 1)));
                    m2 = fmaxf(m2, fmaf(v[j + 2], c22, -__shfl_sync(0xffffffffu, b_col, j + 2)));
                    m3 = fmaxf(m3, fmaf(v[j + 3], c22, -__shfl_sync(0xffffffffu, b_col, j + 3)));
                }
                const bool cand = (fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) > row_bound && valid) || (p.conf_out != nullptr && valid);
                if (!__any_sync(0xffffffffu, cand)) continue;  // almost every 32 x 32 block: nothing above the threshold
#pragma unroll 4
                for (int j = 0; j < 32; ++j) {
                    const float bj = __shfl_sync(0xffffffffu, b_col, j);
                    if (!cand) continue;
                    const float conf = ex2_denorm(fmaf(v[j], c22, -a_row) - bj);
                    if (p.conf_out && nb + j < p.N) p.conf_out[static_cast<long long>(row) * p.N + nb + j] = conf;
                    if (conf > p.thr) {
                        atomicMax(p.col_best + nb + j, pack_best(conf, row));
                        if (conf > best) { best = conf; best_j = nb + j; }
                    }
                }
            }
            if (valid && best >= 0.f) atomicMax(p.row_best + row, pack_best(best, best_j));
        }
    }
};

}  // namespace dfsfm
