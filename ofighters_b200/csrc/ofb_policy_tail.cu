// The pointer head's tail as ONE persistent tcgen05 kernel (sm_100a):
//     UpSampling2D -> Conv(4 -> 8) -> BN -> ReLU -> UpSampling2D -> Conv(8 -> 1) -> argmax      (agents/qlearnIA_V2.py:176-186, :218-220)
// upconv3's 200 x 200 x 8 output never leaves the SM: it is drained from TMEM to bf16 into a ring of shared-memory
// planes that upconv4's block-Toeplitz MMAs read as their A operand; only (x, y) -- 8 bytes per ship -- goes back to HBM.
//
// One "M row" m = i * 26 + xb is a block of 4 pixels (4 xb .. 4 xb + 3) of row i of the 100 x 100 input (xb = 25 is a dummy
// row that keeps a halo slot between image rows); a ship is 2600 M rows = 21 tiles of 128.  BOTH convolutions use the same
// M rows, so the data flows tile by tile with no strips and no recomputed halo:
//   upconv3 (bilinear x2 folded into 4 phases): K = the 6 input pixels x 4 channels the block depends on (+ 8 spare lanes
//     that carry the left / right image-border correction), N = 4 px x 4 phases x 8 channels = 128; 3 vertical taps x 2
//     K-steps = 6 MMAs per tile.  Its output for M row m is the 2 x 8 pixels (Y = 2i + a, X = 8 xb + q) x 8 channels:
//     sixteen 16-byte chunks, stored in plane (a, q) of the ring at row m.
//   upconv4 ("2-row form"): M row m produces the 4 x 16 output pixels (V = 4i .. 4i+3, Z = 16 xb .. 16 xb + 15) from the
//     4 upconv3 rows 2i-1 .. 2i+2 x 10 pixels x 8 channels: 4 vertical taps x 5 K-steps = 20 MMAs with N = 64 (+ 16 columns
//     of border variants, see below).  A vertical tap is the descriptor shifted by +-26 ring rows in the plane of the other
//     parity, a horizontal neighbour the plane of x mod 8 +- 1 (the row's halo slots hold the replicated edge pixels).
//   Its tiles lag 32 M rows behind upconv3's, so that tile t needs the drains of tiles <= t only and a ring of 3 tiles
//     (+ a 64-row mirror in front of it, which makes the wrap-around contiguous for the descriptors) is enough.
// Image borders.  The folded form assumes a replicate-extended input, the convolutions zero-pad their (upsampled) input.
// The true border values are the same contraction with other weights, so they are extra N columns / small extra MMAs, not
// a scalar pass:  upconv3 left / right: 8 spare K lanes carry L[i][0] / L[i][99] with weights that cancel the out-of-range
// taps; upconv3 top / bottom (tiles 0 / 20 only): 4 extra N = 64 MMAs into their own TMEM columns; upconv4 left / right: 8
// extra columns in every MMA (free: these MMAs are bound by reading A); upconv4 top / bottom: 10 extra N = 16 MMAs on
// tiles 0 / 20; the 4 corner pixels of the 400 x 400 map are 32 MACs each in the draining thread that owns them.
// Warp roles: 0-3 / 4-7 drain upconv3's even / odd tiles (TMEM -> +bias, ReLU, bf16 -> ring), 8-11 drain upconv4 (running
// maximum, index recovered only when a value reaches the ship's best so far), 12 bulk-copies the input tiles, 13 / 14 issue
// the MMAs of upconv3 / upconv4.
#include "ofb_common.cuh"
#include "ofb_policy_dev.cuh"
#include "ofb_tc_ptx.cuh"
#include "ofb_policy_tail.cuh"

__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t *r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void named_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// order-preserving map float -> int (for an atomic maximum on values of either sign).  It orders -0.0 below +0.0; the keys are
// taken on v + bias4 with a bias4 that is never -0.0 (pol_tz_tail), and x + (+0.0) is never -0.0.
__device__ __forceinline__ int okey(float v) { const int b = __float_as_int(v); return b >= 0 ? b : b ^ 0x7fffffff; }

// ---- CTA pairs (cta_group::2): M = 256 MMAs over two CTAs of a cluster, each supplying its own 128 A rows and HALF of the B columns
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t *bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
// wait for a phase completed by an arrival from the peer CTA
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
    uint32_t done, spins = 0;
    do {
        if (++spins > (1u << 24)) __trap();
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
template <bool PAIR>
__device__ __forceinline__ void tl_commit(uint64_t *bar) {
    if constexpr (PAIR)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                     "h"((uint16_t)3) : "memory");
    else
        tc_commit(bar);
}
template <bool PAIR>
__device__ __forceinline__ void tl_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (PAIR)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        tc_mma(d_tmem, a_desc, b_desc, idesc, accumulate);
}
// kind::f16 instruction descriptor of the pair: M = 256
__host__ __device__ constexpr uint32_t instr_desc_m(int n, int m) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct TlArgs {
    const uint8_t *in;                // upconv2's output, pairs layout [item][3 planes][TL_UP2_PLANE][16 B]
    const uint8_t *wblob;             // TL_WBYTES of operands + constants (pack_tail in ofb_policy.cu)
    float bias4;
    float *ptr_out;                   // optional dense pointer map [item][400][400]
    int *xy;                          // [item][2]
    __nv_bfloat16 *up3_dbg;           // optional: upconv3's output NHWC [item][200][200][8] (validation taps)
    long long *stamps;                // optional: clock64 stamps of CTA 0, [tile < TL_STAMP_TILES][8] (scripts/tail_stamps.py)
};
#define TL_STAMP_TILES 64
#define TL_STAMP(g, j) do { if (a.stamps && blockIdx.x == 0 && (g) < TL_STAMP_TILES) a.stamps[(g) * 8 + (j)] = clock64(); } while (0)

// shared memory (bytes)
struct TlSmem {
    static constexpr unsigned off_ones = 0;                                          // 128 rows x 16 B: K lane 0 = 1.0 (bias MMA's A operand;
                                                                                     // its second K chunk = the ring rows behind it, x 0)
    static constexpr unsigned off_ring = off_ones + 128 * 16;                        // 16 planes x TL_RING rows x 16 B
    static constexpr unsigned off_w = off_ring + 16 * TL_RING * 16;                  // the weight blob, verbatim
    static constexpr unsigned off_a3 = off_w + TL_WBYTES;                            // 2 stages x 3 planes x TL_A3_SLOTS x 16 B
    static constexpr unsigned off_misc = off_a3 + 2 * 3 * TL_A3_SLOTS * 16;          // corners[2][4], vship, si[4]
    static constexpr unsigned off_bar = off_misc + 32 * 4;
    // barriers: wbar, a3_full[2], a3_empty[2], d3_full[2], d3_empty[2], d3v_empty, ring_full[3], ring_free[3], d4_full[2], d4_empty[2]
    // ... and, for CTA pairs, peer3[2], peer4[2]: the peer's "tile g may be issued" of upconv3 / upconv4 (arrivals from the other CTA)
    static constexpr unsigned n_bar = 1 + 2 + 2 + 2 + 2 + 1 + 3 + 3 + 2 + 2 + 4;
    static constexpr unsigned total = off_bar + n_bar * 8 + 16;
};
static_assert(TlSmem::total <= 232448, "k_tz_tail: shared memory over the 227 KB limit");

#define TL_NT (15 * 32)
#define TL_TM_D3V 256
#define TL_TM_D4 320

// ring row (physical) of row `rel` of the tile in ring slot `slot` (rel may be < 0 or >= 128: the neighbouring tiles)
__device__ __forceinline__ void ring_store(uint4 *ring, int plane, int slot, int rel, const uint4 &v) {
    int phys = TL_MARGIN + 128 * slot + rel;
    if (phys >= TL_RING) phys -= 384;
    ring[plane * TL_RING + phys] = v;
    if (slot == 2 && rel >= 64 && rel < 128) ring[plane * TL_RING + phys - 384] = v;        // mirror in front of slot 0
}

template <bool PAIR>
__global__ void __launch_bounds__(TL_NT, 1)
k_tz_tail(const TlArgs a, const int n_ships) {
    // operand geometry: a CTA of a pair holds HALF of every B operand's N columns (its rank's half), so every operand offset,
    // block stride and chunk distance (LBO) is halved; A operands, TMEM columns and every drain are unchanged
    constexpr uint32_t H = PAIR ? 2u : 1u;
    constexpr int MM = PAIR ? 256 : 128;
    const uint32_t rank = PAIR ? cluster_rank() : 0u;
    const bool leader = !PAIR || rank == 0u;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint4 *ring = reinterpret_cast<uint4 *>(smem + TlSmem::off_ring);
    const float *wf = reinterpret_cast<const float *>(smem + TlSmem::off_w + TL_OFF_AUX / (PAIR ? 2 : 1));   // bias3[8], corner weights [4][2][2][8]
    float *corners = reinterpret_cast<float *>(smem + TlSmem::off_misc);                  // [2][4]
    int *vship = reinterpret_cast<int *>(smem + TlSmem::off_misc) + 8;
    int *si = reinterpret_cast<int *>(smem + TlSmem::off_misc) + 16;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + TlSmem::off_bar);
    uint64_t *wbar = bars, *a3_full = bars + 1, *a3_empty = a3_full + 2, *d3_full = a3_empty + 2, *d3_empty = d3_full + 2,
             *d3v_empty = d3_empty + 2, *ring_full = d3v_empty + 1, *ring_free = ring_full + 3, *d4_full = ring_free + 3,
             *d4_empty = d4_full + 2, *peer3 = d4_empty + 2, *peer4 = peer3 + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + TlSmem::off_bar + TlSmem::n_bar * 8);

    // the ring starts out as zeros: rows nobody has written yet are read (by M rows whose outputs are discarded) and must
    // not hold NaN patterns
    for (int i = tid; i < 16 * TL_RING; i += TL_NT) ring[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid < 128) reinterpret_cast<uint4 *>(smem + TlSmem::off_ones)[tid] = make_uint4(0x3F80u, 0u, 0u, 0u);   // bf16 1.0 in K lane 0
    if (tid == 0) {
        mbar_init(wbar, 1);
        for (int s = 0; s < 2; s++) {
            mbar_init(&a3_full[s], 1);
            mbar_init(&a3_empty[s], 1);
            mbar_init(&d3_full[s], 1);
            mbar_init(&d3_empty[s], 4);
            mbar_init(&d4_full[s], 1);
            mbar_init(&d4_empty[s], 4);
        }
        mbar_init(d3v_empty, 4);
        for (int s = 0; s < 3; s++) { mbar_init(&ring_full[s], 4); mbar_init(&ring_free[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&peer3[s], 1); mbar_init(&peer4[s], 1); }
        *vship = (int)0x80000000;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();                                   // the zeros above vs. the MMAs' (async proxy) reads
    if constexpr (PAIR) {
        __syncthreads();
        cluster_sync_all();                               // both CTAs' barriers exist before anything can arrive on them
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
        }
    } else if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // ships of this CTA; a pair works in lockstep, so both CTAs take the same count (a CTA past the end repeats the last ship)
    const int n_mine = PAIR ? (n_ships + (int)gridDim.x - 1) / (int)gridDim.x : (n_ships - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int n_tiles = n_mine * TL_TILES;
    auto ship_of = [&](int k) { return (size_t)min((long long)blockIdx.x + (long long)k * gridDim.x, (long long)n_ships - 1); };

    if (warp == 12) {
        // ------------------------------------------------------------ producer: weights once, then one input tile per step
        if (lane == 0) {
            constexpr unsigned WB = PAIR ? TL_WBYTES_H : TL_WBYTES;
            const uint8_t *wsrc = a.wblob + (PAIR ? (size_t)rank * TL_WBYTES_H : 0);
            mbar_expect_tx(wbar, WB);
            for (unsigned off = 0; off < WB; off += 30720) bulk_g2s(smem + TlSmem::off_w + off, wsrc + off, min(30720u, WB - off), wbar);
            for (int g = 0; g < n_tiles; g++) {
                const int s = g & 1, k = g / TL_TILES, t = g - k * TL_TILES;
                const size_t ship = ship_of(k);
                if (g >= 2) mbar_wait(&a3_empty[s], (uint32_t)(((g >> 1) - 1) & 1));
                mbar_expect_tx(&a3_full[s], 3u * TL_A3_SLOTS * 16);
                uint8_t *dst = smem + TlSmem::off_a3 + s * (3 * TL_A3_SLOTS * 16);
                const uint8_t *src = a.in + (ship * 3 * TL_UP2_PLANE + (size_t)128 * t) * 16;
#pragma unroll
                for (int pl = 0; pl < 3; pl++)
                    bulk_g2s(dst + pl * TL_A3_SLOTS * 16, src + (size_t)pl * TL_UP2_PLANE * 16, TL_A3_SLOTS * 16, &a3_full[s]);
            }
        }
        __syncwarp();
    } else if (warp == 13) {
        // ------------------------------------------------------------ upconv3 MMAs (converged warp, one elected lane issues).
        // CTA pairs: the leader issues for both CTAs; the peer's warp only reports "my tile g may be issued" (input landed,
        // TMEM stage drained) to the leader; the commits arrive on both CTAs' barriers.
        mbar_wait(wbar, 0);
        const bool elected = elect_one(), issue = elected && leader;
        const uint32_t b3 = smem_u32(smem + TlSmem::off_w + TL_OFF_B3 / H) >> 4, b3v = smem_u32(smem + TlSmem::off_w + TL_OFF_B3V / H) >> 4;
        const uint32_t ones16 = smem_u32(smem + TlSmem::off_ones) >> 4, ring16 = smem_u32(ring) >> 4;
        const uint32_t bias16 = smem_u32(smem + TlSmem::off_w + TL_OFF_BIAS3 / H) >> 4;
        constexpr uint32_t ID128 = instr_desc_m(128, MM), ID64 = instr_desc_m(64, MM);
        int vq = 0;
        for (int g = 0; g < n_tiles; g++) {
            const int s = g & 1, t = g % TL_TILES;
            const bool var_tile = t == 0 || t == TL_TILES - 1;
            mbar_wait(&a3_full[s], (uint32_t)((g >> 1) & 1));
            if (g >= 2) { mbar_wait(&d3_empty[s], (uint32_t)(((g >> 1) - 1) & 1)); tc_fence_after(); }
            if (PAIR && var_tile && vq >= 1) { mbar_wait(d3v_empty, (uint32_t)((vq - 1) & 1)); tc_fence_after(); }
            if constexpr (PAIR) {
                if (!leader) {
                    if (elected) mbar_arrive_remote(&peer3[s], 0u);
                    if (var_tile) vq++;
                    __syncwarp();
                    continue;
                }
                mbar_wait_cluster(&peer3[s], (uint32_t)((g >> 1) & 1));
                tc_fence_after();
            }
            const uint32_t a16 = smem_u32(smem + TlSmem::off_a3 + s * (3 * TL_A3_SLOTS * 16)) >> 4;
            const uint32_t d = tmem_base + (uint32_t)(s * 128);
            // bias: A = a column of ones in K lane 0 (the second K chunk reads ring rows against zero weights)
            const uint64_t ones_d = smem_desc(ones16, ring16 - ones16, 8), bias_d = smem_desc(bias16, 128 / H, 8);
            if (issue) tl_mma<PAIR>(d, ones_d, bias_d, ID128, 0u);
#pragma unroll
            for (int u = 0; u < 3; u++)
#pragma unroll
                for (int ks = 0; ks < 2; ks++) {
                    // ks 0: chunks (PA[e], PB[e]); ks 1: (PA[e + 1], spare[e])
                    const uint64_t ad = smem_desc(a16 + (uint32_t)(26 * u + ks), ks ? 2u * TL_A3_SLOTS - 1u : (uint32_t)TL_A3_SLOTS, 8);
                    const uint64_t bd = smem_desc(b3 + (uint32_t)((u * 2 + ks) * 2 * (128 / H)), 128 / H, 8);
                    if (issue) tl_mma<PAIR>(d, ad, bd, ID128, 1u);
                }
            if (var_tile) {
                // top / bottom image row: the true (zero-padded) phase a = 0 / 1 of row i = 0 / 99 into their own columns
                const int set = t == 0 ? 0 : 1;
                if (!PAIR && vq >= 1) { mbar_wait(d3v_empty, (uint32_t)((vq - 1) & 1)); tc_fence_after(); }
                if (issue) tl_mma<PAIR>(tmem_base + TL_TM_D3V, ones_d, bias_d, ID64, 0u);       // column n of the variant has channel n & 7 too
#pragma unroll
                for (int ui = 0; ui < 2; ui++)
#pragma unroll
                    for (int ks = 0; ks < 2; ks++) {
                        const int u = set == 0 ? ui + 1 : ui;
                        const uint64_t ad = smem_desc(a16 + (uint32_t)(26 * u + ks), ks ? 2u * TL_A3_SLOTS - 1u : (uint32_t)TL_A3_SLOTS, 8);
                        const uint64_t bd = smem_desc(b3v + (uint32_t)((((set * 2 + ui) * 2) + ks) * 2 * (64 / H)), 64 / H, 8);
                        if (issue) tl_mma<PAIR>(tmem_base + TL_TM_D3V, ad, bd, ID64, 1u);
                    }
                vq++;
            }
            if (issue) { tl_commit<PAIR>(&d3_full[s]); tl_commit<PAIR>(&a3_empty[s]); }
            __syncwarp();
        }
    } else if (warp == 14) {
        // ------------------------------------------------------------ upconv4 MMAs
        mbar_wait(wbar, 0);
        const bool elected = elect_one(), issue = elected && leader;
        const uint32_t ring16 = smem_u32(ring) >> 4;
        const uint32_t b4 = smem_u32(smem + TlSmem::off_w + TL_OFF_B4 / H) >> 4, b4v = smem_u32(smem + TlSmem::off_w + TL_OFF_B4V / H) >> 4;
        constexpr uint32_t ID80 = instr_desc_m(80, MM), ID48 = instr_desc_m(48, MM), ID16 = instr_desc_m(16, MM);
        for (int g = 0; g < n_tiles; g++) {
            const int s = g & 1, t = g % TL_TILES, slot = t % 3;
            mbar_wait(&ring_full[slot], (uint32_t)((g / 3) & 1));
            if (lane == 0) TL_STAMP(g, 4);
            if (g >= 2) { mbar_wait(&d4_empty[s], (uint32_t)(((g >> 1) - 1) & 1)); tc_fence_after(); }
            if constexpr (PAIR) {
                if (!leader) {
                    if (elected) mbar_arrive_remote(&peer4[s], 0u);
                    __syncwarp();
                    continue;
                }
                mbar_wait_cluster(&peer4[s], (uint32_t)((g >> 1) & 1));
                tc_fence_after();
            }
            if (lane == 0) TL_STAMP(g, 5);
            const uint32_t base = ring16 + (uint32_t)(TL_MARGIN - TL_UP4_LAG + 128 * slot);       // ring row of M row 128 t - 32
            const uint32_t d = tmem_base + (uint32_t)(TL_TM_D4 + 96 * s);
            // vertical tap dy reads upconv3 row 2i - 1 + dy: parity a = (dy + 1) & 1, ring row m + {-26, 0, 0, +26}
#pragma unroll
            for (int o = 0; o < 4; o++) {
                const int dy = o == 0 ? 1 : (o == 1 ? 2 : (o == 2 ? 0 : 3));       // the full-width taps first (they zero the accumulator)
                const int par = (dy + 1) & 1, voff = dy == 0 ? -TL_P : (dy == 3 ? TL_P : 0);
                const int nn = (dy == 0 || dy == 3) ? 48 : 80;
                const uint32_t boff = (dy == 0 ? 0u : (dy == 1 ? 480u : (dy == 2 ? 1280u : 2080u))) / H;
#pragma unroll
                for (int ks = 0; ks < 5; ks++) {
                    const int q0 = (ks == 0 || ks == 4) ? 0 : 2 * ks - 1, o0 = ks == 4 ? 1 : 0;
                    const uint32_t lbo = (ks == 0 || ks == 4) ? 7u * TL_RING - 1u : (uint32_t)TL_RING;
                    const uint64_t ad = smem_desc(base + (uint32_t)((par * 8 + q0) * TL_RING + voff + o0), lbo, 8);
                    const uint64_t bd = smem_desc(b4 + boff + (uint32_t)(ks * 2 * (nn / (int)H)), (uint32_t)nn / H, 8);
                    if (issue) tl_mma<PAIR>(d + (dy == 3 ? 32u : 0u), ad, bd, nn == 80 ? ID80 : ID48, (o | ks) ? 1u : 0u);
                }
            }
            if (t == 0 || t == TL_TILES - 1) {
                // top / bottom row of the 400 x 400 map (V = 0 / 399): taps dy = 1, 2 with the border weights, 16 pixels per M row
                const int set = t == 0 ? 0 : 1;
#pragma unroll
                for (int dyi = 0; dyi < 2; dyi++)
#pragma unroll
                    for (int ks = 0; ks < 5; ks++) {
                        const int par = dyi == 0 ? 0 : 1;                          // dy = 1 -> row 2i (a = 0), dy = 2 -> row 2i + 1 (a = 1)
                        const int q0 = (ks == 0 || ks == 4) ? 0 : 2 * ks - 1, o0 = ks == 4 ? 1 : 0;
                        const uint32_t lbo = (ks == 0 || ks == 4) ? 7u * TL_RING - 1u : (uint32_t)TL_RING;
                        const uint64_t ad = smem_desc(base + (uint32_t)((par * 8 + q0) * TL_RING + o0), lbo, 8);
                        const uint64_t bd = smem_desc(b4v + (uint32_t)((((set * 2 + dyi) * 5) + ks) * 2 * (16 / H)), 16 / H, 8);
                        if (issue) tl_mma<PAIR>(d + 80u, ad, bd, ID16, (dyi | ks) ? 1u : 0u);
                    }
            }
            if (issue) {
                tl_commit<PAIR>(&d4_full[s]);
                tl_commit<PAIR>(&ring_free[(slot + 2) % 3]);      // tile g - 1's ring slot (and, for a tile of slot 0, the mirror rows): no reader left
            }
            __syncwarp();
        }
    } else if (warp < 8) {
        // ------------------------------------------------------------ upconv3 drain: group grp takes the tiles g = grp (mod 2).
        // TMEM -> ReLU -> bf16 happens BEFORE the wait for the ring slot (the 16 chunks of an M row sit in 64 registers), so
        // that only the stores are in the dependency chain  MMAs of upconv4 (g - 2) -> ring slot free -> MMAs of upconv4 (g).
        mbar_wait(wbar, 0);
        const int grp = warp >> 2, gw = warp & 3, r = tid & 127;
        for (int g = grp; g < n_tiles; g += 2) {
            const int s = grp, k = g / TL_TILES, t = g - k * TL_TILES, slot = t % 3;
            const size_t ship = ship_of(k);
            const int m = 128 * t + r, i = m / TL_P, xb = m - i * TL_P;
            const bool valid = xb < 25 && i < 100;
            mbar_wait(&d3_full[s], (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            if (r == 0) TL_STAMP(g, 0);
            const uint32_t lane_base = tmem_base + ((uint32_t)(gw * 32) << 16);
            const bool var_tile = t == 0 || t == TL_TILES - 1;
            const bool var_warp = (t == 0 && gw == 0) || (t == TL_TILES - 1 && gw < 2);     // warps that hold M rows of i = 0 / 99
            const int var_a = t == 0 ? 0 : 1;
            const bool use_var = var_warp && valid && i == (t == 0 ? 0 : 99);
            uint4 px[16];                                 // chunk xo * 4 + a * 2 + b = pixel (2i + a, 8 xb + 2 xo + b)
#pragma unroll
            for (int xo = 0; xo < 4; xo++) {
                uint32_t rr[32], rv[16];
                tc_ld32(lane_base + (uint32_t)(s * 128 + xo * 32), rr);
                if (var_warp) tc_ld16(lane_base + (uint32_t)(TL_TM_D3V + xo * 16), rv);
                tc_wait_ld();
                if (var_warp && use_var) {                 // compile-time register indices: no local-memory array
                    if (var_a == 0) {
#pragma unroll
                        for (int j = 0; j < 16; j++) rr[j] = rv[j];
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j++) rr[16 + j] = rv[j];
                    }
                }
#pragma unroll
                for (int ph = 0; ph < 4; ph++)
                    px[xo * 4 + ph] = make_uint4(pack_relu_bf2(__uint_as_float(rr[ph * 8]), __uint_as_float(rr[ph * 8 + 1])),
                                                 pack_relu_bf2(__uint_as_float(rr[ph * 8 + 2]), __uint_as_float(rr[ph * 8 + 3])),
                                                 pack_relu_bf2(__uint_as_float(rr[ph * 8 + 4]), __uint_as_float(rr[ph * 8 + 5])),
                                                 pack_relu_bf2(__uint_as_float(rr[ph * 8 + 6]), __uint_as_float(rr[ph * 8 + 7])));
            }
            tc_fence_before();                            // all of this warp's accumulator reads are done: hand the stage back
            __syncwarp();
            if (lane == 0) { mbar_arrive(&d3_empty[s]); if (var_tile) mbar_arrive(d3v_empty); }
            if (r == 0) TL_STAMP(g, 1);
            // Ring slot `slot` (tile g - 3's) is free once upconv4's MMAs of tile g - 2 have completed.  A tile of slot 2 also
            // writes the mirror rows in front of slot 0, which the MMAs of tile g - 2 (slot 0) read: it waits even the first time.
            if (slot == 2) mbar_wait(&ring_free[2], (uint32_t)((g / 3) & 1));
            else if (g >= 3) mbar_wait(&ring_free[slot], (uint32_t)(((g / 3) - 1) & 1));
            if (r == 0) TL_STAMP(g, 2);
            if (valid) {
                uint4 *dst = ring + TL_MARGIN + 128 * slot + r;
#pragma unroll
                for (int c = 0; c < 16; c++) dst[(((c >> 1) & 1) * 8 + 2 * (c >> 2) + (c & 1)) * TL_RING] = px[c];
                if (slot == 2 && r >= 64) {               // mirror in front of slot 0
#pragma unroll
                    for (int c = 0; c < 16; c++) dst[(((c >> 1) & 1) * 8 + 2 * (c >> 2) + (c & 1)) * TL_RING - 384] = px[c];
                }
                // replicated edges (rare lanes): X = -1 := X = 0, X = 200 := X = 199, Y = -1 := Y = 0, Y = 200 := Y = 199
                if (xb == 0) { ring_store(ring, 7, slot, r - 1, px[0]); ring_store(ring, 15, slot, r - 1, px[2]); }
                if (xb == 24) { ring_store(ring, 0, slot, r + 1, px[13]); ring_store(ring, 8, slot, r + 1, px[15]); }
                if (i == 0) {
#pragma unroll
                    for (int c = 0; c < 16; c++)
                        if (((c >> 1) & 1) == 0) ring_store(ring, 8 + 2 * (c >> 2) + (c & 1), slot, r - TL_P, px[c]);
                    if (xb == 0) ring_store(ring, 15, slot, r - TL_P - 1, px[0]);
                    if (xb == 24) ring_store(ring, 8, slot, r - TL_P + 1, px[13]);
                }
                if (i == 99) {
#pragma unroll
                    for (int c = 0; c < 16; c++)
                        if (((c >> 1) & 1) == 1) ring_store(ring, 2 * (c >> 2) + (c & 1), slot, r + TL_P, px[c]);
                    if (xb == 0) ring_store(ring, 7, slot, r + TL_P - 1, px[2]);
                    if (xb == 24) ring_store(ring, 0, slot, r + TL_P + 1, px[15]);
                }
                if ((i == 0 || i == 99) && (xb == 0 || xb == 24)) {
                    // corner pixel of the 400 x 400 map: 2 x 2 upconv3 pixels x 8 channels with both borders' weights
                    const int cid = (i == 0 ? 0 : 2) + (xb == 0 ? 0 : 1);
                    float corner = 0.f;
#pragma unroll
                    for (int ph = 0; ph < 4; ph++) {
                        const uint4 lo = px[ph], hi = px[12 + ph];
                        const uint4 sel = make_uint4(xb == 0 ? lo.x : hi.x, xb == 0 ? lo.y : hi.y, xb == 0 ? lo.z : hi.z, xb == 0 ? lo.w : hi.w);
                        float u3[8];
                        unpack_bf8(sel, u3);
                        const float *cw = wf + 8 + ((cid * 2 + (ph >> 1)) * 2 + (ph & 1)) * 8;
#pragma unroll
                        for (int c = 0; c < 8; c++) corner += u3[c] * cw[c];
                    }
                    corners[(k & 1) * 4 + cid] = corner;
                }
                if (a.up3_dbg) {
#pragma unroll
                    for (int c = 0; c < 16; c++)
                        *reinterpret_cast<uint4 *>(a.up3_dbg + ((ship * 200 + (size_t)(2 * i + ((c >> 1) & 1))) * 200 +
                                                                (size_t)(8 * xb + 2 * (c >> 2) + (c & 1))) * 8) = px[c];
                }
            }
            fence_async_smem();                           // generic-proxy stores -> visible to the MMAs' operand reads
            __syncwarp();
            if (lane == 0) mbar_arrive(&ring_full[slot]);
            if (r == 0) TL_STAMP(g, 3);
        }
    } else if (warp < 12) {
        // ------------------------------------------------------------ upconv4 drain + argmax
        mbar_wait(wbar, 0);
        const int gw = warp & 3, l = tid - 256;
        const uint32_t lane_base = tmem_base + ((uint32_t)(gw * 32) << 16);
        int best_key = (int)0x80000000, best_idx = 0x7fffffff;
        for (int g = 0; g < n_tiles; g++) {
            const int s = g & 1, k = g / TL_TILES, t = g - k * TL_TILES;
            const size_t ship = ship_of(k);
            const int m = 128 * t - TL_UP4_LAG + l, mm = max(m, 0), i = mm / TL_P, xb = mm - i * TL_P;
            const bool valid = m >= 0 && xb < 25 && i < 100;
            const bool var_tile = t == 0 || t == TL_TILES - 1;
            mbar_wait(&d4_full[s], (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            if (l == 0) TL_STAMP(g, 6);
            uint32_t ra[32], rb[32], rc[16], rv[16];
            const uint32_t tm = lane_base + (uint32_t)(TL_TM_D4 + 96 * s);
            tc_ld32(tm, ra);
            tc_ld32(tm + 32, rb);
            tc_ld16(tm + 64, rc);
            if (var_tile) tc_ld16(tm + 80, rv);
            tc_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d4_empty[s]);
            // columns: [0,8) variants of row r = 0 (c * 2 + side), [8,40) row 0: xo * 4 + c * 2 + d, [40,72) row 1, [72,80) variants of row 1
            float v[64];
#pragma unroll
            for (int n = 0; n < 64; n++) {
                const int col = n + 8;
                v[n] = __uint_as_float(col < 32 ? ra[col] : (col < 64 ? rb[col - 32] : rc[col - 64]));
            }
            if (xb == 0) {                                // Z = 0: (xo 0, d 0)
#pragma unroll
                for (int rw = 0; rw < 2; rw++)
#pragma unroll
                    for (int c = 0; c < 2; c++) v[rw * 32 + c * 2] = __uint_as_float(rw == 0 ? ra[c * 2] : rc[8 + c * 2]);
            }
            if (xb == 24) {                               // Z = 399: (xo 7, d 1)
#pragma unroll
                for (int rw = 0; rw < 2; rw++)
#pragma unroll
                    for (int c = 0; c < 2; c++) v[rw * 32 + 28 + c * 2 + 1] = __uint_as_float(rw == 0 ? ra[c * 2 + 1] : rc[8 + c * 2 + 1]);
            }
            if (var_tile) {
                if (t == 0 && i == 0) {                   // V = 0: row r = 0, c = 0
#pragma unroll
                    for (int j = 0; j < 16; j++) v[(j >> 1) * 4 + (j & 1)] = __uint_as_float(rv[j]);
                    if (xb == 0) v[0] = corners[(k & 1) * 4 + 0];
                    if (xb == 24) v[29] = corners[(k & 1) * 4 + 1];
                }
                if (t == TL_TILES - 1 && i == 99) {       // V = 399: row r = 1, c = 1
#pragma unroll
                    for (int j = 0; j < 16; j++) v[32 + (j >> 1) * 4 + 2 + (j & 1)] = __uint_as_float(rv[j]);
                    if (xb == 0) v[32 + 2] = corners[(k & 1) * 4 + 2];
                    if (xb == 24) v[32 + 28 + 3] = corners[(k & 1) * 4 + 3];
                }
            }
            if (a.ptr_out && valid) {
                float *dst = a.ptr_out + ship * 160000 + (size_t)(4 * i) * 400 + 16 * xb;
#pragma unroll
                for (int n = 0; n < 64; n++)
                    dst[((n >> 5) * 2 + ((n >> 1) & 1)) * 400 + 2 * ((n & 31) >> 2) + (n & 1)] = v[n] + a.bias4;
            }
            float mx[32];
#pragma unroll
            for (int n = 0; n < 32; n++) mx[n] = fmaxf(v[n], v[n + 32]);
#pragma unroll
            for (int h = 16; h > 0; h >>= 1)
#pragma unroll
                for (int n = 0; n < h; n++) mx[n] = fmaxf(mx[n], mx[n + h]);
            // the map is v + bias4: fp32 addition is monotone but not injective, so the maximum and its first index are taken
            // on the biased values (two pixels with v1 > v2 can both round to the same v + bias4)
            const float M = mx[0] + a.bias4;
            const int key = okey(M);
            // only a value that reaches the ship's best so far can be its maximum: the index scan is rare
            const bool cand = valid && key >= *reinterpret_cast<volatile int *>(vship);
            if (__any_sync(0xffffffffu, cand)) {
                if (cand) {
                    int cmin = 0x7fffffff;
#pragma unroll
                    for (int n = 0; n < 64; n++) {
                        const int cn = ((n >> 5) * 2 + ((n >> 1) & 1)) * 400 + 2 * ((n & 31) >> 2) + (n & 1);
                        if (v[n] + a.bias4 == M) cmin = min(cmin, cn);
                    }
                    const int idx = 1600 * i + 16 * xb + cmin;
                    if (key > best_key || (key == best_key && idx < best_idx)) { best_key = key; best_idx = idx; }
                    atomicMax(vship, key);
                }
            }
            if (l == 0) TL_STAMP(g, 7);
            if (t == TL_TILES - 1) {
                // the ship is complete: the lowest flat index among the threads that hold its maximum
                named_sync(1, 128);
                const int V = *reinterpret_cast<volatile int *>(vship);
                int bi = best_key == V ? best_idx : 0x7fffffff;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) bi = min(bi, __shfl_xor_sync(0xffffffffu, bi, o));
                if (lane == 0) si[gw] = bi;
                named_sync(1, 128);
                if (l == 0) {
                    const int b = min(min(si[0], si[1]), min(si[2], si[3]));
                    if (a.xy) {
                        a.xy[ship * 2] = b % 400;         // (x, y) = (k % 400, k // 400)   (:219-220, F-order unravel)
                        a.xy[ship * 2 + 1] = b / 400;
                    }
                    *vship = (int)0x80000000;
                }
                best_key = (int)0x80000000;
                best_idx = 0x7fffffff;
                named_sync(1, 128);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) {
        cluster_sync_all();                               // the peer's MMAs / commits no longer touch this CTA
        if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
    } else if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
    }
}

static long long *g_tail_stamps = nullptr;
extern "C" int ofb_policy_tail_stamps(long long *dev_buf) { g_tail_stamps = dev_buf; return OFB_OK; }

int pol_tz_tail(const ofb_policy *p, const __nv_bfloat16 *up2_pairs, float *ptr_out, int32_t *xy, __nv_bfloat16 *up3_dbg, int n_items,
                cudaStream_t st) {
    static thread_local SmemAttrCache attr = {}, attr2 = {};
    int n_sm = 148;
    OFB_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, p->device));
    if (n_items == 0) return OFB_OK;
    TlArgs a = {};
    a.in = reinterpret_cast<const uint8_t *>(up2_pairs);
    a.wblob = reinterpret_cast<const uint8_t *>(p->w.tail_blob);
    a.bias4 = p->u4_bias == 0.f ? 0.f : p->u4_bias;         // +0.0 for a bias of -0.0: -0.0 and +0.0 are one value for the argmax
    a.ptr_out = ptr_out;
    a.xy = xy;
    a.up3_dbg = up3_dbg;
    a.stamps = g_tail_stamps;
    if (p->tail_pair) {
        // CTA pairs: clusters of 2 (one CTA per SM, both SMs of a TPC), an even grid
        OFB_CUDA_CHECK(attr2.ensure(k_tz_tail<true>, (int)TlSmem::total));
        a.wblob = reinterpret_cast<const uint8_t *>(p->w.tail_blob2);
        int grid = n_items < n_sm ? n_items : n_sm;
        grid = (grid + 1) & ~1;
        if (grid > n_sm) grid -= 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(TL_NT);
        cfg.dynamicSmemBytes = TlSmem::total;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        OFB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, k_tz_tail<true>, a, n_items));
        return OFB_OK;
    }
    OFB_CUDA_CHECK(attr.ensure(k_tz_tail<false>, (int)TlSmem::total));
    k_tz_tail<false><<<n_items < n_sm ? n_items : n_sm, TL_NT, TlSmem::total, st>>>(a, n_items);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}
