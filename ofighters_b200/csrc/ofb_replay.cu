// Device-resident replay memory (include/ofb_replay.h) for sm_100a (compiled with -fmad=false: the gather rasterises
// lasers in fp64 with the frame kernel's code, ofb_raster_dev.cuh, so its maps are bit-identical to the frame's).
//
// Ring layout: slot s, tracked arena a -> ring + (s * count + a) * stride, the first bytes of an arena block (header,
// ships, live laser groups) copied from the handle's state.  Per transition id = s * count * P + a * P + p (P policy ships):
// the played action and pointer of frame s, and -- once frame s + 1 was pushed -- valid / reward / done.  An n-step memory
// keeps the same one-step fields: ofb_replay_gather_nstep walks them at gather time.
#include <cstring>
#include <new>
#include "ofb_common.cuh"
#include "ofb_raster_dev.cuh"
#include "../../include/ofb_replay.h"

#define OFB_REPLAY_TILE 2048          // candidates per block of the index kernels: 256 threads x 8
struct PrioStats {                   // written by k_prio_scan for the draws of the same sample
    double total;                    // sum of the valid masses
    float mass_min;                  // smallest non-zero valid mass
    int last_tile;                   // last tile with a non-zero sum
};
struct ofb_replay {
    const ofb_arenas *h;
    ArenaLayout lay;
    int device;
    long long first, count;
    int P, depth;
    int n_step;                  // frames of an n-step return (1 = one-step transitions)
    int32_t *ships;              // [P] ship index of each policy ship
    char *ring;                  // depth * count * stride bytes
    int32_t *act;                // [depth * count * P]
    int2 *xy;                    // [depth * count * P]
    float *reward;               // [depth * count * P]
    uint8_t *valid, *done;       // [depth * count * P]
    int32_t *tile_count;         // [n_tiles] scratch of ofb_replay_index
    long long n_tiles;
    long long pushes;            // frames pushed so far
    int newest;                  // slot of the last push
    size_t bytes;
    // prioritized replay: all NULL until ofb_replay_enable_priorities
    float *mass;                 // [depth * count * P] sampling mass of each transition id
    float *max_mass;             // [1] largest mass set so far (initially 1)
    double *tile_sum;            // [n_tiles] sum of the valid masses of each tile
    double *tile_prefix;         // [n_tiles] exclusive prefix of tile_sum
    float *tile_min;             // [n_tiles] smallest non-zero valid mass of each tile
    int32_t *tile_valid;         // [n_tiles] valid transitions with a non-zero mass in each tile
    PrioStats *stats;            // [1]
    float alpha, eps;
    unsigned long long seed;
    long long samples;           // prioritized samples drawn so far: the Philox counter
};

// ---------------------------------------------------------------- push: one warp per tracked arena
__global__ void __launch_bounds__(128)
k_replay_push(const char *__restrict__ state, const ArenaLayout lay, long long first, long long count,
              const int32_t *__restrict__ ships, int P, char *__restrict__ ring, int slot, int prev, int mslot,
              const int32_t *__restrict__ iaction_in,
              const int2 *__restrict__ xy_in, int32_t *__restrict__ act, int2 *__restrict__ xy, float *__restrict__ reward,
              uint8_t *__restrict__ valid, uint8_t *__restrict__ done, float *__restrict__ mass, const float *__restrict__ max_mass) {
    const long long a = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (a >= count) return;
    const char *src = state + (first + a) * (long long)lay.stride;
    char *dst = ring + ((long long)slot * count + a) * (long long)lay.stride;
    const int *hdr = reinterpret_cast<const int *>(src);
    const int n = hdr[HDR_NLASERS];
    // header + ships + the live laser groups: a multiple of 16 bytes (off_laser and OFB_GROUP_BYTES both are)
    const int n16 = (lay.off_laser + ((n + 7) >> 3) * OFB_GROUP_BYTES) >> 4;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
#pragma unroll 4                                           // (the default unroll spills to local memory)
    for (int i = lane; i < n16; i += 32) d4[i] = s4[i];
    if (lane < P) {
        const long long cP = count * P;
        const long long j = a * P + lane;
        const int si = ships[lane];
        const uint4 rec = reinterpret_cast<const uint4 *>(src + lay.off_ship)[si];
        if (prev >= 0) {                                   // frame t = slot `prev` gets its successor t+1 = this state
            const char *old = ring + ((long long)prev * count + a) * (long long)lay.stride;
            const uint4 orec = reinterpret_cast<const uint4 *>(old + lay.off_ship)[si];
            const bool same_episode = reinterpret_cast<const int *>(old)[HDR_EPISODE] == hdr[HDR_EPISODE];
            valid[prev * cP + j] = (same_episode && (orec.x >> 31)) ? 1 : 0;
            reward[prev * cP + j] = (float)ship_unpack(rec).reward;
            done[prev * cP + j] = (rec.x >> 31) ? 0 : 1;
        }
        // prioritized replay: the frame that becomes a candidate with this push (prev for n = 1) gets the largest mass
        if (mass && mslot >= 0) mass[mslot * cP + j] = *max_mass;
        const long long o = (long long)slot * cP + j;
        valid[o] = 0;                                      // the newest frame has no successor yet
        act[o] = iaction_in[(first + a) * P + lane];
        xy[o] = xy_in[(first + a) * P + lane];
    }
}

// ---------------------------------------------------------------- index: count per tile, scan, scatter in order
// candidate c in [0, nf * cP): frame f = c / cP (0 = oldest complete frame), its transition c % cP
__device__ __forceinline__ long long replay_id(long long c, long long cP, int oldest, int depth) {
    const long long f = c / cP;
    return (long long)((oldest + f) % depth) * cP + (c - f * cP);
}

__global__ void __launch_bounds__(256)
k_replay_count(const uint8_t *__restrict__ valid, long long cP, long long n_cand, int oldest, int depth,
               int32_t *__restrict__ tile_count) {
    __shared__ int s_warp[8];
    const long long c0 = (long long)blockIdx.x * OFB_REPLAY_TILE + threadIdx.x * 8;
    int k = 0;
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (c0 + i < n_cand) k += valid[replay_id(c0 + i, cP, oldest, depth)];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = k;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < 8; w++) t += s_warp[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts in place (one block); the total goes to count_out
__global__ void __launch_bounds__(1024) k_replay_scan(int32_t *tile_count, long long n_tiles, int32_t *count_out) {
    __shared__ int s_sum[1024];
    const long long per = (n_tiles + 1023) / 1024;
    const long long b0 = threadIdx.x * per, b1 = min(n_tiles, b0 + per);
    int k = 0;
    for (long long i = b0; i < b1; i++) k += tile_count[i];
    s_sum[threadIdx.x] = k;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                   // Hillis-Steele inclusive scan of the per-thread sums
        const int v = threadIdx.x >= o ? s_sum[threadIdx.x - o] : 0;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    int run = s_sum[threadIdx.x] - k;
    for (long long i = b0; i < b1; i++) {
        const int c = tile_count[i];
        tile_count[i] = run;
        run += c;
    }
    if (threadIdx.x == 1023) *count_out = s_sum[1023];
}

__global__ void __launch_bounds__(256)
k_replay_scatter(const uint8_t *__restrict__ valid, long long cP, long long n_cand, int oldest, int depth,
                 const int32_t *__restrict__ tile_off, int32_t *__restrict__ ids) {
    __shared__ int s_warp[8];
    const long long c0 = (long long)blockIdx.x * OFB_REPLAY_TILE + threadIdx.x * 8;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long id[8];
    unsigned m = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        id[i] = c0 + i < n_cand ? replay_id(c0 + i, cP, oldest, depth) : 0;
        if (c0 + i < n_cand && valid[id[i]]) m |= 1u << i;
    }
    const int k = __popc(m);
    int incl = k;                                          // warp inclusive scan
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int base = tile_off[blockIdx.x];
    for (int w = 0; w < warp; w++) base += s_warp[w];
    int pos = base + incl - k;
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (m & (1u << i)) ids[pos++] = (int32_t)id[i];
}

// ---------------------------------------------------------------- gather: one CTA per (sample, obs | next)
// One observation of sample b: the snapshot of tracked arena a in ring slot s -> the ship's head (ofb_obs_vec's, k_obs_vec)
// and the two bit maps, rasterised with the frame kernel's code and written with one bulk store.  Every thread of the CTA
// calls it (it synchronises the block).
__device__ __forceinline__ void gather_observation(uint32_t *bits, const char *__restrict__ ring, const ArenaLayout &lay,
                                                   long long count, long long s, long long a, int ship, int b,
                                                   uint32_t *__restrict__ maps, float *__restrict__ vec) {
    const int W = lay.W, H = lay.H;
    const int words = (W * H) >> 5;
    const char *base = ring + (s * count + a) * (long long)lay.stride;
    const int *hdr = reinterpret_cast<const int *>(base);
    const uint4 *shp = reinterpret_cast<const uint4 *>(base + lay.off_ship);

    if (vec && threadIdx.x == 0) {
        const ShipRec r = ship_unpack(shp[ship]);
        float4 *v = reinterpret_cast<float4 *>(vec + (long long)b * 8);
        v[0] = make_float4((float)r.reward, 1.0f, (float)r.px, (float)r.py);
        v[1] = make_float4((float)lay.W, (float)lay.H, (float)r.x, (float)r.y);
    }
    if (!maps) return;

    const int n = hdr[HDR_NLASERS];
    {
        uint4 *b4 = reinterpret_cast<uint4 *>(bits);
        for (int i = threadIdx.x; i < (2 * words) / 4; i += blockDim.x) b4[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    const int rows = 2 * OFB_R_SHIP - 1;
    for (int t = threadIdx.x; t < lay.S * rows; t += blockDim.x)
        raster_ship_row(bits, W, H, shp[t / rows].x, t % rows - (OFB_R_SHIP - 1));
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const double *lp = reinterpret_cast<const double *>(base + laser_off(lay.off_laser, k));
        raster_laser(bits + words, W, H, lp[0], lp[OFB_G_Y / 8]);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned bytes = (unsigned)(2 * words * 4);
        char *dst = reinterpret_cast<char *>(maps) + (long long)b * bytes;
        const unsigned src = (unsigned)__cvta_generic_to_shared(bits);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(src), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

__global__ void __launch_bounds__(256)
k_replay_gather(const char *__restrict__ ring, const ArenaLayout lay, long long count, int P, int depth,
                const int32_t *__restrict__ ships, const int32_t *__restrict__ ids, const int32_t *__restrict__ act,
                const int2 *__restrict__ axy, const float *__restrict__ rew, const uint8_t *__restrict__ dn,
                uint32_t *__restrict__ maps_obs, float *__restrict__ vec_obs, uint32_t *__restrict__ maps_next,
                float *__restrict__ vec_next, int32_t *__restrict__ iaction, int32_t *__restrict__ pointer,
                float *__restrict__ reward, uint8_t *__restrict__ done) {
    extern __shared__ __align__(128) uint32_t bits[];      // [2][words], as k_raster
    const int b = blockIdx.x, next = blockIdx.y;
    const long long cP = count * P;
    const long long id = ids[b];
    const long long slot = id / cP, j = id - slot * cP;
    const long long a = j / P;
    const int p = (int)(j - a * P);
    if (!next && threadIdx.x == 1) {
        if (iaction) iaction[b] = act[id];
        if (pointer) reinterpret_cast<int2 *>(pointer)[b] = axy[id];
        if (reward) reward[b] = rew[id];
        if (done) done[b] = dn[id];
    }
    gather_observation(bits, ring, lay, count, next ? (slot + 1) % depth : slot, a, ships[p], b, next ? maps_next : maps_obs,
                       next ? vec_next : vec_obs);
}

// The n-step window of transition (frame t = `slot`, arena x ship j), from the one-step fields of frames t, t+1, ...:
// k frames, ended by a death (done), by the end of the episode after frame t+k, or at k = n.  R = r[t+k-1], then
// R = r[t+i] + gamma * R for i = k-2 .. 0, and discount = gamma^k as k-1 products from gamma, all rounded without fma.
struct NStepWindow {
    int k;
    int done;
    float ret, discount;
};

__device__ __forceinline__ NStepWindow nstep_window(const uint8_t *__restrict__ valid, const uint8_t *__restrict__ dn,
                                                    const float *__restrict__ rew, long long slot, long long j, long long cP,
                                                    int depth, int n, float gamma) {
    NStepWindow w = {n, 0, 0.0f, 0.0f};
    for (int i = 0; i < n; i++) {
        if (dn[((slot + i) % depth) * cP + j]) { w.k = i + 1; w.done = 1; break; }
        if (i + 1 == n) break;
        if (!valid[((slot + i + 1) % depth) * cP + j]) { w.k = i + 1; break; }   // the episode ends after frame t+i+1
    }
    float R = rew[((slot + w.k - 1) % depth) * cP + j];
    for (int i = w.k - 2; i >= 0; i--) R = __fadd_rn(rew[((slot + i) % depth) * cP + j], __fmul_rn(gamma, R));
    float d = gamma;
    for (int i = 1; i < w.k; i++) d = __fmul_rn(d, gamma);
    w.ret = R;
    w.discount = d;
    return w;
}

// k_replay_gather for n-step transitions: obs = frame t, next = frame t+k.  Thread 0 of the next-CTA walks the window before
// the raster; thread 1 of the obs-CTA walks it again to write the scalar fields (at most n bytes and floats each).
__global__ void __launch_bounds__(256)
k_replay_gather_nstep(const char *__restrict__ ring, const ArenaLayout lay, long long count, int P, int depth, int n_step,
                      float gamma, const int32_t *__restrict__ ships, const int32_t *__restrict__ ids,
                      const int32_t *__restrict__ act, const int2 *__restrict__ axy, const float *__restrict__ rew,
                      const uint8_t *__restrict__ valid, const uint8_t *__restrict__ dn, uint32_t *__restrict__ maps_obs,
                      float *__restrict__ vec_obs, uint32_t *__restrict__ maps_next, float *__restrict__ vec_next,
                      int32_t *__restrict__ iaction, int32_t *__restrict__ pointer, float *__restrict__ ret,
                      uint8_t *__restrict__ done, float *__restrict__ discount, int32_t *__restrict__ steps) {
    extern __shared__ __align__(128) uint32_t bits[];
    __shared__ int s_k;
    const int b = blockIdx.x, next = blockIdx.y;
    const long long cP = count * P;
    const long long id = ids[b];
    const long long slot = id / cP, j = id - slot * cP;
    const long long a = j / P;
    const int p = (int)(j - a * P);
    if (next && threadIdx.x == 0) s_k = nstep_window(valid, dn, rew, slot, j, cP, depth, n_step, gamma).k;
    if (!next && threadIdx.x == 1) {
        const NStepWindow w = nstep_window(valid, dn, rew, slot, j, cP, depth, n_step, gamma);
        if (iaction) iaction[b] = act[id];
        if (pointer) reinterpret_cast<int2 *>(pointer)[b] = axy[id];
        if (ret) ret[b] = w.ret;
        if (done) done[b] = (uint8_t)w.done;
        if (discount) discount[b] = w.discount;
        if (steps) steps[b] = w.k;
    }
    if (next) __syncthreads();                             // s_k (uniform branch: the whole CTA takes it)
    gather_observation(bits, ring, lay, count, next ? (slot + s_k) % depth : slot, a, ships[p], b, next ? maps_next : maps_obs,
                       next ? vec_next : vec_obs);
}

// ---------------------------------------------------------------- prioritized sampling: tile sums, scan, one block per draw
// The candidates and their order are ofb_replay_index's; a candidate's mass counts only while it is valid, so invalid
// transitions, the newest frame and slots overwritten by the ring have mass 0 and are never drawn.
__device__ __forceinline__ float prio_mass(const uint8_t *valid, const float *mass, long long c, long long cP, long long n_cand,
                                           int oldest, int depth) {
    if (c >= n_cand) return 0.0f;
    const long long id = replay_id(c, cP, oldest, depth);
    return valid[id] ? mass[id] : 0.0f;
}

__global__ void __launch_bounds__(256)
k_prio_tiles(const uint8_t *__restrict__ valid, const float *__restrict__ mass, long long cP, long long n_cand, int oldest, int depth,
             double *__restrict__ tile_sum, float *__restrict__ tile_min, int32_t *__restrict__ tile_valid) {
    __shared__ double s_sum[8];
    __shared__ float s_min[8];
    __shared__ int s_cnt[8];
    const long long c0 = (long long)blockIdx.x * OFB_REPLAY_TILE + threadIdx.x * 8;
    double s = 0.0;
    float mn = INFINITY;
    int k = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const float m = prio_mass(valid, mass, c0 + i, cP, n_cand, oldest, depth);
        if (m > 0.0f) { s += (double)m; mn = fminf(mn, m); k++; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        k += __shfl_xor_sync(0xffffffffu, k, o);
    }
    if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = s; s_min[threadIdx.x >> 5] = mn; s_cnt[threadIdx.x >> 5] = k; }
    __syncthreads();
    if (threadIdx.x == 0) {                                // (s, mn, k) already hold warp 0's reduction
        for (int w = 1; w < 8; w++) { s += s_sum[w]; mn = fminf(mn, s_min[w]); k += s_cnt[w]; }
        tile_sum[blockIdx.x] = s;
        tile_min[blockIdx.x] = mn;
        tile_valid[blockIdx.x] = k;
    }
}

// One block: exclusive fp64 prefix of the tile sums, the total, the smallest mass, the drawable count.  The prefix is made
// exactly non-decreasing, which the draws' binary search and their order in b rely on: the per-thread chunk sums are scanned,
// their running maximum M_t (exact) starts chunk t + 1, and chunk t's prefixes are clamped to M_t.  total = M_1023.
__global__ void __launch_bounds__(1024)
k_prio_scan(const double *__restrict__ tile_sum, const float *__restrict__ tile_min, const int32_t *__restrict__ tile_valid,
            long long n_tiles, double *__restrict__ tile_prefix, PrioStats *__restrict__ stats, int32_t *__restrict__ n_valid_out) {
    __shared__ double s_sum[1024];
    __shared__ float s_min[32];
    __shared__ int s_cnt[32], s_last[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long per = (n_tiles + 1023) / 1024;
    const long long b0 = tid * per, b1 = min(n_tiles, b0 + per);
    double s = 0.0;
    float mn = INFINITY;
    int k = 0, last = -1;
    for (long long i = b0; i < b1; i++) {
        const double v = tile_sum[i];
        s += v;
        mn = fminf(mn, tile_min[i]);
        k += tile_valid[i];
        if (v > 0.0) last = (int)i;
    }
    s_sum[tid] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                   // Hillis-Steele inclusive scan of the per-thread sums
        const double v = tid >= o ? s_sum[tid - o] : 0.0;
        __syncthreads();
        s_sum[tid] += v;
        __syncthreads();
    }
    for (int o = 1; o < 1024; o <<= 1) {                   // its running maximum: exact, so non-decreasing
        const double v = tid >= o ? s_sum[tid - o] : 0.0;
        __syncthreads();
        s_sum[tid] = fmax(s_sum[tid], v);
        __syncthreads();
    }
    const double hi = s_sum[tid];
    double run = tid > 0 ? s_sum[tid - 1] : 0.0;
    for (long long i = b0; i < b1; i++) {
        tile_prefix[i] = fmin(run, hi);
        run += tile_sum[i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        k += __shfl_xor_sync(0xffffffffu, k, o);
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if (lane == 0) { s_min[warp] = mn; s_cnt[warp] = k; s_last[warp] = last; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 32; w++) { mn = fminf(mn, s_min[w]); k += s_cnt[w]; last = max(last, s_last[w]); }
        stats->total = s_sum[1023];
        stats->mass_min = mn;
        stats->last_tile = last;
        *n_valid_out = k;
    }
}

// Draw b: u = (b + U) / B * total.  Thread 0 binary-searches the tile prefix, then the block scans that tile's masses in fp64
// and takes the first candidate whose inclusive prefix exceeds u.  When rounding leaves u at or past the tile's (or the
// memory's) sum, the last candidate of non-zero mass is taken instead: a zero mass is never drawn.  Every step is
// non-decreasing in u, and u in b, so the draws of one sample are in age order.
__global__ void __launch_bounds__(256)
k_prio_draw(const uint8_t *__restrict__ valid, const float *__restrict__ mass, long long cP, long long n_cand, int oldest, int depth,
            const double *__restrict__ tile_sum, const double *__restrict__ tile_prefix, const PrioStats *__restrict__ stats,
            unsigned long long seed,
            unsigned long long counter, float beta, int B, int32_t *__restrict__ ids_out, float *__restrict__ weight_out) {
    __shared__ int s_tile, s_first, s_last;
    __shared__ double s_r, s_warp[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const PrioStats st = *stats;
    if (!(st.total > 0.0)) return;                         // no drawable transition: n_valid = 0
    if (tid == 0) {
        uint32_t c[4] = {(uint32_t)b, (uint32_t)counter, (uint32_t)(counter >> 32), 0x50524552u};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        const double U = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);   // 53 bits, [0, 1)
        const double u = ((double)b + U) / (double)B * st.total;
        int lo = 0, hi = st.last_tile;                     // the last tile t <= last_tile with prefix[t] <= u
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (tile_prefix[mid] <= u) lo = mid;
            else hi = mid - 1;
        }
        double r = u - tile_prefix[lo];
        if (tile_sum[lo] == 0.0) {                         // an empty tile whose prefix rounded below the next one's:
            while (tile_sum[lo] == 0.0) lo++;              // the next tile with mass (last_tile at the latest), its first
            r = -1.0;                                      // candidate of non-zero mass
        }
        s_tile = lo;
        s_r = r;
        s_first = 0x7fffffff;
        s_last = -1;
    }
    __syncthreads();
    const long long c0 = (long long)s_tile * OFB_REPLAY_TILE + tid * 8;
    const double r = s_r;
    double m[8], own = 0.0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        m[i] = (double)prio_mass(valid, mass, c0 + i, cP, n_cand, oldest, depth);
        own += m[i];
    }
    double incl = own;                                     // block exclusive scan of the per-thread sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    double run = incl - own;
    for (int w = 0; w < warp; w++) run += s_warp[w];
    int first = 0x7fffffff, last = -1;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        run += m[i];
        if (m[i] > 0.0) {
            last = (int)(c0 + i);
            if (run > r && first == 0x7fffffff) first = (int)(c0 + i);
        }
    }
    if (first != 0x7fffffff) atomicMin(&s_first, first);
    if (last >= 0) atomicMax(&s_last, last);
    __syncthreads();
    if (tid == 0) {
        const long long c = s_first != 0x7fffffff ? s_first : s_last;
        const long long id = replay_id(c, cP, oldest, depth);
        ids_out[b] = (int32_t)id;
        // fp32 pow (the fp64 one spills), within a few ulp; mass >= mass_min makes w <= 1, kept so under that rounding.
        // A ratio r past FLT_MAX (a mass clamped to FLT_MAX over a small m_min) would cast to inf and give w = 0: there
        // r = f * 2^e with f in [1, 2), and r^-beta = f^-beta * 2^phi * 2^n with n + phi = -beta * e, n an integer.
        // Below FLT_MAX, e = 0 and scale = 1 exactly, so w is the plain powf.  mass_min is read again here: st.mass_min,
        // kept live across the fp64 division's slow-path calls, spills.
        const double r = (double)mass[id] / (double)stats->mass_min;
        const long long bits = __double_as_longlong(r);
        const bool big = !(r <= 3.402823466e38);
        const int e = big ? (int)(bits >> 52) - 1023 : 0;
        const float base = big ? (float)__longlong_as_double((bits & 0x000fffffffffffffll) | 0x3ff0000000000000ll) : (float)r;
        const double x = -(double)beta * e, n = fmax(floor(x), -250.0);   // 2^x below 2^-250 is 0 in fp32 anyway
        const int n0 = (int)n / 2, n1 = (int)n - n0;                    // 2^n as two normal factors
        const float scale = exp2f((float)(x - n)) * __int_as_float((127 + n0) << 23) * __int_as_float((127 + n1) << 23);
        weight_out[b] = fminf(powf(base, -beta) * scale, 1.0f);
    }
}

__global__ void k_prio_update(const int32_t *__restrict__ ids, const float *__restrict__ td_act, const float *__restrict__ td_ptr, int B,
                              long long n_ids, float alpha, float eps, float *__restrict__ mass, float *__restrict__ max_mass) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long id = ids[b];
    if (id < 0 || id >= n_ids) return;
    float m = (float)pow(fabs((double)td_act[b]) + fabs((double)td_ptr[b]) + (double)eps, (double)alpha);
    if (!(m <= 3.402823466e38f)) m = 3.402823466e38f;     // a non-finite error must not poison the sampler's sums
    mass[id] = m;
    atomicMax(reinterpret_cast<int *>(max_mass), __float_as_int(m));   // masses are >= 0: their bits order like the values
}

// ---------------------------------------------------------------- C ABI
static void replay_free(ofb_replay *r) {
    cudaFree(r->mass);
    cudaFree(r->max_mass);
    cudaFree(r->tile_sum);
    cudaFree(r->tile_prefix);
    cudaFree(r->tile_min);
    cudaFree(r->tile_valid);
    cudaFree(r->stats);
    cudaFree(r->ring);
    cudaFree(r->act);
    cudaFree(r->xy);
    cudaFree(r->reward);
    cudaFree(r->valid);
    cudaFree(r->done);
    cudaFree(r->tile_count);
    cudaFree(r->ships);
    delete r;
}

extern "C" int ofb_replay_create(const ofb_arenas *h, int64_t first, int64_t count, const int32_t *ship_index_host,
                                 int32_t n_policy, int32_t depth, ofb_replay **out) {
    if (!h || !out || !ship_index_host) { ofb_set_error("ofb_replay_create: null argument"); return OFB_E_ARG; }
    if (first < 0 || count < 1 || first + count > h->n_arenas) {
        ofb_set_error("ofb_replay_create: the tracked arenas must lie in [0, %lld)", (long long)h->n_arenas);
        return OFB_E_ARG;
    }
    if (n_policy < 1 || n_policy > h->lay.S || depth < 2) {
        ofb_set_error("ofb_replay_create: need 1 <= P <= n_ships (%d) policy ships and depth >= 2", h->lay.S);
        return OFB_E_ARG;
    }
    const long long cP = (long long)count * n_policy;
    if ((long long)depth * cP >= (1ll << 31)) {
        ofb_set_error("ofb_replay_create: depth x count x P = %lld transitions does not fit int32 ids", (long long)depth * cP);
        return OFB_E_ARG;
    }
    OFB_CUDA_CHECK(cudaSetDevice(h->device));
    ofb_replay *r = new (std::nothrow) ofb_replay();
    if (!r) return OFB_E_NOMEM;
    for (int p = 0; p < n_policy; p++) {
        const int s = ship_index_host[p];
        bool dup = false;
        for (int q = 0; q < p; q++) dup |= ship_index_host[q] == s;
        if (s < 0 || s >= h->lay.S || dup) {
            delete r;
            ofb_set_error("ofb_replay_create: ship indices must be distinct and below n_ships (%d)", h->lay.S);
            return OFB_E_ARG;
        }
    }
    r->h = h;
    r->lay = h->lay;
    r->device = h->device;
    r->first = first;
    r->count = count;
    r->P = n_policy;
    r->depth = depth;
    r->n_step = 1;
    r->pushes = 0;
    r->newest = depth - 1;
    r->n_tiles = ((long long)(depth - 1) * cP + OFB_REPLAY_TILE - 1) / OFB_REPLAY_TILE;
    const size_t nt = (size_t)depth * cP;
    const size_t ring = (size_t)depth * count * h->lay.stride;
    r->bytes = ring + nt * (sizeof(int32_t) + sizeof(int2) + sizeof(float) + 2) + (size_t)r->n_tiles * sizeof(int32_t) +
               n_policy * sizeof(int32_t);
    if (cudaMalloc(&r->ships, n_policy * sizeof(int32_t)) != cudaSuccess || cudaMalloc(&r->ring, ring) != cudaSuccess ||
        cudaMalloc(&r->act, nt * sizeof(int32_t)) != cudaSuccess ||
        cudaMalloc(&r->xy, nt * sizeof(int2)) != cudaSuccess || cudaMalloc(&r->reward, nt * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&r->valid, nt) != cudaSuccess || cudaMalloc(&r->done, nt) != cudaSuccess ||
        cudaMalloc(&r->tile_count, (size_t)r->n_tiles * sizeof(int32_t)) != cudaSuccess) {
        cudaGetLastError();
        ofb_set_error("ofb_replay_create: cudaMalloc of %zu bytes failed", r->bytes);
        replay_free(r);
        return OFB_E_NOMEM;
    }
    if (cudaMemset(r->valid, 0, nt) != cudaSuccess ||
        cudaMemcpy(r->ships, ship_index_host, n_policy * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess) {
        ofb_set_error("ofb_replay_create: initialisation failed: %s", cudaGetErrorString(cudaGetLastError()));
        replay_free(r);
        return OFB_E_CUDA;
    }
    *out = r;
    return OFB_OK;
}

extern "C" int ofb_replay_destroy(ofb_replay *r) {
    if (!r) return OFB_OK;
    cudaSetDevice(r->device);
    replay_free(r);
    return OFB_OK;
}

extern "C" int64_t ofb_replay_device_bytes(const ofb_replay *r) { return r ? (int64_t)r->bytes : OFB_E_ARG; }
extern "C" int64_t ofb_replay_pushes(const ofb_replay *r) { return r ? (int64_t)r->pushes : OFB_E_ARG; }

extern "C" int ofb_replay_set_n_step(ofb_replay *r, int32_t n) {
    if (!r) { ofb_set_error("ofb_replay_set_n_step: null argument"); return OFB_E_ARG; }
    if (r->pushes > 0) { ofb_set_error("ofb_replay_set_n_step: only before the first push"); return OFB_E_ARG; }
    if (n < 1 || n > r->depth - 1) {
        ofb_set_error("ofb_replay_set_n_step: need 1 <= n <= depth - 1 = %d (got %d)", r->depth - 1, n);
        return OFB_E_ARG;
    }
    r->n_step = n;
    return OFB_OK;
}

// Candidates of ofb_replay_index and ofb_replay_sample_prioritized: the frames [T - filled + 1, T - n] of the ring, starting at
// the oldest slot.  Returns their number of frames.
static long long replay_candidates(const ofb_replay *r, int *oldest) {
    const long long filled = r->pushes < r->depth ? r->pushes : r->depth;
    const long long nf = filled > 0 ? filled - 1 : 0;
    *oldest = (int)((r->newest - nf + r->depth) % r->depth);
    return filled > r->n_step ? filled - r->n_step : 0;
}

extern "C" int ofb_replay_push(ofb_replay *r, const ofb_arenas *h, const int32_t *iaction_dev, const int32_t *xy_dev,
                               void *stream) {
    if (!r || !iaction_dev || !xy_dev) { ofb_set_error("ofb_replay_push: null argument"); return OFB_E_ARG; }
    if (h != r->h) { ofb_set_error("ofb_replay_push: the arenas are not the ones the memory was created on"); return OFB_E_ARG; }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    const int slot = (r->newest + 1) % r->depth;
    const int prev = r->pushes > 0 ? r->newest : -1;
    // frame T - n becomes a candidate with this push of frame T = pushes (prev for n = 1)
    const int mslot = r->pushes >= r->n_step ? (slot - r->n_step + r->depth) % r->depth : -1;
    const long long threads = r->count * 32;
    k_replay_push<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        h->state, r->lay, r->first, r->count, r->ships, r->P, r->ring, slot, prev, mslot, iaction_dev,
        reinterpret_cast<const int2 *>(xy_dev), r->act, r->xy, r->reward, r->valid, r->done, r->mass, r->max_mass);
    OFB_CUDA_CHECK(cudaGetLastError());
    r->newest = slot;
    r->pushes += 1;
    return OFB_OK;
}

extern "C" int ofb_replay_index(ofb_replay *r, int32_t *ids_dev, int32_t *count_dev, void *stream) {
    if (!r || !ids_dev || !count_dev) { ofb_set_error("ofb_replay_index: null argument"); return OFB_E_ARG; }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    cudaStream_t st = (cudaStream_t)stream;
    int oldest = 0;
    const long long cP = r->count * r->P, n_cand = replay_candidates(r, &oldest) * cP;
    if (n_cand == 0) {
        OFB_CUDA_CHECK(cudaMemsetAsync(count_dev, 0, sizeof(int32_t), st));
        return OFB_OK;
    }
    const long long tiles = (n_cand + OFB_REPLAY_TILE - 1) / OFB_REPLAY_TILE;
    k_replay_count<<<(unsigned)tiles, 256, 0, st>>>(r->valid, cP, n_cand, oldest, r->depth, r->tile_count);
    k_replay_scan<<<1, 1024, 0, st>>>(r->tile_count, tiles, count_dev);
    k_replay_scatter<<<(unsigned)tiles, 256, 0, st>>>(r->valid, cP, n_cand, oldest, r->depth, r->tile_count, ids_dev);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_replay_gather(const ofb_replay *r, const int32_t *ids_dev, int32_t batch, uint32_t *maps_obs_dev,
                                 float *vec_obs_dev, uint32_t *maps_next_dev, float *vec_next_dev, int32_t *iaction_dev,
                                 int32_t *pointer_dev, float *reward_dev, uint8_t *done_dev, void *stream) {
    if (!r || !ids_dev || batch < 0) { ofb_set_error("ofb_replay_gather: bad argument"); return OFB_E_ARG; }
    if (r->n_step > 1) {
        ofb_set_error("ofb_replay_gather: the memory holds %d-step transitions: use ofb_replay_gather_nstep", r->n_step);
        return OFB_E_ARG;
    }
    if (batch == 0) return OFB_OK;
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    const size_t smem = (size_t)(r->lay.W * r->lay.H / 32) * 2 * sizeof(uint32_t);
    static thread_local SmemAttrCache attr = {};
    if (smem > 48 * 1024) OFB_CUDA_CHECK(attr.ensure(k_replay_gather, (int)smem));
    k_replay_gather<<<dim3((unsigned)batch, 2), 256, smem, (cudaStream_t)stream>>>(
        r->ring, r->lay, r->count, r->P, r->depth, r->ships, ids_dev, r->act, r->xy, r->reward, r->done, maps_obs_dev,
        vec_obs_dev, maps_next_dev, vec_next_dev, iaction_dev, pointer_dev, reward_dev, done_dev);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_replay_gather_nstep(const ofb_replay *r, const int32_t *ids_dev, int32_t batch, float gamma,
                                       uint32_t *maps_obs_dev, float *vec_obs_dev, uint32_t *maps_next_dev, float *vec_next_dev,
                                       int32_t *iaction_dev, int32_t *pointer_dev, float *return_dev, uint8_t *done_dev,
                                       float *discount_dev, int32_t *steps_dev, void *stream) {
    if (!r || !ids_dev || batch < 0) { ofb_set_error("ofb_replay_gather_nstep: bad argument"); return OFB_E_ARG; }
    if (!(gamma >= 0.0f && gamma <= 3.402823466e38f)) {
        ofb_set_error("ofb_replay_gather_nstep: need a finite gamma >= 0 (got %g)", gamma);
        return OFB_E_ARG;
    }
    if (batch == 0) return OFB_OK;
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    const size_t smem = (size_t)(r->lay.W * r->lay.H / 32) * 2 * sizeof(uint32_t);
    static thread_local SmemAttrCache attr = {};
    if (smem > 48 * 1024) OFB_CUDA_CHECK(attr.ensure(k_replay_gather_nstep, (int)smem));
    k_replay_gather_nstep<<<dim3((unsigned)batch, 2), 256, smem, (cudaStream_t)stream>>>(
        r->ring, r->lay, r->count, r->P, r->depth, r->n_step, gamma, r->ships, ids_dev, r->act, r->xy, r->reward, r->valid,
        r->done, maps_obs_dev, vec_obs_dev, maps_next_dev, vec_next_dev, iaction_dev, pointer_dev, return_dev, done_dev,
        discount_dev, steps_dev);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}

// ---------------------------------------------------------------- prioritized replay
extern "C" int ofb_replay_enable_priorities(ofb_replay *r, const ofb_replay_prio_config *cfg) {
    if (!r || !cfg) { ofb_set_error("ofb_replay_enable_priorities: null argument"); return OFB_E_ARG; }
    if (r->mass) { ofb_set_error("ofb_replay_enable_priorities: priorities are already enabled"); return OFB_E_ARG; }
    if (r->pushes > 0) { ofb_set_error("ofb_replay_enable_priorities: only before the first push"); return OFB_E_ARG; }
    if (!(cfg->alpha >= 0.0f && cfg->alpha <= 3.402823466e38f) || !(cfg->eps >= 0.0f && cfg->eps <= 3.402823466e38f)) {
        ofb_set_error("ofb_replay_enable_priorities: need finite alpha >= 0 and eps >= 0 (got %g, %g)", cfg->alpha, cfg->eps);
        return OFB_E_ARG;
    }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    const size_t nt = (size_t)r->depth * r->count * r->P, tiles = (size_t)r->n_tiles;
    const size_t bytes = nt * sizeof(float) + sizeof(float) + tiles * (2 * sizeof(double) + sizeof(float) + sizeof(int32_t)) +
                         sizeof(PrioStats);
    if (cudaMalloc(&r->mass, nt * sizeof(float)) != cudaSuccess || cudaMalloc(&r->max_mass, sizeof(float)) != cudaSuccess ||
        cudaMalloc(&r->tile_sum, tiles * sizeof(double)) != cudaSuccess ||
        cudaMalloc(&r->tile_prefix, tiles * sizeof(double)) != cudaSuccess || cudaMalloc(&r->tile_min, tiles * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&r->tile_valid, tiles * sizeof(int32_t)) != cudaSuccess || cudaMalloc(&r->stats, sizeof(PrioStats)) != cudaSuccess) {
        cudaGetLastError();
        ofb_set_error("ofb_replay_enable_priorities: cudaMalloc of %zu bytes failed", bytes);
        cudaFree(r->mass); cudaFree(r->max_mass); cudaFree(r->tile_sum); cudaFree(r->tile_prefix); cudaFree(r->tile_min);
        cudaFree(r->tile_valid); cudaFree(r->stats);
        r->mass = r->max_mass = r->tile_min = nullptr;
        r->tile_sum = r->tile_prefix = nullptr;
        r->tile_valid = nullptr;
        r->stats = nullptr;
        return OFB_E_NOMEM;
    }
    const float one = 1.0f;
    OFB_CUDA_CHECK(cudaMemset(r->mass, 0, nt * sizeof(float)));
    OFB_CUDA_CHECK(cudaMemset(r->stats, 0, sizeof(PrioStats)));
    OFB_CUDA_CHECK(cudaMemcpy(r->max_mass, &one, sizeof(float), cudaMemcpyHostToDevice));
    r->alpha = cfg->alpha;
    r->eps = cfg->eps;
    r->seed = cfg->seed;
    r->samples = 0;
    r->bytes += bytes;
    return OFB_OK;
}

extern "C" int ofb_replay_sample_prioritized(ofb_replay *r, int32_t batch, float beta, int32_t *ids_out, float *weight_out,
                                             int32_t *n_valid_out, void *stream) {
    if (!r || !ids_out || !weight_out || !n_valid_out) { ofb_set_error("ofb_replay_sample_prioritized: null argument"); return OFB_E_ARG; }
    if (!r->mass) { ofb_set_error("ofb_replay_sample_prioritized: priorities are not enabled"); return OFB_E_ARG; }
    if (batch < 1 || !(beta >= 0.0f && beta <= 3.402823466e38f)) {
        ofb_set_error("ofb_replay_sample_prioritized: need batch >= 1 and finite beta >= 0 (got %d, %g)", batch, beta);
        return OFB_E_ARG;
    }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    cudaStream_t st = (cudaStream_t)stream;
    int oldest = 0;
    const long long cP = r->count * r->P, n_cand = replay_candidates(r, &oldest) * cP;
    if (n_cand == 0) {
        OFB_CUDA_CHECK(cudaMemsetAsync(n_valid_out, 0, sizeof(int32_t), st));
        return OFB_OK;
    }
    const long long tiles = (n_cand + OFB_REPLAY_TILE - 1) / OFB_REPLAY_TILE;
    k_prio_tiles<<<(unsigned)tiles, 256, 0, st>>>(r->valid, r->mass, cP, n_cand, oldest, r->depth, r->tile_sum, r->tile_min,
                                                 r->tile_valid);
    k_prio_scan<<<1, 1024, 0, st>>>(r->tile_sum, r->tile_min, r->tile_valid, tiles, r->tile_prefix, r->stats, n_valid_out);
    k_prio_draw<<<(unsigned)batch, 256, 0, st>>>(r->valid, r->mass, cP, n_cand, oldest, r->depth, r->tile_sum, r->tile_prefix,
                                                 r->stats, r->seed,
                                                 (unsigned long long)r->samples, beta, batch, ids_out, weight_out);
    OFB_CUDA_CHECK(cudaGetLastError());
    r->samples += 1;
    return OFB_OK;
}

extern "C" int ofb_replay_update_priorities(ofb_replay *r, const int32_t *ids_dev, const float *td_act_dev, const float *td_ptr_dev,
                                            int32_t batch, void *stream) {
    if (!r || !ids_dev || !td_act_dev || !td_ptr_dev || batch < 1) {
        ofb_set_error("ofb_replay_update_priorities: bad argument");
        return OFB_E_ARG;
    }
    if (!r->mass) { ofb_set_error("ofb_replay_update_priorities: priorities are not enabled"); return OFB_E_ARG; }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    k_prio_update<<<(unsigned)((batch + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        ids_dev, td_act_dev, td_ptr_dev, batch, (long long)r->depth * r->count * r->P, r->alpha, r->eps, r->mass, r->max_mass);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_replay_read_priorities(const ofb_replay *r, float *mass_dev, float *max_mass_dev, double *last_total_dev,
                                          void *stream) {
    if (!r) { ofb_set_error("ofb_replay_read_priorities: null argument"); return OFB_E_ARG; }
    if (!r->mass) { ofb_set_error("ofb_replay_read_priorities: priorities are not enabled"); return OFB_E_ARG; }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nt = (size_t)r->depth * r->count * r->P;
    if (mass_dev) OFB_CUDA_CHECK(cudaMemcpyAsync(mass_dev, r->mass, nt * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (max_mass_dev) OFB_CUDA_CHECK(cudaMemcpyAsync(max_mass_dev, r->max_mass, sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (last_total_dev) OFB_CUDA_CHECK(cudaMemcpyAsync(last_total_dev, &r->stats->total, sizeof(double), cudaMemcpyDeviceToDevice, st));
    return OFB_OK;
}

// ---------------------------------------------------------------- prioritized replay sharded over ranks
__global__ void k_prio_sample_stats(const PrioStats *__restrict__ stats, double *__restrict__ out) {
    out[0] = stats->total;
    out[1] = (double)stats->mass_min;
}

// w[b] *= ((m_min / M) / g)^(-beta): Schaul's weight over the union of the ranks' memories (include/ofb_replay.h)
__global__ void k_prio_rescale(float *__restrict__ w, int B, float beta, const double *__restrict__ local,
                               const double *__restrict__ g) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double total = local[0], gr = g[0];
    if (!(total > 0.0) || !(gr > 0.0)) return;
    const double f = pow((local[1] / total) / gr, -(double)beta);
    w[b] = (float)((double)w[b] * f);
}

extern "C" int ofb_replay_sample_stats(const ofb_replay *r, double *out_dev, void *stream) {
    if (!r || !out_dev) { ofb_set_error("ofb_replay_sample_stats: null argument"); return OFB_E_ARG; }
    if (!r->mass) { ofb_set_error("ofb_replay_sample_stats: priorities are not enabled"); return OFB_E_ARG; }
    OFB_CUDA_CHECK(cudaSetDevice(r->device));
    k_prio_sample_stats<<<1, 1, 0, (cudaStream_t)stream>>>(r->stats, out_dev);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_replay_rescale_weights(float *weight_dev, int32_t batch, float beta, const double *local_stats_dev,
                                          const double *global_ratio_dev, void *stream) {
    if (!weight_dev || !local_stats_dev || !global_ratio_dev || batch < 1 || !(beta >= 0.0f && beta <= 3.402823466e38f)) {
        ofb_set_error("ofb_replay_rescale_weights: bad argument (need buffers, batch >= 1 and a finite beta >= 0)");
        return OFB_E_ARG;
    }
    k_prio_rescale<<<(unsigned)((batch + 127) / 128), 128, 0, (cudaStream_t)stream>>>(weight_dev, batch, beta, local_stats_dev,
                                                                                    global_ratio_dev);
    OFB_CUDA_CHECK(cudaGetLastError());
    return OFB_OK;
}
