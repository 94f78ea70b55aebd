// ssd_b200.cu -- sm_100a kernels + C ABI of the batched SSD grid-world simulator.
//
// Design (DESIGN.md): one warp owns one env instance for a whole step.
//   * lanes 0..n-1 ARE the agents during move/rotate, conflict resolution, consume and beams:
//     collisions, swaps, chains and cycles are resolved with __ballot/__shfl/redux (bit-filter pre-tests
//     with REDUX.OR, exact shuffle loops only on a possible hit), keeping the reference's sequential
//     phase structure (map_env.py:477-661);
//   * lanes are spawn candidates during apple/waste spawning (4 apple points or 2 waste
//     points per Philox4x32-10 call);
//   * lanes are output pixel ROWS during the egocentric render.  Small views (N <= 16, Cleanup) are
//     gathered straight from the staged byte grid; large views (Harvest, N = 31) read one run of N
//     nibbles from a zero-padded nibble-packed index map (or its transpose) held in shared memory.
//     Either way a lane colours 4 pixels per PRMT through an 8-entry register LUT and writes the
//     finished row with one 256-bit (st.global.v8.b32, SASS STG.E.ENL2.256) or 128-bit store per plane.
// The env's grid is staged in shared memory for the whole step.  No tensor cores: nothing here is a
// contraction.  HBM traffic per env-step is the algorithmic 2G + n(3N^2+11)+3 bytes (+ row padding),
// ~98% of it observation WRITES.
//
// Reference citations are relative to drdh/Homophily-MARL.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <new>
#include <mutex>

#include "ssd_b200.h"

namespace {

constexpr int kWarps = 4;                 // env instances per CTA
constexpr int kMinBlocks = 8;             // __launch_bounds__ minimum of resident CTAs per SM
using ColourLuts = uint32_t[kWarps][16];  // ssd_kernel's static shared memory: one colour LUT per warp
constexpr uint16_t kNoPoint = 0xFFFF;
constexpr int kMaxDevices = 64;

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_RENDER = 2, MODE_STEP_RESET = 3 };   // MODE_STEP_RESET: ssd_step_autoreset

// -DSSD_BOUNDS_CHECK builds the checked variant (libssd_b200_check.so): every data-dependent shared-memory index is
// tested against its tile and violations are counted (compute-sanitizer is closed on the GPU pool).
#ifdef SSD_BOUNDS_CHECK
__device__ unsigned long long g_oob_count = 0;
#define SSD_CHECK(cond) do { if (!(cond)) atomicAdd(&g_oob_count, 1ull); } while (0)
#else
#define SSD_CHECK(cond) do { } while (0)
#endif

// Static per-map tables, resident in global memory (read through the L1 read-only path).
struct MapDev {
    uint8_t  base_grid[SSD_MAX_CELLS];        // reset grid in cell codes
    uint16_t apple_pts[SSD_MAX_CELLS + 4];    // row-major, padded to x4 with kNoPoint
    uint16_t waste_pts[SSD_MAX_CELLS + 4];    // padded to x2
    uint16_t spawn_pts[SSD_MAX_SPAWN];
    uint32_t thr_apple[SSD_MAX_CELLS + 1];
    uint32_t thr_waste[SSD_MAX_CELLS + 1];
};

// One env variant (ssd_set_variants): its map tables and the scalars that may differ between the variants of a handle.
struct VarDev {
    MapDev map;
    int n_apple, n_waste, n_spawn, n_apple4, n_waste2;
    int base_apples, base_waste;
    int fire_cost, hit_penalty, tag_timeout;
    uint32_t thr_harvest[4];
};

// ------------------------------------------------------------------ geometry
// Everything that follows from (kind, H, W, V).  Computed by ONE constexpr function used by the host
// (ssd_create) and, for the reference's shipped maps, at compile time by the kernels (GeoS), so that index
// arithmetic folds into immediates; any other geometry runs the same code on runtime values (GeoD).
struct GeoVals {
    int kind, H, W, V, G, GS, N, RP, PS, AS, LPn, nw8M, nw8T, pitchM, pitchT, PMS;
    int off_map[4];                           // byte offset of the nibble map read by orientation: 0,1 (LEFT/RIGHT) -> MT, 2,3 -> M
    int direct, padF, padB;                   // small views (RP <= 16) are gathered straight from the staged grid: no maps, but
                                              // V rows of slack before / after the grid so that column runs need no bounds test
    uint32_t maskM8;                          // valid-nibble mask of the last word of a map row
    int RS4, AS4;                             // SSD_OBS_INDEX4: bytes per row (ceil(N/2) rounded to 4) and per agent (rounded to 16)
};
__host__ __device__ constexpr int cround_up(int v, int m) { return (v + m - 1) / m * m; }
__host__ __device__ constexpr GeoVals make_geo(int kind, int H, int W, int V) {
    GeoVals g{};
    g.kind = kind; g.H = H; g.W = W; g.V = V; g.G = H * W; g.GS = cround_up(H * W, 16);
    g.N = 2 * V + 1; g.RP = cround_up(g.N, 4); g.PS = g.N * g.RP; g.AS = cround_up(3 * g.PS, 16);
    // nibble-packed padded maps; word pitch kept odd so that lanes gathering consecutive rows hit distinct banks
    g.LPn = cround_up(V, 8); g.nw8M = (W + 7) / 8; g.nw8T = (H + 7) / 8;
    g.maskM8 = (W & 7) ? (1u << (4 * (W & 7))) - 1u : 0xffffffffu;
    int wm = (g.LPn + W + V + 7) / 8; if (wm < g.LPn / 8 + g.nw8M) wm = g.LPn / 8 + g.nw8M; if ((wm & 1) == 0) ++wm;
    int wt = (g.LPn + H + V + 7) / 8; if (wt < g.LPn / 8 + g.nw8T) wt = g.LPn / 8 + g.nw8T; if ((wt & 1) == 0) ++wt;
    g.pitchM = 4 * wm; g.pitchT = 4 * wt;
    const int szM = cround_up((H + 2 * V) * g.pitchM, 16) + 16, szT = cround_up((W + 2 * V) * g.pitchT, 16) + 16;
    g.off_map[0] = 16; g.off_map[1] = 16; g.off_map[2] = 16 + szT; g.off_map[3] = 16 + szT;
    g.PMS = szT + szM + 32;
    g.direct = g.RP <= 16;
    g.padF = g.direct ? cround_up(V * W + 48, 16) : 16;      // + 32 bytes at the very front for the (class, rank) -> lane table
    g.padB = g.direct ? cround_up(V * W + 32, 16) : 32;
    if (g.direct) g.PMS = 0;
    g.RS4 = cround_up((g.N + 1) / 2, 4); g.AS4 = cround_up(g.N * g.RS4, 16);
    return g;
}

struct KParams {
    GeoVals geo;                              // make_geo(kind, H, W, V)
    int B, n;
    int env0, env1;                           // this launch covers env instances [env0, env1) of the B resident ones
    int pdl;                                  // launched with the programmatic-serialization attribute (set per launch)
    int NA;                                   // agent stride (ssd_layout)
    int agents_uniform;                       // all agent colours equal -> no per-agent repaint
    int episode_limit, fire_cost, hit_penalty, beam_len, n_actions;
    int n_apple, n_waste, n_spawn, n_apple4, n_waste2;
    int random_spawn, spawn_rot;
    int base_apples, base_waste;              // 'A' / 'H' cells of the reset grid (cell counts are carried in ssd_state.counts)
    uint32_t invN20, invW20, invMW20;         // GeoD's divisions: floor(x / d) == (x * inv) >> 20 on the used ranges
    uint32_t seed_lo, seed_hi, gid_base;
    uint32_t thr_harvest[4];
    uint32_t lut[16];
    uint32_t lut8[6];                         // 8-entry colour LUT per plane (lo, hi words): R, G, B
    const MapDev* map;
    uint8_t* grid; uint32_t* agent; int32_t* ep_ret; int32_t* t; uint32_t* tick; uint32_t* counts;
    const uint8_t* actions; const uint8_t* mask;
    int8_t* reward; uint8_t* clean; uint16_t* apple_cnt; uint8_t* done; uint8_t* obs; uint8_t* state_rgb;
    const uint32_t* d_prio; const uint32_t* d_uapple; const uint32_t* d_uwaste; const uint32_t* d_wkey;
    const uint32_t* d_spawnkey; const uint8_t* d_rot;
    int tag_timeout;                          // steps a FIRE-hit agent stays off the map (0: never; DESIGN.md §3 item 11)
    int state_idx4;                           // state_rgb holds packed colour indices (SSD_OBS_INDEX4; DESIGN.md §3 item 13)
    uint8_t* end_obs; uint8_t* end_state; int32_t* end_ep_ret;   // MODE_STEP_RESET: ssd_episode_end (DESIGN.md §3 item 14)
    const uint8_t* variant_of;                // [B] variant id per env (ssd_set_env_variants), or NULL: the fields above (variant 0)
    const VarDev* variants;                   // the variant table (n_variants records), read only when variant_of is set
    int n_variants;
    uint32_t* stats; uint32_t* end_stats;     // STATS kernels: per-agent episode counters (ssd_set_stats; DESIGN.md §3 item 16)
};

// STATS: one agent's counter deltas of a step, packed in one register so that the step's live registers stay flat.  Bits: 0 ate an
// apple, 1 fired, 2 started the step out of play, 3-4 FIRE rays of its beam that hit an agent (<= 3), 5-10 rays that hit it
// (<= 3 per shooter, <= 48).
constexpr uint32_t kSdAte = 1u, kSdFire = 2u, kSdOut = 4u;
constexpr int kSdDealt = 3, kSdTaken = 5;

// The variant an env runs (DESIGN.md §3 item 15).  VAR = false (no id array): every read is the KParams field it always was, and
// the kernel is the code it was before variants existed.  VAR: a load from the env's record in the variant table.  Warp-uniform:
// one warp owns one env.
template <bool VAR>
struct Var {
    static constexpr bool kVar = VAR;
    const KParams& p;
    int id;
    __device__ __forceinline__ const VarDev* d() const { return p.variants + id; }
    __device__ __forceinline__ const MapDev* map() const { return VAR ? &d()->map : p.map; }
#define SSD_VAR_FIELD(f) __device__ __forceinline__ int f() const { return VAR ? __ldg(&d()->f) : p.f; }
    SSD_VAR_FIELD(n_apple4) SSD_VAR_FIELD(n_waste) SSD_VAR_FIELD(n_waste2) SSD_VAR_FIELD(n_spawn)
    SSD_VAR_FIELD(base_apples) SSD_VAR_FIELD(base_waste) SSD_VAR_FIELD(fire_cost) SSD_VAR_FIELD(hit_penalty)
    SSD_VAR_FIELD(tag_timeout)
#undef SSD_VAR_FIELD
    __device__ __forceinline__ uint32_t thr_harvest(int k) const { return VAR ? __ldg(&d()->thr_harvest[k]) : p.thr_harvest[k]; }
};

// The geometry accessors, over D::vals(): compile-time constants (GeoS) or the launch's KParams::geo (GeoD).  Only the
// divisions and the by-orientation map offset are written per class: GeoS folds constants where GeoD indexes its values.
template <class D>
struct GeoAccess {
    __device__ __forceinline__ int kind() const { return v().kind; }
    __device__ __forceinline__ int H() const { return v().H; }
    __device__ __forceinline__ int W() const { return v().W; }
    __device__ __forceinline__ int V() const { return v().V; }
    __device__ __forceinline__ int G() const { return v().G; }
    __device__ __forceinline__ int GS() const { return v().GS; }
    __device__ __forceinline__ int N() const { return v().N; }
    __device__ __forceinline__ int RP() const { return v().RP; }
    __device__ __forceinline__ int PS() const { return v().PS; }
    __device__ __forceinline__ int AS() const { return v().AS; }
    __device__ __forceinline__ int RS4() const { return v().RS4; }
    __device__ __forceinline__ int AS4() const { return v().AS4; }
    __device__ __forceinline__ int LPn() const { return v().LPn; }
    __device__ __forceinline__ int nw8M() const { return v().nw8M; }
    __device__ __forceinline__ int nw8T() const { return v().nw8T; }
    __device__ __forceinline__ int pitchM() const { return v().pitchM; }
    __device__ __forceinline__ int pitchT() const { return v().pitchT; }
    __device__ __forceinline__ int PMS() const { return v().PMS; }
    __device__ __forceinline__ bool direct() const { return v().direct != 0; }
    __device__ __forceinline__ int padF() const { return v().padF; }
    __device__ __forceinline__ int padB() const { return v().padB; }
    __device__ __forceinline__ uint32_t maskM8() const { return v().maskM8; }
private:
    __device__ __forceinline__ decltype(auto) v() const { return static_cast<const D*>(this)->vals(); }
};

template <int KIND_, int H_, int W_, int V_>
struct GeoS : GeoAccess<GeoS<KIND_, H_, W_, V_>> {          // compile-time geometry
    static constexpr GeoVals v = make_geo(KIND_, H_, W_, V_);
    __device__ __forceinline__ explicit GeoS(const KParams&) {}
    __device__ __forceinline__ static constexpr GeoVals vals() { return v; }
    __device__ __forceinline__ int off_map(int o) const {
        constexpr int o0 = v.off_map[0], o1 = v.off_map[1], o2 = v.off_map[2], o3 = v.off_map[3];
        return o == 0 ? o0 : (o == 1 ? o1 : (o == 2 ? o2 : o3));
    }
    __device__ __forceinline__ int divW(int x) const { return (int)((unsigned)x / (unsigned)v.W); }
    __device__ __forceinline__ int divN(int x) const { return (int)((unsigned)x / (unsigned)v.N); }
    __device__ __forceinline__ int divMW(int x) const { return (int)((unsigned)x / (unsigned)v.nw8M); }
};

struct GeoD : GeoAccess<GeoD> {                               // runtime geometry (any wall-enclosed map)
    const KParams& p;
    __device__ __forceinline__ explicit GeoD(const KParams& p_) : p(p_) {}
    __device__ __forceinline__ const GeoVals& vals() const { return p.geo; }
    __device__ __forceinline__ int off_map(int o) const { return p.geo.off_map[o]; }
    __device__ __forceinline__ int divW(int x) const { return (int)(((uint32_t)x * p.invW20) >> 20); }
    __device__ __forceinline__ int divN(int x) const { return (int)(((uint32_t)x * p.invN20) >> 20); }
    __device__ __forceinline__ int divMW(int x) const { return (int)(((uint32_t)x * p.invMW20) >> 20); }
};

// ------------------------------------------------------------------ Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint32_t pick(const uint4& v, int i) {
    return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}
// The lanes of the warp that owns an env instance, and the full-warp collectives the device functions use.
struct Warp {
    int lane;
    __device__ __forceinline__ explicit Warp(int lane_) : lane(lane_) {}
    __device__ __forceinline__ unsigned ballot(bool pred) const { return __ballot_sync(0xffffffffu, pred); }
    template <typename T> __device__ __forceinline__ T shfl(T v, int src) const { return __shfl_sync(0xffffffffu, v, src); }
    template <typename T> __device__ __forceinline__ T rmin(T v) const { return __reduce_min_sync(0xffffffffu, v); }
    template <typename T> __device__ __forceinline__ T rmax(T v) const { return __reduce_max_sync(0xffffffffu, v); }
    template <typename T> __device__ __forceinline__ T radd(T v) const { return __reduce_add_sync(0xffffffffu, v); }
    __device__ __forceinline__ unsigned ror(unsigned v) const { return __reduce_or_sync(0xffffffffu, v); }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};

// lanes j < n whose value equals this lane's: what __match_any_sync returns for the agent lanes, from n pipelined shuffles
// (MATCH.ANY costs 3-4 % of a Cleanup step per use, profiles/r2_notes.md)
__device__ __forceinline__ unsigned equal_lanes(const Warp& w, int v, int n) {
    unsigned m = 0;
    for (int j = 0; j < n; ++j) m |= (unsigned)(w.shfl(v, j) == v) << j;
    return m;
}
// Cheap sufficient test for "the values of the lanes in `who` are pairwise distinct": two 32-bucket bit filters, OR-reduced over
// the warp (REDUX.OR); if either filter shows one bit per participating lane there is no duplicate.  False alarms (hash
// collisions) only send the caller to the exact shuffle loop.
__device__ __forceinline__ bool surely_distinct(const Warp& w, int v, bool in, unsigned who) {
    const int cnt = __popc(who);
    const unsigned f0 = w.ror(in ? 1u << (v & 31) : 0u);
    if (__popc(f0) == cnt) return true;
    const unsigned f1 = w.ror(in ? 1u << ((v >> 5) & 31) : 0u);
    return __popc(f1) == cnt;
}

// warp-strided loop with the first trip peeled (trip counts here are almost always 0 or 1)
template <typename F>
__device__ __forceinline__ void warp_for(int n, int lane, F f) {
    int i = lane;
    if (i < n) f(i);
    for (i += 32; i < n; i += 32) f(i);
}
// draw streams: 0 mover priority, 1 apple, 2 waste (u, order key), 3 spawn key, 4 spawn rotation
__device__ __forceinline__ uint32_t philox_word(const KParams& p, uint32_t gid, uint32_t tick, uint32_t stream, uint32_t idx) {
    const uint4 r = philox4x32_10(gid, tick, stream, idx >> 2, p.seed_lo, p.seed_hi);
    return pick(r, idx & 3);
}

// agent i is drawn as the first char of str(i % 10 + 1)  (map_env.py:370 into a <U1 array)
__device__ __forceinline__ int agent_colour_index(int i) {
    const int v = i % 10 + 1;
    return 6 + (v == 10 ? 1 : v);
}

// ------------------------------------------------------------------ update_moves (map_env.py:477-661)
// lanes < n hold one agent each: pos (cell index), ori, act.  Non-agent lanes carry unique
// negative positions so they never match a cell.
template <class GEO>
__device__ __forceinline__ void update_moves(const Warp& w, const GEO& g, const KParams& p, const uint8_t* __restrict__ sg, int lane, bool is_agent,
                                             int act, int& pos, int& ori, int env, uint32_t gid, uint32_t tick) {
    // turns take effect immediately (map_env.py:509-511, 843-861)
    if (act == 5) ori = (0x0132 >> (4 * ori)) & 3;           // CW : LEFT->UP, RIGHT->DOWN, UP->RIGHT, DOWN->LEFT
    else if (act == 6) ori = (0x1023 >> (4 * ori)) & 3;      // CCW: LEFT->DOWN, RIGHT->UP, UP->LEFT, DOWN->RIGHT
    const bool mover = is_agent && act <= 4;
    int prop = pos;
    if (mover && act < 4) {
        // (drow, dcol) of action a under orientation o, 2-bit fields holding value+1 (map_env.py:826-835)
        //   LEFT : (0,+1) (0,-1) (-1,0) (+1,0)   RIGHT: (0,-1) (0,+1) (+1,0) (-1,0)
        //   UP   : (-1,0) (+1,0) (0,-1) (0,+1)   DOWN : (+1,0) (-1,0) (0,+1) (0,-1)
        constexpr uint32_t kDr = (1u) | (1u << 2) | (0u << 4) | (2u << 6) | (1u << 8) | (1u << 10) | (2u << 12) | (0u << 14) |
                                 (0u << 16) | (2u << 18) | (1u << 20) | (1u << 22) | (2u << 24) | (0u << 26) | (1u << 28) | (1u << 30);
        constexpr uint32_t kDc = (2u) | (0u << 2) | (1u << 4) | (1u << 6) | (0u << 8) | (2u << 10) | (1u << 12) | (1u << 14) |
                                 (1u << 16) | (1u << 18) | (0u << 20) | (2u << 22) | (1u << 24) | (1u << 26) | (2u << 28) | (0u << 30);
        const int f = 2 * (ori * 4 + act);
        const int dr = (int)((kDr >> f) & 3u) - 1, dc = (int)((kDc >> f) & 3u) - 1;
        const int q = pos + dr * g.W() + dc;
        SSD_CHECK(q >= 0 && q < g.G());
        prop = sg[q] == SSD_CELL_WALL ? pos : q;             // agent.py:111-119
    }
    unsigned in_moves = w.ballot(mover);
    if (in_moves == 0) return;                                // map_env.py:534
    int mv = prop;                                            // live agent_moves[i]

    // ---- phase 1: contested cells in lexicographic order of the ORIGINAL proposals (543-609)
    unsigned pending = 0;                                     // movers whose proposal is shared with another mover
    if (!surely_distinct(w, prop, mover, in_moves)) {
        const unsigned grp = equal_lanes(w, mover ? prop : -1000 - lane, p.n);
        pending = w.ballot(mover && __popc(grp) >= 2);
    }
    if (pending) {
        uint32_t prio = 0;
        if (mover) prio = p.d_prio ? p.d_prio[(size_t)env * p.n + lane] : philox_word(p, gid, tick, 0, (uint32_t)lane);
        while (pending) {
            const int cell = w.rmin(((pending >> lane) & 1u) ? prop : 0x7fffffff);
            const bool in_cont = mover && prop == cell;
            const unsigned cont = w.ballot(in_cont);
            const unsigned occm = w.ballot(pos == cell);          // live positions (567)
            bool free_cell = true;
            if (occm) {
                const int occ = 31 - __clz(occm);                              // dict build: last index wins (516)
                const int mv_occ = w.shfl(mv, occ);
                const bool occ_moves = (in_moves >> occ) & 1u;
                const bool c1 = (cont >> occ) & 1u;                            // (1) 578
                const bool c2 = !occ_moves || mv_occ == cell;                  // (2) 584-586
                const unsigned swp = w.ballot(in_cont && mv_occ == pos);   // (3) 590-594
                free_cell = !(c1 || c2 || swp != 0);
            }
            if (free_cell) {                                                   // winner = first in shuffled order (598-601)
                const uint32_t mk = w.rmin(in_cont ? prio : 0xffffffffu);
                const unsigned eq = w.ballot(in_cont && prio == mk);
                if (lane == __ffs(eq) - 1) pos = cell;
            }
            if (in_cont) mv = pos;                                             // 604-609
            pending &= ~cont;
        }
    }
    // ---- phase 2: iterate until every move is made or dropped (612-661)
    // Fast path: if no mover's target is occupied by ANOTHER agent, the sequential walk below moves every mover (targets are
    // unique after phase 1 or the mover's own cell, and nobody enters a cell that is somebody's target), so all move at once.
    // (A mover whose target is its own cell never changes anything, whoever else stands there.)  The occupancy test is first
    // made against a 32-bucket bit filter of all agents' cells; only a possible hit pays for the exact shuffle loop.
    {
        const bool mine = (in_moves >> lane) & 1u;
        const unsigned cells = w.ror(is_agent ? 1u << (pos & 31) : 0u);
        bool blocked = mine && mv != pos && ((cells >> (mv & 31)) & 1u);
        if (w.ballot(blocked)) {
            blocked = false;
            for (int j = 0; j < p.n; ++j) blocked |= (w.shfl(pos, j) == mv) && (j != lane);
            blocked = blocked && mine && mv != pos;
        }
        if (w.ballot(blocked) == 0) {
            if (mine) pos = mv;
            return;
        }
    }
    while (in_moves) {
        const int spos = pos;                                  // snapshot dict of this pass (613)
        const unsigned snap = in_moves;
        unsigned todo = snap;
        while (todo) {
            const int i = __ffs(todo) - 1;
            todo &= todo - 1;
            if (!((in_moves >> i) & 1u)) continue;             // deleted earlier in this pass (619-620)
            const int mvi = w.shfl(mv, i);
            const int posi = w.shfl(pos, i);
            const unsigned live = w.ballot(pos == mvi);            // 621
            if (!live) {                                                       // 650-653
                if (lane == i) pos = mvi;
                in_moves &= ~(1u << i);
                continue;
            }
            const unsigned sm = w.ballot(spos == mvi);
            if (!sm) { in_moves &= ~(1u << i); continue; }                     // reference KeyError; unreachable (DESIGN.md)
            const int occ = 31 - __clz(sm);
            const int pos_occ = w.shfl(pos, occ);
            const int mv_occ = w.shfl(mv, occ);
            const int occ_mv = ((in_moves >> occ) & 1u) ? mv_occ : pos_occ;
            if (occ == i) in_moves &= ~(1u << i);                                              // (1) 630
            else if (!((snap >> occ) & 1u) || pos_occ == occ_mv) in_moves &= ~(1u << i);       // (2) 636-639
            else if (mv_occ == posi && mvi == pos_occ) in_moves &= ~((1u << i) | (1u << occ)); // (3) 642-648
        }
        if (in_moves == snap) {                                // nobody could move: rotate cycles together (658-661)
            if ((in_moves >> lane) & 1u) pos = mv;
            break;
        }
    }
}

// Agent occupancy is kept IN the staged grid: bit 7 of a cell byte is set while an agent stands on it
// (the dict `agent_by_pos` / `[r, c] in self.agent_pos` tests of the reference become one bit test).
constexpr uint8_t kOcc = 0x80;

// ------------------------------------------------------------------ beams (map_env.py:663-769)
// TAG: every agent a FIRE ray hits (the one hit_penalty charges) sets `tagged`; it stays on the map until all beams are done.
// In a TAG launch an env whose variant has tag_timeout 0 tags nobody, exactly like the kernel without TAG.
template <bool TAG, class GEO, class VR>
__device__ __forceinline__ void beams(const Warp& w, const GEO& g, const KParams& p, const VR& vr, uint8_t* sg, int lane, bool is_agent,
                                      int act, int pos, int ori, int& reward, int& clean_num, int& waste, bool& tagged) {
    const bool fire = is_agent && act == 7;
    const bool clean = is_agent && act == 8 && g.kind() == SSD_KIND_CLEANUP;
    if (fire) reward -= vr.fire_cost();                       // agent.py:188-190, 239-241
    unsigned need = w.ballot(clean || (fire && (TAG || vr.hit_penalty() != 0)));
    while (need) {                                            // agent index order, map effects applied per agent (669-671)
        const int i = __ffs(need) - 1;
        need &= need - 1;
        const int posi = w.shfl(pos, i), orii = w.shfl(ori, i);
        const bool is_clean = w.shfl(act, i) == 8;
        // firing direction ORIENTATIONS[o] and its right-hand rotation (map_env.py:28-31, 840-841)
        const int dr = orii == 0 ? -1 : (orii == 1 ? 1 : 0), dc = orii == 2 ? -1 : (orii == 3 ? 1 : 0);
        const int rr = orii == 2 ? 1 : (orii == 3 ? -1 : 0), rc = orii == 0 ? -1 : (orii == 1 ? 1 : 0);
        const int d = dr * g.W() + dc, rs = rr * g.W() + rc;
        int upd = -1, hit = -1;
        if (lane < 3) {                                       // the three parallel rays (728-730)
            int q = posi + (lane == 0 ? d : (lane == 1 ? rs : -rs));
            for (int k = 0; k < p.beam_len; ++k) {            // maps are wall-enclosed: a ray cannot leave the map
                SSD_CHECK(q >= 0 && q < g.G());
                const int v = sg[q], code = v & 0x7f;
                if (code == SSD_CELL_WALL) break;             // 737
                if (v & kOcc) {                               // agents absorb beams (741-749)
                    if (!is_clean) hit = q;
                    if (is_clean && code == SSD_CELL_WASTE) upd = q;
                    break;
                }
                if (is_clean && code == SSD_CELL_WASTE) { upd = q; break; }   // 752-760
                q += d;
            }
        }
        w.sync();
        if (upd >= 0) sg[upd] = (uint8_t)(SSD_CELL_RIVER | (sg[upd] & kOcc));
        w.sync();
        const unsigned um = w.ballot(upd >= 0);
        if (lane == i && is_clean) clean_num = __popc(um);    // 672-673
        waste -= __popc(um);                                  // only CLEAN produces updates: 'H' -> 'R'
        if (TAG || vr.hit_penalty() != 0) {                   // hit(): the LAST index standing on the cell (agent.py:184-186)
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const int hq = w.shfl(hit, s);
                const unsigned on = w.ballot(hq >= 0 && pos == hq);
                if (on && lane == 31 - __clz(on)) {
                    reward -= vr.hit_penalty();
                    if (TAG && (!VR::kVar || vr.tag_timeout() != 0)) tagged = true;   // without variants TAG means tag_timeout > 0
                }
            }
        }
    }
}

// STATS: the FIRE rays of the step once more, for the episode counters (DESIGN.md §3 item 16), after beams() and before the tagged
// leave the map.  A FIRE ray stops at a wall or at the first cell an agent in play stands on, and neither changes during the beam
// phase (CLEAN only turns waste into river; tagged agents stay on the map until every beam is done), so this walk finds the cells
// beams() hit, whatever order the beams ran in.  Returns the lane's kSdFire, kSdDealt and kSdTaken bits.  A pass of its own:
// walking FIRE rays inside beams() whatever hit_penalty is spilled the Harvest V=15 auto-reset kernel with variants.
template <class GEO>
__device__ __forceinline__ uint32_t fire_counts(const Warp& w, const GEO& g, const KParams& p, const uint8_t* sg, int lane, bool is_agent,
                                                int act, int pos, int ori) {
    const bool fire = is_agent && act == 7;
    uint32_t sd = fire ? kSdFire : 0u;
    unsigned need = w.ballot(fire);
    while (need) {
        const int i = __ffs(need) - 1;
        need &= need - 1;
        const int posi = w.shfl(pos, i), orii = w.shfl(ori, i);
        const int dr = orii == 0 ? -1 : (orii == 1 ? 1 : 0), dc = orii == 2 ? -1 : (orii == 3 ? 1 : 0);
        const int rr = orii == 2 ? 1 : (orii == 3 ? -1 : 0), rc = orii == 0 ? -1 : (orii == 1 ? 1 : 0);
        const int d = dr * g.W() + dc, rs = rr * g.W() + rc;
        int hit = -1;
        if (lane < 3) {
            int q = posi + (lane == 0 ? d : (lane == 1 ? rs : -rs));
            for (int k = 0; k < p.beam_len; ++k) {
                SSD_CHECK(q >= 0 && q < g.G());
                const int v = sg[q];
                if ((v & 0x7f) == SSD_CELL_WALL) break;
                if (v & kOcc) { hit = q; break; }
                q += d;
            }
        }
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int hq = w.shfl(hit, s);
            const unsigned on = w.ballot(hq >= 0 && pos == hq);
            if (on && lane == 31 - __clz(on)) sd += 1u << kSdTaken;   // the agent hit_penalty charges
            if (on && lane == i) sd += 1u << kSdDealt;
        }
    }
    return sd;
}

// ------------------------------------------------------------------ spawning (cleanup.py:165-204, harvest.py:92-122)
// `apples` / `waste` are the env's running cell counts (ssd_state.counts): the reference recounts the map every step
// (map_env.py:291-292, cleanup.py:206-212); here consume / clean / spawn keep them up to date, which is the same number.
template <class GEO, class VR>
__device__ __forceinline__ void spawn(const Warp& w, const GEO& g, const KParams& p, const VR& vr, uint8_t* sg, int lane, int env,
                                      uint32_t gid, uint32_t tick, int& apples, int& waste) {
    const MapDev* __restrict__ m = vr.map();
    uint32_t tA = 1, tW = 0;
    if (g.kind() == SSD_KIND_CLEANUP) {
        SSD_CHECK(waste >= 0 && waste <= vr.n_waste());
        tA = __ldg(&m->thr_apple[waste]);
        tW = __ldg(&m->thr_waste[waste]);
    }
    // apples: 4 candidate points per lane per Philox call; decisions use the pre-spawn grid.  In Cleanup a decision reads
    // only its own cell (and apple points and waste points are different cells), so the apple is written at once; Harvest's
    // 3x3 neighbour count needs every decision to see the pre-spawn grid, so its apples are applied in a second pass.
    unsigned long long decided = 0;
    int n_new = 0;
    if (tA != 0) {
        int it = 0;
        for (int j = lane; j < vr.n_apple4(); j += 32, ++it) {
            const ushort4 pts = __ldg(reinterpret_cast<const ushort4*>(m->apple_pts) + j);
            const uint16_t c4[4] = { pts.x, pts.y, pts.z, pts.w };
            uint4 r = make_uint4(0, 0, 0, 0);
            if (!p.d_uapple) r = philox4x32_10(gid, tick, 1u, (uint32_t)j, p.seed_lo, p.seed_hi);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int c = c4[q];
                if (c == kNoPoint) continue;
                const int v = sg[c];
                if ((v & kOcc) || v == SSD_CELL_APPLE) continue;               // cleanup.py:171, harvest.py:105
                uint32_t thr = tA;
                if (g.kind() == SSD_KIND_HARVEST) {
                    int cnt = 0;                                               // j^2+k^2 <= 2: the 3x3 block (harvest.py:107-116)
#pragma unroll
                    SSD_CHECK(c - g.W() - 1 >= 0 && c + g.W() + 1 < g.G());
#pragma unroll
                    for (int a = -1; a <= 1; ++a)
#pragma unroll
                        for (int b = -1; b <= 1; ++b) cnt += sg[c + a * g.W() + b] == SSD_CELL_APPLE;
                    thr = vr.thr_harvest(cnt < 3 ? cnt : 3);
                }
                const uint32_t u = p.d_uapple ? p.d_uapple[(size_t)env * g.G() + c] : pick(r, q);
                if (u < thr) {
                    if (g.kind() == SSD_KIND_CLEANUP) { sg[c] = SSD_CELL_APPLE; ++n_new; }
                    else decided |= 1ull << (it * 4 + q);
                }
            }
        }
    }
    // waste: visit eligible waste points in ascending (order key, cell); the first success spawns one 'H'
    int wcell = -1;
    if (tW != 0) {
        uint32_t bk = 0xffffffffu, bc = 0xffffffffu;
        for (int j = lane; j < vr.n_waste2(); j += 32) {
            const ushort2 pts = __ldg(reinterpret_cast<const ushort2*>(m->waste_pts) + j);
            uint4 r = make_uint4(0, 0, 0, 0);
            if (!p.d_uwaste) r = philox4x32_10(gid, tick, 2u, (uint32_t)j, p.seed_lo, p.seed_hi);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const uint32_t c = q ? pts.y : pts.x;
                if (c == kNoPoint || (sg[c] & 0x7f) == SSD_CELL_WASTE) continue;   // cleanup.py:182
                const uint32_t u = p.d_uwaste ? p.d_uwaste[(size_t)env * g.G() + c] : (q ? r.z : r.x);
                const uint32_t key = p.d_uwaste ? p.d_wkey[(size_t)env * g.G() + c] : (q ? r.w : r.y);
                if (u < tW && (key < bk || (key == bk && c < bc))) { bk = key; bc = c; }
            }
        }
        const bool have = bc != 0xffffffffu;
        if (w.ballot(have)) {
            const uint32_t mk = w.rmin(have ? bk : 0xffffffffu);
            wcell = (int)w.rmin((have && bk == mk) ? bc : 0xffffffffu);
        }
    }
    w.sync();                                             // every decision read the pre-spawn grid
    if (g.kind() == SSD_KIND_HARVEST && decided) {
        int it = 0;
        for (int j = lane; j < vr.n_apple4(); j += 32, ++it) {
            const ushort4 pts = __ldg(reinterpret_cast<const ushort4*>(m->apple_pts) + j);
            const uint16_t c4[4] = { pts.x, pts.y, pts.z, pts.w };
#pragma unroll
            for (int q = 0; q < 4; ++q) if ((decided >> (it * 4 + q)) & 1ull) sg[c4[q]] = SSD_CELL_APPLE;
        }
    }
    if (wcell >= 0 && lane == 0) sg[wcell] = (uint8_t)(SSD_CELL_WASTE | (sg[wcell] & kOcc));
    w.sync();
    if (g.kind() == SSD_KIND_HARVEST) n_new = __popcll(decided);
    if (w.ballot(n_new != 0)) apples += w.radd(n_new);
    waste += wcell >= 0;
}

// ------------------------------------------------------------------ agent placement (map_env.py:771-793)
// The agents in `who` take, in index order, the free spawn point with the largest (key, cell); lanes are spawn points.  At reset
// every point is free; a respawn after tagging-out (RESPAWN) also skips the points in-play agents stand on (occupancy bits).
template <bool RESPAWN, class GEO, class VR>
__device__ __forceinline__ void place_agents(const Warp& w, const GEO& g, const KParams& p, const VR& vr, const uint8_t* sg, int lane,
                                             int env, uint32_t gid, uint32_t tick, unsigned who, int& pos) {
    const bool is_sp = lane < vr.n_spawn();
    const int mycell = is_sp ? (int)__ldg(&vr.map()->spawn_pts[lane]) : -1;
    bool taken = RESPAWN && is_sp && (sg[mycell] & kOcc);
    for (int i = 0; i < p.n; ++i) {
        if (!((who >> i) & 1u)) continue;
        uint32_t key = 0;
        if (p.random_spawn && is_sp)
            key = p.d_spawnkey ? p.d_spawnkey[((size_t)env * p.n + i) * g.G() + mycell]
                               : philox_word(p, gid, tick, 3u, (uint32_t)(i * vr.n_spawn() + lane));
        const bool cand = is_sp && !taken;
        const uint32_t mk = w.rmax(cand ? key : 0u);
        const unsigned eq = w.ballot(cand && key == mk);
        const int win = 31 - __clz(eq);
        const int cell = w.shfl(mycell, win);
        if (lane == win) taken = true;
        if (lane == i) pos = cell;
    }
}
// spawn_rotation (map_env.py:786-793)
__device__ __forceinline__ int spawn_orientation(const KParams& p, int env, uint32_t gid, uint32_t tick, int lane) {
    if (p.spawn_rot >= 0) return p.spawn_rot;
    return p.d_rot ? (int)(p.d_rot[(size_t)env * p.n + lane] & 3) : (int)(philox_word(p, gid, tick, 4u, (uint32_t)lane) >> 30);
}

// ------------------------------------------------------------------ render (map_env.py:360-379, 418-446, 795-815, 923-957)
__device__ __forceinline__ void st_row32(uint8_t* dst, const uint32_t* w) {     // one full 32-byte sector per lane
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(dst), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
}
__device__ __forceinline__ void st_row16(uint8_t* dst, const uint32_t* w) {
    asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" :: "l"(dst), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
}
__device__ __forceinline__ void st_row8(uint8_t* dst, uint32_t w0, uint32_t w1) {
    asm volatile("st.global.v2.b32 [%0], {%1,%2};" :: "l"(dst), "r"(w0), "r"(w1) : "memory");
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {   // raw PRMT: no selector masking
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// Row gather from NIBBLE-PACKED padded index maps.
// Two zero-padded copies of the map live in shared memory as 4-bit colour indices (8 cells per word):
//   M [padded row][col]   and   MT [padded col][row]
// so that for every orientation an output row of the rotated egocentric window (np.rot90 k=1,3,0,2 for
// LEFT, RIGHT, UP, DOWN; map_env.py:806-813) is ONE run of N nibbles:
//   UP    out[y][x] = M [r-V+y][c-V+x]  ascending       DOWN  out[y][x] = M [r+V-y][c+V-x]  descending
//   LEFT  out[y][x] = MT[c+V-y][r-V+x]  ascending       RIGHT out[y][x] = MT[c-V+y][r+V-x]  descending
// A lane owns one (agent, y) output row: it loads the <=5 words holding the run (nibble-reversing them for a
// descending run: one PRMT byte swap + one shift/merge), funnel-shifts them to pixel 0 (SHF), and every 16 bits
// of the result ARE the PRMT selector that looks 4 pixels up in the 8-entry colour LUT held in two registers
// per plane.  The finished row leaves the SM as one 32-byte (st.global.v8.b32 -> STG.E.ENL2.256) or 16-byte
// store per plane.  Indices: 0-5 cell codes, 6 outside, 7 agent.
// IDX (SSD_OBS_INDEX4): the funnel-shifted words ARE the packed output row (pixel x = nibble x, little-endian), so they are
// stored as they are, pad nibbles masked: one 16-byte store for N = 31, word stores otherwise; no PRMT.  In IDX kernels a
// full-colour agent is staged as its own index 7..15 (the row maps and the direct gather carry any index below 16).
__device__ __forceinline__ uint32_t nibble_reverse(uint32_t x) {
    const uint32_t y = prmt(x, 0u, 0x0123);
    return ((y << 4) & 0xf0f0f0f0u) | ((y >> 4) & 0x0f0f0f0fu);
}

template <int OCT_T>
struct RowUnit {                                              // one (agent, y) output row in flight
    uint32_t L[OCT_T > 0 ? OCT_T + 1 : 1];
    const uint32_t* w;
    uint8_t* dst;
    uint32_t sh, rev;
    uint32_t keep;                                            // 0 for the rows of an agent that is out of play: written as zeros
    bool valid;
};

template <int OCT_T, bool IDX, class GEO>
__device__ __forceinline__ void fetch_row(const Warp& w, const GEO& g, const KParams& p, const uint8_t* pmap, uint8_t* gobs, int lane, int it, int units,
                                          uint32_t abase_sh, int astep, unsigned outm, RowUnit<OCT_T>& U) {
    const int u = it * 32 + lane;
    U.valid = u < units;
    const int al = U.valid ? g.divN(u) : 0;
    U.keep = ((outm >> al) & 1u) ? 0u : 0xffffffffu;
    const int y = u - al * g.N();
    const uint32_t ab = w.shfl(abase_sh, al);
    const int as = w.shfl(astep, al);
    U.w = reinterpret_cast<const uint32_t*>(pmap + (ab & 0xffffu) + (U.valid ? y * as : 0));
    U.sh = (ab >> 16) & 31u;
    U.rev = (ab >> 24) & 1u;
    U.dst = IDX ? gobs + al * g.AS4() + y * g.RS4() : gobs + al * g.AS() + y * g.RP();
    {   // the <= OCT+1 words of the run, ascending or descending, must lie inside this warp's map tile
        const int nwords = (OCT_T > 0 ? OCT_T : ((g.RP() >> 2) + 1) >> 1) + 1;
        const long off = reinterpret_cast<const uint8_t*>(U.w) - pmap;
        SSD_CHECK(off >= (U.rev ? 4L * (nwords - 1) : 0L) && off + (U.rev ? 4L : 4L * nwords) <= g.PMS());
    }
    if constexpr (OCT_T > 0) {
        if (U.rev) {                                          // descending run: words walk down, nibbles are reversed
#pragma unroll
            for (int k = 0; k <= OCT_T; ++k) U.L[k] = nibble_reverse(*(U.w - k));
        } else {
#pragma unroll
            for (int k = 0; k <= OCT_T; ++k) U.L[k] = U.w[k]; // always in bounds: invalid lanes read agent 0's row 0
        }
    }
}

template <int OCT_T, bool IDX, class GEO>
__device__ __forceinline__ void emit_row(const GEO& g, const KParams& p, const RowUnit<OCT_T>& U, uint32_t lastmask) {
    if (!U.valid) return;
    const uint32_t sh = U.sh;
    if constexpr (IDX) {                                      // lastmask: valid nibbles of the row's last word
        if constexpr (OCT_T > 0) {
            uint32_t o[OCT_T];
#pragma unroll
            for (int k = 0; k < OCT_T; ++k) o[k] = __funnelshift_r(U.L[k], U.L[k + 1], sh) & U.keep;
            o[OCT_T - 1] &= lastmask;
            st_row16(U.dst, o);                               // OCT_T == 4: N = 29..31, 16 bytes a row
        } else {
            const int OCT = ((g.RP() >> 2) + 1) >> 1;         // == RS4 / 4 words of 8 pixels
            uint32_t prev = U.rev ? nibble_reverse(U.w[0]) : U.w[0];
            for (int k = 0; k < OCT; ++k) {
                const uint32_t cur = U.rev ? nibble_reverse(*(U.w - (k + 1))) : U.w[k + 1];
                const uint32_t m = k == OCT - 1 ? lastmask : 0xffffffffu;
                *reinterpret_cast<uint32_t*>(U.dst + 4 * k) = __funnelshift_r(prev, cur, sh) & m & U.keep;
                prev = cur;
            }
        }
    } else if constexpr (OCT_T > 0) {
        uint32_t v[2 * OCT_T];
#pragma unroll
        for (int k = 0; k < OCT_T; ++k) { v[2 * k] = __funnelshift_r(U.L[k], U.L[k + 1], sh); v[2 * k + 1] = v[2 * k] >> 16; }
#pragma unroll
        for (int pl = 0; pl < 3; ++pl) {                      // one colour plane at a time: 2*OCT PRMTs, then one wide store
            const uint32_t t0 = p.lut8[2 * pl] & U.keep, t1 = p.lut8[2 * pl + 1] & U.keep;
            uint32_t o[2 * OCT_T];
#pragma unroll
            for (int k = 0; k < 2 * OCT_T; ++k) o[k] = prmt(t0, t1, v[k]);
            o[2 * OCT_T - 1] &= lastmask;
            if (OCT_T == 4) st_row32(U.dst + pl * g.PS(), o);
            else st_row16(U.dst + pl * g.PS(), o);
        }
    } else {
        const int WR = g.RP() >> 2, OCT = (WR + 1) >> 1;
        uint32_t prev = U.rev ? nibble_reverse(U.w[0]) : U.w[0];
        for (int k = 0; k < OCT; ++k) {
            const uint32_t cur = U.rev ? nibble_reverse(*(U.w - (k + 1))) : U.w[k + 1];
            uint32_t v = __funnelshift_r(prev, cur, sh);
            prev = cur;
            for (int hlf = 0; hlf < 2; ++hlf, v >>= 16) {
                const int wd = 2 * k + hlf;
                if (wd >= WR) break;
                const uint32_t m = wd == WR - 1 ? lastmask : 0xffffffffu;
#pragma unroll
                for (int pl = 0; pl < 3; ++pl)
                    *reinterpret_cast<uint32_t*>(U.dst + pl * g.PS() + 4 * wd) = prmt(p.lut8[2 * pl], p.lut8[2 * pl + 1], v) & m & U.keep;
            }
        }
    }
}

template <int OCT_T, bool IDX, class GEO>
__device__ __forceinline__ void gather_rows(const Warp& w, const GEO& g, const KParams& p, const uint8_t* pmap, uint8_t* gobs, int lane,
                                            uint32_t abase_sh, int astep, unsigned outm) {
    const int WR = g.RP() >> 2;
    const uint32_t lastmask = IDX ? 0xffffffffu >> (4 * (8 * ((WR + 1) >> 1) - g.N())) : 0xffffffffu >> (8 * (4 * WR - g.N()));
    const int units = p.n * g.N(), iters = (units + 31) / 32;
    RowUnit<OCT_T> cur, nxt;
    fetch_row<OCT_T, IDX>(w, g, p, pmap, gobs, lane, 0, units, abase_sh, astep, outm, cur);
    for (int it = 0; it < iters; ++it) {                      // software pipeline: row it+1 is fetched while row it is emitted
        if (it + 1 < iters) fetch_row<OCT_T, IDX>(w, g, p, pmap, gobs, lane, it + 1, units, abase_sh, astep, outm, nxt);
        emit_row<OCT_T, IDX>(g, p, cur, lastmask);
        cur = nxt;
    }
}

// Nibble-packed padded maps, built one aligned 32-bit word (8 cells) at a time.  Map cells start at nibble
// LPn (V rounded up to 8) of a padded row, so only the last word of a row needs its tail set to "outside".
template <class GEO>
__device__ __forceinline__ void build_rowmap(const Warp& w, const GEO& g, const KParams& p, const uint8_t* sg, uint8_t* map, int lane) {
    const uint32_t* sgw = reinterpret_cast<const uint32_t*>(sg);
    const int total = g.H() * g.nw8M();
#pragma unroll 4
    for (int i = lane; i < total; i += 32) {
        const int r = g.divMW(i), j = i - r * g.nw8M();
        const int sb = r * g.W() + 8 * j, wi = sb >> 2;       // first source byte of this word (grid row r, col 8j)
        const uint32_t sel = 0x3210u + 0x1111u * (sb & 3);
        SSD_CHECK(wi >= 0 && 4 * (wi + 3) <= g.GS() + g.PMS());          // the last words may run into the (ignored) map tile
        const uint32_t a0 = sgw[wi], a1 = sgw[wi + 1], a2 = sgw[wi + 2];
        const uint32_t x0 = prmt(a0, a1, sel), x1 = prmt(a1, a2, sel);
        uint32_t w = prmt(x0 | (x0 >> 4), x1 | (x1 >> 4), 0x6420);            // 8 bytes -> 8 nibbles
        if (j == g.nw8M() - 1) w = (w & g.maskM8()) | (0x66666666u & ~g.maskM8());
        SSD_CHECK((r + g.V()) * g.pitchM() + (g.LPn() >> 1) + 4 * j + 4 <= (g.H() + 2 * g.V()) * g.pitchM());
        *reinterpret_cast<uint32_t*>(map + (r + g.V()) * g.pitchM() + (g.LPn() >> 1) + 4 * j) = w;
    }
}
// Transposed map from M: one lane transposes one 8 x 8 block of nibbles (8 words in, 8 words out) with three butterfly
// stages (swap 1-, 2-, 4-nibble sub-blocks across the diagonal).  Rows below the map come from M's first padding row and
// columns right of the map from M's tail nibbles, both "outside", which is exactly what MT's own padding holds.
template <class GEO>
__device__ __forceinline__ void build_colmap(const Warp& w, const GEO& g, const KParams& p, const uint8_t* M, uint8_t* MT, int lane) {
    const int total = g.nw8T() * g.nw8M();
    for (int blk = lane; blk < total; blk += 32) {
        const int i = g.divMW(blk), j = blk - i * g.nw8M();   // rows 8i.., columns 8j..
        uint32_t a[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int r = min(8 * i + k, g.H());              // H = first bottom padding row of M
            SSD_CHECK((r + g.V()) * g.pitchM() + (g.LPn() >> 1) + 4 * j + 4 <= (g.H() + 2 * g.V()) * g.pitchM());
            a[k] = *reinterpret_cast<const uint32_t*>(M + (r + g.V()) * g.pitchM() + (g.LPn() >> 1) + 4 * j);
        }
#pragma unroll
        for (int k = 0; k < 8; k += 2) {                      // 1-nibble sub-blocks
            const uint32_t t = ((a[k] >> 4) ^ a[k + 1]) & 0x0f0f0f0fu;
            a[k + 1] ^= t; a[k] ^= t << 4;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) if (!(k & 2)) {           // 2-nibble sub-blocks
            const uint32_t t = ((a[k] >> 8) ^ a[k + 2]) & 0x00ff00ffu;
            a[k + 2] ^= t; a[k] ^= t << 8;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {                         // 4-nibble sub-blocks
            const uint32_t t = ((a[k] >> 16) ^ a[k + 4]) & 0x0000ffffu;
            a[k + 4] ^= t; a[k] ^= t << 16;
        }
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            const int c = 8 * j + x;
            if (c < g.W()) {
                SSD_CHECK((c + g.V()) * g.pitchT() + (g.LPn() >> 1) + 4 * i + 4 <= (g.W() + 2 * g.V()) * g.pitchT());
                *reinterpret_cast<uint32_t*>(MT + (c + g.V()) * g.pitchT() + (g.LPn() >> 1) + 4 * i) = a[x];
            }
        }
    }
}

// "outside the map" everywhere (utility_funcs.py:58-116 without np.pad); issued while the state loads are in flight
template <class GEO>
__device__ __forceinline__ void fill_outside(const Warp& w, const GEO& g, const KParams& p, uint8_t* pmap, int lane) {
    const uint4 v6 = make_uint4(0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u);
    uint4* q = reinterpret_cast<uint4*>(pmap);
    const int n16 = g.PMS() >> 4;
#pragma unroll 8
    for (int i = lane; i < n16; i += 32) q[i] = v6;           // trip count is a compile-time constant for the shipped maps
}

// Direct gather for small views (N <= 16, i.e. every Cleanup configuration): a lane owns one (agent, y) output row and
// reads its N cells straight from the staged byte grid -- one unaligned 16-byte run for UP / DOWN (5 aligned words + funnel
// shifts), N byte loads down a column for LEFT / RIGHT -- packs them to nibbles, replaces the cells outside the map by
// index 6, reverses the run for DOWN / RIGHT, and colours 4 pixels per PRMT as the map path does.  No padded maps are built.
// The grid tile has V rows of slack on both sides (zeroed at kernel start), so no load needs a bounds test; agents were
// written into the staged grid as index 7 by the caller.
template <bool COLS, bool IDX, class GEO>
__device__ __forceinline__ void gather_class(const Warp& w, const GEO& g, const KParams& p, const uint8_t* sg, const uint8_t* rank2lane,
                                             uint8_t* gobs, int lane, uint32_t apack, int n_in_class, unsigned outm) {
    const int N = g.N(), V = g.V(), W = g.W(), units = n_in_class * N, WR = g.RP() >> 2;
    const uint32_t lastmask = 0xffffffffu >> (8 * (4 * WR - N));
    for (int u0 = 0; u0 < units; u0 += 32) {
        const int u = u0 + lane;
        const bool valid = u < units;
        const int rank = valid ? g.divN(u) : 0;
        const int y = u - rank * N;
        const int al = rank2lane[rank];
        const uint32_t ap = w.shfl(apack, al);
        if (!valid) continue;
        const int ar = (int)(ap & 0xffu), ac = (int)((ap >> 8) & 0xffu), o = (int)(ap >> 16);
        uint32_t b0, b1, b2, b3;                              // element i of the run (ascending map coordinate) in byte i
        int lo, hi;                                           // elements inside the map: [lo, hi)
        if (!COLS) {                                          // UP / DOWN: a run along map row R
            const int R = o == 2 ? ar - V + y : ar + V - y;
            const bool rv = (unsigned)R < (unsigned)g.H();
            lo = rv ? max(0, V - ac) : 0;
            hi = rv ? min(N, W + V - ac) : 0;
            const int start = (rv ? R : 0) * W + ac - V;      // >= -V: inside the front slack
            SSD_CHECK(start >= -g.padF() + 32 && start + 20 <= g.GS() + g.padB());
            const uint32_t* wp = reinterpret_cast<const uint32_t*>(sg + (start & ~3));
            const uint32_t sh = (uint32_t)(start & 3) * 8u;
            const uint32_t a0 = wp[0], a1 = wp[1], a2 = wp[2], a3 = wp[3], a4 = wp[4];
            b0 = __funnelshift_r(a0, a1, sh); b1 = __funnelshift_r(a1, a2, sh);
            b2 = __funnelshift_r(a2, a3, sh); b3 = __funnelshift_r(a3, a4, sh);
        } else {                                              // LEFT / RIGHT: a run down map column C
            const int C = o == 0 ? ac + V - y : ac - V + y;
            const bool cv = (unsigned)C < (unsigned)W;
            lo = cv ? max(0, V - ar) : 0;
            hi = cv ? min(N, g.H() + V - ar) : 0;
            const uint8_t* col = sg + (ar - V) * W + (cv ? C : 0);     // rows ar-V .. ar+V: at most V rows into either slack
            SSD_CHECK((ar - V) * W >= -g.padF() + 32 && (ar + V) * W + W <= g.GS() + g.padB());
            uint32_t e[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) e[i] = i < N ? (uint32_t)col[i * W] : 0u;
            b0 = e[0] | (e[1] << 8) | (e[2] << 16) | (e[3] << 24);
            b1 = e[4] | (e[5] << 8) | (e[6] << 16) | (e[7] << 24);
            b2 = e[8] | (e[9] << 8) | (e[10] << 16) | (e[11] << 24);
            b3 = e[12] | (e[13] << 8) | (e[14] << 16) | (e[15] << 24);
        }
        // bytes -> nibbles (every byte is a colour index < 8), cells outside the map -> 6
        uint32_t n0 = prmt(b0 | (b0 >> 4), b1 | (b1 >> 4), 0x6420);
        uint32_t n1 = prmt(b2 | (b2 >> 4), b3 | (b3 >> 4), 0x6420);
        const unsigned long long vm = (hi >= 16 ? ~0ull : ((1ull << (4 * hi)) - 1ull)) & ~((1ull << (4 * lo)) - 1ull);
        const uint32_t m0 = (uint32_t)vm, m1 = (uint32_t)(vm >> 32);
        n0 = (n0 & m0) | (0x66666666u & ~m0);
        n1 = (n1 & m1) | (0x66666666u & ~m1);
        if (o & 1) {                                          // RIGHT / DOWN: out[x] = element N-1-x (np.rot90 k=3 / k=2)
            const uint32_t r1 = nibble_reverse(n0), r0w = nibble_reverse(n1);       // nibble j of (r1:r0w) = element 15-j
            const unsigned long long rr = (((unsigned long long)r1 << 32) | r0w) >> (4 * (16 - N));   // up to 60 bits for tiny views
            n0 = (uint32_t)rr;
            n1 = (uint32_t)(rr >> 32);
        }
        if constexpr (IDX) {                                  // (n0, n1) is the packed row: keep its N nibbles
            const uint32_t keep = ((outm >> al) & 1u) ? 0u : 0xffffffffu;
            uint8_t* dst = gobs + al * g.AS4() + y * g.RS4();
            if (g.RS4() == 8) st_row8(dst, n0 & keep, n1 & (0xffffffffu >> (4 * (16 - N))) & keep);
            else *reinterpret_cast<uint32_t*>(dst) = n0 & (0xffffffffu >> (4 * (8 - N))) & keep;
            continue;
        }
        const uint32_t v[4] = { n0, n0 >> 16, n1, n1 >> 16 };
        uint8_t* dst = gobs + al * g.AS() + y * g.RP();
        const uint32_t keep = ((outm >> al) & 1u) ? 0u : 0xffffffffu;       // an agent out of play sees zeros
#pragma unroll
        for (int pl = 0; pl < 3; ++pl) {
            const uint32_t t0 = p.lut8[2 * pl] & keep, t1 = p.lut8[2 * pl + 1] & keep;
            uint32_t o4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) o4[k] = prmt(t0, t1, v[k]);
            if (WR == 4) { o4[3] &= lastmask; st_row16(dst + pl * g.PS(), o4); }
            else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (k < WR) *reinterpret_cast<uint32_t*>(dst + pl * g.PS() + 4 * k) = k == WR - 1 ? (o4[k] & lastmask) : o4[k];
            }
        }
    }
}

// The rows of UP / DOWN agents and of LEFT / RIGHT agents are gathered in two separate passes, so that a trip of the warp runs
// ONE of the two load schemes instead of both under divergence.  `tbl` (32 bytes at the very start of the tile's front slack,
// never touched by a gather load) maps (class, rank within class) -> agent lane.
template <bool IDX, class GEO>
__device__ __forceinline__ void gather_direct(const Warp& w, const GEO& g, const KParams& p, const uint8_t* sg, uint8_t* tbl, uint8_t* gobs, int lane,
                                              bool is_agent, int r0, int c0, int ori, unsigned outm) {
    const uint32_t apack = (uint32_t)r0 | ((uint32_t)c0 << 8) | ((uint32_t)ori << 16);
    const unsigned m_rows = w.ballot(is_agent && ori >= 2), m_cols = w.ballot(is_agent && ori < 2);
    if (is_agent) {
        const bool cols = ori < 2;
        tbl[(cols ? 16 : 0) + __popc((cols ? m_cols : m_rows) & ((1u << lane) - 1u))] = (uint8_t)lane;
    }
    w.sync();
    if (m_rows) gather_class<false, IDX>(w, g, p, sg, tbl, gobs, lane, apack, __popc(m_rows), outm);
    if (m_cols) gather_class<true, IDX>(w, g, p, sg, tbl + 16, gobs, lane, apack, __popc(m_cols), outm);
}

// live: the lane's agent is on the map; outm: agents out of play (tagged out), whose views are written as zeros.  Their rows go
// through the same gather at cell (0, 0), masked, so that a warp trip never mixes two kinds of row.
template <bool IDX, class GEO>
__device__ __forceinline__ void render(const Warp& w, const GEO& g, const KParams& p, const uint8_t* sg, uint8_t* pmap, const uint32_t* lut_s,
                                       int lane, bool is_agent, bool live, int pos, int ori, int env, unsigned same, unsigned outm,
                                       bool end) {
    // end (MODE_STEP_RESET): into the episode-end buffers instead of the step outputs.  Each pointer is read from the launch
    // parameters where it is used, as before: a pointer held in registers across the state block costs the fused kernels spills.
    uint8_t* const state = end ? p.end_state : p.state_rgb;
    const bool top = live && lane == 31 - __clz(same);       // later index overwrites (map_env.py:370); same = lanes on this lane's cell
    if (state) {
        if (p.state_idx4) {                                   // get_state as packed colour indices (DESIGN.md §3 item 13)
            // One lane assembles one 32-bit word, 8 cells of a row, as build_rowmap does, and stores it.  A row is nw8M
            // words (ceil(W/2) rounded up to 4 bytes); the nibbles past W and the words past the last row are 0.
            // RGB-observation kernels staged every agent as 7, so in the full-colour scheme the top agent's own colour index
            // is staged for the pack and 7 restored before the observation gather.  (r0, c0 are computed after this block:
            // live across the pack loop they cost the render kernels registers.)
            uint8_t* sgm = const_cast<uint8_t*>(sg);
            const bool repaint = !IDX && !p.agents_uniform;
            if (repaint) { if (top) sgm[pos] = (uint8_t)agent_colour_index(lane); w.sync(); }
            const int words = cround_up(g.H() * g.nw8M(), 4);
            uint32_t* out = reinterpret_cast<uint32_t*>(state) + (size_t)env * words;
            const uint32_t* sgw = reinterpret_cast<const uint32_t*>(sg);
#pragma unroll 1                                              // 1-5 trips on the shipped maps
            for (int i = lane; i < words; i += 32) {
                const int r = g.divMW(i), j = i - r * g.nw8M();
                uint32_t v = 0u;
                if (r < g.H()) {
                    const int sb = r * g.W() + 8 * j, wi = sb >> 2;   // first cell of this word (row r, column 8j)
                    const uint32_t sel = 0x3210u + 0x1111u * (sb & 3);
                    SSD_CHECK(wi >= 0 && 4 * (wi + 3) <= g.GS() + g.padB());   // the last words may read into the back slack
                    const uint32_t a0 = sgw[wi], a1 = sgw[wi + 1], a2 = sgw[wi + 2];
                    const uint32_t x0 = prmt(a0, a1, sel), x1 = prmt(a1, a2, sel);
                    v = prmt(x0 | (x0 >> 4), x1 | (x1 >> 4), 0x6420);          // 8 bytes -> 8 nibbles
                    if (j == g.nw8M() - 1) v &= g.maskM8();
                }
                out[i] = v;
            }
            if (repaint) { w.sync(); if (top) sgm[pos] = 7; w.sync(); }
        } else {                                              // get_state: unrotated full map (map_env.py:950-957)
            uint8_t* out = state + (size_t)env * 3 * g.G();
            for (int c = lane; c < g.G(); c += 32) {
                const uint32_t rgb = lut_s[sg[c]];
                out[c] = (uint8_t)rgb; out[g.G() + c] = (uint8_t)(rgb >> 8); out[2 * g.G() + c] = (uint8_t)(rgb >> 16);
            }
            w.sync();                                         // orders the agent overlay after the cell colours
            if (top) {
                const uint32_t rgb = lut_s[agent_colour_index(lane)];
                out[pos] = (uint8_t)rgb; out[g.G() + pos] = (uint8_t)(rgb >> 8); out[2 * g.G() + pos] = (uint8_t)(rgb >> 16);
            }
        }
    }
    uint8_t* const obs = end ? p.end_obs : p.obs;
    if (!obs) return;
    int r0 = 0, c0 = 0;
    if (live) { r0 = g.divW(pos); c0 = pos - r0 * g.W(); }
    uint8_t* gobs = obs + (size_t)env * (p.n * (IDX ? g.AS4() : g.AS()));

    if (g.direct()) {
        gather_direct<IDX>(w, g, p, sg, const_cast<uint8_t*>(sg) - g.padF(), gobs, lane, is_agent, r0, c0, ori, outm);
    } else {
        // the maps were pre-filled with "outside the map" at kernel start (fill_outside); now the cells (agents are already in
        // the staged grid as index 7)
        // per agent: which map, first word of its window row 0, row step, funnel shift, direction   (o: 0 LEFT 1 RIGHT 2 UP 3 DOWN)
        const bool colmap = ori < 2, rev = (ori == 1) || (ori == 3);
        const int rowc = colmap ? c0 : r0;                        // coordinate that selects the map row
        const int runc = colmap ? r0 : c0;                        // coordinate along the run
        const int pitch = colmap ? g.pitchT() : g.pitchM();
        const bool down = (ori == 0) || (ori == 3);               // window row y walks towards smaller map rows
        const int s = g.LPn() + runc + (rev ? g.V() : -g.V());    // first pixel of the run (highest nibble when descending)
        const uint32_t abase_sh = (uint32_t)(g.off_map(ori) + (rowc + (down ? 2 * g.V() : 0)) * pitch + ((s >> 3) << 2))
                                  | ((uint32_t)((rev ? 7 - (s & 7) : (s & 7)) * 4) << 16) | ((uint32_t)rev << 24);
        const int astep = down ? -pitch : pitch;
        const bool needT = w.ballot(live && ori < 2) != 0;
        uint8_t* MT = pmap + g.off_map(0);
        uint8_t* M = pmap + g.off_map(2);
        build_rowmap(w, g, p, sg, M, lane);
        w.sync();
        if (needT) {                                              // LEFT / RIGHT views read the transpose (agents included)
            build_colmap(w, g, p, M, MT, lane);
            w.sync();
        }
        if (g.RP() == 32) gather_rows<4, IDX>(w, g, p, pmap, gobs, lane, abase_sh, astep, outm);
        else gather_rows<0, IDX>(w, g, p, pmap, gobs, lane, abase_sh, astep, outm);
    }
    if constexpr (IDX) {                                          // pad bytes per agent block (8 for N = 15)
        const int body = g.N() * g.RS4(), tail = g.AS4() - body;
        if (tail) for (int i = lane; i < p.n * (tail >> 2); i += 32)
            *reinterpret_cast<uint32_t*>(gobs + (i / (tail >> 2)) * g.AS4() + body + 4 * (i % (tail >> 2))) = 0u;
    } else {
        const int tail = g.AS() - 3 * g.PS();                     // pad bytes per agent block (0 for the shipped views)
        if (tail) for (int i = lane; i < p.n * (tail >> 2); i += 32)
            *reinterpret_cast<uint32_t*>(gobs + (i / (tail >> 2)) * g.AS() + 3 * g.PS() + 4 * (i % (tail >> 2))) = 0u;
    }
    if (!IDX && !p.agents_uniform) {
        // full-colour scheme: every visible agent is re-painted with its own colour (after the row stores)
        w.sync();
        const uint32_t apack = (uint32_t)r0 | ((uint32_t)c0 << 10) | ((uint32_t)ori << 20);
        const int pairs = p.n * p.n, iters = (pairs + 31) / 32;
        for (int it = 0; it < iters; ++it) {
            const int q = it * 32 + lane;
            const bool valid = q < pairs;
            const int al = valid ? q / p.n : 0, j = valid ? q - al * p.n : 0;
            const uint32_t api = w.shfl(apack, al), apj = w.shfl(apack, j);
            const bool topj = w.shfl((int)top, j);
            if (!valid || !topj || ((outm >> al) & 1u)) continue;
            const int a = (int)(apj & 1023) - (int)(api & 1023) + g.V(), b = (int)((apj >> 10) & 1023) - (int)((api >> 10) & 1023) + g.V();
            if (a < 0 || a >= g.N() || b < 0 || b >= g.N()) continue;
            const int o = api >> 20;
            int y, x;
            if (o == 2) { y = a; x = b; } else if (o == 0) { x = a; y = g.N() - 1 - b; }
            else if (o == 3) { y = g.N() - 1 - a; x = g.N() - 1 - b; } else { x = g.N() - 1 - a; y = b; }
            const uint32_t rgb = lut_s[agent_colour_index(j)];
            uint8_t* d = gobs + al * g.AS() + y * g.RP() + x;
            d[0] = (uint8_t)rgb; d[g.PS()] = (uint8_t)(rgb >> 8); d[2 * g.PS()] = (uint8_t)(rgb >> 16);
        }
    }
}

// ------------------------------------------------------------------ the kernel's stages
// setup_agents (map_env.py:771-784) and custom_map_update (313) on the base grid staged in sg: MODE_RESET's body.  The reset
// env's t, tick and counts are stored; its agents are all in play.
template <class GEO, class VR>
__device__ __forceinline__ void reset_env(const Warp& w, const GEO& g, const KParams& p, const VR& vr, uint8_t* sg, int lane, bool is_agent,
                                          int env, uint32_t gid, uint32_t tick, int& pos, int& ori, int& apples, int& waste) {
    place_agents<false>(w, g, p, vr, sg, lane, env, gid, tick, ~0u, pos);
    if (is_agent) ori = spawn_orientation(p, env, gid, tick, lane);
    if (is_agent) sg[pos] |= kOcc;                         // distinct spawn points: no two lanes share a cell
    w.sync();
    apples = vr.base_apples(); waste = vr.base_waste();
    spawn(w, g, p, vr, sg, lane, env, gid, tick, apples, waste);
    if (lane == 0) { p.t[env] = 0; p.tick[env] = tick + 1; p.counts[env] = (uint32_t)apples | ((uint32_t)waste << 16); }
}

// The write-back of a reset env (every agent in play on a cell of its own, no timer, ep_ret 0).  The step's write-back in
// ssd_kernel stays written out there: calling a shared function from it moves the register allocation of the Harvest V=15
// tagging step kernels.
template <class GEO>
__device__ __forceinline__ void write_back_reset(const Warp& w, const GEO& g, const KParams& p, uint8_t* sg, int lane, bool is_agent,
                                                 int env, int pos, int ori) {
    if (is_agent) sg[pos] &= 0x7f;
    w.sync();
    uint4* dst = reinterpret_cast<uint4*>(p.grid + (size_t)env * g.GS());
    warp_for(g.GS() >> 4, lane, [&](int i) { dst[i] = reinterpret_cast<const uint4*>(sg)[i]; });
    if (is_agent) {
        const int r = g.divW(pos);
        p.agent[(size_t)env * p.NA + lane] = (uint32_t)r | ((uint32_t)(pos - r * g.W()) << 8) | ((uint32_t)ori << 16);
        p.ep_ret[(size_t)env * p.NA + lane] = 0;
    }
}

// The agent overlay, then render (`end`: into the episode-end buffers).
template <bool TAG, bool IDX, class GEO>
__device__ __forceinline__ void draw(const Warp& w, const GEO& g, const KParams& p, uint8_t* sg, uint8_t* pmap, const uint32_t* lut_s, int lane,
                                     bool is_agent, bool live, int pos, int ori, int env, unsigned same, bool end) {
    // agent overlay: every occupied cell shows an agent (index 7; which agent only matters for the full-colour repaint and
    // the state image, both handled in render).  Same value from every lane on a shared cell: no race.
    // IDX: the top agent of a cell is staged as its own colour index (7 in the simplified scheme), so no repaint follows.
    w.sync();                                          // the write-back has read the staged grid
    if (IDX) { if (live && lane == 31 - __clz(same)) sg[pos] = (uint8_t)(p.agents_uniform ? 7 : agent_colour_index(lane)); }
    else if (live) sg[pos] = 7;
    w.sync();
    const unsigned outm = TAG ? w.ballot(is_agent && !live) : 0u;
    render<IDX>(w, g, p, sg, pmap, lut_s, lane, is_agent, live, pos, ori, env, same, outm, end);
}

// ------------------------------------------------------------------ the kernel
// TAG: tagging-out timers are on (p.tag_timeout > 0, or with variants any variant's; every mode but MODE_RESET, DESIGN.md §3 item 11).
// IDX: observations are written as packed colour indices (SSD_OBS_INDEX4, DESIGN.md §3 item 12) instead of RGB planes.
// MODE_STEP_RESET: MODE_STEP, then an env whose episode the step ended renders the finished step into the episode-end
// buffers, runs MODE_RESET's body keyed by the post-step tick and renders its first observation (DESIGN.md §3 item 14).  A mode
// of its own, not a runtime flag, so that the other instantiations keep their code.  Its two render call sites inline two copies
// of the render: a two-pass loop around one call site spilled in the Harvest V=15 and runtime-geometry kernels
// (profiles/r7_notes.md).
// VAR: envs run the variants of p.variant_of (DESIGN.md §3 item 15).  A template parameter, not a runtime switch on variant_of,
// because the switch moved the register allocation of most kernels without variants and spilled one (profiles/r8_notes.md).
// STATS (MODE_STEP, MODE_STEP_RESET): the step adds its events to the per-agent episode counters p.stats (DESIGN.md §3 item 16).
// A template parameter for the same reason as VAR: the kernels without counters keep their code.
template <int MODE, class GEO, bool TAG, bool IDX, bool VAR, bool STATS>
__global__ void __launch_bounds__(kWarps * 32, kMinBlocks) ssd_kernel(const __grid_constant__ KParams p) {
    constexpr bool STEP = MODE == MODE_STEP || MODE == MODE_STEP_RESET;
    const GEO g(p);
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ ColourLuts lut_all;                            // colour LUT, one private copy per warp: no CTA barrier anywhere
    const int warp = threadIdx.x >> 5;
    const Warp w(threadIdx.x & 31);
    const int lane = w.lane;
    uint32_t* lut_s = lut_all[warp];
    // per-env tile: [front slack][grid GS][back slack][nibble maps (map path only)]
    uint8_t* tile = smem + (size_t)warp * (g.padF() + g.GS() + g.padB() + g.PMS());
    uint8_t* sg = tile + g.padF();
    uint8_t* pmap = sg + g.GS() + g.padB();
    const bool is_agent = lane < p.n;
    // One env instance per warp and per launch.  (A persistent loop over env instances was measured and dropped: warps that
    // start together stay phase-locked -- everybody resolves moves, then everybody stores observations -- which turns a
    // 65536-env launch into 14 back-to-back single-wave steps: Harvest 204 us instead of 167 us.  Letting the block scheduler
    // start a fresh CTA whenever one retires decorrelates the phases; profiles/r2_notes.md.)  Two envs per warp (16 lanes each)
    // was measured slower on every workload but the largest Cleanup launch (profiles/r1_notes.md, profiles/r2_notes.md §2).
    const int env = p.env0 + blockIdx.x * kWarps + warp;
    if (env >= p.env1) return;
    // Prologue that touches nothing an earlier launch writes (colour LUT, slack / "outside" fill of the staging tile).  Under
    // programmatic dependent launch (small launches, p.pdl) it runs first, while the previous launch of the stream is still
    // storing observations, and the state loads follow the grid dependency; otherwise it runs under the state loads.
    auto prologue = [&]() {
        if (lane < 16) lut_s[lane] = p.lut[lane];             // (made visible by w.sync below)
        if (p.obs || (MODE == MODE_STEP_RESET && p.end_obs)) {
            if (g.direct()) {                                 // zero the slack around the grid (read, then masked, by the gather)
                for (int i = lane; i < (g.padF() >> 4); i += 32) reinterpret_cast<uint4*>(tile)[i] = make_uint4(0, 0, 0, 0);
                for (int i = lane; i < (g.padB() >> 4); i += 32) reinterpret_cast<uint4*>(sg + g.GS())[i] = make_uint4(0, 0, 0, 0);
            } else fill_outside(w, g, p, pmap, lane);         // "outside the map"
        }
    };
    if (p.pdl) {
        prologue();
        asm volatile("griddepcontrol.wait;" ::: "memory");    // the previous launch of the stream has completed, its writes are visible
    }
    {
        if (MODE == MODE_RESET && p.mask && __ldcg(p.mask + env) == 0) return;
        const uint32_t gid = p.gid_base + (uint32_t)env;
        int vid = 0;                                          // the env's variant: ids past the table run the last variant
        if (VAR) {
            vid = __ldcg(p.variant_of + env);
            SSD_CHECK(vid < p.n_variants);
            vid = min(vid, p.n_variants - 1);
        }
        const Var<VAR> vr{p, vid};
        // every global load of the step is issued up front.  Mutable state is read past L1 (ld.global.cg): each entry is read once
        // per step anyway, and a launch that became resident before its predecessors finished (programmatic dependent launch,
        // concurrent env ranges sharing a cache line at a range boundary) must never see a line an earlier CTA left in this SM's L1.
        const uint32_t tick = __ldcg(p.tick + env);
        const int t_prev = STEP ? __ldcg(p.t + env) : 0;
        const uint32_t cnt = STEP ? __ldcg(p.counts + env) : 0u;
        int act = (STEP && is_agent) ? (int)__ldcg(p.actions + (size_t)env * p.n + lane) : 255;
        int pos = -1 - lane, ori = 0, ep_ret = 0;
        uint32_t a_rec = 0;
        if (MODE != MODE_RESET && is_agent) {
            a_rec = __ldcg(p.agent + (size_t)env * p.NA + lane);
            ep_ret = __ldcg(p.ep_ret + (size_t)env * p.NA + lane);
        }
        const int n16 = g.GS() >> 4;
        {
            const uint4* src = MODE == MODE_RESET ? reinterpret_cast<const uint4*>(vr.map()->base_grid)
                                                  : reinterpret_cast<const uint4*>(p.grid + (size_t)env * g.GS());
            uint4 g0 = make_uint4(0, 0, 0, 0);
            if (lane < n16) g0 = __ldcg(src + lane);
            if (!p.pdl) prologue();                           // while the state loads are in flight
            if (lane < n16) reinterpret_cast<uint4*>(sg)[lane] = g0;
            for (int i = lane + 32; i < n16; i += 32) reinterpret_cast<uint4*>(sg)[i] = __ldcg(src + i);
        }
        // Tagging-out (TAG): an agent whose timer (bits 24..31 of its record) is non-zero is out of play for the whole step.  Its
        // lane then acts like a lane without an agent (unique negative pos, no action), and `home` keeps the cell of its record.
        bool live = is_agent;
        int timer = 0, home = 0;
        if (MODE != MODE_RESET && is_agent) {
            pos = (int)(a_rec & 0xff) * g.W() + (int)((a_rec >> 8) & 0xff);
            ori = (int)((a_rec >> 16) & 3);
            if (TAG) {
                timer = (int)(a_rec >> 24);
                home = pos;
                if (timer) { live = false; pos = -1 - lane; act = 255; }
            }
        }
        w.sync();

        int apples = (int)(cnt & 0xffffu), waste = (int)(cnt >> 16);
        // lanes standing on this lane's cell: MATCH.ANY is slow (3-4 % of the step each in the profile), positions do not change
        // after update_moves, so it is evaluated once and shared by consume, the occupancy strip and the render
        unsigned same = 1u << lane;                            // reset: distinct spawn points
        if (MODE == MODE_RENDER) same = equal_lanes(w, pos, p.n);
        bool ended = false;                                        // MODE_STEP_RESET: this step ended the episode
        if (STEP) {
            int reward = 0, clean_num = 0;
            bool tagged = false;
            uint32_t sd = 0;                                       // STATS: the step's counter deltas (kSd* bits)
            update_moves(w, g, p, sg, lane, live, act, pos, ori, env, gid, tick);                     // map_env.py:251
            // consume in index order: the lowest index on a cell eats the apple (253-256); mark occupancy
            same = surely_distinct(w, pos, live, w.ballot(live)) ? (1u << lane) : equal_lanes(w, pos, p.n);
            const int here = live ? sg[pos] : 0;
            const bool first = live && lane == __ffs(same) - 1;
            const unsigned ate = w.ballot(first && here == SSD_CELL_APPLE);
            w.sync();
            if (first) {
                if (here == SSD_CELL_APPLE) { reward += 1; sg[pos] = kOcc | SSD_CELL_EMPTY; }
                else sg[pos] = (uint8_t)(kOcc | here);
            }
            apples -= __popc(ate);
            if (STATS && ((ate >> lane) & 1u)) sd = kSdAte;
            w.sync();
            beams<TAG>(w, g, p, vr, sg, lane, live, act, pos, ori, reward, clean_num, waste, tagged);    // 259-260
            if (STATS) sd |= fire_counts(w, g, p, sg, lane, live, act, pos, ori);
            if (STATS && is_agent) {
                // Every count of the step is known here (t, whether the step ends the episode, the stage-in timer), so the
                // counters are updated before spawn and nothing of them is live across spawn or the render: the non-zero deltas
                // are added in L2 (RED.ADD, no register waits for a load).  Loading the seven counters and storing them with the
                // agent records spilled in the Harvest V=15 and runtime-geometry auto-reset kernels.  An episode that ends in a
                // MODE_STEP_RESET step loads its counters (past L1, after griddepcontrol.wait), writes them to end_stats if set
                // and stores zeros: the reset that follows starts from 0.
                const uint32_t t = (uint32_t)t_prev + 1u;
                if (TAG && timer != 0) sd |= kSdOut;
                const uint32_t d[SSD_N_STATS] = { sd & 1u, (sd & 1u) ? t : 0u, (sd >> 1) & 1u, (sd >> kSdDealt) & 3u,
                                                  (sd >> kSdTaken) & 63u, (sd >> 2) & 1u, (uint32_t)clean_num };
                uint32_t* const s = p.stats + (size_t)env * SSD_N_STATS * p.NA + lane;
                if (MODE == MODE_STEP_RESET && (int)t >= p.episode_limit) {
                    uint32_t v[SSD_N_STATS];
#pragma unroll
                    for (int f = 0; f < SSD_N_STATS; ++f) v[f] = __ldcg(s + f * p.NA) + d[f];
                    uint32_t* const e = p.end_stats + (size_t)env * SSD_N_STATS * p.NA + lane;
#pragma unroll
                    for (int f = 0; f < SSD_N_STATS; ++f) {
                        if (p.end_stats) e[f * p.NA] = v[f];
                        s[f * p.NA] = 0u;
                    }
                } else {
#pragma unroll
                    for (int f = 0; f < SSD_N_STATS; ++f) if (d[f]) atomicAdd(s + f * p.NA, d[f]);
                }
            }
            unsigned gone = 0;
            if (TAG) {                                 // the tagged leave the map; a cell stays occupied while an untagged agent is on it
                gone = w.ballot(tagged);
                if (gone) {
                    if (live && lane == __ffs(same) - 1 && (same & ~gone) == 0) sg[pos] &= 0x7f;
                    w.sync();
                    if (tagged) { home = pos; pos = -1 - lane; live = false; }
                }
            }
            spawn(w, g, p, vr, sg, lane, env, gid, tick, apples, waste);                              // 263, 291-292
            if (TAG) {                                 // the agents out during this step count down; those reaching 0 return
                const bool back = timer == 1;
                timer = tagged ? vr.tag_timeout() : (timer ? timer - 1 : 0);
                const unsigned who = w.ballot(back);
                if (who) {
                    place_agents<true>(w, g, p, vr, sg, lane, env, gid, tick, who, pos);
                    if (back) { ori = spawn_orientation(p, env, gid, tick, lane); live = true; sg[pos] |= kOcc; }
                    w.sync();
                }
                if (gone | who) same = equal_lanes(w, pos, p.n);
            }
            const int t = t_prev + 1;
            if (is_agent) {
                p.reward[(size_t)env * p.n + lane] = (int8_t)reward;
                p.clean[(size_t)env * p.n + lane] = (uint8_t)clean_num;
                ep_ret += reward;                                                               // 885-888
            }
            if (lane == 0) {
                p.apple_cnt[env] = (uint16_t)apples;
                p.done[env] = t >= p.episode_limit;                                             // 890-894
                p.t[env] = t;
                p.tick[env] = tick + 1;
                p.counts[env] = (uint32_t)apples | ((uint32_t)waste << 16);
            }
            if (MODE == MODE_STEP_RESET) ended = t >= p.episode_limit;
        } else if (MODE == MODE_RESET) {
            reset_env(w, g, p, vr, sg, lane, is_agent, env, gid, tick, pos, ori, apples, waste);
            ep_ret = 0;
        }

        // the next launch of this stream may become resident now (its prologue overlaps this launch's stores; it still waits
        // for this whole grid before it reads any state)
        if (p.pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (MODE != MODE_RENDER) {                                 // strip the occupancy bits, write the state back
            if (live && lane == __ffs(same) - 1) sg[pos] &= 0x7f;
            w.sync();
            uint4* dst = reinterpret_cast<uint4*>(p.grid + (size_t)env * g.GS());
            warp_for(g.GS() >> 4, lane, [&](int i) { dst[i] = reinterpret_cast<const uint4*>(sg)[i]; });
            if (is_agent) {                                        // an agent out of play keeps the cell it left the map from
                const int cell = (TAG && !live) ? home : pos;
                const int r = g.divW(cell);
                p.agent[(size_t)env * p.NA + lane] = (uint32_t)r | ((uint32_t)(cell - r * g.W()) << 8) | ((uint32_t)ori << 16)
                                                     | (TAG ? (uint32_t)timer << 24 : 0u);
                p.ep_ret[(size_t)env * p.NA + lane] = ep_ret;
            }
        }
        if constexpr (MODE == MODE_STEP_RESET) {
            // An env whose episode ended renders the finished step into the episode-end buffers and is reset (MODE_RESET's body on
            // the base grid staged again, the draws keyed by the post-step tick, as a masked ssd_reset after this step would key
            // them); every env then renders into the step outputs below.
            if (ended) {
                if (is_agent && p.end_ep_ret) p.end_ep_ret[(size_t)env * p.NA + lane] = ep_ret;
                if (p.end_obs || p.end_state) draw<TAG, IDX>(w, g, p, sg, pmap, lut_s, lane, is_agent, live, pos, ori, env, same, true);
                // The base grid is staged again.  Nothing else needs restoring: a render never writes the slack or the "outside"
                // fill of the maps, and it rebuilds every map cell it reads.
                w.sync();                                          // the render has read the staged grid
                const uint4* src = reinterpret_cast<const uint4*>(vr.map()->base_grid);
                warp_for(g.GS() >> 4, lane, [&](int i) { reinterpret_cast<uint4*>(sg)[i] = __ldcg(src + i); });
                w.sync();
                reset_env(w, g, p, vr, sg, lane, is_agent, env, gid, tick + 1, pos, ori, apples, waste);
                write_back_reset(w, g, p, sg, lane, is_agent, env, pos, ori);
                live = is_agent; same = 1u << lane;
            }
        }
        if (p.obs || p.state_rgb) draw<TAG, IDX>(w, g, p, sg, pmap, lut_s, lane, is_agent, live, pos, ori, env, same, false);
    }
}

// ------------------------------------------------------------------ incentive bookkeeping (homophily_learner.py:98-115)
__global__ void incentive_kernel(const long long* __restrict__ a_inc, const float* __restrict__ reward, long long rows, int n,
                                 float incentive, float cost, float ratio, float T, int recip,
                                 float* __restrict__ r_env, float* __restrict__ r_inc, float* __restrict__ sgn) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * n) return;
    const long long row = idx / n;
    const int k = (int)(idx - row * n);
    const long long* a = a_inc + row * n * n;
    int give = 0, rp = 0, rn = 0;
    for (int j = 0; j < n; ++j) {
        if (j == k) continue;                                  // inc_mask_actions = 1 - eye
        give += a[k * n + j] != 0;
        const long long v = a[j * n + k];
        rp += v == 1; rn += v == 2;
    }
    const float rv = (float)(rp - rn), r = reward[idx];
    const float e = __fadd_rn(r, __fmul_rn(__fmul_rn(rv, ratio), incentive));
    const float c = __fsub_rn(r, __fmul_rn(__fmul_rn((float)give, cost), incentive));
    if (recip) { const float inv = __fdiv_rn(1.0f, T); r_env[idx] = __fmul_rn(e, inv); r_inc[idx] = __fmul_rn(c, inv); }
    else { r_env[idx] = __fdiv_rn(e, T); r_inc[idx] = __fdiv_rn(c, T); }
    if (sgn) sgn[idx] = rv > 0.f ? 1.f : (rv < 0.f ? -1.f : 0.f);
}

// ------------------------------------------------------------------ episode counters of a reset (ssd_reset with ssd_set_stats)
// Zeroes the SSD_N_STATS x agent_stride counters of every env whose mask byte is non-zero (mask NULL: every env).  A kernel of its
// own, so that the MODE_RESET instantiations keep their code.  ssd_reset also runs it over the shaping traces (per_env =
// agent_stride words; 0.0f is the all-zero word).
__global__ void __launch_bounds__(256) zero_stats_kernel(uint32_t* __restrict__ stats, const uint8_t* __restrict__ mask,
                                                         long long total, int per_env) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    if (mask && mask[i / per_env] == 0) return;
    stats[i] = 0u;
}

// ------------------------------------------------------------------ shaped rewards (ssd_set_reward_shaping; DESIGN.md §3 item 17)
// One parameter set as the kernel reads it: a = alpha/(n-1), b = beta/(n-1) and w1 = 1 - w are precomputed on the host in fp32.
struct ShapeDev { float a, b, decay, w, w1; };

struct ShapeParams {
    const int8_t* reward;                     // [B][n] the step's rewards
    const uint8_t* done;                      // [B] auto-reset launches only (NULL otherwise): a done env's trace restarts at 0
    const uint8_t* variant_of;                // [B] or NULL: every env uses params[0]
    const ShapeDev* params; int n_params;
    float* trace; float* shaped;              // [B][NA]
    int n, NA, env0, env1;
};

// One warp per env and one lane per agent, as in ssd_kernel.  Every operation is an explicitly rounded fp32 intrinsic, so nothing
// is contracted into an FMA and the result is bit-exact against a NumPy float32 restatement (tests/shaping_ref.py).  The n-way
// sums run over n shuffles in ascending j.  A kernel of its own after the step launch, so that no ssd_kernel instantiation
// changes.
__global__ void __launch_bounds__(kWarps * 32) shape_rewards_kernel(const __grid_constant__ ShapeParams p) {
    // Under programmatic dependent launch (small launches, as the step launch before it): wait for the step's outputs, and let
    // the next step launch of the stream become resident and run its prologue meanwhile (it still waits for this whole grid).
    // Both are no-ops in a plain launch.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int lane = threadIdx.x & 31;
    const int env = p.env0 + blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (env >= p.env1) return;
    const int pid = p.variant_of ? min((int)__ldcg(p.variant_of + env), p.n_params - 1) : 0;
    const ShapeDev s = p.params[pid];
    const bool is_agent = lane < p.n;
    // mutable buffers are read past L1, as in ssd_kernel: concurrent env ranges may share a line at a range boundary
    const int ri = is_agent ? (int)__ldcg(p.reward + (size_t)env * p.n + lane) : 0;
    const size_t at = (size_t)env * p.NA + lane;
    const float r = (float)ri;
    const float e = __fadd_rn(__fmul_rn(is_agent ? __ldcg(p.trace + at) : 0.0f, s.decay), r);
    int sum = 0;
    float D = 0.0f, A = 0.0f;
    for (int j = 0; j < p.n; ++j) {
        const float ej = __shfl_sync(0xffffffffu, e, j);
        sum += __shfl_sync(0xffffffffu, ri, j);
        if (j != lane) {
            D = __fadd_rn(D, fmaxf(__fsub_rn(ej, e), 0.0f));
            A = __fadd_rn(A, fmaxf(__fsub_rn(e, ej), 0.0f));
        }
    }
    const float c = __fdiv_rn((float)sum, (float)p.n);
    const float m = __fadd_rn(__fmul_rn(s.w1, r), __fmul_rn(s.w, c));
    const float u = __fsub_rn(__fsub_rn(m, __fmul_rn(s.a, D)), __fmul_rn(s.b, A));
    if (is_agent) {
        p.shaped[at] = u;
        p.trace[at] = (p.done && __ldcg(p.done + env)) ? 0.0f : e;
    }
}

// ------------------------------------------------------------------ index4 -> f32 RGB (ssd_expand_obs, ssd_expand_state)
// One CTA per block of rows x cols nibbles (an agent view, or an env's state image), one thread per pixel:
// f32 [3][rows][cols] = color_lut[nibble] / 256, exactly what u8 RGB / 256 gives.
struct ExpandParams {
    const uint8_t* in;                        // first block of the range in the index4 buffer
    float* out;                               // [blocks][3][rows][cols]
    int rows, cols, row_stride, block_stride; // block_stride: bytes between blocks (agent or env stride)
    uint32_t lut[16];                         // R | G << 8 | B << 16 per colour index
};
__global__ void __launch_bounds__(256) expand_index4_kernel(const __grid_constant__ ExpandParams p) {
    const uint8_t* __restrict__ in = p.in + (size_t)blockIdx.x * p.block_stride;
    const int NN = p.rows * p.cols;
    float* __restrict__ out = p.out + (size_t)blockIdx.x * 3 * NN;
    for (int q = threadIdx.x; q < NN; q += blockDim.x) {
        const int y = q / p.cols, x = q - y * p.cols;
        const uint32_t rgb = p.lut[(__ldg(in + y * p.row_stride + (x >> 1)) >> (4 * (x & 1))) & 15u];
        out[q] = (float)(rgb & 0xffu) * (1.0f / 256.0f);
        out[NN + q] = (float)((rgb >> 8) & 0xffu) * (1.0f / 256.0f);
        out[2 * NN + q] = (float)((rgb >> 16) & 0xffu) * (1.0f / 256.0f);
    }
}

thread_local int g_last_cuda_error = 0;

inline int cuda_fail(cudaError_t e) { g_last_cuda_error = (int)e; return SSD_ERR_CUDA; }
#define SSD_CUDA(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_); } while (0)

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Makes the handle's device current for the duration of a call and restores the caller's device afterwards.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) { err = cudaSetDevice(dev); switched = err == cudaSuccess; }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

uint32_t magic20(int d, int max_x) {
    // smallest m with floor(x*m / 2^20) == floor(x / d) for all 0 <= x <= max_x (verified exhaustively)
    uint32_t m = (uint32_t)(((1u << 20) + d - 1) / d);
    for (int x = 0; x <= max_x; ++x)
        if ((int)(((uint64_t)x * m) >> 20) != x / d) return 0;
    return m;
}

// Observation strides of one format (ssd_get_obs_layout; ssd_step_host copies B * env_stride bytes).
ssd_obs_layout obs_layout(const KParams& k, int32_t format) {
    const GeoVals& g = k.geo;
    if (format == SSD_OBS_INDEX4) return { format, g.RS4, 0, g.AS4, k.n * g.AS4 };
    return { format, g.RP, g.PS, g.AS, k.n * g.AS };
}

// State image strides of one format (ssd_get_state_layout; ssd_step_host copies B * env_stride bytes).  An index4 row is
// nw8M words, which is ceil(W/2) rounded up to 4 bytes.
ssd_state_layout state_layout(const KParams& k, int32_t format) {
    const GeoVals& g = k.geo;
    if (format == SSD_OBS_INDEX4) return { format, 4 * g.nw8M, 0, 4 * round_up(g.H * g.nw8M, 4) };
    return { format, g.W, g.G, 3 * g.G };
}

}  // namespace

struct ssd_handle {
    KParams kp;
    MapDev* d_map;
    int device;
    size_t smem_bytes;
    mutable int64_t launches;                                 // also counts ssd_expand_obs / _state, which take a const handle
    int force_generic;                                        // SSD_B200_GENERIC=1: always use the runtime-geometry kernels
    int pdl;                                                  // programmatic dependent launch for small launches (SSD_B200_PDL=0 turns it off)
    int obs_format;                                           // SSD_OBS_RGB (at creation) or SSD_OBS_INDEX4
    int state_format;                                         // the same, for the state image
    VarDev* d_vars;                                           // variant table: SSD_MAX_VARIANTS records, allocated once when first needed
    VarDev* base;                                             // host copy of the creation config's record (ssd_set_variants(h, 0, ...))
    int tag_any;                                              // some variant of the table has tag_timeout > 0
    ShapeDev* d_shape;                                        // shaping table: SSD_MAX_VARIANTS records, allocated once when first needed
    int n_shape;                                              // entries in use; 0 = shaping off
    float* shape_trace; float* shaped;                        // caller-owned [B][NA] (ssd_set_reward_shaping)
};

static int fill_common(const ssd_handle* h, const ssd_state* st, const ssd_draws* d, KParams& k) {
    if (!h || !st || !st->grid || !st->agent || !st->ep_ret || !st->t || !st->tick || !st->counts) return SSD_ERR_INVALID;
    k = h->kp;
    k.env0 = 0; k.env1 = k.B;
    k.state_idx4 = h->state_format == SSD_OBS_INDEX4;
    k.grid = st->grid; k.agent = st->agent; k.ep_ret = st->ep_ret; k.t = st->t; k.tick = st->tick; k.counts = st->counts;
    if (d) {
        if ((d->u_waste == nullptr) != (d->wkey == nullptr)) return SSD_ERR_INVALID;
        k.d_prio = d->prio; k.d_uapple = d->u_apple; k.d_uwaste = d->u_waste; k.d_wkey = d->wkey;
        k.d_spawnkey = d->spawn_key; k.d_rot = d->rot;
    }
    return SSD_OK;
}

template <int MODE, class GEO, bool TAG, bool IDX, bool VAR, bool STATS>
static int launch_kernel(ssd_handle* h, const KParams& k, void* stream) {
    DeviceGuard guard(h->device);
    SSD_CUDA(guard.err);
    {   // cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel FUNCTION (per device), not to a handle: all
        // runtime-geometry handles share one instantiation, so the limit is only ever raised (high-water mark).
        static std::mutex mu;
        static int high_water[kMaxDevices] = {};
        std::lock_guard<std::mutex> lock(mu);
        const int dev = h->device;
        if (dev < 0 || dev >= kMaxDevices) return SSD_ERR_INVALID;
        if ((int)h->smem_bytes > high_water[dev]) {
            SSD_CUDA(cudaFuncSetAttribute(ssd_kernel<MODE, GEO, TAG, IDX, VAR, STATS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
            high_water[dev] = (int)h->smem_bytes;
        }
    }
    const int grid = (k.env1 - k.env0 + kWarps - 1) / kWarps;
    if (grid <= 0) return SSD_OK;

    if (k.pdl) {                                               // programmatic dependent launch (see launch_geo)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kWarps * 32); cfg.dynamicSmemBytes = h->smem_bytes;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        SSD_CUDA(cudaLaunchKernelEx(&cfg, ssd_kernel<MODE, GEO, TAG, IDX, VAR, STATS>, k));
    } else {
        ssd_kernel<MODE, GEO, TAG, IDX, VAR, STATS><<<grid, kWarps * 32, h->smem_bytes, (cudaStream_t)stream>>>(k);
    }
    ++h->launches;
    SSD_CUDA(cudaGetLastError());
    return SSD_OK;
}

// Launches of at most a few waves are bound by the latency of their own chain (launch -> state loads -> logic -> stores), so
// consecutive launches of a stream are chained programmatically: the next one becomes resident and runs its prologue while this
// one stores observations (cleanup5, 4 096 envs in 8 ranges: 8.7 -> 7.2 us per step; harvest5: 12.1 -> 10.2 us).  Large
// launches gain nothing and pay for the prologue no longer running under the state loads, so they keep the plain launch.
constexpr int kPdlMaxEnvs = 2048;

static bool use_pdl(const ssd_handle* h, const KParams& k) { return h->pdl && (k.env1 - k.env0) <= kPdlMaxEnvs; }

// The shaped rewards of the step launch just queued with `k` (ssd_set_reward_shaping): shape_rewards_kernel on the same stream
// over the same envs, chained programmatically exactly when the step launch is.  done: the step's done flags for an auto-reset
// step (the traces of the envs it reset restart at 0), NULL otherwise.  Nothing is launched while shaping is off.
static int launch_shaping(ssd_handle* h, const KParams& k, const uint8_t* done, void* stream) {
    if (!h->n_shape) return SSD_OK;
    const int grid = (k.env1 - k.env0 + kWarps - 1) / kWarps;
    if (grid <= 0) return SSD_OK;
    DeviceGuard guard(h->device);
    SSD_CUDA(guard.err);
    ShapeParams s;
    s.reward = k.reward; s.done = done; s.variant_of = k.variant_of; s.params = h->d_shape; s.n_params = h->n_shape;
    s.trace = h->shape_trace; s.shaped = h->shaped;
    s.n = k.n; s.NA = k.NA; s.env0 = k.env0; s.env1 = k.env1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kWarps * 32); cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    if (use_pdl(h, k)) { cfg.attrs = attr; cfg.numAttrs = 1; }
    SSD_CUDA(cudaLaunchKernelEx(&cfg, shape_rewards_kernel, s));
    ++h->launches;
    SSD_CUDA(cudaGetLastError());
    return SSD_OK;
}

// Zeroes `per_env` u32 words of every env whose mask byte is non-zero (mask NULL: every env): ssd_reset's counter and trace reset.
static int zero_masked(ssd_handle* h, uint32_t* buf, const uint8_t* mask, int B, int per_env, void* stream) {
    DeviceGuard guard(h->device);
    SSD_CUDA(guard.err);
    const long long total = (long long)B * per_env;
    zero_stats_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, mask, total, per_env);
    ++h->launches;
    SSD_CUDA(cudaGetLastError());
    return SSD_OK;
}

template <int MODE, class GEO, bool VAR, bool STATS>
static int launch_var(ssd_handle* h, const KParams& k, void* stream) {
    const bool idx = h->obs_format == SSD_OBS_INDEX4;          // packed colour-index observations: their own instantiations
    if constexpr (MODE != MODE_RESET) {                        // tagging-out timers: their own instantiation
        if (k.variant_of ? h->tag_any : k.tag_timeout != 0)
            return idx ? launch_kernel<MODE, GEO, true, true, VAR, STATS>(h, k, stream)
                       : launch_kernel<MODE, GEO, true, false, VAR, STATS>(h, k, stream);
    }
    return idx ? launch_kernel<MODE, GEO, false, true, VAR, STATS>(h, k, stream)
               : launch_kernel<MODE, GEO, false, false, VAR, STATS>(h, k, stream);
}

template <int MODE, class GEO>
static int launch_geo(ssd_handle* h, const KParams& k_in, void* stream) {
    KParams k = k_in;
    k.pdl = use_pdl(h, k);
    // episode counters (ssd_set_stats): their own step instantiations
    if constexpr (MODE == MODE_STEP || MODE == MODE_STEP_RESET) {
        if (k.stats) return k.variant_of ? launch_var<MODE, GEO, true, true>(h, k, stream) : launch_var<MODE, GEO, false, true>(h, k, stream);
    }
    // per-env variants: their own instantiations (a render reads nothing a variant sets, but draws no agent out of play when
    // any variant tags)
    if constexpr (MODE != MODE_RENDER) {
        if (k.variant_of) return launch_var<MODE, GEO, true, false>(h, k, stream);
    }
    return launch_var<MODE, GEO, false, false>(h, k, stream);
}

// The reference's shipped geometries (constants.py maps x yaml view sizes) get compile-time index arithmetic.
template <int MODE>
static int launch(ssd_handle* h, const KParams& k, void* stream) {
    const GeoVals& v = k.geo;
    if (!h->force_generic) {
        if (v.kind == SSD_KIND_HARVEST && v.H == 9 && v.W == 38 && v.V == 15) return launch_geo<MODE, GeoS<SSD_KIND_HARVEST, 9, 38, 15>>(h, k, stream);
        if (v.kind == SSD_KIND_HARVEST && v.H == 9 && v.W == 38 && v.V == 7) return launch_geo<MODE, GeoS<SSD_KIND_HARVEST, 9, 38, 7>>(h, k, stream);
        if (v.kind == SSD_KIND_CLEANUP && v.H == 25 && v.W == 18 && v.V == 7) return launch_geo<MODE, GeoS<SSD_KIND_CLEANUP, 25, 18, 7>>(h, k, stream);
        if (v.kind == SSD_KIND_CLEANUP && v.H == 48 && v.W == 18 && v.V == 7) return launch_geo<MODE, GeoS<SSD_KIND_CLEANUP, 48, 18, 7>>(h, k, stream);
        if (v.kind == SSD_KIND_CLEANUP && v.H == 10 && v.W == 10 && v.V == 7) return launch_geo<MODE, GeoS<SSD_KIND_CLEANUP, 10, 10, 7>>(h, k, stream);
    }
    return launch_geo<MODE, GeoD>(h, k, stream);
}

// One variant of a handle of kind `kind`, H x W and n agents, checked as ssd_create checks its config: the int8 reward bound and the
// 8-bit timer (SSD_ERR_INVALID), a wall-enclosed map in the kind's alphabet (SSD_ERR_MAP), at least n spawn points (SSD_ERR_SPAWN),
// at most SSD_MAX_SPAWN of them, the Cleanup LUT length (#waste points + 1) and the apple point limit of spawn (SSD_ERR_INVALID).
// Every point slot past the lists holds kNoPoint, so a launch that pairs a table with a stale count never reads a bogus cell.
static int compile_variant(int kind, int H, int W, int n, const char* ascii_map, uint32_t n_waste_lut, const uint32_t* thr_apple,
                           const uint32_t* thr_waste, const uint32_t thr_harvest[4], int fire_cost, int hit_penalty, int tag_timeout,
                           VarDev* v) {
    if (!ascii_map) return SSD_ERR_INVALID;
    if (abs(fire_cost) + n * abs(hit_penalty) + 1 > 127) return SSD_ERR_INVALID;   // reward is int8
    if (tag_timeout < 0 || tag_timeout > 255) return SSD_ERR_INVALID;              // 8-bit timer in the agent record
    memset(v, 0, sizeof(VarDev));
    MapDev* hm = &v->map;
    for (int k = 0; k < SSD_MAX_CELLS + 4; ++k) hm->apple_pts[k] = hm->waste_pts[k] = kNoPoint;
    const int G = H * W;
    int na = 0, nw = 0, ns = 0;
    for (int c = 0; c < G; ++c) {
        const char ch = ascii_map[c];
        const int r = c / W, col = c % W;
        const bool border = r == 0 || col == 0 || r == H - 1 || col == W - 1;
        if (border && ch != '@') return SSD_ERR_MAP;
        uint8_t code = SSD_CELL_EMPTY;
        switch (ch) {
            case '@': code = SSD_CELL_WALL; break;
            case ' ': break;
            case 'P': if (ns < SSD_MAX_SPAWN) hm->spawn_pts[ns] = (uint16_t)c; ++ns; break;   // map_env.py:143-146
            case 'A': if (kind == SSD_KIND_HARVEST) { code = SSD_CELL_APPLE; hm->apple_pts[na++] = (uint16_t)c; } break;
            case 'B': if (kind == SSD_KIND_CLEANUP) hm->apple_pts[na++] = (uint16_t)c; break;   // cleanup.py:81-82
            case 'H': if (kind == SSD_KIND_CLEANUP) { code = SSD_CELL_WASTE; hm->waste_pts[nw++] = (uint16_t)c; } break;
            case 'R': if (kind == SSD_KIND_CLEANUP) code = SSD_CELL_RIVER; break;
            case 'S': if (kind == SSD_KIND_CLEANUP) code = SSD_CELL_STREAM; break;
            default: return SSD_ERR_MAP;
        }
        hm->base_grid[c] = code;
    }
    if (ns < n) return SSD_ERR_SPAWN;
    if (ns > SSD_MAX_SPAWN) return SSD_ERR_INVALID;
    if (kind == SSD_KIND_CLEANUP) {
        if (n_waste_lut != (uint32_t)nw + 1 || !thr_apple || !thr_waste) return SSD_ERR_INVALID;
        memcpy(hm->thr_apple, thr_apple, sizeof(uint32_t) * (nw + 1));
        memcpy(hm->thr_waste, thr_waste, sizeof(uint32_t) * (nw + 1));
    }
    v->n_apple = na; v->n_waste = nw; v->n_spawn = ns; v->n_apple4 = (na + 3) / 4; v->n_waste2 = (nw + 1) / 2;
    if (v->n_apple4 > 32 * 16) return SSD_ERR_INVALID;                               // spawn's 64-bit decision mask
    for (int c = 0; c < G; ++c) { v->base_apples += hm->base_grid[c] == SSD_CELL_APPLE; v->base_waste += hm->base_grid[c] == SSD_CELL_WASTE; }
    v->fire_cost = fire_cost; v->hit_penalty = hit_penalty; v->tag_timeout = tag_timeout;
    for (int i = 0; i < 4; ++i) v->thr_harvest[i] = thr_harvest[i];
    return SSD_OK;
}

// The scalars of variant 0 live in KParams, where every launch without an id array reads them.
static void set_variant0(KParams& k, const VarDev& v) {
    k.n_apple = v.n_apple; k.n_waste = v.n_waste; k.n_spawn = v.n_spawn; k.n_apple4 = v.n_apple4; k.n_waste2 = v.n_waste2;
    k.base_apples = v.base_apples; k.base_waste = v.base_waste;
    k.fire_cost = v.fire_cost; k.hit_penalty = v.hit_penalty; k.tag_timeout = v.tag_timeout;
    for (int i = 0; i < 4; ++i) k.thr_harvest[i] = v.thr_harvest[i];
}

// Allocates the variant table at its full size, every record the creation config, the first time a call needs it.  It is never
// reallocated, so no launch, queued or captured in a CUDA graph, can read a freed table.
static int ensure_variant_table(ssd_handle* h) {
    if (h->d_vars) return SSD_OK;
    VarDev* d = nullptr;
    SSD_CUDA(cudaMalloc(&d, sizeof(VarDev) * SSD_MAX_VARIANTS));
    for (int i = 0; i < SSD_MAX_VARIANTS; ++i) {
        const cudaError_t e = cudaMemcpy(d + i, h->base, sizeof(VarDev), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFree(d); return cuda_fail(e); }
    }
    h->d_vars = d;
    h->kp.variants = d;
    return SSD_OK;
}

extern "C" {

int ssd_abi_version(void) { return SSD_B200_ABI_VERSION; }

const char* ssd_error_string(int code) {
    switch (code) {
        case SSD_OK: return "ok";
        case SSD_ERR_INVALID: return "invalid argument or unsupported geometry";
        case SSD_ERR_CUDA: return "CUDA runtime error";
        case SSD_ERR_SPAWN: return "There are not enough spawn points! Check your map?";
        case SSD_ERR_MAP: return "map must be wall-enclosed and use the reference alphabet";
        default: return "unknown error";
    }
}

int ssd_last_cuda_error(void) { return g_last_cuda_error; }

uint32_t ssd_prob_to_threshold(double p) {
    if (!(p > 0.0)) return 0u;
    const double t = ceil(p * 4294967296.0);
    return t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
}

int ssd_create(const ssd_config* cfg, ssd_handle** out) {
    if (!cfg || !out || !cfg->ascii_map) return SSD_ERR_INVALID;
    *out = nullptr;
    const int H = cfg->height, W = cfg->width, G = H * W, n = cfg->n_agents, V = cfg->view;
    if (cfg->kind != SSD_KIND_CLEANUP && cfg->kind != SSD_KIND_HARVEST) return SSD_ERR_INVALID;
    if (H < 3 || W < 3 || H > 255 || W > 255 || G > SSD_MAX_CELLS) return SSD_ERR_INVALID;
    if (n < 1 || n > SSD_MAX_AGENTS || V < 1 || V > 31 || cfg->n_envs < 1) return SSD_ERR_INVALID;
    if (cfg->beam_len < 0 || cfg->episode_limit < 1 || cfg->spawn_rotation > 3) return SSD_ERR_INVALID;
    if (abs(cfg->fire_cost) + n * abs(cfg->hit_penalty) + 1 > 127) return SSD_ERR_INVALID;   // reward is int8
    if (cfg->tag_timeout < 0 || cfg->tag_timeout > 255) return SSD_ERR_INVALID;              // 8-bit timer in the agent record

    VarDev* v0 = new (std::nothrow) VarDev;
    if (!v0) return SSD_ERR_INVALID;
    {
        const int rc = compile_variant(cfg->kind, H, W, n, cfg->ascii_map, cfg->n_waste_lut, cfg->thr_apple, cfg->thr_waste,
                                       cfg->thr_harvest, cfg->fire_cost, cfg->hit_penalty, cfg->tag_timeout, v0);
        if (rc) { delete v0; return rc; }
    }
    const MapDev* hm = &v0->map;

    ssd_handle* h = new (std::nothrow) ssd_handle;
    if (!h) { delete v0; return SSD_ERR_INVALID; }
    memset(h, 0, sizeof(*h));
    KParams& k = h->kp;
    k.geo = make_geo(cfg->kind, H, W, V);
    const GeoVals& gv = k.geo;
    k.B = cfg->n_envs; k.n = n; k.NA = round_up(n, 4);
    k.episode_limit = cfg->episode_limit;
    k.beam_len = cfg->beam_len; k.n_actions = cfg->kind == SSD_KIND_CLEANUP ? 9 : 8;
    set_variant0(k, *v0);
    k.n_variants = 1;
    h->base = v0;
    k.random_spawn = cfg->random_spawn_point != 0; k.spawn_rot = cfg->spawn_rotation < 0 ? -1 : cfg->spawn_rotation;
    k.invN20 = magic20(gv.N, SSD_MAX_AGENTS * gv.N + 64); k.invW20 = magic20(W, G + 1);
    k.seed_lo = (uint32_t)cfg->seed; k.seed_hi = (uint32_t)(cfg->seed >> 32); k.gid_base = cfg->env_gid_base;
    for (int i = 0; i < 16; ++i)
        k.lut[i] = (uint32_t)cfg->color_lut[i][0] | ((uint32_t)cfg->color_lut[i][1] << 8) | ((uint32_t)cfg->color_lut[i][2] << 16);
    k.agents_uniform = 1;
    for (int i = 8; i < 16; ++i) if (k.lut[i] != k.lut[7]) k.agents_uniform = 0;
    for (int ch = 0; ch < 3; ++ch) {                          // 8-entry per-plane LUT: indices 0-6 + 7 = agent
        uint32_t lo = 0, hi = 0;
        for (int i = 0; i < 4; ++i) { lo |= (uint32_t)cfg->color_lut[i][ch] << (8 * i); hi |= (uint32_t)cfg->color_lut[4 + i][ch] << (8 * i); }
        k.lut8[2 * ch] = lo; k.lut8[2 * ch + 1] = hi;
    }
    if (k.invN20 == 0 || k.invW20 == 0) { delete v0; delete h; return SSD_ERR_INVALID; }

    k.invMW20 = magic20(gv.nw8M, H * gv.nw8M + 32);
    if (k.invMW20 == 0 || gv.PMS >= 60000) { delete v0; delete h; return SSD_ERR_INVALID; }
    h->smem_bytes = (size_t)kWarps * (gv.padF + gv.GS + gv.padB + gv.PMS);     // one staging tile per warp
    { const char* e = getenv("SSD_B200_GENERIC"); h->force_generic = e && e[0] == '1'; }
    { const char* e = getenv("SSD_B200_PDL"); h->pdl = !(e && e[0] == '0'); }
    h->device = cfg->device;

    DeviceGuard guard(cfg->device);
    cudaError_t e = guard.err;
    if (e == cudaSuccess) {                                   // the launch needs smem_bytes dynamic + the static LUTs
        int optin = 0;
        e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
        if (e == cudaSuccess && h->smem_bytes + sizeof(ColourLuts) > (size_t)optin) { delete v0; delete h; return SSD_ERR_INVALID; }
    }
    if (e == cudaSuccess) e = cudaMalloc(&h->d_map, sizeof(MapDev));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_map, hm, sizeof(MapDev), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        if (h->d_map) cudaFree(h->d_map);
        delete v0;
        delete h;
        return cuda_fail(e);
    }
    k.map = h->d_map;
    *out = h;
    return SSD_OK;
}

int ssd_destroy(ssd_handle* h) {
    if (!h) return SSD_ERR_INVALID;
    DeviceGuard guard(h->device);
    cudaFree(h->d_map);
    if (h->d_vars) cudaFree(h->d_vars);
    if (h->d_shape) cudaFree(h->d_shape);
    delete h->base;
    delete h;
    return SSD_OK;
}

int ssd_get_layout(const ssd_handle* h, ssd_layout* o) {
    if (!h || !o) return SSD_ERR_INVALID;
    const KParams& k = h->kp;
    const GeoVals& g = k.geo;
    o->n_actions = k.n_actions; o->n_cells = g.G; o->obs_n = g.N; o->grid_stride = g.GS; o->agent_stride = k.NA;
    o->obs_plane_stride = g.PS; o->obs_agent_stride = g.AS; o->obs_env_stride = obs_layout(k, SSD_OBS_RGB).env_stride;
    o->n_apple_pts = k.n_apple; o->n_waste_pts = k.n_waste; o->n_spawn_pts = k.n_spawn; o->obs_row_stride = g.RP;
    return SSD_OK;
}

int ssd_get_obs_layout(const ssd_handle* h, int32_t format, ssd_obs_layout* o) {
    if (!h || !o || (format != SSD_OBS_RGB && format != SSD_OBS_INDEX4)) return SSD_ERR_INVALID;
    *o = obs_layout(h->kp, format);
    return SSD_OK;
}

int ssd_set_obs_format(ssd_handle* h, int32_t format) {
    if (!h || (format != SSD_OBS_RGB && format != SSD_OBS_INDEX4)) return SSD_ERR_INVALID;
    h->obs_format = format;
    return SSD_OK;
}

int ssd_get_state_layout(const ssd_handle* h, int32_t format, ssd_state_layout* o) {
    if (!h || !o || (format != SSD_OBS_RGB && format != SSD_OBS_INDEX4)) return SSD_ERR_INVALID;
    *o = state_layout(h->kp, format);
    return SSD_OK;
}

int ssd_set_state_format(ssd_handle* h, int32_t format) {
    if (!h || (format != SSD_OBS_RGB && format != SSD_OBS_INDEX4)) return SSD_ERR_INVALID;
    h->state_format = format;
    return SSD_OK;
}

int ssd_set_variants(ssd_handle* h, int32_t n_variants, const ssd_variant* variants) {
    if (!h || n_variants < 0 || n_variants > SSD_MAX_VARIANTS || (n_variants > 0 && !variants)) return SSD_ERR_INVALID;
    const int m = n_variants > 0 ? n_variants : 1;
    VarDev* recs = new (std::nothrow) VarDev[m];
    if (!recs) return SSD_ERR_INVALID;
    const GeoVals& g = h->kp.geo;
    if (n_variants == 0) recs[0] = *h->base;
    for (int i = 0; i < n_variants; ++i) {
        const ssd_variant& v = variants[i];
        const int rc = compile_variant(g.kind, g.H, g.W, h->kp.n, v.ascii_map, v.n_waste_lut, v.thr_apple, v.thr_waste, v.thr_harvest,
                                       v.fire_cost, v.hit_penalty, v.tag_timeout, &recs[i]);
        if (rc) { delete[] recs; return rc; }
    }
    DeviceGuard guard(h->device);
    cudaError_t e = guard.err;
    if (e == cudaSuccess) {
        const int rc = ensure_variant_table(h);
        if (rc) { delete[] recs; return rc; }
        e = cudaDeviceSynchronize();                          // no launch in flight reads the table or the map while they change
    }
    if (e == cudaSuccess) e = cudaMemcpy(h->d_vars, recs, sizeof(VarDev) * m, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_map, &recs[0].map, sizeof(MapDev), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete[] recs; return cuda_fail(e); }
    set_variant0(h->kp, recs[0]);
    h->kp.n_variants = m;
    h->tag_any = 0;
    for (int i = 0; i < m; ++i) h->tag_any |= recs[i].tag_timeout != 0;
    delete[] recs;
    return SSD_OK;
}

int ssd_set_env_variants(ssd_handle* h, const uint8_t* variant_of) {
    if (!h) return SSD_ERR_INVALID;
    if (variant_of) {
        DeviceGuard guard(h->device);
        SSD_CUDA(guard.err);
        const int rc = ensure_variant_table(h);
        if (rc) return rc;
    }
    h->kp.variant_of = variant_of;
    return SSD_OK;
}

int ssd_set_stats(ssd_handle* h, uint32_t* stats, uint32_t* end_stats) {
    if (!h || (end_stats && !stats)) return SSD_ERR_INVALID;
    if (stats && h->kp.episode_limit > 65535) return SSD_ERR_INVALID;   // APPLE_T of an episode stays below 2^31
    h->kp.stats = stats; h->kp.end_stats = end_stats;
    return SSD_OK;
}

int ssd_set_reward_shaping(ssd_handle* h, int32_t n_params, const ssd_shaping* params, float* trace, float* shaped) {
    if (!h || n_params < 0 || n_params > SSD_MAX_VARIANTS || (n_params > 0 && !params)) return SSD_ERR_INVALID;
    if ((trace == nullptr) != (shaped == nullptr) || (trace != nullptr) != (n_params > 0)) return SSD_ERR_INVALID;
    ShapeDev recs[SSD_MAX_VARIANTS];
    const int n = h->kp.n;
    for (int i = 0; i < n_params; ++i) {
        const ssd_shaping& q = params[i];
        if (!isfinite(q.alpha) || !isfinite(q.beta) || !isfinite(q.decay) || !isfinite(q.prosocial)) return SSD_ERR_INVALID;
        if (q.alpha < 0.0f || q.beta < 0.0f || q.decay < 0.0f || q.decay > 1.0f || q.prosocial < 0.0f || q.prosocial > 1.0f)
            return SSD_ERR_INVALID;
        const float others = (float)(n - 1);
        recs[i].a = n > 1 ? q.alpha / others : 0.0f;
        recs[i].b = n > 1 ? q.beta / others : 0.0f;
        recs[i].decay = q.decay; recs[i].w = q.prosocial; recs[i].w1 = 1.0f - q.prosocial;
    }
    if (n_params > 0) {
        DeviceGuard guard(h->device);
        SSD_CUDA(guard.err);
        if (!h->d_shape) {                                    // allocated once at full size: no launch ever reads a freed table
            ShapeDev* d = nullptr;
            SSD_CUDA(cudaMalloc(&d, sizeof(ShapeDev) * SSD_MAX_VARIANTS));
            h->d_shape = d;
        }
        SSD_CUDA(cudaDeviceSynchronize());                    // no launch in flight reads the table while it changes
        SSD_CUDA(cudaMemcpy(h->d_shape, recs, sizeof(ShapeDev) * n_params, cudaMemcpyHostToDevice));
    }
    h->n_shape = n_params; h->shape_trace = trace; h->shaped = shaped;
    return SSD_OK;
}

int ssd_reset(ssd_handle* h, const ssd_state* st, const uint8_t* mask, const ssd_draws* draws, uint8_t* obs, void* stream) {
    KParams k;
    const int rc = fill_common(h, st, draws, k);
    if (rc) return rc;
    k.mask = mask; k.obs = obs;
    int lrc = launch<MODE_RESET>(h, k, stream);
    if (!lrc && k.stats) lrc = zero_masked(h, k.stats, mask, k.B, SSD_N_STATS * k.NA, stream);
    if (!lrc && h->n_shape) lrc = zero_masked(h, reinterpret_cast<uint32_t*>(h->shape_trace), mask, k.B, k.NA, stream);
    return lrc;
}

int ssd_step(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
             const ssd_step_out* out, void* stream) {
    return ssd_step_range(h, st, actions, draws, out, 0, h ? h->kp.B : 0, stream);
}

// The arguments of a step over envs [env_begin, env_begin + env_count), validated before any CUDA call.
static int fill_step(const ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
                     const ssd_step_out* out, int32_t env_begin, int32_t env_count, KParams& k) {
    const int rc = fill_common(h, st, draws, k);
    if (rc) return rc;
    if (!actions || !out || !out->reward || !out->clean || !out->apple_cnt || !out->done) return SSD_ERR_INVALID;
    if (env_begin < 0 || env_count < 0 || (int64_t)env_begin + env_count > k.B) return SSD_ERR_INVALID;
    k.env0 = env_begin; k.env1 = env_begin + env_count;
    k.actions = actions; k.reward = out->reward; k.clean = out->clean; k.apple_cnt = out->apple_cnt; k.done = out->done;
    k.obs = out->obs; k.state_rgb = out->state_rgb;
    return SSD_OK;
}

int ssd_step_range(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
                   const ssd_step_out* out, int32_t env_begin, int32_t env_count, void* stream) {
    KParams k;
    const int rc = fill_step(h, st, actions, draws, out, env_begin, env_count, k);
    if (rc) return rc;
    const int lrc = launch<MODE_STEP>(h, k, stream);
    return lrc ? lrc : launch_shaping(h, k, nullptr, stream);
}

int ssd_step_autoreset(ssd_handle* h, const ssd_state* st, const uint8_t* actions, const ssd_draws* draws,
                       const ssd_step_out* out, const ssd_episode_end* end, int32_t env_begin, int32_t env_count,
                       void* stream) {
    KParams k;
    const int rc = fill_step(h, st, actions, draws, out, env_begin, env_count, k);
    if (rc) return rc;
    if (end) { k.end_obs = end->obs; k.end_state = end->state_rgb; k.end_ep_ret = end->ep_ret; }
    const int lrc = launch<MODE_STEP_RESET>(h, k, stream);
    return lrc ? lrc : launch_shaping(h, k, k.done, stream);
}

int ssd_render(ssd_handle* h, const ssd_state* st, uint8_t* obs, uint8_t* state_rgb, void* stream) {
    KParams k;
    const int rc = fill_common(h, st, nullptr, k);
    if (rc) return rc;
    if (!obs && !state_rgb) return SSD_ERR_INVALID;
    k.obs = obs; k.state_rgb = state_rgb;
    return launch<MODE_RENDER>(h, k, stream);
}

int ssd_step_host(ssd_handle* h, const ssd_state* st, const uint8_t* h_actions, uint8_t* d_actions,
                  const ssd_step_out* d_out, const ssd_step_out* h_out, void* stream) {
    if (!h || !h_actions || !d_actions || !d_out || !h_out) return SSD_ERR_INVALID;
    DeviceGuard guard(h->device);
    SSD_CUDA(guard.err);
    const KParams& k = h->kp;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = (size_t)k.B;
    SSD_CUDA(cudaMemcpyAsync(d_actions, h_actions, B * k.n, cudaMemcpyHostToDevice, s));
    KParams ks;                                               // ssd_step, except that a host step leaves the episode counters alone
    int rc = fill_step(h, st, d_actions, nullptr, d_out, 0, k.B, ks);
    if (rc) return rc;
    ks.stats = ks.end_stats = nullptr;
    rc = launch<MODE_STEP>(h, ks, stream);
    if (!rc) rc = launch_shaping(h, ks, nullptr, stream);     // the shaped rewards are updated like ssd_step's
    if (rc) return rc;
    if (h_out->reward) SSD_CUDA(cudaMemcpyAsync(h_out->reward, d_out->reward, B * k.n, cudaMemcpyDeviceToHost, s));
    if (h_out->clean) SSD_CUDA(cudaMemcpyAsync(h_out->clean, d_out->clean, B * k.n, cudaMemcpyDeviceToHost, s));
    if (h_out->apple_cnt) SSD_CUDA(cudaMemcpyAsync(h_out->apple_cnt, d_out->apple_cnt, B * 2, cudaMemcpyDeviceToHost, s));
    if (h_out->done) SSD_CUDA(cudaMemcpyAsync(h_out->done, d_out->done, B, cudaMemcpyDeviceToHost, s));
    const size_t ES = (size_t)obs_layout(k, h->obs_format).env_stride;
    if (h_out->obs && d_out->obs) SSD_CUDA(cudaMemcpyAsync(h_out->obs, d_out->obs, B * ES, cudaMemcpyDeviceToHost, s));
    if (h_out->state_rgb && d_out->state_rgb)
        SSD_CUDA(cudaMemcpyAsync(h_out->state_rgb, d_out->state_rgb, B * (size_t)state_layout(k, h->state_format).env_stride,
                                 cudaMemcpyDeviceToHost, s));
    SSD_CUDA(cudaStreamSynchronize(s));
    return SSD_OK;
}

int ssd_incentive(const int64_t* actions_inc, const float* reward, int64_t rows, int32_t n_agents,
                  float incentive, float cost, float ratio, int32_t max_seq_length,
                  float* rewards_for_env, float* rewards_for_inc, float* recv_sign, void* stream) {
    if (!actions_inc || !reward || !rewards_for_env || !rewards_for_inc || rows < 0 || n_agents < 1 || max_seq_length == 0)
        return SSD_ERR_INVALID;
    if (rows == 0) return SSD_OK;
    // max_seq_length > 0: true division (torch CPU); < 0: multiply by 1/|T| (torch CUDA scalar-divisor path)
    const int recip = max_seq_length < 0;
    const float T = (float)abs(max_seq_length);
    const long long total = (long long)rows * n_agents;
    const int threads = 256;
    incentive_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(actions_inc), reward, rows, n_agents, incentive, cost, ratio, T, recip,
        rewards_for_env, rewards_for_inc, recv_sign);
    SSD_CUDA(cudaGetLastError());
    return SSD_OK;
}

// One expand_index4_kernel launch over `blocks` blocks of rows x cols nibbles, `block_stride` bytes apart from `in`.
static int launch_expand(const ssd_handle* h, const uint8_t* in, int64_t blocks, int rows, int cols, int row_stride,
                         int block_stride, float* out, void* stream) {
    DeviceGuard guard(h->device);
    SSD_CUDA(guard.err);
    ExpandParams e;
    e.in = in; e.out = out;
    e.rows = rows; e.cols = cols; e.row_stride = row_stride; e.block_stride = block_stride;
    for (int i = 0; i < 16; ++i) e.lut[i] = h->kp.lut[i];
    expand_index4_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(e);
    ++h->launches;
    SSD_CUDA(cudaGetLastError());
    return SSD_OK;
}

int ssd_expand_obs(const ssd_handle* h, const uint8_t* obs_index4, int32_t env_begin, int32_t env_count, float* out, void* stream) {
    if (!h || !obs_index4 || !out) return SSD_ERR_INVALID;
    const KParams& k = h->kp;
    if (env_begin < 0 || env_count < 0 || (int64_t)env_begin + env_count > k.B) return SSD_ERR_INVALID;
    if (env_count == 0) return SSD_OK;
    const GeoVals& g = k.geo;
    return launch_expand(h, obs_index4 + (size_t)env_begin * k.n * g.AS4, (int64_t)env_count * k.n, g.N, g.N, g.RS4, g.AS4,
                         out, stream);
}

int ssd_expand_state(const ssd_handle* h, const uint8_t* state_index4, int32_t env_begin, int32_t env_count, float* out,
                     void* stream) {
    if (!h || !state_index4 || !out) return SSD_ERR_INVALID;
    const KParams& k = h->kp;
    if (env_begin < 0 || env_count < 0 || (int64_t)env_begin + env_count > k.B) return SSD_ERR_INVALID;
    if (env_count == 0) return SSD_OK;
    const ssd_state_layout s = state_layout(k, SSD_OBS_INDEX4);
    return launch_expand(h, state_index4 + (size_t)env_begin * s.env_stride, env_count, k.geo.H, k.geo.W, s.row_stride,
                         s.env_stride, out, stream);
}

int64_t ssd_launch_count(const ssd_handle* h) { return h ? h->launches : -1; }

int64_t ssd_debug_oob_count(void) {
#ifdef SSD_BOUNDS_CHECK
    unsigned long long v = 0;
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(&v, g_oob_count, sizeof(v)) != cudaSuccess) return -2;
    return (int64_t)v;
#else
    return -1;
#endif
}

}  // extern "C"
