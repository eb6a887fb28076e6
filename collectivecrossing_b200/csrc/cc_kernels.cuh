// cc_kernels.cuh — sm_100a kernels of the batched CollectiveCrossing step / reset path.
//
// Mapping (DESIGN.md §3): a TILE of LPE lanes (4, 8, 16 or 32) owns one env; a lane owns APL
// agents (agent a = lane_in_tile + slot*LPE).  A warp therefore processes EPW = 32/LPE
// consecutive envs per iteration of a persistent grid-stride loop, and every per-agent array
// ([N][A], env-major) is read / written as one contiguous run of bytes per warp.
//
// The semantics follow the reference function by function (file:line cited at each device
// function; paths relative to /root/reference/src/collectivecrossing/).  oracle/cc_oracle.c is
// the CPU restatement the tests diff this file against.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>
#include <stdint.h>

#include "../../include/ccb200.h"

#ifndef CCB_MIN_BLOCKS_APL2
#define CCB_MIN_BLOCKS_APL2 2   // crews of 33-64 agents (two agents per lane): at most 128 registers, 2 CTAs per SM (3 CTAs at 76 registers measured slower: 1.63 vs 1.49 ms int8, 3.04 vs 2.77 ms float32 per 262 k envs)
#endif
#ifndef CCB_LANES_PREFETCH
#define CCB_LANES_PREFETCH 1   // one env per warp: request the next env's record before stepping the current one
#endif
#ifndef CCB_LANES_PARMOVES
#define CCB_LANES_PARMOVES 1   // one env per warp: resolve the ordered moves in parallel (shared-memory cell maps)
#endif
#ifndef CCB_LANES_UNROLL
#define CCB_LANES_UNROLL 4     // plain-vector loop of the int8 rows of big crews
#endif
#ifndef CCB_MIN_BLOCKS
#define CCB_MIN_BLOCKS 4  // resident CTAs per SM the register allocator must allow (A/B in DESIGN.md §6)
#endif

// Checked build (make CHECKS=1 -> libccb200_checked.so; tests/test_gpu_checked_build.py runs parity cases through it):
// device-side asserts on every data-dependent shared-memory index and on the bulk-copy sizes.  compute-sanitizer is closed
// on this pool (profiles/r2_compute_sanitizer_closed_on_this_pool.txt), so these are the bounds checks of the hot path.
#ifdef CCB_CHECKS
#include <cassert>
#define CCB_CHECK(cond) assert(cond)
#else
#define CCB_CHECK(cond) ((void)0)
#endif

namespace ccb {

constexpr int kPlainUnroll = CCB_LANES_UNROLL;
#ifndef CCB_LANE_IMG_RING
#define CCB_LANE_IMG_RING 2
#endif
constexpr int kMaxImgIter = 9;    // an 8-row chunk of the largest crew (128 agents) is 259 vectors = 9 per lane
constexpr int kLaneImgRing = CCB_LANE_IMG_RING;   // chunk images per warp (int8 rows of big crews)
constexpr int kWarpsPerCta = 8;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kResetAttemptCap = 4096;   // same cap as the oracle

enum Mode { kModeStep = 0, kModeReset = 1, kModePolicy = 2, kModeObserve = 3 };
// OR-ed into the OBS template argument of a step / reset kernel: placements come from the env's numpy generator
// (KParams::gen, cc_set_reset_rng) instead of Philox.  A flag of an existing argument, not a new one, so that the
// Philox instantiations keep their symbols and their code.
constexpr int kNpReset = 0x100;
struct Pcg64State;
enum StatSlot { kStEnvSteps = 0, kStEpisodes, kStTermAll, kStTruncAll, kStArrivals, kStEpLen, kStEpRet, kStRewardSum, kStCount };
enum ErrBit { kErrInvalidAction = 1, kErrResetStuck = 2 };

struct KParams {
    // lowered config (cc_config) + derived
    int W, H, D, TL, TR, DL, DR, DC, YB, YE, B, A;
    int max_steps, reward_kind, terminated_kind;
    double rp[4];
    // shard
    long long n_envs;
    unsigned long long genv_offset, seed;
    unsigned t;
    // persistent state
    int8_t *x, *y;
    uint8_t *flags;
    int32_t *step;
    float *ep_ret;
    // step io
    const int8_t *actions, *order;
    const uint8_t *mask;  // reset mode
    int8_t *actions_out;
    void *obs, *reward;
    uint8_t *agent_flags, *agent_info, *env_flags;
    int policy, auto_reset, reward_f64;
    // bookkeeping
    unsigned long long *stats;  // kStCount 8-byte slots (int64 / double bit patterns)
    int *err;
    // shared-memory layout (bytes from the dynamic smem base)
    int R;               // pairs per observation row = 3 + 2A
    int pairs_per_env;   // A * R
    int lut_entries;     // EPW * A * R
    int stage_pairs;     // 3 + EPW * 2A (per warp)
    int walk_words;      // words of one padded-lattice bitmap: ceil((W+3)(H+3)/32)
    int off_stage, off_bitmap, off_desc;
    float rpf[4];        // reward parameters rounded to float32 once
    unsigned reward_category_mask;  // 0xF for the default reward (category overrides apply), else 0
    long long n_groups;
    int smem_total;
    int tpe_bm_words;    // thread-per-env kernel: words of the private lattice bitmap (0 = compare-based occupancy)
    int tpe_bm_rows;     // ... 1: one word per padded lattice ROW (at most 32 padded columns), else bit index = cell
    unsigned *tpe_counter, *tpe_counter_next;   // thread-per-env kernel: work counters of this / the next launch
    int tpe_reverse;              // step kernels: process the groups from the last to the first (alternates between launches)
    // thread-per-env kernel, fused multi-step launches (cc_rollout_fused): every output is time-major [n_steps][...]
    // lane-group kernel, int8 rows of one-env-per-warp crews (A > 16) whose env block is a whole number of 16-byte
    // vectors: 8 copies of the row template, shifted by 0, 2, ..., 14 bytes, so that most output vectors are ONE
    // aligned 16-byte shared-memory load (shift_tst = 0: not used)
    int shift_tst;                // bytes of one shifted copy (multiple of 16)
    int off_shift;                // [warp][8][shift_tst]
    int off_vlist;                // unsigned plain[nvec_env], unsigned short special[nvec_env], counts[2], starts[2][n_chunks+1], special LUT
    int img_vecs, n_chunks;       // the env block leaves the SM in n_chunks bulk copies of (at most) img_vecs vectors = img_rows rows
    int img_rows;                 // rows per chunk: a multiple of 8 (8 rows are the smallest run of rows that is whole 16-byte vectors)
    int off_img;                  // [warp][kLaneImgRing][img_vecs * 16] image ring
    int max_special;              // rows of the special-vector LUT
    int nvec_env;                 // 16-byte vectors of an env's observation block
    long long obs_env_offset;     // lane-group kernel: the observation rows of env n go to row block n + obs_env_offset of p.obs
    int n_steps;                  // env-steps per env in this launch (1 for cc_step)
    const void *t2_tables;        // small-lattice kernel: its tables, built once per handle (cc_kernel_tpe2.cuh: T2Tables)
    // lane-group kernel, one env per warp (crews above 16): per-warp byte maps of the padded lattice for the parallel
    // resolution of the ordered moves — [own: which ACTIVE agent stands on the cell][win: first contender for the cell]
    // [128 status bytes] (cellmap_cells = bytes of one map, a multiple of 16; 0 = sequential turns only)
    int off_cellmap, cellmap_cells;
    long long slice_agents;       // elements of one time slice of a per-agent array: n_envs * A
    long long slice_envs;         // ... of a per-env array: n_envs
    long long slice_obs_bytes;    // ... of the observation tensor, in bytes
    // numpy-mode placements (cc_set_reset_rng): the per-env generators of envs [first, first + n_envs) of the handle;
    // read by the instantiations that carry kNpReset only.  (Last member: the offsets of the others stay as they were.)
    Pcg64State *gen;
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (counter-based; auto-reset placement and random actions).  Same constants and
// counter layout as oracle/cc_oracle.c:orc_draw.
// ---------------------------------------------------------------------------------------------
struct U4 { unsigned v0, v1, v2, v3; };

__device__ __forceinline__ U4 philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        unsigned h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        unsigned h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        unsigned n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}
enum { kStreamReset = 0, kStreamAction = 1 };
__device__ __forceinline__ U4 draw(const KParams &p, unsigned long long genv, unsigned stream, unsigned idx) {
    return philox4x32_10((unsigned)genv, (unsigned)(genv >> 32), p.t, (stream << 24) | (idx & 0xFFFFFFu),
                         (unsigned)p.seed, (unsigned)(p.seed >> 32));
}
// (same stream at an explicit counter word: step t of a fused multi-step launch draws what launch t would)
__device__ __forceinline__ U4 draw_at(const KParams &p, unsigned t, unsigned long long genv, unsigned stream, unsigned idx) {
    return philox4x32_10((unsigned)genv, (unsigned)(genv >> 32), t, (stream << 24) | (idx & 0xFFFFFFu),
                         (unsigned)p.seed, (unsigned)(p.seed >> 32));
}
__device__ __forceinline__ int bounded(unsigned r, int n) { return (int)__umulhi(r, (unsigned)n); }

// ---------------------------------------------------------------------------------------------
// geometry predicates
// ---------------------------------------------------------------------------------------------
// collectivecrossing.py:509-534 _is_valid_position.  (:565-588 _would_hit_tram_wall rejects a
// subset of what this rejects, so _is_move_valid's geometric part is exactly this test.)
__device__ __forceinline__ bool valid_position(const KParams &p, int x, int y) {
    bool ok = (unsigned)x <= (unsigned)p.W && (unsigned)y <= (unsigned)p.H;
    if (y == p.D) ok = ok && (p.DL < x) && (x < p.DR);
    if (y >= p.D) ok = ok && (p.TL < x) && (x < p.TR);
    return ok;
}
// collectivecrossing.py:551-554 is_in_tram_area (inclusive)
__device__ __forceinline__ bool in_tram_area(const KParams &p, int x, int y) { return y >= p.D && p.TL <= x && x <= p.TR; }
// collectivecrossing.py:556-563 is_at_tram_door
__device__ __forceinline__ bool at_tram_door(const KParams &p, int x, int y) { return y == p.D && (x == p.DL - 1 || x == p.DR + 1); }
// ---------------------------------------------------------------------------------------------
// reset(seed=s), bit-exact with the reference's generator: numpy Generator(PCG64(SeedSequence(s)))
// (gymnasium seeding; collectivecrossing.py:95,105-106,134-137).  One thread per env — the draw
// stream is inherently sequential.  Restated from numpy's bit_generator.pyx (SeedSequence),
// _pcg64 / pcg64.h (seeding, XSL-RR 128/64 output, 32-bit buffering) and distributions.c
// (Lemire bounded uint32), see oracle/cc_oracle.c for the CPU twin.
// ---------------------------------------------------------------------------------------------
struct Pcg64 {
    unsigned long long hi, lo, inc_hi, inc_lo;
    unsigned buffered;
    bool has_buffered;
    __device__ __forceinline__ void advance() {
        const unsigned long long MH = 2549297995355413924ULL, ML = 4865540595714422341ULL;
        unsigned long long nlo = lo * ML;
        unsigned long long nhi = __umul64hi(lo, ML) + hi * ML + lo * MH;
        unsigned long long slo = nlo + inc_lo;
        nhi += inc_hi + (slo < nlo ? 1ULL : 0ULL);
        hi = nhi; lo = slo;
    }
    __device__ __forceinline__ unsigned long long next64() {
        advance();
        unsigned long long v = hi ^ lo;
        unsigned rot = (unsigned)(hi >> 58);
        return (v >> rot) | (v << ((64u - rot) & 63u));
    }
    __device__ __forceinline__ unsigned next32() {
        if (has_buffered) { has_buffered = false; return buffered; }
        unsigned long long n = next64();
        has_buffered = true; buffered = (unsigned)(n >> 32);
        return (unsigned)n;
    }
    __device__ __forceinline__ long long integers(long long low, long long high) {  // [low, high)
        unsigned rng = (unsigned)(high - low) - 1u;
        if (rng == 0u) return low;
        unsigned excl = rng + 1u;
        unsigned long long m = (unsigned long long)next32() * excl;
        unsigned left = (unsigned)m;
        if (left < excl) {
            unsigned thr = (0xFFFFFFFFu - rng) % excl;
            while (left < thr) { m = (unsigned long long)next32() * excl; left = (unsigned)m; }
        }
        return low + (long long)(m >> 32);
    }
    __device__ void seed(unsigned long long s) {
        unsigned ent[2] = {(unsigned)s, (unsigned)(s >> 32)};
        int n_ent = (s >> 32) ? 2 : 1;
        unsigned pool[4], hc = 0x43b0d7e5u;
        auto hashmix = [&](unsigned v) { v ^= hc; hc *= 0x931e8875u; v *= hc; v ^= v >> 16; return v; };
        auto mix = [](unsigned a, unsigned b) { unsigned r = 0xca01f9ddu * a - 0x4973f715u * b; r ^= r >> 16; return r; };
        for (int i = 0; i < 4; ++i) pool[i] = hashmix(i < n_ent ? ent[i] : 0u);
        for (int a = 0; a < 4; ++a)
            for (int b = 0; b < 4; ++b)
                if (a != b) pool[b] = mix(pool[b], hashmix(pool[a]));
        unsigned st[8], hb = 0x8b51f9ddu;
        for (int i = 0; i < 8; ++i) { unsigned v = pool[i & 3]; v ^= hb; hb *= 0x58f38dedu; v *= hb; v ^= v >> 16; st[i] = v; }
        unsigned long long w0 = st[0] | ((unsigned long long)st[1] << 32), w1 = st[2] | ((unsigned long long)st[3] << 32);
        unsigned long long w2 = st[4] | ((unsigned long long)st[5] << 32), w3 = st[6] | ((unsigned long long)st[7] << 32);
        // pcg_setseq_128_srandom_r(initstate = w0:w1, initseq = w2:w3)
        inc_hi = (w2 << 1) | (w3 >> 63); inc_lo = (w3 << 1) | 1ULL;
        hi = 0; lo = 0;
        advance();
        unsigned long long slo = lo + w1;
        hi += w0 + (slo < lo ? 1ULL : 0ULL); lo = slo;
        advance();
        has_buffered = false; buffered = 0;
    }
};

// persistent generator of one env (what gymnasium keeps in env.np_random): 6 x 8 bytes
struct Pcg64State { unsigned long long hi, lo, inc_hi, inc_lo, buffered, has_buffered; };


__device__ __forceinline__ Pcg64 np_load(const Pcg64State &st) {
    Pcg64 g;
    g.hi = st.hi; g.lo = st.lo; g.inc_hi = st.inc_hi; g.inc_lo = st.inc_lo;
    g.buffered = (unsigned)st.buffered; g.has_buffered = st.has_buffered != 0;
    return g;
}
__device__ __forceinline__ Pcg64State np_save(const Pcg64 &g) {
    return Pcg64State{g.hi, g.lo, g.inc_hi, g.inc_lo, (unsigned long long)g.buffered, g.has_buffered ? 1ull : 0ull};
}

// One candidate of reset()'s rejection loop from the env's numpy generator: integers(0, W), integers(0, D) for a
// boarding agent (collectivecrossing.py:103-117), integers(TL, TR + 1), integers(D, H) for an exiting one (:132-140).
// Returns the geometric test; the occupancy test against the agents already placed is the caller's.
__device__ __forceinline__ bool np_candidate(Pcg64 &g, const KParams &p, bool boarding, int &px, int &py) {
    if (boarding) {
        px = (int)g.integers(0, p.W); py = (int)g.integers(0, p.D);
        return valid_position(p, px, py) && !(p.DL <= px && px <= p.DR && py == p.D - 1);
    }
    px = (int)g.integers(p.TL, p.TR + 1); py = (int)g.integers(p.D, p.H);
    return valid_position(p, px, py);
}
// reset()'s placement of one agent with the numpy generator: candidates until one passes the geometric test and
// free(x, y) (no agent j < i stands there).  At kResetAttemptCap attempts the last candidate is kept and false returned.
// cc_reset_seeded_kernel and the thread-per-env step kernels place every agent through this; the lane-group kernel
// draws through np_candidate with the same attempt count (its occupancy test is a ballot); tests/native/cc_oracle_np.c restates it.
template <typename Free>
__device__ __forceinline__ bool np_place_agent(Pcg64 &g, const KParams &p, bool boarding, Free free, int &px, int &py) {
    bool ok = false;
    for (int attempt = 0; attempt < kResetAttemptCap && !ok; ++attempt) ok = np_candidate(g, p, boarding, px, py) && free(px, py);
    return ok;
}

// actions.py:18-24 ACTION_TO_DIRECTION
__device__ __forceinline__ int act_dx(int a) { return (a == CC_ACT_RIGHT) - (a == CC_ACT_LEFT); }
__device__ __forceinline__ int act_dy(int a) { return (a == CC_ACT_UP) - (a == CC_ACT_DOWN); }

__device__ __forceinline__ unsigned pack_pos(int x, int y) { return ((unsigned)(x & 0xff) << 8) | (unsigned)(y & 0xff); }
__device__ __forceinline__ int pos_x(unsigned q) { return (int)(int8_t)(q >> 8); }
__device__ __forceinline__ int pos_y(unsigned q) { return (int)(int8_t)(q & 0xff); }

// the geometric half of collectivecrossing.py:378-408 _move_agent: bit31 = "wants to move and the
// target passes _is_valid_position", low 16 bits = packed target
__device__ __forceinline__ unsigned move_request(const KParams &p, unsigned pos, int action, bool active) {
    int nx = pos_x(pos) + act_dx(action), ny = pos_y(pos) + act_dy(action);
    bool go = active && (unsigned)action < 4u && valid_position(p, nx, ny);
    return (go ? 0x80000000u : 0u) | pack_pos(nx, ny);
}

template <int APL>
__device__ __forceinline__ unsigned pick(const unsigned (&v)[APL], int slot) {
    unsigned r = v[0];
#pragma unroll
    for (int k = 1; k < APL; ++k) r = (slot == k) ? v[k] : r;
    return r;
}
template <int APL>
__device__ __forceinline__ int picki(const int (&v)[APL], int slot) {
    int r = v[0];
#pragma unroll
    for (int k = 1; k < APL; ++k) r = (slot == k) ? v[k] : r;
    return r;
}

template <typename T> struct PairOf;
template <> struct PairOf<float> { using type = float2; };
template <> struct PairOf<int8_t> { using type = char2; };
template <typename T> __device__ __forceinline__ typename PairOf<T>::type mk_pair(int a, int b);
template <> __device__ __forceinline__ float2 mk_pair<float>(int a, int b) { return make_float2((float)a, (float)b); }
template <> __device__ __forceinline__ char2 mk_pair<int8_t>(int a, int b) { return make_char2((signed char)a, (signed char)b); }

// ---------------------------------------------------------------------------------------------
// per-warp context
// ---------------------------------------------------------------------------------------------
template <int LPE, int APL>
struct Tile {
    static constexpr int EPW = 32 / LPE;
    static constexpr unsigned MASK = (LPE == 32) ? 0xffffffffu : ((1u << (LPE & 31)) - 1u);
    static constexpr int LOG = (LPE == 4) ? 2 : (LPE == 8) ? 3 : (LPE == 16) ? 4 : 5;
    int lane, li, tile, tshift;
    __device__ __forceinline__ Tile() {
        lane = threadIdx.x & 31;
        li = lane & (LPE - 1);
        tile = lane >> LOG;
        tshift = tile * LPE;
    }
    __device__ __forceinline__ unsigned tballot(bool pred) const { return (__ballot_sync(kFull, pred) >> tshift) & MASK; }
    __device__ __forceinline__ unsigned tshfl(unsigned v, int src_in_tile) const { return __shfl_sync(kFull, v, src_in_tile, LPE); }
};

// ---------------------------------------------------------------------------------------------
// Observation expansion.
// Row i of an env is  [P_i, K1, K2, S_0a, S_0b, S_1a, S_1b, ...] with S_ia,S_ib replaced by M
// (observations.py:62-94), in PAIR units: P_i=(x_i,y_i) K1=(DC,D) K2=(DL,DR) S_ja=(x_j,y_j)
// S_jb=(type_j,active_j) M=(-1,-1).  A warp stages one row TEMPLATE per env in shared memory,
//      T_e = [unused, K1, K2, S_0a, S_0b, ..., S_(A-1)b, M]          (2A+4 pairs)
// so output pair q of any row reads T_e[q] — consecutive output pairs read consecutive addresses, which
// keeps the gather free of bank conflicts — except q = 0 (reads S_ia = T_e[3+2i]) and the own block
// (reads M = T_e[2A+3]).  gather_index() is loop-invariant: it is evaluated once per kernel into
// per-lane descriptors when the chunk is small (A <= 13), else into a shared-memory LUT.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int gather_index(const KParams &p, int P) {
    const int A = p.A, R = p.R, ppe = p.pairs_per_env;
    int tile = P / ppe, q0 = P - tile * ppe;
    int i = q0 / R, q = q0 - i * R;
    int base = tile * (2 * A + 4);
    if (q == 0) return base + 3 + 2 * i;
    if (q >= 3 && ((q - 3) >> 1) == i) return base + 2 * A + 3;
    return base + q;
}

// generic path: `count` pairs starting at global pair index gp0, 16-byte vectors wherever a whole
// vector lies inside the range (everywhere except the ends of an unaligned / odd-sized chunk)
template <typename T>
__device__ __forceinline__ void emit_obs_lut(T *obs, long long gp0, int count, const uint16_t *lut,
                                             const typename PairOf<T>::type *stage, int lane) {
    using P2 = typename PairOf<T>::type;
    constexpr int PPV = 16 / (int)sizeof(P2);  // pairs per 16-byte vector: 2 (fp32) or 8 (int8)
    const long long v_first = gp0 / PPV;
    const int head = (int)(gp0 - v_first * PPV);            // pairs of the first vector before the chunk
    const int nvec = (head + count + PPV - 1) / PPV;
    P2 *out = reinterpret_cast<P2 *>(obs) + v_first * PPV;  // vector-aligned base
    for (int v = lane; v < nvec; v += 32) {
        const int p0 = v * PPV - head;
        if (p0 >= 0 && p0 + PPV <= count) {
            union { uint4 u; P2 e[PPV]; } pk;
#pragma unroll
            for (int e = 0; e < PPV; ++e) pk.e[e] = stage[lut[p0 + e]];
            __stcs(reinterpret_cast<uint4 *>(out) + v, pk.u);
        } else {
#pragma unroll
            for (int e = 0; e < PPV; ++e)
                if (p0 + e >= 0 && p0 + e < count) out[v * PPV + e] = stage[lut[p0 + e]];
        }
    }
}

constexpr int kDescWords = 24;                 // cached gather descriptors per lane (one per output pair)
constexpr int kDescPairs = 32 * kDescWords;    // = 768 output pairs per warp chunk
constexpr int kRtabSize = 400;                 // reward-table index = |x-DC| (<= 128) + biased y distance (< 256)
constexpr int kYBias = 128;
constexpr int kMaxGeom = 120;                  // largest width / height the tables are sized for (reference: 100)
constexpr int kMaxPad = kMaxGeom + 4;          // padded lattice side
constexpr int kMaxWalkWords = 512;             // >= ceil(kMaxPad^2 / 32) = 481; a power of two so garbage indices can be masked
constexpr int kNumYClass = 5;                  // far / door level / beyond: up, down, at destination
constexpr int kPolicyRows = 2 * kNumYClass * 3;  // (type, y class, x class)

// Geometry tables (per CTA, built once).  A word has its additive fields in the low bits and its
// predicate flags in the top byte, so for an agent at (x, y) of type t
//      u = yt[t][y] + xt[x]   ->  bits 0-7  row of act_tab (greedy decision),  bits 8-16 reward-table index
//      f = (yt & xt) >> 24    ->  bit0 in_tram_area, bit1 at_tram_door, bit3 at destination  (= CC_I_* bits)
__device__ __forceinline__ unsigned make_xt(const KParams &p, int x) {
    const unsigned tramx = p.TL <= x && x <= p.TR, adj = (x == p.DL - 1 || x == p.DR + 1);
    const unsigned xcmp = x < p.DC ? 0u : (x == p.DC ? 1u : 2u);
    const unsigned xdist = p.reward_kind == CC_REWARD_DEFAULT ? (unsigned)abs(x - p.DC) : 0u;  // rewards.py:82-84,95-98
    return xcmp | (xdist << 8) | ((tramx | (adj << 1) | 8u) << 24);
}
__device__ __forceinline__ unsigned make_yt(const KParams &p, int type, int y) {
    const int dest = type == 0 ? p.YB : p.YE;
    const unsigned ytram = y >= p.D, isd = y == p.D, arrived = y == dest;
    // y class of the greedy policy (greedy_policy.py:117-158)
    unsigned cls;
    if (type == 0) cls = y < p.D - 1 ? 0u : (y == p.D - 1 ? 1u : (y < dest ? 2u : (y > dest ? 3u : 4u)));
    else           cls = y > p.D + 1 ? 0u : (y == p.D + 1 ? 1u : (y < dest ? 2u : (y > dest ? 3u : 4u)));
    int ydist;
    if (p.reward_kind == CC_REWARD_DEFAULT) ydist = type == 0 ? p.D - y : y - p.D;   // rewards.py:83,97
    else ydist = abs(y - dest);                                                        // utils/geometry.py:54-55
    ydist = min(max(ydist + kYBias, 0), 255);
    return ((unsigned)(type * kNumYClass + (int)cls) * 3u) | ((unsigned)ydist << 8) | ((ytram | (isd << 1) | (arrived << 3)) << 24);
}
// greedy decision for (type, y class, x class) and the 4-bit mask of valid moves (bit a = action a valid):
// baseline_policies/greedy_policy.py:64-88 (preferred move if valid) and :277-449 (fallback lists)
__device__ __forceinline__ int greedy_decision(int row, unsigned vmask) {
    const int type = row / (kNumYClass * 3), cls = (row / 3) % kNumYClass, xc = row % 3;
    const int vert = type == 0 ? CC_ACT_UP : CC_ACT_DOWN, toward = xc == 0 ? CC_ACT_RIGHT : CC_ACT_LEFT;
    int want;
    unsigned pref;  // 4 nibbles, first choice lowest
    if (cls <= 1) {
        want = (cls == 1 && xc != 1) ? toward : vert;
        if (type == 0) pref = xc == 0 ? 0x3210u : (xc == 2 ? 0x3012u : 0x3201u);   // RULD | LURD | URLD
        else           pref = xc == 0 ? 0x1230u : (xc == 2 ? 0x1032u : 0x1203u);   // RDLU | LDRU | DRLU
    } else {
        want = cls == 2 ? CC_ACT_UP : (cls == 3 ? CC_ACT_DOWN : CC_ACT_WAIT);       // sign(dest - y), :178-182
        pref = type == 0 ? 0x3201u : 0x1203u;
    }
    if (want == CC_ACT_WAIT || ((vmask >> want) & 1u)) return want;
    for (int c = 0; c < 4; ++c) { const int cand = (pref >> (4 * c)) & 15; if ((vmask >> cand) & 1u) return cand; }
    return CC_ACT_WAIT;
}

// ---------------------------------------------------------------------------------------------
// the fused kernel
// ---------------------------------------------------------------------------------------------
// OBSF: the obs dtype, with kNpReset for numpy-mode placements (step and reset modes)
template <int LPE, int APL, int OBSF, int MODE>
// (two agents per lane: the float32-row instantiation keeps its registers — 122, measured 8 % faster than capped at 128 / 2 CTAs)
__global__ void __launch_bounds__(kThreads, (MODE != kModeStep) ? 1 : (APL == 1 ? CCB_MIN_BLOCKS : (APL == 2 ? ((OBSF & ~kNpReset) == CC_OBS_FP32 ? 1 : CCB_MIN_BLOCKS_APL2) : 1))) cc_kernel(const __grid_constant__ KParams p) {
    constexpr int OBS = OBSF & ~kNpReset;
    constexpr bool kNp = (OBSF & kNpReset) != 0;
    using TL_ = Tile<LPE, APL>;
    using OT = typename std::conditional<OBS == CC_OBS_FP32, float, int8_t>::type;
    using P2 = typename PairOf<OT>::type;
    constexpr int EPW = TL_::EPW;
    constexpr int PPV = 16 / (int)sizeof(P2);  // output pairs per 16-byte vector: 2 (fp32) or 8 (int8)
    constexpr bool kHasObs = OBS == CC_OBS_INT8 || OBS == CC_OBS_FP32;   // the reference's rows
    constexpr bool kTable = OBS == CC_OBS_TABLE;                            // the compact [A][4] table
    constexpr bool kCanCache = kHasObs && LPE <= 16;
    constexpr bool kHasPolicy = MODE == kModeStep || MODE == kModePolicy;
    constexpr bool kMoves = MODE == kModeStep;
    extern __shared__ __align__(16) unsigned char smem[];

    const TL_ T;
    const int warp = threadIdx.x >> 5;
    const int A = p.A;
    const int PW = p.W + 3, PH = p.H + 3;  // lattice padded by one ring: x in [-1, W+1] -> column x+1
    // fixed-size tables live in STATIC shared memory: their addresses are immediates, nothing has to
    // be kept in (or rematerialised into) registers to reach them
    __shared__ unsigned xt[kMaxPad], yt[2 * kMaxPad], walk[kMaxWalkWords];
    __shared__ float rtab[2 * kRtabSize];
    __shared__ uint8_t act_tab[kPolicyRows * 16];
    __shared__ unsigned long long red_all[kWarpsPerCta * kStCount];
    uint16_t *lut = reinterpret_cast<uint16_t *>(smem);
    P2 *stage = reinterpret_cast<P2 *>(smem + p.off_stage) + warp * p.stage_pairs;
    unsigned *blocked = reinterpret_cast<unsigned *>(smem + p.off_bitmap) + (warp * EPW + T.tile) * p.walk_words;

    // ---- once per CTA: gather descriptors / LUT, geometry tables -----------------------------------
    const int chunk_pairs = EPW * p.pairs_per_env;
    constexpr bool kPairwise = false;             // (8-byte pair-wise stores measured slower than 16-byte vectors: 0.308 vs 0.276 ms)
    const bool cached = kCanCache && chunk_pairs <= kDescPairs && (kPairwise || ((chunk_pairs % PPV) == 0 && (p.obs_env_offset * p.pairs_per_env) % PPV == 0));
    uint4 *desc_sm = reinterpret_cast<uint4 *>(smem + p.off_desc) + threadIdx.x;  // [kDescWords/4][kThreads], conflict-free
    if (kHasObs) {
        if (cached) {
            // descriptor = byte offset (from the dynamic shared-memory base) of the template pair that
            // feeds one output pair.  fp32: word w serves output pair lane + 32 w (stored pair-wise);
            // int8: word w serves pair w % 8 of the lane's 16-byte vector number w / 8.
            const unsigned stage_off = (unsigned)(reinterpret_cast<unsigned char *>(stage) - smem);
#pragma unroll
            for (int q = 0; q < kDescWords / 4; ++q) {
                unsigned d[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int w = q * 4 + c;
                    const int P = kPairwise ? T.lane + 32 * w : (T.lane + 32 * (w / PPV)) * PPV + (w % PPV);
                    d[c] = stage_off + (unsigned)sizeof(P2) * (unsigned)(P < chunk_pairs ? gather_index(p, P) : 0);
                }
                desc_sm[q * kThreads] = make_uint4(d[0], d[1], d[2], d[3]);
            }
        } else {
            for (int P = threadIdx.x; P < p.lut_entries; P += blockDim.x) lut[P] = (uint16_t)gather_index(p, P);   // (no entries with shifted rows)
        }
        for (int e = T.lane; e < EPW; e += 32) {   // the constant pairs of every env template of this warp
            P2 *t = stage + e * (2 * A + 4);
            t[0] = mk_pair<OT>(0, 0); t[1] = mk_pair<OT>(p.DC, p.D); t[2] = mk_pair<OT>(p.DL, p.DR); t[2 * A + 3] = mk_pair<OT>(-1, -1);
        }
    }
    // int8 rows of big crews (one env per warp).  Row i of an env is the row template [P K1 K2 S_0a ... S_(A-1)b] with pair 0
    // replaced by S_ia and the own block by M; a row is 6 + 4A = 2 x odd bytes, so rows start at every even alignment.  The warp
    // keeps 8 copies of the template, copy c shifted by 2c bytes, each followed by the first 16 bytes of the template again:
    // ANY 16-byte vector of the output — also one that straddles two rows — is then 16 consecutive bytes of the copy whose
    // shift matches, i.e. ONE aligned 16-byte load, up to the bytes that differ from row to row (pair 0 and the own block),
    // which are patched in the assembled image.  img_src[j] = offset of the source of vector j of an 8-row chunk.
    constexpr bool kShiftable = kHasObs && OBS == CC_OBS_INT8 && LPE == 32 && MODE != kModeReset;
    unsigned char *shifted = smem + p.off_shift + warp * 8 * p.shift_tst;
    const bool shift_rows = kShiftable && p.shift_tst > 0;
    const int lrow = 6 + 4 * A;
    unsigned *img_src = reinterpret_cast<unsigned *>(smem + p.off_vlist);   // [vector of a chunk]: where its 16 bytes lie in the shifted copies
    if (shift_rows) {
        for (int j = threadIdx.x; j < p.img_vecs; j += blockDim.x) {
            const int b0 = 16 * j, r0 = b0 % lrow, c = ((16 - (r0 & 15)) >> 1) & 7;   // copy whose shift aligns template byte r0
            img_src[j] = (unsigned)(c * p.shift_tst + 2 * c + r0);
        }
        // constant head of every copy and of its 16-byte tail: template bytes 2..5 = K1, K2 (bytes 0..1, pair 0, are patched)
        if (T.lane < 8) {
            unsigned char *t = shifted + T.lane * p.shift_tst + 2 * T.lane;
            t[2] = t[lrow + 2] = (unsigned char)p.DC; t[3] = t[lrow + 3] = (unsigned char)p.D;
            t[4] = t[lrow + 4] = (unsigned char)p.DL; t[5] = t[lrow + 5] = (unsigned char)p.DR;
        }
    }
    for (int i = threadIdx.x; i < PW; i += blockDim.x) xt[i] = make_xt(p, i - 1);
    for (int i = threadIdx.x; i < 2 * PH; i += blockDim.x) yt[(i / PH) * kMaxPad + i % PH] = make_yt(p, i / PH, i % PH - 1);
    if (kHasPolicy)
        for (int i = threadIdx.x; i < kPolicyRows * 16; i += blockDim.x) act_tab[i] = (uint8_t)greedy_decision(i >> 4, (unsigned)i & 15u);
    // distance rewards: entry k holds float((double)(-d) * f) (boarding / simple distance) or
    // float((double)d * f) (exiting, default reward) for d = k - kYBias: the reference's float64 product
    // (rewards.py:85,99,127) rounded once — no FP64 in the loop
    if (kMoves) {
        const double f = p.reward_kind == CC_REWARD_DEFAULT ? p.rp[3] : p.rp[0];
        for (int i = threadIdx.x; i < 2 * kRtabSize; i += blockDim.x) {
            const int type = i / kRtabSize, d = i % kRtabSize - kYBias;
            const bool negate = type == 0 || p.reward_kind == CC_REWARD_SIMPLE_DISTANCE;
            float v = (float)((double)(negate ? -d : d) * f);
            if (p.reward_kind == CC_REWARD_BINARY) v = p.rpf[1];                  // rewards.py:152-159 (never goal_reward)
            if (p.reward_kind == CC_REWARD_CONSTANT_NEGATIVE) v = p.rpf[0];       // rewards.py:179-182
            rtab[i] = v;
        }
    }
    // static map of walkable lattice points (collectivecrossing.py:509-534), one bit per point of
    // the padded lattice; the padding ring is not walkable, so neighbour tests need no bounds check
    for (int w = threadIdx.x; w < p.walk_words; w += blockDim.x) {
        unsigned bits = 0;
        for (int b = 0; b < 32; ++b) {
            const int idx = w * 32 + b, yy = idx / PW - 1, xx = idx - (yy + 1) * PW - 1;
            bits |= valid_position(p, xx, yy) ? (1u << b) : 0u;
        }
        walk[w] = bits;
    }
    if (kMoves && LPE == 32 && p.cellmap_cells > 0)   // empty maps: no agent (0xFF) on any cell
        for (int i = threadIdx.x; i < kWarpsPerCta * (2 * p.cellmap_cells + 128) / 4; i += blockDim.x)
            reinterpret_cast<unsigned *>(smem + p.off_cellmap)[i] = 0xFFFFFFFFu;
    // statistics: arrivals and the reward sum change every step and stay in registers; the
    // episode-end sums are updated on the (rare) step an episode ends, in the warp's smem slot
    unsigned long long *red = red_all + warp * kStCount;
    if (kMoves && T.lane < kStCount) red[T.lane] = 0ull;
    __syncthreads();
    unsigned st_arrivals = 0;
    double st_rsum = 0.0;
    int errbits = 0;
    int img_slot = 0;   // next image of the warp's ring (int8 rows of big crews)
    unsigned long long l2_evict_first = 0;   // (the rows are written once and not read by this kernel)
    if (kHasObs && OBS == CC_OBS_INT8 && LPE == 32) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_evict_first));

    // ---- per-lane constants ---------------------------------------------------------------------------
    int aidx[APL], aload[APL], ytoff[APL], rtoff[APL];
    bool avalid[APL];
#pragma unroll
    for (int k = 0; k < APL; ++k) {
        aidx[k] = T.li + k * LPE;
        avalid[k] = aidx[k] < A;
        aload[k] = T.tile * A + min(aidx[k], A - 1);   // lanes beyond A re-read agent A-1 (never stored)
        ytoff[k] = aidx[k] < p.B ? 0 : kMaxPad;         // row of yt for this agent's type
        rtoff[k] = aidx[k] < p.B ? 0 : kRtabSize;       // half of rtab for this agent's type
    }
    const unsigned tile_bits = TL_::MASK << T.tshift;
    const int group_stride = EPW * A;

    const int total_warps = (int)gridDim.x * kWarpsPerCta;
    const int n_groups = (int)p.n_groups;
    // (Fetching the record of group g + total_warps while group g is processed was measured: no gain.)
    struct Record { unsigned x[APL], y[APL], fl[APL]; int act[APL]; int step; float ep_ret; };
    auto fetch = [&](int gg, Record &r) {
        const long long m0 = (long long)gg * EPW;
        const bool ok = T.tile < (int)min((long long)EPW, p.n_envs - m0);   // false only in the ragged last group
        const int tl = ok ? T.tile : 0;                                       // tiles beyond the end re-read env 0 of the group
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            const int o = gg * group_stride + (ok ? aload[k] : aload[k] - T.tile * A);
            r.x[k] = (unsigned)(uint8_t)p.x[o];
            r.y[k] = (unsigned)(uint8_t)p.y[o];
            r.fl[k] = p.flags[o];
            r.act[k] = CC_ACT_WAIT;
            if (kMoves && p.policy == CC_POLICY_EXTERNAL) r.act[k] = p.actions[o];
        }
        r.step = p.step[(int)m0 + tl];
        r.ep_ret = kMoves ? p.ep_ret[(int)m0 + tl] : 0.f;
    };
    // (step launches alternate the direction: a launch starts on the groups the previous one wrote last, whose state is
    // still in L2)
    auto group_of = [&](int w) { return (MODE == kModeStep && p.tpe_reverse) ? n_groups - 1 - w : w; };
    // one env per warp (crews above 16): the record of the warp's NEXT env is requested before the current one is
    // stepped — a warp works ~25k cycles on an env, and 13 % of its stall samples were this load (profiles/r2_ncu_summary.txt)
    // (not with float32 rows: that mode is at the HBM roofline and measured 8 % slower with either change — the rows leave
    // through st.global there, and warps that reach the row phase sooner only collide in the load/store pipe)
    constexpr bool kPrefetch = CCB_LANES_PREFETCH && LPE == 32 && MODE == kModeStep && OBS != CC_OBS_FP32;
    Record ahead;
    {
        const int gw0 = (int)blockIdx.x * kWarpsPerCta + warp;
        if (kPrefetch && gw0 < n_groups) fetch(group_of(gw0), ahead);
    }
    for (int gw = (int)blockIdx.x * kWarpsPerCta + warp; gw < n_groups; gw += total_warps) {
        const int g = group_of(gw);
        Record next;
        if (kPrefetch) {
            next = ahead;
            if (gw + total_warps < n_groups) fetch(group_of(gw + total_warps), ahead);
        } else fetch(g, next);
        const long long n0 = (long long)g * EPW;
        const int envs_here = (int)min((long long)EPW, p.n_envs - n0);
        const bool env_ok = T.tile < envs_here;           // false only in the ragged last group
        const int row0 = g * group_stride;                // first agent slot of the group (N*A < 2^31, checked by the host)
        const unsigned long long genv = p.genv_offset + (unsigned long long)(n0 + T.tile);
        int off[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) off[k] = row0 + (env_ok ? aload[k] : aload[k] - T.tile * A);

        // ---- the env's record (one contiguous run of bytes per array per warp) ------------------------
        unsigned pos[APL];   // x << 8 | y (both 0..126 for every reachable state)
        unsigned fl[APL];
        int action[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            pos[k] = (next.x[k] << 8) | next.y[k];
            fl[k] = (env_ok && avalid[k]) ? next.fl[k] : 0u;
            action[k] = next.act[k];
        }
        int step = next.step;
        float ep_ret = next.ep_ret;

        // table coordinates (clamped: set_state promises in-lattice positions; the clamp only keeps
        // shared-memory reads in bounds for garbage) and the padded-lattice cell of every owned agent
        int cell[APL];
        unsigned geo_u[APL], geo_f[APL];
        auto lookup = [&](int k) {
            const int cx = min((int)(pos[k] >> 8), p.W + 1) + 1, cy = min((int)(pos[k] & 0xffu), p.H + 1) + 1;
            CCB_CHECK(cx >= 0 && cx < kMaxPad && cy >= 0 && ytoff[k] + cy < 2 * kMaxPad);
            const unsigned xv = xt[cx], yv = yt[ytoff[k] + cy];
            cell[k] = cy * PW + cx;
            geo_u[k] = yv + xv;
            geo_f[k] = (yv & xv) >> 24;
        };

        // ---- on-device policies (baseline_policies/*.py at randomness_factor 0) ---------------
        bool geo_known = false;  // chosen moves already passed the geometric test
        if (kHasPolicy && p.policy != CC_POLICY_EXTERNAL) {
            if (p.policy == CC_POLICY_RANDOM) {
#pragma unroll
                for (int k = 0; k < APL; ++k) {
                    action[k] = bounded(draw(p, genv, kStreamAction, (unsigned)aidx[k]).v0, 5);
                    lookup(k);
                }
            } else {
                // blocked = walls | cells held by ACTIVE agents (collectivecrossing.py:345-369 as
                // one bit test; the asking agent's own cell is never one of its neighbour cells)
                for (int w = T.li; w < p.walk_words; w += LPE) blocked[w] = ~walk[w];
                __syncwarp();
                bool pending = false;
#pragma unroll
                for (int k = 0; k < APL; ++k) {
                    lookup(k);
                    CCB_CHECK(cell[k] >= PW && cell[k] + PW < p.walk_words * 32);   // the four neighbours lie inside the padded lattice
                    if (fl[k] & CC_F_ACTIVE) atomicOr(&blocked[cell[k] >> 5], 1u << (cell[k] & 31));
                    // waiting_policy.py:118-131: some exiting agent that is not done has not arrived
                    pending |= avalid[k] && aidx[k] >= p.B && (fl[k] & 6u) == 0u && env_ok && !(geo_f[k] & 8u);
                }
                __syncwarp();
                const bool exiting_pending = p.policy == CC_POLICY_WAITING && (__ballot_sync(kFull, pending) & tile_bits) != 0u;
#pragma unroll
                for (int k = 0; k < APL; ++k) {
                    // validity of the four moves (greedy_policy.py:238-264 -> _is_move_valid)
                    const int c = cell[k];
                    auto is_free = [&](int idx) { return ((blocked[idx >> 5] >> (idx & 31)) & 1u) ^ 1u; };
                    const unsigned vmask = is_free(c + 1) | (is_free(c + PW) << 1) | (is_free(c - 1) << 2) | (is_free(c - PW) << 3);
                    CCB_CHECK((((geo_u[k] & 0xffu) << 4) | vmask) < kPolicyRows * 16);
                    const int a = act_tab[((geo_u[k] & 0xffu) << 4) | vmask];
                    const bool asks = (fl[k] & 7u) == CC_F_ACTIVE;                         // active, not done
                    const bool waits = exiting_pending && aidx[k] < p.B && !(geo_f[k] & 1u);  // waiting_policy.py:74-108
                    action[k] = (asks && !waits) ? a : CC_ACT_WAIT;
                }
                geo_known = true;
                __syncwarp();
            }
        } else if (kHasPolicy) {
#pragma unroll
            for (int k = 0; k < APL; ++k) lookup(k);
        }
        if (MODE == kModePolicy) {
#pragma unroll
            for (int k = 0; k < APL; ++k)
                if (env_ok && avalid[k]) __stcs(reinterpret_cast<signed char *>(p.actions_out) + off[k], (signed char)action[k]);
            continue;
        }

        bool need_reset = false;
        unsigned eflags = 0;
        if (kMoves) {
            if (p.actions_out) {
#pragma unroll
                for (int k = 0; k < APL; ++k)
                    if (env_ok && avalid[k]) __stcs(reinterpret_cast<signed char *>(p.actions_out) + off[k], (signed char)action[k]);
            }
            // ---- collectivecrossing.py:188 ---------------------------------------------------
            step += 1;
            unsigned alive_prev[APL];  // 1 iff neither terminated nor truncated at step start
#pragma unroll
            for (int k = 0; k < APL; ++k) alive_prev[k] = (avalid[k] && (fl[k] & 6u) == 0u) ? 1u : 0u;

            // ---- collectivecrossing.py:197-202: ordered moves -------------------------------
            // cmp[k] = packed position of an ACTIVE agent, else a sentinel no target can equal;
            // a request is the packed target cell, or kNoMove.  A mover's target never equals its
            // own cell, so the occupancy ballot (:536-541) needs no self-exclusion.
            // A request that must not move is the owner's own cmp value: the owner (or every ghost) hits it
            // in the ballot, so it can never be committed and needs no separate test.
            constexpr unsigned kGhost = 0xFFFFFFFFu;
            unsigned cmp[APL];
#pragma unroll
            for (int k = 0; k < APL; ++k) cmp[k] = (fl[k] & CC_F_ACTIVE) ? pos[k] : kGhost;
            auto make_request = [&](int my_cell, int my_act, unsigned my_cmp) -> unsigned {
                // packed (dx << 8 | dy) mod 2^16 of actions 0..3 (actions.py:18-24)
                const unsigned delta = (unsigned)((0xFFFFFF0000010100ull >> (16 * (my_act & 3))) & 0xffffull);
                bool go = my_cmp != kGhost && (unsigned)my_act < 4u;                    // :398, wait
                if (!geo_known) {                                                       // :509-534 via the static map
                    const int t = my_cell + ((my_act & 1) ? PW : 1) * ((my_act & 2) ? -1 : 1);
                    go = go && ((walk[(t >> 5) & 0x1ff] >> (t & 31)) & 1u);  // (mask: garbage positions stay inside the table)
                }
                return go ? ((my_cmp + delta) & 0xffffu) : my_cmp;
            };
            if (p.order == nullptr) {
                // every agent has an entry: :707-711 applies to all of them
                unsigned req[APL];
#pragma unroll
                for (int k = 0; k < APL; ++k) {
                    if (env_ok && avalid[k] && (unsigned)action[k] > 4u) errbits |= kErrInvalidAction;
                    req[k] = make_request(cell[k], action[k], cmp[k]);
                }
                auto turn = [&](const int s, const int l) {
                    const unsigned rq = T.tshfl(req[s], l);
                    bool hit = false;
#pragma unroll
                    for (int k = 0; k < APL; ++k) hit |= cmp[k] == rq;
                    const unsigned occ = __ballot_sync(kFull, hit) & tile_bits;
                    if (T.li == l && !occ) cmp[s] = rq;                                     // :406-408
                };
                // ---- one env per warp: the ordered turns resolved in PARALLEL --------------------------------------
                // The reference moves agent 0, 1, 2, ... (collectivecrossing.py:197-202); agent i's move succeeds iff its
                // target is free AT ITS TURN.  With every agent moving at most once that is decidable without the loop:
                //   * a target that held an ACTIVE agent j at step start is free at turn i iff j < i and j's own move succeeded
                //     (j > i has not moved yet; a j that does not move never leaves);
                //   * among the agents that ask for one cell and are not ruled out by that, the FIRST in agent order enters,
                //     all later ones find it taken.
                // `own[cell]` (who stands there), `win[cell]` (first contender) and a status byte per agent live in shared
                // memory; dependencies point to smaller agent indices only, so the chains end and are followed in rounds.
                // Stacked ACTIVE agents (only injectable states) fall back to the sequential turns below.
                bool sequential = true;
                if constexpr (LPE == 32) {
                    if (CCB_LANES_PARMOVES && OBS != CC_OBS_FP32 && p.cellmap_cells > 0) {
                        unsigned char *own = smem + p.off_cellmap + warp * (2 * p.cellmap_cells + 128);
                        unsigned char *win = own + p.cellmap_cells, *stat = win + p.cellmap_cells;
                        enum { kFail = 0, kOk = 1, kUnknown = 2 };
                        int tcell[APL];
                        bool mover[APL], active[APL];
#pragma unroll
                        for (int k = 0; k < APL; ++k) {
                            active[k] = cmp[k] != kGhost;
                            mover[k] = req[k] != cmp[k];                                    // a request that passed the geometric test
                            tcell[k] = cell[k] + ((action[k] & 1) ? PW : 1) * ((action[k] & 2) ? -1 : 1);
                            CCB_CHECK(!active[k] || cell[k] < p.cellmap_cells);
                            CCB_CHECK(!mover[k] || (tcell[k] >= 0 && tcell[k] < p.cellmap_cells));
                            if (active[k]) own[cell[k]] = (unsigned char)aidx[k];
                            stat[aidx[k]] = mover[k] ? kUnknown : kFail;
                        }
                        __syncwarp();
                        bool stacked = false;
#pragma unroll
                        for (int k = 0; k < APL; ++k) stacked |= active[k] && own[cell[k]] != (unsigned char)aidx[k];
                        if (!__any_sync(kFull, stacked)) {
                            sequential = false;
                            int dep[APL];
                            bool cand[APL];
#pragma unroll
                            for (int k = 0; k < APL; ++k) {
                                dep[k] = -1;
                                cand[k] = mover[k];
                                if (mover[k]) {
                                    const int o = own[tcell[k]];
                                    if (o != 0xFF) {
                                        if (o > aidx[k] || stat[o] == kFail) cand[k] = false;   // still there at my turn / never leaves
                                        else dep[k] = o;
                                    }
                                }
                            }
                            bool wrote;
                            do {   // win[cell] = smallest agent index among the contenders (each round can only lower it)
                                bool lower[APL];
#pragma unroll
                                for (int k = 0; k < APL; ++k) lower[k] = cand[k] && win[tcell[k]] > aidx[k];
                                __syncwarp();
                                wrote = false;
#pragma unroll
                                for (int k = 0; k < APL; ++k)
                                    if (lower[k]) { win[tcell[k]] = (unsigned char)aidx[k]; wrote = true; }
                                __syncwarp();
                            } while (__any_sync(kFull, wrote));
                            int st[APL];
#pragma unroll
                            for (int k = 0; k < APL; ++k) {
                                st[k] = kFail;
                                if (cand[k]) st[k] = win[tcell[k]] != aidx[k] ? kFail : (dep[k] < 0 ? kOk : kUnknown);
                                if (mover[k]) stat[aidx[k]] = (unsigned char)st[k];
                            }
                            __syncwarp();
                            bool changed;
                            do {   // follow the chains: an agent that waits for j's cell succeeds iff j did
                                int seen[APL];
#pragma unroll
                                for (int k = 0; k < APL; ++k) seen[k] = st[k] == kUnknown ? (int)stat[dep[k]] : (int)kUnknown;
                                __syncwarp();
                                changed = false;
#pragma unroll
                                for (int k = 0; k < APL; ++k)
                                    if (st[k] == kUnknown && seen[k] != kUnknown) { st[k] = seen[k]; stat[aidx[k]] = (unsigned char)seen[k]; changed = true; }
                                __syncwarp();
                            } while (__any_sync(kFull, changed));
#pragma unroll
                            for (int k = 0; k < APL; ++k) {
                                if (st[k] == kOk) cmp[k] = req[k];                           // :406-408
                                if (cand[k]) win[tcell[k]] = 0xFF;                           // leave the map empty
                            }
                        }
#pragma unroll
                        for (int k = 0; k < APL; ++k)
                            if (active[k]) own[cell[k]] = 0xFF;
                        __syncwarp();
                    }
                }
                if (!sequential) {
                } else if (APL == 1 && A == LPE) {
#pragma unroll
                    for (int l = 0; l < LPE; ++l) turn(0, l);
                } else {
#pragma unroll
                    for (int s = 0; s < APL; ++s) {
                        const int lim = min(LPE, A - s * LPE);
#pragma unroll 4
                        for (int l = 0; l < lim; ++l) turn(s, l);
                    }
                }
            } else {
                int ord[APL];
#pragma unroll
                for (int k = 0; k < APL; ++k) ord[k] = (env_ok && avalid[k]) ? (int)p.order[off[k]] : -1;
                bool stop = !env_ok;
                for (int k = 0; k < A; ++k) {
                    const int oi = (int)T.tshfl((unsigned)picki<APL>(ord, k >> TL_::LOG), k & (LPE - 1));
                    stop = stop || oi < 0;
                    bool live = !stop;
                    if (live && oi >= A) { errbits |= kErrInvalidAction; live = false; }  // :701-705
                    const int ol = oi & (LPE - 1), os = (oi >> TL_::LOG) & (APL - 1);
                    const int my_act = picki<APL>(action, os);
                    const unsigned my_cmp = pick<APL>(cmp, os);
                    const bool owner = live && T.li == ol;
                    if (owner && (unsigned)my_act > 4u) errbits |= kErrInvalidAction;   // :707-711
                    // the cell is recomputed: an agent listed twice has moved since the top of the step
                    const int my_cell = (min((int)(my_cmp & 0xffu), p.H + 1) + 1) * PW + min((int)((my_cmp >> 8) & 0xffu), p.W + 1) + 1;
                    unsigned rq = T.tshfl(make_request(my_cell, my_act, my_cmp), ol);
                    bool hit = !live;   // a dead turn hits itself everywhere
#pragma unroll
                    for (int s = 0; s < APL; ++s) hit |= cmp[s] == rq;
                    const unsigned occ = __ballot_sync(kFull, hit) & tile_bits;
                    if (owner && !occ) {
#pragma unroll
                        for (int s = 0; s < APL; ++s) if (s == os) cmp[s] = rq;
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < APL; ++k) pos[k] = (fl[k] & CC_F_ACTIVE) ? cmp[k] : pos[k];   // ghosts never move

            // ---- :210-212 deactivate arrivals; rewards; terminated; truncated --------------
            bool lane_not_arr = false, lane_new_arr = false;
            unsigned arr[APL];
#pragma unroll
            for (int k = 0; k < APL; ++k) {
                lookup(k);                                             // geometry of the post-move cell
                arr[k] = avalid[k] ? (geo_f[k] >> 3) & 1u : 0u;        // :663-683 (y only)
                const bool newly = env_ok && arr[k] && (fl[k] & CC_F_ACTIVE);
                fl[k] &= ~arr[k];                                      // types.py:46-51 (CC_F_ACTIVE == 1)
                if (APL == 1) lane_new_arr = newly;
                else st_arrivals += __popc(__ballot_sync(kFull, newly));   // counted warp-wide on every lane; lane 0's copy is used
                lane_not_arr = lane_not_arr || (avalid[k] && !arr[k]);
            }
            if (APL == 1) st_arrivals += __popc(__ballot_sync(kFull, lane_new_arr));
            const bool all_arrived = (__ballot_sync(kFull, lane_not_arr) & tile_bits) == 0u;
            const bool over_limit = step >= p.max_steps;                // truncateds.py:61
            bool lane_alive = false;
            float rsum_lane = 0.f;
            float rew[APL];
            unsigned oflag[APL];
#pragma unroll
            for (int k = 0; k < APL; ++k) {
                // One path for the four reward functions: the distance table holds the per-kind value
                // (a constant for binary / constant_negative), and the DefaultReward categories
                // (rewards.py:78-99) override it where their mask bits are set (masks are 0 for the others).
                const unsigned f = geo_f[k];
                CCB_CHECK(rtoff[k] + (int)((geo_u[k] >> 8) & 0x1ffu) < 2 * kRtabSize);
                float r = rtab[rtoff[k] + (int)((geo_u[k] >> 8) & 0x1ffu)];       // :82-85 / :95-99 (positive, sic) / :127
                const bool boarding = aidx[k] < p.B;
                const float special = boarding ? ((f & 2u) ? p.rpf[1] : p.rpf[2]) : p.rpf[2];  // door / tram area | exiting outside (sic)
                const unsigned in_special = boarding ? (f & 3u) : ((f & 1u) ^ 1u);
                r = (in_special & p.reward_category_mask) ? special : r;
                r = (f & 8u & p.reward_category_mask) ? p.rpf[0] : r;              // :78-79 and :88-89 (same parameter, sic)
                r = alive_prev[k] ? r : 0.f;                            // rewards.py:65-66 etc.
                rew[k] = r;
                rsum_lane += r;
                lane_alive |= alive_prev[k] != 0u;
                const unsigned tval = (p.terminated_kind == CC_TERM_ALL_AT_DESTINATION) ? (unsigned)all_arrived : arr[k];  // terminateds.py:56-60,82
                const unsigned cval = alive_prev[k] & (unsigned)over_limit;   // truncateds.py:57-61
                // collectivecrossing.py:229-243: sticky flags; an entry is returned for agents that were
                // alive at step start and for agents whose terminated flag flips now
                const unsigned present = alive_prev[k] | (tval & ~(fl[k] >> 1) & 1u);
                fl[k] |= (tval << 1) | (cval << 2);
                oflag[k] = (fl[k] & 7u) | (alive_prev[k] << 3) | (tval << 4) | (cval << 5) | (present << 6);
            }
            const bool any_alive = (__ballot_sync(kFull, lane_alive) & tile_bits) != 0u;
            const bool term_all = all_arrived;                          // :256 (terminateds holds every agent)
            const bool trunc_all = any_alive && over_limit;             // :257
            // reward sum: balanced tree over the tile's lanes (fixed association order; the oracle
            // reproduces it), accumulated into the env's float32 episode return
            float rsum = rsum_lane;
#pragma unroll
            for (int w = LPE / 2; w >= 1; w >>= 1) rsum += __shfl_xor_sync(kFull, rsum, w, LPE);
            ep_ret += rsum;
            const bool done = term_all || trunc_all;
            eflags = (term_all ? CC_E_TERMINATED_ALL : 0u) | (trunc_all ? CC_E_TRUNCATED_ALL : 0u);

            // ---- outputs of the finished step ----------------------------------------------
#pragma unroll
            for (int k = 0; k < APL; ++k)
                if (env_ok && avalid[k]) {
                    if (p.reward_f64) {
                        // single-env facade: the reference's float64 value itself
                        const int x = (int)(pos[k] >> 8), y = (int)(pos[k] & 0xffu);
                        const bool boarding = aidx[k] < p.B;
                        double r = 0.0;
                        if (alive_prev[k]) {
                            switch (p.reward_kind) {
                            case CC_REWARD_DEFAULT:
                                if (arr[k]) r = p.rp[0];
                                else if (boarding) r = at_tram_door(p, x, y) ? p.rp[1] : in_tram_area(p, x, y) ? p.rp[2] : (double)(-(abs(x - p.DC) + (p.D - y))) * p.rp[3];
                                else r = !in_tram_area(p, x, y) ? p.rp[2] : (double)(abs(x - p.DC) + (y - p.D)) * p.rp[3];
                                break;
                            case CC_REWARD_SIMPLE_DISTANCE: r = (double)(-abs(y - (boarding ? p.YB : p.YE))) * p.rp[0]; break;
                            case CC_REWARD_BINARY: r = p.rp[1]; break;
                            default: r = p.rp[0]; break;
                            }
                        }
                        __stcs(reinterpret_cast<double *>(p.reward) + off[k], r);
                    } else __stcs(reinterpret_cast<float *>(p.reward) + off[k], rew[k]);
                    // (per-step outputs are written once and never read by the kernels: streaming stores keep them from
                    // displacing the state in L2 — measured on the thread-per-env kernel: 0.2545 -> 0.2422 ms per launch)
                    __stcs(reinterpret_cast<unsigned char *>(p.agent_flags) + off[k], (unsigned char)oflag[k]);
                    // :248-254: in_tram_area | at_door | active | at_destination
                    if (p.agent_info) __stcs(reinterpret_cast<unsigned char *>(p.agent_info) + off[k], (unsigned char)((geo_f[k] & 0xBu) | ((fl[k] & 1u) << 2)));
                }
            const bool leader = env_ok && T.li == 0;
            if (leader) st_rsum += (double)rsum;
            const bool ended = leader && done && any_alive;             // the step the last agents finished on
            const unsigned ended_mask = __ballot_sync(kFull, ended);
            if (ended_mask) {                                           // rare: fold this warp's finished episodes into its slot
                unsigned n_term = __popc(__ballot_sync(kFull, ended && term_all)), n_trunc = __popc(__ballot_sync(kFull, ended && trunc_all));
                unsigned len = ended ? (unsigned)step : 0u;
                double ret = ended ? (double)ep_ret : 0.0;
#pragma unroll
                for (int w = 16; w >= 1; w >>= 1) { len += __shfl_xor_sync(kFull, len, w); ret += __shfl_xor_sync(kFull, ret, w); }
                if (T.lane == 0) {
                    red[kStEpisodes] += __popc(ended_mask); red[kStTermAll] += n_term; red[kStTruncAll] += n_trunc; red[kStEpLen] += len;
                    red[kStEpRet] = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)red[kStEpRet]) + ret);
                }
            }
            need_reset = env_ok && done && p.auto_reset;
            if (need_reset) { eflags |= CC_E_WAS_RESET; ep_ret = 0.f; }
        }
        if (MODE == kModeReset) need_reset = env_ok && (p.mask == nullptr || p.mask[(int)n0 + T.tile] != 0);

        // ---- collectivecrossing.py:91-150 reset(): rejection-sampled placement ---------------
        // Agent i's k-th candidate is Philox(seed; genv, t, RESET, i<<16|k); it takes the first
        // candidate that passes the geometric test and is not occupied by an agent j < i.  The
        // candidates are drawn by all lanes at once, the acceptance sweep is sequential.
        if ((MODE == kModeStep || MODE == kModeReset) && __any_sync(kFull, need_reset)) {
          if constexpr (kNp) {
            // numpy mode: the env's generator is sequential, so the tile's lane 0 holds it, draws the candidates of agent `fin`
            // one at a time (np_candidate) and broadcasts them; the occupancy ballot accepts a candidate or asks for the next
            // draw.  Draws, attempt cap and result are those of np_place_agent / cc_reset_seeded_kernel.
            bool placed[APL];
#pragma unroll
            for (int k = 0; k < APL; ++k) placed[k] = false;
            int fin = need_reset ? 0 : A;  // agents placed so far (tile-uniform)
            int attempt = 0;               // draws for agent fin (lane 0)
            Pcg64 g;
            if (need_reset && T.li == 0) g = np_load(p.gen[n0 + T.tile]);
            while (__any_sync(kFull, fin < A)) {
                const bool act_tile = fin < A;
                unsigned rq = 0;   // bit 31: passes the geometric test, bit 16: attempt cap reached, low 16 bits: packed candidate
                if (act_tile && T.li == 0) {
                    int cx, cy;
                    const bool ok = np_candidate(g, p, fin < p.B, cx, cy);
                    attempt += 1;
                    rq = pack_pos(cx, cy) | (ok ? 0x80000000u : 0u) | (attempt >= kResetAttemptCap ? 0x10000u : 0u);
                }
                rq = T.tshfl(rq, 0);
                bool hit = false;
#pragma unroll
                for (int s = 0; s < APL; ++s) hit |= placed[s] && pos[s] == (rq & 0xffffu);
                const unsigned occ = __ballot_sync(kFull, hit) & tile_bits;
                const bool good = (rq >> 31) && !occ;
                if (act_tile && (good || (rq & 0x10000u))) {   // accepted, or the cap is hit: the last candidate stays
                    if (T.li == (fin & (LPE - 1))) {
#pragma unroll
                        for (int s = 0; s < APL; ++s) if (s == (fin >> TL_::LOG)) { placed[s] = true; pos[s] = rq & 0xffffu; }
                    }
                    if (!good && T.li == 0) errbits |= kErrResetStuck;
                    fin += 1;
                    attempt = 0;
                }
            }
            if (need_reset && T.li == 0) p.gen[n0 + T.tile] = np_save(g);
          } else {
            bool placed[APL], has_cand[APL];
            unsigned cand[APL];
            int attempt[APL];
#pragma unroll
            for (int k = 0; k < APL; ++k) { placed[k] = false; has_cand[k] = false; cand[k] = 0; attempt[k] = 0; }
            int fin = need_reset ? 0 : A;  // agents finalised so far (tile-uniform)
            while (__any_sync(kFull, fin < A)) {
#pragma unroll
                for (int k = 0; k < APL; ++k) {
                    if (fin < A && avalid[k] && !placed[k] && !has_cand[k]) {
                        const U4 r = draw(p, genv, kStreamReset, ((unsigned)aidx[k] << 16) | (unsigned)attempt[k]);
                        int cx, cy;
                        bool ok;
                        if (aidx[k] < p.B) {                            // :103-117
                            cx = bounded(r.v0, p.W); cy = bounded(r.v1, p.D);
                            ok = valid_position(p, cx, cy) && !(p.DL <= cx && cx <= p.DR && cy == p.D - 1);
                        } else {                                        // :132-140
                            cx = p.TL + bounded(r.v0, p.TR + 1 - p.TL); cy = p.D + bounded(r.v1, p.H - p.D);
                            ok = valid_position(p, cx, cy);
                        }
                        attempt[k] += 1;
                        cand[k] = pack_pos(cx, cy);
                        has_cand[k] = ok;
                        if (!ok && attempt[k] >= kResetAttemptCap) { has_cand[k] = true; cand[k] |= 0x10000u; errbits |= kErrResetStuck; }
                    }
                }
                bool progress = true;
                while (__any_sync(kFull, progress && fin < A)) {
                    const bool act_tile = progress && fin < A;
                    const int fi = act_tile ? fin : 0;
                    const int ol = fi & (LPE - 1), os = fi >> TL_::LOG;
                    unsigned mine = pick<APL>(cand, os);
                    bool mine_has = false;
#pragma unroll
                    for (int s = 0; s < APL; ++s) mine_has = (s == os) ? has_cand[s] : mine_has;
                    const unsigned rq = T.tshfl(mine | (mine_has ? 0x80000000u : 0u), ol);
                    const bool forced = (rq & 0x10000u) != 0;  // attempt cap hit: place regardless
                    bool hit = false;
#pragma unroll
                    for (int s = 0; s < APL; ++s) hit |= placed[s] && pos[s] == (rq & 0xffffu);
                    const unsigned occ = __ballot_sync(kFull, hit) & tile_bits;
                    if (act_tile && (rq >> 31)) {
                        if (!occ || forced) {
                            if (T.li == ol) {
#pragma unroll
                                for (int s = 0; s < APL; ++s) if (s == os) { placed[s] = true; pos[s] = rq & 0xffffu; }
                            }
                            fin += 1;
                        } else {
                            if (T.li == ol) {
#pragma unroll
                                for (int s = 0; s < APL; ++s)
                                    if (s == os) {
                                        has_cand[s] = false;
                                        if (attempt[s] >= kResetAttemptCap) { has_cand[s] = true; cand[s] |= 0x10000u; errbits |= kErrResetStuck; }
                                    }
                            }
                            progress = false;
                        }
                    } else progress = false;
                }
            }
          }
            if (need_reset) {
                step = 0;                                               // :97
#pragma unroll
                for (int k = 0; k < APL; ++k) fl[k] = avalid[k] ? (unsigned)CC_F_ACTIVE : 0u;
                if (MODE == kModeReset) ep_ret = 0.f;
            }
        }

        // ---- write back the persistent state ----------------------------------------------------
        if (MODE == kModeStep || MODE == kModeReset) {
            const bool wr = env_ok && (MODE == kModeStep || need_reset);
#pragma unroll
            for (int k = 0; k < APL; ++k)
                if (wr && avalid[k]) {
                    p.x[off[k]] = (int8_t)(pos[k] >> 8);
                    p.y[off[k]] = (int8_t)(pos[k] & 0xffu);
                    p.flags[off[k]] = (uint8_t)(fl[k] & 7u);
                }
            if (wr && T.li == 0) {
                p.step[(int)n0 + T.tile] = step;
                p.ep_ret[(int)n0 + T.tile] = ep_ret;
                if (MODE == kModeStep) __stcs(reinterpret_cast<unsigned char *>(p.env_flags) + (int)n0 + T.tile, (unsigned char)eflags);
            }
        }

        // ---- CC_OBS_TABLE: (x_j, y_j, type_j, active_j) of observations.py:80-91, one 32-bit word per agent ----
        if (kTable && p.obs != nullptr) {
            const bool wr = env_ok && (MODE != kModeReset || need_reset);   // reset: only the envs that were reset
            unsigned *tab = reinterpret_cast<unsigned *>(p.obs) + p.obs_env_offset * A;
#pragma unroll
            for (int k = 0; k < APL; ++k)
                if (wr && avalid[k])
                    __stcs(tab + off[k], (pos[k] >> 8 & 0xffu) | ((pos[k] & 0xffu) << 8) | ((aidx[k] < p.B ? 0u : 1u) << 16) | ((fl[k] & 1u) << 24));
        }

        // ---- observations.py:43-94 from the post-step (post-reset) state ------------------------
        if (kHasObs && p.obs != nullptr) {
            P2 *tstage = stage + T.tile * (2 * A + 4) + 3;
#pragma unroll
            for (int k = 0; k < APL; ++k)
                if (avalid[k]) {
                    tstage[2 * aidx[k]] = mk_pair<OT>((int)(int8_t)(pos[k] >> 8), (int)(int8_t)(pos[k] & 0xffu));
                    tstage[2 * aidx[k] + 1] = mk_pair<OT>(aidx[k] < p.B ? 0 : 1, (int)(fl[k] & 1u));
                    if (shift_rows) {
                        // the agent's 4 bytes into the 8 shifted copies (template byte 6 + 4a at copy byte 2c + 6 + 4a)
                        const unsigned lo = (pos[k] >> 8 & 0xffu) | ((pos[k] & 0xffu) << 8), hi = (aidx[k] < p.B ? 0u : 1u) | ((fl[k] & 1u) << 8);
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            unsigned char *d = shifted + c * p.shift_tst + 2 * c + 6 + 4 * aidx[k];
                            if (c & 1) *reinterpret_cast<unsigned *>(d) = lo | (hi << 16);
                            else { *reinterpret_cast<unsigned short *>(d) = (unsigned short)lo; *reinterpret_cast<unsigned short *>(d + 2) = (unsigned short)hi; }
                            if (aidx[k] < 3) {   // the 16-byte tail repeats the head of the template (a row is 2 mod 4 bytes long)
                                unsigned char *d2 = d + lrow;
                                *reinterpret_cast<unsigned short *>(d2) = (unsigned short)lo; *reinterpret_cast<unsigned short *>(d2 + 2) = (unsigned short)hi;
                            }
                        }
                    }
                }
            __syncwarp();
            OT *obs = reinterpret_cast<OT *>(p.obs);
            const long long gp0 = (n0 + p.obs_env_offset) * (long long)p.pairs_per_env;   // (offset: time slice of a rollout buffer)
            P2 *out = reinterpret_cast<P2 *>(obs) + gp0;
            const int count = envs_here * p.pairs_per_env;        // output pairs of this group
            if (MODE == kModeReset) {
                // only the envs that were reset get their rows rewritten
                const unsigned tiles = __ballot_sync(kFull, need_reset);
                for (int P = T.lane; P < count; P += 32)
                    if ((tiles >> ((P / p.pairs_per_env) * LPE)) & 1u) out[P] = stage[gather_index(p, P)];
            } else if (kCanCache && cached && (kPairwise || envs_here == EPW)) {
                uint4 d4 = make_uint4(0, 0, 0, 0);
                if (kPairwise) {
                    // lane <-> output pair: 32 lanes store 256 contiguous bytes per instruction
                    P2 *o = out + T.lane;
#pragma unroll
                    for (int w = 0; w < kDescWords; ++w) {
                        if (w * 32 < count) {                             // uniform
                            if (w % 4 == 0) d4 = desc_sm[(w / 4) * kThreads];
                            const unsigned a = (w % 4 == 0) ? d4.x : (w % 4 == 1) ? d4.y : (w % 4 == 2) ? d4.z : d4.w;
                            const P2 v = *reinterpret_cast<const P2 *>(smem + a);
                            if (w * 32 + 32 <= count || T.lane + w * 32 < count) __stcs(reinterpret_cast<float2 *>(o + 32 * w), reinterpret_cast<const float2 &>(v));
                        }
                    }
                } else {
                    // whole, vector-aligned chunk: each lane assembles its 16-byte vectors
                    uint4 *outv = reinterpret_cast<uint4 *>(out) + T.lane;
                    const int nvec = chunk_pairs / PPV;
#pragma unroll
                    for (int j = 0; j < kDescWords / PPV; ++j) {
                        if (j * 32 < nvec) {                              // uniform
                            union { uint4 u; P2 e[PPV]; } pk;
#pragma unroll
                            for (int h = 0; h < PPV; ++h) {
                                const int w = j * PPV + h;
                                if (w % 4 == 0) d4 = desc_sm[(w / 4) * kThreads];
                                const unsigned a = (w % 4 == 0) ? d4.x : (w % 4 == 1) ? d4.y : (w % 4 == 2) ? d4.z : d4.w;
                                pk.e[h] = *reinterpret_cast<const P2 *>(smem + a);
                            }
                            if (j * 32 + 32 <= nvec || T.lane + j * 32 < nvec) __stcs(outv + 32 * j, pk.u);
                        }
                    }
                }
            } else if (shift_rows) {
                if constexpr (kShiftable) {
                    // The env block leaves the SM chunk by chunk (8 rows = img_vecs vectors): the warp assembles a chunk in one of
                    // kLaneImgRing shared-memory images — a plain vector is ONE aligned 16-byte load from the shifted template,
                    // a special one is gathered pair by pair — and one lane hands the image to the TMA unit (cp.async.bulk).
                    // Stores issued with st.global stall the SM's load/store pipe, and with it the other warps' shared-memory
                    // work, whenever HBM pushes back (profiles/probes/lsu_coupling_probe.cu; DESIGN.md §3.1).
                    // (32-bit shared-memory addresses: the copy of a vector is its source offset (ld.shared.u32), one ld.shared.v4 and one st.shared.v4)
                    const unsigned src_s = (unsigned)__cvta_generic_to_shared(img_src) + 4u * (unsigned)T.lane;
                    const unsigned ring_s = (unsigned)__cvta_generic_to_shared(smem + p.off_img + warp * (kLaneImgRing * p.img_vecs * 16));
                    const unsigned shifted_s = (unsigned)__cvta_generic_to_shared(shifted);
                    unsigned char *dst = reinterpret_cast<unsigned char *>(out);
                    const unsigned chunk_bytes = (unsigned)p.img_vecs * 16u;
                    for (int c = 0; c < p.n_chunks; ++c) {
                        const unsigned img_s = ring_s + (unsigned)img_slot * chunk_bytes;
                        img_slot = img_slot + 1 == kLaneImgRing ? 0 : img_slot + 1;
                        const int rows_here = min(p.img_rows, A - c * p.img_rows);          // (the last chunk may be shorter)
                        const int vecs_here = rows_here * lrow / 16;
                        if (T.lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kLaneImgRing - 1) : "memory");   // the copy that read this image is done
                        __syncwarp();
#pragma unroll
                        for (int k = 0; k < kMaxImgIter; ++k)
                            if (T.lane + 32 * k < vecs_here) {
                                uint4 v;
                                unsigned so;
                                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(so) : "r"(src_s + 128u * k));
                                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(shifted_s + so));
                                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(img_s + 16u * (unsigned)(T.lane + 32 * k)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
                            }
                        __syncwarp();
                        if (T.lane < rows_here) {   // row i of the env: own position in front, -1 over the own block (observations.py:62-64,92-93)
                            const int i = c * p.img_rows + T.lane;
                            const unsigned row_s = img_s + (unsigned)(T.lane * lrow);
                            const unsigned short own = *reinterpret_cast<const unsigned short *>(stage + 3 + 2 * i);
                            asm volatile("st.shared.u16 [%0], %1;" ::"r"(row_s), "h"(own) : "memory");
                            asm volatile("st.shared.u16 [%0], %1;" ::"r"(row_s + 6u + 4u * (unsigned)i), "h"((unsigned short)0xffffu) : "memory");
                            asm volatile("st.shared.u16 [%0], %1;" ::"r"(row_s + 8u + 4u * (unsigned)i), "h"((unsigned short)0xffffu) : "memory");
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async-proxy read
                        __syncwarp();
                        if (T.lane == 0) {
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                                         ::"l"(dst + (size_t)c * chunk_bytes), "r"(img_s), "r"((unsigned)vecs_here * 16u), "l"(l2_evict_first) : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                    }
                }
            } else if (cached) {
                // ragged last group of an int8 run that otherwise uses the descriptors: the LUT was not
                // built, gather with the index function directly (at most once per launch)
                for (int P = T.lane; P < count; P += 32) out[P] = stage[gather_index(p, P)];
            } else {
                emit_obs_lut<OT>(obs, gp0, count, lut, stage, T.lane);
            }
            __syncwarp();
        }
    }

    if (kShiftable && T.lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // shared memory stays valid until the copies are done
    // ---- statistics: per-warp slots in shared memory -> one atomic per slot per CTA ----------------
    if (MODE == kModeStep) {
        // every lane counted arrivals warp-wide: lane 0's copy is the warp's count
        double rs = st_rsum;
#pragma unroll
        for (int w = 16; w >= 1; w >>= 1) rs += __shfl_xor_sync(kFull, rs, w);
        if (T.lane == 0) {
            red[kStArrivals] += st_arrivals;
            red[kStRewardSum] = (unsigned long long)__double_as_longlong(rs);
        }
        __syncthreads();
        const unsigned long long *all = red_all;
        if (threadIdx.x >= 1 && threadIdx.x < 6) {
            unsigned long long v = 0;
            for (int w = 0; w < kWarpsPerCta; ++w) v += all[w * kStCount + threadIdx.x];
            if (v) atomicAdd(&p.stats[threadIdx.x], v);
        } else if (threadIdx.x == 6 || threadIdx.x == 7) {
            double v = 0.0;
            for (int w = 0; w < kWarpsPerCta; ++w) v += __longlong_as_double((long long)all[w * kStCount + threadIdx.x]);
            if (v != 0.0) atomicAdd(reinterpret_cast<double *>(&p.stats[threadIdx.x]), v);
        } else if (threadIdx.x == 0 && blockIdx.x == 0) {
            atomicAdd(&p.stats[kStEnvSteps], (unsigned long long)p.n_envs);
        }
    }
    if (errbits) atomicOr(p.err, errbits);
}

// seeds != nullptr: reset(seed=seeds[n]) — a fresh generator per env (gymnasium Env.reset(seed=s));
// seeds == nullptr: reset() — every env keeps drawing from its stored generator.
// (a plain function, not a template: defined in the one translation unit that sets CCB_WITH_RESET_SEEDED)
#ifdef CCB_WITH_RESET_SEEDED
__global__ void __launch_bounds__(128) cc_reset_seeded_kernel(const __grid_constant__ KParams p, const long long *seeds, Pcg64State *gen) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= p.n_envs) return;
    Pcg64 g;
    if (seeds) g.seed((unsigned long long)seeds[n]);
    else g = np_load(gen[n]);
    int8_t *x = p.x + n * p.A, *y = p.y + n * p.A;
    int stuck = 0;
    for (int i = 0; i < p.A; ++i) {
        int px = 0, py = 0;
        const bool ok = np_place_agent(g, p, i < p.B, [&](int cx, int cy) {
            for (int j = 0; j < i; ++j)
                if (x[j] == cx && y[j] == cy) return false;
            return true;
        }, px, py);
        if (!ok) stuck = 1;
        x[i] = (int8_t)px; y[i] = (int8_t)py;
        p.flags[n * p.A + i] = CC_F_ACTIVE;
    }
    p.step[n] = 0;
    p.ep_ret[n] = 0.f;
    gen[n] = np_save(g);
    if (stuck) atomicOr(p.err, kErrResetStuck);
}
#endif  // CCB_WITH_RESET_SEEDED

}  // namespace ccb
