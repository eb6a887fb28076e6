// cc_kernel_tpe2.cuh — thread-per-env step kernel for SMALL lattices and the compact output modes.
//
// cc_step_tpe_kernel (cc_kernel_tpe.cuh) is bound by HBM when it writes the reference's float32 rows, but its compact
// modes (no observations, int8 rows, the compact table) are bound by instruction issue: ~2,000 warp-instructions per
// 32 env-steps (profiles/r1_ncu_summary.txt).  This kernel restates the same step (same semantics, same RNG streams,
// bit-identical results — tests/test_gpu_parity.py runs every eligible case through it) with a third of the instructions:
//
//   * a position is ONE byte, the agent's cell of the padded lattice: c = (y+1)*PW + (x+1) <= 255.  The 8 cells of an
//     env come out of the packed x / y state words with one multiply-add per 4 agents (byte lanes never carry);
//   * everything the step needs to know about a cell is one 8-byte table entry per (cell, agent type), read with a single
//     ld.shared.v2: greedy-table row, in-tram / at-door / arrived bits, x, y, walkable-neighbour masks — and the float32
//     REWARD itself (collectivecrossing.py:509-563, rewards.py:41-182 evaluated once per cell when the table is built);
//   * per-agent flag logic (types.py:16-73, collectivecrossing.py:229-243, truncateds.py:57-61, terminateds.py:56-82) runs
//     on 4 agents per 32-bit word (SWAR); per-agent selects use PRMT sign-fill masks instead of predicates;
//   * ordered moves (collectivecrossing.py:197-202) compare the one-byte target with the 8 cells of the ACTIVE agents;
//     an agent that must not move asks for its own cell (or, a ghost, for the ghost sentinel) and so blocks itself;
//   * int8 rows: every thread composes its env's 304-byte block with 19 conflict-free 16-byte shared-memory stores and the
//     warp's 9,728 contiguous bytes leave the SM as ONE bulk asynchronous copy (TMA, SASS UBLKCP).
//
// Eligibility (host side, cc_launch_tpe.cu): crews of at most 8, padded lattice (W+3)(H+3) <= 256 with at most 32 columns
// and 16 rows (README config: 15 x 11 = 165), obs in {none, table, int8 (8 agents)}.  Every other case runs
// cc_step_tpe_kernel / cc_kernel.  Reference paths are relative to /root/reference/src/collectivecrossing/.
#pragma once
#include "cc_kernel_tpe.cuh"

#ifndef CCB_T2_MIN_BLOCKS
#define CCB_T2_MIN_BLOCKS 6    // resident 128-thread CTAs per SM the register allocator must allow (<= 80 registers)
#endif

namespace ccb {

constexpr int kT2Warps = 4;            // warps per CTA (2 for batches that fit in one wave: finer CTAs balance the SMs better)
constexpr int kT2Threads = kT2Warps * 32;
constexpr int kT2MaxRows = 16, kT2MaxCols = 32, kT2MaxCells = 256;
constexpr int kT2BitmapBytesPerWarp = kT2MaxRows * 128;   // row r of lane l at r * 128 + l * 4

// geo word of a table entry (low half of the 8-byte entry; the high half is the float32 reward of an agent of that type
// standing on the cell, rewards.py:41-182):
//   byte 0  bits 0-4 row of the greedy decision table (type, y class, x class; greedy_policy.py:117-158),
//           bit 5 in_tram_area (:551-554), bit 6 at_tram_door (:556-563), bit 7 at destination (:663-683)
//   byte 1  x
//   byte 2  bits 0-3 y, bits 4-7 walkable neighbours in ACTION order (bit a: the cell in direction a passes :509-534)
//   byte 3  bits 0-3 walkable neighbours in BITMAP order (bit0 left, bit1 up, bit2 right, bit3 down),
//           bit 4 the cell itself is a valid position, bit 5 the cell is excluded from boarding spawns (:110-115)
enum { kT2InTram = 1u << 5, kT2AtDoor = 1u << 6, kT2Arrived = 1u << 7, kT2Valid = 1u << 28, kT2SpawnExcluded = 1u << 29 };

// The tables of one config, built once per handle by cc_t2_tables_kernel and copied into shared memory by every CTA.
struct T2Tables {
    uint2 tab[2 * kT2MaxCells];            // [cell][type] {geo, reward}
    uint8_t act2[kPolicyRows * 16];        // greedy decision by (table row, free-neighbour mask in bitmap order)
    int dcell[8];                          // cell delta of actions 0..3 (actions.py:18-24); 0 for wait / invalid
};
static_assert(sizeof(T2Tables) % 16 == 0, "copied as 16-byte vectors");

template <int A, int OBS>
struct T2Layout {
    static constexpr bool kImage = OBS == CC_OBS_INT8;                 // 8 agents: an env's block is 19 x 16 bytes
    static constexpr int kEnvBytes = A * (6 + 4 * A);
    static constexpr int kImageBytes = kImage ? 32 * kEnvBytes : 0;    // 9,728 B: the warp's 32 blocks, contiguous like the output
    // float32 rows (even crews): the row templates + image ring of cc_kernel_tpe.cuh, emitted by tpe_emit_group_tma
    using L1 = TpeLayout<A, CC_OBS_FP32>;
    static constexpr bool kRows32 = OBS == CC_OBS_FP32;
    static constexpr int kRows32Bytes = kRows32 ? L1::kStageBytesPerWarp : 0;
    // the policy bitmap aliases the image / the image ring (idle while the warp steps): it is zeroed before every use there
    static constexpr bool kDirtyBitmap = kImage || kRows32;
    static constexpr int kBitmapOffset = kRows32 ? L1::kTplBytesPerWarp : 0;
    static constexpr int kBytesNeeded = kImage ? kImageBytes : (kRows32 ? kRows32Bytes : 0);
    static constexpr int kBytesPerWarp = kBytesNeeded > kBitmapOffset + kT2BitmapBytesPerWarp ? kBytesNeeded : kBitmapOffset + kT2BitmapBytesPerWarp;
    static constexpr int kDynBytes = kT2Warps * kBytesPerWarp;
};

// 0xFFFFFFFF if bit 7 of byte k of w is set, else 0 (PRMT with the sign-replicate selector)
// (k is a constant after unrolling: the selector is an immediate)
// (inline PTX: the __byte_perm intrinsic documents only the 3 index bits of a selector nibble)
__device__ __forceinline__ unsigned t2_fill(unsigned w, int k) {
    unsigned r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0u), "r"(0x8888u | ((unsigned)k * 0x1111u)));
    return r;
}
// bytes B of a, b, c, d -> one word (a in byte 0)
template <int B>
__device__ __forceinline__ unsigned t2_gather4(unsigned a, unsigned b, unsigned c, unsigned d) {
    const unsigned lo = __byte_perm(a, b, (unsigned)(B | ((4 + B) << 4)));
    const unsigned hi = __byte_perm(c, d, (unsigned)(B | ((4 + B) << 4)));
    return __byte_perm(lo, hi, 0x5410u);
}
// byte B of the geo words of the (up to) 8 agents, agents 0-3 in w[0], 4-7 in w[1]
template <int A, int B>
__device__ __forceinline__ void t2_gather(const uint2 (&e)[A], unsigned (&w)[2]) {
    auto g = [&](int k) { return e[k < A ? k : A - 1].x; };
    w[0] = t2_gather4<B>(g(0), g(1), g(2), g(3));
    w[1] = A > 4 ? t2_gather4<B>(g(4), g(5), g(6), g(7)) : 0u;
}
// A bytes of env `env` of an [N][A] byte array from two packed words
template <int A, bool STREAM>
__device__ __forceinline__ void t2_store_packed(void *base, int env, unsigned w0, unsigned w1) {
    unsigned char *q = static_cast<unsigned char *>(base) + (size_t)env * A;
    if constexpr (A == 8) {
        if constexpr (STREAM) __stcs(reinterpret_cast<uint2 *>(q), make_uint2(w0, w1));
        else *reinterpret_cast<uint2 *>(q) = make_uint2(w0, w1);
    } else if constexpr (A == 4) {
        if constexpr (STREAM) __stcs(reinterpret_cast<unsigned *>(q), w0);
        else *reinterpret_cast<unsigned *>(q) = w0;
    } else {
#pragma unroll
        for (int k = 0; k < A; ++k) q[k] = (unsigned char)((k < 4 ? w0 : w1) >> (8 * (k & 3)));
    }
}

// one block: the tables of a config (collectivecrossing.py:509-563, rewards.py:41-182, greedy_policy.py:64-449 per cell)
// (a plain function, not a template: defined in the one translation unit that sets CCB_WITH_T2_TABLES)
#ifdef CCB_WITH_T2_TABLES
__global__ void __launch_bounds__(256) cc_t2_tables_kernel(const __grid_constant__ KParams p, T2Tables *out) {
    const int PW = p.W + 3, PH = p.H + 3;
    uint2 *tab = out->tab;
    uint8_t *act2 = out->act2;
    int *dcell = out->dcell;
    for (int i = threadIdx.x; i < 2 * kT2MaxCells; i += blockDim.x) {
        const int cell = i >> 1, type = i & 1;
        const int yy = cell / PW - 1, xx = cell - (yy + 1) * PW - 1;
        unsigned geo = 0;
        float rew = 0.f;
        if (cell < PW * PH && xx >= 0 && xx <= p.W && yy >= 0 && yy <= p.H) {
            const unsigned xv = make_xt(p, xx), yv = make_yt(p, type, yy);
            const unsigned u = xv + yv, f = (xv & yv) >> 24;   // f: bit0 in_tram, bit1 at_door, bit3 arrived (cc_kernels.cuh)
            const bool in_tram = f & 1u, at_door = f & 2u, arrived = f & 8u;
            const unsigned right = valid_position(p, xx + 1, yy), up = valid_position(p, xx, yy + 1), left = valid_position(p, xx - 1, yy),
                           down = valid_position(p, xx, yy - 1);
            geo = (u & 31u) | (in_tram ? kT2InTram : 0u) | (at_door ? kT2AtDoor : 0u) | (arrived ? kT2Arrived : 0u) | ((unsigned)xx << 8) |
                  ((unsigned)yy << 16) | ((right | (up << 1) | (left << 2) | (down << 3)) << 20) | ((left | (up << 1) | (right << 2) | (down << 3)) << 24) |
                  (valid_position(p, xx, yy) ? kT2Valid : 0u) | ((p.DL <= xx && xx <= p.DR && yy == p.D - 1) ? kT2SpawnExcluded : 0u);
            // the reward of an agent of this type on this cell, float32 of the reference's float64 value (rounded once)
            const bool boarding = type == 0;
            switch (p.reward_kind) {
            case CC_REWARD_DEFAULT:                                   // rewards.py:78-99
                if (arrived) rew = p.rpf[0];
                else if (boarding) rew = at_door ? p.rpf[1] : (in_tram ? p.rpf[2] : (float)((double)(-(abs(xx - p.DC) + (p.D - yy))) * p.rp[3]));
                else rew = !in_tram ? p.rpf[2] : (float)((double)(abs(xx - p.DC) + (yy - p.D)) * p.rp[3]);   // positive (sic)
                break;
            case CC_REWARD_SIMPLE_DISTANCE: rew = (float)((double)(-abs(yy - (boarding ? p.YB : p.YE))) * p.rp[0]); break;   // rewards.py:127
            case CC_REWARD_BINARY: rew = p.rpf[1]; break;              // rewards.py:152-159 (never goal_reward)
            default: rew = p.rpf[0]; break;                            // rewards.py:179-182
            }
        } else {
            // padding ring / beyond the lattice: never a position of a valid state; keep x, y inside the bitmap
            geo = ((unsigned)min(max(xx, 0), p.W) << 8) | ((unsigned)min(max(yy, 0), p.H) << 16);
        }
        tab[i] = make_uint2(geo, __float_as_uint(rew));
    }
    for (int i = threadIdx.x; i < kPolicyRows * 16; i += blockDim.x) {
        const unsigned m = (unsigned)i & 15u;   // bitmap order -> action order (0 right, 1 up, 2 left, 3 down)
        act2[i] = (uint8_t)greedy_decision(i >> 4, ((m >> 2) & 1u) | (m & 2u) | ((m & 1u) << 2) | (m & 8u));
    }
    if (threadIdx.x < 8) dcell[threadIdx.x] = threadIdx.x == 0 ? 1 : (threadIdx.x == 1 ? PW : (threadIdx.x == 2 ? -1 : (threadIdx.x == 3 ? -PW : 0)));
}
#endif  // CCB_WITH_T2_TABLES

// BT >= 0: the number of boarding agents is known at compile time (the README crew, 5 + 3: the type of agent k and with it
// the table half it reads, the boarding / exiting byte masks ... are immediates); BT = -1: any crew (p.B).
// OBSF: the obs dtype, with kNpReset for numpy-mode auto-reset placements (instantiated for BT = -1 only)
template <int A, int OBSF, int BT>
__global__ void __launch_bounds__(kT2Threads, CCB_T2_MIN_BLOCKS) cc_step_tpe2_kernel(const __grid_constant__ KParams p) {
    constexpr int OBS = OBSF & ~kNpReset;
    constexpr bool kNp = (OBSF & kNpReset) != 0;
    using L = T2Layout<A, OBS>;
    const int B = BT >= 0 ? BT : p.B;
    static_assert(A >= 1 && A <= 8, "thread-per-env mapping is for crews of at most 8");
    static_assert(OBS == CC_OBS_NONE || OBS == CC_OBS_TABLE || (OBS == CC_OBS_INT8 && A == 8) || (OBS == CC_OBS_FP32 && A % 2 == 0),
                  "int8 rows: 8 agents; float32 rows: even crews (an env's block must be whole 16-byte vectors for the bulk copies)");
    static_assert(!L::kRows32 || L::L1::kTma, "float32 rows leave through the TMA image ring");
    constexpr unsigned kOnes = 0x01010101u;
    // byte lanes of the agents that exist (k < A)
    constexpr unsigned kM0 = A >= 4 ? kOnes : (kOnes >> (8 * (4 - A)));
    constexpr unsigned kM1 = A <= 4 ? 0u : (A == 8 ? kOnes : (kOnes >> (8 * (8 - A))));
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ __align__(16) T2Tables tb;
    __shared__ unsigned long long red_all[kT2Warps * kStCount];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int PW = p.W + 3, PH = p.H + 3;

    // ---- once per CTA: the tables (L2-resident, 4.7 KB) and a clean bitmap ------------------------------------------
    for (int i = threadIdx.x; i < (int)(sizeof(T2Tables) / 16); i += blockDim.x)
        reinterpret_cast<uint4 *>(&tb)[i] = static_cast<const uint4 *>(p.t2_tables)[i];
    const int n_warps = (int)blockDim.x >> 5;   // 4, or 2 for small batches (cc_launch_tpe.cu)
    for (int i = threadIdx.x; i < n_warps * L::kBytesPerWarp / 4; i += blockDim.x) reinterpret_cast<unsigned *>(smem)[i] = 0u;
    __shared__ __align__(16) unsigned lut[L::kRows32 ? L::L1::kLutWords : 4];   // float32 rows: emission table of tpe_emit_group_tma
    if constexpr (L::kRows32) {
        __syncthreads();   // (the zero fill above must not overtake the constants below)
        using L1 = typename L::L1;
        for (int w = threadIdx.x; w < L1::kLutWords; w += blockDim.x) {
            // entry (j, lane): pair w = lane + 32 j of ANY env (offset inside that env's template)
            const int src = w < L1::PPE ? tpe_source<A>(w / L1::R, w % L1::R) : kSrcM;
            lut[w] = src >= 0 ? (unsigned)(src * L1::PSZ) : (0x80000000u | (unsigned)(-src));
        }
        // the constant pairs of this thread's template
        float2 *t = reinterpret_cast<float2 *>(smem + warp * L::kBytesPerWarp + lane * L1::TSB);
        t[2 * A] = make_float2((float)p.DC, (float)p.D); t[2 * A + 1] = make_float2((float)p.DL, (float)p.DR); t[2 * A + 2] = make_float2(-1.f, -1.f);
    }
    const TpeConstPairs kc = {make_uint2(__float_as_uint((float)p.DC), __float_as_uint((float)p.D)),
                              make_uint2(__float_as_uint((float)p.DL), __float_as_uint((float)p.DR)),
                              make_uint2(__float_as_uint(-1.f), __float_as_uint(-1.f))};
    unsigned long long *red = red_all + warp * kStCount;
    if (lane < kStCount) red[lane] = 0ull;
    if (blockIdx.x == 0 && threadIdx.x == 0) *p.tpe_counter_next = 0u;   // the counter the NEXT launch uses
    __syncthreads();

    const unsigned tab_s = (unsigned)__cvta_generic_to_shared(tb.tab), act_s = (unsigned)__cvta_generic_to_shared(tb.act2),
                   dc_s = (unsigned)__cvta_generic_to_shared(tb.dcell);
    unsigned char *wsmem = smem + warp * L::kBytesPerWarp;
    const unsigned img_s = (unsigned)__cvta_generic_to_shared(wsmem);
    const unsigned bm = img_s + (unsigned)L::kBitmapOffset + 4u * lane;   // this thread's bitmap row r at bm + 128 r
    unsigned tbase[A];                                          // table base of agent k's type
#pragma unroll
    for (int k = 0; k < A; ++k) tbase[k] = tab_s + (k < B ? 0u : 8u);
    // bytes 0x01 of the boarding agents; destination test and type byte are in the table
    unsigned boardw[2];
    boardw[0] = (B >= 4 ? kOnes : (B <= 0 ? 0u : (kOnes >> (8 * (4 - B))))) & kM0;
    boardw[1] = (B <= 4 ? 0u : (B >= 8 ? kOnes : (kOnes >> (8 * (8 - B))))) & kM1;
    const unsigned typew0 = kM0 & ~boardw[0], typew1 = kM1 & ~boardw[1];   // observations.py:86: 0 boarding, 1 exiting

    auto lookup = [&](unsigned c, int k) {
        CCB_CHECK(c < (unsigned)kT2MaxCells);
        uint2 e;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(tbase[k] + c * 16u));
        return e;
    };
    auto lds32 = [&](unsigned addr) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; };
    auto sts32 = [&](unsigned addr, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); };

    unsigned st_arrivals = 0;
    double st_rsum = 0.0;
    int errbits = 0;
    const int total_warps = (int)gridDim.x * n_warps;
    const int n_groups = (int)p.n_groups;
    int gw = (int)blockIdx.x * n_warps + warp;
    int g_next = 0;
    for (; gw < n_groups; gw = g_next) {
        const int g = p.tpe_reverse ? n_groups - 1 - gw : gw;
        const long long nn = (long long)g * 32 + lane;
        const int nl = nn < p.n_envs ? (int)nn : (int)p.n_envs - 1;    // threads beyond the end re-read the last env (never stored)
        const uint2 xw_in = tpe_fetch_row<A>(p.x, nl), yw_in = tpe_fetch_row<A>(p.y, nl), fw_in = tpe_fetch_row<A>(p.flags, nl);
        int step = p.step[nl];
        float ep_ret = p.ep_ret[nl];
#if CCB_TPE_DYNAMIC
        if (lane == 0) g_next = total_warps + (int)atomicAdd(p.tpe_counter, 1u);
#else
        g_next = gw + total_warps;
#endif
        const int n = g * 32 + lane;
        const int envs_here = (int)min(32ll, p.n_envs - (long long)g * 32);
        const bool env_ok = lane < envs_here;                 // false only in the ragged last group
        const unsigned long long genv = p.genv_offset + (unsigned long long)n;
        const unsigned m0e = env_ok ? kM0 : 0u, m1e = env_ok ? kM1 : 0u;

        // ---- the env's record, in registers for all the steps of this launch ----------------------------------------
        // cells: (y+1)*PW + (x+1) for 4 agents per multiply-add (every byte lane stays below 256 for in-lattice positions)
        unsigned c[A];
        {
            const unsigned bias = (unsigned)(PW + 1) * kOnes;
            const unsigned cw0 = yw_in.x * (unsigned)PW + xw_in.x + bias, cw1 = yw_in.y * (unsigned)PW + xw_in.y + bias;
#pragma unroll
            for (int k = 0; k < A; ++k) c[k] = ((k < 4 ? cw0 : cw1) >> (8 * (k & 3))) & 0xffu;
        }
        unsigned fl[2] = {env_ok ? fw_in.x & 0x07070707u & (kM0 * 7u) : 0u, env_ok ? fw_in.y & 0x07070707u & (kM1 * 7u) : 0u};
        uint2 e[A];                                            // table entries of the agents' current cells
#pragma unroll
        for (int k = 0; k < A; ++k) e[k] = lookup(c[k], k);
        unsigned fb[2];                                        // byte 0 of the entries (in_tram / at_door / arrived bits)
        t2_gather<A, 0>(e, fb);

      for (int tt = 0; tt < p.n_steps; ++tt) {   // (body indented as one step: time slice tt of every output)
        const size_t slice_a = (size_t)tt * (size_t)p.slice_agents;
        const unsigned t_rng = p.t + (unsigned)tt;
        unsigned act[A];
        bool geo_known = false;                                // chosen moves already passed the geometric test
        if (p.policy == CC_POLICY_EXTERNAL) {
            const uint2 aw = tpe_fetch_row<A>(p.actions + slice_a, env_ok ? n : (int)p.n_envs - 1);
            // collectivecrossing.py:707-711: an action outside {0..4} is an error (sticky flag) and moves nothing
            const unsigned bad0 = (((aw.x & 0x7f7f7f7fu) + 0x7b7b7b7bu) | aw.x) & 0x80808080u & (m0e * 0x80u);
            const unsigned bad1 = (((aw.y & 0x7f7f7f7fu) + 0x7b7b7b7bu) | aw.y) & 0x80808080u & (m1e * 0x80u);
            if (bad0 | bad1) errbits |= kErrInvalidAction;
#pragma unroll
            for (int k = 0; k < A; ++k) act[k] = min(((k < 4 ? aw.x : aw.y) >> (8 * (k & 3))) & 0xffu, 4u);
        } else if (p.policy == CC_POLICY_RANDOM) {
#pragma unroll
            for (int k = 0; k < A; ++k) act[k] = (unsigned)bounded(draw_at(p, t_rng, genv, kStreamAction, (unsigned)k).v0, 5);
        } else {
            // ---- baseline_policies/greedy_policy.py:64-88, waiting_policy.py:62-131 at randomness_factor 0 ----------
            // occupancy of the padded lattice, one word per row, private to the thread (walls are in the table)
            if constexpr (L::kDirtyBitmap) {   // the image(s) the bitmap aliases must have been read by the previous group's copies
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncwarp();
            }
            // (the bitmap is clean: zeroed at kernel start and after every use; where it aliases the image, zeroed here)
            if constexpr (L::kDirtyBitmap) {
#pragma unroll
                for (int r = 0; r < kT2MaxRows; ++r)
                    if (r < PH) sts32(bm + 128u * r, 0u);
            }
            unsigned arow[A];
#pragma unroll
            for (int k = 0; k < A; ++k) {
                arow[k] = bm + 128u + ((e[k].x >> 9) & 0x780u);                       // row y + 1
                CCB_CHECK(arow[k] >= bm + 128u && arow[k] + 128u < bm + 128u * (unsigned)PH && ((e[k].x >> 8) & 31u) + 2u <= 31u);
                if ((fl[k >> 2] >> (8 * (k & 3))) & 1u)                               // column x + 1
                    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(arow[k]), "r"(2u << ((e[k].x >> 8) & 31u)) : "memory");
            }
            // waiting_policy.py:118-131: some exiting agent that is not done has not arrived
            const unsigned nd0 = ~((fl[0] >> 1) | (fl[0] >> 2)) & m0e, nd1 = ~((fl[1] >> 1) | (fl[1] >> 2)) & m1e;
            const bool exiting_pending = p.policy == CC_POLICY_WAITING && ((((nd0 & ~boardw[0] & ~(fb[0] >> 7)) | (nd1 & ~boardw[1] & ~(fb[1] >> 7))) & kOnes) != 0u);
            // asks: active and not done (greedy_policy.py callers); waits: boarding agent outside the tram area (waiting_policy.py:74-108)
            unsigned go7[2];
            go7[0] = (fl[0] & nd0 & (exiting_pending ? ~(boardw[0] & ~(fb[0] >> 5)) : ~0u) & kOnes) << 7;
            go7[1] = (fl[1] & nd1 & (exiting_pending ? ~(boardw[1] & ~(fb[1] >> 5)) : ~0u) & kOnes) << 7;
#pragma unroll
            for (int k = 0; k < A; ++k) {
                // greedy_policy.py:238-264 -> _is_move_valid (collectivecrossing.py:345-369): walkable and not held by an ACTIVE agent
                const unsigned x = (e[k].x >> 8) & 31u;
                const unsigned here = lds32(arow[k]) >> x, above = lds32(arow[k] + 128u) >> x, below = lds32(arow[k] - 128u) >> x;
                // here: bit0 left, bit1 self, bit2 right; above / below: bit1
                const unsigned occ = (here & 5u) | (above & 2u) | ((below & 2u) << 2);
                const unsigned vmask = (e[k].x >> 24) & 15u & ~occ;
                unsigned a;
                CCB_CHECK((((e[k].x & 31u) << 4) | vmask) < (unsigned)(kPolicyRows * 16));
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(a) : "r"(act_s + (((e[k].x & 31u) << 4) | vmask)));
                const unsigned m = t2_fill(k < 4 ? go7[0] : go7[1], k & 3);
                act[k] = ((a ^ (unsigned)CC_ACT_WAIT) & m) ^ (unsigned)CC_ACT_WAIT;
            }
            if constexpr (!L::kDirtyBitmap) {
#pragma unroll
                for (int k = 0; k < A; ++k)
                    if ((fl[k >> 2] >> (8 * (k & 3))) & 1u) sts32(arow[k], 0u);
            }
            geo_known = true;
        }
        if (p.actions_out && env_ok) {
            auto a_ = [&](int k) { return act[k < A ? k : A - 1]; };
            const unsigned w0 = a_(0) | (a_(1) << 8) | (a_(2) << 16) | (a_(3) << 24), w1 = A > 4 ? (a_(4) | (a_(5) << 8) | (a_(6) << 16) | (a_(7) << 24)) : 0u;
            t2_store_packed<A, true>(p.actions_out + slice_a, n, w0, w1);
        }

        // ---- collectivecrossing.py:188 ------------------------------------------------------------------------------
        step += 1;
        // alive_prev: neither terminated nor truncated at step start (bytes 0x01)
        const unsigned alive0 = ~((fl[0] >> 1) | (fl[0] >> 2)) & m0e, alive1 = ~((fl[1] >> 1) | (fl[1] >> 2)) & m1e;

        // ---- collectivecrossing.py:197-202: moves, strictly in agent order -----------------------------------------------
        // cmp[k]: cell of an ACTIVE agent, else the ghost sentinel (inactive agents do not block, :536-541).  An agent that
        // must not move (wait, invalid, blocked by a wall, ghost) asks for its own cmp value and so finds it occupied.
        {
            const unsigned act7_0 = (fl[0] & kOnes) << 7, act7_1 = (fl[1] & kOnes) << 7;
            unsigned cmp[A], am[A];
#pragma unroll
            for (int k = 0; k < A; ++k) {
                am[k] = t2_fill(k < 4 ? act7_0 : act7_1, k & 3);
                cmp[k] = c[k] | ~am[k];
            }
            // one agent's turn: the target is committed unless some cmp value equals it — a chain of setp.eq.or on ONE predicate
            // (the compiler's own rendering of the same test is a compare + select per pair)
            auto turn = [&](const int k, const int d) {
                CCB_CHECK(act[k] <= 4u && (am[k] == 0u || c[k] + (unsigned)d < (unsigned)kT2MaxCells));
                const unsigned target = (c[k] + (unsigned)d) | ~am[k];
                auto cm = [&](int j) { return cmp[j < A ? j : 0]; };
                asm("{\n\t.reg .pred q;\n\t"
                    "setp.eq.u32 q, %1, %9;\n\tsetp.eq.or.u32 q, %2, %9, q;\n\tsetp.eq.or.u32 q, %3, %9, q;\n\tsetp.eq.or.u32 q, %4, %9, q;\n\t"
                    "setp.eq.or.u32 q, %5, %9, q;\n\tsetp.eq.or.u32 q, %6, %9, q;\n\tsetp.eq.or.u32 q, %7, %9, q;\n\tsetp.eq.or.u32 q, %8, %9, q;\n\t"
                    "selp.u32 %0, %10, %9, q;\n\t}"                                           // :406-408
                    : "=r"(cmp[k]) : "r"(cm(0)), "r"(cm(1)), "r"(cm(2)), "r"(cm(3)), "r"(cm(4)), "r"(cm(5)), "r"(cm(6)), "r"(cm(7)), "r"(target), "r"(cmp[k]));
            };
            if (geo_known) {
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    int d;
                    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(d) : "r"(dc_s + act[k] * 4u));
                    turn(k, d);
                }
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    int d;
                    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(d) : "r"(dc_s + act[k] * 4u));
                    d = ((e[k].x >> (20u + act[k])) & 1u) ? d : 0;   // :509-534 through the table (wait / invalid: d is 0 already)
                    turn(k, d);
                }
            }
#pragma unroll
            for (int k = 0; k < A; ++k) c[k] = (cmp[k] & am[k]) | (c[k] & ~am[k]);      // ghosts never move
        }

        // ---- :210-212 deactivate arrivals; rewards; terminated; truncated (4 agents per word) -------------------------------
#pragma unroll
        for (int k = 0; k < A; ++k) e[k] = lookup(c[k], k);
        t2_gather<A, 0>(e, fb);
        const unsigned arr0 = (fb[0] >> 7) & kM0, arr1 = (fb[1] >> 7) & kM1;           // :663-683 (y only)
        st_arrivals += __popc(arr0 & fl[0]) + __popc(arr1 & fl[1]);                     // active agents that arrive now (fl is 0 beyond the end)
        fl[0] &= ~arr0; fl[1] &= ~arr1;                                                 // types.py:46-51 (CC_F_ACTIVE == 1)
        const bool all_arrived = (((arr0 ^ kM0) | (arr1 ^ kM1)) == 0u);
        const bool over_limit = step >= p.max_steps;                                    // truncateds.py:61
        const bool all_mode = p.terminated_kind == CC_TERM_ALL_AT_DESTINATION;
        const unsigned tval0 = all_mode ? (all_arrived ? kM0 : 0u) : arr0, tval1 = all_mode ? (all_arrived ? kM1 : 0u) : arr1;   // terminateds.py:56-60,82
        const unsigned cval0 = over_limit ? alive0 : 0u, cval1 = over_limit ? alive1 : 0u;                                    // truncateds.py:57-61
        const unsigned pres0 = alive0 | (tval0 & ~(fl[0] >> 1)), pres1 = alive1 | (tval1 & ~(fl[1] >> 1));                    // collectivecrossing.py:243
        fl[0] |= (tval0 << 1) | (cval0 << 2); fl[1] |= (tval1 << 1) | (cval1 << 2);                                           // :229-241
        const unsigned of0 = fl[0] | (alive0 << 3) | (tval0 << 4) | (cval0 << 5) | ((pres0 & kOnes) << 6);
        const unsigned of1 = fl[1] | (alive1 << 3) | (tval1 << 4) | (cval1 << 5) | ((pres1 & kOnes) << 6);
        const bool any_alive = (alive0 | alive1) != 0u;
        const bool term_all = all_arrived;                          // :256
        const bool trunc_all = any_alive && over_limit;             // :257
        // rewards: the table value where the agent was alive at step start (rewards.py:65-66), else 0
        float rew[A];
        {
            const unsigned a7_0 = alive0 << 7, a7_1 = alive1 << 7;
#pragma unroll
            for (int k = 0; k < A; ++k) rew[k] = __uint_as_float(e[k].y & (t2_fill(k < 4 ? a7_0 : a7_1, k & 3)));
        }
        // reward sum of the env: the balanced float32 tree the other kernels and the oracle use
        float rsum;
        {
            constexpr int LPE = A <= 4 ? 4 : 8;
            float leaf[LPE];
#pragma unroll
            for (int l = 0; l < LPE; ++l) leaf[l] = l < A ? 0.f + rew[l < A ? l : 0] : 0.f;
#pragma unroll
            for (int w = LPE / 2; w >= 1; w >>= 1)
#pragma unroll
                for (int l = 0; l < w; ++l) leaf[l] = leaf[l] + leaf[l + w];
            rsum = leaf[0];
        }
        ep_ret += rsum;
        const bool done = term_all || trunc_all;
        unsigned eflags = (term_all ? CC_E_TERMINATED_ALL : 0u) | (trunc_all ? CC_E_TRUNCATED_ALL : 0u);

        // ---- outputs of the finished step -------------------------------------------------------------------------------
        if (env_ok) {
            float *rw = reinterpret_cast<float *>(p.reward) + slice_a + (size_t)n * A;
            if constexpr (A % 4 == 0) {
#pragma unroll
                for (int k = 0; k < A; k += 4) __stcs(reinterpret_cast<float4 *>(rw + k), make_float4(rew[k], rew[k + 1], rew[k + 2], rew[k + 3]));
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k) rw[k] = rew[k];
            }
            t2_store_packed<A, true>(p.agent_flags + slice_a, n, of0, of1);
            if (p.agent_info) {   // :248-254: in_tram_area | at_door << 1 | active << 2 | at_destination << 3
                const unsigned i0 = ((fb[0] >> 5) & 0x03030303u) | ((fb[0] >> 4) & 0x08080808u) | ((fl[0] & kOnes) << 2);
                const unsigned i1 = ((fb[1] >> 5) & 0x03030303u) | ((fb[1] >> 4) & 0x08080808u) | ((fl[1] & kOnes) << 2);
                t2_store_packed<A, true>(p.agent_info + slice_a, n, i0 & (kM0 * 15u), i1 & (kM1 * 15u));
            }
            st_rsum += (double)rsum;
        }
        const bool ended = env_ok && done && any_alive;             // the step the last agents finished on
        const unsigned ended_mask = __ballot_sync(kFull, ended);
        if (ended_mask) {                                           // rare: fold this warp's finished episodes into its slot
            const unsigned n_term = __popc(__ballot_sync(kFull, ended && term_all)), n_trunc = __popc(__ballot_sync(kFull, ended && trunc_all));
            unsigned len = ended ? (unsigned)step : 0u;
            double ret = ended ? (double)ep_ret : 0.0;
#pragma unroll
            for (int w = 16; w >= 1; w >>= 1) { len += __shfl_xor_sync(kFull, len, w); ret += __shfl_xor_sync(kFull, ret, w); }
            if (lane == 0) {
                red[kStEpisodes] += __popc(ended_mask); red[kStTermAll] += n_term; red[kStTruncAll] += n_trunc; red[kStEpLen] += len;
                red[kStEpRet] = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)red[kStEpRet]) + ret);
            }
        }

        // ---- collectivecrossing.py:91-150 reset(): rejection-sampled placement (auto-reset) ----------------------------------
        // Agent i's k-th candidate is Philox(seed; genv, t, RESET, i<<16|k); it takes the first candidate that passes the
        // geometric test and is not held by an agent j < i (cc_oracle.c:orc_reset_env).
        if (env_ok && done && p.auto_reset) {
            eflags |= CC_E_WAS_RESET;
            ep_ret = 0.f;
            step = 0;                                               // :97
          if constexpr (kNp) {
            // numpy mode: the env's generator (loaded and stored only here), placement of cc_reset_seeded_kernel
            Pcg64 g = np_load(p.gen[n]);
#pragma unroll
            for (int i = 0; i < A; ++i) {
                int px = 0, py = 0;
                const bool ok = np_place_agent(g, p, i < B, [&](int cx, int cy) {
                    const unsigned cell = (unsigned)((cy + 1) * PW + cx + 1);
                    bool free = true;
#pragma unroll
                    for (int j = 0; j < i; ++j) free = free && c[j] != cell;
                    return free;
                }, px, py);
                if (!ok) errbits |= kErrResetStuck;                 // cap hit: keep the last candidate
                c[i] = (unsigned)((py + 1) * PW + px + 1) & 255u;
            }
            p.gen[n] = np_save(g);
          } else {
#pragma unroll
            for (int i = 0; i < A; ++i) {
                unsigned cand = 0;
                bool ok = false;
                for (int attempt = 0; attempt < kResetAttemptCap && !ok; ++attempt) {
                    const U4 r = draw_at(p, t_rng, genv, kStreamReset, ((unsigned)i << 16) | (unsigned)attempt);
                    int cx, cy;
                    if (i < B) { cx = bounded(r.v0, p.W); cy = bounded(r.v1, p.D); }                                   // :103-117
                    else { cx = p.TL + bounded(r.v0, p.TR + 1 - p.TL); cy = p.D + bounded(r.v1, p.H - p.D); }            // :132-140
                    cand = (unsigned)((cy + 1) * PW + cx + 1);
                    CCB_CHECK(cand < (unsigned)(PW * PH));
                    const unsigned ge = tb.tab[(cand & 255u) * 2].x;
                    ok = (ge & kT2Valid) && !(i < B && (ge & kT2SpawnExcluded));
#pragma unroll
                    for (int j = 0; j < i; ++j) ok = ok && c[j] != cand;
                }
                if (!ok) errbits |= kErrResetStuck;                 // cap hit: keep the last candidate
                c[i] = cand & 255u;
            }
          }
            fl[0] = kM0; fl[1] = kM1;                               // everyone active, nobody done
#pragma unroll
            for (int k = 0; k < A; ++k) e[k] = lookup(c[k], k);
            t2_gather<A, 0>(e, fb);
        }
        if (env_ok) __stcs(reinterpret_cast<unsigned char *>(p.env_flags) + (size_t)tt * (size_t)p.slice_envs + n, (unsigned char)eflags);

        // ---- observations.py:43-94 from the post-step (post-reset) state ----------------------------------------------------
        if constexpr (OBS == CC_OBS_FP32) {
            // the env's row template [S_0a S_0b ... K1 K2 M] (cc_kernel_tpe.cuh), then the warp's 32 blocks through the TMA image ring
            using L1 = typename L::L1;
            float2 *tpl = reinterpret_cast<float2 *>(wsmem + lane * L1::TSB);
#pragma unroll
            for (int k = 0; k < A; ++k) {
                tpl[2 * k] = make_float2((float)(int)((e[k].x >> 8) & 0xffu), (float)(int)((e[k].x >> 16) & 0xfu));
                tpl[2 * k + 1] = make_float2(k < B ? 0.f : 1.f, (float)(int)(((k < 4 ? fl[0] : fl[1]) >> (8 * (k & 3))) & 1u));
            }
            __syncwarp();
            void *obs_t = static_cast<unsigned char *>(p.obs) + (size_t)tt * (size_t)p.slice_obs_bytes;
            tpe_emit_group_tma<A, CC_OBS_FP32>(lut, img_s, obs_t, g, envs_here, lane, kc);
            __syncwarp();
        } else if constexpr (OBS != CC_OBS_NONE) {
            // T_k = (x_k, y_k, type_k, active_k): the agent's block of every row (observations.py:80-91)
            unsigned T[A];
#pragma unroll
            for (int k = 0; k < A; ++k)
                T[k] = ((e[k].x >> 8) & 0x0fffu) | ((((k < 4 ? typew0 : typew1) >> (8 * (k & 3))) & 1u) << 16) | ((((k < 4 ? fl[0] : fl[1]) >> (8 * (k & 3))) & 1u) << 24);
            if constexpr (OBS == CC_OBS_TABLE) {
                if (env_ok) {
                    unsigned *dst = reinterpret_cast<unsigned *>(static_cast<unsigned char *>(p.obs) + (size_t)tt * (size_t)p.slice_obs_bytes) + (size_t)n * A;
                    if constexpr (A % 4 == 0) {
#pragma unroll
                        for (int k = 0; k < A; k += 4) __stcs(reinterpret_cast<uint4 *>(dst + k), make_uint4(T[k], T[k + 1], T[k + 2], T[k + 3]));
                    } else {
#pragma unroll
                        for (int k = 0; k < A; ++k) __stcs(dst + k, T[k]);
                    }
                }
            } else {
                // int8 rows of 8 agents.  Row i = [x_i y_i | DC D DL DR | T_0 .. T_7 with T_i = -1] is 38 bytes, so rows come in
                // pairs of 19 words: the even row starts word-aligned (its table is shifted by two bytes), the odd row's table
                // is word-aligned.  The thread's 8 rows are 19 16-byte vectors at stride 304 B: conflict-free (19 is odd).
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the image is free again
                __syncwarp();
                const unsigned K1 = (unsigned)(p.DC & 0xff) | ((unsigned)(p.D & 0xff) << 8), K2 = (unsigned)(p.DL & 0xff) | ((unsigned)(p.DR & 0xff) << 8);
                const unsigned KK = K1 | (K2 << 16);
                unsigned S[7];                                       // S_j = high half of T_j, low half of T_(j+1)
#pragma unroll
                for (int j = 0; j < 7; ++j) S[j] = __byte_perm(T[j], T[j + 1], 0x5432u);
                unsigned wv[76];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const int a = 2 * m, b = 2 * m + 1;              // the pair's even and odd row
                    unsigned *w = wv + 19 * m;
                    w[0] = (T[a] & 0xffffu) | (K1 << 16);            // x_a y_a DC D
                    // even row: DL DR T0.lo | S_0 .. S_6 | T7.hi (x_b y_b), with agent a's block masked
                    w[1] = K2 | ((a == 0 ? 0xffffu : (T[0] & 0xffffu)) << 16);
#pragma unroll
                    for (int j = 0; j < 7; ++j) w[2 + j] = (j == a - 1) ? (S[j] | 0xffff0000u) : ((j == a) ? (S[j] | 0x0000ffffu) : S[j]);
                    w[9] = (a == 7 ? 0xffffu : (T[7] >> 16)) | (T[b] << 16);   // ... T7.hi | x_b y_b  (a is even: a != 7)
                    w[10] = KK;                                      // DC D DL DR of the odd row
#pragma unroll
                    for (int j = 0; j < 8; ++j) w[11 + j] = j == b ? 0xffffffffu : T[j];
                }
                const unsigned dst_s = img_s + (unsigned)lane * (unsigned)L::kEnvBytes;
                CCB_CHECK(dst_s + 19u * 16u <= img_s + (unsigned)L::kBytesPerWarp && envs_here * L::kEnvBytes <= L::kImageBytes && (envs_here * L::kEnvBytes) % 16 == 0);
#pragma unroll
                for (int v = 0; v < 19; ++v)
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst_s + 16u * v), "r"(wv[4 * v]), "r"(wv[4 * v + 1]), "r"(wv[4 * v + 2]), "r"(wv[4 * v + 3]) : "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async-proxy read
                __syncwarp();
                if (lane == 0) {
                    unsigned char *dst = static_cast<unsigned char *>(p.obs) + (size_t)tt * (size_t)p.slice_obs_bytes + (size_t)g * 32 * L::kEnvBytes;
                    unsigned long long l2_evict_first;
                    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_evict_first));
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                                 ::"l"(dst), "r"(img_s), "r"((unsigned)(envs_here * L::kEnvBytes)), "l"(l2_evict_first) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
        }
      }   // steps of this launch

        // ---- write back the persistent state --------------------------------------------------------------------------------
        if (env_ok) {
            unsigned xw[2], yw[2];
            t2_gather<A, 1>(e, xw);
            t2_gather<A, 2>(e, yw);
            t2_store_packed<A, false>(p.x, n, xw[0], xw[1]);
            t2_store_packed<A, false>(p.y, n, yw[0] & 0x0f0f0f0fu, yw[1] & 0x0f0f0f0fu);
            t2_store_packed<A, false>(p.flags, n, fl[0], fl[1]);
            p.step[n] = step;
            p.ep_ret[n] = ep_ret;
        }
#if CCB_TPE_DYNAMIC
        g_next = __shfl_sync(kFull, g_next, 0);
#endif
    }

    if (L::kDirtyBitmap && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // shared memory stays valid until the copies are done
    // ---- statistics: per-warp slots in shared memory -> one atomic per slot per CTA -----------------------------------------
    {
        double rs = st_rsum;
        unsigned ar = st_arrivals;
#pragma unroll
        for (int w = 16; w >= 1; w >>= 1) { rs += __shfl_xor_sync(kFull, rs, w); ar += __shfl_xor_sync(kFull, ar, w); }
        if (lane == 0) {
            red[kStArrivals] += ar;
            red[kStRewardSum] = (unsigned long long)__double_as_longlong(rs);
        }
        __syncthreads();
        const unsigned long long *all = red_all;
        if (threadIdx.x >= 1 && threadIdx.x < 6) {
            unsigned long long v = 0;
            for (int w = 0; w < n_warps; ++w) v += all[w * kStCount + threadIdx.x];
            if (v) atomicAdd(&p.stats[threadIdx.x], v);
        } else if (threadIdx.x == 6 || threadIdx.x == 7) {
            double v = 0.0;
            for (int w = 0; w < n_warps; ++w) v += __longlong_as_double((long long)all[w * kStCount + threadIdx.x]);
            if (v != 0.0) atomicAdd(reinterpret_cast<double *>(&p.stats[threadIdx.x]), v);
        } else if (threadIdx.x == 0 && blockIdx.x == 0) {
            atomicAdd(&p.stats[kStEnvSteps], (unsigned long long)p.n_envs * (unsigned long long)p.n_steps);
        }
    }
    if (errbits) atomicOr(p.err, errbits);
}

}  // namespace ccb
