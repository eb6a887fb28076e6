// cc_kernel_tpe.cuh — the step kernel for small crews (A <= 8): one THREAD owns one env.
//
// Why a second mapping (DESIGN.md §3): with one lane per agent (cc_kernels.cuh) a README env costs
// ~160 warp-instructions per step and the kernel is bound by the issue rate, not by HBM.  For A <= 8
// the whole env fits in the registers of one thread, the reference's sequential move loop
// (collectivecrossing.py:197-202) becomes straight-line code, and a warp steps 32 envs with the
// instruction count the lane-group mapping needs for 4.  What is left is the byte traffic:
//   * state / actions / per-agent outputs: an env's A bytes are ONE 8-byte (A = 8) or 4-byte (A = 4)
//     word per thread — consecutive threads, consecutive words: coalesced without staging;
//   * observations (float32): every thread writes its env's 2A+3-pair row template into shared memory
//     (conflict-free 8-byte stores); then, env by env, the warp assembles the env's block of A rows in a
//     shared-memory image — lane l gathers output pairs l, l+32, ... through a per-CTA table of
//     template offsets — and one lane hands the image to the TMA unit (cp.async.bulk, SASS UBLKCP).
//     Stores issued with st.global would stall the SM's load/store pipe, and with it every other
//     warp's shared-memory work, whenever HBM pushes back (profiles/probes/lsu_coupling_probe.cu);
//   * a launch may run n_steps > 1 steps per env with the state in registers (cc_rollout_fused).
// Semantics, quirks and RNG streams are those of cc_kernels.cuh / oracle/cc_oracle.c; every block
// cites the reference lines it restates (paths relative to /root/reference/src/collectivecrossing/).
#pragma once
#include "cc_kernels.cuh"

#ifndef CCB_TPE_MIN_BLOCKS
#define CCB_TPE_MIN_BLOCKS 3   // resident CTAs per SM the register allocator must allow
#endif
#ifndef CCB_TPE_TMA
#define CCB_TPE_TMA 1          // float32 rows leave the SM through cp.async.bulk (TMA) instead of st.global, see DESIGN.md §3
#endif
#ifndef CCB_TPE_CONST_REGS
#define CCB_TPE_CONST_REGS 0   // TMA gather: 1 = lanes whose pair is K1 / K2 / M keep it in a register (predicated load, no bank
                               // conflicts, 4 instructions per pair); 0 = every lane loads from the template (1 instruction, 2-way conflicts)
#endif
#ifndef CCB_TPE_STATE_STREAM
#define CCB_TPE_STATE_STREAM 0 // state rows: 0 = default caching, 1 = streaming (evict-first) operators, 2 = L2 evict_last hints
                               // (measured, 1M envs: single-step launch 0.2423 / 0.2537 ms, fused 0.2014 / 0.2041 ms for 0 / 1)
#endif
#ifndef CCB_TPE_DYNAMIC
#define CCB_TPE_DYNAMIC 1      // warps take their next group of 32 envs from an atomic counter (no tail round, ascending writes)
#endif

namespace ccb {

constexpr int kTpeWarps = 8;
constexpr int kTpeThreads = kTpeWarps * 32;
constexpr int kTpeMaxBitmapWords = 16;   // private policy bitmaps up to 512 padded lattice points (16 KB per CTA)

constexpr int tpe_gcd(int a, int b) { return b == 0 ? a : tpe_gcd(b, a % b); }

template <int A, int OBS>
struct TpeLayout {
    using OT = typename std::conditional<OBS == CC_OBS_FP32, float, int8_t>::type;
    using P2 = typename PairOf<OT>::type;
    static constexpr bool kHasObs = OBS == CC_OBS_INT8 || OBS == CC_OBS_FP32;   // the reference's rows (CC_OBS_TABLE needs no staging)
    static constexpr int R = 3 + 2 * A;                  // pairs per observation row
    static constexpr int PPE = A * R;                    // pairs per env
    static constexpr int PSZ = (int)sizeof(P2);          // 8 (float32) or 2 (int8)
    static constexpr int PPV = 16 / PSZ;                 // pairs per 16-byte vector
    static constexpr bool kVectorisable = PPE % PPV == 0;
    static constexpr int VPE = PPE / PPV;                // 16-byte vectors per env
    // Row template of one env in shared memory: [S_0a, S_0b, ..., S_(A-1)a, S_(A-1)b, K1, K2, M], 2A+3 pairs.
    //   float32: 8-byte pairs, stride exactly 2A+3 pairs (an odd number of 8-byte units), written with
    //            8-byte stores: the 16 threads of a half-warp then hit 16 distinct bank pairs;
    //   int8:    2-byte pairs, stride an odd number of 4-byte words, written with 4-byte stores.
    // The constant pairs K1, K2, M are written once per kernel.
    static constexpr int TPL_PAIRS = 2 * A + 3;
    static constexpr int TSB = OBS == CC_OBS_FP32 ? TPL_PAIRS * 8 : (((TPL_PAIRS * PSZ + 3) / 4) | 1) * 4;
    // float32 rows are assembled env by env in a ring of kImgRing shared-memory images of one env's
    // observation block (A rows = kImgBytes) and leave the SM as bulk asynchronous copies (TMA): stores
    // issued with st.global stall the whole load/store pipe of the SM while HBM pushes back, and with it
    // the shared-memory work of the warps that are stepping envs (profiles/probes/lsu_coupling_probe.cu)
    static constexpr bool kTma = OBS == CC_OBS_FP32 && CCB_TPE_TMA != 0 && (PPE * PSZ) % 16 == 0;   // bulk copies move multiples of 16 bytes: even crews
    static constexpr int kImgBytes = PPE * PSZ;          // 1216 B for A = 8; a multiple of 16 whenever A is even
    static constexpr int kImgRing = 3;
    static constexpr int kImgInstr = (PPE + 31) / 32;    // warp instructions that cover an env's pairs
    static constexpr int kTplBytesPerWarp = kHasObs ? (32 * TSB + 15) / 16 * 16 : 0;
    static constexpr int kStageBytesPerWarp = kTplBytesPerWarp + (kTma ? kImgRing * kImgBytes : 0);
    static constexpr int kStageBytes = kTpeWarps * kStageBytesPerWarp;
    // Emission: the 32 envs of a warp are NB blocks of EB envs; a block is a whole number (JB) of
    // 32-unit rows, so unit j of lane l lies at the same place of every block and ONE table entry per
    // (j, lane) — the offset of its source from the block's first template — serves all blocks.
    //   float32: unit = one 8-byte pair (lane <-> pair).  A warp instruction gathers 32 CONSECUTIVE output
    //            pairs: but for the own position, the door constants and the masked block these are
    //            consecutive template pairs (2-way bank conflicts at most, none with CCB_TPE_CONST_REGS).
    //            With TMA rows the table has one entry per (j, lane) for ANY env (offset inside its template).
    //   int8:    unit = one 16-byte vector of 8 pairs.
    static constexpr bool kPairwise = OBS == CC_OBS_FP32;
    static constexpr int UPE = kPairwise ? PPE : VPE;    // emission units per env
    static constexpr int G = tpe_gcd(UPE > 0 ? UPE : 1, 32);
    static constexpr int NB = G, EB = 32 / G, JB = UPE / G;
    static constexpr int kLutEntryWords = kPairwise ? 1 : 4;   // one coded source, or 8 x 16-bit offsets
    static constexpr int kLutWords = kHasObs ? (kTma ? kImgInstr * 32 : JB * 32 * kLutEntryWords) : 4;
};

// Source of output pair q of row i (observations.py:62-94: own position, door constants, then every
// agent's block with the own block masked): index of a pair of the agent table S (>= 0), or one of the
// constant pairs.
enum { kSrcK1 = -1, kSrcK2 = -2, kSrcM = -3 };
template <int A>
__device__ __forceinline__ int tpe_source(int i, int q) {
    if (q == 0) return 2 * i;                     // (x_i, y_i) = S_ia
    if (q == 1) return kSrcK1;                    // (door centre, division)
    if (q == 2) return kSrcK2;                    // (door left, door right)
    return ((q - 3) >> 1) == i ? kSrcM : q - 3;   // (-1, -1) over the own block
}
// int8 template: byte offset of the pair feeding output pair P (0 .. A*R-1) of an env; constants follow the table
template <int A, int PSZ>
__device__ __forceinline__ unsigned tpe_pair_offset(int P) {
    constexpr int R = 3 + 2 * A;
    const int src = tpe_source<A>(P / R, P % R);
    return (unsigned)((src >= 0 ? src : 2 * A - 1 - src) * PSZ);
}

// A bytes of env `env` of an [N][A] byte array: one 8-byte (A = 8) or 4-byte (A = 4) word per thread, bytes otherwise.
// Loading (packed) and unpacking are separate so that the next group's record can be fetched early.
template <int A>
__device__ __forceinline__ uint2 tpe_fetch_row(const void *base, int env) {
    const unsigned char *q = static_cast<const unsigned char *>(base) + (size_t)env * A;
    if constexpr (A == 8) {
#if CCB_TPE_STATE_STREAM == 2
        uint2 w; unsigned long long pol;
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("ld.global.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(w.x), "=r"(w.y) : "l"(q), "l"(pol));
        return w;
#else
        return CCB_TPE_STATE_STREAM ? __ldcs(reinterpret_cast<const uint2 *>(q)) : *reinterpret_cast<const uint2 *>(q);
#endif
    }
    else if constexpr (A == 4) return make_uint2(CCB_TPE_STATE_STREAM == 1 ? __ldcs(reinterpret_cast<const unsigned *>(q)) : *reinterpret_cast<const unsigned *>(q), 0u);
    else {   // other crews: rows are not word-aligned, byte loads (the warp still covers one contiguous run of 32 A bytes)
        uint2 w = make_uint2(0u, 0u);
#pragma unroll
        for (int k = 0; k < A; ++k) (k < 4 ? w.x : w.y) |= (unsigned)q[k] << (8 * (k & 3));
        return w;
    }
}
template <int A>
__device__ __forceinline__ void tpe_unpack_row(uint2 w, unsigned (&v)[A]) {
#pragma unroll
    for (int k = 0; k < A; ++k) v[k] = ((k < 4 ? w.x : w.y) >> (8 * (k & 3))) & 0xffu;
}
// STREAM: per-step outputs are written once and not read again by the kernels: st.global.cs (evict first)
template <int A, bool STREAM = false>
__device__ __forceinline__ void tpe_store_row(void *base, int env, const unsigned (&v)[A]) {
    unsigned char *q = static_cast<unsigned char *>(base) + (size_t)env * A;
    if constexpr (A == 8) {
        uint2 w;
        w.x = (v[0] & 0xffu) | ((v[1] & 0xffu) << 8) | ((v[2] & 0xffu) << 16) | (v[3] << 24);
        w.y = (v[4] & 0xffu) | ((v[5] & 0xffu) << 8) | ((v[6] & 0xffu) << 16) | (v[7] << 24);
        if constexpr (STREAM) __stcs(reinterpret_cast<uint2 *>(q), w);
        else if constexpr (CCB_TPE_STATE_STREAM == 2) {
            unsigned long long pol;
            asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
            asm volatile("st.global.L2::cache_hint.v2.u32 [%0], {%1, %2}, %3;" ::"l"(q), "r"(w.x), "r"(w.y), "l"(pol) : "memory");
        } else *reinterpret_cast<uint2 *>(q) = w;
    } else if constexpr (A == 4) {
        const unsigned w = (v[0] & 0xffu) | ((v[1] & 0xffu) << 8) | ((v[2] & 0xffu) << 16) | (v[3] << 24);
        if constexpr (STREAM) __stcs(reinterpret_cast<unsigned *>(q), w);
        else *reinterpret_cast<unsigned *>(q) = w;
    } else {
#pragma unroll
        for (int k = 0; k < A; ++k) q[k] = (unsigned char)v[k];
    }
}

struct TpeConstPairs { uint2 k1, k2, m; };   // (DC, D), (DL, DR), (-1, -1) as float32 bit patterns

// ---------------------------------------------------------------------------------------------------
// float32 observation rows through TMA: the rows of the group whose templates sit in the warp's template
// buffer (`sbase`, shared address).  Every env's block (A rows) is assembled in one of kImgRing image
// buffers — lane l gathers pairs l, l+32, ... through the per-CTA offset table — and leaves the SM as
// ONE bulk asynchronous copy.  (Measured alternatives, DESIGN.md §5: spreading these envs over the phases
// of the next group's step as a software pipeline, 2 or 4 envs at a time, was slower — every
// fence.proxy.async is also a MEMBAR that drains the step's own loads and stores.)
// ---------------------------------------------------------------------------------------------------
template <int A, int OBS>
__device__ __forceinline__ void tpe_emit_group_tma(const unsigned *lut, unsigned sbase, void *obs, int g, int envs_here, int lane, const TpeConstPairs &kc) {
    using L = TpeLayout<A, OBS>;
    static_assert(L::kImgRing == 3, "the env loop is unrolled by the ring size");
    // src[j]: shared address, inside the template of the env being emitted, of the pair that feeds output
    // pair lane + 32 j (the same offsets for every env).  With CCB_TPE_CONST_REGS a lane whose pair is one of
    // the constants K1, K2, M (src = 0xFFFFFFFF) keeps it in val[j] for the whole group and makes no
    // shared-memory access, so the other lanes of a half-warp read consecutive template pairs without bank
    // conflicts; measured, the conflicts cost nothing and the predication 400 instructions per 32 envs.
    unsigned src[L::kImgInstr];
    unsigned long long val[L::kImgInstr];
#pragma unroll
    for (int j = 0; j < L::kImgInstr; ++j) {
        const unsigned d = lut[j * 32 + lane];
#if CCB_TPE_CONST_REGS
        src[j] = (d >> 31) ? 0xFFFFFFFFu : sbase + d;
        const uint2 c = (d & 3u) == 1u ? kc.k1 : ((d & 3u) == 2u ? kc.k2 : kc.m);
        val[j] = (unsigned long long)c.x | ((unsigned long long)c.y << 32);
#else
        src[j] = sbase + ((d >> 31) ? (unsigned)((2 * A - 1 + (int)(d & 3u)) * L::PSZ) : d);   // constants follow the agent table
        val[j] = 0ull;
#endif
    }
    const unsigned img0 = sbase + L::kTplBytesPerWarp;                   // image ring of this warp
    const unsigned islot = img0 + 8u * lane;                             // this lane's pair slot of image 0
    unsigned char *dst = static_cast<unsigned char *>(obs) + (size_t)g * 32 * L::kImgBytes;
    unsigned long long l2_evict_first;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_evict_first));
    auto emit_env = [&](const unsigned t_imm, const unsigned buf) {      // both compile-time after inlining
        // the image buffer is free once the bulk copy issued kImgRing envs ago has read it
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(L::kImgRing - 1) : "memory");
        __syncwarp();
#pragma unroll
        for (int j = 0; j < L::kImgInstr; ++j) {
#if CCB_TPE_CONST_REGS
            asm volatile("{\n\t.reg .pred pl;\n\tsetp.ne.u32 pl, %1, 0xFFFFFFFF;\n\t@pl ld.shared.b64 %0, [%2];\n\t}"
                         : "+l"(val[j]) : "r"(src[j]), "r"(src[j] + t_imm));
#else
            CCB_CHECK(src[j] + t_imm >= sbase && src[j] + t_imm + 8u <= sbase + (unsigned)L::kTplBytesPerWarp);
            asm volatile("ld.shared.b64 %0, [%1];" : "=l"(val[j]) : "r"(src[j] + t_imm));
#endif
            if (j * 32 + 32 <= L::PPE || lane + j * 32 < L::PPE)
                asm volatile("st.shared.b64 [%0], %1;" ::"r"(islot + buf + 256u * j), "l"(val[j]) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async-proxy read
        __syncwarp();
        CCB_CHECK(buf + (unsigned)L::kImgBytes <= (unsigned)(L::kImgRing * L::kImgBytes) && (reinterpret_cast<uintptr_t>(dst) & 15) == 0);
        if (lane == 0) {
            // (evict_first: the rows are written once and not read by this kernel; they must not push the state out of L2)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                         ::"l"(dst), "r"(img0 + buf), "n"(L::kImgBytes), "l"(l2_evict_first) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        dst += L::kImgBytes;
    };
    // a group starts on buffer 0 whatever the previous group ended on: all earlier copies must have been read
    // (they were issued a whole step ago; this does not wait in practice)
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    int e = 0;
    for (; e + 3 <= envs_here; e += 3) {
        emit_env(0u, 0u);
        emit_env((unsigned)L::TSB, (unsigned)L::kImgBytes);
        emit_env(2u * L::TSB, 2u * L::kImgBytes);
#pragma unroll
        for (int j = 0; j < L::kImgInstr; ++j) src[j] = (CCB_TPE_CONST_REGS && src[j] == 0xFFFFFFFFu) ? src[j] : src[j] + 3u * L::TSB;
    }
    if (e < envs_here) emit_env(0u, 0u);                                              // 32 = 10 x 3 + 2
    if (e + 1 < envs_here) emit_env((unsigned)L::TSB, (unsigned)L::kImgBytes);
}

// The same rows with st.global (CCB_TPE_TMA = 0): blocks [B0, B1) of the group, a
// block being EB envs = JB rows of 32 consecutive pairs (256 contiguous bytes per store instruction).
template <int A, int OBS, int B0, int B1>
__device__ __forceinline__ void tpe_emit_blocks_stg(const unsigned *lut, unsigned sbase, const unsigned char *wstage, void *obs, int g_prev,
                                                    int envs_prev, int lane) {
    using L = TpeLayout<A, OBS>;
    if (g_prev < 0) return;                              // warp-uniform
    uint2 *outp = reinterpret_cast<uint2 *>(obs) + (size_t)g_prev * 32 * L::PPE + lane;
    if (envs_prev == 32) {
#pragma unroll
        for (int j = 0; j < L::JB; ++j) {
            const unsigned a0 = sbase + lut[j * 32 + lane];
#pragma unroll
            for (int b = B0; b < B1; ++b) {
                uint2 o;
                asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(o.x), "=r"(o.y) : "r"(a0 + (unsigned)(b * L::EB * L::TSB)));
                __stcs(outp + b * L::EB * L::PPE + 32 * j, o);
            }
        }
    } else if (B0 == 0) {
        // ragged last group of a launch: plain index arithmetic, once, at most one warp per launch
        const int npair = envs_prev * L::PPE;
        for (int v = lane; v < npair; v += 32) {
            const int e = v / L::PPE, r = v % L::PPE;
            __stcs(outp + (v - lane), *reinterpret_cast<const uint2 *>(wstage + e * L::TSB + tpe_pair_offset<A, L::PSZ>(r)));
        }
    }
}

// OBSF: the obs dtype, with kNpReset for numpy-mode auto-reset placements
template <int A, int OBSF>
__global__ void __launch_bounds__(kTpeThreads, CCB_TPE_MIN_BLOCKS) cc_step_tpe_kernel(const __grid_constant__ KParams p) {
    constexpr int OBS = OBSF & ~kNpReset;
    constexpr bool kNp = (OBSF & kNpReset) != 0;
    using L = TpeLayout<A, OBS>;
    using OT = typename L::OT;
    using P2 = typename L::P2;
    constexpr bool kHasObs = L::kHasObs;
    constexpr unsigned kGhost = 0xFFFFFFFFu;
    static_assert(A >= 1 && A <= 8, "thread-per-env mapping is for crews of at most 8");
    static_assert(OBS != CC_OBS_INT8 || L::kVectorisable, "an env's observation block must be a whole number of 16-byte vectors");
    extern __shared__ __align__(16) unsigned char smem[];   // row templates: [warp][32 envs][TSB]

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int PW = p.W + 3, PH = p.H + 3;  // lattice padded by one ring: x in [-1, W+1] -> column x+1
    __shared__ unsigned xt[kMaxPad], yt[2 * kMaxPad], walk[kMaxWalkWords];
    __shared__ unsigned walk_row[kTpeMaxBitmapWords];   // row y of the padded lattice as one word (lattices up to 32 columns)
    __shared__ float rtab[kRtabSize];   // value for a boarding agent; exiting agents of the default reward get the negative
    __shared__ uint8_t act_tab[kPolicyRows * 16];
    __shared__ unsigned long long red_all[kTpeWarps * kStCount];
    __shared__ __align__(16) unsigned lut[L::kLutWords];   // emission table, see TpeLayout
    unsigned char *wstage = smem + warp * L::kStageBytesPerWarp;   // this warp's 32 templates
    unsigned char *tpl = wstage + lane * L::TSB;                    // this thread's env
    // private lattice bitmap of the policies: word w of this thread at bm[w * kBmStride].  With TMA rows it
    // lives in the warp's image ring, which is idle while the warp steps its envs (kBmStride = 32 lanes);
    // otherwise in its own region behind the templates (kBmStride = threads of the CTA).
    constexpr int kBmStride = L::kTma ? 32 : kTpeThreads;
    unsigned *bm_ptr = L::kTma ? reinterpret_cast<unsigned *>(wstage + L::kTplBytesPerWarp) + lane
                               : reinterpret_cast<unsigned *>(smem + L::kStageBytes) + threadIdx.x;
    // (accessed through its 32-bit shared-space address: the word index is data dependent, and generic 64-bit
    // address arithmetic per access was a fifth of the policy's instructions)
    const unsigned bm = (unsigned)__cvta_generic_to_shared(bm_ptr);
    constexpr unsigned kBmWord = 4u * kBmStride;   // bytes between consecutive words of one thread
    // (checked build: a word of the private bitmap lies inside the region it aliases — the warp's image ring — or its own)
    auto bm_load = [&](unsigned word) { CCB_CHECK((int)word < p.tpe_bm_words && (!L::kTma || (word + 1) * kBmWord <= (unsigned)(L::kImgRing * L::kImgBytes))); unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(bm + word * kBmWord)); return v; };
    auto bm_store = [&](unsigned word, unsigned v) { CCB_CHECK((int)word < p.tpe_bm_words && (!L::kTma || (word + 1) * kBmWord <= (unsigned)(L::kImgRing * L::kImgBytes))); asm volatile("st.shared.u32 [%0], %1;" ::"r"(bm + word * kBmWord), "r"(v) : "memory"); };

    // ---- once per CTA: tables (same contents as cc_kernels.cuh) -------------------------------------
    for (int i = threadIdx.x; i < PW; i += blockDim.x) xt[i] = make_xt(p, i - 1);
    for (int i = threadIdx.x; i < 2 * PH; i += blockDim.x) yt[(i / PH) * kMaxPad + i % PH] = make_yt(p, i / PH, i % PH - 1);
    for (int i = threadIdx.x; i < kPolicyRows * 16; i += blockDim.x) act_tab[i] = (uint8_t)greedy_decision(i >> 4, (unsigned)i & 15u);
    {
        // distance rewards: float((double)(-+d) * f), the reference's float64 product rounded once
        // (rewards.py:85,99,127); constants for binary / constant_negative (rewards.py:152-159,179-182)
        const double f = p.reward_kind == CC_REWARD_DEFAULT ? p.rp[3] : p.rp[0];
        for (int i = threadIdx.x; i < kRtabSize; i += blockDim.x) {
            const int d = i - kYBias;
            float v = (float)((double)(-d) * f);      // boarding / simple distance; exiting (default): float((double)d * f) = 0 - v exactly
            if (p.reward_kind == CC_REWARD_BINARY) v = p.rpf[1];
            if (p.reward_kind == CC_REWARD_CONSTANT_NEGATIVE) v = p.rpf[0];
            rtab[i] = v;
        }
    }
    // collectivecrossing.py:509-534 as a bitmap of the padded lattice: a warp builds one word per ballot
    for (int w = warp; w < p.walk_words; w += kTpeWarps) {
        const int idx = w * 32 + lane, yy = idx / PW - 1, xx = idx - (yy + 1) * PW - 1;
        const unsigned bits = __ballot_sync(kFull, valid_position(p, xx, yy));
        if (lane == 0) walk[w] = bits;
    }
    if (p.tpe_bm_rows && threadIdx.x < PH) {
        unsigned bits = 0;
        for (int c = 0; c < PW; ++c) bits |= valid_position(p, c - 1, (int)threadIdx.x - 1) ? (1u << c) : 0u;
        walk_row[threadIdx.x] = bits;
    }
    if (kHasObs) {
        for (int w = threadIdx.x; w < L::kLutWords; w += blockDim.x) {
            // entry (j, lane) describes unit v = lane + 32 j of a block: env e = v / UPE, unit r = v % UPE of that env
            const int entry = w / L::kLutEntryWords, part = w % L::kLutEntryWords;
            const int v = (entry & 31) + 32 * (entry >> 5), e = v / (L::UPE > 0 ? L::UPE : 1), r = v % (L::UPE > 0 ? L::UPE : 1);
            if (L::kTma) {
                // entry (j, lane): pair w = lane + 32 j of ANY env (offset inside that env's template)
                const int src = w < L::PPE ? tpe_source<A>(w / L::R, w % L::R) : kSrcM;
                lut[w] = src >= 0 ? (unsigned)(src * L::PSZ) : (0x80000000u | (unsigned)(-src));
            } else if (L::kPairwise) {
                lut[w] = (unsigned)(e * L::TSB) + tpe_pair_offset<A, L::PSZ>(r);
            } else {
                lut[w] = ((unsigned)(e * L::TSB) + tpe_pair_offset<A, L::PSZ>(8 * r + 2 * part)) |
                         (((unsigned)(e * L::TSB) + tpe_pair_offset<A, L::PSZ>(8 * r + 2 * part + 1)) << 16);
            }
        }
        {   // the constant pairs of this thread's template
            P2 *t = reinterpret_cast<P2 *>(tpl);
            t[2 * A] = mk_pair<OT>(p.DC, p.D); t[2 * A + 1] = mk_pair<OT>(p.DL, p.DR); t[2 * A + 2] = mk_pair<OT>(-1, -1);
        }
    }
    const TpeConstPairs kc = {make_uint2(__float_as_uint((float)p.DC), __float_as_uint((float)p.D)),
                              make_uint2(__float_as_uint((float)p.DL), __float_as_uint((float)p.DR)),
                              make_uint2(__float_as_uint(-1.f), __float_as_uint(-1.f))};
    unsigned long long *red = red_all + warp * kStCount;
    if (lane < kStCount) red[lane] = 0ull;
    if (blockIdx.x == 0 && threadIdx.x == 0) *p.tpe_counter_next = 0u;   // the counter the NEXT launch uses
    __syncthreads();
    unsigned st_arrivals = 0;
    double st_rsum = 0.0;
    int errbits = 0;

    const int total_warps = (int)gridDim.x * kTpeWarps;
    const int n_groups = (int)p.n_groups;   // groups of 32 envs
    // Work distribution: every warp starts on group (its global index); later groups come from an
    // atomic counter, fetched one iteration ahead so that the round trip is hidden.  Compared with a
    // fixed stride this has no partially filled last round, and the groups in flight stay a compact,
    // ascending window of the output (profiles/probes/store_pattern_probe.cu: 6.2 -> 6.9 TB/s).
    // (De-phasing the warps of an SM at launch with a per-warp delay was measured: no effect.)
    // The record of a group: one word per byte row, step counter, return.  (Fetching it one group ahead,
    // before the previous group's rows are streamed out, was measured: no gain, 10 more live registers.)
    struct Record { uint2 x, y, fl; int step; float ep_ret; };
    auto fetch = [&](int gg, Record &r) {
        const long long n = (long long)gg * 32 + lane;
        const int nl = n < p.n_envs ? (int)n : (int)p.n_envs - 1;    // threads beyond the end re-read the last env (never stored)
        r.x = tpe_fetch_row<A>(p.x, nl);
        r.y = tpe_fetch_row<A>(p.y, nl);
        r.fl = tpe_fetch_row<A>(p.flags, nl);
        r.step = CCB_TPE_STATE_STREAM == 1 ? __ldcs(p.step + nl) : p.step[nl];
        r.ep_ret = CCB_TPE_STATE_STREAM == 1 ? __ldcs(p.ep_ret + nl) : p.ep_ret[nl];
    };
    // Work items are handed out in ascending order; with tpe_reverse (every other single-step launch) item w is
    // group n_groups-1-w, so a launch starts on the groups the previous launch wrote LAST — the part of the
    // state that is still in L2.
    int gw = (int)blockIdx.x * kTpeWarps + warp;
    int g_next = 0;
    Record rec;
    for (; gw < n_groups; gw = g_next) {
        const int g = p.tpe_reverse ? n_groups - 1 - gw : gw;
        fetch(g, rec);
#if CCB_TPE_DYNAMIC
        if (lane == 0) g_next = total_warps + (int)atomicAdd(p.tpe_counter, 1u);
#else
        g_next = gw + total_warps;
#endif
        const int n = g * 32 + lane;
        const int envs_here = (int)min(32ll, p.n_envs - (long long)g * 32);
        const bool env_ok = lane < envs_here;                 // false only in the ragged last group
        const unsigned long long genv = p.genv_offset + (unsigned long long)n;

        // ---- the env's record: in registers for all the steps this launch takes (cc_rollout_fused: n_steps > 1) ----
        unsigned pos[A], fl[A];
        {
            unsigned px[A], py[A];
            tpe_unpack_row<A>(rec.x, px);
            tpe_unpack_row<A>(rec.y, py);
            tpe_unpack_row<A>(rec.fl, fl);
#pragma unroll
            for (int k = 0; k < A; ++k) { pos[k] = (px[k] << 8) | py[k]; fl[k] = env_ok ? fl[k] : 0u; }
        }
        int step = rec.step;
        float ep_ret = rec.ep_ret;
      for (int tt = 0; tt < p.n_steps; ++tt) {   // (body indented as one step: time slice tt of every output)
        const size_t slice_a = (size_t)tt * (size_t)p.slice_agents;   // offset of slice tt in a per-agent array (elements)
        const unsigned t_rng = p.t + (unsigned)tt;                     // RNG counter word of this step
        unsigned action[A];
        if (p.policy == CC_POLICY_EXTERNAL) tpe_unpack_row<A>(tpe_fetch_row<A>(p.actions + slice_a, env_ok ? n : (int)p.n_envs - 1), action);
        else {
#pragma unroll
            for (int k = 0; k < A; ++k) action[k] = CC_ACT_WAIT;
        }

        int cell[A];
        unsigned geo_u[A], geo_f[A];
        auto lookup = [&](int k) {
            // (clamped to the lattice: set_state promises in-lattice positions, the clamp only keeps the
            // table and bitmap reads of garbage in bounds — all four neighbours lie in the padded lattice)
            const int cx = min((int)(pos[k] >> 8), p.W) + 1, cy = min((int)(pos[k] & 0xffu), p.H) + 1;
            CCB_CHECK(cx >= 1 && cx <= p.W + 1 && cy >= 1 && cy <= p.H + 1);
            const unsigned xv = xt[cx], yv = yt[(k < p.B ? 0 : kMaxPad) + cy];
            cell[k] = cy * PW + cx;
            geo_u[k] = yv + xv;
            geo_f[k] = (yv & xv) >> 24;
        };
        auto walkable = [&](int c) { return (walk[(c >> 5) & (kMaxWalkWords - 1)] >> (c & 31)) & 1u; };
        // cmp[k] = packed position of an ACTIVE agent, else a sentinel no target can equal: inactive
        // agents are ghosts (collectivecrossing.py:536-541)
        unsigned cmp[A];
#pragma unroll
        for (int k = 0; k < A; ++k) cmp[k] = (fl[k] & CC_F_ACTIVE) ? pos[k] : kGhost;
        auto occupied = [&](unsigned target) {
            bool hit = false;
#pragma unroll
            for (int j = 0; j < A; ++j) hit |= cmp[j] == target;
            return hit;
        };

        // ---- on-device policies (baseline_policies/*.py at randomness_factor 0) --------------------
        bool geo_known = false;   // chosen moves already passed the geometric test
        if (p.policy == CC_POLICY_RANDOM) {
#pragma unroll
            for (int k = 0; k < A; ++k) {
                action[k] = (unsigned)bounded(draw_at(p, t_rng, genv, kStreamAction, (unsigned)k).v0, 5);
                lookup(k);
            }
        } else if (p.policy != CC_POLICY_EXTERNAL) {
            bool pending = false;
#pragma unroll
            for (int k = 0; k < A; ++k) {
                lookup(k);
                // waiting_policy.py:118-131: some exiting agent that is not done has not arrived
                pending |= k >= p.B && (fl[k] & 6u) == 0u && env_ok && !(geo_f[k] & 8u);
            }
            const bool exiting_pending = p.policy == CC_POLICY_WAITING && pending;
            // validity of the four moves of every agent (greedy_policy.py:238-264 -> _is_move_valid,
            // collectivecrossing.py:345-369): a walkable target that no ACTIVE agent holds (the asking
            // agent's own cell is never one of its targets)
            unsigned vmask[A];
            if (p.tpe_bm_words > 0) {
                // small lattice: the thread keeps a private bitmap "wall or occupied" of the padded
                // lattice in shared memory (word w at bm[w * kBmStride]: a thread only ever touches
                // its own bank), so a move is valid iff ONE bit is clear
                if constexpr (L::kTma) {   // the ring must have been read by the previous group's copies (issued long ago)
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    __syncwarp();
                }
                if (p.tpe_bm_rows) {
                    // lattices of at most 32 padded columns: ONE word per row, so an agent at (cx, cy) reads the three
                    // rows around it once and tests four bits (cell = cy * PW + cx)
                    for (int w = 0; w < p.tpe_bm_words; ++w) bm_store((unsigned)w, ~walk_row[w]);
#pragma unroll
                    for (int k = 0; k < A; ++k)
                        if (fl[k] & CC_F_ACTIVE) {
                            const unsigned cy = min(pos[k] & 0xffu, (unsigned)p.H) + 1u, cx = min(pos[k] >> 8, (unsigned)p.W) + 1u;
                            bm_store(cy, bm_load(cy) | (1u << cx));
                        }
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        const unsigned cy = min(pos[k] & 0xffu, (unsigned)p.H) + 1u, cx = min(pos[k] >> 8, (unsigned)p.W) + 1u;
                        const unsigned below = bm_load(cy - 1u), here = bm_load(cy), above = bm_load(cy + 1u);
                        const unsigned blocked = ((here >> (cx + 1u)) & 1u) | (((above >> cx) & 1u) << 1) | (((here >> (cx - 1u)) & 1u) << 2) | (((below >> cx) & 1u) << 3);
                        vmask[k] = blocked ^ 15u;
                    }
                } else {
                    for (int w = 0; w < p.tpe_bm_words; ++w) bm_store((unsigned)w, ~walk[w]);
#pragma unroll
                    for (int k = 0; k < A; ++k)
                        if (fl[k] & CC_F_ACTIVE) bm_store((unsigned)cell[k] >> 5, bm_load((unsigned)cell[k] >> 5) | (1u << (cell[k] & 31)));
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        const int c = cell[k];
                        auto blocked = [&](int idx) { return (bm_load((unsigned)idx >> 5) >> (idx & 31)) & 1u; };
                        vmask[k] = (blocked(c + 1) | (blocked(c + PW) << 1) | (blocked(c - 1) << 2) | (blocked(c - PW) << 3)) ^ 15u;
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    const int c = cell[k];
                    const unsigned q = pos[k];
                    const unsigned v0 = walkable(c + 1) & (unsigned)!occupied((q + 0x100u) & 0xffffu);
                    const unsigned v1 = walkable(c + PW) & (unsigned)!occupied((q + 1u) & 0xffffu);
                    const unsigned v2 = walkable(c - 1) & (unsigned)!occupied((q - 0x100u) & 0xffffu);
                    const unsigned v3 = walkable(c - PW) & (unsigned)!occupied((q - 1u) & 0xffffu);
                    vmask[k] = v0 | (v1 << 1) | (v2 << 2) | (v3 << 3);
                }
            }
#pragma unroll
            for (int k = 0; k < A; ++k) {
                CCB_CHECK((((geo_u[k] & 0xffu) << 4) | vmask[k]) < kPolicyRows * 16);
                const unsigned a = act_tab[((geo_u[k] & 0xffu) << 4) | vmask[k]];
                const bool asks = (fl[k] & 7u) == CC_F_ACTIVE;                         // active, not done
                const bool waits = exiting_pending && k < p.B && !(geo_f[k] & 1u);    // waiting_policy.py:74-108
                action[k] = (asks && !waits) ? a : (unsigned)CC_ACT_WAIT;
            }
            geo_known = true;
        } else {
#pragma unroll
            for (int k = 0; k < A; ++k) lookup(k);
        }
        if (p.actions_out && env_ok) tpe_store_row<A, true>(p.actions_out + slice_a, n, action);

        // ---- collectivecrossing.py:188 ---------------------------------------------------------------
        step += 1;
        unsigned alive_prev[A];   // 1 iff neither terminated nor truncated at step start
#pragma unroll
        for (int k = 0; k < A; ++k) alive_prev[k] = (env_ok && (fl[k] & 6u) == 0u) ? 1u : 0u;

        // ---- collectivecrossing.py:197-202: moves, strictly in agent order ----------------------
#pragma unroll
        for (int k = 0; k < A; ++k) {
            const unsigned a = action[k];
            if (env_ok && a > 4u) errbits |= kErrInvalidAction;                          // :707-711
            // packed (dx << 8 | dy) mod 2^16 of actions 0..3 (actions.py:18-24)
            const unsigned delta = (unsigned)((0xFFFFFF0000010100ull >> (16 * (a & 3u))) & 0xffffull);
            bool go = (fl[k] & CC_F_ACTIVE) && a < 4u;                                   // :398, wait
            if (!geo_known) go = go && walkable(cell[k] + ((a & 1u) ? PW : 1) * ((a & 2u) ? -1 : 1));  // :509-534
            const unsigned target = (pos[k] + delta) & 0xffffu;
            if (go && !occupied(target)) cmp[k] = target;                                // :406-408
        }
#pragma unroll
        for (int k = 0; k < A; ++k) pos[k] = (fl[k] & CC_F_ACTIVE) ? cmp[k] : pos[k];    // ghosts never move

        // ---- :210-212 deactivate arrivals; rewards; terminated; truncated ----------------------
        unsigned arr[A];
        bool all_arrived = true;
#pragma unroll
        for (int k = 0; k < A; ++k) {
            lookup(k);                                             // geometry of the post-move cell
            arr[k] = (geo_f[k] >> 3) & 1u;                         // :663-683 (y only)
            st_arrivals += (env_ok && arr[k] && (fl[k] & CC_F_ACTIVE)) ? 1u : 0u;
            fl[k] &= ~arr[k];                                      // types.py:46-51 (CC_F_ACTIVE == 1)
            all_arrived = all_arrived && arr[k];
        }
        const bool over_limit = step >= p.max_steps;               // truncateds.py:61
        bool any_alive = false;
        float rew[A];
        unsigned oflag[A];
#pragma unroll
        for (int k = 0; k < A; ++k) {
            // one path for the four reward functions, see cc_kernels.cuh (rewards.py:65-66,78-99,127,152-159,179-182)
            const unsigned f = geo_f[k];
            CCB_CHECK((int)((geo_u[k] >> 8) & 0x1ffu) < kRtabSize);
            float r = rtab[(int)((geo_u[k] >> 8) & 0x1ffu)];
            if (k >= p.B && p.reward_kind == CC_REWARD_DEFAULT) r = 0.f - r;   // rewards.py:95-99: the exiting term is positive (sic)
            const bool boarding = k < p.B;
            const float special = boarding ? ((f & 2u) ? p.rpf[1] : p.rpf[2]) : p.rpf[2];
            const unsigned in_special = boarding ? (f & 3u) : ((f & 1u) ^ 1u);
            r = (in_special & p.reward_category_mask) ? special : r;
            r = (f & 8u & p.reward_category_mask) ? p.rpf[0] : r;
            r = alive_prev[k] ? r : 0.f;
            rew[k] = r;
            any_alive |= alive_prev[k] != 0u;
            const unsigned tval = (p.terminated_kind == CC_TERM_ALL_AT_DESTINATION) ? (unsigned)all_arrived : arr[k];  // terminateds.py:56-60,82
            const unsigned cval = alive_prev[k] & (unsigned)over_limit;                   // truncateds.py:57-61
            const unsigned present = alive_prev[k] | (tval & ~(fl[k] >> 1) & 1u);         // collectivecrossing.py:243
            fl[k] |= (tval << 1) | (cval << 2);                                           // :229-241
            oflag[k] = (fl[k] & 7u) | (alive_prev[k] << 3) | (tval << 4) | (cval << 5) | (present << 6);
        }
        const bool term_all = all_arrived;                          // :256
        const bool trunc_all = any_alive && over_limit;             // :257
        // reward sum of the env: the balanced float32 tree the lane-group kernel and the oracle use
        // (leaves = lanes of a 4- or 8-lane tile, missing leaves 0)
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

        // ---- outputs of the finished step ----------------------------------------------------------
        if (env_ok) {
            float *rw = reinterpret_cast<float *>(p.reward) + slice_a + (size_t)n * A;
            if constexpr (A % 4 == 0) {
#pragma unroll
                for (int k = 0; k < A; k += 4) __stcs(reinterpret_cast<float4 *>(rw + k), make_float4(rew[k], rew[k + 1], rew[k + 2], rew[k + 3]));
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k) rw[k] = rew[k];
            }
            tpe_store_row<A, true>(p.agent_flags + slice_a, n, oflag);
            if (p.agent_info) {
                unsigned info[A];
#pragma unroll
                for (int k = 0; k < A; ++k) info[k] = (geo_f[k] & 0xBu) | ((fl[k] & 1u) << 2);   // :248-254
                tpe_store_row<A, true>(p.agent_info + slice_a, n, info);
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

        // ---- collectivecrossing.py:91-150 reset(): rejection-sampled placement (auto-reset) -------
        // Agent i's k-th candidate is Philox(seed; genv, t, RESET, i<<16|k); it takes the first candidate
        // that passes the geometric test and is not held by an agent j < i (cc_oracle.c:orc_reset_env).
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
                const bool ok = np_place_agent(g, p, i < p.B, [&](int cx, int cy) {
                    bool free = true;
#pragma unroll
                    for (int j = 0; j < i; ++j) free = free && pos[j] != pack_pos(cx, cy);
                    return free;
                }, px, py);
                if (!ok) errbits |= kErrResetStuck;                 // cap hit: keep the last candidate
                pos[i] = pack_pos(px, py);
                fl[i] = CC_F_ACTIVE;
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
                    if (i < p.B) {                                  // :103-117
                        cx = bounded(r.v0, p.W); cy = bounded(r.v1, p.D);
                        ok = valid_position(p, cx, cy) && !(p.DL <= cx && cx <= p.DR && cy == p.D - 1);
                    } else {                                        // :132-140
                        cx = p.TL + bounded(r.v0, p.TR + 1 - p.TL); cy = p.D + bounded(r.v1, p.H - p.D);
                        ok = valid_position(p, cx, cy);
                    }
                    cand = pack_pos(cx, cy);
#pragma unroll
                    for (int j = 0; j < i; ++j) ok = ok && pos[j] != cand;
                }
                if (!ok) errbits |= kErrResetStuck;                 // cap hit: keep the last candidate
                pos[i] = cand;
                fl[i] = CC_F_ACTIVE;
            }
          }
        }

        if (env_ok) __stcs(reinterpret_cast<unsigned char *>(p.env_flags) + (size_t)tt * (size_t)p.slice_envs + n, (unsigned char)eflags);
#pragma unroll
        for (int k = 0; k < A; ++k) fl[k] &= 7u;

        // ---- CC_OBS_TABLE: (x_j, y_j, type_j, active_j) of observations.py:80-91 from the post-step (post-reset) state,
        // one 32-bit word per agent: an env's 4A bytes leave the thread as 16-byte vectors (A = 4, 8) or words ----
        if constexpr (OBS == CC_OBS_TABLE) {
            if (env_ok) {
                unsigned tw[A];
#pragma unroll
                for (int k = 0; k < A; ++k) tw[k] = (pos[k] >> 8) | ((pos[k] & 0xffu) << 8) | ((k < p.B ? 0u : 1u) << 16) | ((fl[k] & 1u) << 24);
                unsigned *dst = reinterpret_cast<unsigned *>(static_cast<unsigned char *>(p.obs) + (size_t)tt * (size_t)p.slice_obs_bytes) + (size_t)n * A;
                if constexpr (A % 4 == 0) {
#pragma unroll
                    for (int k = 0; k < A; k += 4) __stcs(reinterpret_cast<uint4 *>(dst + k), make_uint4(tw[k], tw[k + 1], tw[k + 2], tw[k + 3]));
                } else {
#pragma unroll
                    for (int k = 0; k < A; ++k) __stcs(dst + k, tw[k]);
                }
            }
        }

        // ---- observations.py:43-94 from the post-step (post-reset) state --------------------------
        if (kHasObs) {
            if constexpr (OBS == CC_OBS_FP32) {
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    reinterpret_cast<float2 *>(tpl)[2 * k] = make_float2((float)(int)(pos[k] >> 8), (float)(int)(pos[k] & 0xffu));
                    reinterpret_cast<float2 *>(tpl)[2 * k + 1] = make_float2(k < p.B ? 0.f : 1.f, (float)(fl[k] & 1u));
                }
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k)
                    reinterpret_cast<unsigned *>(tpl)[k] = (pos[k] >> 8) | ((pos[k] & 0xffu) << 8) | ((k < p.B ? 0u : 1u) << 16) | ((fl[k] & 1u) << 24);
            }
            __syncwarp();
            const unsigned sbase = (unsigned)__cvta_generic_to_shared(wstage);
            void *obs_t = static_cast<unsigned char *>(p.obs) + (size_t)tt * (size_t)p.slice_obs_bytes;
            if constexpr (L::kTma) {
                tpe_emit_group_tma<A, OBS>(lut, sbase, obs_t, g, envs_here, lane, kc);
            } else if constexpr (L::kPairwise) {
                tpe_emit_blocks_stg<A, OBS, 0, L::NB>(lut, sbase, wstage, obs_t, g, envs_here, lane);
            } else {
                uint4 *outv = reinterpret_cast<uint4 *>(obs_t) + (size_t)g * 32 * L::VPE + lane;
                if (envs_here == 32) {
#pragma unroll
                    for (int j = 0; j < L::JB; ++j) {
                        const uint4 d = reinterpret_cast<const uint4 *>(lut)[j * 32 + lane];
#pragma unroll
                        for (int b = 0; b < L::NB; ++b) {
                            auto two = [&](unsigned w) {
                                unsigned short lo, hi;
                                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(lo) : "r"(sbase + (w & 0xffffu) + (unsigned)(b * L::EB * L::TSB)));
                                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(hi) : "r"(sbase + (w >> 16) + (unsigned)(b * L::EB * L::TSB)));
                                return (unsigned)lo | ((unsigned)hi << 16);
                            };
                            __stcs(outv + b * L::EB * L::VPE + 32 * j, make_uint4(two(d.x), two(d.y), two(d.z), two(d.w)));
                        }
                    }
                } else {
                    const int nvec = envs_here * L::VPE;
                    for (int v = lane; v < nvec; v += 32) {
                        const int e = v / (L::VPE > 0 ? L::VPE : 1), r = v % (L::VPE > 0 ? L::VPE : 1);
                        const unsigned char *tb = wstage + e * L::TSB;
                        union { uint4 u; P2 q[L::PPV]; } o;
#pragma unroll
                        for (int c = 0; c < L::PPV; ++c) o.q[c] = *reinterpret_cast<const P2 *>(tb + tpe_pair_offset<A, L::PSZ>(L::PPV * r + c));
                        __stcs(outv + (v - lane), o.u);
                    }
                }
            }
            __syncwarp();
        }
      }   // steps of this launch

        // ---- write back the persistent state ----------------------------------------------------
        if (env_ok) {
            unsigned px[A], py[A];
#pragma unroll
            for (int k = 0; k < A; ++k) { px[k] = pos[k] >> 8; py[k] = pos[k] & 0xffu; }
            tpe_store_row<A, CCB_TPE_STATE_STREAM == 1>(p.x, n, px);
            tpe_store_row<A, CCB_TPE_STATE_STREAM == 1>(p.y, n, py);
            tpe_store_row<A, CCB_TPE_STATE_STREAM == 1>(p.flags, n, fl);
            if (CCB_TPE_STATE_STREAM == 1) { __stcs(p.step + n, step); __stcs(p.ep_ret + n, ep_ret); }
            else { p.step[n] = step; p.ep_ret[n] = ep_ret; }
        }
#if CCB_TPE_DYNAMIC
        g_next = __shfl_sync(kFull, g_next, 0);
#endif
    }

    if (L::kTma && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // shared memory stays valid until the copies are done
    // ---- statistics: per-warp slots in shared memory -> one atomic per slot per CTA ----------------
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
            for (int w = 0; w < kTpeWarps; ++w) v += all[w * kStCount + threadIdx.x];
            if (v) atomicAdd(&p.stats[threadIdx.x], v);
        } else if (threadIdx.x == 6 || threadIdx.x == 7) {
            double v = 0.0;
            for (int w = 0; w < kTpeWarps; ++w) v += __longlong_as_double((long long)all[w * kStCount + threadIdx.x]);
            if (v != 0.0) atomicAdd(reinterpret_cast<double *>(&p.stats[threadIdx.x]), v);
        } else if (threadIdx.x == 0 && blockIdx.x == 0) {
            atomicAdd(&p.stats[kStEnvSteps], (unsigned long long)p.n_envs * (unsigned long long)p.n_steps);
        }
    }
    if (errbits) atomicOr(p.err, errbits);
}

}  // namespace ccb
