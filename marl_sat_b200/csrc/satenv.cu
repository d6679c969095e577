// Batched SATEnv kernels for sm_100a: formula-bank compiler, reset / step(+auto-reset) / get_obs,
// and the SATState exporter.  Reference semantics: src/envs/multi_agent_sat_env.py (cited as env:LINE)
// and src/learners/mappo_gnn_sat_learner.py:422-464 (auto-reset).  See DESIGN.md section 4.
#include <type_traits>

#include "internal.h"

namespace msat {

// =====================================================================================
// K_compile: one CTA per formula.  Evaluates the agent<->clause and agent<->neighbour
// relations of _compute_observation_maps (env:99-128) once per formula and stores them as a
// flat A*D-bit mask stream in observation order [own(n) | clauses(m) | neighbours(n)] per agent,
// next to the literals packed literal-major as u16 codes ((var << 1) | negated, 0xFFFF for a 0 padding literal).
// =====================================================================================
__global__ void __launch_bounds__(256) compile_bank_kernel(Dims d, const int32_t* __restrict__ clauses,
                                                           uint8_t* __restrict__ bank) {
    extern __shared__ uint32_t csm[];
    uint32_t* clause_agents = csm;                 // [m][agw]  agents related to clause c
    uint32_t* var_agents = csm + d.m * d.agw;      // [n][agw]  agents that see variable v in a related clause
    const int tid = threadIdx.x, nt = blockDim.x;
    const int32_t* cl = clauses + (size_t)blockIdx.x * d.m * d.k;
    uint8_t* rec = bank + (size_t)blockIdx.x * d.rec_bytes;
    uint16_t* lits = reinterpret_cast<uint16_t*>(rec);
    uint32_t* mflat = reinterpret_cast<uint32_t*>(rec + d.lits_bytes);

    for (int i = tid; i < (d.m + d.n) * d.agw; i += nt) csm[i] = 0u;
    for (int i = tid; i < d.lits_bytes / 2; i += nt) lits[i] = lit_pad(d);     // spare column and tail stay padding
    for (int i = d.lits_bytes / 4 + d.fw + 1 + tid; i < d.rec_bytes / 4; i += nt)
        reinterpret_cast<uint32_t*>(rec)[i] = 0u;
    __syncthreads();

    for (int c = tid; c < d.m; c += nt) {
        uint32_t* ca = clause_agents + c * d.agw;
        for (int j = 0; j < d.k; ++j) {
            const int lit = cl[c * d.k + j];
            uint16_t code;
            if (lit == 0) {
                // env:100,106: |0|-1 = -1 equals the -1 padding of every agent that owns fewer than
                // V variables, so the clause becomes "related" to all of those agents.
                code = lit_pad(d);
                if (d.rem > 0)
                    for (int a = d.rem; a < d.A; ++a) ca[a >> 5] |= 1u << (a & 31);
            } else {
                int v = (lit < 0 ? -lit : lit) - 1;
                v = v < d.n ? v : d.n - 1;
                code = (uint16_t)((v << 1) | (lit < 0 ? 1 : 0));
                const int a = var_to_agent(d, v);
                ca[a >> 5] |= 1u << (a & 31);
            }
            lits[lit_index(d.ms, c, j)] = code;
        }
    }
    __syncthreads();
    // env:116-121: every real variable of a related clause is a candidate neighbour.
    for (int c = tid; c < d.m; c += nt) {
        for (int j = 0; j < d.k; ++j) {
            const uint16_t code = lits[lit_index(d.ms, c, j)];
            if (code == lit_pad(d)) continue;
            const int v = code >> 1;
            for (int w = 0; w < d.agw; ++w) {
                const uint32_t x = clause_agents[c * d.agw + w];
                if (x) atomicOr(&var_agents[v * d.agw + w], x);
            }
        }
    }
    __syncthreads();
    for (int w = tid; w < d.fw + 1; w += nt) {
        uint32_t bits = 0u;
        for (int b = 0; b < 32; ++b) {
            const int j = w * 32 + b;
            if (j >= d.AD) break;
            const int a = j / d.D, p = j - a * d.D;
            uint32_t bit;
            if (p < d.n) {
                bit = var_to_agent(d, p) == a;                                         // env:355
            } else if (p < d.n + d.m) {
                bit = (clause_agents[(p - d.n) * d.agw + (a >> 5)] >> (a & 31)) & 1u;  // env:112
            } else {
                const int v = p - d.n - d.m;
                bit = ((var_agents[v * d.agw + (a >> 5)] >> (a & 31)) & 1u) && var_to_agent(d, v) != a;   // env:123
            }
            bits |= bit << b;
        }
        mflat[w] = bits;
    }
    if (d.cnt_words) {
        // var -> clause occurrence lists for the incremental clause update: row_off[v] .. row_off[v+1] index
        // occ[], an entry is (clause << 1) | negated; rows are filled in clause-major literal order
        int* cnt = reinterpret_cast<int*>(csm + (d.m + d.n) * d.agw);      // [n + 1]
        uint16_t* row_off = reinterpret_cast<uint16_t*>(rec + d.csr_off);
        uint16_t* occ = row_off + ((d.n + 1 + 7) & ~7);
        __syncthreads();
        for (int i = tid; i <= d.n; i += nt) cnt[i] = 0;
        __syncthreads();
        for (int i = tid; i < d.m * d.k; i += nt) {
            const uint32_t code = lits[lit_index(d.ms, i / d.k, i % d.k)];
            if (code != lit_pad(d)) atomicAdd(&cnt[code >> 1], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int run = 0;
            for (int v = 0; v < d.n; ++v) {
                const int c = cnt[v];
                cnt[v] = run;
                row_off[v] = (uint16_t)run;
                run += c;
            }
            row_off[d.n] = (uint16_t)run;
        }
        __syncthreads();
        for (int v = tid; v < d.n; v += nt) {
            int o = cnt[v];
            for (int i = 0; i < d.m * d.k; ++i) {
                const int c = i / d.k;
                const uint32_t code = lits[lit_index(d.ms, c, i - c * d.k)];
                if (code != lit_pad(d) && (int)(code >> 1) == v) occ[o++] = (uint16_t)((c << 1) | (code & 1u));
            }
        }
    }
}

// =====================================================================================
// Device pieces of the env kernel.  One group of GS threads owns one env.
// =====================================================================================

// Literal truth table of the current assignment: tt[code] for code = (var << 1) | negated, i.e. tt[2v] = a_v,
// tt[2v+1] = !a_v, and tt[2n] = 0 for the 0-padding literal (never true, env:141-144).  2n + 1 bytes per
// env, rebuilt after every change of the assignment; it turns one literal evaluation into one byte load.
template <int GS>
__device__ __forceinline__ void build_truth_table(const Dims& d, const uint32_t* assign, uint8_t* tt, int gt) {
    const int n2 = 2 * d.n;
    for (int w = gt; 4 * w <= n2; w += GS) {          // four codes (two variables) per 32-bit store
        const int v = 2 * w;
        const uint32_t word = assign[v >> 5] >> (v & 31);      // v is even: v and v+1 sit in the same word
        const uint32_t a0 = word & 1u, a1 = (word >> 1) & 1u;
        uint32_t b = a0 | ((a0 ^ 1u) << 8) | (a1 << 16) | ((a1 ^ 1u) << 24);
        if (v >= d.n) b = 0u;                                   // codes 2n .. : padding literal
        else if (v + 1 >= d.n) b &= 0x0000FFFFu;
        reinterpret_cast<uint32_t*>(tt)[w] = b;
    }
}

// Clause truth via warp ballots (env:130-156): lane = clause, ballot word = 32 clause-status bits, __popc for
// the number of (un)satisfied clauses; the evaluators follow the bulk-store helpers below.

// Publish the number of unsatisfied clauses.  nsat: the satisfied clauses this thread's warp (sub-warp group for
// GS < 32) evaluated, the same in each of its lanes.  A group of at most one warp stores m - nsat; the warps of a
// wider group subtract their counts from *nunsat, which the caller set to m.
template <int GS>
__device__ __forceinline__ void publish_unsat(const Dims& d, int* nunsat, int nsat, int gt) {
    if (GS <= 32) *nunsat = d.m - nsat;
    else if ((gt & 31) == 0 && nsat) atomicAdd(nunsat, -nsat);
}

// ---- bulk (TMA) store shared -> global ----------------------------------------------------------------
__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING their shared-memory source
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all committed bulk stores of this thread have completed (their writes are done, not only their reads)
__device__ __forceinline__ void tma_store_wait() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Clause evaluation for a GNN-style consumer (learner:165-195): besides status bits and the unsatisfied
// count it emits clause_features float[m][3] = {is_sat, #true literals / 3.0, 1} -- the literal 3.0 of
// learner:185 for every clause width.  The floats of up to kCfStageClauses clauses are staged in shared
// memory (lane = clause, three conflict-free 4-byte stores) at the same 16-byte phase as their global
// destination and leave as ONE bulk (TMA) store per pass; the <= 3 floats before / after the 16-byte
// aligned body go out as scalars.

// number of true literals of clause c (lane = clause); K3: three literals per clause, no loop
template <bool K3>
__device__ __forceinline__ uint32_t true_literals(const Dims& d, const uint16_t* lits, const uint8_t* tt, int c) {
    if (K3) {
        const uint32_t l0 = lits[c], l1 = lits[d.ms + c], l2 = lits[2 * d.ms + c];   // independent loads first
        return (uint32_t)tt[l0] + tt[l1] + tt[l2];
    }
    uint32_t cnt = 0u;
#pragma unroll 4
    for (int j = 0; j < d.k; ++j) cnt += tt[lits[lit_index(d.ms, c, j)]];
    return cnt;
}

// cf01[t] = {t > 0 ? 1 : 0, t / 3.0} for t = 0..15: the first two clause features of a clause with t true literals
// True-literal count of clause c for the evaluators below.  INCR: the 4-bit count carried in the state (kept
// up to date by flip_and_update_counts); otherwise from the staged literals, optionally packed into `cnt_store`
// (zeroed by the caller) so that a state of an incremental plan leaves every kernel with valid counts.
template <bool K3, bool INCR, bool STORE = true>
__device__ __forceinline__ uint32_t clause_count(const Dims& d, const uint16_t* lits, const uint8_t* tt,
                                                 uint32_t* cntw, int c) {
    if (INCR) return (cntw[c >> 3] >> (4 * (c & 7))) & 15u;
    const uint32_t cnt = true_literals<K3>(d, lits, tt, c);
    if (STORE && cntw && cnt) atomicOr(&cntw[c >> 3], cnt << (4 * (c & 7)));
    return cnt;
}

template <int GS, bool K3, bool INCR, bool STORE>
__device__ __forceinline__ void eval_clauses_gnn(const Dims& d, const uint16_t* lits, const uint8_t* tt, uint32_t* cntw,
                                                 uint32_t* satw, int* nunsat, const float2* cf01, uint8_t* stage,
                                                 float* __restrict__ cf_out, int gid, int gt) {
    const int lane = gt & 31;
    int nsat = 0;                                       // popc of the rounds this warp evaluates (warp-uniform)
    constexpr int kRoundsPerPass = kCfStageClauses / 32;
    const int full = d.m >> 5;                          // rounds in which every lane has a clause
    for (int w0 = 0; w0 < d.sw; w0 += kRoundsPerPass) {
        const int c0 = w0 * 32;
        const int c1 = min(d.m, c0 + kCfStageClauses);
        uint8_t* gdst = reinterpret_cast<uint8_t*>(cf_out + 3 * (size_t)c0);
        const uint32_t phase16 = (uint32_t)(reinterpret_cast<uintptr_t>(gdst) & 15u);
        if (w0 > 0) {
            if (gt == 0) tma_store_wait_read();        // the previous pass has left the staging buffer
            group_sync<GS>(gid);
        }
        const int wend = min(d.sw, w0 + kRoundsPerPass);
        float* o = reinterpret_cast<float*>(stage + phase16) + 3 * (32 * (gt >> 5) + lane);
        int w = w0 + (gt >> 5);
        for (; w < min(wend, full); w += GS / 32, o += 3 * GS) {
            const uint32_t cnt = clause_count<K3, INCR, STORE>(d, lits, tt, cntw, w * 32 + lane);
            const float2 f = cf01[cnt];
            o[0] = f.x;
            o[1] = f.y;
            o[2] = 1.0f;
            const uint32_t word = __ballot_sync(0xffffffffu, cnt != 0u);
            nsat += __popc(word);
            if (lane == 0) satw[w] = word;
        }
        if (w < wend) {                                 // the ragged last round (w == full)
            const int c = w * 32 + lane;
            uint32_t cnt = 0u;
            if (c < d.m) {
                cnt = clause_count<K3, INCR, STORE>(d, lits, tt, cntw, c);
                const float2 f = cf01[cnt];
                o[0] = f.x;
                o[1] = f.y;
                o[2] = 1.0f;
            }
            const uint32_t word = __ballot_sync(0xffffffffu, cnt != 0u);
            nsat += __popc(word);
            if (lane == 0) satw[w] = word;
        }
        fence_proxy_async();                           // staged floats -> visible to the bulk-copy engine
        group_sync<GS>(gid);
        const uint32_t len = 12u * (uint32_t)(c1 - c0);
        uint32_t head = (16u - phase16) & 15u;
        head = head < len ? head : len;
        const uint32_t body = (len - head) & ~15u;
        if (gt == 0 && body) {
            tma_store_1d(gdst + head, stage + phase16 + head, body);
            tma_store_commit();
        }
        if (gt >= 1 && gt < 8) {                        // scalar head (lanes 1-3) and tail (lanes 4-6)
            const uint32_t i = gt < 4 ? (uint32_t)(gt - 1) * 4u : head + body + (uint32_t)(gt - 4) * 4u;
            const bool mine = gt < 4 ? i < head : i < len;
            if (mine) *reinterpret_cast<float*>(gdst + i) = *reinterpret_cast<const float*>(stage + phase16 + i);
        }
    }
    publish_unsat<GS>(d, nunsat, nsat, gt);
}

// Paired evaluation for k == 3 in launches without observations: a lane owns two ADJACENT clauses, so one aligned
// 32-bit load fetches both codes of a literal column (3 loads instead of 6), the six feature floats of the pair
// are contiguous in the staging buffer (three 8-byte stores when the destination phase allows) and the number of
// satisfied clauses is a per-lane sum reduced once per warp -- no ballots, and no status words: nothing in such a
// launch reads them (callers that do -- shaped reward, incremental plans -- take the lane = clause evaluators).
template <int GS, bool CF>
__device__ __forceinline__ void eval_clauses_pairs(const Dims& d, const uint16_t* lits, const uint8_t* tt, int* nunsat,
                                                   const float2* cf01, uint8_t* stage, float* __restrict__ cf_out,
                                                   int gid, int gt) {
    const uint32_t* l32 = reinterpret_cast<const uint32_t*>(lits);
    const int ms2 = d.ms >> 1;
    int nsat = 0;
    auto counts = [&](int pp, uint32_t& ca, uint32_t& cb) {       // pair pp = clauses 2pp, 2pp + 1
        const uint32_t w0 = l32[pp], w1 = l32[ms2 + pp], w2 = l32[2 * ms2 + pp];
        ca = (uint32_t)tt[w0 & 0xFFFFu] + tt[w1 & 0xFFFFu] + tt[w2 & 0xFFFFu];
        cb = (uint32_t)tt[w0 >> 16] + tt[w1 >> 16] + tt[w2 >> 16];    // spare column of an odd m: padding codes, 0
        nsat += (ca != 0u) + (cb != 0u);
    };
    if constexpr (!CF) {
        const int npairs = (d.m + 1) >> 1;
        for (int pp = gt; pp < npairs; pp += GS) {
            uint32_t ca, cb;
            counts(pp, ca, cb);
        }
    } else {
        for (int c0 = 0; c0 < d.m; c0 += kCfStageClauses) {
            const int c1 = min(d.m, c0 + kCfStageClauses);
            uint8_t* gdst = reinterpret_cast<uint8_t*>(cf_out + 3 * (size_t)c0);
            const uint32_t phase16 = (uint32_t)(reinterpret_cast<uintptr_t>(gdst) & 15u);
            if (c0 > 0) {
                if (gt == 0) tma_store_wait_read();        // the previous pass has left the staging buffer
                group_sync<GS>(gid);
            }
            const int npass = (c1 - c0 + 1) >> 1;            // pairs of this pass (the last may be half valid)
            const int p0 = c0 >> 1;
            if ((phase16 & 7u) == 0u) {                      // 8-byte aligned pair slots: three 64-bit stores
                for (int q = gt; q < npass; q += GS) {
                    uint32_t ca, cb;
                    counts(p0 + q, ca, cb);
                    const float2 f = cf01[ca], g = cf01[cb];
                    float2* o = reinterpret_cast<float2*>(stage + phase16 + 24 * q);
                    o[0] = f;
                    o[1] = make_float2(1.0f, g.x);
                    o[2] = make_float2(g.y, 1.0f);
                }
            } else {
                for (int q = gt; q < npass; q += GS) {
                    uint32_t ca, cb;
                    counts(p0 + q, ca, cb);
                    const float2 f = cf01[ca], g = cf01[cb];
                    float* o = reinterpret_cast<float*>(stage + phase16 + 24 * q);
                    o[0] = f.x; o[1] = f.y; o[2] = 1.0f;
                    o[3] = g.x; o[4] = g.y; o[5] = 1.0f;
                }
            }
            fence_proxy_async();                           // staged floats -> visible to the bulk-copy engine
            group_sync<GS>(gid);
            const uint32_t len = 12u * (uint32_t)(c1 - c0);
            uint32_t head = (16u - phase16) & 15u;
            head = head < len ? head : len;
            const uint32_t body = (len - head) & ~15u;
            if (gt == 0 && body) {
                tma_store_1d(gdst + head, stage + phase16 + head, body);
                tma_store_commit();
            }
            if (gt >= 1 && gt < 8) {                        // scalar head (lanes 1-3) and tail (lanes 4-6)
                const uint32_t i = gt < 4 ? (uint32_t)(gt - 1) * 4u : head + body + (uint32_t)(gt - 4) * 4u;
                const bool mine = gt < 4 ? i < head : i < len;
                if (mine) *reinterpret_cast<float*>(gdst + i) = *reinterpret_cast<const float*>(stage + phase16 + i);
            }
        }
    }
    nsat = __reduce_add_sync(0xffffffffu, nsat);
    if (nunsat) publish_unsat<GS>(d, nunsat, nsat, gt);
}

// Plain evaluation (no clause features): status bits + number of unsatisfied clauses (optional).
// STORE: also pack the counts into cntw (plans with the incremental update only).
template <int GS, bool K3, bool INCR, bool STORE>
__device__ __forceinline__ void eval_clauses_impl(const Dims& d, const uint16_t* lits, const uint8_t* tt, uint32_t* cntw,
                                                  uint32_t* satw, int* nunsat, int gt) {
    const int lane = gt & 31;
    int nsat = 0;
    if constexpr (GS < 32) {
        // several envs per warp: rounds of GS clauses, ballots over the env's own lanes, status bits stored as
        // GS-bit pieces of the 32-bit status words (little endian)
        using piece_t = typename std::conditional<GS == 16, uint16_t, uint8_t>::type;
        piece_t* piece = reinterpret_cast<piece_t*>(satw);
        const uint32_t sh = subwarp_shift<GS>();
        const uint32_t mask = subwarp_mask<GS>();
        const int full = d.m / GS;                       // rounds in which every lane has a clause
        int r = 0;
        for (; r < full; ++r) {
            const uint32_t cnt = clause_count<K3, INCR, STORE>(d, lits, tt, cntw, r * GS + gt);
            const uint32_t bits = (__ballot_sync(mask, cnt != 0u) >> sh) & ((1u << GS) - 1u);
            nsat += __popc(bits);
            if (gt == 0) piece[r] = (piece_t)bits;
        }
        if (full * GS < d.m) {                           // the ragged round
            const int c = r * GS + gt;
            const uint32_t cnt = c < d.m ? clause_count<K3, INCR, STORE>(d, lits, tt, cntw, c) : 0u;
            const uint32_t bits = (__ballot_sync(mask, cnt != 0u) >> sh) & ((1u << GS) - 1u);
            nsat += __popc(bits);
            if (gt == 0) piece[r] = (piece_t)bits;
            ++r;
        }
        if (gt == 0)
            for (; r < (32 / GS) * d.sw; ++r) piece[r] = 0;      // rest of the last status word
    } else {
        for (int w = gt >> 5; w < d.sw; w += GS / 32) {
            const int c = w * 32 + lane;
            const uint32_t cnt = c < d.m ? clause_count<K3, INCR, STORE>(d, lits, tt, cntw, c) : 0u;
            const uint32_t word = __ballot_sync(0xffffffffu, cnt != 0u);
            nsat += __popc(word);
            if (lane == 0) satw[w] = word;
        }
    }
    if (nunsat) publish_unsat<GS>(d, nunsat, nsat, gt);
}
// Half-warp groups, k == 3: a lane owns two ADJACENT clauses (one aligned 32-bit load per literal column fetches
// both codes), so one trip of the 16 lanes covers a whole 32-bit status word: the ballots of the even and the odd
// clauses are interleaved back into clause order (the observation writer reads the status bits in place).
__device__ __forceinline__ uint32_t spread16(uint32_t x) {       // bit i -> bit 2i
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    return (x | (x << 1)) & 0x55555555u;
}
__device__ __forceinline__ void eval_clauses_pairs16(const Dims& d, const uint16_t* lits, const uint8_t* tt,
                                                     uint32_t* satw, int* nunsat, int gt) {
    const uint32_t* l32 = reinterpret_cast<const uint32_t*>(lits);
    const int ms2 = d.ms >> 1;
    const uint32_t sh = subwarp_shift<16>();
    const uint32_t mask = subwarp_mask<16>();
    int nsat = 0;
    for (int w = 0; w < d.sw; ++w) {
        const int pp = 16 * w + gt;                               // clauses 2pp, 2pp + 1
        uint32_t ca = 0u, cb = 0u;
        if (pp < ms2) {
            const uint32_t w0 = l32[pp], w1 = l32[ms2 + pp], w2 = l32[2 * ms2 + pp];
            ca = (uint32_t)tt[w0 & 0xFFFFu] + tt[w1 & 0xFFFFu] + tt[w2 & 0xFFFFu];
            cb = (uint32_t)tt[w0 >> 16] + tt[w1 >> 16] + tt[w2 >> 16];     // spare column of an odd m: padding, 0
        }
        const uint32_t ev = (__ballot_sync(mask, ca != 0u) >> sh) & 0xFFFFu;
        const uint32_t od = (__ballot_sync(mask, cb != 0u) >> sh) & 0xFFFFu;
        const uint32_t word = spread16(ev) | (spread16(od) << 1);
        nsat += __popc(word);
        if (gt == 0) satw[w] = word;
    }
    if (nunsat) publish_unsat<16>(d, nunsat, nsat, gt);
}

template <int GS, bool K3, bool INCR>
__device__ __forceinline__ void eval_clauses(const Dims& d, const uint16_t* lits, const uint8_t* tt, uint32_t* cntw,
                                             uint32_t* satw, int* nunsat, int gt) {
    if constexpr (GS == 16 && K3 && !INCR) {
        // pays from ~4 status words on (uf35-149: -8 % step time; uf20-91, 3 words: +4 % instructions)
        if (!cntw && d.sw >= 4) {
            eval_clauses_pairs16(d, lits, tt, satw, nunsat, gt);
            return;
        }
    }
    if (!INCR && cntw) eval_clauses_impl<GS, K3, INCR, true>(d, lits, tt, cntw, satw, nunsat, gt);
    else eval_clauses_impl<GS, K3, INCR, false>(d, lits, tt, cntw, satw, nunsat, gt);
}

// assign = randint(key, (n,), 0, 2) (env:162): bit 0 of threefry_2x32(split(key)[1], arange(n)).
template <int GS>
__device__ __forceinline__ void threefry_assign(const Dims& d, uint32_t k0, uint32_t k1, uint32_t* assign, int gt) {
    uint32_t ka[2], kb[2];
    split2(k0, k1, ka, kb);
    const int half = (d.n + 1) >> 1;
    for (int i = gt; i < half; i += GS) {
        uint32_t x0 = (uint32_t)i;
        uint32_t x1 = (half + i < d.n) ? (uint32_t)(half + i) : 0u;
        threefry2x32(kb[0], kb[1], x0, x1);
        if (x0 & 1u) atomicOr(&assign[i >> 5], 1u << (i & 31));
        const int v = half + i;
        if (v < d.n && (x1 & 1u)) atomicOr(&assign[v >> 5], 1u << (v & 31));
    }
}

// State import: pack a given int32[n] assignment (nonzero reads as 1) into the assignment words.  Lane v % 32 (v % 16
// in half-warp groups) loads variable v, so consecutive lanes read consecutive ints, and one ballot makes a word
// (half a word for GS = 16, stored as a 16-bit piece: little endian, as the half-warp status words).  Every word,
// including the bits past n, is written in full.
template <int GS>
__device__ __forceinline__ void load_assign(const Dims& d, const int32_t* __restrict__ src, uint32_t* assign, int gt) {
    if constexpr (GS < 32) {
        uint16_t* piece = reinterpret_cast<uint16_t*>(assign);
        const uint32_t sh = subwarp_shift<16>();
        const uint32_t mask = subwarp_mask<16>();
        for (int r = 0; r < 2 * d.aw; ++r) {
            const int v = 16 * r + gt;
            const bool bit = v < d.n && src[v] != 0;
            const uint32_t bits = (__ballot_sync(mask, bit) >> sh) & 0xFFFFu;
            if (gt == 0) piece[r] = (uint16_t)bits;
        }
    } else {
        const int lane = gt & 31;
        for (int w = gt >> 5; w < d.aw; w += GS / 32) {
            const int v = 32 * w + lane;
            const uint32_t word = __ballot_sync(0xffffffffu, v < d.n && src[v] != 0);
            if (lane == 0) assign[w] = word;
        }
    }
}

// Start state (msat_apply_start_states) into zeroed assignment words: bit v = start bit v XOR (u_v < thr), where
// u_v = threefry_2x32(ka, arange(n))[v] and (ka, kb) = split(key) -- the half of the key randint leaves unused
// (threefry_assign reads kb), with randint's counter layout.  Start bits past n are dropped.  XOR commutes, so
// the start words and the flips go in with atomics in any order.
template <int GS>
__device__ __forceinline__ void start_assign(const Dims& d, const uint32_t* __restrict__ start, uint32_t thr,
                                             uint32_t k0, uint32_t k1, uint32_t* assign, int gt) {
    for (int w = gt; w < d.aw; w += GS) {
        const int tail = d.n - 32 * w;
        const uint32_t word = start[w] & (tail >= 32 ? 0xFFFFFFFFu : (1u << tail) - 1u);
        if (word) atomicXor(&assign[w], word);
    }
    uint32_t ka[2], kb[2];
    split2(k0, k1, ka, kb);
    const int half = (d.n + 1) >> 1;
    for (int i = gt; i < half; i += GS) {
        uint32_t x0 = (uint32_t)i;
        uint32_t x1 = (half + i < d.n) ? (uint32_t)(half + i) : 0u;
        threefry2x32(ka[0], ka[1], x0, x1);
        if (x0 < thr) atomicXor(&assign[i >> 5], 1u << (i & 31));
        const int v = half + i;
        if (v < d.n && x1 < thr) atomicXor(&assign[v >> 5], 1u << (v & 31));
    }
}

// Decode all agents' actions of env e (env:233-250) and call flip(v) once for every variable that flips; the flips
// are simultaneous, so flip must commute (atomics).  has_pre: the caller already holds act[gt] (mode 0) in `pre`
// (loaded early, next to the state record).
template <int GS, typename F>
__device__ __forceinline__ void for_each_flip(const Dims& d, const int32_t* __restrict__ actions, int e, int gt,
                                              bool has_pre, int pre, F flip) {
    if (d.action_mode == 0) {
        const int32_t* act = actions + (size_t)e * d.A;
        for (int a = gt; a < d.A; a += GS) {
            const int x = (has_pre && a == gt) ? pre : act[a];
            const int size = group_size(d, a);
            if (x >= size) continue;                       // env:236 no-op
            int idx = x < size - 1 ? x : size - 1;         // env:238
            if (idx < 0) idx += d.V;                       // JAX gather: wrap once, then clamp
            idx = idx < 0 ? 0 : (idx > d.V - 1 ? d.V - 1 : idx);
            if (idx >= size) continue;                     // landed on a -1 pad: one_hot(-1) = 0 (env:243)
            flip(group_start(d, a) + idx);
        }
    } else {
        const int32_t* act = actions + (size_t)e * d.A * d.V;
        for (int i = gt; i < d.A * d.V; i += GS) {
            const int a = i / d.V, j = i - a * d.V;
            if (j < group_size(d, a) && (act[i] & 1))      // env:246-250 (actions are 0/1)
                flip(group_start(d, a) + j);
        }
    }
}

// Incremental clause update (env:130-156 restricted to the clauses adjacent to the flipped variables): every
// flipping (agent, variable) walks the variable's occurrence list -- staged in shared memory by a TMA bulk copy
// of the record's CSR block -- and moves the 4-bit true-literal count of each adjacent clause by +-1.  A variable flips at most
// once per step (agents own disjoint variables), so its new value is the old one inverted; the partial sums
// of a clause's updates stay within [0, k] in any order, so the packed nibbles never carry or borrow.
__device__ __forceinline__ void flip_and_update_counts(const Dims& d, const uint8_t* csr, int v,
                                                       uint32_t* assign, uint32_t* cntw) {
    const uint16_t* row_off = reinterpret_cast<const uint16_t*>(csr);
    const uint16_t* occ = row_off + ((d.n + 1 + 7) & ~7);
    const uint32_t bit = 1u << (v & 31);
    const uint32_t now_true = ((assign[v >> 5] & bit) == 0u) ? 1u : 0u;      // value after the flip
    atomicXor(&assign[v >> 5], bit);
    const int o1 = row_off[v + 1];
    for (int o = row_off[v]; o < o1; ++o) {
        const uint32_t code = occ[o];
        const uint32_t c = code >> 1;
        const uint32_t unit = 1u << (4 * (c & 7));
        if ((code & 1u) ^ now_true) atomicAdd(&cntw[c >> 3], unit);           // this literal became true
        else atomicSub(&cntw[c >> 3], unit);
    }
}

// Four observation ints from a 4-bit mask nibble and a 4-bit value nibble: out = mask ? value : -1.
// The nibbles are spread to one byte per element with a multiply, combined bytewise into
// {0xFF, 0x00, 0x01} and sign-extended to int32 with one PRMT each.
__device__ __forceinline__ int4 expand_nibble(uint32_t mn, uint32_t xn) {
    const uint32_t m4 = (mn * 0x00204081u) & 0x01010101u;          // bit i -> byte i
    const uint32_t r = 0xFFFFFFFFu - m4 * 0xFFu;                   // byte: mask ? 0x00 : 0xFF
    const uint32_t c = ((xn * 0x00204081u) & 0x01010101u) | r;     // byte: mask ? value : 0xFF
    // prmt.b32 selector nibble: bits 2:0 pick the byte, bit 3 replicates its sign instead (the
    // __byte_perm intrinsic masks bit 3 away, hence inline PTX): byte i sign-extended to 32 bits.
    int4 v;
    asm("prmt.b32 %0, %1, %1, 0x8880;" : "=r"(v.x) : "r"(c));
    asm("prmt.b32 %0, %1, %1, 0x9991;" : "=r"(v.y) : "r"(c));
    asm("prmt.b32 %0, %1, %1, 0xAAA2;" : "=r"(v.z) : "r"(c));
    asm("prmt.b32 %0, %1, %1, 0xBBB3;" : "=r"(v.w) : "r"(c));
    return v;
}

// Observation writer (env:345-398).  Per env the A*D output ints are one flat range of the
// [B,A,D] tensor.  out[i] = mask[i] ? value[i] : -1 where mask is the bank's flat bit stream and
// value is [assign | clause status | assign] repeated per agent.  Both streams are re-based to the
// 128-byte aligned start of the range so every lane owns whole 16-byte chunks (st.global.cs.v4).
// Four observation BYTES (int8) of a mask / value nibble pair: mask ? value : -1 (0xFF).
__device__ __forceinline__ uint32_t expand_nibble_i8(uint32_t mn, uint32_t xn) {
    const uint32_t m4 = (mn * 0x00204081u) & 0x01010101u;
    return ((xn * 0x00204081u) & 0x01010101u) | (0xFFFFFFFFu - m4 * 0xFFu);
}

// I8 (msat_plan_set_obs_dtype): the same flat range with one byte per element -- `obs` then points to int8 data,
// a 16-byte chunk covers 16 elements (half a mask / value word pair) and at most 15 bytes at each end of an
// env's range go out as scalar byte stores.
template <int GS, bool I8>
__device__ __forceinline__ void emit_obs(const Dims& d, long long row, const uint32_t* assign, const uint32_t* satw,
                                         uint32_t* X, uint2* smx, const uint32_t* mflat,
                                         int32_t* __restrict__ obs, int gid, int gt) {
    for (int w = gt; w < d.xw; w += GS) {
        const int pos = 32 * w;
        X[w] = extract32(assign, d.aw, pos) | extract32(satw, d.sw, pos - d.n) |
               extract32(assign, d.aw, pos - d.n - d.m);
    }
    group_sync<GS>(gid);

    const long long g_start = row * d.AD;
    const int s = (int)(g_start & 31);
    const int nw = (s + d.AD + 31) >> 5;
    for (int w = gt; w < nw; w += GS) {
        const int j0 = 32 * w - s;
        const uint32_t mw = extract32(mflat, d.fw + 1, j0);
        uint32_t xw = 0u;
        int j = j0 > 0 ? j0 : 0;
        const int jend = (j0 + 32 < d.AD) ? j0 + 32 : d.AD;
        if (d.D >= 32) {
            // a 32-bit window crosses at most one row boundary: the value stream is X repeated with period D, and
            // bits before / after the env's range are never stored (their mask bits are zero)
            const int jj = j0 < 0 ? j0 + d.D : j0;
            int arow = (int)__umulhi((uint32_t)jj, d.inv_D);
            if (arow * d.D > jj) --arow;
            const int p = jj - arow * d.D;                       // 0 <= p < D; X has one clean word past D
            xw = __funnelshift_r(X[p >> 5], X[(p >> 5) + 1], p & 31);
            const int rem = d.D - p;
            if (rem < 32) xw |= X[0] << rem;
        } else if (j < jend) {
            int arow = (int)__umulhi((uint32_t)j, d.inv_D);     // j / D with a rounded-up reciprocal (+0/+1)
            if (arow * d.D > j) --arow;
            int p = j - arow * d.D;
            while (j < jend) {
                int len = d.D - p;
                if (len > jend - j) len = jend - j;
                uint32_t bits = extract32(X, d.xw, p);
                if (len < 32) bits &= (1u << len) - 1u;
                xw |= bits << (j - j0);
                j += len;
                p = 0;
            }
        }
        smx[w] = make_uint2(mw, xw);
    }
    group_sync<GS>(gid);

    if constexpr (I8) {
        // ---- int8: chunk q covers elements [16q, 16q+16) of the re-based range (32-byte aligned base) ----
        int8_t* out8 = reinterpret_cast<int8_t*>(obs) + (g_start - s);
        const int lo = s, hi = s + d.AD;
        const int q_lo = (lo + 15) >> 4, q_hi = hi >> 4;
        {
            int q = q_lo + gt;                      // GS is even: a lane keeps the same half of its word pair
            const int sh = (q & 1) * 16;
            const uint2* sp = smx + (q >> 1);
            uint4* op = reinterpret_cast<uint4*>(out8) + q;
#pragma unroll 2
            for (; q < q_hi; q += GS, sp += GS / 2, op += GS) {
                const uint2 mx = *sp;
                const uint32_t m16 = mx.x >> sh, x16 = mx.y >> sh;
                __stcs(op, make_uint4(expand_nibble_i8(m16 & 0xFu, x16 & 0xFu),
                                      expand_nibble_i8((m16 >> 4) & 0xFu, (x16 >> 4) & 0xFu),
                                      expand_nibble_i8((m16 >> 8) & 0xFu, (x16 >> 8) & 0xFu),
                                      expand_nibble_i8((m16 >> 12) & 0xFu, (x16 >> 12) & 0xFu)));
            }
        }
        // the < 16 elements before the first / after the last complete chunk (or the whole range when it is short)
        const int head_end = min(16 * q_lo, hi);
        const int tail_start = max(16 * q_hi, head_end);
        auto put = [&](int i) {
            const uint2 mx = smx[i >> 5];
            out8[i] = ((mx.x >> (i & 31)) & 1u) ? (int8_t)((mx.y >> (i & 31)) & 1u) : (int8_t)-1;
        };
        for (int i = lo + gt; i < head_end; i += GS) put(i);
        for (int i = tail_start + gt; i < hi; i += GS) put(i);
        return;
    }
    // ---- streaming stores: chunk q covers ints [4q, 4q+4) of the re-based range ----
    int32_t* out = obs + (g_start - s);
    const int lo_valid = s, hi_valid = s + d.AD;
    const int q_lo = (lo_valid + 3) >> 2;       // first chunk that lies completely inside the env's range
    const int q_hi = hi_valid >> 2;             // one past the last complete chunk
    {
        // GS is a multiple of 8, so a lane keeps the same nibble position in every iteration.
        int q = q_lo + gt;
        const int sh = (q & 7) * 4;
        const uint2* sp = smx + (q >> 3);
        int4* op = reinterpret_cast<int4*>(out) + q;
#pragma unroll 4
        for (; q < q_hi; q += GS, sp += GS / 8, op += GS) {
            const uint2 mx = *sp;
            __stcs(op, expand_nibble((mx.x >> sh) & 0xFu, (mx.y >> sh) & 0xFu));
        }
    }
    // at most one partial chunk at each end (the env's range is only 4-byte aligned): scalar stores
    if (gt < 8) {
        const int q = (gt < 4) ? q_lo - 1 : q_hi;
        const int i = 4 * q + (gt & 3);
        const bool partial = (gt < 4) ? (4 * q_lo != lo_valid) : (4 * q_hi != hi_valid);
        if (partial && q >= 0 && i >= lo_valid && i < hi_valid) {
            const uint2 mx = smx[i >> 5];
            out[i] = ((mx.x >> (i & 31)) & 1u) ? (int)((mx.y >> (i & 31)) & 1u) : -1;
        }
    }
}

// `count` 4-byte values f(0..count-1) to a 4-byte aligned destination with 16-byte streaming stores: the
// (at most 3) elements before the first 16-byte boundary and after the last complete chunk go out as scalars.
template <int GS, typename F>
__device__ __forceinline__ void store_words_vec4(uint32_t* __restrict__ dst, int count, int gt, F f) {
    int head = (int)(((16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2);
    head = head < count ? head : count;
    const int n4 = (count - head) >> 2;
    uint4* d4 = reinterpret_cast<uint4*>(dst + head);
    for (int q = gt; q < n4; q += GS) {
        const int i = head + 4 * q;
        __stcs(d4 + q, make_uint4(f(i), f(i + 1), f(i + 2), f(i + 3)));
    }
    if (gt < head) dst[gt] = f(gt);
    const int i = head + 4 * n4 + gt;
    if (gt < 3 && i < count) dst[i] = f(i);
}

// Assignment part of the dynamic GNN input (learner:165): int32[n] per env as 16-byte stores.
template <int GS>
__device__ __forceinline__ void emit_gnn_assignment(const Dims& d, long long row, const uint32_t* assign,
                                                    int32_t* __restrict__ gnn_assign, int gt) {
    store_words_vec4<GS>(reinterpret_cast<uint32_t*>(gnn_assign) + row * d.n, d.n, gt,
                         [&](int v) { return (assign[v >> 5] >> (v & 31)) & 1u; });
}

// Dispatch on clause width (k == 3 has its own unrolled path) and on whether clause features are wanted.
// pairs: the launch writes no observations and nothing reads the clause-status words (see eval_clauses_pairs).
template <int GS, bool INCR, bool OBS>
__device__ __forceinline__ void run_eval(const Dims& d, const uint16_t* lits, const uint8_t* tt, uint32_t* cntw,
                                         uint32_t* satw, int* nunsat, const float2* cf01, uint8_t* stage, float* cf_row,
                                         bool pairs, int gid, int gt) {
    if constexpr (!OBS && !INCR && GS >= 32) {
        if (pairs) {
            if (cf_row) eval_clauses_pairs<GS, true>(d, lits, tt, nunsat, cf01, stage, cf_row, gid, gt);
            else eval_clauses_pairs<GS, false>(d, lits, tt, nunsat, cf01, stage, cf_row, gid, gt);
            return;
        }
    }
    if (GS >= 32 && cf_row) {          // half-warp groups exist only for observation-writing launches
        if constexpr (GS >= 32) {
            const bool store = !INCR && cntw != nullptr;       // pack the counts for an incremental plan's state
            if (d.k == 3) {
                if (store) eval_clauses_gnn<GS, true, INCR, true>(d, lits, tt, cntw, satw, nunsat, cf01, stage, cf_row, gid, gt);
                else eval_clauses_gnn<GS, true, INCR, false>(d, lits, tt, cntw, satw, nunsat, cf01, stage, cf_row, gid, gt);
            } else {
                if (store) eval_clauses_gnn<GS, false, INCR, true>(d, lits, tt, cntw, satw, nunsat, cf01, stage, cf_row, gid, gt);
                else eval_clauses_gnn<GS, false, INCR, false>(d, lits, tt, cntw, satw, nunsat, cf01, stage, cf_row, gid, gt);
            }
        }
    } else {
        if (d.k == 3) eval_clauses<GS, true, INCR>(d, lits, tt, cntw, satw, nunsat, gt);
        else eval_clauses<GS, false, INCR>(d, lits, tt, cntw, satw, nunsat, gt);
    }
}

// One rollout step of the rng alone (learner:397,416,426): rng <- split(rng)[0]; rng <- split(rng)[0];
// rng <- split(rng, 3)[0].
__device__ __forceinline__ void rng_advance(uint32_t& r0, uint32_t& r1) {
    uint32_t a[2], b[2];
    split2(r0, r1, a, b);
    split2(a[0], a[1], a, b);
    uint32_t x0 = 0u, x1 = 3u, y0 = 1u, y1 = 4u;
    threefry2x32(a[0], a[1], x0, x1);
    threefry2x32(a[0], a[1], y0, y1);
    r0 = x0;
    r1 = y0;
}

// =====================================================================================
// K_env<GS, MODE, OBS, MULTI, INCR>: reset / step (+ fused auto-reset, + K fused steps) / get_obs.
// 256-thread CTAs, 256/GS envs each (GS = 16: two envs per warp, observation-writing launches only).
// OBS = the launch writes local observations (whole bank record staged, observation re-basing buffers);
// !OBS = literal block only (or, INCR, the CSR occurrence lists), optional GNN-input outputs.
// MULTI = K steps per launch (msat_rollout_steps); INCR = incremental clause update (step launches of a plan
// with MSAT_CLAUSES_INCREMENTAL that write no observations).
// MODE_IMPORT (msat_import_state) is the reset with the assignment, step and done flag taken from memory.
// MODE_START (msat_apply_start_states) is the reset of the envs that just restarted on a problem with a start state,
// in place, with the assignment built from that start (start_assign); the other groups leave after reading two words.
// =====================================================================================
template <int GS, int MODE, bool OBS, bool MULTI, bool INCR>
__global__ void __launch_bounds__(kCtaThreads, (MULTI || !OBS) ? 4 : 8) env_kernel(const Dims d, const EnvArgs a) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    constexpr int NG = kCtaThreads / GS;
    // builds a state instead of reading one
    constexpr bool FRESH = MODE == MODE_RESET || MODE == MODE_IMPORT || MODE == MODE_START;
    const int gid = threadIdx.x / GS, gt = threadIdx.x % GS;
    const int e = blockIdx.x * NG + gid;
    const GroupLayout& L = a.L;
    const int K = MULTI ? a.num_steps : 1;          // MULTI only with MODE_STEP

    // ---- K > 1 with fused keys: the K chains {rng', act, step, prob, reset} of learner:397-434, once per CTA
    uint32_t* s_chain = reinterpret_cast<uint32_t*>(smem_raw + (size_t)NG * L.total);
    if (MULTI && a.rng_in) {
        if (threadIdx.x == 0) {
            uint32_t r0 = a.rng_in[0], r1 = a.rng_in[1];
            for (int j = 0; j < K; ++j) {          // the dependent part: three Threefry levels per step
                s_chain[10 * j] = r0;
                s_chain[10 * j + 1] = r1;
                rng_advance(r0, r1);
            }
        }
        __syncthreads();
        if ((int)threadIdx.x < K) {
            uint32_t c[10];
            rng_chain_compute(s_chain[10 * threadIdx.x], s_chain[10 * threadIdx.x + 1], c);
            for (int i = 0; i < 10; ++i) s_chain[10 * threadIdx.x + i] = c[i];
        }
        __syncthreads();
        if (blockIdx.x == 0 && threadIdx.x < 10) a.chain_out[threadIdx.x] = s_chain[10 * (K - 1) + threadIdx.x];
    }
    if (e >= a.B) return;   // whole group leaves together
    int start_pidx = 0;
    if constexpr (MODE == MODE_START) {
        // only an env that has just (re)started (step 0) on a problem with a start is rewritten; the group reads the
        // same two words in every lane, so it leaves together
        const uint32_t* tail = a.state_in + (size_t)e * d.state_words + d.aw;
        start_pidx = clamp_problem((int)tail[ST_PIDX], a.P);
        if (tail[ST_STEP] != 0u || (a.has_start && !a.has_start[start_pidx])) return;
    }

    uint8_t* base = smem_raw + (size_t)gid * L.total;
    uint8_t* rec = base + L.rec;
    uint32_t* st = reinterpret_cast<uint32_t*>(base + L.st);
    uint32_t* satw = reinterpret_cast<uint32_t*>(base + L.satw);
    uint32_t* satw_old = reinterpret_cast<uint32_t*>(base + L.satw_old);
    uint32_t* X = reinterpret_cast<uint32_t*>(base + L.x);
    uint2* smx = reinterpret_cast<uint2*>(base + L.smx);
    uint8_t* tt = base + L.tt;
    uint8_t* stage = base + L.stage;
    uint64_t* bar = reinterpret_cast<uint64_t*>(base + L.bar);
    int* misc = reinterpret_cast<int*>(base + L.misc);
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(rec);
    const uint32_t* mflat = reinterpret_cast<const uint32_t*>(rec + d.lits_bytes);
    uint32_t* st_tail = st + d.aw;
    const uint32_t tma_bytes = OBS ? (uint32_t)d.rec_copy_bytes : (uint32_t)d.lits_bytes;
    // per-clause true-literal counts of an incremental plan live in the state record behind the scalars
    uint32_t* cntw = d.cnt_words ? st + d.aw + 4 : nullptr;
    uint32_t* cnt_store = (MODE != MODE_OBS) ? cntw : nullptr;     // full evaluations refresh the counts
    const bool want_cf = !OBS && a.gnn_cf != nullptr;
    // k == 3 launches without observations whose clause-status words nobody reads: paired evaluation
    const bool pairs = !OBS && d.k == 3 && cnt_store == nullptr && cntw == nullptr && a.reward_mode == 0;
    float2* cf01 = reinterpret_cast<float2*>(misc + 4);  // {t > 0, t / 3.0} for t = 0..15 true literals (learner:185)

    // ---- stage the state record (plain loads) ----
    // The two global loads every step waits for -- this lane's piece of the state record and its first action --
    // are issued back to back before anything consumes them, so their latencies overlap each other and the
    // shared-memory set-up below instead of adding up.
    // state records are multiples of 16 bytes (state_words % 4 == 0) in a 16-byte aligned array
    const uint4* sin = FRESH ? nullptr : reinterpret_cast<const uint4*>(a.state_in + (size_t)e * d.state_words);
    const int sw4 = d.state_words >> 2;
    uint4 s0 = make_uint4(0u, 0u, 0u, 0u);
    if (!FRESH && gt < sw4) s0 = sin[gt];
    if constexpr (GS < 32) {            // issue-bound half-warp groups: no registers to spare for the overlap
        if (gt < sw4) reinterpret_cast<uint4*>(st)[gt] = s0;
    }
    int act_pre = 0;
    const bool act_pre_ok = GS >= 32 && MODE == MODE_STEP && !INCR && d.action_mode == 0 && gt < d.A;
    if (act_pre_ok) act_pre = a.actions[(size_t)e * d.A + gt];
    if (gt == 0) {
        misc[0] = d.m;              // #unsatisfied accumulator of multi-warp groups: m minus the satisfied counts
        mbar_init(bar, 1);
    }
    if (want_cf && gt < 16) cf01[gt] = make_float2(gt > 0 ? 1.0f : 0.0f, __fdiv_rn((float)gt, 3.0f));
    if constexpr (GS >= 32) {
        if (gt < sw4) reinterpret_cast<uint4*>(st)[gt] = s0;
    }
    if (!FRESH) {
#pragma unroll 1
        for (int i = gt + GS; i < sw4; i += GS) reinterpret_cast<uint4*>(st)[i] = sin[i];
    } else {
#pragma unroll 1
        for (int i = gt + GS; i < sw4; i += GS) reinterpret_cast<uint4*>(st)[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    group_sync<GS>(gid);

    // Every thread keeps its own copy of the scalar state fields in registers from here on: thread 0 rewrites
    // them in shared memory only after the last step, and a warp that read `step` from shared memory after
    // such a write would disagree with the others about `done` and wait at a group barrier nobody else reaches.
    // an imported step is stored verbatim: states exported after stepping past `done` carry step >= max_steps
    int step_cur = (MODE == MODE_RESET || MODE == MODE_START) ? 0
                 : (MODE == MODE_IMPORT) ? (a.step_in ? a.step_in[e] : 0) : (int)st_tail[ST_STEP];
    int nunsat_prev = FRESH ? 0 : (int)st_tail[ST_NUNSAT];
    uint32_t flags = (MODE == MODE_RESET || MODE == MODE_START) ? 0u
                   : (MODE == MODE_IMPORT) ? ((a.done_in && a.done_in[e]) ? 1u : 0u) : st_tail[ST_FLAGS];
    int pidx;
    if (MODE == MODE_START) pidx = start_pidx;
    else if (FRESH) pidx = a.prob_idx[e];
    else pidx = (int)st_tail[ST_PIDX];
    pidx = clamp_problem(pidx, a.P);
    int loaded_pidx = -1;           // formula whose block sits in the record slot ...
    bool loaded_csr = false;        // ... and whether that block is its occurrence lists (incremental steps) or its literals
    uint32_t phase = 0u;
    int nunsat = nunsat_prev;

    for (int j = 0; j < K; ++j) {
        const bool last = j == K - 1;
        const bool emit = last || a.emit_every_step;
        const long long row = (a.emit_every_step ? (long long)j * a.B : 0LL) + e;     // row of obs / GNN outputs
        const long long orow = (long long)j * a.B + e;                                  // row of reward / done / info

        // ---- formula record: TMA bulk copy unless the env's formula is already staged (an incremental step
        //      needs the literals only when the episode restarts) ----
        if (!INCR && loaded_pidx != pidx && gt == 0) {
            if (j > 0) fence_proxy_async();
            mbar_expect_tx(bar, tma_bytes);
            tma_load_1d(rec, a.bank + (size_t)pidx * d.rec_bytes, tma_bytes, bar);
        }
        // incremental step: the var -> clause occurrence lists of the formula instead (the literals are needed
        // only when the episode restarts)
        const bool need_csr = INCR && !(loaded_csr && loaded_pidx == pidx);
        if (need_csr && gt == 0) {
            if (j > 0) fence_proxy_async();
            mbar_expect_tx(bar, (uint32_t)d.csr_bytes);
            tma_load_1d(rec, a.bank + (size_t)pidx * d.rec_bytes + d.csr_off, (uint32_t)d.csr_bytes, bar);
        }
        if (MODE == MODE_STEP && a.reward_mode) {
            // shaped reward (env:201-223): clause status of the state BEFORE the flips
            if (INCR) {
                run_eval<GS, true, OBS>(d, lits, tt, cntw, satw_old, nullptr, cf01, stage, nullptr, false, gid, gt);
            } else {
                if (loaded_pidx != pidx) {
                    mbar_wait(bar, phase);
                    phase ^= 1u;
                    loaded_pidx = pidx;
                }
                build_truth_table<GS>(d, st, tt, gt);
                group_sync<GS>(gid);
                run_eval<GS, false, OBS>(d, lits, tt, nullptr, satw_old, nullptr, cf01, stage, nullptr, false, gid, gt);
            }
            group_sync<GS>(gid);
        }

        // ---- new assignment while the record is in flight ----
        if (MODE == MODE_RESET) {
            threefry_assign<GS>(d, a.keys[2 * (size_t)e], a.keys[2 * (size_t)e + 1], st, gt);
        } else if (MODE == MODE_IMPORT) {
            load_assign<GS>(d, a.assign_in + (size_t)e * d.n, st, gt);
        } else if (MODE == MODE_START) {
            // the env's reset key, as msat_env_keys and the fused step derive it: split(reset_key, Bg)[env_off + e]
            uint32_t key[2];
            env_reset_key(a.reset_key[0], a.reset_key[1], a.Bg, a.env_off + (uint32_t)e, key);
            start_assign<GS>(d, a.start_words + (size_t)pidx * d.aw, a.flip_thr[pidx], key[0], key[1], st, gt);
        } else if (MODE == MODE_STEP) {
            if (INCR) {
                if (need_csr) {
                    mbar_wait(bar, phase);
                    phase ^= 1u;
                    loaded_pidx = pidx;
                    loaded_csr = true;
                }
                for_each_flip<GS>(d, a.actions + (long long)j * a.act_step_stride, e, gt, false, 0,
                                  [&](int v) { flip_and_update_counts(d, rec, v, st, cntw); });
            } else {
                for_each_flip<GS>(d, a.actions + (long long)j * a.act_step_stride, e, gt, act_pre_ok && j == 0, act_pre,
                                  [&](int v) { atomicXor(&st[v >> 5], 1u << (v & 31)); });
            }
        }
        if (!INCR && cnt_store)
            for (int i = gt; i < d.cnt_words; i += GS) cnt_store[i] = 0u;
        group_sync<GS>(gid);
        if (!INCR) {
            build_truth_table<GS>(d, st, tt, gt);
            if (loaded_pidx != pidx) {
                mbar_wait(bar, phase);
                phase ^= 1u;
                loaded_pidx = pidx;
            }
            group_sync<GS>(gid);
        }

        float* cf_row = (want_cf && emit) ? a.gnn_cf + row * d.m * 3 : nullptr;
        run_eval<GS, INCR, OBS>(d, lits, tt, INCR ? cntw : cnt_store, satw, &misc[0], cf01, stage, cf_row, pairs, gid, gt);
        group_sync<GS>(gid);
        nunsat = misc[0];

        if (MODE == MODE_STEP) {
            if (!MULTI && a.rng_in && blockIdx.x == 0 && threadIdx.x == 0) {
                // advance the rollout rng once per step (learner:397,416,426); chain_out never aliases rng_in
                uint32_t c[10];
                rng_chain_compute(a.rng_in[0], a.rng_in[1], c);
                for (int i = 0; i < 10; ++i) a.chain_out[i] = c[i];
            }
            const bool solved = nunsat == 0;                                  // env:257
            const bool done = solved || (step_cur + 1 >= d.max_steps);        // env:258-259
            // pre-reset outputs stored in the Transition (learner:467-478)
            int newly = 0;
            float r = solved ? 1.0f : 0.0f;                                   // env:193
            if (a.reward_mode) {
                for (int w = 0; w < d.sw; ++w) newly += __popc(satw[w] & ~satw_old[w]);
                // env:207-221, f32 with one rounding per operation
                const float r_pbrs = __fsub_rn(__fmul_rn(a.r_gamma, (float)(-nunsat)), (float)(-nunsat_prev));
                const float r_cl = __fmul_rn((float)newly, a.r_clause);
                r = __fadd_rn(__fadd_rn(r_pbrs, r_cl), solved ? a.r_sat : 0.0f);
            }
            if (a.reward) {
                float* rp = a.reward + orow * a.reward_cols;
#pragma unroll 1
                for (int i = gt; i < a.reward_cols; i += GS) rp[i] = r;
            }
            if (a.done) {
                uint8_t* dp = a.done + orow * a.done_cols;
#pragma unroll 1
                for (int i = gt; i < a.done_cols; i += GS) dp[i] = done ? 1 : 0;
            }
            if (gt == 0) {
                if (a.solved) a.solved[orow] = solved ? 1 : 0;
                if (a.num_unsat) a.num_unsat[orow] = nunsat;
                if (a.episode_step) a.episode_step[orow] = step_cur + 1;     // env:281
                if (a.newly_sat) a.newly_sat[orow] = newly;
            }
            if (done && a.auto_reset) {
                // learner:425-464: swap in a fresh episode on a newly drawn formula (group-uniform branch)
                group_sync<GS>(gid);   // everyone is done reading the old record / misc
                uint32_t rk0, rk1;
                if (a.rng_in) {
                    // fused key derivation (learner:426-434) from the rollout rng, global env index
                    // the first four lanes of the group share the Threefry blocks (five dependent levels
                    // instead of thirteen blocks on one thread while the rest of the group waits)
                    if (gt < 4) {
                        const int base_lane = GS < 32 ? (int)(threadIdx.x & 31u & (32u - GS)) : 0;
                        uint32_t c6 = 0u, c7 = 0u, c8 = 0u, c9 = 0u, r0 = 0u, r1 = 0u, np, k0, k1;
                        if (MULTI) {
                            c6 = s_chain[10 * j + 6]; c7 = s_chain[10 * j + 7];
                            c8 = s_chain[10 * j + 8]; c9 = s_chain[10 * j + 9];
                        } else {
                            r0 = a.rng_in[0]; r1 = a.rng_in[1];
                        }
                        env_reset_inputs_4lanes(0xFu << base_lane, gt, base_lane, MULTI, r0, r1, c6, c7, c8, c9, a.Bg,
                                                a.env_off + (uint32_t)e, (uint32_t)a.P, np, k0, k1);
                        if (gt == 0) {
                            misc[1] = (int)np;
                            misc[2] = (int)k0;
                            misc[3] = (int)k1;
                        }
                    }
                    group_sync<GS>(gid);
                    pidx = misc[1];
                    rk0 = (uint32_t)misc[2];
                    rk1 = (uint32_t)misc[3];
                } else {
                    pidx = a.prob_idx[e];
                    rk0 = a.keys[2 * (size_t)e];
                    rk1 = a.keys[2 * (size_t)e + 1];
                }
                pidx = clamp_problem(pidx, a.P);
                // the full evaluation of the new episode needs the literal block (an incremental step had the
                // occurrence lists in the slot)
                const bool need_lits = pidx != loaded_pidx || (INCR && loaded_csr);
                if (gt == 0) {
                    misc[0] = d.m;
                    if (a.reset_count) atomicAdd(a.reset_count, 1ULL);
                    if (need_lits) {
                        fence_proxy_async();
                        mbar_expect_tx(bar, tma_bytes);
                        tma_load_1d(rec, a.bank + (size_t)pidx * d.rec_bytes, tma_bytes, bar);
                    }
                }
                for (int i = gt; i < d.aw; i += GS) st[i] = 0u;
                if (cnt_store)
                    for (int i = gt; i < d.cnt_words; i += GS) cnt_store[i] = 0u;
                group_sync<GS>(gid);
                threefry_assign<GS>(d, rk0, rk1, st, gt);
                group_sync<GS>(gid);
                build_truth_table<GS>(d, st, tt, gt);
                if (need_lits) {
                    mbar_wait(bar, phase);
                    phase ^= 1u;
                    loaded_pidx = pidx;
                    loaded_csr = false;
                }
                group_sync<GS>(gid);
                // the clause features of the finished episode are already on their way to the same rows: let
                // those bulk stores complete before the new episode's features are sent after them
                if (cf_row) {
                    if (gt == 0) tma_store_wait();
                    group_sync<GS>(gid);
                }
                run_eval<GS, false, OBS>(d, lits, tt, cnt_store, satw, &misc[0], cf01, stage, cf_row, pairs, gid, gt);
                group_sync<GS>(gid);
                nunsat = misc[0];
                step_cur = 0;
                flags = 0u;
            } else {
                step_cur += 1;                                               // env:269
                flags = done ? 1u : 0u;                                      // env:270
            }
            nunsat_prev = nunsat;
        }
        if (emit) {
            if (!OBS && a.gnn_assign) emit_gnn_assignment<GS>(d, row, st, a.gnn_assign, gt);
            if (OBS && a.obs) {
                if (a.obs_i8) emit_obs<GS, true>(d, row, st, satw, X, smx, mflat, a.obs, gid, gt);
                else emit_obs<GS, false>(d, row, st, satw, X, smx, mflat, a.obs, gid, gt);
            }
        }
        if (!last) {
            if (cf_row && gt == 0) tma_store_wait_read();   // the staging buffer is rewritten by the next step
            group_sync<GS>(gid);           // every lane has read misc[0] / the state of this step
            if (gt == 0) misc[0] = d.m;    // published by the barrier after the next step's flips
        }
    }

    // a CTA must not retire while the bulk-copy engine still reads its shared memory
    if (want_cf && gt == 0) tma_store_wait_read();
    if (MODE != MODE_OBS) {
        group_sync<GS>(gid);
        if (gt == 0) {
            st_tail[ST_STEP] = (uint32_t)step_cur;                           // env:170,269
            st_tail[ST_PIDX] = (uint32_t)pidx;
            st_tail[ST_NUNSAT] = (uint32_t)nunsat;
            st_tail[ST_FLAGS] = flags;                                       // env:171,270
        }
        group_sync<GS>(gid);
        uint4* sout = reinterpret_cast<uint4*>(a.state_out + (size_t)e * d.state_words);
#pragma unroll 1
        for (int i = gt; i < (d.state_words >> 2); i += GS) sout[i] = reinterpret_cast<const uint4*>(st)[i];
    }
}

template <int GS, bool OBS>
static cudaError_t launch_env_gs(const msat_plan* plan, EnvMode mode, const EnvArgs& a, cudaStream_t s, int smem_bytes) {
    const int groups = kCtaThreads / GS;
    const int grid = (a.B + groups - 1) / groups;
    if (grid == 0) return cudaSuccess;
    // every instantiation a launch with this (GS, OBS) can select: the shared-memory opt-in below covers them all.
    // The single-step kernels sit at index `mode`, then the multi-step one, then the incremental clause update's
    // single- and multi-step kernels (step launches without observations on a plan that carries the counts).
    constexpr int kFns = OBS ? 6 : 8;
    const void* fns[8] = {(const void*)env_kernel<GS, MODE_RESET, OBS, false, false>,
                          (const void*)env_kernel<GS, MODE_STEP, OBS, false, false>,
                          (const void*)env_kernel<GS, MODE_OBS, OBS, false, false>,
                          (const void*)env_kernel<GS, MODE_IMPORT, OBS, false, false>,
                          (const void*)env_kernel<GS, MODE_START, OBS, false, false>,
                          (const void*)env_kernel<GS, MODE_STEP, OBS, true, false>,
                          OBS ? nullptr : (const void*)env_kernel<GS, MODE_STEP, false, false, true>,
                          OBS ? nullptr : (const void*)env_kernel<GS, MODE_STEP, false, true, true>};
    const bool multi = mode == MODE_STEP && a.num_steps > 1;
    const bool incr = !OBS && mode == MODE_STEP && plan->d.cnt_words > 0;
    if (multi) smem_bytes += 40 * a.num_steps;
    if (smem_bytes > 48 * 1024) {
        // opt in to > 48 KB of dynamic shared memory once per (plan, device), not once per launch
        int dev = 0;
        cudaError_t err = cudaGetDevice(&dev);
        if (err != cudaSuccess) return err;
        const unsigned long long bit = 1ULL << ((OBS ? 0 : 32) + (dev & 31));
        if (!(plan->prepared_devices.load(std::memory_order_acquire) & bit)) {
            for (int i = 0; i < kFns; ++i) {
                err = cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemOptin);
                if (err != cudaSuccess) return err;
            }
            plan->prepared_devices.fetch_or(bit, std::memory_order_release);
        }
    }
    const void* fn = fns[incr ? 6 + (int)multi : (multi ? 5 : (int)mode)];
    Dims d = plan->d;
    EnvArgs args = a;
    void* params[] = {&d, &args};
    return cudaLaunchKernel(fn, dim3(grid), dim3(kCtaThreads), params, (size_t)smem_bytes, s);
}

cudaError_t launch_env(const msat_plan* plan, EnvMode mode, const EnvArgs& a0, cudaStream_t s) {
    // the group size follows the work per env: observation-writing launches use the plan's GS, launches
    // without observations the small-group variant
    EnvArgs a = a0;
    if (a.num_steps < 1) a.num_steps = 1;
    const bool noobs = a.obs == nullptr;
    a.L = noobs ? plan->layout_noobs : plan->layout_obs;
    a.obs_i8 = plan->obs_i8;
    const int gs = noobs ? plan->group_threads_noobs : plan->group_threads;
    const int smem = noobs ? plan->smem_bytes_noobs : plan->smem_bytes;
    if (noobs) {
        switch (gs) {
            case 32: return launch_env_gs<32, false>(plan, mode, a, s, smem);
            case 64: return launch_env_gs<64, false>(plan, mode, a, s, smem);
            case 128: return launch_env_gs<128, false>(plan, mode, a, s, smem);
            default: return launch_env_gs<256, false>(plan, mode, a, s, smem);
        }
    }
    switch (gs) {
        case 16: return launch_env_gs<16, true>(plan, mode, a, s, smem);
        case 32: return launch_env_gs<32, true>(plan, mode, a, s, smem);
        case 64: return launch_env_gs<64, true>(plan, mode, a, s, smem);
        case 128: return launch_env_gs<128, true>(plan, mode, a, s, smem);
        default: return launch_env_gs<256, true>(plan, mode, a, s, smem);
    }
}

cudaError_t launch_compile_bank(const msat_plan* plan, const int32_t* clauses, int P, uint8_t* bank, cudaStream_t s) {
    if (P == 0) return cudaSuccess;
    if (plan->compile_smem_bytes > 48 * 1024) {
        cudaError_t err = cudaFuncSetAttribute((const void*)compile_bank_kernel,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, plan->compile_smem_bytes);
        if (err != cudaSuccess) return err;
    }
    compile_bank_kernel<<<P, 256, plan->compile_smem_bytes, s>>>(plan->d, clauses, bank);
    return cudaGetLastError();
}

// =====================================================================================
// K_export: reference-shaped SATState leaves (env:13-24) from packed state + bank.  Off the hot
// path (API fidelity, parity tests); one 128-thread CTA per env, global-memory reads only.
// =====================================================================================
__global__ void __launch_bounds__(128) export_kernel(const Dims d, const ExportArgs a) {
    const int e = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const uint32_t* st = a.state + (size_t)e * d.state_words;
    const uint32_t* tail = st + d.aw;
    const int pidx = clamp_problem((int)tail[ST_PIDX], a.P);
    const uint8_t* rec = a.bank + (size_t)pidx * d.rec_bytes;
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(rec);
    const uint32_t* mflat = reinterpret_cast<const uint32_t*>(rec + d.lits_bytes);
    if (a.assign)
        for (int v = tid; v < d.n; v += nt) a.assign[(size_t)e * d.n + v] = (st[v >> 5] >> (v & 31)) & 1u;
    if (a.sat)
        for (int c = tid; c < d.m; c += nt) {
            bool sat = false;
            for (int j = 0; j < d.k; ++j) {
                const uint32_t code = lits[lit_index(d.ms, c, j)];
                if (code != lit_pad(d)) {
                    const uint32_t v = code >> 1;
                    sat |= (((st[v >> 5] >> (v & 31)) ^ code) & 1u) != 0u;
                }
            }
            a.sat[(size_t)e * d.m + c] = sat ? 1 : 0;
        }
    if (tid == 0) {
        if (a.num_unsat) a.num_unsat[e] = (int)tail[ST_NUNSAT];
        if (a.step) a.step[e] = (int)tail[ST_STEP];
        if (a.pidx) a.pidx[e] = pidx;
    }
    if (a.done)
        for (int i = tid; i < d.A; i += nt) a.done[(size_t)e * d.A + i] = (uint8_t)(tail[ST_FLAGS] & 1u);
    if (a.clauses || a.l2a)
        for (int i = tid; i < d.m * d.k; i += nt) {
            const uint32_t code = lits[lit_index(d.ms, i / d.k, i % d.k)];
            const int v = (code == lit_pad(d)) ? -1 : (int)(code >> 1);
            if (a.clauses) a.clauses[(size_t)e * d.m * d.k + i] = v < 0 ? 0 : ((code & 1u) ? -(v + 1) : (v + 1));
            // env:160: index -1 wraps to the last variable
            if (a.l2a) a.l2a[(size_t)e * d.m * d.k + i] = var_to_agent(d, v < 0 ? d.n - 1 : v);
        }
    if (a.acm)
        for (int i = tid; i < d.A * d.m; i += nt) {
            const int ag = i / d.m, c = i - ag * d.m;
            const int j = ag * d.D + d.n + c;
            a.acm[(size_t)e * d.A * d.m + i] = ((mflat[j >> 5] >> (j & 31)) & 1u) ? 1 : -1;
        }
    if (a.anm)
        for (int i = tid; i < d.A * d.n; i += nt) {
            const int ag = i / d.n, v = i - ag * d.n;
            const int j = ag * d.D + d.n + d.m + v;
            a.anm[(size_t)e * d.A * d.n + i] = ((mflat[j >> 5] >> (j & 31)) & 1u) ? 1 : -1;
        }
}

cudaError_t launch_export(const msat_plan* plan, const ExportArgs& a, cudaStream_t s) {
    if (a.B == 0) return cudaSuccess;
    export_kernel<<<a.B, 128, 0, s>>>(plan->d, a);
    return cudaGetLastError();
}

}  // namespace msat
