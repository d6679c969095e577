// Batched WalkSAT/SKC over packed env states (msat_walksat; the algorithm contract is in
// include/marl_sat_b200.h and oracle/walksat.py).  One warp owns one env: it stages the formula's literal block
// with one TMA bulk copy, builds the var -> clause occurrence lists, the u8 true-literal counts and the
// unsatisfied-clause bits in its own slice of shared memory, and then runs the whole flip loop warp-locally --
// no global-memory traffic and no CTA barrier until it writes the state back.  A warp retires as soon as its
// env is solved.
#include "internal.h"

namespace msat {

namespace {

constexpr uint32_t kFull = 0xFFFFFFFFu;

__device__ __forceinline__ int warp_incl_scan(int x, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(kFull, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

// bit position of the nth (0-based) set bit of x; x has more than nth set bits
__device__ __forceinline__ int nth_set_bit(uint32_t x, int nth) {
    int pos = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int lo = __popc(x & ((1u << s) - 1u));
        if (nth >= lo) {
            nth -= lo;
            x >>= s;
            pos += s;
        }
    }
    return pos;
}

// index of the rank-th (0-based) set bit of the sw-word bit array `bits`; rank < total popcount
__device__ __forceinline__ int rank_select(const uint32_t* bits, int sw, uint32_t rank, int lane) {
    for (int w0 = 0; w0 < sw; w0 += 32) {
        const uint32_t word = w0 + lane < sw ? bits[w0 + lane] : 0u;
        const int pc = __popc(word);
        const int incl = warp_incl_scan(pc, lane);
        const uint32_t total = (uint32_t)__shfl_sync(kFull, incl, 31);
        if (rank < total) {
            const int L = __ffs(__ballot_sync(kFull, (uint32_t)incl > rank)) - 1;
            const uint32_t wl = __shfl_sync(kFull, word, L);
            const int before = __shfl_sync(kFull, incl - pc, L);
            return (w0 + L) * 32 + nth_set_bit(wl, (int)rank - before);
        }
        rank -= total;
    }
    return 0;   // not reached: rank < popcount
}

}  // namespace

__global__ void __launch_bounds__(kWalksatMaxWarps * 32) walksat_kernel(const Dims d, const WalksatLayout L,
                                                                        const WalksatArgs a) {
    extern __shared__ __align__(128) uint8_t ls_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int e = blockIdx.x * (blockDim.x >> 5) + wid;
    if (e >= a.B) return;                       // whole warp leaves together

    uint8_t* base = ls_smem + (size_t)wid * L.total;
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(base + L.lits);
    uint16_t* occ = reinterpret_cast<uint16_t*>(base + L.occ);
    int* row = reinterpret_cast<int*>(base + L.row);
    uint8_t* cnt8 = base + L.cnt;
    uint32_t* cntw = reinterpret_cast<uint32_t*>(base + L.cnt);
    uint32_t* unsat = reinterpret_cast<uint32_t*>(base + L.unsat);
    uint32_t* dupw = reinterpret_cast<uint32_t*>(base + L.dup);
    uint32_t* assign = reinterpret_cast<uint32_t*>(base + L.assign);
    int* brk = reinterpret_cast<int*>(base + L.brk);
    uint64_t* bar = reinterpret_cast<uint64_t*>(base + L.bar);
    uint32_t* st = a.state + (size_t)e * d.state_words;
    const uint32_t pad = lit_pad(d);

    const int pidx = clamp_problem((int)st[d.aw + ST_PIDX], a.P);
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, (uint32_t)d.lits_bytes);
        tma_load_1d(base + L.lits, a.bank + (size_t)pidx * d.rec_bytes, (uint32_t)d.lits_bytes, bar);
    }
    // while the literal block is in flight
    for (int i = lane; i < d.aw; i += 32) assign[i] = st[i];
    for (int v = lane; v < d.n; v += 32) row[v] = 0;
    const uint32_t k0 = a.keys[2 * (size_t)e], k1 = a.keys[2 * (size_t)e + 1];
    __syncwarp();
    mbar_wait(bar, 0u);

    // ---- per clause (lane = clause): true-literal count, repeated variable, occurrence counts ----
    int U = 0;
    for (int c0 = 0; c0 < d.m; c0 += 32) {
        const int c = c0 + lane;
        uint32_t ntrue = 0u;
        bool dup = false;
        if (c < d.m) {
            for (int j = 0; j < d.k; ++j) {
                const uint32_t code = lits[lit_index(d.ms, c, j)];
                if (code == pad) continue;
                const uint32_t v = code >> 1;
                atomicAdd(&row[v], 1);
                ntrue += ((assign[v >> 5] >> (v & 31)) ^ code) & 1u;
                for (int i = 0; i < j; ++i) dup |= (uint32_t)(lits[lit_index(d.ms, c, i)] >> 1) == v;   // padding: n != v
            }
            cnt8[c] = (uint8_t)ntrue;
        }
        const uint32_t uw = __ballot_sync(kFull, c < d.m && ntrue == 0u);
        const uint32_t dw = __ballot_sync(kFull, c < d.m && dup);
        if (lane == 0) {
            unsat[c0 >> 5] = uw;
            dupw[c0 >> 5] = dw;
        }
        U += __popc(uw);
    }
    __syncwarp();
    // exclusive prefix of the occurrence counts
    int carry = 0;
    for (int v0 = 0; v0 < d.n; v0 += 32) {
        const int v = v0 + lane;
        const int x = v < d.n ? row[v] : 0;
        const int incl = warp_incl_scan(x, lane);
        if (v < d.n) row[v] = carry + incl - x;
        carry += __shfl_sync(kFull, incl, 31);
    }
    __syncwarp();
    // scatter: afterwards row[v] is the end of v's list and row[v - 1] (0 for v = 0) its start
    for (int c = lane; c < d.m; c += 32)
        for (int j = 0; j < d.k; ++j) {
            const uint32_t code = lits[lit_index(d.ms, c, j)];
            if (code == pad) continue;
            occ[atomicAdd(&row[code >> 1], 1)] = (uint16_t)((c << 1) | (code & 1u));
        }
    __syncwarp();

    // ---- flip loop ----
    int t = 0;
    for (; t < a.max_flips && U > 0; ++t) {
        uint32_t x0 = (uint32_t)a.flip_offset + (uint32_t)t, x1 = 0u;
        threefry2x32(k0, k1, x0, x1);
        const int c = rank_select(unsat, d.sw, __umulhi(x0, (uint32_t)U), lane);
        // candidates: lane j = literal column j of the picked clause
        const uint32_t code = lane < d.k ? lits[lit_index(d.ms, c, lane)] : pad;
        const bool cand = code != pad;
        const uint32_t cmask = __ballot_sync(kFull, cand);
        if (cmask == 0u) continue;                              // all-padding clause: the iteration still counts
        const int v = (int)(code >> 1);
        const int vs = cand ? (v ? row[v - 1] : 0) : 0;
        const int deg = cand ? row[v] - vs : 0;
        const int incl = warp_incl_scan(deg, lane);
        const int excl = incl - deg;
        const int total = __shfl_sync(kFull, incl, 31);
        brk[lane] = 0;
        __syncwarp();
        // break counts: lanes spread over the (candidate, occurrence) pairs
        for (int p0 = 0; p0 < total; p0 += 32) {
            const int p = p0 + lane;
            int j = 0;
            for (int jj = 1; jj < d.k; ++jj) {                  // the column whose pair range holds p
                const int s = __shfl_sync(kFull, excl, jj), dg = __shfl_sync(kFull, deg, jj);
                if (dg > 0 && p >= s) j = jj;
            }
            const int vj = __shfl_sync(kFull, v, j), sj = __shfl_sync(kFull, vs, j), ej = __shfl_sync(kFull, excl, j);
            if (p < total) {
                const int idx = sj + (p - ej);
                const uint32_t ent = occ[idx];
                const int cc = (int)(ent >> 1);
                const uint32_t av = (assign[vj >> 5] >> (vj & 31)) & 1u;
                bool b = false;
                if ((av ^ ent) & 1u) {                          // this literal is true
                    const uint32_t nt = cnt8[cc];
                    if (!((dupw[cc >> 5] >> (cc & 31)) & 1u)) {
                        b = nt == 1u;                           // it is the clause's only true literal
                    } else {
                        // the variable occurs more than once in the clause: count the clause once (at its first
                        // entry in v's list) and only if every true literal is on v and none is false
                        bool first = true;
                        for (int q = sj; q < idx; ++q) first &= (int)(occ[q] >> 1) != cc;
                        uint32_t tv = 0u, fv = 0u;
                        for (int i = 0; i < d.k; ++i) {
                            const uint32_t ci = lits[lit_index(d.ms, cc, i)];
                            if (ci == pad || (int)(ci >> 1) != vj) continue;
                            if ((av ^ ci) & 1u) ++tv;
                            else ++fv;
                        }
                        b = first && fv == 0u && nt == tv;
                    }
                }
                if (b) atomicAdd(&brk[j], 1);
            }
        }
        __syncwarp();
        const int bj = cand ? brk[lane] : 0x7FFFFFFF;
        const uint32_t zmask = __ballot_sync(kFull, cand && bj == 0);
        int col;
        if (zmask) {
            col = __ffs(zmask) - 1;                                            // freebie
        } else if ((x1 >> 8) < a.thr) {
            col = nth_set_bit(cmask, (int)(((x1 & 0xFFu) * (uint32_t)__popc(cmask)) >> 8));   // random walk
        } else {
            const int mn = __reduce_min_sync(kFull, bj);
            col = __ffs(__ballot_sync(kFull, cand && bj == mn)) - 1;           // greedy
        }
        // flip: lanes spread over the flipped variable's occurrences
        const int fv = __shfl_sync(kFull, v, col), fs = __shfl_sync(kFull, vs, col), fd = __shfl_sync(kFull, deg, col);
        const uint32_t af = (assign[fv >> 5] >> (fv & 31)) & 1u;
        int du = 0;
        for (int q = lane; q < fd; q += 32) {
            const uint32_t ent = occ[fs + q];
            const int cc = (int)(ent >> 1);
            const bool was_true = ((af ^ ent) & 1u) != 0u;
            const int sh = 8 * (cc & 3);
            // a count never drops below the number of true literals being removed, so no borrow leaves the byte
            const uint32_t old = atomicAdd(&cntw[cc >> 2], was_true ? 0u - (1u << sh) : 1u << sh);
            const uint32_t ob = (old >> sh) & 0xFFu, nb = was_true ? ob - 1u : ob + 1u;
            if ((ob == 0u) != (nb == 0u)) {
                atomicXor(&unsat[cc >> 5], 1u << (cc & 31));
                du += nb == 0u ? 1 : -1;
            }
        }
        U += __reduce_add_sync(kFull, du);
        __syncwarp();
        if (lane == 0) assign[fv >> 5] ^= 1u << (fv & 31);
        __syncwarp();
    }

    // ---- write back: assignment, num_unsatisfied and an incremental plan's 4-bit counts ----
    for (int i = lane; i < d.aw; i += 32) st[i] = assign[i];
    for (int i = lane; i < d.cnt_words; i += 32) {
        uint32_t w = 0u;
        for (int q = 0; q < 8 && 8 * i + q < d.m; ++q) w |= (uint32_t)cnt8[8 * i + q] << (4 * q);
        st[d.aw + 4 + i] = w;
    }
    if (lane == 0) {
        st[d.aw + ST_NUNSAT] = (uint32_t)U;
        if (a.solved) a.solved[e] = U == 0 ? 1 : 0;
        if (a.flips) a.flips[e] = t;
    }
}

cudaError_t launch_walksat(const msat_plan* plan, const WalksatArgs& a, cudaStream_t s) {
    if (a.B == 0) return cudaSuccess;
    const Dims& d = plan->d;
    const WalksatLayout L = walksat_layout(d);
    const int warps = walksat_warps(d);
    const int smem = warps * L.total;
    if (smem > 48 * 1024) {
        // opt in to > 48 KB of dynamic shared memory once per (plan, device), not once per launch
        int dev = 0;
        cudaError_t err = cudaGetDevice(&dev);
        if (err != cudaSuccess) return err;
        const unsigned long long bit = 1ULL << (dev & 63);
        if (!(plan->prepared_walksat.load(std::memory_order_acquire) & bit)) {
            err = cudaFuncSetAttribute((const void*)walksat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kMaxSmemOptin);
            if (err != cudaSuccess) return err;
            plan->prepared_walksat.fetch_or(bit, std::memory_order_release);
        }
    }
    walksat_kernel<<<(a.B + warps - 1) / warps, 32 * warps, smem, s>>>(d, L, a);
    return cudaGetLastError();
}

}  // namespace msat
