// nastar_generic.cuh — engine for maps of any shape (H or W > 32): forward search and backward replay.
//
// Same state machine as the warp32 engine (DifferentiableAstar.forward loop + backtrack,
// /root/reference/src/neural_astar/planner/differentiable_astar.py:187-255), one map per warp,
// but rows no longer fit a lane's registers:
//   * passable / open / closed / path rows are bit arrays in shared memory ([H][ceil(W/32)]);
//   * every row caches its best open cell (f key, column) in shared memory; lane l folds the rows
//     {l, l+32, ...} into a register pair, so selection is still two REDUX.MINs;
//   * a step relaxes <= 8 neighbours (lanes 0..8 take one cell each), rescans only row r with all
//     lanes, and re-folds the <= 3 touched rows — O(W/32 + H/32) per step, never O(H*W);
//   * h is evaluated lazily when a cell is first opened, so the g / f / parent planes need no
//     initialisation; the parent is stored as a 1-byte Moore direction code.
//   kGlobal = false: cost (TMA bulk copy), g, f, parent live in shared memory (N <= ~16k cells,
//                    i.e. up to 128x128);
//   kGlobal = true : g, f, parent live in a per-CTA slot of the HBM workspace (L2 resident),
//                    cost is read through the read-only path; persistent CTAs loop over maps.
#pragma once
#include "../../include/nastar_b200.h"
#include "nastar_common.cuh"

namespace nastar {

struct GenericLayout {
    int H, W, N, Wd, nbits;  // nbits = H*Wd words per bit array
    __host__ __device__ GenericLayout(int h, int w) : H(h), W(w), N(h * w), Wd((w + 31) >> 5), nbits(h * ((w + 31) >> 5)) {}
    __host__ __device__ int npad() const { return (N + 3) & ~3; }
    // shared-memory bytes that every variant needs: 3 bit arrays (the path rows reuse the passable rows once the
    // search is over) + row-min cache + mbarrier
    __host__ __device__ size_t smem_common() const { return size_t(3) * nbits * 4 + size_t(H) * 8 + 16; }
    // planes kept in shared memory by the !kGlobal variant: cost, g, f (fp32) + parent (u8)
    __host__ __device__ size_t smem_planes() const { return size_t(npad()) * 13; }
    // per-CTA workspace slot of the kGlobal variant: g, f (fp32) + parent (u8)
    __host__ __device__ size_t slot_bytes() const { return (size_t(npad()) * 9 + 255) & ~size_t(255); }
    // backward adds per slot, always in the workspace: acc (fp64), A0 and B0 (fp64: prefix sums at the start of the
    // cell's current open interval) and v (fp32) — 28 B per cell
    __host__ __device__ size_t bwd_bytes() const { return (size_t(npad()) * 28 + 255) & ~size_t(255); }
    __host__ __device__ size_t slot_total(bool global_state, bool bwd) const {
        return (global_state ? slot_bytes() : 0) + (bwd ? bwd_bytes() : 0);
    }
};

// kBwd = true replays the search for *T_batch steps and accumulates the closed-form gradient (SURVEY App. B)
// EVENT-BASED (IntervalPlanes, nastar_common.cuh): S and D are maintained incrementally in fp64 from the <= 9 events
// of a step — O(1) work per step instead of a dense O(N/32) softmax pass (round 1).  Per-cell state (v, A(t0), B(t0),
// acc) lives in the per-CTA workspace slot.
// kNoExit (forward only): NASTAR_FWD_NO_EARLY_EXIT — keep stepping after the solve step, exactly T steps.
template <bool kGlobal, bool kTrace, bool kBwd, bool kNoExit = false>
__global__ void __launch_bounds__(32) astar_generic_kernel(const SearchArgs a) {
    constexpr bool kContinue = kBwd || kNoExit;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const nastar_fwd_params& p = a.f;
    const int lane = threadIdx.x;
    const GenericLayout L(p.H, p.W);
    const int H = L.H, W = L.W, N = L.N, Wd = L.Wd;
    const int np = L.npad();

    // ---- carve shared memory ----------------------------------------------------------------
    unsigned char* sp = smem_raw;
    float* sCost = nullptr;
    float* G;
    float* F;
    uint8_t* Par;
    if (!kGlobal) {
        sCost = reinterpret_cast<float*>(sp); sp += size_t(np) * 4;
        G = reinterpret_cast<float*>(sp); sp += size_t(np) * 4;
        F = reinterpret_cast<float*>(sp); sp += size_t(np) * 4;
        Par = reinterpret_cast<uint8_t*>(sp); sp += size_t(np);
    } else {
        unsigned char* slot = static_cast<unsigned char*>(p.workspace) + size_t(blockIdx.x) * L.slot_total(true, kBwd);
        G = reinterpret_cast<float*>(slot);
        F = G + np;
        Par = reinterpret_cast<uint8_t*>(F + np);
    }
    IntervalPlanes iv{};    // backward only
    if (kBwd) {
        unsigned char* slot = static_cast<unsigned char*>(p.workspace) + size_t(blockIdx.x) * L.slot_total(kGlobal, true) +
                              (kGlobal ? L.slot_bytes() : 0);
        iv.acc = reinterpret_cast<double*>(slot);
        iv.a0 = iv.acc + np;
        iv.b0 = iv.a0 + np;
        iv.v = reinterpret_cast<float*>(iv.b0 + np);
    }
    uint32_t* sPass = reinterpret_cast<uint32_t*>(sp); sp += size_t(L.nbits) * 4;
    uint32_t* sOpen = reinterpret_cast<uint32_t*>(sp); sp += size_t(L.nbits) * 4;
    uint32_t* sClosed = reinterpret_cast<uint32_t*>(sp); sp += size_t(L.nbits) * 4;
    uint32_t* sPath = sPass;  // the passable rows are dead once the loop ends; the backtrack reuses them
    uint32_t* sRmKey = reinterpret_cast<uint32_t*>(sp); sp += size_t(H) * 4;
    int32_t* sRmCol = reinterpret_cast<int32_t*>(sp); sp += size_t(H) * 4;
    uint64_t* bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(sp) + 7) & ~uintptr_t(7));

    const float gr = p.g_ratio, omg = p.one_minus_g_ratio;
    const int Tb = kBwd ? *a.T_batch : 0;
    const int T = kBwd ? Tb : p.T;
    const bool stationary_ok = (gr >= 0.5f);
    uint32_t bar_parity = 0;
    if (!kGlobal) {
        if (lane == 0) { mbar_init(bar, 1); fence_mbar_init(); }
        __syncwarp();
    }

    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
        if (!kBwd && a.redo != nullptr && a.redo[b] == 0) continue;
        const float* gCost = p.cost + int64_t(b) * p.cost_stride;
        const float* gStart = p.start + int64_t(b) * p.start_stride;
        const float* gGoal = p.goal + int64_t(b) * p.goal_stride;
        const float* gObst = p.obst + int64_t(b) * p.obst_stride;

        // ---- prologue: cost plane -> smem (TMA), bit rows from obstacle/start/goal planes -------
        if (!kGlobal) {
            const bool tma_ok = ((N & 3) == 0) && aligned16(gCost);
            if (tma_ok) {
                if (lane == 0) {
                    fence_proxy_async();  // earlier generic-proxy accesses to sCost (previous map) are ordered
                    mbar_expect_tx(bar, uint32_t(N) * 4u);
                    tma_load_1d(sCost, gCost, uint32_t(N) * 4u, bar);
                }
            } else {
                for (int i = lane; i < N; i += 32) sCost[i] = __ldg(gCost + i);
            }
            (void)tma_ok;
        }
        int start_idx = -1, goal_idx = -1;
        const bool vec = ((W & 31) == 0) && aligned16(gObst) && aligned16(gStart) && aligned16(gGoal);
        if (vec) {
            // Rows are whole 32-bit words (flat bit index == row-word index): stream the planes with
            // 128-bit loads, kUnroll segments of 128 cells in flight per plane (the prologue is a pure
            // HBM stream; with one warp per map the only way to cover DRAM latency is load-level parallelism)
            constexpr int kUnroll = 8;
            const int nseg = (N + 127) >> 7;   // the last segment may be partial (N is a multiple of 32, not of 128)
            const int nq = N >> 2;             // float4 count of a plane
            const float4* o4 = reinterpret_cast<const float4*>(gObst);
            const float4* s4 = reinterpret_cast<const float4*>(gStart);
            const float4* g4 = reinterpret_cast<const float4*>(gGoal);
            for (int seg0 = 0; seg0 < nseg; seg0 += kUnroll) {
                float4 vo[kUnroll], vs[kUnroll], vg[kUnroll];
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) {
                    const int q = ((seg0 + u) << 5) + lane;
                    const bool in = q < nq;
                    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    vo[u] = in ? __ldg(o4 + q) : z;
                    vs[u] = in ? __ldg(s4 + q) : z;
                    vg[u] = in ? __ldg(g4 + q) : z;
                }
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) {
                    if ((seg0 + u) < nseg) {
                        // lane l holds cells 4l..4l+3 of the segment; word k = lanes 8k..8k+7
                        uint32_t nib = (vo[u].x != 0.f ? 1u : 0u) | (vo[u].y != 0.f ? 2u : 0u) |
                                       (vo[u].z != 0.f ? 4u : 0u) | (vo[u].w != 0.f ? 8u : 0u);
                        uint32_t word = nib << ((lane & 7) << 2);
                        word |= __shfl_xor_sync(kFull, word, 1);
                        word |= __shfl_xor_sync(kFull, word, 2);
                        word |= __shfl_xor_sync(kFull, word, 4);
                        if ((lane & 7) == 0 && ((seg0 + u) << 2) + (lane >> 3) < L.nbits)
                            sPass[((seg0 + u) << 2) + (lane >> 3)] = word;
                        const bool hs = (vs[u].x != 0.f) | (vs[u].y != 0.f) | (vs[u].z != 0.f) | (vs[u].w != 0.f);
                        const bool hg = (vg[u].x != 0.f) | (vg[u].y != 0.f) | (vg[u].z != 0.f) | (vg[u].w != 0.f);
                        const uint32_t bs = __ballot_sync(kFull, hs), bg = __ballot_sync(kFull, hg);
                        if (start_idx < 0 && bs) {
                            const int src = __ffs(bs) - 1;
                            const int e = (vs[u].x != 0.f) ? 0 : (vs[u].y != 0.f) ? 1 : (vs[u].z != 0.f) ? 2 : 3;
                            start_idx = ((seg0 + u) << 7) + (src << 2) + __shfl_sync(kFull, e, src);
                        }
                        if (goal_idx < 0 && bg) {
                            const int src = __ffs(bg) - 1;
                            const int e = (vg[u].x != 0.f) ? 0 : (vg[u].y != 0.f) ? 1 : (vg[u].z != 0.f) ? 2 : 3;
                            goal_idx = ((seg0 + u) << 7) + (src << 2) + __shfl_sync(kFull, e, src);
                        }
                    }
                }
            }
        } else {
            for (int y = 0; y < H; ++y) {
                for (int w = 0; w < Wd; ++w) {
                    const int x = (w << 5) + lane;
                    const bool in = x < W;
                    const int i = y * W + x;
                    const float vo = in ? __ldg(gObst + i) : 0.f;
                    const float vs = in ? __ldg(gStart + i) : 0.f;
                    const float vg = in ? __ldg(gGoal + i) : 0.f;
                    const uint32_t wo = __ballot_sync(kFull, vo != 0.f);
                    const uint32_t ws = __ballot_sync(kFull, vs != 0.f);
                    const uint32_t wg = __ballot_sync(kFull, vg != 0.f);
                    if (lane == 0) sPass[y * Wd + w] = wo;
                    if (start_idx < 0 && ws) start_idx = y * W + (w << 5) + __ffs(ws) - 1;
                    if (goal_idx < 0 && wg) goal_idx = y * W + (w << 5) + __ffs(wg) - 1;
                }
            }
        }
        if (goal_idx < 0) goal_idx = 0;
        for (int i = lane; i < L.nbits; i += 32) { sOpen[i] = 0u; sClosed[i] = 0u; }
        for (int y = lane; y < H; y += 32) { sRmKey[y] = kKeyInf; sRmCol[y] = 0; }
        if (!kGlobal) {
            if (((N & 3) == 0) && aligned16(gCost)) { mbar_wait(bar, bar_parity); bar_parity ^= 1u; }
        }
        __syncwarp();
        const int gy = goal_idx / W, gx = goal_idx - gy * W;
        auto cost_at = [&](int i) -> float { return kGlobal ? __ldg(gCost + i) : sCost[i]; };

        int ts_in = NASTAR_TS_CAPPED;
        bool blocked = false;
        const float* gG = nullptr;
        if (kBwd) {
            ts_in = a.t_solve_in[b];
            blocked = (ts_in >= 0) && (ts_in < Tb - 1);   // goal clamp, differentiable_astar.py:222-223
            gG = a.grad_hist + int64_t(b) * a.grad_stride;
            for (int i = lane; i < N; i += 32) { iv.v[i] = 0.f; iv.acc[i] = 0.0; }
            __syncwarp();
        }
        // backward running sums (replicated in every lane): S = sum of v over the open set, D = <Gh, v>,
        // A / B = prefix sums of 1/S and D/S^2 over the steps executed so far
        double Ssum = 0.0, Slo = 0.0, Dsum = 0.0, Dlo = 0.0, Acum = 0.0, Bcum = 0.0;   // (Ssum,Slo), (Dsum,Dlo): double-double
        auto gh_at = [&](int i) -> float { return (blocked && i == goal_idx) ? 0.f : __ldg(gG + i); };
        if (start_idx >= 0 && lane == 0) {
            const int sy = start_idx / W, sx = start_idx - sy * W;
            const float h0 = __fadd_rn(heuristic(sy, sx, gy, gx), cost_at(start_idx));
            const float f0 = f_value(gr, omg, 0.f, h0);
            G[start_idx] = 0.f;
            F[start_idx] = f0;
            if (kBwd) { iv.v[start_idx] = expf(__fdiv_rn(-f0, a.sqrt_w)); iv.a0[start_idx] = 0.0; iv.b0[start_idx] = 0.0; }
            sOpen[sy * Wd + (sx >> 5)] = 1u << (sx & 31);
            sRmKey[sy] = fkey(f0);
            sRmCol[sy] = sx;
        }
        __syncwarp();
        if (kBwd && start_idx >= 0) {
            Ssum = double(iv.v[start_idx]);
            Dsum = double(gh_at(start_idx)) * Ssum;
        }
        uint32_t bk = kKeyInf;
        int by = 0;
        for (int y = lane; y < H; y += 32) {
            const uint32_t k = sRmKey[y];
            if (k < bk) { bk = k; by = y; }
        }

        // ---- search loop -----------------------------------------------------------------------
        int t_solve = NASTAR_TS_CAPPED;
        int steps = 0;
        int32_t* trace = kTrace ? (p.trace + int64_t(b) * T) : nullptr;
        for (int t = 0; t < T; ++t) {
            const uint32_t m = __reduce_min_sync(kFull, bk);
            if (m == kKeyInf) { t_solve = NASTAR_TS_EXHAUSTED; break; }
            double A1 = 0.0, B1 = 0.0;   // prefix sums INCLUDING step t (events of step t take effect from t+1 on)
            if (kBwd) {
                const double inv = 1.0 / (Ssum + Slo);
                const double a_t = inv, b_t = (Dsum + Dlo) * inv * inv;
                const bool last = stationary_ok && (ts_in >= 0) && (t == ts_in + 1);
                if (last) {
                    // the map is solved and re-selects its goal with a frozen open set until step T_batch-1
                    // (SURVEY App. A.4): the remaining Tb - t steps advance the prefix sums linearly
                    Acum += double(Tb - t) * a_t;
                    Bcum += double(Tb - t) * b_t;
                    break;
                }
                A1 = Acum + a_t;
                B1 = Bcum + b_t;
            }
            const int r = int(__reduce_min_sync(kFull, (bk == m) ? uint32_t(by) : 0x7FFFFFFFu));
            const int c = sRmCol[r];
            const int ind = r * W + c;
            steps = t + 1;
            if (kTrace && lane == 0) trace[t] = ind;
            const bool solved = (ind == goal_idx);
            if (lane == 0) {
                sClosed[r * Wd + (c >> 5)] |= 1u << (c & 31);
                if (!solved) sOpen[r * Wd + (c >> 5)] &= ~(1u << (c & 31));
            }
            __syncwarp();
            // rescan of row r over its remaining, pre-expansion open cells (ascending x => first min)
            uint32_t rs_key = kKeyInf;
            int rs_col = 0;
            for (int x = lane; x < W; x += 32) {
                if ((sOpen[r * Wd + (x >> 5)] >> (x & 31)) & 1u) {
                    const uint32_t k = fkey(F[ind - c + x]);
                    if (k < rs_key) { rs_key = k; rs_col = x; }
                }
            }
            // neighbour cell of this lane (lanes 0..8, centre excluded)
            const int k9 = lane;
            const int dr = k9 / 3 - 1, dc = k9 - (k9 / 3) * 3 - 1;
            const int y = r + dr, x = c + dc;
            const bool valid = (lane < 9) && (lane != 4) && (unsigned(y) < unsigned(H)) && (unsigned(x) < unsigned(W));
            const int n = y * W + x;
            bool passable = false, isopen = false, isclosed = false;
            float gn = 0.f;
            if (valid) {
                const int wi = y * Wd + (x >> 5);
                const uint32_t bit = 1u << (x & 31);
                passable = sPass[wi] & bit;
                isopen = sOpen[wi] & bit;
                isclosed = sClosed[wi] & bit;
                if (passable && isopen) gn = G[n];
            }
            const float g2 = __fadd_rn(G[ind], cost_at(ind));
            __syncwarp();  // every read of the pre-expansion open bits is done
            const bool upd = valid && passable && (isopen ? (gn > g2) : !isclosed);
            uint32_t key = kKeyInf;
            double dS = 0.0, dD = 0.0;   // backward: this lane's change of S and D
            if (upd) {
                const float hn = __fadd_rn(heuristic(y, x, gy, gx), cost_at(n));
                const float fn = f_value(gr, omg, g2, hn);
                G[n] = g2;
                F[n] = fn;
                Par[n] = uint8_t(k9);
                atomicOr(&sOpen[y * Wd + (x >> 5)], 1u << (x & 31));
                key = fkey(fn);
                if (kBwd) {
                    const float v_new = expf(__fdiv_rn(-fn, a.sqrt_w));
                    const double gh = double(gh_at(n));
                    dS = iv.event(n, gh, v_new, A1, B1);
                    dD = gh * dS;
                }
            }
            if (kBwd) {
                if (lane == 9 && !solved) {
                    // event: the selected cell leaves the open set (the goal stays open, :224)
                    const double gh = double(gh_at(ind));
                    dS = iv.leave(ind, gh, A1, B1);
                    dD = gh * dS;
                }
#pragma unroll
                for (int o = 8; o; o >>= 1) {          // events sit on lanes 0..9
                    dS += __shfl_xor_sync(kFull, dS, o);
                    dD += __shfl_xor_sync(kFull, dD, o);
                }
                dS = __shfl_sync(kFull, dS, 0);
                dD = __shfl_sync(kFull, dD, 0);
                dd_add(Ssum, Slo, dS);
                dd_add(Dsum, Dlo, dD);
                Acum = A1;
                Bcum = B1;
            }
            if (solved && t_solve < 0) t_solve = t;
            if (!kContinue && solved) break;
            // per-row minimum of the freshly written keys: lanes {0,1,2} {3,4,5} {6,7,8}
            const uint32_t k1 = __shfl_down_sync(kFull, key, 1), k2 = __shfl_down_sync(kFull, key, 2);
            const int x1 = __shfl_down_sync(kFull, x, 1), x2 = __shfl_down_sync(kFull, x, 2);
            uint32_t best = key;
            int bx = x;
            if (k1 < best) { best = k1; bx = x1; }
            if (k2 < best) { best = k2; bx = x2; }
            const uint32_t mr = __reduce_min_sync(kFull, rs_key);
            const int mc = int(__reduce_min_sync(kFull, (rs_key == mr) ? uint32_t(rs_col) : 0x7FFFFFFFu));
            if (lane == 0 || lane == 3 || lane == 6) {
                const int yy = r + lane / 3 - 1;
                if (unsigned(yy) < unsigned(H)) {
                    uint32_t ck;
                    int cc;
                    if (lane == 3) { ck = mr; cc = mc; } else { ck = sRmKey[yy]; cc = sRmCol[yy]; }
                    if (best < ck || (best == ck && bx < cc)) { ck = best; cc = bx; }
                    sRmKey[yy] = ck;
                    sRmCol[yy] = cc;
                }
            }
            __syncwarp();
            if (((lane - (r - 1)) & 31) < 3) {  // lanes owning rows r-1, r, r+1 re-fold their rows
                bk = kKeyInf;
                by = 0;
                for (int yy = lane; yy < H; yy += 32) {
                    const uint32_t k = sRmKey[yy];
                    if (k < bk) { bk = k; by = yy; }
                }
            }
        }
        __syncwarp();

        if (kBwd) {
            // close the intervals of the cells still open at the end, then scale
            const float coef = -omg / a.sqrt_w;
            float* gOut = a.grad_cost + int64_t(b) * N;
            for (int i = lane; i < N; i += 32) gOut[i] = float(double(coef) * iv.close(i, Acum, Bcum, [&] { return double(gh_at(i)); }));
            __syncwarp();
        }
        if (!kBwd) {
        // ---- backtrack (differentiable_astar.py:96-125): follow direction codes ---------------
        for (int i = lane; i < L.nbits; i += 32) sPath[i] = 0u;   // sPath aliases sPass
        __syncwarp();
        if (lane == 0) {
            sPath[gy * Wd + (gx >> 5)] |= 1u << (gx & 31);
            const bool goal_has_parent = (sOpen[gy * Wd + (gx >> 5)] >> (gx & 31)) & 1u;
            if (goal_has_parent && goal_idx != start_idx) {
                int loc = goal_idx;
                const int hops = (t_solve >= 0) ? N : (T - 1);
                for (int k = 0; k < hops; ++k) {
                    const int code = Par[loc];
                    // code = (dr+1)*3 + (dc+1) of this cell relative to its parent
                    loc -= (code / 3 - 1) * W + (code - (code / 3) * 3 - 1);
                    const int yy = loc / W, xx = loc - yy * W;
                    sPath[yy * Wd + (xx >> 5)] |= 1u << (xx & 31);
                    if (loc == start_idx) break;
                }
            }
        }
        __syncwarp();

        // ---- epilogue: coalesced stores --------------------------------------------------------
        float* gHist = p.histories + int64_t(b) * N;
        long long* gPath = reinterpret_cast<long long*>(p.paths) + int64_t(b) * N;
        if (((W & 31) == 0) && aligned16(gHist) && aligned16(gPath)) {
            // flat bit index == row-word index: each lane expands 4 cells per segment into one 128-bit
            // histories store and two 128-bit paths stores (fully coalesced)
            const int nseg = (N + 127) >> 7;
            const int nq = N >> 2;
            const int sh = (lane & 7) << 2;
            for (int seg = 0; seg < nseg; ++seg) {
                const int wi = (seg << 2) + (lane >> 3);
                const int q = (seg << 5) + lane;
                if (q >= nq) continue;            // partial last segment
                const uint32_t cb = sClosed[wi] >> sh, pb = sPath[wi] >> sh;
                reinterpret_cast<float4*>(gHist)[q] = make_float4((cb & 1u) ? 1.f : 0.f, (cb & 2u) ? 1.f : 0.f,
                                                                  (cb & 4u) ? 1.f : 0.f, (cb & 8u) ? 1.f : 0.f);
                reinterpret_cast<longlong2*>(gPath)[2 * q] = make_longlong2((pb & 1u) ? 1ll : 0ll, (pb & 2u) ? 1ll : 0ll);
                reinterpret_cast<longlong2*>(gPath)[2 * q + 1] = make_longlong2((pb & 4u) ? 1ll : 0ll, (pb & 8u) ? 1ll : 0ll);
            }
        } else {
            for (int y = 0; y < H; ++y) {
                for (int x = lane; x < W; x += 32) {
                    const int wi = y * Wd + (x >> 5);
                    gHist[y * W + x] = ((sClosed[wi] >> (x & 31)) & 1u) ? 1.f : 0.f;
                    gPath[y * W + x] = ((sPath[wi] >> (x & 31)) & 1u) ? 1ll : 0ll;
                }
            }
        }
        int n_closed = 0, n_path = 0;
        if (p.n_closed || p.path_len) {
            for (int i = lane; i < L.nbits; i += 32) { n_closed += __popc(sClosed[i]); n_path += __popc(sPath[i]); }
            n_closed = __reduce_add_sync(kFull, n_closed);
            n_path = __reduce_add_sync(kFull, n_path);
        }
        if (lane == 0) {
            if (p.t_solve) p.t_solve[b] = t_solve;
            if (p.n_steps) p.n_steps[b] = steps;
            if (p.n_closed) p.n_closed[b] = n_closed;
            if (p.path_len) p.path_len[b] = n_path;
        }
        }  // !kBwd
        __syncwarp();
    }
}

}  // namespace nastar
