// nastar_warp.cuh — warp-resident engines: astar_warp32_kernel (H, W <= 32) and astar_warp64_kernel (H, W <= 64,
// not both <= 32), forward and backward.
//
// Replaces the T-step loop + backtrack of DifferentiableAstar.forward
// (/root/reference/src/neural_astar/planner/differentiable_astar.py:187-255) and the autograd
// through it, one map per warp.  Design (DESIGN.md "warp32 engine"):
//   * the map lives in shared memory in a PADDED kW x kW layout (cell id rc = y*kW + x, kW = 32 or 64), so every
//     index is a shift/mask and every plane sits at a compile-time offset;
//   * lane l owns grid rows l (and l+32 when kW = 64): passable / open / closed rows are kW-bit masks in registers,
//     and the lane caches each row's best open cell (order-preserving f key, column);
//   * node selection (:206-209; softmax+argmax == arg-min of (f, flat index), SURVEY App. A.2)
//     is two REDUX.MINs over the cached row minima: min key, then min (row*kW + col) among ties;
//   * expansion (:228-249) touches <= 8 cells in rows r-1..r+1: the lanes owning those rows relax their
//     <= 3 cells with branch-free mask algebra and fold the new keys into their cached minimum —
//     insertions/decreases never need a rescan;
//   * only row r lost its minimum (the selected cell): all 32 lanes rescan that one row (one
//     conflict-free LDS per 32 columns + two REDUX.MINs);
//   * planes are staged with 1-D TMA bulk copies (cp.async.bulk + mbarrier) when W == kW and
//     results leave as coalesced 128-bit stores; the loop itself never touches HBM.
//   kBwd = true replays the same state machine and accumulates the closed-form gradient of the
//   straight-through softmax (SURVEY App. B) — same code path, so the replay cannot drift; the
//   accumulation is event-based (IntervalPlanes, nastar_common.cuh: O(1) per step).
// The shared-memory layouts, the heuristic table and the backward's interval algebra are shared; each kernel keeps its
// own prologue, step loop and epilogue, because ptxas schedules the tuned step loops differently as soon as the code
// around them changes (shared kW templates for the staging / h pass / epilogue cost 1-13 instructions per step).
#pragma once
#include <type_traits>

#include "../../include/nastar_b200.h"
#include "nastar_common.cuh"

namespace nastar {

// heuristic(|dy|, |dx|) for every offset on a 64x64 grid (the 32-wide engine uses its top-left corner), filled once
// per device by heur_init_kernel with the very same device function the generic engine evaluates inline — the
// per-map h pass becomes one cached load + one add per cell instead of an IEEE sqrt chain.
constexpr int kHeurCells = 64 * 64;
__device__ float g_heur[kHeurCells];

__global__ void heur_init_kernel() {
    const int i = threadIdx.x + blockIdx.x * blockDim.x;
    if (i < kHeurCells) g_heur[i] = heuristic(i >> 6, i & 63, 0, 0);
}

// one row of the padded map as a bit mask
template <int kW>
using RowMask = std::conditional_t<kW == 32, uint32_t, unsigned long long>;

template <int kW>
struct __align__(16) WarpSmem {
    static constexpr int kCells = kW * kW;
    float cost[kCells];        // staged cost plane (padded)
    uint32_t key[kCells];      // order-preserving key of f = g_ratio*g + (1-g_ratio)*h, opened cells only
    float2 ghbuf[kCells + 4];  // {g, h} per cell at ghbuf[2 + rc]; 2 guard cells on either side make the
                               // c-1 / c+1 window loads of the first/last cell addressable (16-B aligned body)
    int8_t par[kCells];        // parent link of opened cells as a signed offset: parent = rc - par[rc], in [-kW-1, kW+1]
    RowMask<kW> open_row[kW];  // every lane's open rows, refreshed each step (rescan input)
    RowMask<kW> bits_a[kW];    // closed rows for the epilogue
    RowMask<kW> bits_b[kW];    // path rows for the epilogue
    unsigned long long bar;    // mbarrier for the TMA prologue
};

// backward-only planes (dynamic shared memory): the event-based closed form's per-cell state
template <int kW>
struct __align__(16) WarpBwd {
    static constexpr int kCells = kW * kW;
    double acc[kCells];
    double a0[kCells];
    double b0[kCells];
    float v[kCells];
    float gh[kCells];     // upstream gradient (goal zeroed when the clamp blocks it)
    __device__ __forceinline__ IntervalPlanes planes() { return IntervalPlanes{acc, a0, b0, v}; }
};

// the warp32 forward's 17.4 KB is what lets a search CTA sit beside the encoder's last conv CTA in the pipelined
// step (DESIGN.md §5); the warp64 backward must stay under the 227 KB per-CTA limit
static_assert(sizeof(WarpSmem<32>) == 17840 && sizeof(WarpBwd<32>) == 32768, "warp32 shared-memory footprint");
static_assert(sizeof(WarpSmem<64>) == 71216 && sizeof(WarpBwd<64>) == 131072, "warp64 shared-memory footprint");

// kNoExit (forward only): NASTAR_FWD_NO_EARLY_EXIT — keep stepping after the solve step, exactly T steps.
// kFused (forward only): the prologue may have to finish the encoder (NASTAR_COST_LOGIT / NASTAR_COST_TAPS); kept out
// of the plain instantiation so that its cold instruction footprint stays small.
template <bool kTrace, bool kBwd, bool kNoExit = false, bool kFused = false>
__global__ void __launch_bounds__(32, 12) astar_warp32_kernel(const SearchArgs a) {
    constexpr bool kContinue = kBwd || kNoExit;   // the loop does not stop at the solve step
    __shared__ WarpSmem<32> S;
    extern __shared__ __align__(16) unsigned char bwd_raw[];  // backward only: WarpBwd<32>
    WarpBwd<32>& Bw = *reinterpret_cast<WarpBwd<32>*>(bwd_raw);
    const nastar_fwd_params& p = a.f;
    float2* const sGH = S.ghbuf + 2;
    const int lane = threadIdx.x;
    const int b = blockIdx.x;                    // output slot
    const int H = p.H, W = p.W, N = H * W;
    // NASTAR_FWD_PAIR: CTAs B..2B-1 search the same problems with cost = obstacles (VanillaAstar, astar.py:93-94)
    const bool vanilla_half = !kBwd && (p.flags & NASTAR_FWD_PAIR) && (b >= p.B);
    const int bi = vanilla_half ? (b - p.B) : b;  // input map

    const float* gStart = p.start + int64_t(bi) * p.start_stride;
    const float* gGoal = p.goal + int64_t(bi) * p.goal_stride;
    const float* gObst = p.obst + int64_t(bi) * p.obst_stride;
    const float* gCost = vanilla_half ? gObst : (p.cost + int64_t(bi) * p.cost_stride);
    const int cost_kind = (!kFused || kBwd || vanilla_half) ? NASTAR_COST_PLANE : p.cost_kind;
    const bool cost_plane = (cost_kind == NASTAR_COST_PLANE);
    const bool obst_is_cost = cost_plane && (gObst == gCost);

    // ---------------- prologue: stage planes, build row masks ------------------------------
    uint32_t pass = 0u;
    int start_rc = -1, goal_rc = -1;
    const bool tma = (W == 32) && (!cost_plane || aligned16(gCost)) && aligned16(gStart) && aligned16(gGoal) && aligned16(gObst);
    if (tma) {
        // flat layout == padded layout: bulk-copy whole planes (start/goal/obstacles are parked in the
        // f and {g,h} planes, which are not live yet)
        float* tStart = reinterpret_cast<float*>(S.key);
        float* tGoal = reinterpret_cast<float*>(sGH);
        float* tObst = tGoal + WarpSmem<32>::kCells;
        uint64_t* bar = reinterpret_cast<uint64_t*>(&S.bar);
        if (lane == 0) {
            mbar_init(bar, 1);
            fence_mbar_init();
            const uint32_t bytes = uint32_t(N) * 4u;
            mbar_expect_tx(bar, bytes * ((obst_is_cost ? 3u : 4u) - (cost_plane ? 0u : 1u)));
            if (cost_plane) tma_load_1d(S.cost, gCost, bytes, bar);
            tma_load_1d(tStart, gStart, bytes, bar);
            tma_load_1d(tGoal, gGoal, bytes, bar);
            if (!obst_is_cost) tma_load_1d(tObst, gObst, bytes, bar);
        }
        __syncwarp();
        if (kFused && !cost_plane) {
            // fused encoder hand-off (SURVEY 8(f)-3): the cost plane is produced here from the encoder's raw
            // output while the TMA copies of the other planes are in flight
#pragma unroll 4      // four rows of gathers in flight: the prologue is a chain of L2 round trips for one warp
            for (int y = 0; y < H; ++y)
                S.cost[(y << 5) + lane] = cost_value(cost_kind, gCost, y, lane, H, W, p.cost_bias, p.cost_scale);
        }
        mbar_wait(bar, 0);
        const float* sObst = obst_is_cost ? S.cost : tObst;
#pragma unroll 4
        for (int y = 0; y < H; ++y) {
            const int i = (y << 5) + lane;
            const uint32_t wo = __ballot_sync(kFull, sObst[i] != 0.f);
            const uint32_t ws = __ballot_sync(kFull, tStart[i] != 0.f);
            const uint32_t wg = __ballot_sync(kFull, tGoal[i] != 0.f);
            if (lane == y) pass = wo;
            if (start_rc < 0 && ws) start_rc = (y << 5) + __ffs(ws) - 1;
            if (goal_rc < 0 && wg) goal_rc = (y << 5) + __ffs(wg) - 1;
        }
    } else {
        // W < 32 (or unaligned planes): rows are shorter than a warp; issue 8 rows of loads per plane
        // before consuming them so that DRAM latency is paid H/8 times, not H times
        const bool in = lane < W;
        constexpr int kRows = 8;
        for (int y0 = 0; y0 < H; y0 += kRows) {
            float vc[kRows], vo[kRows], vs[kRows], vg[kRows];
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                const bool ok = in && (y0 + u < H);
                const int i = (y0 + u) * W + lane;
                vc[u] = ok ? (kFused ? cost_value(cost_kind, gCost, y0 + u, lane, H, W, p.cost_bias, p.cost_scale)
                                     : __ldg(gCost + i)) : 0.f;
                vo[u] = obst_is_cost ? vc[u] : (ok ? __ldg(gObst + i) : 0.f);
                vs[u] = ok ? __ldg(gStart + i) : 0.f;
                vg[u] = ok ? __ldg(gGoal + i) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                const int y = y0 + u;
                if (y < H) {
                    S.cost[(y << 5) + lane] = vc[u];
                    const uint32_t wo = __ballot_sync(kFull, vo[u] != 0.f);
                    const uint32_t ws = __ballot_sync(kFull, vs[u] != 0.f);
                    const uint32_t wg = __ballot_sync(kFull, vg[u] != 0.f);
                    if (lane == y) pass = wo;
                    if (start_rc < 0 && ws) start_rc = (y << 5) + __ffs(ws) - 1;
                    if (goal_rc < 0 && wg) goal_rc = (y << 5) + __ffs(wg) - 1;
                }
            }
        }
    }
    if (goal_rc < 0) goal_rc = 0;  // argmax of an all-zero plane (differentiable_astar.py:197)
    const int gy = goal_rc >> 5, gx = goal_rc & 31;
    __syncwarp();
    // h = heuristic + cost (:191-192), one row per iteration; overwrites the parked planes
    {
        const int adx = (lane > gx) ? (lane - gx) : (gx - lane);
#pragma unroll 8
        for (int y = 0; y < H; ++y) {
            const int i = (y << 5) + lane;
            const int ady = (y > gy) ? (y - gy) : (gy - y);
            sGH[i] = make_float2(0.f, __fadd_rn(__ldg(&g_heur[(ady << 6) | adx]), S.cost[i]));
        }
    }
    __syncwarp();

    const float gr = p.g_ratio, omg = p.one_minus_g_ratio;
    uint32_t open = 0u, closed = 0u;
    uint32_t rm_key = kKeyInf;
    int rm_col = 0;

    // backward: running sums replicated in every lane (S = sum of v over the open set, D = <Gh, v>, A / B = prefix
    // sums of 1/S and D/S^2 over the executed steps)
    double Ssum = 0.0, Slo = 0.0, Dsum = 0.0, Dlo = 0.0, Acum = 0.0, Bcum = 0.0;   // (Ssum,Slo), (Dsum,Dlo): double-double
    int Tb = 0, ts_in = NASTAR_TS_CAPPED;
    if (kBwd) {
        Tb = *a.T_batch;
        ts_in = a.t_solve_in[b];
        const float* gG = a.grad_hist + int64_t(b) * a.grad_stride;
        // clamp(hist + sel) blocks the gradient at a goal that is re-selected after its solve step
        // (pre-clamp value 2, differentiable_astar.py:222-223; SURVEY App. B)
        const bool blocked = (ts_in >= 0) && (ts_in < Tb - 1);
        for (int y = 0; y < 32; ++y) {
            const int i = (y << 5) + lane;
            Bw.acc[i] = 0.0;
            Bw.v[i] = 0.f;
            Bw.gh[i] = (y < H && lane < W && !(blocked && i == goal_rc)) ? __ldg(gG + y * W + lane) : 0.f;
        }
        __syncwarp();
    }
    if (lane == 0) S.par[goal_rc] = 0;  // parents are initialised to the goal (:195-198): a self link at the goal
    if (start_rc >= 0) {
        const float f0 = f_value(gr, omg, 0.f, sGH[start_rc].y);
        if (lane == 0) {
            S.key[start_rc] = fkey(f0);              // g = 0 already (:193)
            if (kBwd) { Bw.v[start_rc] = expf(__fdiv_rn(-f0, a.sqrt_w)); Bw.a0[start_rc] = 0.0; Bw.b0[start_rc] = 0.0; }  // :207
        }
        if (lane == (start_rc >> 5)) {
            open = 1u << (start_rc & 31);            // open_maps = start_maps (:187)
            rm_key = fkey(f0);
            rm_col = start_rc & 31;
        }
    }
    S.open_row[lane] = open;
    __syncwarp();
    if (kBwd && start_rc >= 0) {
        Ssum = double(Bw.v[start_rc]);
        Dsum = double(Bw.gh[start_rc]) * Ssum;
    }

    // ---------------- the search loop (differentiable_astar.py:203-252) --------------------
    const int T = kBwd ? Tb : p.T;
    // post-solve steps are stationary when g_ratio >= 0.5 (the goal keeps being re-selected and
    // nothing changes, SURVEY App. A.4): the backward then adds them in one go
    const bool stationary_ok = (gr >= 0.5f);
    int t_solve = NASTAR_TS_CAPPED;
    int32_t* trace = kTrace ? (p.trace + int64_t(b) * p.T) : nullptr;
    const float2* ghrow = sGH + (lane << 5);      // this lane's row of {g,h}
    int t = 0;
    for (; t < T; ++t) {
        // -- select: lexicographic arg-min of (f key, row, col) with two REDUX.MINs -----------
        const uint32_t m = __reduce_min_sync(kFull, rm_key);
        if (m == kKeyInf) { t_solve = NASTAR_TS_EXHAUSTED; break; }
        double A1 = 0.0, B1 = 0.0;   // prefix sums INCLUDING step t (the events of step t act from t+1 on)
        if (kBwd) {
            const double inv = 1.0 / (Ssum + Slo);
            const double a_t = inv, b_t = (Dsum + Dlo) * inv * inv;
            if (stationary_ok && (ts_in >= 0) && (t == ts_in + 1)) {
                // solved: the goal is re-selected with a frozen open set until step T_batch-1 (App. A.4)
                Acum += double(Tb - t) * a_t;
                Bcum += double(Tb - t) * b_t;
                break;
            }
            A1 = Acum + a_t;
            B1 = Bcum + b_t;
        }
        const uint32_t ind = __reduce_min_sync(kFull, (rm_key == m) ? uint32_t((lane << 5) | rm_col) : 0xFFFFFFFFu);
        const int r = int(ind >> 5), c = int(ind & 31u);
        if (kTrace && lane == 0) trace[t] = r * W + c;
        const bool solved = (int(ind) == goal_rc);          // :219-220
        const uint32_t m1 = 1u << c;                        // column masks of the 3-wide window;
        const uint32_t m0 = m1 >> 1, m2 = m1 << 1;          // they fall off the row at c == 0 / 31
        // -- rescan inputs for row r (pre-expansion open cells minus the selected one); stale f
        //    values of cells relaxed this step are upper bounds and the fresh keys are merged below
        const uint32_t open_r = (kContinue && solved) ? S.open_row[r] : (S.open_row[r] & ~m1);
        const uint32_t krs = S.key[(r << 5) + lane];
        const uint32_t rs_key = ((open_r >> lane) & 1u) ? krs : kKeyInf;
        // the rescan's two reductions are issued here, ahead of the expansion's ALU chain, so that their latency
        // overlaps it instead of extending the tail of the step (their inputs are pre-step values only)
        const uint32_t mr = __reduce_min_sync(kFull, rs_key);
        const uint32_t mc = __reduce_min_sync(kFull, (rs_key == mr) ? uint32_t(lane) : 0xFFFFFFFFu);
        // -- expansion inputs ----------------------------------------------------------------
        const int dr = lane - r;
        const bool isr = (dr == 0);
        const bool near = (unsigned(dr + 1) <= 2u);
        // only the three row lanes load (rows are 256 B apart = same banks; 32 lanes would serialise)
        float2 n0 = make_float2(0.f, 0.f), n1 = n0, n2 = n0;
        if (near) { n0 = ghrow[c - 1]; n1 = ghrow[c]; n2 = ghrow[c + 1]; }   // guard cells make c-1/c+1 safe
        const float g2 = __fadd_rn(sGH[ind].x, S.cost[ind]);               // :234, cost of the SELECTED node
        __syncwarp();   // every shared-memory read of this step precedes every write below (no intra-warp WAR)
        // -- closed/open update of the selected cell (:222-225) ------------------------------
        if (isr) {
            closed |= m1;
            if (!solved) open &= ~m1;                       // the goal stays open once selected
            rm_key = kKeyInf;                               // this row's minimum is rebuilt below
        }
        // -- expansion (:228-249) as mask algebra on this lane's row ---------------------------
        //    idx = ((1-open)(1-hist) + open*(g > g2)) * neighbours * obstacles   (:235-236)
        const uint32_t win = isr ? (m0 | m2) : (m0 | m1 | m2);
        const uint32_t cand = near ? (win & pass) : 0u;
        const uint32_t gt = ((n0.x > g2) ? m0 : 0u) | ((n1.x > g2) ? m1 : 0u) | ((n2.x > g2) ? m2 : 0u);
        const uint32_t upd = cand & ((open & gt) | ~(open | closed));
        open |= upd;                                        // :242
        const float ag = __fmul_rn(gr, g2);
        const float f0n = __fadd_rn(ag, __fmul_rn(omg, n0.y));
        const float f1n = __fadd_rn(ag, __fmul_rn(omg, n1.y));
        const float f2n = __fadd_rn(ag, __fmul_rn(omg, n2.y));
        const bool u0 = (upd & m0) != 0u, u1 = (upd & m1) != 0u, u2 = (upd & m2) != 0u;
        const int cell = (lane << 5) + c;
        const uint32_t q0 = fkey(f0n), q1 = fkey(f1n), q2 = fkey(f2n);
        const int off = (dr << 5) - 1;                      // (this row, column c-1) minus the selected cell
        if (u0) { sGH[cell - 1].x = g2; S.key[cell - 1] = q0; S.par[cell - 1] = int8_t(off); }       // :238, :246-249
        if (u1) { sGH[cell].x = g2;     S.key[cell] = q1;     S.par[cell] = int8_t(off + 1); }
        if (u2) { sGH[cell + 1].x = g2; S.key[cell + 1] = q2; S.par[cell + 1] = int8_t(off + 2); }
        if (kBwd) {
            double dS = 0.0, dD = 0.0;   // this lane's change of S and D
            auto event = [&](int cl, float v_new) {
                const double gh = double(Bw.gh[cl]);
                const double dv = Bw.planes().event(cl, gh, v_new, A1, B1);
                dS += dv;
                dD += gh * dv;
            };
            if (u0) event(cell - 1, expf(__fdiv_rn(-f0n, a.sqrt_w)));   // :207
            if (u1) event(cell, expf(__fdiv_rn(-f1n, a.sqrt_w)));
            if (u2) event(cell + 1, expf(__fdiv_rn(-f2n, a.sqrt_w)));
            if (isr && !solved) event(int(ind), 0.f);                    // the selected cell leaves the open set
            // the events sit on the lanes of rows r-1, r, r+1
            const double s0 = __shfl_sync(kFull, dS, max(r - 1, 0)), s1 = __shfl_sync(kFull, dS, r),
                         s2 = __shfl_sync(kFull, dS, min(r + 1, 31));
            const double d0 = __shfl_sync(kFull, dD, max(r - 1, 0)), d1 = __shfl_sync(kFull, dD, r),
                         d2 = __shfl_sync(kFull, dD, min(r + 1, 31));
            dd_add(Ssum, Slo, (r > 0 ? s0 : 0.0) + s1 + (r < 31 ? s2 : 0.0));
            dd_add(Dsum, Dlo, (r > 0 ? d0 : 0.0) + d1 + (r < 31 ? d2 : 0.0));
            Acum = A1;
            Bcum = B1;
        }
        // fold the fresh keys (ascending column, strict < keeps the lowest column on ties)
        const uint32_t k0 = u0 ? q0 : kKeyInf, k1 = u1 ? q1 : kKeyInf, k2 = u2 ? q2 : kKeyInf;
        uint32_t bk = k0;
        int bc = c - 1;
        if (k1 < bk) { bk = k1; bc = c; }
        if (k2 < bk) { bk = k2; bc = c + 1; }
        if ((bk < rm_key) | ((bk == rm_key) & (bc < rm_col))) { rm_key = bk; rm_col = bc; }
        if (solved && t_solve < 0) t_solve = t;             // first step at which the goal was selected
        if (!kContinue && solved) break;                    // :251-252 (per-map early exit, App. A.4)
        if (near) S.open_row[lane] = open;
        // -- fold the rescan into lane r's cached minimum -------------------------------------
        const bool take = isr & ((mr < rm_key) | ((mr == rm_key) & (int(mc) < rm_col)));
        rm_key = take ? mr : rm_key;
        rm_col = take ? int(mc) : rm_col;
        __syncwarp();
    }
    __syncwarp();
    // selection steps executed: t on exhaustion / cap, t+1 when the loop left through the solve step
    const int steps = (!kContinue && t_solve >= 0) ? (t + 1) : t;

    if (kBwd) {
        // close the intervals of the cells still open; dL/dcost = -(1-g_ratio)/sqrt(W) * acc
        // (h = heuristic + cost, f = g_ratio*g + (1-g_ratio)*h)
        const double coef = -double(omg) / double(a.sqrt_w);
        float* gOut = a.grad_cost + int64_t(b) * N;
        for (int y = 0; y < H; ++y) {
            const int i = (y << 5) + lane;
            if (lane < W) {
                const double acc = Bw.planes().close(i, Acum, Bcum, [&] { return double(Bw.gh[i]); });
                gOut[y * W + lane] = float(coef * acc);
            }
        }
        return;
    }

    // ---------------- backtrack (differentiable_astar.py:96-125, App. A.3) ------------------
    uint32_t path = 0u;
    {
        if (lane == gy) path |= 1u << gx;
        // the start's parent is the goal in the reference (the initial value); the walk stops at the start
        // before following it, which marks the same cells (App. A.3)
        int loc = goal_rc - S.par[goal_rc];
        const int hops = (t_solve >= 0) ? N : (p.T - 1);
        for (int k = 0; k < hops; ++k) {
            if (lane == (loc >> 5)) path |= 1u << (loc & 31);
            if (loc == start_rc || loc == goal_rc) break;   // reached the start (or the goal's self link)
            loc -= S.par[loc];
        }
    }

    // ---------------- epilogue: coalesced stores of histories / paths -----------------------
    S.bits_a[lane] = closed;
    S.bits_b[lane] = path;
    __syncwarp();
    float* gHist = p.histories + int64_t(b) * N;
    long long* gPath = reinterpret_cast<long long*>(p.paths) + int64_t(b) * N;
    if (W == 32 && aligned16(gHist) && aligned16(gPath)) {
        const int x = (lane & 7) << 2;
#pragma unroll 4
        for (int j = 0; j < 8; ++j) {
            const int y = (lane >> 3) + 4 * j;
            if (y < H) {
                const int i4 = lane + 32 * j;
                const uint32_t cb = S.bits_a[y] >> x, pb = S.bits_b[y] >> x;
                reinterpret_cast<float4*>(gHist)[i4] = make_float4((cb & 1u) ? 1.f : 0.f, (cb & 2u) ? 1.f : 0.f,
                                                                   (cb & 4u) ? 1.f : 0.f, (cb & 8u) ? 1.f : 0.f);
                reinterpret_cast<longlong2*>(gPath)[2 * i4] = make_longlong2((pb & 1u) ? 1ll : 0ll, (pb & 2u) ? 1ll : 0ll);
                reinterpret_cast<longlong2*>(gPath)[2 * i4 + 1] = make_longlong2((pb & 4u) ? 1ll : 0ll, (pb & 8u) ? 1ll : 0ll);
            }
        }
    } else {
        for (int y = 0; y < H; ++y) {
            if (lane < W) {
                gHist[y * W + lane] = ((S.bits_a[y] >> lane) & 1u) ? 1.f : 0.f;
                gPath[y * W + lane] = ((S.bits_b[y] >> lane) & 1u) ? 1ll : 0ll;
            }
        }
    }
    // per-map counts for the validation metrics (utils/training.py:71-85): histories.sum(), paths.sum()
    const int n_closed = __reduce_add_sync(kFull, __popc(closed));
    const int n_path = __reduce_add_sync(kFull, __popc(path));
    if (lane == 0) {
        if (p.t_solve) p.t_solve[b] = t_solve;
        if (p.n_steps) p.n_steps[b] = steps;
        if (p.n_closed) p.n_closed[b] = n_closed;
        if (p.path_len) p.path_len[b] = n_path;
    }
}

// 64-wide engine: lane l owns rows l and l+32 (two 64-bit passable/open/closed masks and two cached row minima), so
// selection first takes the local min of the lane's two rows; of a lane's two rows at most one is within r-1..r+1, so the
// row lanes pick that slot with selects and run the same branch-free 3-cell mask algebra on 64-bit masks; the rescan of
// row r checks columns l and l+32.  ~70 KB of shared memory per map (198 KB with the backward), 3 maps per SM.
// kFused (forward only): as in the 32-wide engine; kept out of the plain instantiations.
template <bool kTrace, bool kBwd, bool kNoExit = false, bool kFused = false>
__global__ void __launch_bounds__(32) astar_warp64_kernel(const SearchArgs a) {
    constexpr bool kContinue = kBwd || kNoExit;
    const nastar_fwd_params& p = a.f;
    extern __shared__ __align__(16) unsigned char smem64_raw[];
    WarpSmem<64>& S = *reinterpret_cast<WarpSmem<64>*>(smem64_raw);
    WarpBwd<64>& Bw = *reinterpret_cast<WarpBwd<64>*>(smem64_raw + sizeof(WarpSmem<64>));
    float2* const sGH = S.ghbuf + 2;
    const int lane = threadIdx.x;
    const int b = blockIdx.x;
    const int H = p.H, W = p.W, N = H * W;
    typedef unsigned long long u64;

    const float* gCost = p.cost + int64_t(b) * p.cost_stride;
    const float* gStart = p.start + int64_t(b) * p.start_stride;
    const float* gGoal = p.goal + int64_t(b) * p.goal_stride;
    const float* gObst = p.obst + int64_t(b) * p.obst_stride;
    const int cost_kind = (kFused && !kBwd) ? p.cost_kind : NASTAR_COST_PLANE;
    const bool cost_plane = (cost_kind == NASTAR_COST_PLANE);
    const bool obst_is_cost = cost_plane && (gObst == gCost);

    // ---------------- prologue ----------------------------------------------------------------
    u64 pass[2] = {0ull, 0ull};
    int start_rc = -1, goal_rc = -1;
    const bool tma = (W == 64) && (!cost_plane || aligned16(gCost)) && aligned16(gStart) && aligned16(gGoal) && aligned16(gObst);
    if (tma) {
        float* tStart = reinterpret_cast<float*>(S.key);
        float* tGoal = reinterpret_cast<float*>(sGH);
        float* tObst = tGoal + WarpSmem<64>::kCells;
        uint64_t* bar = reinterpret_cast<uint64_t*>(&S.bar);
        if (lane == 0) {
            mbar_init(bar, 1);
            fence_mbar_init();
            const uint32_t bytes = uint32_t(N) * 4u;
            mbar_expect_tx(bar, bytes * ((obst_is_cost ? 3u : 4u) - (cost_plane ? 0u : 1u)));
            if (cost_plane) tma_load_1d(S.cost, gCost, bytes, bar);
            tma_load_1d(tStart, gStart, bytes, bar);
            tma_load_1d(tGoal, gGoal, bytes, bar);
            if (!obst_is_cost) tma_load_1d(tObst, gObst, bytes, bar);
        }
        __syncwarp();
        if (kFused && !cost_plane) {
            // fused encoder hand-off: the cost plane is produced here from the encoder's raw output while the TMA copies
            // of the other planes are in flight
#pragma unroll 2
            for (int y = 0; y < H; ++y) {
                S.cost[(y << 6) + lane] = cost_value(cost_kind, gCost, y, lane, H, W, p.cost_bias, p.cost_scale);
                S.cost[(y << 6) + lane + 32] = cost_value(cost_kind, gCost, y, lane + 32, H, W, p.cost_bias, p.cost_scale);
            }
        }
        mbar_wait(bar, 0);
        const float* sObst = obst_is_cost ? S.cost : tObst;
#pragma unroll 2
        for (int y = 0; y < H; ++y) {
            const int i = (y << 6) + lane;
            const uint32_t wo0 = __ballot_sync(kFull, sObst[i] != 0.f), wo1 = __ballot_sync(kFull, sObst[i + 32] != 0.f);
            const uint32_t ws0 = __ballot_sync(kFull, tStart[i] != 0.f), ws1 = __ballot_sync(kFull, tStart[i + 32] != 0.f);
            const uint32_t wg0 = __ballot_sync(kFull, tGoal[i] != 0.f), wg1 = __ballot_sync(kFull, tGoal[i + 32] != 0.f);
            if (lane == (y & 31)) {
                if (y >> 5) pass[1] = u64(wo0) | (u64(wo1) << 32);
                else pass[0] = u64(wo0) | (u64(wo1) << 32);
            }
            if (start_rc < 0 && (ws0 | ws1)) start_rc = (y << 6) + (ws0 ? __ffs(ws0) - 1 : 32 + __ffs(ws1) - 1);
            if (goal_rc < 0 && (wg0 | wg1)) goal_rc = (y << 6) + (wg0 ? __ffs(wg0) - 1 : 32 + __ffs(wg1) - 1);
        }
    } else {
        const bool in0 = lane < W, in1 = lane + 32 < W;
        constexpr int kRows = 4;
        for (int y0 = 0; y0 < H; y0 += kRows) {
            float vc[kRows][2], vo[kRows][2], vs[kRows][2], vg[kRows][2];
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool ok = (hf ? in1 : in0) && (y0 + u < H);
                    const int i = (y0 + u) * W + lane + 32 * hf;
                    vc[u][hf] = ok ? (kFused ? cost_value(cost_kind, gCost, y0 + u, lane + 32 * hf, H, W, p.cost_bias, p.cost_scale)
                                             : __ldg(gCost + i)) : 0.f;
                    vo[u][hf] = obst_is_cost ? vc[u][hf] : (ok ? __ldg(gObst + i) : 0.f);
                    vs[u][hf] = ok ? __ldg(gStart + i) : 0.f;
                    vg[u][hf] = ok ? __ldg(gGoal + i) : 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                const int y = y0 + u;
                if (y < H) {
                    S.cost[(y << 6) + lane] = vc[u][0];
                    S.cost[(y << 6) + lane + 32] = vc[u][1];
                    const uint32_t wo0 = __ballot_sync(kFull, vo[u][0] != 0.f), wo1 = __ballot_sync(kFull, vo[u][1] != 0.f);
                    const uint32_t ws0 = __ballot_sync(kFull, vs[u][0] != 0.f), ws1 = __ballot_sync(kFull, vs[u][1] != 0.f);
                    const uint32_t wg0 = __ballot_sync(kFull, vg[u][0] != 0.f), wg1 = __ballot_sync(kFull, vg[u][1] != 0.f);
                    if (lane == (y & 31)) {
                        if (y >> 5) pass[1] = u64(wo0) | (u64(wo1) << 32);
                        else pass[0] = u64(wo0) | (u64(wo1) << 32);
                    }
                    if (start_rc < 0 && (ws0 | ws1)) start_rc = (y << 6) + (ws0 ? __ffs(ws0) - 1 : 32 + __ffs(ws1) - 1);
                    if (goal_rc < 0 && (wg0 | wg1)) goal_rc = (y << 6) + (wg0 ? __ffs(wg0) - 1 : 32 + __ffs(wg1) - 1);
                }
            }
        }
    }
    if (goal_rc < 0) goal_rc = 0;
    const int gy = goal_rc >> 6, gx = goal_rc & 63;
    __syncwarp();
    {
        const int adx0 = (lane > gx) ? (lane - gx) : (gx - lane);
        const int adx1 = (lane + 32 > gx) ? (lane + 32 - gx) : (gx - lane - 32);
#pragma unroll 4
        for (int y = 0; y < H; ++y) {
            const int i = (y << 6) + lane;
            const int ady = (y > gy) ? (y - gy) : (gy - y);
            sGH[i] = make_float2(0.f, __fadd_rn(__ldg(&g_heur[(ady << 6) | adx0]), S.cost[i]));
            sGH[i + 32] = make_float2(0.f, __fadd_rn(__ldg(&g_heur[(ady << 6) | adx1]), S.cost[i + 32]));
        }
    }
    __syncwarp();

    const float gr = p.g_ratio, omg = p.one_minus_g_ratio;
    u64 open[2] = {0ull, 0ull}, closed[2] = {0ull, 0ull};
    uint32_t rm_key[2] = {kKeyInf, kKeyInf};
    int rm_col[2] = {0, 0};
    if (lane == 0) S.par[goal_rc] = 0;
    if (start_rc >= 0) {
        const float f0 = f_value(gr, omg, 0.f, sGH[start_rc].y);
        const int sy = start_rc >> 6, sx = start_rc & 63;
        if (lane == 0) S.key[start_rc] = fkey(f0);
        if (lane == (sy & 31)) {
            if (sy >> 5) { open[1] = 1ull << sx; rm_key[1] = fkey(f0); rm_col[1] = sx; }
            else         { open[0] = 1ull << sx; rm_key[0] = fkey(f0); rm_col[0] = sx; }
        }
    }
    S.open_row[lane] = open[0];
    S.open_row[lane + 32] = open[1];
    // backward state: running sums replicated in every lane
    double Ssum = 0.0, Slo = 0.0, Dsum = 0.0, Dlo = 0.0, Acum = 0.0, Bcum = 0.0;   // (Ssum,Slo), (Dsum,Dlo): double-double
    int Tb = 0, ts_in = NASTAR_TS_CAPPED;
    if (kBwd) {
        Tb = *a.T_batch;
        ts_in = a.t_solve_in[b];
        // clamp(hist + sel) blocks the gradient at a goal that is re-selected after its solve step
        // (pre-clamp value 2, differentiable_astar.py:222-223; SURVEY App. B)
        const bool blocked = (ts_in >= 0) && (ts_in < Tb - 1);
        const float* gG = a.grad_hist + int64_t(b) * a.grad_stride;
        for (int i = lane; i < WarpBwd<64>::kCells; i += 32) {
            const int y = i >> 6, x = i & 63;
            Bw.acc[i] = 0.0;
            Bw.v[i] = 0.f;
            Bw.gh[i] = (y < H && x < W && !(blocked && i == goal_rc)) ? __ldg(gG + y * W + x) : 0.f;
        }
        __syncwarp();
        if (start_rc >= 0) {
            const float f0 = f_value(gr, omg, 0.f, sGH[start_rc].y);
            const float v0 = expf(__fdiv_rn(-f0, a.sqrt_w));                 // :207
            if (lane == 0) { Bw.v[start_rc] = v0; Bw.a0[start_rc] = 0.0; Bw.b0[start_rc] = 0.0; }
            Ssum = double(v0);
            Dsum = double(Bw.gh[start_rc]) * Ssum;
        }
    }
    __syncwarp();

    // ---------------- search loop --------------------------------------------------------------
    const int T = kBwd ? Tb : p.T;
    const bool stationary_ok = (gr >= 0.5f);   // post-solve steps are stationary (SURVEY App. A.4)
    int t_solve = NASTAR_TS_CAPPED;
    int32_t* trace = kTrace ? (p.trace + int64_t(b) * T) : nullptr;
    int t = 0;
    for (; t < T; ++t) {
        // local best of the lane's two rows (strict <: the lower row wins ties)
        uint32_t bk = rm_key[0];
        int bid = (lane << 6) | rm_col[0];
        if (rm_key[1] < bk) { bk = rm_key[1]; bid = ((lane + 32) << 6) | rm_col[1]; }
        const uint32_t m = __reduce_min_sync(kFull, bk);
        if (m == kKeyInf) { t_solve = NASTAR_TS_EXHAUSTED; break; }
        double A1 = 0.0, B1 = 0.0;   // prefix sums INCLUDING step t (the events of step t act from t+1 on)
        if (kBwd) {
            const double inv = 1.0 / (Ssum + Slo);
            const double a_t = inv, b_t = (Dsum + Dlo) * inv * inv;
            if (stationary_ok && (ts_in >= 0) && (t == ts_in + 1)) {
                // solved: the goal is re-selected with a frozen open set until step T_batch-1
                Acum += double(Tb - t) * a_t;
                Bcum += double(Tb - t) * b_t;
                break;
            }
            A1 = Acum + a_t;
            B1 = Bcum + b_t;
        }
        const uint32_t ind = __reduce_min_sync(kFull, (bk == m) ? uint32_t(bid) : 0xFFFFFFFFu);
        const int r = int(ind >> 6), c = int(ind & 63u);
        if (kTrace && lane == 0) trace[t] = r * W + c;
        const bool solved = (int(ind) == goal_rc);
        const u64 m1 = 1ull << c, m0 = m1 >> 1, m2 = m1 << 1;
        // rescan inputs: columns lane and lane+32 of row r
        const u64 open_r = (kContinue && solved) ? S.open_row[r] : (S.open_row[r] & ~m1);
        const uint32_t ka = S.key[(r << 6) + lane], kb = S.key[(r << 6) + 32 + lane];
        uint32_t rs_key = ((open_r >> lane) & 1ull) ? ka : kKeyInf;
        int rs_col = lane;
        {
            const uint32_t kb2 = ((open_r >> (lane + 32)) & 1ull) ? kb : kKeyInf;
            if (kb2 < rs_key) { rs_key = kb2; rs_col = lane + 32; }
        }
        // which of this lane's rows (if any) is in r-1..r+1
        const int d0 = lane - r, d1 = lane + 32 - r;
        const bool near1 = (unsigned(d1 + 1) <= 2u);
        const bool near = (unsigned(d0 + 1) <= 2u) | near1;
        const int dr = near1 ? d1 : d0;
        const bool isr = near & (dr == 0);
        const int myrow = near1 ? (lane + 32) : lane;
        u64 myopen = near1 ? open[1] : open[0];
        u64 myclosed = near1 ? closed[1] : closed[0];
        const u64 mypass = near1 ? pass[1] : pass[0];
        uint32_t mykey = near1 ? rm_key[1] : rm_key[0];
        int mycol = near1 ? rm_col[1] : rm_col[0];
        const int cell = (myrow << 6) + c;
        float2 n0 = make_float2(0.f, 0.f), n1 = n0, n2 = n0;
        if (near) { n0 = sGH[cell - 1]; n1 = sGH[cell]; n2 = sGH[cell + 1]; }
        const float g2 = __fadd_rn(sGH[ind].x, S.cost[ind]);
        __syncwarp();   // read phase ends
        if (isr) {
            myclosed |= m1;
            if (!solved) myopen &= ~m1;
            mykey = kKeyInf;
        }
        const u64 win = isr ? (m0 | m2) : (m0 | m1 | m2);
        const u64 cand = near ? (win & mypass) : 0ull;
        const u64 gt = ((n0.x > g2) ? m0 : 0ull) | ((n1.x > g2) ? m1 : 0ull) | ((n2.x > g2) ? m2 : 0ull);
        const u64 upd = cand & ((myopen & gt) | ~(myopen | myclosed));
        myopen |= upd;
        const float ag = __fmul_rn(gr, g2);
        const float f0n = __fadd_rn(ag, __fmul_rn(omg, n0.y));
        const float f1n = __fadd_rn(ag, __fmul_rn(omg, n1.y));
        const float f2n = __fadd_rn(ag, __fmul_rn(omg, n2.y));
        const bool u0 = (upd & m0) != 0ull, u1 = (upd & m1) != 0ull, u2 = (upd & m2) != 0ull;
        const uint32_t q0 = fkey(f0n), q1 = fkey(f1n), q2 = fkey(f2n);
        const int off = (dr << 6) - 1;
        if (u0) { sGH[cell - 1].x = g2; S.key[cell - 1] = q0; S.par[cell - 1] = int8_t(off); }
        if (u1) { sGH[cell].x = g2;     S.key[cell] = q1;     S.par[cell] = int8_t(off + 1); }
        if (u2) { sGH[cell + 1].x = g2; S.key[cell + 1] = q2; S.par[cell + 1] = int8_t(off + 2); }
        if (kBwd) {
            double dS = 0.0, dD = 0.0;   // this lane's change of S and D
            auto event = [&](int cl, float v_new) {
                const double gh = double(Bw.gh[cl]);
                const double dv = Bw.planes().event(cl, gh, v_new, A1, B1);
                dS += dv;
                dD += gh * dv;
            };
            if (u0) event(cell - 1, expf(__fdiv_rn(-f0n, a.sqrt_w)));     // :207
            if (u1) event(cell, expf(__fdiv_rn(-f1n, a.sqrt_w)));
            if (u2) event(cell + 1, expf(__fdiv_rn(-f2n, a.sqrt_w)));
            if (isr && !solved) event(int(ind), 0.f);                      // the selected cell leaves the open set
            // the events sit on the (at most three) lanes that own rows r-1, r, r+1
            const int l0 = (r - 1) & 31, l1 = r & 31, l2 = (r + 1) & 31;
            dd_add(Ssum, Slo, __shfl_sync(kFull, dS, l0) + __shfl_sync(kFull, dS, l1) + __shfl_sync(kFull, dS, l2));
            dd_add(Dsum, Dlo, __shfl_sync(kFull, dD, l0) + __shfl_sync(kFull, dD, l1) + __shfl_sync(kFull, dD, l2));
            Acum = A1;
            Bcum = B1;
        }
        const uint32_t k0 = u0 ? q0 : kKeyInf, k1 = u1 ? q1 : kKeyInf, k2 = u2 ? q2 : kKeyInf;
        uint32_t fk = k0;
        int fc = c - 1;
        if (k1 < fk) { fk = k1; fc = c; }
        if (k2 < fk) { fk = k2; fc = c + 1; }
        if ((fk < mykey) | ((fk == mykey) & (fc < mycol))) { mykey = fk; mycol = fc; }
        if (near) {
            if (near1) { open[1] = myopen; closed[1] = myclosed; rm_key[1] = mykey; rm_col[1] = mycol; }
            else       { open[0] = myopen; closed[0] = myclosed; rm_key[0] = mykey; rm_col[0] = mycol; }
            S.open_row[myrow] = myopen;
        }
        if (solved && t_solve < 0) t_solve = t;
        if (!kContinue && solved) break;
        // fold the rescan into the cached minimum of row r (lane r&31, slot r>>5)
        // (kept AFTER the expansion: hoisting these two reductions above it, as the warp32 engine does, lands them inside
        // the divergent region of the `near` lanes here and REDUX then takes its slow divergent path — 3.6x slower)
        const uint32_t mr = __reduce_min_sync(kFull, rs_key);
        const uint32_t mc = __reduce_min_sync(kFull, (rs_key == mr) ? uint32_t(rs_col) : 0xFFFFFFFFu);
        if (lane == (r & 31)) {
            if (r >> 5) {
                if ((mr < rm_key[1]) | ((mr == rm_key[1]) & (int(mc) < rm_col[1]))) { rm_key[1] = mr; rm_col[1] = int(mc); }
            } else {
                if ((mr < rm_key[0]) | ((mr == rm_key[0]) & (int(mc) < rm_col[0]))) { rm_key[0] = mr; rm_col[0] = int(mc); }
            }
        }
        __syncwarp();
    }
    __syncwarp();
    const int steps = (!kContinue && t_solve >= 0) ? (t + 1) : t;

    if (kBwd) {
        // close the intervals of the cells still open, scale: dL/dcost = -(1-g_ratio)/sqrt(W) * acc
        const double coef = -double(omg) / double(a.sqrt_w);
        float* gOut = a.grad_cost + int64_t(b) * N;
        for (int i = lane; i < WarpBwd<64>::kCells; i += 32) {
            const int y = i >> 6, x = i & 63;
            if (y < H && x < W) {
                const double acc = Bw.planes().close(i, Acum, Bcum, [&] { return double(Bw.gh[i]); });
                gOut[y * W + x] = float(coef * acc);
            }
        }
        return;
    }

    // ---------------- backtrack ------------------------------------------------------------------
    u64 path0 = 0ull, path1 = 0ull;
    {
        const int myslot_row0 = lane, myslot_row1 = lane + 32;
#define NASTAR_MARK(LOC)                                                   \
        {                                                                  \
            const int y_ = (LOC) >> 6;                                     \
            const u64 bit_ = 1ull << ((LOC) & 63);                         \
            path0 |= (y_ == myslot_row0) ? bit_ : 0ull;                    \
            path1 |= (y_ == myslot_row1) ? bit_ : 0ull;                    \
        }
        NASTAR_MARK(goal_rc)
        int loc = goal_rc - S.par[goal_rc];
        const int hops = (t_solve >= 0) ? N : (T - 1);
        for (int k = 0; k < hops; ++k) {
            NASTAR_MARK(loc)
            if (loc == start_rc || loc == goal_rc) break;
            loc -= S.par[loc];
        }
#undef NASTAR_MARK
    }

    // ---------------- epilogue -------------------------------------------------------------------
    S.bits_a[lane] = closed[0];
    S.bits_a[lane + 32] = closed[1];
    S.bits_b[lane] = path0;
    S.bits_b[lane + 32] = path1;
    __syncwarp();
    float* gHist = p.histories + int64_t(b) * N;
    long long* gPath = reinterpret_cast<long long*>(p.paths) + int64_t(b) * N;
    if (W == 64 && aligned16(gHist) && aligned16(gPath)) {
        const int x = (lane & 15) << 2;
        const int n4 = N >> 2;
        for (int i4 = lane; i4 < n4; i4 += 32) {
            const int y = i4 >> 4;
            const uint32_t cb = uint32_t(S.bits_a[y] >> x), pb = uint32_t(S.bits_b[y] >> x);
            reinterpret_cast<float4*>(gHist)[i4] = make_float4((cb & 1u) ? 1.f : 0.f, (cb & 2u) ? 1.f : 0.f,
                                                               (cb & 4u) ? 1.f : 0.f, (cb & 8u) ? 1.f : 0.f);
            reinterpret_cast<longlong2*>(gPath)[2 * i4] = make_longlong2((pb & 1u) ? 1ll : 0ll, (pb & 2u) ? 1ll : 0ll);
            reinterpret_cast<longlong2*>(gPath)[2 * i4 + 1] = make_longlong2((pb & 4u) ? 1ll : 0ll, (pb & 8u) ? 1ll : 0ll);
        }
    } else {
        for (int y = 0; y < H; ++y) {
            for (int x = lane; x < W; x += 32) {
                gHist[y * W + x] = ((S.bits_a[y] >> x) & 1ull) ? 1.f : 0.f;
                gPath[y * W + x] = ((S.bits_b[y] >> x) & 1ull) ? 1ll : 0ll;
            }
        }
    }
    const int n_closed = __reduce_add_sync(kFull, __popcll(closed[0]) + __popcll(closed[1]));
    const int n_path = __reduce_add_sync(kFull, __popcll(path0) + __popcll(path1));
    if (lane == 0) {
        if (p.t_solve) p.t_solve[b] = t_solve;
        if (p.n_steps) p.n_steps[b] = steps;
        if (p.n_closed) p.n_closed[b] = n_closed;
        if (p.path_len) p.path_len[b] = n_path;
    }
}

}  // namespace nastar
