// nastar_common.cuh — device helpers shared by the A* engines (sm_100a).
//
// Arithmetic contract (SURVEY.md App. A): every fp32 operation of the reference's loop is a
// separately rounded IEEE op (ATen element-wise kernels; no FMA contraction), so all
// numerics that feed comparisons go through __fmul_rn/__fadd_rn/__fsqrt_rn here.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/nastar_b200.h"

namespace nastar {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr uint32_t kKeyInf = 0xFFFFFFFFu;  // "no open cell" sentinel, above every float key

// Kernel arguments of every search engine: the forward parameters plus the extra fields of nastar_bwd_params.
struct SearchArgs {
    nastar_fwd_params f;
    // backward only
    float sqrt_w;
    const int32_t* T_batch;     // device scalar: loop iterations the reference would execute
    const int32_t* t_solve_in;  // forward's t_solve[] (goal clamp blocking, App. B)
    const float* grad_hist;
    int64_t grad_stride;
    float* grad_cost;
    // generic engine, forward only, nullable: per-map flags written by the bin16 engine (nastar_bin16.cuh); when
    // given, only maps with redo[b] != 0 are processed (the others were already finished on-chip)
    const int32_t* redo;
};

// Order-preserving map float -> uint32 (a < b  <=>  key(a) < key(b) for non-NaN a, b).
__device__ __forceinline__ uint32_t fkey(float f) {
    uint32_t b = __float_as_uint(f);
    return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}

// f = g_ratio*g + (1-g_ratio)*h   (differentiable_astar.py:206) — three roundings.
__device__ __forceinline__ float f_value(float gr, float omg, float g, float h) {
    return __fadd_rn(__fmul_rn(gr, g), __fmul_rn(omg, h));
}

// get_heuristic (differentiable_astar.py:26-52): chebyshev + 0.001 * euclid, all in fp32.
__device__ __forceinline__ float heuristic(int y, int x, int gy, int gx) {
    int idy = y - gy, idx = x - gx;
    int ady = idy < 0 ? -idy : idy, adx = idx < 0 ? -idx : idx;
    float cheb = static_cast<float>(ady + adx - (ady < adx ? ady : adx));   // exact
    float euc = __fsqrt_rn(static_cast<float>(ady * ady + adx * adx));       // exact int -> IEEE sqrt
    return __fadd_rn(cheb, __fmul_rn(0.001f, euc));
}

// encoder.py:32-34, cost = sigmoid(x) * const, with the operation sequence of ATen's CUDA sigmoid
// (1 / (1 + exp(-x)), full-precision expf and IEEE division) followed by a separately rounded multiply.
__device__ __forceinline__ float sigmoid_scaled(float x, float scale) {
    return __fmul_rn(__fdiv_rn(1.f, __fadd_rn(1.f, expf(-x))), scale);
}

// NASTAR_COST_TAPS: logit(y,x) = bias + sum_k taps[y+ky-1][x+kx-1][k], k = ky*3+kx ascending, zero padding —
// the 9->1 gather that finishes the encoder's single-output-channel 3x3 convolution (planner/encoder.py
// `_conv3x3_single_output`).  taps is one map's [H*W][9] block.
__device__ __forceinline__ float cost_from_taps(const float* __restrict__ taps, int y, int x, int H, int W,
                                                float bias, float scale) {
    float acc = bias;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int yy = y + ky - 1;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int xx = x + kx - 1;
            if (unsigned(yy) < unsigned(H) && unsigned(xx) < unsigned(W))
                acc = __fadd_rn(acc, __ldg(taps + (int64_t(yy) * W + xx) * 9 + (ky * 3 + kx)));
        }
    }
    return sigmoid_scaled(acc, scale);
}

// one cost value under nastar_fwd_params.cost_kind (include/nastar_b200.h NASTAR_COST_*)
__device__ __forceinline__ float cost_value(int kind, const float* __restrict__ src, int y, int x, int H, int W,
                                            float bias, float scale) {
    if (kind == 0) return __ldg(src + y * W + x);
    if (kind == 1) return sigmoid_scaled(__ldg(src + y * W + x), scale);
    return cost_from_taps(src, y, x, H, W, bias, scale);
}

// Double-double accumulator for the running sums of the event-based backward (S = sum of exp(-f/sqrt(W)) over the
// open set, D = <Gh, v>).  Over a long search S decays by many orders of magnitude (the selected cell is always the
// LARGEST term): a plain fp64 running sum keeps an absolute error of 1e-16 x the early, large values, which becomes
// a large relative error once S has shrunk by 1e-10 or more (cost x10, 64x64 maps).  With an error-free TwoSum the
// pair (hi, lo) carries ~106 bits, so removed terms cancel exactly against the identical values added earlier.
__device__ __forceinline__ void dd_add(double& hi, double& lo, double x) {
    const double s = __dadd_rn(hi, x);
    const double bb = __dadd_rn(s, -hi);
    const double err = __dadd_rn(__dadd_rn(hi, -__dadd_rn(s, -bb)), __dadd_rn(x, -bb));
    lo = __dadd_rn(lo, err);
    const double t = __dadd_rn(s, lo);
    lo = __dadd_rn(lo, -__dadd_rn(t, -s));
    hi = t;
}

// Per-cell state of the event-based backward (SURVEY App. B), in shared memory or in a workspace slot.
// dL/dcost[p] = -(1-g_ratio)/sqrt(W) * sum_t y_t[p] * (Gh[p] - <Gh, y_t>) with y_t = v_t / S_t over the open set.
// A cell's softmax weight v = exp(-f/sqrt(W)) only changes when it is opened, relaxed or closed, so its contribution
// over an interval [t0, t1) of constant v is v * (Gh * (A(t1)-A(t0)) - (B(t1)-B(t0))) with the prefix sums
// A(t) = sum_{tau<t} 1/S_tau and B(t) = sum_{tau<t} D_tau/S_tau^2, D_t = <Gh, v_t>.
struct IntervalPlanes {
    double* acc;  // closed intervals: sum of v * (Gh * dA - dB)
    double* a0;   // A(t0), B(t0) of the cell's current open interval
    double* b0;
    float* v;     // softmax numerator of open cells, else 0

    // The weight of cell i changes to v_new (0: the cell leaves the open set) from the next step on; A1, B1 are the
    // prefix sums including the current step.  Returns the change of v.
    __device__ __forceinline__ double event(int i, double gh, float v_new, double A1, double B1) const {
        const float v_old = v[i];
        if (v_old != 0.f) acc[i] += double(v_old) * (gh * (A1 - a0[i]) - (B1 - b0[i]));
        v[i] = v_new;
        a0[i] = A1;
        b0[i] = B1;
        return double(v_new) - double(v_old);
    }
    // The open cell i is closed (the generic engine's selection event): its last interval ends at A1, B1; A(t0) and
    // B(t0) are left stale, a closed cell is never reopened.  Returns the change of v.
    __device__ __forceinline__ double leave(int i, double gh, double A1, double B1) const {
        const float v_old = v[i];
        acc[i] += double(v_old) * (gh * (A1 - a0[i]) - (B1 - b0[i]));
        v[i] = 0.f;
        return -double(v_old);
    }
    // acc of cell i with its open interval (if any) closed at the end of the search, prefix sums A, B; gh_at() gives
    // the cell's upstream gradient and is only evaluated for open cells
    template <typename GhAt>
    __device__ __forceinline__ double close(int i, double A, double B, GhAt gh_at) const {
        double r = acc[i];
        const float vi = v[i];
        if (vi != 0.f) r += double(vi) * (gh_at() * (A - a0[i]) - (B - b0[i]));
        return r;
    }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP) -------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace nastar
