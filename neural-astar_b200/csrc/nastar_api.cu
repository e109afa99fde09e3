// nastar_api.cu — C-ABI entry points of libnastar_b200.so (see include/nastar_b200.h).
// Host side only validates, picks an engine and launches; no torch types, no CPU fallback.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>

#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "../../include/nastar_b200.h"
#include "nastar_bin16.cuh"
#include "nastar_generic.cuh"
#include "nastar_glue.cuh"
#include "nastar_warp.cuh"

namespace {
std::atomic<uint64_t> g_launches{0};
cudaError_t g_last_err = cudaSuccess;

constexpr size_t kMaxDynSmem = 232448;  // 227 KB opt-in limit per CTA on sm_100
constexpr int kGlobalCtasPerSm = 8;

int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

// one-time fill of the warp engines' heuristic table on the current device (stream-ordered before first use)
cudaError_t ensure_heur(cudaStream_t stream) {
    static std::atomic<uint64_t> done_mask{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = uint64_t(1) << (dev & 63);
    if (done_mask.load(std::memory_order_acquire) & bit) return cudaSuccess;
    nastar::heur_init_kernel<<<nastar::kHeurCells / 256, 256, 0, stream>>>();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // later launches on OTHER streams must also see the table: finish the fill before publishing
    e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return e;
    done_mask.fetch_or(bit, std::memory_order_release);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaSuccess;
}

// Calls f with each runtime flag as a std::integral_constant<bool>, so that f can pick the kernel template
// instantiation: with_flags(f, x, y) calls f(bool_constant<x>, bool_constant<y>).
template <typename F>
auto with_flags(F&& f) {
    return f();
}
template <typename F, typename... Flags>
auto with_flags(F&& f, bool first, Flags... rest) {
    if (first) return with_flags([&](auto... c) { return f(std::true_type{}, c...); }, rest...);
    return with_flags([&](auto... c) { return f(std::false_type{}, c...); }, rest...);
}

// the kernels' arguments for a backward call; the loop bound comes from *T_batch on the device (f.T = 0)
nastar::SearchArgs backward_args(const nastar_bwd_params* p) {
    nastar::SearchArgs a{};
    a.f.cost = p->cost;   a.f.cost_stride = p->cost_stride;
    a.f.start = p->start; a.f.start_stride = p->start_stride;
    a.f.goal = p->goal;   a.f.goal_stride = p->goal_stride;
    a.f.obst = p->obst;   a.f.obst_stride = p->obst_stride;
    a.f.B = p->B; a.f.H = p->H; a.f.W = p->W;
    a.f.g_ratio = p->g_ratio;
    a.f.one_minus_g_ratio = p->one_minus_g_ratio;
    a.f.workspace = p->workspace;
    a.f.workspace_bytes = p->workspace_bytes;
    a.sqrt_w = p->sqrt_w;
    a.T_batch = p->T_batch;
    a.t_solve_in = p->t_solve;
    a.grad_hist = p->grad_histories;
    a.grad_stride = p->grad_stride;
    a.grad_cost = p->grad_cost;
    return a;
}

// Launches kernel with `smem` bytes of dynamic shared memory (opting in above the 48 KB default).
template <typename Kernel>
cudaError_t launch_dyn(Kernel kernel, int grid, size_t smem, cudaStream_t stream, const nastar::SearchArgs& a) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32, smem, stream>>>(a);
    return cudaSuccess;
}

// generic engine variant for a shape: 2 = state in shared memory, 3 = state in the HBM workspace, 0 = too large
int generic_engine_for(int32_t H, int32_t W) {
    if (H <= 0 || W <= 0 || int64_t(H) * W > (int64_t(1) << 30)) return 0;
    const nastar::GenericLayout L(H, W);
    if (L.smem_common() + L.smem_planes() <= kMaxDynSmem) return 2;
    if (L.smem_common() <= kMaxDynSmem) return 3;
    return 0;
}

int generic_slots(int B) {
    const int cap = num_sms() * kGlobalCtasPerSm;
    return B < cap ? B : cap;
}

// ---- engine 5 (nastar_bin16.cuh): binary-cost maps, one CTA per map --------------------------------------
// NASTAR_B200_BIN16=0 in the environment disables it (A/B measurements against engines 2/3)
bool bin16_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = std::getenv("NASTAR_B200_BIN16");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v != 0;
}

bool bin16_shape_ok(int32_t H, int32_t W) {
    if (H <= 0 || W <= 0 || (H <= 64 && W <= 64)) return false;   // engines 1 / 4 keep their shapes
    if (generic_engine_for(H, W) == 0) return false;
    const nastar::Bin16Layout L(H, W);
    return L.supported() && L.smem_bytes() <= kMaxDynSmem;
}

// head of the workspace when engine 5 may run: [0,256) work-queue counter, then B redo flags (256-B granules)
size_t bin16_aux_bytes(int32_t B) { return 256 + ((size_t(B) * 4 + 255) & ~size_t(255)); }

inline int cuda_fail(cudaError_t e) {
    g_last_err = e;
    return NASTAR_ECUDA;
}

__global__ void batch_steps_kernel(const int32_t* __restrict__ t_solve, const int32_t* __restrict__ n_steps,
                                   int B, int T, int32_t* __restrict__ out) {
    // T_batch = number of iterations of the reference's batch-synchronous loop
    // (differentiable_astar.py:203,251-252): it stops right after the slowest map's solve step,
    // or runs all T iterations if some map never reaches its goal.
    int m = 0;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        const int ts = t_solve[i];
        const int v = (ts >= 0) ? (ts + 1) : T;
        m = max(m, v);
        (void)n_steps;
    }
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    __shared__ int sm[32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : 0;
        for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
        if (threadIdx.x == 0) out[0] = min(m, T);
    }
}
}  // namespace

namespace {
template <int C>
cudaError_t launch_head(const float* x, int64_t P, const float* w_host, float* taps, cudaStream_t stream) {
    nastar::HeadWeights<C> hw;
    for (int i = 0; i < C * 9; ++i) hw.w[i] = w_host[i];
    const int64_t want = ((P + 31) / 32 + nastar::kHeadWarps - 1) / nastar::kHeadWarps;   // one 32-pixel group per warp
    const int64_t cap = int64_t(num_sms()) * 16;
    nastar::head_taps_kernel<C><<<unsigned(want < cap ? want : cap), 32 * nastar::kHeadWarps, 0, stream>>>(x, P, hw, taps);
    return cudaGetLastError();
}
}  // namespace

extern "C" {

int nastar_b200_abi_version(void) { return NASTAR_B200_ABI_VERSION; }

int nastar_b200_engine_for(int32_t H, int32_t W) {
    if (H <= 0 || W <= 0) return 0;
    if (H <= 32 && W <= 32) return 1;
    if (H <= 64 && W <= 64) return 4;   // forward and (event-based) backward on the warp-resident 64-wide engine
    return generic_engine_for(H, W);
}

int nastar_b200_bin16_supported(int32_t H, int32_t W) { return bin16_shape_ok(H, W) ? 1 : 0; }

size_t nastar_b200_forward_workspace_bytes(int32_t B, int32_t H, int32_t W) {
    if (B <= 0) return 0;
    const int engine = nastar_b200_engine_for(H, W);
    if (engine != 2 && engine != 3) return 0;
    size_t n = (engine == 3) ? size_t(generic_slots(B)) * nastar::GenericLayout(H, W).slot_bytes() : 0;
    if (bin16_enabled() && bin16_shape_ok(H, W)) n += bin16_aux_bytes(B);
    return n;
}

size_t nastar_b200_backward_workspace_bytes(int32_t B, int32_t H, int32_t W) {
    if (B <= 0 || nastar_b200_engine_for(H, W) == 1 || nastar_b200_engine_for(H, W) == 4) return 0;
    const int e = generic_engine_for(H, W);
    if (e == 0) return 0;
    return size_t(generic_slots(B)) * nastar::GenericLayout(H, W).slot_total(e == 3, true);
}

int nastar_b200_forward(const nastar_fwd_params* p, void* stream_v) {
    if (!p || !p->cost || !p->start || !p->goal || !p->obst || !p->histories || !p->paths) return NASTAR_EINVAL;
    if (p->B <= 0 || p->H <= 0 || p->W <= 0 || p->T < 1) return NASTAR_EINVAL;
    if (p->cost_kind < NASTAR_COST_PLANE || p->cost_kind > NASTAR_COST_TAPS) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const int engine = nastar_b200_engine_for(p->H, p->W);
    if (engine == 0) return NASTAR_EUNSUPPORTED;
    if (p->cost_kind != NASTAR_COST_PLANE && engine != 1 && engine != 4) return NASTAR_EUNSUPPORTED;   // fused hand-off: H,W <= 64
    const bool pair = (p->flags & NASTAR_FWD_PAIR) != 0;
    if (pair && engine != 1) {
        // two halves back to back: the learned-cost search, then the same problems with cost = obstacles
        const int64_t N = int64_t(p->H) * p->W;
        nastar_fwd_params h = *p;
        h.flags &= ~NASTAR_FWD_PAIR;
        int st = nastar_b200_forward(&h, stream_v);
        if (st != NASTAR_OK) return st;
        h.cost = p->obst;
        h.cost_stride = p->obst_stride;
        h.cost_kind = NASTAR_COST_PLANE;
        h.histories = p->histories + int64_t(p->B) * N;
        h.paths = p->paths + int64_t(p->B) * N;
        if (p->t_solve) h.t_solve = p->t_solve + p->B;
        if (p->n_steps) h.n_steps = p->n_steps + p->B;
        if (p->trace) h.trace = p->trace + int64_t(p->B) * p->T;
        if (p->n_closed) h.n_closed = p->n_closed + p->B;
        if (p->path_len) h.path_len = p->path_len + p->B;
        return nastar_b200_forward(&h, stream_v);
    }
    const int nmaps = pair ? 2 * p->B : p->B;   // output slots (= CTAs of the warp32 engine)
    if (p->trace) {
        cudaError_t e = cudaMemsetAsync(p->trace, 0xFF, size_t(nmaps) * size_t(p->T) * sizeof(int32_t), stream);
        if (e != cudaSuccess) return cuda_fail(e);
    }
    const bool trace = (p->trace != nullptr);
    const bool noexit = (p->flags & NASTAR_FWD_NO_EARLY_EXIT) != 0;
    const bool fused = (p->cost_kind != NASTAR_COST_PLANE);
    if (engine == 1 || engine == 4) {
        cudaError_t e = ensure_heur(stream);
        if (e != cudaSuccess) return cuda_fail(e);
        nastar::SearchArgs a{};
        a.f = *p;
        if (engine == 1) {
            with_flags([&](auto kTrace, auto kNoExit, auto kFused) {
                nastar::astar_warp32_kernel<kTrace, false, kNoExit, kFused><<<nmaps, 32, 0, stream>>>(a);
            }, trace, noexit, fused);
        } else {
            e = with_flags([&](auto kTrace, auto kNoExit, auto kFused) {
                return launch_dyn(nastar::astar_warp64_kernel<kTrace, false, kNoExit, kFused>, p->B,
                                  sizeof(nastar::WarpSmem<64>), stream, a);
            }, trace, noexit, fused);
            if (e != cudaSuccess) return cuda_fail(e);
        }
        g_launches.fetch_add(1, std::memory_order_relaxed);
    } else {
        const nastar::GenericLayout L(p->H, p->W);
        const bool global = (engine == 3);
        const size_t smem = L.smem_common() + (global ? 0 : L.smem_planes());
        int grid = p->B;
        const size_t slots_bytes = global ? size_t(generic_slots(p->B)) * L.slot_bytes() : 0;
        if (global) {
            grid = generic_slots(p->B);
            if (!p->workspace || p->workspace_bytes < slots_bytes) return NASTAR_EWORKSPACE;
        }
        nastar::SearchArgs ga{};
        ga.f = *p;
        // engine 5 first when the cost plane IS the binary obstacle plane (VanillaAstar / Config 5): whole map on
        // chip, one CTA per SM pulling maps from a queue; maps it flags are re-run below by the generic engine
        const bool aliased = (p->obst == p->cost) && (p->obst_stride == p->cost_stride);
        const size_t aux = bin16_aux_bytes(p->B);
        if (bin16_enabled() && aliased && !p->trace && p->flags == 0 && bin16_shape_ok(p->H, p->W) && p->workspace &&
            p->workspace_bytes >= aux + slots_bytes) {
            unsigned char* ws = static_cast<unsigned char*>(p->workspace);
            nastar::Bin16Args ba{};
            ba.f = *p;
            ba.queue = reinterpret_cast<int32_t*>(ws);
            ba.redo = reinterpret_cast<int32_t*>(ws + 256);
            cudaError_t e = cudaMemsetAsync(ba.queue, 0, 256, stream);
            if (e != cudaSuccess) return cuda_fail(e);
            const size_t bsmem = nastar::Bin16Layout(p->H, p->W).smem_bytes();
            auto launch16 = [&](auto kernel) -> cudaError_t {
                cudaError_t e2 = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bsmem));
                if (e2 != cudaSuccess) return e2;
                int per_sm = 1;   // resident CTAs per SM (1 at 256x256, a few for smaller maps)
                e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nastar::kBin16Threads, bsmem);
                if (e2 != cudaSuccess) return e2;
                per_sm = per_sm < 1 ? 1 : per_sm;
                const int bgrid = p->B < num_sms() * per_sm ? p->B : num_sms() * per_sm;
                kernel<<<bgrid, nastar::kBin16Threads, bsmem, stream>>>(ba);
                return cudaGetLastError();
            };
            e = (p->H <= 256) ? launch16(nastar::astar_bin16_kernel<8>) : launch16(nastar::astar_bin16_kernel<16>);
            if (e != cudaSuccess) return cuda_fail(e);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            ga.redo = ba.redo;
            ga.f.workspace = ws + aux;
            ga.f.workspace_bytes = p->workspace_bytes - aux;
        }
        const cudaError_t e = with_flags([&](auto kGlobal, auto kTrace, auto kNoExit) {
            return launch_dyn(nastar::astar_generic_kernel<kGlobal, kTrace, false, kNoExit>, grid, smem, stream, ga);
        }, global, trace, noexit);
        if (e != cudaSuccess) return cuda_fail(e);
        g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_backward(const nastar_bwd_params* p, void* stream_v) {
    if (!p || !p->cost || !p->start || !p->goal || !p->obst || !p->grad_histories || !p->grad_cost || !p->T_batch ||
        !p->t_solve)
        return NASTAR_EINVAL;
    if (p->B <= 0 || p->H <= 0 || p->W <= 0) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const int engine = nastar_b200_engine_for(p->H, p->W);
    if (engine == 0) return NASTAR_EUNSUPPORTED;
    const nastar::SearchArgs a = backward_args(p);
    cudaError_t e;
    if (engine == 1 || engine == 4) {
        e = ensure_heur(stream);
        if (e != cudaSuccess) return cuda_fail(e);
        // the event-based closed form keeps its per-cell interval state in dynamic shared memory (WarpBwd): 32 KB
        // next to the warp32 engine's 17.4 KB of static planes, 128 KB behind the warp64 engine's planes
        if (engine == 1) e = launch_dyn(nastar::astar_warp32_kernel<false, true>, p->B, sizeof(nastar::WarpBwd<32>), stream, a);
        else e = launch_dyn(nastar::astar_warp64_kernel<false, true>, p->B, sizeof(nastar::WarpSmem<64>) + sizeof(nastar::WarpBwd<64>), stream, a);
    } else {
        const nastar::GenericLayout L(p->H, p->W);
        const bool global = (engine == 3);
        const int grid = generic_slots(p->B);
        if (!p->workspace || p->workspace_bytes < size_t(grid) * L.slot_total(global, true)) return NASTAR_EWORKSPACE;
        const size_t smem = L.smem_common() + (global ? 0 : L.smem_planes());
        e = with_flags([&](auto kGlobal) {
            return launch_dyn(nastar::astar_generic_kernel<kGlobal, false, true>, grid, smem, stream, a);
        }, global);
    }
    if (e != cudaSuccess) return cuda_fail(e);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_batch_steps(const int32_t* t_solve, const int32_t* n_steps, int32_t B, int32_t T, int32_t* T_batch,
                            void* stream_v) {
    if (!t_solve || !T_batch || B <= 0 || T < 1) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    batch_steps_kernel<<<1, 256, 0, stream>>>(t_solve, n_steps, B, T, T_batch);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_pack_inputs(const float* map_designs, int32_t C, int32_t Hm, int32_t Wm, const float* start,
                            int64_t start_stride, const float* goal, int64_t goal_stride, int32_t B, int32_t H,
                            int32_t W, float* out, void* stream_v) {
    if (!map_designs || !start || !goal || !out || C <= 0 || Hm <= 0 || Wm <= 0 || B <= 0 || H <= 0 || W <= 0)
        return NASTAR_EINVAL;
    if ((C == 1 && (reinterpret_cast<uintptr_t>(out) & 7)) || (C == 3 && (reinterpret_cast<uintptr_t>(out) & 15)))
        return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const int64_t npix = int64_t(B) * Hm * Wm;
    const int64_t want = (npix + 255) / 256;
    const int grid = int(want < int64_t(num_sms()) * 16 ? want : int64_t(num_sms()) * 16);
    nastar::pack_inputs_kernel<<<grid, 256, 0, stream>>>(map_designs, C, Hm, Wm, start, start_stride, goal, goal_stride,
                                                         B, H, W, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_cost_from_taps(const float* taps, int32_t B, int32_t H, int32_t W, float bias, float scale,
                               float* cost, void* stream_v) {
    if (!taps || !cost || B <= 0 || H <= 0 || W <= 0) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    const int64_t total = int64_t(B) * H * W;
    const int64_t want = (total + 255) / 256;
    const int grid = int(want < int64_t(num_sms()) * 16 ? want : int64_t(num_sms()) * 16);
    nastar::cost_from_taps_kernel<<<grid, 256, 0, stream>>>(taps, B, H, W, bias, scale, cost);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_conv1_marks(const float* map_designs, const float* start, int64_t start_stride, const float* goal,
                            int64_t goal_stride, int32_t B, int32_t H, int32_t W, const float* w_host,
                            const float* bias_host, float* out, void* stream_v) {
    if (!map_designs || !start || !goal || !w_host || !bias_host || !out || B <= 0 || H <= 0 || W <= 0) return NASTAR_EINVAL;
    if (reinterpret_cast<uintptr_t>(out) & 15) return NASTAR_EINVAL;
    const int64_t n_pix = int64_t(B) * H * W;
    if (n_pix > (int64_t(1) << 30)) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    nastar::Conv1Weights cw;
    std::memcpy(cw.w, w_host, sizeof(cw.w));
    std::memcpy(cw.b, bias_host, sizeof(cw.b));
    const int64_t want = (n_pix + 32 * nastar::kConv1Warps - 1) / (32 * nastar::kConv1Warps);
    const int grid = int(want < int64_t(num_sms()) * 8 ? want : int64_t(num_sms()) * 8);
    nastar::conv1_marks_kernel<<<grid, 32 * nastar::kConv1Warps, 0, stream>>>(map_designs, start, start_stride, goal,
                                                                             goal_stride, int(n_pix), H, W, cw, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

int nastar_b200_head_taps(const float* x, int64_t P, int32_t C, const float* w_host, float* taps, void* stream_v) {
    if (!x || !w_host || !taps || P <= 0 || (reinterpret_cast<uintptr_t>(x) & 15)) return NASTAR_EINVAL;
    if (P > (int64_t(1) << 31) * 127) return NASTAR_EINVAL;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    cudaError_t e;
    switch (C) {
        case 32: e = launch_head<32>(x, P, w_host, taps, stream); break;
        case 64: e = launch_head<64>(x, P, w_host, taps, stream); break;
        case 128: e = launch_head<128>(x, P, w_host, taps, stream); break;
        case 256: e = launch_head<256>(x, P, w_host, taps, stream); break;
        default: return NASTAR_EUNSUPPORTED;
    }
    if (e != cudaSuccess) return cuda_fail(e);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return NASTAR_OK;
}

int nastar_b200_selftest_sqrt(int32_t n, int32_t* mismatches, void* stream_v) {
    if (n <= 0 || !mismatches) return NASTAR_EINVAL;
    nastar::sqrt_rn_int_check_kernel<<<num_sms() * 4, 256, 0, static_cast<cudaStream_t>(stream_v)>>>(n, mismatches);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e);
    return NASTAR_OK;
}

uint64_t nastar_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* nastar_b200_status_string(int s) {
    switch (s) {
        case NASTAR_OK: return "ok";
        case NASTAR_EINVAL: return "invalid argument";
        case NASTAR_EUNSUPPORTED: return "unsupported map shape or feature";
        case NASTAR_ECUDA: return "CUDA runtime error";
        case NASTAR_EWORKSPACE: return "workspace too small";
        default: return "unknown status";
    }
}

const char* nastar_b200_last_cuda_error(void) { return cudaGetErrorString(g_last_err); }

}  // extern "C"
