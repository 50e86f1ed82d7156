// C ABI of the risvec library (include/risvec.h): handle, state arena, launches.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"
#include "geom.cuh"
#include "ris.cuh"
#include "step.cuh"
#include "sarl_mma.cuh"
#include "sarl_mma_big.cuh"
#include "sarl_umma.cuh"
#include "marl_tma.cuh"
#include "pairing.cuh"
#include "episode.cuh"
#include "episode_log.cuh"
#include "replay.cuh"

using namespace risvec;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                             \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) return fail(RISVEC_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

// Every entry point runs on the handle's device and then gives the caller its own current device back
// (a single-process multi-GPU program must not find torch's current device changed by a library call).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
        else prev = -1;  // already current: nothing to restore
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
#define ENTER_DEVICE(dev)        \
    DeviceGuard _dev_guard(dev); \
    if (!_dev_guard.ok) return fail(RISVEC_ERR_CUDA, "cudaSetDevice(%d) failed", (int)(dev))

struct FieldDesc {
    size_t offset;
    int64_t rows, cols;
    int elem_bytes, is_float;
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// RISVEC_SARL_PATH pins the SARL rollout kernel for tests and A/B runs: auto (also spelled mma, and any unknown
// spelling) | mma-ldg (k_sarl_mma, no TMA staging) | mma-sync (k_sarl_mma_big for the shapes of k_sarl_umma) | v8 |
// generic (the FP32-pipe kernels)
enum SarlPath { kPathAuto, kPathMmaLdg, kPathMmaSync, kPathV8, kPathGeneric };
struct Overrides {
    SarlPath sarl;       // RISVEC_FORCE_GENERIC=1 makes it kPathGeneric
    bool marl_v8;        // RISVEC_MARL_PATH=v8: the MARL fast path stays on k_marl_v8
    bool force_generic;  // RISVEC_FORCE_GENERIC=1: the shape-generic kernels everywhere (tests)
};
Overrides read_overrides() {  // at risvec_create
    const char *fg = getenv("RISVEC_FORCE_GENERIC"), *sp = getenv("RISVEC_SARL_PATH"), *mp = getenv("RISVEC_MARL_PATH");
    const char* const sarl_names[] = {"auto", "mma-ldg", "mma-sync", "v8", "generic"};  // SarlPath order
    Overrides o{};
    o.force_generic = fg != nullptr && fg[0] == '1';
    o.marl_v8 = mp != nullptr && !strcmp(mp, "v8");
    for (int i = 1; i < 5; ++i)
        if (sp != nullptr && !strcmp(sp, sarl_names[i])) o.sarl = (SarlPath)i;
    if (o.force_generic) o.sarl = kPathGeneric;
    return o;
}

}  // namespace

struct risvec_env {
    Dims dims;
    State st;
    risvec_params_t params;
    int device;
    char* arena;
    size_t arena_bytes;
    FieldDesc fields[RISVEC_F_COUNT];
    unsigned long long reset_calls, mob_calls, chan_calls;
    int64_t launches;
    // device staging for the *_host entry points (grow-only) + their copy pipeline
    char* stage;
    size_t stage_bytes;
    char* scratch;  // |S|^2 hand-over between the cascade and scan kernels (grow-only)
    size_t scratch_bytes;
    int pipe_ready;
    cudaStream_t s_in, s_out;
    cudaEvent_t ev[2 * 64 + 3];  // 2 * kMaxChunks + 3: per chunk in / kernel, start, in done, done
    Overrides ovr;  // the kernel overrides of tests and A/B runs
    const char* step_kernel;  // name of the kernel(s) the latest rollout launched (risvec_last_step_kernel)
    double* stats_slots;      // attached statistics accumulator (risvec_attach_stats_accumulator) or null
    int stats_folded;         // the latest rollout kernel added its statistics itself
    unsigned char* ep_bits;   // [E] in the arena: stage bits of the current tick (episode clock, unfused shapes)
    int* ep_keys;             // [E] in the arena: episode index that keys the tick's draws (same)
    const double* env_params; // attached per-env parameter table [E, RISVEC_ENVP_COLS] (risvec_attach_env_params) or null
    const int32_t* ris_elem;  // attached per-env RIS size [E] (risvec_attach_ris_elements) or null
};

struct risvec_replay {
    ReplayMem m;
    int device;
    long long mem_cntr;      // host-counter mode
    int devcnt;              // device-counter mode (risvec_replay_use_device_counter): the count is *ctr.count
    ReplayCtr ctr;           // in the arena's tail, zero at creation
    char* base;
    size_t off[RISVEC_RB_COUNT + 1];
    int64_t launches;
};

namespace {

int check_launch(risvec_env* env, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RISVEC_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    env->launches += 1;
    return RISVEC_OK;
}
int check_step_launch(risvec_env* env, const char* what) {  // a rollout kernel: remember which one ran
    if (int rc = check_launch(env, what)) return rc;
    env->step_kernel = what;
    return RISVEC_OK;
}

int validate_params(const risvec_params_t* p) {
    if (p->n_up < 1 || p->n_down < 1 || p->n_left < 1 || p->n_right < 1 || p->n_up > RISVEC_MAX_LANES ||
        p->n_down > RISVEC_MAX_LANES || p->n_left > RISVEC_MAX_LANES || p->n_right > RISVEC_MAX_LANES)
        return fail(RISVEC_ERR_INVALID, "lane counts must be in [1, %d]", RISVEC_MAX_LANES);
    if (!(p->time_fast > 0) || !(p->time_slow > 0)) return fail(RISVEC_ERR_INVALID, "time_fast/time_slow must be > 0");
    if (p->data_buf_size - 1 <= 5) return fail(RISVEC_ERR_INVALID, "data_buf_size must be > 6");
    return RISVEC_OK;
}

void bind_state(risvec_env* env) {
    auto P = [&](int f) { return (void*)(env->arena + env->fields[f].offset); };
    State& s = env->st;
    s.pos_x = (double*)P(RISVEC_F_POS_X); s.pos_y = (double*)P(RISVEC_F_POS_Y);
    s.dir = (int*)P(RISVEC_F_DIR); s.vel = (int*)P(RISVEC_F_VEL);
    s.dist = (double*)P(RISVEC_F_DIST); s.angle = (double*)P(RISVEC_F_ANGLE); s.amp = (double*)P(RISVEC_F_AMP);
    s.theta_re = (double*)P(RISVEC_F_THETA_RE); s.theta_im = (double*)P(RISVEC_F_THETA_IM);
    s.phase_real = (float*)P(RISVEC_F_PHASE_REAL);
    s.gains = (double*)P(RISVEC_F_GAINS); s.databuf = (double*)P(RISVEC_F_DATABUF);
    s.data_t = (float*)P(RISVEC_F_DATA_T); s.data_p = (float*)P(RISVEC_F_DATA_P);
    s.over_data = (float*)P(RISVEC_F_OVER_DATA); s.over_power = (float*)P(RISVEC_F_OVER_POWER);
    s.rate = (float*)P(RISVEC_F_RATE); s.data_r = (int*)P(RISVEC_F_DATA_R);
    s.reward_user = (float*)P(RISVEC_F_REWARD_USER); s.reward = (float*)P(RISVEC_F_REWARD);
    s.mecq = (double*)P(RISVEC_F_MECQ); s.stats = (float*)P(RISVEC_F_STATS);
    s.last_power = (float*)P(RISVEC_F_LAST_POWER); s.step_ctr = (long long*)P(RISVEC_F_STEP_CTR);
}

int ensure_stage(risvec_env* env, size_t bytes) {
    if (bytes <= env->stage_bytes) return RISVEC_OK;
    if (env->stage) cudaFree(env->stage);
    env->stage = nullptr;
    env->stage_bytes = 0;
    CUDA_TRY(cudaMalloc((void**)&env->stage, bytes));
    env->stage_bytes = bytes;
    return RISVEC_OK;
}

// -------------------------------------------------------------------------- launch helpers
int ensure_scratch(risvec_env* env, size_t bytes) {
    if (bytes <= env->scratch_bytes) return RISVEC_OK;
    if (env->scratch) cudaFree(env->scratch);
    env->scratch = nullptr;
    env->scratch_bytes = 0;
    CUDA_TRY(cudaMalloc((void**)&env->scratch, bytes));
    env->scratch_bytes = bytes;
    return RISVEC_OK;
}

// f(std::true_type{}) while a per-env parameter table is attached (the PE instantiations), else f(std::false_type{})
template <typename F>
int dispatch_pe(const risvec_env* env, F&& f) {
    return env->env_params ? f(std::true_type{}) : f(std::false_type{});
}
// the same for an attached per-env RIS size (the NE instantiations)
template <typename F>
int dispatch_re(const risvec_env* env, F&& f) {
    return env->ris_elem ? f(std::true_type{}) : f(std::false_type{});
}

// f(std::integral_constant<int, VP>{}) for the least power of two VP >= V (V <= 32); dispatch_vp<8> starts at 8
template <int VP = 1, typename F>
int dispatch_vp(int V, F&& f) {
    if constexpr (VP < 32)
        if (V > VP) return dispatch_vp<2 * VP>(V, f);
    return f(std::integral_constant<int, VP>{});
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }
inline bool aligned8(const void* p) { return ((uintptr_t)p & 7u) == 0; }

// ---- tensor maps over the caller's arrays, encoded per call
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {  // cuTensorMapEncodeTiled through the runtime (no link-time libcuda dependency)
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        else
            cudaGetLastError();
    }
    return fn;
}
// rows x inner 4-byte elements, dense; box = box_rows x box_inner
bool tensor_map_2d(CUtensorMap* m, CUtensorMapDataType dt, const void* base, uint64_t inner, uint64_t rows,
                   uint32_t box_inner, uint32_t box_rows) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[2] = {inner, rows}, strides[1] = {inner * 4};
    const cuuint32_t box[2] = {box_inner, box_rows}, estr[2] = {1, 1};
    return enc(m, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
           CUDA_SUCCESS;
}
// the [T][E * V] float traces of a rollout, 16 steps x box_inner floats per box
template <int N>
bool trace_maps(CUtensorMap (&m)[N], float* const (&traces)[N], const Dims& d, int T, uint32_t box_inner) {
    for (int n = 0; n < N; ++n)
        if (!tensor_map_2d(&m[n], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, traces[n], (uint64_t)d.E * d.V, T, box_inner, 16))
            return false;
    return true;
}

// ---- SARL: the rollout kernels in the order they are tried (choose_sarl)
enum SarlKernel { kSarlMmaTma, kSarlMma, kSarlUmma, kSarlMmaBig, kSarlV8, kSarlRollout, kSarlCascade };

bool sarl_traces(const risvec_sarl_out_t& o) {  // every per-vehicle trace given, 16-byte aligned
    const float* const t[6] = {o.DataBuf, o.data_t, o.data_p, o.over_power, o.over_data, o.rate};
    for (const float* p : t)
        if (!p || !aligned16(p)) return false;
    return true;
}
// k_sarl_mma_tma covers the BASELINE shape: V = 8, E % 4 == 0, M = 16 or 40, every trace + the arrivals supplied,
// 16-byte aligned streams, 32-bit element indices
bool sarl_tma_covers(const Dims& d, const SarlArgs& a) {
    return d.V == 8 && d.E % 4 == 0 && (d.M == 16 || d.M == 40) && sarl_traces(a.out) && a.arrivals &&
           a.out.reward && aligned16(a.phase) && aligned16(a.action) && aligned16(a.arrivals) &&
           aligned16(a.out.reward) && (uint64_t)a.T * d.E * std::max(d.M, 16) < (1ull << 31);
}
// k_sarl_umma / k_sarl_mma_big: one block per env for many vehicles or elements (config 4)
bool sarl_big_covers(const Dims& d, const SarlArgs& a) {
    return d.V % 4 == 0 && d.V <= 32 && d.M % 2 == 0 && d.M <= 256 && (d.V > 8 || d.M > 64) && sarl_traces(a.out) &&
           aligned8(a.phase) && (uint64_t)a.T * d.E * std::max(d.M, 2 * d.V) < (1ull << 31);
}

// The kernel of a SARL rollout (`a.in_rec`: packed records, `a.raw`: the fused driver step), the first candidate
// from `from` on that takes the call; a caller whose tensor maps cannot be encoded asks again from the next one.
SarlKernel choose_sarl(const risvec_env* env, const SarlArgs& a, int from = kSarlMmaTma) {
    const Dims& d = env->dims;
    const SarlPath p = env->ovr.sarl;
    if (a.in_rec) return kSarlV8;  // the caller checked the packed shape
    // an attached per-env parameter table or RIS size: only k_sarl_mma and the generic kernels have PE / NE
    // instantiations
    const bool pe = env->env_params != nullptr || env->ris_elem != nullptr;
    const bool mma = p == kPathAuto || p == kPathMmaLdg || p == kPathMmaSync;
    // tensor cores, one warp per env: V <= 8, M even, M <= 64
    const bool mma_fits = mma && d.V <= 8 && d.M % 2 == 0 && d.M <= 64 && (!a.raw || aligned8(a.raw));
    if (from <= kSarlMmaTma && mma_fits && !pe && p != kPathMmaLdg && sarl_tma_covers(d, a)) return kSarlMmaTma;
    if (from <= kSarlMma && mma_fits) return kSarlMma;
    const bool big = mma && !pe && p != kPathMmaLdg && sarl_big_covers(d, a);
    if (from <= kSarlUmma && big && p != kPathMmaSync) return kSarlUmma;
    if (from <= kSarlMmaBig && big && p == kPathMmaSync) return kSarlMmaBig;
    if (d.V <= 8 && d.M <= 40 && p != kPathGeneric && !pe) return kSarlV8;  // elements split over the env's 8 lanes
    return d.M <= 40 ? kSarlRollout : kSarlCascade;
}

// tensor cores + TMA staging (sarl_mma.cuh); dynamic + static shared memory stay under the 48 KB default
int launch_sarl_mma_tma(risvec_env* env, const SarlArgs& a, cudaStream_t st, bool* launched) {
    const Dims& d = env->dims;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    CUtensorMap tm_ph, tm_ac, tm_ar;
    SarlOutMaps tm_out;
    const risvec_sarl_out_t& o = a.out;
    // the block's four envs x 8 vehicles = one 128-byte line per (trace, step)
    if (!tensor_map_2d(&tm_ph, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.phase, (uint64_t)E * M, T, M, kSarlTmaRows) ||
        !tensor_map_2d(&tm_ac, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.action, (uint64_t)E * 2 * V, T, 2 * V, kSarlTmaRows) ||
        !tensor_map_2d(&tm_ar, CU_TENSOR_MAP_DATA_TYPE_INT32, a.arrivals, (uint64_t)E * V, T, V, kSarlTmaRows) ||
        !tensor_map_2d(&tm_out.reward, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, o.reward, (uint64_t)E, T, 4, kSarlTmaRows) ||
        !trace_maps(tm_out.trace, {o.DataBuf, o.data_t, o.data_p, o.over_power, o.over_data, o.rate}, d, T, 4 * V))
        return RISVEC_OK;
    SarlArgs af = a;
    af.stats_slots = env->stats_slots;  // the statistics pass rides in the kernel's tail
    env->stats_folded = env->stats_slots != nullptr;
    const int KT = M == 16 ? 2 : 5;
    auto kern = KT == 2 ? k_sarl_mma_tma<2> : k_sarl_mma_tma<5>;
    kern<<<E / 4, 128, sarl_tma_smem_bytes(KT), st>>>(d, env->st, sarl_consts(env->params), af, tm_ph, tm_ac, tm_ar,
                                                       tm_out);
    *launched = true;
    return check_step_launch(env, "k_sarl_mma_tma");
}

// tensor cores, LDG (sarl_mma.cuh): one warp per env, 4 envs per block; KT k-tiles of 8 elements, M <= 8 KT
// [per-env RIS size][per-env table][fused][KT]
using SarlMmaRow = std::array<decltype(&k_sarl_mma<1>), 5>;  // over KT
template <bool FUSED, bool PE, bool NE>
SarlMmaRow sarl_mma_row() {
    return {k_sarl_mma<1, FUSED, PE, NE>, k_sarl_mma<2, FUSED, PE, NE>, k_sarl_mma<3, FUSED, PE, NE>,
            k_sarl_mma<5, FUSED, PE, NE>, k_sarl_mma<8, FUSED, PE, NE>};
}
int launch_sarl_mma(risvec_env* env, const SarlArgs& a, cudaStream_t st) {
    static const SarlMmaRow kerns[2][2][2] = {
        {{sarl_mma_row<false, false, false>(), sarl_mma_row<true, false, false>()},
         {sarl_mma_row<false, true, false>(), sarl_mma_row<true, true, false>()}},
        {{sarl_mma_row<false, false, true>(), sarl_mma_row<true, false, true>()},
         {sarl_mma_row<false, true, true>(), sarl_mma_row<true, true, true>()}}};
    const int M = env->dims.M, kt = M <= 8 ? 0 : M <= 16 ? 1 : M <= 24 ? 2 : M <= 40 ? 3 : 4;
    const auto kern = kerns[env->ris_elem != nullptr][env->env_params != nullptr][a.raw != nullptr][kt];
    kern<<<(env->dims.E + 3) / 4, 128, 0, st>>>(env->dims, env->st, env->params, a, env->env_params, env->ris_elem);
    return check_step_launch(env, "k_sarl_mma");
}

// one block per env: k_sarl_umma (tcgen05, sarl_umma.cuh) or, RISVEC_SARL_PATH=mma-sync, its mma.sync form
// k_sarl_mma_big; KQ = 2, 4, 8 for M <= 64, 128, 256
int launch_sarl_big(risvec_env* env, const SarlArgs& a, cudaStream_t st, bool umma, bool* launched) {
    const Dims& d = env->dims;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const risvec_sarl_out_t& o = a.out;
    SarlBigOutMaps tm;
    if (!trace_maps(tm.trace, {o.DataBuf, o.data_t, o.data_p, o.over_power, o.over_data, o.rate}, d, T, V))
        return RISVEC_OK;
    CUtensorMap tm_ac, tm_ar;  // k_sarl_umma: a stage's action rows [16][2 V] and arrivals [16][V] of the block's env
    const uint64_t EV = (uint64_t)E * V;
    if (umma && (!tensor_map_2d(&tm_ac, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.action, 2 * EV, T, 2 * V, 16) ||
                 (a.arrivals && !tensor_map_2d(&tm_ar, CU_TENSOR_MAP_DATA_TYPE_INT32, a.arrivals, EV, T, V, 16))))
        return RISVEC_OK;
    if (umma && !a.arrivals) tm_ar = tm_ac;  // unused: arrivals are drawn on the device
    auto go = [&](auto kq) -> int {
        constexpr int KQ = decltype(kq)::value;
        const SarlConsts c = sarl_consts(env->params);
        if (umma) {
            const int smem = sarl_umma_smem_request(KQ, V);
            CUDA_TRY(cudaFuncSetAttribute(k_sarl_umma<KQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k_sarl_umma<KQ><<<E, kUmmaThreads, smem, st>>>(d, env->st, c, a, tm, tm_ac, tm_ar);
        } else {
            const int smem = sarl_big_smem_bytes(KQ, V);
            CUDA_TRY(cudaFuncSetAttribute(k_sarl_mma_big<KQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k_sarl_mma_big<KQ><<<E, kBigThreads, smem, st>>>(d, env->st, c, a, tm);
        }
        *launched = true;
        return check_step_launch(env, umma ? "k_sarl_umma" : "k_sarl_mma_big");
    };
    return M <= 64 ? go(std::integral_constant<int, 2>{})
                   : M <= 128 ? go(std::integral_constant<int, 4>{}) : go(std::integral_constant<int, 8>{});
}

// FP32 pipe, the env's 8 lanes split the elements (MPI per lane); packed records: V == 8, M == 8 MPI
template <int MPI>
int launch_sarl_v8(risvec_env* env, const SarlArgs& a, cudaStream_t st) {
    const int warps = (env->dims.E + 3) / 4;
    const bool mfull = env->dims.M == 8 * MPI;
    const risvec_sarl_out_t& o = a.out;
    const bool full = a.arrivals && o.reward && o.DataBuf && o.data_t && o.data_p && o.over_power && o.over_data &&
                      o.rate;
    if (a.in_rec != nullptr)
        k_sarl_v8<MPI, true, true, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a);
    else if (mfull && full)
        k_sarl_v8<MPI, true, true, false><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a);
    else if (mfull)
        k_sarl_v8<MPI, true, false, false><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a);
    else
        k_sarl_v8<MPI, false, false, false><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a);
    return check_step_launch(env, "k_sarl_v8");
}

// FP32 pipe, 32 / VP envs per warp: M / WPE elements per lane, a register-resident table of MPL complex floats
template <int VP, int MPL, int WPE>
int launch_sarl_cfg(risvec_env* env, const SarlArgs& a_in, cudaStream_t st) {
    constexpr int EPW = 32 / VP;
    SarlArgs a = a_in;
    const int E = env->dims.E, V = env->dims.V;
    const int blocks = (E + EPW - 1) / EPW;
    const size_t MS = (size_t)((env->dims.M + 4 * WPE + 7) / 4) * 4;  // must match the kernel
    if constexpr (WPE == 1) {  // one warp per env group: fused step kernel
        const size_t smem = 6 * EPW * MS * sizeof(float);
        return dispatch_pe(env, [&](auto pe) {
            return dispatch_re(env, [&](auto re) {
                auto kern = k_sarl_rollout<VP, MPL, WPE, decltype(pe)::value, decltype(re)::value>;
                if (smem > 48 * 1024)
                    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                kern<<<blocks, 32 * WPE, smem, st>>>(env->dims, env->st, env->params, a, env->env_params,
                                                     env->ris_elem);
                return check_step_launch(env, "k_sarl_rollout");
            });
        });
    } else {
        // several warps per env (large M): cascade kernel over (env group, time chunk) -> |S|^2 scratch,
        // then the per-vehicle scan kernel
        if (int rc = ensure_scratch(env, (size_t)a.T * E * V * sizeof(float))) return rc;
        a.g2 = (float*)env->scratch;
        int chunk = 32;
        while (chunk > 2 && (long long)blocks * ((a.T + chunk - 1) / chunk) < 4 * 148) chunk >>= 1;  // fill the SMs
        a.t_chunk = chunk;
        const size_t smem2 = 8 * EPW * MS * sizeof(float) + 4 * WPE * 32 * sizeof(float2);
        if (int rc = dispatch_re(env, [&](auto re) {
                auto kern = k_sarl_cascade2<VP, MPL, WPE, decltype(re)::value>;
                if (smem2 > 48 * 1024)
                    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
                kern<<<dim3(blocks, (a.T + chunk - 1) / chunk), 32 * WPE, smem2, st>>>(env->dims, env->st, a,
                                                                                         env->ris_elem);
                return check_launch(env, "k_sarl_cascade2");
            }))
            return rc;
        const long long total = (long long)E * VP;
        // the scan reads the step parameters: the cascade only forms |S|^2
        if (int rc = dispatch_pe(env, [&](auto pe) {
                k_sarl_scan<VP, decltype(pe)::value><<<(int)((total + 127) / 128), 128, 0, st>>>(
                    env->dims, env->st, env->params, a, env->env_params);
                return check_launch(env, "k_sarl_scan");
            }))
            return rc;
        env->step_kernel = "k_sarl_cascade2+k_sarl_scan";
        return RISVEC_OK;
    }
}
template <int VP>
int launch_sarl_fp32(risvec_env* env, const SarlArgs& a, cudaStream_t st) {
    const int M = env->dims.M;
    if (M <= 16) return launch_sarl_cfg<VP, 16, 1>(env, a, st);
    if (M <= 40) return launch_sarl_cfg<VP, 40, 1>(env, a, st);
    if constexpr (VP >= 8) {  // M > 40 runs at VP >= 8: 32 / VP envs per warp would not fit shared memory
        if (M <= 64) return launch_sarl_cfg<VP, 32, 2>(env, a, st);
        if (M <= 128) return launch_sarl_cfg<VP, 32, 4>(env, a, st);
        if (M <= 256) return launch_sarl_cfg<VP, 32, 8>(env, a, st);
        if (M <= 512) return launch_sarl_cfg<VP, 32, 16>(env, a, st);
        if (M <= 1024) return launch_sarl_cfg<VP, 64, 16>(env, a, st);
        return fail(RISVEC_ERR_UNSUPPORTED, "M = %d > 1024 is not covered by the SARL rollout kernel", M);
    } else {  // choose_sarl sends M > 40 only with VP >= 8 (dispatch_vp<8>): not reached
        return fail(RISVEC_ERR_INVALID, "internal: M = %d > 40 with VP = %d < 8", M, VP);
    }
}

int launch_sarl(risvec_env* env, const SarlArgs& a, cudaStream_t st) {
    const int V = env->dims.V, M = env->dims.M;
    auto fp32 = [&](auto vp) { return launch_sarl_fp32<decltype(vp)::value>(env, a, st); };
    for (int from = kSarlMmaTma;;) {
        const SarlKernel k = choose_sarl(env, a, from);
        bool launched = false;
        int rc = RISVEC_OK;
        switch (k) {
            case kSarlMmaTma: rc = launch_sarl_mma_tma(env, a, st, &launched); break;
            case kSarlMma: return launch_sarl_mma(env, a, st);
            case kSarlUmma:
            case kSarlMmaBig: rc = launch_sarl_big(env, a, st, k == kSarlUmma, &launched); break;
            case kSarlV8: return M <= 16 ? launch_sarl_v8<2>(env, a, st) : launch_sarl_v8<5>(env, a, st);
            case kSarlRollout: return dispatch_vp(V, fp32);
            case kSarlCascade: return dispatch_vp<8>(V, fp32);
        }
        if (rc != RISVEC_OK || launched) return rc;
        from = k + 1;  // a tensor map could not be encoded here: the next candidate
    }
}

// ---- MARL: the rollout kernels in the order they are tried (choose_marl)
enum MarlKernel { kMarlTma, kMarlV8, kMarlRollout };

// the six bench traces + injected arrivals, no over_power
bool marl_full(const MarlArgs& a) {
    const risvec_marl_out_t& o = a.out;
    return a.arrivals && o.reward_user && o.reward && o.DataBuf && o.data_t && o.data_p && o.rate && !o.over_power;
}
// k_marl_tma covers the BASELINE shape: V = 8, E % 4 == 0, marl_full, 16-byte aligned streams, 32-bit indices
bool marl_tma_covers(const Dims& d, const MarlArgs& a) {
    const risvec_marl_out_t& o = a.out;
    return marl_full(a) && d.V == 8 && d.E % 4 == 0 && aligned16(a.action) && aligned16(a.arrivals) &&
           aligned16(o.reward_user) && aligned16(o.reward) && aligned16(o.DataBuf) && aligned16(o.data_t) &&
           aligned16(o.data_p) && aligned16(o.rate) && (uint64_t)a.T * d.E * 16 < (1ull << 31);
}
// The kernel of a MARL rollout (`a.in_rec`: packed records, `a.raw`: the fused driver step), as choose_sarl
MarlKernel choose_marl(const risvec_env* env, const MarlArgs& a, int from = kMarlTma) {
    if (a.in_rec) return kMarlV8;  // the caller checked the packed shape
    // 4 envs per warp, lane = vehicle
    const bool v8 = env->dims.V <= 8 && !env->ovr.force_generic && !a.out.stats && !a.out.last_power &&
                    (!a.raw || aligned8(a.raw));
    // an attached per-env parameter table: k_marl_tma has no PE instantiation
    if (from <= kMarlTma && v8 && !env->ovr.marl_v8 && !env->env_params && marl_tma_covers(env->dims, a))
        return kMarlTma;
    return v8 ? kMarlV8 : kMarlRollout;
}

// time-parallel, one warp per env, TMA in / out (marl_tma.cuh); dynamic + static shared memory stay under the
// 48 KB default
int launch_marl_tma(risvec_env* env, const MarlArgs& a_in, cudaStream_t st, bool* launched) {
    const Dims& d = env->dims;
    const int E = d.E, V = 8, T = a_in.T;
    const risvec_marl_out_t& o = a_in.out;
    CUtensorMap tm_ac, tm_ar;
    MarlOutMaps tm;
    if (!tensor_map_2d(&tm_ac, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a_in.action, (uint64_t)E * 2 * V, T, 2 * V, 16) ||
        !tensor_map_2d(&tm_ar, CU_TENSOR_MAP_DATA_TYPE_INT32, a_in.arrivals, (uint64_t)E * V, T, V, 16) ||
        !tensor_map_2d(&tm.reward, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, o.reward, (uint64_t)E, T, 4, 16) ||
        !trace_maps(tm.trace, {o.reward_user, o.DataBuf, o.data_t, o.data_p, o.rate}, d, T, 4 * V))
        return RISVEC_OK;
    MarlArgs a = a_in;
    a.stats_slots = env->stats_slots;  // the statistics pass rides in the kernel's tail
    env->stats_folded = env->stats_slots != nullptr;
    k_marl_tma<<<E / 4, 128, kMarlSmemBytes, st>>>(d, env->st, marl_consts(env->params), a, tm_ac, tm_ar, tm);
    *launched = true;
    return check_step_launch(env, "k_marl_tma");
}

int launch_marl_v8(risvec_env* env, const MarlArgs& a, cudaStream_t st) {
    const int warps = (env->dims.E + 3) / 4;
    const double* const ep = env->env_params;
    if (a.in_rec)  // the packed entry points refuse an attached table
        k_marl_v8<true, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, nullptr);
    else if (a.raw && ep)
        k_marl_v8<false, false, true, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, ep);
    else if (a.raw)  // action mapping in the prologue, marl_get_state of the new state in the epilogue
        k_marl_v8<false, false, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, nullptr);
    else if (marl_full(a) && ep)
        k_marl_v8<true, false, false, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, ep);
    else if (marl_full(a))
        k_marl_v8<true, false><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, nullptr);
    else if (ep)
        k_marl_v8<false, false, false, true><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, ep);
    else
        k_marl_v8<false, false><<<warps, 32, 0, st>>>(env->dims, env->st, env->params, a, nullptr);
    return check_step_launch(env, "k_marl_v8");
}

int launch_marl(risvec_env* env, const MarlArgs& a, cudaStream_t st) {
    for (int from = kMarlTma;;) {
        const MarlKernel k = choose_marl(env, a, from);
        if (k == kMarlV8) return launch_marl_v8(env, a, st);
        if (k == kMarlRollout)
            return dispatch_vp(env->dims.V, [&](auto vp) {
                constexpr int VP = decltype(vp)::value;
                const long long total = (long long)env->dims.E * VP;
                return dispatch_pe(env, [&](auto pe) {
                    k_marl_rollout<VP, decltype(pe)::value><<<(int)((total + 127) / 128), 128, 0, st>>>(
                        env->dims, env->st, env->params, a, env->env_params);
                    return check_step_launch(env, "k_marl_rollout");
                });
            });
        bool launched = false;
        const int rc = launch_marl_tma(env, a, st, &launched);
        if (rc != RISVEC_OK || launched) return rc;
        from = k + 1;  // a tensor map could not be encoded here: the next candidate
    }
}

struct Carver {
    char* base;
    size_t off;
    template <typename T>
    T* take(size_t n) {
        T* p = (T*)(base + off);
        off = align_up(off + n * sizeof(T), 256);
        return p;
    }
};

__global__ void __launch_bounds__(1024) k_shard_stats(Dims d, State s, double* out) {
    // block b sums the envs b*64 + row, + 64*gridDim.x, ... : thread (row, col) reads stats column
    // col (coalesced 64 B rows), float64 partial sums, shared-memory tree over the 64 rows, then
    // 17 float64 atomics per block into `out` (zeroed by the caller unless it accumulates)
    __shared__ double red[64][RISVEC_NSTAT + 1];
    const int col = threadIdx.x & 15, row = threadIdx.x >> 4;
    double acc = 0.0, racc = 0.0;
    for (int e = blockIdx.x * 64 + row; e < d.E; e += 64 * gridDim.x) {
        acc += (double)s.stats[(size_t)e * RISVEC_NSTAT + col];
        if (col == 0) racc += (double)s.reward[e];
    }
    red[row][col] = acc;
    if (col == 0) red[row][RISVEC_NSTAT] = racc;
    __syncthreads();
    for (int half = 32; half > 0; half >>= 1) {
        if (row < half) {
            red[row][col] += red[row + half][col];
            if (col == 0) red[row][RISVEC_NSTAT] += red[row + half][RISVEC_NSTAT];
        }
        __syncthreads();
    }
    if (threadIdx.x <= RISVEC_NSTAT) atomicAdd(out + threadIdx.x, red[0][threadIdx.x]);
}

int launch_make_new_game(risvec_env* env, const uint8_t* env_mask, const int32_t* reset_ints, int n_ints,
                         const int32_t* reset_dirs, int n_dirs, EnvGate g, void* stream);
int launch_renew_positions(risvec_env* env, const double* uniforms, int n, int32_t* used_out, EnvGate g, void* stream);
int launch_compute_parms(risvec_env* env, EnvGate g, void* stream);
int launch_bcd(risvec_env* env, EnvGate g, void* stream);
int launch_gains(risvec_env* env, const double* chan_rand, const double* chan_normal, const double* chan_exp, EnvGate g,
                 void* stream);
int launch_pair_reset(risvec_env* env, const uint8_t* env_mask, EnvGate g, void* stream);

}  // namespace

// ======================================================================================
extern "C" {

int risvec_abi_version(void) { return RISVEC_ABI_VERSION; }
const char* risvec_last_error(void) { return g_err; }

int risvec_default_params(int variant, risvec_params_t* p) {
    if (!p) return fail(RISVEC_ERR_INVALID, "params is NULL");
    memset(p, 0, sizeof(*p));
    // lane constants of the drivers (marl_train_bcd.py:446-449, ddpg_train.py:17-20)
    const double up[4] = {(400 + 3.5 / 2) / 2.0, (400 + 3.5 + 3.5 / 2) / 2.0, (800 + 3.5 / 2) / 2.0,
                          (800 + 3.5 + 3.5 / 2) / 2.0};
    const double down[4] = {(400 - 3.5 - 3.5 / 2) / 2.0, (400 - 3.5 / 2) / 2.0, (800 - 3.5 - 3.5 / 2) / 2.0,
                            (800 - 3.5 / 2) / 2.0};
    p->n_up = p->n_down = p->n_left = p->n_right = 4;
    for (int i = 0; i < 4; ++i) {
        p->up_lanes[i] = up[i]; p->left_lanes[i] = up[i];
        p->down_lanes[i] = down[i]; p->right_lanes[i] = down[i];
    }
    p->width = 400; p->height = 400;
    p->time_slow = 0.1; p->time_fast = 0.001; p->bandwidth = 1.0; p->k = 1e-28; p->L = 500.0; p->rate = 3.0;
    p->data_buf_size = 10;
    p->channel_model = RISVEC_CHANNEL_FREE;
    p->noise_power = pow(10.0, (-174.0 - 30.0) / 10.0) * 1.0e6;  // MARL:74-76
    p->P_max = 1.0; p->power_scale = 0.7; p->f_local_max = 1.0e9; p->f_edge_max = 2.0e9; p->cycles_per_bit = 500.0;
    p->cpu_share_floor = 0.10; p->w_d = 0.5; p->w_e = 3.0; p->R_min_bpsHz = 0.20; p->D_max_s = 0.10;
    p->qos_penalty = 5.0; p->reward_clip = 50.0; p->qos_enable = 1;
    p->fc_GHz = 3.5; p->shadow_std_los = 4.0; p->shadow_std_nlos = 7.0; p->rician_K_dB = 0.0; p->veh_ant_gain = 3.0;
    p->t_factor1 = 1.0; p->t_factor2 = 0.6; p->penalty1 = 2.0; p->penalty2 = 2.0;
    (void)variant;
    return RISVEC_OK;
}

int risvec_create(const risvec_params_t* params, int variant, int E, int V, int M, int control_bit, int device,
                  uint64_t seed, int64_t env_index_base, risvec_env_t** out) {
    if (!out) return fail(RISVEC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!params) return fail(RISVEC_ERR_INVALID, "params is NULL");
    if (variant != RISVEC_VARIANT_MARL && variant != RISVEC_VARIANT_SARL)
        return fail(RISVEC_ERR_INVALID, "unknown variant %d", variant);
    if (E < 1 || V < 1 || M < 1) return fail(RISVEC_ERR_INVALID, "E, V, M must be >= 1 (got %d, %d, %d)", E, V, M);
    if (control_bit < 0 || control_bit > 10) return fail(RISVEC_ERR_INVALID, "control_bit must be in [0, 10]");
    if (V > 32) return fail(RISVEC_ERR_UNSUPPORTED, "V = %d > 32 vehicles per env is not covered by the kernels", V);
    if (M > 1024) return fail(RISVEC_ERR_UNSUPPORTED, "M = %d > 1024 RIS elements is not covered by the kernels", M);
    if (int rc = validate_params(params)) return rc;

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        return fail(RISVEC_ERR_NODEVICE, "no CUDA device visible: this library has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(RISVEC_ERR_INVALID, "device %d out of range [0, %d)", device, ndev);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(RISVEC_ERR_NODEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device,
                    prop.major, prop.minor);
    ENTER_DEVICE(device);

    risvec_env* env = new (std::nothrow) risvec_env();
    if (!env) return fail(RISVEC_ERR_INVALID, "out of host memory");
    memset(env, 0, sizeof(*env));
    env->device = device;
    env->params = *params;
    env->ovr = read_overrides();
    env->step_kernel = "";
    Dims& d = env->dims;
    d.E = E; d.V = V; d.M = M; d.ncand = 1 << control_bit; d.variant = variant;
    d.seed = seed; d.env_base = env_index_base;
    d.dist_BR = sqrt((kBsX - kRisX) * (kBsX - kRisX) + (kBsY - kRisY) * (kBsY - kRisY) + (kBsZ - kRisZ) * (kBsZ - kRisZ));
    d.angle_BR = (kRisX - kBsX) / d.dist_BR;  // MARL:175-177

    struct Spec { int f; int64_t rows, cols; int eb, fl; };
    const Spec specs[RISVEC_F_COUNT] = {
        {RISVEC_F_POS_X, E, V, 8, 1}, {RISVEC_F_POS_Y, E, V, 8, 1}, {RISVEC_F_DIR, E, V, 4, 0},
        {RISVEC_F_VEL, E, V, 4, 0}, {RISVEC_F_DIST, E, V, 8, 1}, {RISVEC_F_ANGLE, E, V, 8, 1},
        {RISVEC_F_AMP, E, V, 8, 1}, {RISVEC_F_THETA_RE, E, M, 8, 1}, {RISVEC_F_THETA_IM, E, M, 8, 1},
        {RISVEC_F_PHASE_REAL, E, M, 4, 1}, {RISVEC_F_GAINS, E, V, 8, 1}, {RISVEC_F_DATABUF, E, V, 8, 1},
        {RISVEC_F_DATA_T, E, V, 4, 1}, {RISVEC_F_DATA_P, E, V, 4, 1}, {RISVEC_F_OVER_DATA, E, V, 4, 1},
        {RISVEC_F_OVER_POWER, E, V, 4, 1}, {RISVEC_F_RATE, E, V, 4, 1}, {RISVEC_F_DATA_R, E, V, 4, 0},
        {RISVEC_F_REWARD_USER, E, V, 4, 1}, {RISVEC_F_REWARD, E, 1, 4, 1}, {RISVEC_F_MECQ, E, 1, 8, 1},
        {RISVEC_F_STATS, E, RISVEC_NSTAT, 4, 1}, {RISVEC_F_LAST_POWER, E, 2 * V, 4, 1},
        {RISVEC_F_STEP_CTR, E, 1, 8, 0},
        {RISVEC_F_V2I_SHADOWING, E, V, 8, 1},
        {RISVEC_F_PAIR_HIST, E, V * V, 4, 1}, {RISVEC_F_PAIR_STREAK, E, V, 4, 0}, {RISVEC_F_PAIR_TAU, E, 1, 8, 1},
        {RISVEC_F_PAIR_K, E, 1, 4, 0}, {RISVEC_F_PAIR_MASK, E, V * V, 1, 0}, {RISVEC_F_PAIR_ROUNDS, E, 1, 4, 0},
        {RISVEC_F_NOMA_PARTNER, E, V, 4, 0}, {RISVEC_F_NOMA_NGROUPS, E, 1, 4, 0}, {RISVEC_F_NOMA_PAIRS, E, V, 4, 0},
        {RISVEC_F_NOMA_NPAIRS, E, 1, 4, 0},
        {RISVEC_F_EP_STEP, E, 1, 4, 0}, {RISVEC_F_EP_INDEX, E, 1, 4, 0}};
    size_t off = 0;
    for (int i = 0; i < RISVEC_F_COUNT; ++i) {
        const Spec& sp = specs[i];
        env->fields[sp.f] = {off, sp.rows, sp.cols, sp.eb, sp.fl};
        off = align_up(off + (size_t)sp.rows * sp.cols * sp.eb, 256);
    }
    const size_t ep_bits_off = off;  // hand-over of the episode clock to the per-stage kernels (not a field)
    off = align_up(off + (size_t)E, 256);
    const size_t ep_keys_off = off;
    off = align_up(off + (size_t)E * 4, 256);
    env->arena_bytes = off;
    cudaError_t ce = cudaMalloc((void**)&env->arena, env->arena_bytes);
    if (ce != cudaSuccess) {
        delete env;
        return fail(RISVEC_ERR_CUDA, "cudaMalloc(%zu bytes of env state): %s", off, cudaGetErrorString(ce));
    }
    ce = cudaMemset(env->arena, 0, env->arena_bytes);  // Environ.__init__ zero-fills everything
    if (ce != cudaSuccess) {
        cudaFree(env->arena);
        delete env;
        return fail(RISVEC_ERR_CUDA, "cudaMemset: %s", cudaGetErrorString(ce));
    }
    bind_state(env);
    env->ep_bits = (unsigned char*)(env->arena + ep_bits_off);
    env->ep_keys = (int*)(env->arena + ep_keys_off);
    *out = env;
    return RISVEC_OK;
}

int risvec_destroy(risvec_env_t* env) {
    if (!env) return RISVEC_OK;
    DeviceGuard _dev_guard(env->device);
    if (env->arena) cudaFree(env->arena);
    if (env->stage) cudaFree(env->stage);
    if (env->scratch) cudaFree(env->scratch);
    if (env->pipe_ready) {
        cudaStreamDestroy(env->s_in);
        cudaStreamDestroy(env->s_out);
        for (cudaEvent_t e : env->ev) cudaEventDestroy(e);
    }
    delete env;
    return RISVEC_OK;
}

int risvec_set_params(risvec_env_t* env, const risvec_params_t* params) {
    if (!env || !params) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (int rc = validate_params(params)) return rc;
    env->params = *params;
    return RISVEC_OK;
}

int risvec_get_params(const risvec_env_t* env, risvec_params_t* out) {
    if (!env || !out) return fail(RISVEC_ERR_INVALID, "NULL argument");
    *out = env->params;
    return RISVEC_OK;
}

int risvec_field(risvec_env_t* env, int field, void** dev_ptr, int64_t* rows, int64_t* cols, int* elem_bytes,
                 int* is_float) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (field < 0 || field >= RISVEC_F_COUNT) return fail(RISVEC_ERR_INVALID, "unknown field %d", field);
    const FieldDesc& f = env->fields[field];
    if (dev_ptr) *dev_ptr = env->arena + f.offset;
    if (rows) *rows = f.rows;
    if (cols) *cols = f.cols;
    if (elem_bytes) *elem_bytes = f.elem_bytes;
    if (is_float) *is_float = f.is_float;
    return RISVEC_OK;
}

int risvec_make_new_game(risvec_env_t* env, const int32_t* reset_ints, int n_ints, const int32_t* reset_dirs,
                         int n_dirs, void* stream) {
    return risvec_make_new_game_masked(env, nullptr, reset_ints, n_ints, reset_dirs, n_dirs, stream);
}

int risvec_make_new_game_masked(risvec_env_t* env, const uint8_t* env_mask, const int32_t* reset_ints, int n_ints,
                                const int32_t* reset_dirs, int n_dirs, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    const int V = env->dims.V;
    const int need = 9 * (V / 4) + 3 * (V % 4) + 1;
    if (reset_ints != nullptr && n_ints < need)
        return fail(RISVEC_ERR_INVALID, "reset_ints needs %d draws per env for V = %d (got %d)", need, V, n_ints);
    if (reset_ints != nullptr && (V % 4) != 0 && (reset_dirs == nullptr || n_dirs < V % 4))
        return fail(RISVEC_ERR_INVALID, "reset_dirs needs %d headings per env", V % 4);
    if (reset_ints == nullptr && reset_dirs != nullptr)
        return fail(RISVEC_ERR_INVALID, "reset_dirs given without reset_ints");
    ENTER_DEVICE(env->device);
    return launch_make_new_game(env, env_mask, reset_ints, n_ints, reset_dirs, n_dirs, EnvGate{}, stream);
}

int risvec_renew_positions(risvec_env_t* env, const double* uniforms, int n, int32_t* used_out, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (uniforms != nullptr && n < 1) return fail(RISVEC_ERR_INVALID, "uniforms given with n = %d", n);
    ENTER_DEVICE(env->device);
    return launch_renew_positions(env, uniforms, n, used_out, EnvGate{}, stream);
}

int risvec_compute_parms(risvec_env_t* env, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    ENTER_DEVICE(env->device);
    return launch_compute_parms(env, EnvGate{}, stream);
}

int risvec_set_phase(risvec_env_t* env, const float* phase, void* stream) {
    if (!env || !phase) return fail(RISVEC_ERR_INVALID, "NULL argument");
    ENTER_DEVICE(env->device);
    const long long n = (long long)env->dims.E * env->dims.M;
    const int threads = 256, blocks = (int)((n + threads - 1) / threads);
    k_set_phase<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, phase);
    return check_launch(env, "k_set_phase");
}

int risvec_optimize_phase_shift(risvec_env_t* env, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    ENTER_DEVICE(env->device);
    return launch_bcd(env, EnvGate{}, stream);
}

int risvec_update_channel_gains(risvec_env_t* env, const double* chan_rand, const double* chan_normal,
                                const double* chan_exp, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    const bool any = chan_rand || chan_normal || chan_exp;
    if (env->params.channel_model != RISVEC_CHANNEL_FREE && any && !(chan_rand && chan_normal && chan_exp))
        return fail(RISVEC_ERR_INVALID, "chan_rand, chan_normal and chan_exp must be given together");
    ENTER_DEVICE(env->device);
    return launch_gains(env, chan_rand, chan_normal, chan_exp, EnvGate{}, stream);
}

}  // extern "C"

namespace {
// The per-stage launches behind the plain entry points; `g` restricts them to some envs (the episode-start calls
// on the shapes k_begin_episode does not take).  A zero gate is exactly the plain entry point.
int launch_make_new_game(risvec_env* env, const uint8_t* env_mask, const int32_t* reset_ints, int n_ints,
                         const int32_t* reset_dirs, int n_dirs, EnvGate g, void* stream) {
    const int threads = 128, blocks = (env->dims.E + threads - 1) / threads;
    const unsigned long long call = g.call ? 0 : env->reset_calls++;
    k_make_new_game<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, env->params, reset_ints, n_ints,
                                                                  reset_dirs, n_dirs, call, env_mask, g);
    return check_launch(env, "k_make_new_game");
}
int launch_renew_positions(risvec_env* env, const double* uniforms, int n, int32_t* used_out, EnvGate g, void* stream) {
    const int threads = 128, blocks = (env->dims.E + threads - 1) / threads;
    const unsigned long long call = g.call ? 0 : env->mob_calls++;
    k_renew_positions<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, env->params, uniforms, n,
                                                                    used_out, call, g);
    return check_launch(env, "k_renew_positions");
}
int launch_compute_parms(risvec_env* env, EnvGate g, void* stream) {
    const long long n = (long long)env->dims.E * env->dims.V;
    const int threads = 256, blocks = (int)((n + threads - 1) / threads);
    k_compute_parms<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, g);
    return check_launch(env, "k_compute_parms");
}
int launch_bcd(risvec_env* env, EnvGate g, void* stream) {
    return dispatch_re(env, [&](auto re) {
        constexpr bool NE = decltype(re)::value;
        if (env->dims.ncand <= 8 && env->dims.V <= 8 && env->dims.M <= 256 && !env->ovr.force_generic) {
            // 4 envs per warp, lane = (env, candidate)
            const int wpb = env->dims.M <= 64 ? 4 : 1;
            const int blocks = (env->dims.E + 4 * wpb - 1) / (4 * wpb);
            const size_t smem = (size_t)wpb * 4 * 2 * env->dims.M * sizeof(double2);
            if (smem > 48 * 1024)
                CUDA_TRY(cudaFuncSetAttribute(k_bcd_v8<NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_bcd_v8<NE><<<blocks, 32 * wpb, smem, (cudaStream_t)stream>>>(env->dims, env->st, g, env->ris_elem);
            return check_launch(env, "k_bcd_v8");
        }
        const int wpb = 4, threads = 32 * wpb, blocks = (env->dims.E + wpb - 1) / wpb;
        const size_t smem = (size_t)wpb * 2 * env->dims.M * sizeof(double2);
        if (smem > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(k_bcd<NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_bcd<NE><<<blocks, threads, smem, (cudaStream_t)stream>>>(env->dims, env->st, g, env->ris_elem);
        return check_launch(env, "k_bcd");
    });
}
int launch_gains(risvec_env* env, const double* chan_rand, const double* chan_normal, const double* chan_exp, EnvGate g,
                 void* stream) {
    if (env->params.channel_model == RISVEC_CHANNEL_FREE)
        return dispatch_re(env, [&](auto re) {
            constexpr bool NE = decltype(re)::value;
            if (!env->ovr.force_generic)  // lane = (env, vehicle), sequential over the elements
                return dispatch_vp(env->dims.V, [&](auto vp) {
                    constexpr int VP = decltype(vp)::value;
                    const long long n = (long long)env->dims.E * VP;
                    const int threads = 128, blocks = (int)((n + threads - 1) / threads);
                    k_gains_free_v<VP, NE><<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, g,
                                                                                          env->ris_elem);
                    return check_launch(env, "k_gains_free_v");
                });
            const int wpb = 4, threads = 32 * wpb, blocks = (env->dims.E + wpb - 1) / wpb;
            k_gains_free<NE><<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, g, env->ris_elem);
            return check_launch(env, "k_gains_free");
        });
    // the 3GPP branch has no RIS term: it takes no per-env RIS size
    const long long n = (long long)env->dims.E * env->dims.V;
    const int threads = 128, blocks = (int)((n + threads - 1) / threads);
    const unsigned long long call = g.call ? 0 : env->chan_calls++;
    k_gains_3gpp<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, env->st, env->params, chan_rand, chan_normal,
                                                               chan_exp, call, g);
    return check_launch(env, "k_gains_3gpp");
}

// Argument checks shared by each rollout entry point and its `_host` form: both refuse the same input with the same
// message, and the `_host` form does so before it enqueues a copy.
int check_marl_args(const risvec_env* env, int T, const void* action, const void* partner, const void* ngroups) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_MARL) return fail(RISVEC_ERR_INVALID, "handle is not a MARL env");
    if (T < 1) return fail(RISVEC_ERR_INVALID, "T must be >= 1 (got %d)", T);
    if (!action || !partner || !ngroups) return fail(RISVEC_ERR_INVALID, "action, partner and ngroups are required");
    return RISVEC_OK;
}
int check_sarl_args(const risvec_env* env, int T, const void* action, const void* phase) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_SARL) return fail(RISVEC_ERR_INVALID, "handle is not a SARL env");
    if (T < 1) return fail(RISVEC_ERR_INVALID, "T must be >= 1 (got %d)", T);
    if (!action || !phase) return fail(RISVEC_ERR_INVALID, "action and phase are required");
    return RISVEC_OK;
}
// ---- packed record layout (include/risvec.h): one input / one output stream per rollout
const char kPackedEnvParamsMsg[] =
    "packed records take no per-env parameter table: a table is attached (risvec_attach_env_params); detach it or use "
    "the per-array entry points";
int check_sarl_packed_args(const risvec_env* env, int T, const void* in_rec, const void* out_rec, const void* reward) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_SARL) return fail(RISVEC_ERR_INVALID, "handle is not a SARL env");
    if (T < 1 || !in_rec || !out_rec || !reward) return fail(RISVEC_ERR_INVALID, "T >= 1 and all three buffers are required");
    if (env->dims.V != 8 || env->dims.E % 4 != 0 || (env->dims.M != 16 && env->dims.M != 40))
        return fail(RISVEC_ERR_UNSUPPORTED, "packed SARL records need V == 8, E %% 4 == 0 and M in {16, 40} "
                    "(got V = %d, E = %d, M = %d)", env->dims.V, env->dims.E, env->dims.M);
    if (env->env_params) return fail(RISVEC_ERR_UNSUPPORTED, "%s", kPackedEnvParamsMsg);
    if (env->ris_elem)
        return fail(RISVEC_ERR_UNSUPPORTED, "packed SARL records take no per-env RIS size: one is attached "
                    "(risvec_attach_ris_elements); detach it or use the per-array entry points");
    return RISVEC_OK;
}
int check_marl_packed_args(const risvec_env* env, int T, const void* in_rec, const void* partner, const void* ngroups,
                           const void* out_rec, const void* reward) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_MARL) return fail(RISVEC_ERR_INVALID, "handle is not a MARL env");
    if (T < 1 || !in_rec || !partner || !ngroups || !out_rec || !reward)
        return fail(RISVEC_ERR_INVALID, "T >= 1 and all buffers are required");
    if (env->dims.V != 8 || env->dims.E % 4 != 0)
        return fail(RISVEC_ERR_UNSUPPORTED, "packed MARL records need V == 8 and E %% 4 == 0 (got V = %d, E = %d)",
                    env->dims.V, env->dims.E);
    if (env->env_params) return fail(RISVEC_ERR_UNSUPPORTED, "%s", kPackedEnvParamsMsg);
    return RISVEC_OK;
}
}  // namespace

extern "C" {

// statistics accumulator attached: kernels that fold the statistics pass set env->stats_folded, every other kernel
// is followed by k_shard_stats into slot 0
static int rollout_marl_impl(risvec_env_t* env, int T, const float* action, const int32_t* partner, const int32_t* ngroups,
                             const int32_t* arrivals, const risvec_marl_out_t* out, void* stream);
static int rollout_sarl_impl(risvec_env_t* env, int T, const float* action, const float* phase, const int32_t* arrivals,
                             const risvec_sarl_out_t* out, void* stream);
static int finish_rollout(risvec_env_t* env, int rc, void* stream) {
    if (rc == RISVEC_OK && env->stats_slots != nullptr && !env->stats_folded) rc = risvec_shard_stats(env, env->stats_slots, 1, stream);
    return rc;
}
int risvec_rollout_marl(risvec_env_t* env, int T, const float* action, const int32_t* partner, const int32_t* ngroups,
                        const int32_t* arrivals, const risvec_marl_out_t* out, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    env->stats_folded = 0;
    return finish_rollout(env, rollout_marl_impl(env, T, action, partner, ngroups, arrivals, out, stream), stream);
}
int risvec_rollout_sarl(risvec_env_t* env, int T, const float* action, const float* phase, const int32_t* arrivals,
                        const risvec_sarl_out_t* out, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    env->stats_folded = 0;
    return finish_rollout(env, rollout_sarl_impl(env, T, action, phase, arrivals, out, stream), stream);
}

static int rollout_marl_impl(risvec_env_t* env, int T, const float* action, const int32_t* partner, const int32_t* ngroups,
                             const int32_t* arrivals, const risvec_marl_out_t* out, void* stream) {
    if (int rc = check_marl_args(env, T, action, partner, ngroups)) return rc;
    ENTER_DEVICE(env->device);
    MarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = T; a.action = action; a.partner = partner; a.ngroups = ngroups; a.arrivals = arrivals;
    if (out) a.out = *out;
    return launch_marl(env, a, (cudaStream_t)stream);
}

static int rollout_sarl_impl(risvec_env_t* env, int T, const float* action, const float* phase, const int32_t* arrivals,
                             const risvec_sarl_out_t* out, void* stream) {
    if (int rc = check_sarl_args(env, T, action, phase)) return rc;
    ENTER_DEVICE(env->device);
    SarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = T; a.action = action; a.phase = phase; a.arrivals = arrivals;
    if (out) a.out = *out;
    return launch_sarl(env, a, (cudaStream_t)stream);
}

int risvec_rollout_sarl_packed(risvec_env_t* env, int T, const void* in_rec, float* out_rec, float* reward,
                               void* stream) {
    if (int rc = check_sarl_packed_args(env, T, in_rec, out_rec, reward)) return rc;
    ENTER_DEVICE(env->device);
    SarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = T; a.in_rec = (const float*)in_rec; a.out_rec = out_rec; a.out.reward = reward;
    return launch_sarl(env, a, (cudaStream_t)stream);
}

int risvec_rollout_marl_packed(risvec_env_t* env, int T, const void* in_rec, const int32_t* partner,
                               const int32_t* ngroups, float* out_rec, float* reward, void* stream) {
    if (int rc = check_marl_packed_args(env, T, in_rec, partner, ngroups, out_rec, reward)) return rc;
    ENTER_DEVICE(env->device);
    MarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = T; a.in_rec = (const float*)in_rec; a.partner = partner; a.ngroups = ngroups; a.out_rec = out_rec;
    a.out.reward = reward;
    return launch_marl(env, a, (cudaStream_t)stream);
}

}  // extern "C"

// ---- host-buffer variants.  The T steps are cut into chunks and pipelined over three streams:
// chunk c+1 is copied in (H2D engine) while chunk c computes on the caller's stream and
// chunk c-1 is copied out (D2H engine), so the call runs at PCIe speed of the larger direction.
namespace {

constexpr int kMaxChunks = 64;

int ensure_pipe(risvec_env* env) {
    if (env->pipe_ready) return RISVEC_OK;
    CUDA_TRY(cudaStreamCreateWithFlags(&env->s_in, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&env->s_out, cudaStreamNonBlocking));
    for (cudaEvent_t& e : env->ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    env->pipe_ready = 1;
    return RISVEC_OK;
}

int chunk_steps(int T, size_t in_bytes_per_step) {
    // ~RISVEC_HOST_CHUNK_MB (default 24) MB of input per chunk, at most kMaxChunks chunks
    static const int mb = [] { const char* v = getenv("RISVEC_HOST_CHUNK_MB"); int m = v ? atoi(v) : 24; return m < 1 ? 1 : m; }();
    size_t per = (size_t)mb << 20;
    int tc = (int)(per / (in_bytes_per_step ? in_bytes_per_step : 1));
    if (tc < 1) tc = 1;
    int n = (T + tc - 1) / tc;
    if (n > kMaxChunks) n = kMaxChunks;
    int steps = (T + n - 1) / n;
    // chunks start on 16-step boundaries: the stage tiling of the time-parallel kernels (k_sarl_mma_tma,
    // k_marl_tma) is then the same as in one device launch over all T steps, and so is every result bit
    if (steps > 16) steps = (steps + 15) / 16 * 16;
    return steps;
}

enum HostDir { kIn, kOnce, kOut };  // step-major input | step-independent input | step-major output

// One host array of a `_host` rollout.  A NULL `host` is an array the caller did not pass (an output it does not
// want, arrivals drawn on the device): it gets no staging, and the launch sees a NULL device pointer.
struct HostBuf {
    HostDir dir;
    const void* host;  // an output's is the caller's writable array
    size_t bytes;      // per step; kOnce: in all
    size_t total(int T) const { return dir == kOnce ? bytes : bytes * (size_t)T; }
};

cudaError_t join(cudaStream_t to, cudaStream_t from, cudaEvent_t ev) {  // `to` waits for all work queued on `from`
    const cudaError_t e = cudaEventRecord(ev, from);
    return e != cudaSuccess ? e : cudaStreamWaitEvent(to, ev, 0);
}

// The pipeline of every `_host` entry point.  The staging holds each array in `b` whole.  The kOnce inputs go first,
// then the kIn inputs chunk by chunk, all on s_in; each chunk then runs `launch(tn, d)` on `stream`, where d[i] is
// the device copy of b[i] at the chunk's first step, and its kOut outputs are copied back on s_out.
// `chunk_bytes_per_step` sets the chunk length (chunk_steps).
template <size_t N, typename Launch>
int host_pipeline(risvec_env* env, int T, size_t chunk_bytes_per_step, const HostBuf (&b)[N], void* stream,
                  Launch launch) {
    if (int rc = ensure_pipe(env)) return rc;
    size_t need = 0;
    for (const HostBuf& x : b)
        if (x.host) need += align_up(x.total(T), 256);
    if (int rc = ensure_stage(env, need)) return rc;
    Carver c{env->stage, 0};
    char* dev[N];
    for (size_t i = 0; i < N; ++i) dev[i] = b[i].host ? c.take<char>(b[i].total(T)) : nullptr;

    cudaStream_t st = (cudaStream_t)stream, si = env->s_in, so = env->s_out;
    cudaEvent_t* ev_in = env->ev;
    cudaEvent_t* ev_k = env->ev + kMaxChunks;
    cudaEvent_t ev_start = env->ev[2 * kMaxChunks], ev_done = env->ev[2 * kMaxChunks + 1];
    cudaEvent_t ev_in_done = env->ev[2 * kMaxChunks + 2];
    CUDA_TRY(cudaEventRecord(ev_start, st));  // staging may still be read by earlier work on `stream`
    CUDA_TRY(cudaStreamWaitEvent(si, ev_start, 0));
    CUDA_TRY(cudaStreamWaitEvent(so, ev_start, 0));
    const int Tc = chunk_steps(T, chunk_bytes_per_step);
    const int rc = [&]() -> int {
        for (size_t i = 0; i < N; ++i)
            if (b[i].dir == kOnce && b[i].host)
                CUDA_TRY(cudaMemcpyAsync(dev[i], b[i].host, b[i].bytes, cudaMemcpyHostToDevice, si));
        for (int t0 = 0, ci = 0; t0 < T; t0 += Tc, ++ci) {
            const size_t tn = std::min(Tc, T - t0);
            for (size_t i = 0; i < N; ++i)
                if (b[i].dir == kIn && b[i].host)
                    CUDA_TRY(cudaMemcpyAsync(dev[i] + t0 * b[i].bytes, (const char*)b[i].host + t0 * b[i].bytes,
                                             tn * b[i].bytes, cudaMemcpyHostToDevice, si));
            CUDA_TRY(cudaEventRecord(ev_in[ci], si));
        }
        for (int t0 = 0, ci = 0; t0 < T; t0 += Tc, ++ci) {
            const int tn = std::min(Tc, T - t0);
            void* d[N];
            for (size_t i = 0; i < N; ++i) d[i] = dev[i] && b[i].dir != kOnce ? dev[i] + (size_t)t0 * b[i].bytes : dev[i];
            CUDA_TRY(cudaStreamWaitEvent(st, ev_in[ci], 0));
            double* const slots = env->stats_slots;
            if (t0 + tn < T) env->stats_slots = nullptr;  // the statistics are those of the rollout's last step
            const int rc = launch(tn, d);
            env->stats_slots = slots;
            if (rc) return rc;
            CUDA_TRY(cudaEventRecord(ev_k[ci], st));
            CUDA_TRY(cudaStreamWaitEvent(so, ev_k[ci], 0));
            for (size_t i = 0; i < N; ++i)
                if (b[i].dir == kOut && b[i].host)
                    CUDA_TRY(cudaMemcpyAsync((char*)b[i].host + t0 * b[i].bytes, d[i], tn * b[i].bytes,
                                             cudaMemcpyDeviceToHost, so));
        }
        return RISVEC_OK;
    }();
    // every exit, a failed chunk's too, joins both copy streams into `stream`: the caller only has to synchronise
    // `stream`, and the next call cannot overwrite the staging under copies still queued here
    const cudaError_t ji = join(st, si, ev_in_done), jo = join(st, so, ev_done);
    if (rc != RISVEC_OK) return rc;
    if (ji != cudaSuccess || jo != cudaSuccess)
        return fail(RISVEC_ERR_CUDA, "joining the copy streams: %s", cudaGetErrorString(ji != cudaSuccess ? ji : jo));
    return RISVEC_OK;
}

}  // namespace

extern "C" {

int risvec_rollout_marl_host(risvec_env_t* env, int T, const float* action, const int32_t* partner,
                             const int32_t* ngroups, const int32_t* arrivals, const risvec_marl_out_t* out,
                             void* stream) {
    if (int rc = check_marl_args(env, T, action, partner, ngroups)) return rc;
    ENTER_DEVICE(env->device);
    const size_t E = env->dims.E, ev = E * env->dims.V * 4;  // ev: bytes of one step of an [T,E,V] array
    const risvec_marl_out_t h = out ? *out : risvec_marl_out_t{};
    const HostBuf b[] = {{kIn, action, 2 * ev}, {kIn, arrivals, ev}, {kOnce, partner, ev}, {kOnce, ngroups, E * 4},
                         {kOut, h.reward_user, ev}, {kOut, h.reward, E * 4}, {kOut, h.DataBuf, ev}, {kOut, h.data_t, ev},
                         {kOut, h.data_p, ev}, {kOut, h.rate, ev}, {kOut, h.over_power, ev},
                         {kOut, h.stats, E * RISVEC_NSTAT * 4}, {kOut, h.last_power, 2 * ev}};
    // the chunk length counts the arrivals whether or not they are passed
    return host_pipeline(env, T, 3 * ev, b, stream, [&](int tn, void* const* d) {
        const risvec_marl_out_t o = {(float*)d[4], (float*)d[5], (float*)d[6], (float*)d[7], (float*)d[8],
                                     (float*)d[9], (float*)d[10], (float*)d[11], (float*)d[12]};
        return risvec_rollout_marl(env, tn, (float*)d[0], (int32_t*)d[2], (int32_t*)d[3], (int32_t*)d[1], &o, stream);
    });
}

int risvec_rollout_sarl_host(risvec_env_t* env, int T, const float* action, const float* phase,
                             const int32_t* arrivals, const risvec_sarl_out_t* out, void* stream) {
    if (int rc = check_sarl_args(env, T, action, phase)) return rc;
    ENTER_DEVICE(env->device);
    const size_t E = env->dims.E, ev = E * env->dims.V * 4, em = E * env->dims.M * 4;
    const risvec_sarl_out_t h = out ? *out : risvec_sarl_out_t{};
    const HostBuf b[] = {{kIn, action, 2 * ev}, {kIn, phase, em}, {kIn, arrivals, ev}, {kOut, h.reward, E * 4},
                         {kOut, h.DataBuf, ev}, {kOut, h.data_t, ev}, {kOut, h.data_p, ev}, {kOut, h.over_power, ev},
                         {kOut, h.over_data, ev}, {kOut, h.rate, ev}};
    // the chunk length counts the arrivals whether or not they are passed
    return host_pipeline(env, T, 3 * ev + em, b, stream, [&](int tn, void* const* d) {
        const risvec_sarl_out_t o = {(float*)d[3], (float*)d[4], (float*)d[5], (float*)d[6],
                                     (float*)d[7], (float*)d[8], (float*)d[9]};
        return risvec_rollout_sarl(env, tn, (float*)d[0], (float*)d[1], (int32_t*)d[2], &o, stream);
    });
}

int risvec_rollout_sarl_packed_host(risvec_env_t* env, int T, const void* in_rec, float* out_rec, float* reward,
                                    void* stream) {
    if (int rc = check_sarl_packed_args(env, T, in_rec, out_rec, reward)) return rc;
    ENTER_DEVICE(env->device);
    const size_t E = env->dims.E, in = E * RISVEC_SARL_IN_WORDS(env->dims.M) * 4;
    const HostBuf b[] = {{kIn, in_rec, in}, {kOut, out_rec, E * RISVEC_SARL_OUT_WORDS * 4}, {kOut, reward, E * 4}};
    return host_pipeline(env, T, in, b, stream, [&](int tn, void* const* d) {
        return risvec_rollout_sarl_packed(env, tn, d[0], (float*)d[1], (float*)d[2], stream);
    });
}

int risvec_rollout_marl_packed_host(risvec_env_t* env, int T, const void* in_rec, const int32_t* partner,
                                    const int32_t* ngroups, float* out_rec, float* reward, void* stream) {
    if (int rc = check_marl_packed_args(env, T, in_rec, partner, ngroups, out_rec, reward)) return rc;
    ENTER_DEVICE(env->device);
    const size_t E = env->dims.E, in = E * RISVEC_MARL_IN_WORDS * 4;
    const HostBuf b[] = {{kIn, in_rec, in}, {kOnce, partner, E * 8 * 4}, {kOnce, ngroups, E * 4},
                         {kOut, out_rec, E * RISVEC_MARL_OUT_WORDS * 4}, {kOut, reward, E * 4}};
    return host_pipeline(env, T, in, b, stream, [&](int tn, void* const* d) {
        return risvec_rollout_marl_packed(env, tn, d[0], (int32_t*)d[1], (int32_t*)d[2], (float*)d[3], (float*)d[4],
                                          stream);
    });
}

int risvec_observe(risvec_env_t* env, float* obs, void* stream) {
    if (!env || !obs) return fail(RISVEC_ERR_INVALID, "NULL argument");
    ENTER_DEVICE(env->device);
    const int n_theta = env->dims.variant == RISVEC_VARIANT_SARL ? env->dims.M / env->dims.V : 0;
    const long long n = (long long)env->dims.E * env->dims.V;
    k_observe<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(env->dims, env->st, obs, n_theta);
    return check_launch(env, "k_observe");
}

int risvec_map_actions(risvec_env_t* env, const float* raw, float* action, float* phase, void* stream) {
    if (!env || !raw || !action) return fail(RISVEC_ERR_INVALID, "NULL argument");
    ENTER_DEVICE(env->device);
    const Dims& d = env->dims;
    if (d.variant == RISVEC_VARIANT_MARL) {
        const long long n = (long long)d.E * d.V;
        k_map_actions_marl<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, env->params, raw, action);
        return check_launch(env, "k_map_actions_marl");
    }
    if (!phase) return fail(RISVEC_ERR_INVALID, "SARL action mapping needs the phase output");
    const long long n = (long long)d.E * (2 * d.V + d.M);
    k_map_actions_sarl<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, raw, action, phase);
    return check_launch(env, "k_map_actions_sarl");
}

int risvec_step_marl_fused(risvec_env_t* env, const float* raw, const int32_t* partner, const int32_t* ngroups,
                           const int32_t* arrivals, float* obs, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_MARL) return fail(RISVEC_ERR_INVALID, "handle is not a MARL env");
    if (!raw || !partner || !ngroups || !obs) return fail(RISVEC_ERR_INVALID, "raw, partner, ngroups and obs are required");
    ENTER_DEVICE(env->device);
    const Dims& d = env->dims;
    MarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = 1; a.raw = raw; a.obs = obs; a.partner = partner; a.ngroups = ngroups; a.arrivals = arrivals;
    if (choose_marl(env, a) == kMarlV8) {
        // ONE launch: action mapping in the prologue, Environ.step, marl_get_state of the new state in the epilogue
        env->stats_folded = 0;  // an attached statistics accumulator is served by k_shard_stats
        return finish_rollout(env, launch_marl_v8(env, a, (cudaStream_t)stream), stream);
    }
    // shapes the fused kernel does not take: the same three steps as separate launches (scratch action in the stage)
    if (int rc = ensure_stage(env, (size_t)d.E * 2 * d.V * 4 + 256)) return rc;
    Carver c{env->stage, 0};
    float* act = c.take<float>((size_t)d.E * 2 * d.V);
    if (int rc = risvec_map_actions(env, raw, act, nullptr, stream)) return rc;
    if (int rc = risvec_rollout_marl(env, 1, act, partner, ngroups, arrivals, nullptr, stream)) return rc;
    return risvec_observe(env, obs, stream);
}

int risvec_step_sarl_fused(risvec_env_t* env, const float* raw, const int32_t* arrivals, float* obs, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (env->dims.variant != RISVEC_VARIANT_SARL) return fail(RISVEC_ERR_INVALID, "handle is not a SARL env");
    if (!raw || !obs) return fail(RISVEC_ERR_INVALID, "raw and obs are required");
    ENTER_DEVICE(env->device);
    const Dims& d = env->dims;
    SarlArgs a;
    memset(&a, 0, sizeof(a));
    a.T = 1; a.raw = raw; a.obs = obs; a.arrivals = arrivals;
    if (choose_sarl(env, a) == kSarlMma) {
        // ONE launch: action mapping in the prologue, Environ.step, get_state of the new state in the epilogue
        env->stats_folded = 0;  // an attached statistics accumulator is served by k_shard_stats
        return finish_rollout(env, launch_sarl_mma(env, a, (cudaStream_t)stream), stream);
    }
    // shapes the fused kernel does not take: the same three steps as separate launches (scratch in the stage)
    if (int rc = ensure_stage(env, (size_t)d.E * (2 * d.V + d.M) * 4 + 512)) return rc;
    Carver c{env->stage, 0};
    float* act = c.take<float>((size_t)d.E * 2 * d.V);
    float* ph = c.take<float>((size_t)d.E * d.M);
    if (int rc = risvec_map_actions(env, raw, act, ph, stream)) return rc;
    if (int rc = risvec_rollout_sarl(env, 1, act, ph, arrivals, nullptr, stream)) return rc;
    return risvec_observe(env, obs, stream);
}

int risvec_random_phase(risvec_env_t* env, const int32_t* idx, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    ENTER_DEVICE(env->device);
    const long long n = (long long)env->dims.E * env->dims.M;
    k_random_phase<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(env->dims, env->st, idx, env->chan_calls++);
    return check_launch(env, "k_random_phase");
}

int risvec_direct_link(risvec_env_t* env, const double* normals, double* path_loss, double* shadowing, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (!path_loss && !shadowing) return fail(RISVEC_ERR_INVALID, "both outputs are NULL");
    ENTER_DEVICE(env->device);
    const long long n = (long long)env->dims.E * env->dims.V;
    const double* shadow_state = (const double*)(env->arena + env->fields[RISVEC_F_V2I_SHADOWING].offset);
    k_direct_link<<<(int)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(env->dims, env->st, env->params, shadow_state,
                                                                       normals, path_loss, shadowing, env->chan_calls++);
    return check_launch(env, "k_direct_link");
}

int risvec_default_pairing(int n_veh, int yaml, risvec_pairing_t* out) {
    if (!out) return fail(RISVEC_ERR_INVALID, "out is NULL");
    if (n_veh < 1) return fail(RISVEC_ERR_INVALID, "n_veh must be >= 1");
    memset(out, 0, sizeof(*out));
    out->min_pair_target = n_veh / 4 > 1 ? n_veh / 4 : 1;
    out->mwm_backoff_rounds = 5; out->relax_topk_step = 1; out->qos_enable = 1;
    out->mwm_accept_quantile = 0.10; out->mwm_accept_q_step = 0.05; out->completion_min_quantile = 0.30;
    out->relax_tau_factor_per_round = 0.95; out->tau_back_floor_db = 3.0;
    out->score_w_delta_db = 1.0; out->score_w_history = 0.3; out->abs_gain_min_db = -INFINITY;
    out->qos_soft_penalty_dbscore = 6.0; out->pair_hist_decay = 0.97;
    if (yaml) {  // config.yaml: min_pair_target 3, mwm_backoff_rounds 3, abs_gain_min_db -120
        out->min_pair_target = 3; out->mwm_backoff_rounds = 3; out->abs_gain_min_db = -120.0;
    }
    return RISVEC_OK;
}

// Smallest double x >= 0 with log2(1.0 + x) >= R_min as this host's libm evaluates it (the
// reference's test is `np.log2(1.0 + max(0.0, sinr)) >= R_min`, marl_train_bcd.py:877-881; the
// left side is monotone in sinr).  R_min <= 0 is always satisfied.
static double qos_sinr_threshold(double R_min) {
    if (!(R_min > 0.0)) return -INFINITY;
    if (!(R_min < 1000.0)) return INFINITY;
    double lo = 0.0, hi = exp2(R_min) * 1.0000001;      // predicate false at lo, true at hi
    while (!(log2(1.0 + hi) >= R_min)) hi *= 2.0;
    int64_t a, b;
    memcpy(&a, &lo, 8);
    memcpy(&b, &hi, 8);
    while (b - a > 1) {     // non-negative doubles are ordered like their bit patterns
        const int64_t mid = a + (b - a) / 2;
        double x;
        memcpy(&x, &mid, 8);
        if (log2(1.0 + x) >= R_min) b = mid; else a = mid;
    }
    memcpy(&hi, &b, 8);
    return hi;
}

static PairArgs pair_state_args(risvec_env* env) {
    auto P = [&](int f) { return (void*)(env->arena + env->fields[f].offset); };
    PairArgs a;
    memset(&a, 0, sizeof(a));
    a.hist = (float*)P(RISVEC_F_PAIR_HIST); a.streak = (int*)P(RISVEC_F_PAIR_STREAK);
    a.tau = (double*)P(RISVEC_F_PAIR_TAU); a.lastk = (int*)P(RISVEC_F_PAIR_K);
    a.mask = (unsigned char*)P(RISVEC_F_PAIR_MASK); a.rounds = (int*)P(RISVEC_F_PAIR_ROUNDS);
    a.partner = (int*)P(RISVEC_F_NOMA_PARTNER); a.ngroups = (int*)P(RISVEC_F_NOMA_NGROUPS);
    a.pairs = (int*)P(RISVEC_F_NOMA_PAIRS); a.npairs = (int*)P(RISVEC_F_NOMA_NPAIRS);
    return a;
}

// the launch shared by risvec_pair_noma and risvec_pair_noma_episodes: `a` carries the state pointers and the
// per-call episode arguments, the knobs of `cfg` are added here
static int pair_noma_launch(risvec_env* env, const risvec_pairing_t* cfg, PairArgs a, void* stream) {
    const int V = env->dims.V;
    a.min_pairs = cfg->min_pair_target > 1 ? cfg->min_pair_target : 1;
    a.backoff_rounds = cfg->mwm_backoff_rounds;
    a.accept_q = cfg->mwm_accept_quantile; a.accept_q_step = cfg->mwm_accept_q_step;
    a.completion_q = cfg->completion_min_quantile;
    a.relax_topk_step = cfg->relax_topk_step;
    a.relax_tau_factor = cfg->relax_tau_factor_per_round; a.tau_floor = cfg->tau_back_floor_db;
    a.w_delta = cfg->score_w_delta_db; a.abs_min_db = cfg->abs_gain_min_db; a.qos_pen = cfg->qos_soft_penalty_dbscore;
    a.w_hist = (float)cfg->score_w_history; a.decay_f = (float)cfg->pair_hist_decay;
    a.qos_enable = cfg->qos_enable != 0;
    a.noise = env->params.noise_power; a.P_max = env->params.P_max;
    a.sinr_min = qos_sinr_threshold(env->params.R_min_bpsHz);
    const size_t per = pair_smem_bytes(V);
    const int wpc = V <= 8 ? 4 : (V <= 10 ? 2 : 1);
    const int blocks = (env->dims.E + wpc - 1) / wpc;
    const double* const ep = env->env_params;  // per-env noise_power / P_max of the QoS test
    switch (V) {
#define RISVEC_PAIR_CASE(n)                                                                                    \
    case n:                                                                                                    \
        if (ep) k_pair_noma<n, true><<<blocks, 32 * wpc, per * wpc, (cudaStream_t)stream>>>(env->dims, env->st, a, ep); \
        else k_pair_noma<n><<<blocks, 32 * wpc, per * wpc, (cudaStream_t)stream>>>(env->dims, env->st, a, nullptr);     \
        break;
        RISVEC_PAIR_CASE(1) RISVEC_PAIR_CASE(2) RISVEC_PAIR_CASE(3) RISVEC_PAIR_CASE(4) RISVEC_PAIR_CASE(5)
        RISVEC_PAIR_CASE(6) RISVEC_PAIR_CASE(7) RISVEC_PAIR_CASE(8) RISVEC_PAIR_CASE(9) RISVEC_PAIR_CASE(10)
        RISVEC_PAIR_CASE(11) RISVEC_PAIR_CASE(12)
#undef RISVEC_PAIR_CASE
    }
    return check_launch(env, "k_pair_noma");
}

int risvec_pair_noma(risvec_env_t* env, const risvec_pairing_t* cfg, const float* p01, int64_t p01_env_stride,
                     int topk, double tau_q, int recalc_mask, const int32_t* reuse, int decay, int new_episode,
                     void* stream) {
    if (!env || !cfg || !p01) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (new_episode && !recalc_mask)
        return fail(RISVEC_ERR_INVALID, "new_episode needs recalc_mask (the first step of an episode builds the mask)");
    const int V = env->dims.V;
    if (V > RISVEC_PAIR_MAX_V)
        return fail(RISVEC_ERR_UNSUPPORTED, "pairing is an exact matching over 2^V subsets: V = %d > %d", V,
                    RISVEC_PAIR_MAX_V);
    if (p01_env_stride < V) return fail(RISVEC_ERR_INVALID, "p01_env_stride %lld < V", (long long)p01_env_stride);
    if (!(tau_q >= 0.0 && tau_q <= 1.0)) return fail(RISVEC_ERR_INVALID, "tau_q must be in [0, 1]");
    ENTER_DEVICE(env->device);
    PairArgs a = pair_state_args(env);
    a.p01 = p01; a.p01_stride = p01_env_stride; a.reuse = reuse;
    a.topk = topk; a.tau_q = tau_q; a.recalc = recalc_mask != 0; a.decay = decay != 0; a.fresh = new_episode != 0;
    return pair_noma_launch(env, cfg, a, stream);
}

int risvec_pair_noma_episodes(risvec_env_t* env, const risvec_pairing_t* cfg, const float* p01, int64_t p01_env_stride,
                              const risvec_pair_schedule_t* schedule, const uint8_t* start, const int32_t* reuse,
                              int decay, void* stream) {
    if (!env || !cfg || !p01 || !schedule || !start) return fail(RISVEC_ERR_INVALID, "NULL argument");
    const int V = env->dims.V;
    if (V > RISVEC_PAIR_MAX_V)
        return fail(RISVEC_ERR_UNSUPPORTED, "pairing is an exact matching over 2^V subsets: V = %d > %d", V,
                    RISVEC_PAIR_MAX_V);
    if (p01_env_stride < V) return fail(RISVEC_ERR_INVALID, "p01_env_stride %lld < V", (long long)p01_env_stride);
    const double q0 = schedule->tau_q_start, q1 = schedule->tau_q_end;
    if (!(q0 >= 0.0 && q0 <= 1.0 && q1 >= 0.0 && q1 <= 1.0))
        return fail(RISVEC_ERR_INVALID, "schedule tau_q_start / tau_q_end must be in [0, 1]");
    ENTER_DEVICE(env->device);
    PairArgs a = pair_state_args(env);
    a.p01 = p01; a.p01_stride = p01_env_stride; a.reuse = reuse; a.decay = decay != 0;
    a.start = start;
    a.ep_index = (const int*)(env->arena + env->fields[RISVEC_F_EP_INDEX].offset);
    a.sched_topk_start = schedule->topk_start; a.sched_topk_end = schedule->topk_end;
    a.sched_warmup = schedule->warmup_episodes;
    a.sched_tau_q_start = q0; a.sched_tau_q_end = q1;
    return pair_noma_launch(env, cfg, a, stream);
}

int risvec_pair_reset(risvec_env_t* env, void* stream) { return risvec_pair_reset_masked(env, nullptr, stream); }

int risvec_pair_reset_masked(risvec_env_t* env, const uint8_t* env_mask, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    ENTER_DEVICE(env->device);
    return launch_pair_reset(env, env_mask, EnvGate{}, stream);
}

}  // extern "C"

namespace {
int launch_pair_reset(risvec_env* env, const uint8_t* env_mask, EnvGate g, void* stream) {
    PairArgs a = pair_state_args(env);
    const long long n = (long long)env->dims.E * env->dims.V * env->dims.V;
    const int threads = 256, blocks = (int)((n + threads - 1) / threads);
    k_pair_reset<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->dims, a, env_mask, g);
    return check_launch(env, "k_pair_reset");
}

constexpr int kEpAll = RISVEC_EP_RESET | RISVEC_EP_POSITIONS | RISVEC_EP_CHANNEL | RISVEC_EP_PAIRING;

// k_begin_episode takes the shapes of k_bcd_v8 with the free channel
bool episode_fused(const risvec_env* env) {
    const Dims& d = env->dims;
    return d.V <= 8 && d.ncand <= 8 && d.M <= 256 && env->params.channel_model == RISVEC_CHANNEL_FREE &&
           !env->ovr.force_generic;
}

template <bool CLOCK>
int launch_begin_episode(risvec_env* env, const EpisodeArgs& a, void* stream) {
    const int wpb = env->dims.M <= 64 ? 4 : 1;  // as k_bcd_v8: 4 envs per warp, 2 M double2 of shared memory per env
    const int blocks = (env->dims.E + 4 * wpb - 1) / (4 * wpb);
    const size_t smem = (size_t)wpb * 4 * 2 * env->dims.M * sizeof(double2);
    return dispatch_re(env, [&](auto re) {
        auto kern = k_begin_episode<CLOCK, decltype(re)::value>;
        if (smem > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<blocks, 32 * wpb, smem, (cudaStream_t)stream>>>(env->dims, env->st, env->params, pair_state_args(env), a,
                                                               env->ris_elem);
        return check_launch(env, "k_begin_episode");
    });
}

// the stages `stages` as separate kernels restricted by `g` (g.bits null = every env), in the fixed order
int episode_stages_separate(risvec_env* env, int stages, EnvGate g, const double* uniforms, int n_uni, int32_t* used_out,
                            void* stream) {
    auto gate = [&](unsigned bit) { EnvGate h = g; h.bit = bit; return h; };
    if (stages & RISVEC_EP_RESET)
        if (int rc = launch_make_new_game(env, nullptr, nullptr, 0, nullptr, 0, gate(RISVEC_EP_RESET), stream)) return rc;
    if (stages & RISVEC_EP_POSITIONS) {
        if (int rc = launch_renew_positions(env, uniforms, n_uni, used_out, gate(RISVEC_EP_POSITIONS), stream)) return rc;
        if (int rc = launch_compute_parms(env, gate(RISVEC_EP_POSITIONS), stream)) return rc;
    }
    if (stages & RISVEC_EP_CHANNEL) {
        if (int rc = launch_bcd(env, gate(RISVEC_EP_CHANNEL), stream)) return rc;
        if (int rc = launch_gains(env, nullptr, nullptr, nullptr, gate(RISVEC_EP_CHANNEL), stream)) return rc;
    }
    if (stages & RISVEC_EP_PAIRING)
        if (int rc = launch_pair_reset(env, nullptr, gate(RISVEC_EP_PAIRING), stream)) return rc;
    return RISVEC_OK;
}
}  // namespace

extern "C" {

int risvec_begin_episode(risvec_env_t* env, const uint8_t* stages_env, int stages, const double* uniforms, int n_uni,
                         int32_t* used_out, void* stream) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (stages & ~kEpAll) return fail(RISVEC_ERR_INVALID, "unknown stage bits 0x%x", stages & ~kEpAll);
    if (uniforms != nullptr && n_uni < 1) return fail(RISVEC_ERR_INVALID, "uniforms given with n_uni = %d", n_uni);
    if (stages == 0) return RISVEC_OK;
    if (!(stages & RISVEC_EP_POSITIONS)) {  // nothing renews: the uniforms and used_out are not touched
        uniforms = nullptr;
        used_out = nullptr;
    }
    ENTER_DEVICE(env->device);
    if (!episode_fused(env)) {
        EnvGate g{};
        g.bits = stages_env;
        return episode_stages_separate(env, stages, g, uniforms, n_uni, used_out, stream);
    }
    EpisodeArgs a;
    memset(&a, 0, sizeof(a));
    a.stages = (unsigned)stages; a.stages_env = stages_env;
    a.uniforms = uniforms; a.n_uni = n_uni; a.used_out = used_out;
    a.reset_call = env->reset_calls; a.mob_call = env->mob_calls;
    if (int rc = launch_begin_episode<false>(env, a, stream)) return rc;
    // the counters advance as the separate calls advance them (the free channel draws nothing)
    if (stages & RISVEC_EP_RESET) env->reset_calls++;
    if (stages & RISVEC_EP_POSITIONS) env->mob_calls++;
    return RISVEC_OK;
}

int risvec_episode_tick(risvec_env_t* env, const risvec_episode_schedule_t* schedule, uint8_t* start_out,
                        uint8_t* done_out, void* stream) {
    if (!env || !schedule) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (schedule->steps_per_episode < 1 || schedule->positions_every < 1)
        return fail(RISVEC_ERR_INVALID, "steps_per_episode and positions_every must be >= 1");
    if (schedule->stages & ~kEpAll) return fail(RISVEC_ERR_INVALID, "unknown stage bits 0x%x", schedule->stages & ~kEpAll);
    ENTER_DEVICE(env->device);
    EpisodeArgs a;
    memset(&a, 0, sizeof(a));
    a.stages = (unsigned)schedule->stages;
    a.ep_step = (int*)(env->arena + env->fields[RISVEC_F_EP_STEP].offset);
    a.ep_index = (int*)(env->arena + env->fields[RISVEC_F_EP_INDEX].offset);
    a.steps_per_episode = schedule->steps_per_episode; a.positions_every = schedule->positions_every;
    a.start_out = start_out; a.done_out = done_out;
    if (episode_fused(env)) return launch_begin_episode<true>(env, a, stream);
    // other shapes: the clock writes each env's bits and draw key, then the stage kernels run for those envs
    a.bits_out = env->ep_bits; a.key_out = env->ep_keys;
    k_episode_clock<<<(env->dims.E + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->dims, a);
    if (int rc = check_launch(env, "k_episode_clock")) return rc;
    EnvGate g{};
    g.bits = env->ep_bits;
    g.call = env->ep_keys;
    return episode_stages_separate(env, schedule->stages, g, nullptr, 0, nullptr, stream);
}

int risvec_replay_create(int device, int64_t mem_size, int input_shape, int n_actions, int n_agents,
                         risvec_replay_t** out) {
    if (!out) return fail(RISVEC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (mem_size < 1 || input_shape < 1 || n_actions < 1 || n_agents < 1)
        return fail(RISVEC_ERR_INVALID, "mem_size, input_shape, n_actions, n_agents must be >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        return fail(RISVEC_ERR_NODEVICE, "no CUDA device visible: this library has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(RISVEC_ERR_INVALID, "device %d out of range [0, %d)", device, ndev);
    ENTER_DEVICE(device);
    risvec_replay* rb = new (std::nothrow) risvec_replay();
    if (!rb) return fail(RISVEC_ERR_INVALID, "out of host memory");
    memset(rb, 0, sizeof(*rb));
    rb->device = device;
    ReplayMem& m = rb->m;
    m.mem_size = mem_size; m.N = n_agents; m.S = input_shape * n_agents; m.A = n_actions * n_agents;
    const size_t sz[RISVEC_RB_COUNT] = {(size_t)mem_size * m.S * 4, (size_t)mem_size * m.A * 4, (size_t)mem_size * 4,
                                        (size_t)mem_size * m.N * 4, (size_t)mem_size * m.S * 4, (size_t)mem_size,
                                        (size_t)mem_size * m.N * m.N * 4};
    size_t off = 0;
    for (int i = 0; i < RISVEC_RB_COUNT; ++i) { rb->off[i] = off; off = align_up(off + sz[i], 256); }
    rb->off[RISVEC_RB_COUNT] = off;   // tail: the device counter (int64) and its ticket (uint32)
    off += sizeof(long long) + sizeof(unsigned);
    cudaError_t ce = cudaMalloc((void**)&rb->base, off);
    if (ce == cudaSuccess) ce = cudaMemset(rb->base, 0, off);
    if (ce != cudaSuccess) {
        if (rb->base) cudaFree(rb->base);
        delete rb;
        return fail(RISVEC_ERR_CUDA, "replay memory of %zu bytes: %s", off, cudaGetErrorString(ce));
    }
    m.state = (float*)(rb->base + rb->off[RISVEC_RB_STATE]); m.action = (float*)(rb->base + rb->off[RISVEC_RB_ACTION]);
    m.reward_g = (float*)(rb->base + rb->off[RISVEC_RB_REWARD_G]);
    m.reward_l = (float*)(rb->base + rb->off[RISVEC_RB_REWARD_L]);
    m.state_ = (float*)(rb->base + rb->off[RISVEC_RB_NEW_STATE]);
    m.terminal = (unsigned char*)(rb->base + rb->off[RISVEC_RB_TERMINAL]);
    m.mask = (float*)(rb->base + rb->off[RISVEC_RB_MASK]);
    rb->ctr.count = (long long*)(rb->base + rb->off[RISVEC_RB_COUNT]);
    rb->ctr.ticket = (unsigned*)(rb->ctr.count + 1);
    *out = rb;
    return RISVEC_OK;
}

int risvec_replay_destroy(risvec_replay_t* rb) {
    if (!rb) return RISVEC_OK;
    DeviceGuard _dev_guard(rb->device);
    if (rb->base) cudaFree(rb->base);
    delete rb;
    return RISVEC_OK;
}

int risvec_replay_field(risvec_replay_t* rb, int field, void** dev_ptr, int64_t* rows, int64_t* cols, int* elem_bytes) {
    if (!rb) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (field < 0 || field >= RISVEC_RB_COUNT) return fail(RISVEC_ERR_INVALID, "unknown replay field %d", field);
    const ReplayMem& m = rb->m;
    const int64_t c[RISVEC_RB_COUNT] = {m.S, m.A, 1, m.N, m.S, 1, (int64_t)m.N * m.N};
    if (dev_ptr) *dev_ptr = rb->base + rb->off[field];
    if (rows) *rows = m.mem_size;
    if (cols) *cols = c[field];
    if (elem_bytes) *elem_bytes = field == RISVEC_RB_TERMINAL ? 1 : 4;
    return RISVEC_OK;
}

int64_t risvec_replay_count(const risvec_replay_t* rb) { return rb ? (rb->devcnt ? -1 : rb->mem_cntr) : 0; }

static const char kDevcntMsg[] =
    "the handle counts on the device: use risvec_replay_store_devcnt / risvec_replay_store_marl_devcnt / "
    "risvec_replay_sample_devcnt, and the counter pointer of risvec_replay_use_device_counter for the count";

int risvec_replay_set_count(risvec_replay_t* rb, int64_t mem_cntr) {
    if (!rb || mem_cntr < 0) return fail(RISVEC_ERR_INVALID, "NULL handle or negative count");
    if (rb->devcnt) return fail(RISVEC_ERR_INVALID, "%s", kDevcntMsg);
    rb->mem_cntr = mem_cntr;
    return RISVEC_OK;
}

}  // extern "C"
namespace risvec {
__global__ void k_replay_seed_counter(ReplayCtr c, long long count) {
    *c.count = count;
    *c.ticket = 0;
}
}  // namespace risvec
extern "C" {

int risvec_replay_use_device_counter(risvec_replay_t* rb, int64_t** dev_count, void* stream) {
    if (!rb || !dev_count) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (rb->devcnt) return fail(RISVEC_ERR_INVALID, "the handle already counts on the device");
    ENTER_DEVICE(rb->device);
    k_replay_seed_counter<<<1, 1, 0, (cudaStream_t)stream>>>(rb->ctr, rb->mem_cntr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RISVEC_ERR_CUDA, "launch of k_replay_seed_counter failed: %s", cudaGetErrorString(e));
    rb->launches += 1;
    rb->devcnt = 1;
    *dev_count = (int64_t*)rb->ctr.count;
    return RISVEC_OK;
}

// The path choice (flat float4, vec4 or scalar) depends on shapes and pointers only, never on the count, so a
// device-counter store takes the same path as a host-counter store of the same arguments.
static int replay_store(risvec_replay* rb, int E, const ReplaySrc& src, int marl, int devcnt, cudaStream_t st) {
    const ReplayMem& m = rb->m;
    auto al16 = [](const void* q) { return ((uintptr_t)q & 15) == 0; };   // float4 path needs aligned sources
    const bool vec4 = m.S % 4 == 0 && m.A % 4 == 0 && m.N % 4 == 0 && al16(src.state) && al16(src.state_) &&
                      al16(src.action) && al16(src.reward_l);
    const int vec = vec4 ? 4 : 1;
    const long long total = (long long)E * ((2 * m.S + m.A + m.N + m.N * m.N) / vec + 1);
    const int threads = 256;
    long long blocks = (total + threads - 1) / threads;
    if (blocks > 148 * 64) blocks = 148 * 64;   // grid-stride beyond 64 blocks per SM
    const bool mask_ok = marl ? (src.mask_u8 == nullptr || (((uintptr_t)src.mask_u8) & 3) == 0)
                              : (src.mask_f == nullptr || al16(src.mask_f));
    const ReplayCtr ctr = devcnt ? rb->ctr : ReplayCtr{};
    const long long first = devcnt ? 0 : rb->mem_cntr;
    if (vec4 && mask_ok && (long long)E * (m.A > m.N * m.N ? m.A : m.N * m.N) < (1ll << 31)) {
        // flat float4 copies, one grid row per field (no per-element row arithmetic)
        const long long slot0 = first % m.mem_size;
        const int n_wrap = (int)((m.mem_size - slot0) < E ? (m.mem_size - slot0) : E);
        const long long big = (long long)E * ((m.A > m.S ? m.A : m.S) / 4);
        long long bx = (big + threads - 1) / threads;
        if (bx > 148 * 8) bx = 148 * 8;
        const dim3 grid((unsigned)bx, 6);
        if (marl && devcnt) k_replay_store_flat<1, 1><<<grid, threads, 0, st>>>(m, slot0, n_wrap, E, src, ctr);
        else if (marl) k_replay_store_flat<1, 0><<<grid, threads, 0, st>>>(m, slot0, n_wrap, E, src, ctr);
        else if (devcnt) k_replay_store_flat<0, 1><<<grid, threads, 0, st>>>(m, slot0, n_wrap, E, src, ctr);
        else k_replay_store_flat<0, 0><<<grid, threads, 0, st>>>(m, slot0, n_wrap, E, src, ctr);
    } else {
        using K = void (*)(ReplayMem, long long, int, ReplaySrc, ReplayCtr);
        static const K ks[2][2][2] = {{{k_replay_store<1, 0, 0>, k_replay_store<1, 0, 1>},
                                       {k_replay_store<1, 1, 0>, k_replay_store<1, 1, 1>}},
                                      {{k_replay_store<4, 0, 0>, k_replay_store<4, 0, 1>},
                                       {k_replay_store<4, 1, 0>, k_replay_store<4, 1, 1>}}};
        ks[vec4][marl != 0][devcnt != 0]<<<(int)blocks, threads, 0, st>>>(m, first, E, src, ctr);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RISVEC_ERR_CUDA, "launch of k_replay_store failed: %s", cudaGetErrorString(e));
    rb->launches += 1;
    if (!devcnt) rb->mem_cntr += E;
    return RISVEC_OK;
}

static int store_checks(risvec_replay* rb, int E, int devcnt) {
    if (E < 1 || E > rb->m.mem_size) return fail(RISVEC_ERR_INVALID, "E = %d must be in [1, mem_size]", E);
    if (rb->devcnt && !devcnt) return fail(RISVEC_ERR_INVALID, "%s", kDevcntMsg);
    if (!rb->devcnt && devcnt)
        return fail(RISVEC_ERR_INVALID, "the handle counts on the host: call risvec_replay_use_device_counter first");
    return RISVEC_OK;
}

static int store_flat(risvec_replay_t* rb, int E, const float* state, const float* action, const float* reward_g,
                      const float* reward_l, const float* state_, const uint8_t* done, int done_all,
                      const float* mask_flat, void* stream, int devcnt) {
    if (!rb || !state || !action || !reward_g || !reward_l || !state_) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (int rc = store_checks(rb, E, devcnt)) return rc;
    ENTER_DEVICE(rb->device);
    ReplaySrc src;
    memset(&src, 0, sizeof(src));
    src.state = state; src.state_ = state_; src.action = action; src.reward_g = reward_g; src.reward_l = reward_l;
    src.mask_f = mask_flat; src.done = done; src.done_all = done_all;
    return replay_store(rb, E, src, 0, devcnt, (cudaStream_t)stream);
}

static int store_marl(risvec_replay_t* rb, int E, const float* state, const float* intent_probs,
                      const float* power_raw, const float* reward_g, const float* reward_l, const float* state_,
                      const uint8_t* done, int done_all, const uint8_t* mask_u8, void* stream, int devcnt) {
    if (!rb || !state || !intent_probs || !power_raw || !reward_g || !reward_l || !state_)
        return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (int rc = store_checks(rb, E, devcnt)) return rc;
    if (rb->m.A != rb->m.N * (rb->m.N + 2))
        return fail(RISVEC_ERR_INVALID, "store_marl needs n_actions = n_agents + 2 (got %d per agent)", rb->m.A / rb->m.N);
    ENTER_DEVICE(rb->device);
    ReplaySrc src;
    memset(&src, 0, sizeof(src));
    src.state = state; src.state_ = state_; src.probs = intent_probs; src.power = power_raw; src.reward_g = reward_g;
    src.reward_l = reward_l; src.mask_u8 = mask_u8; src.done = done; src.done_all = done_all;
    return replay_store(rb, E, src, 1, devcnt, (cudaStream_t)stream);
}

int risvec_replay_store(risvec_replay_t* rb, int E, const float* state, const float* action, const float* reward_g,
                        const float* reward_l, const float* state_, const uint8_t* done, int done_all,
                        const float* mask_flat, void* stream) {
    return store_flat(rb, E, state, action, reward_g, reward_l, state_, done, done_all, mask_flat, stream, 0);
}

int risvec_replay_store_devcnt(risvec_replay_t* rb, int E, const float* state, const float* action,
                               const float* reward_g, const float* reward_l, const float* state_, const uint8_t* done,
                               int done_all, const float* mask_flat, void* stream) {
    return store_flat(rb, E, state, action, reward_g, reward_l, state_, done, done_all, mask_flat, stream, 1);
}

int risvec_replay_store_marl(risvec_replay_t* rb, int E, const float* state, const float* intent_probs,
                             const float* power_raw, const float* reward_g, const float* reward_l,
                             const float* state_, const uint8_t* done, int done_all, const uint8_t* mask_u8,
                             void* stream) {
    return store_marl(rb, E, state, intent_probs, power_raw, reward_g, reward_l, state_, done, done_all, mask_u8,
                      stream, 0);
}

int risvec_replay_store_marl_devcnt(risvec_replay_t* rb, int E, const float* state, const float* intent_probs,
                                    const float* power_raw, const float* reward_g, const float* reward_l,
                                    const float* state_, const uint8_t* done, int done_all, const uint8_t* mask_u8,
                                    void* stream) {
    return store_marl(rb, E, state, intent_probs, power_raw, reward_g, reward_l, state_, done, done_all, mask_u8,
                      stream, 1);
}

static int replay_sample(risvec_replay_t* rb, int B, const int64_t* idx, float* states, float* actions,
                         float* rewards_g, float* rewards_l, float* states_, uint8_t* dones, float* masks,
                         void* stream, int devcnt) {
    if (!rb || !idx || !states || !actions || !rewards_g || !rewards_l || !states_ || !dones || !masks)
        return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (B < 1) return fail(RISVEC_ERR_INVALID, "B must be >= 1");
    if (devcnt && !rb->devcnt)
        return fail(RISVEC_ERR_INVALID, "the handle counts on the host: call risvec_replay_use_device_counter first");
    ENTER_DEVICE(rb->device);
    if (devcnt)
        k_replay_sample<1><<<B, 128, 0, (cudaStream_t)stream>>>(rb->m, B, (const long long*)idx, states, actions,
                                                               rewards_g, rewards_l, states_, dones, masks,
                                                               rb->ctr.count);
    else
        k_replay_sample<0><<<B, 128, 0, (cudaStream_t)stream>>>(rb->m, B, (const long long*)idx, states, actions,
                                                               rewards_g, rewards_l, states_, dones, masks, nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RISVEC_ERR_CUDA, "launch of k_replay_sample failed: %s", cudaGetErrorString(e));
    rb->launches += 1;
    return RISVEC_OK;
}

int risvec_replay_sample(risvec_replay_t* rb, int B, const int64_t* idx, float* states, float* actions,
                         float* rewards_g, float* rewards_l, float* states_, uint8_t* dones, float* masks,
                         void* stream) {
    return replay_sample(rb, B, idx, states, actions, rewards_g, rewards_l, states_, dones, masks, stream, 0);
}

int risvec_replay_sample_devcnt(risvec_replay_t* rb, int B, const int64_t* draws, float* states, float* actions,
                                float* rewards_g, float* rewards_l, float* states_, uint8_t* dones, float* masks,
                                void* stream) {
    return replay_sample(rb, B, draws, states, actions, rewards_g, rewards_l, states_, dones, masks, stream, 1);
}

}  // extern "C"
namespace risvec {
__global__ void k_atomic_add_f64(double* __restrict__ dst, const double* __restrict__ src, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(dst + i, src[i]);    // dst may be peer memory: a red.global.add.f64 over NVLink
}
}  // namespace risvec
extern "C" {

int risvec_shard_stats(risvec_env_t* env, double* out, int accumulate, void* stream) {
    if (!env || !out) return fail(RISVEC_ERR_INVALID, "NULL argument");
    ENTER_DEVICE(env->device);
    if (!accumulate) CUDA_TRY(cudaMemsetAsync(out, 0, (RISVEC_NSTAT + 1) * sizeof(double), (cudaStream_t)stream));
    int blocks = (env->dims.E + 63) / 64;   // 64 envs per block and pass; at most one block per SM
    if (blocks > 148) blocks = 148;
    k_shard_stats<<<blocks, 1024, 0, (cudaStream_t)stream>>>(env->dims, env->st, out);
    return check_launch(env, "k_shard_stats");
}

int risvec_episode_accumulate(risvec_env_t* env, double* running, const uint8_t* done, int done_all,
                              double* records, int64_t capacity, unsigned long long* count, void* stream) {
    if (!env || !running || !records || !count) return fail(RISVEC_ERR_INVALID, "NULL argument");
    if (capacity < 1) return fail(RISVEC_ERR_INVALID, "capacity must be >= 1 (got %lld)", (long long)capacity);
    ENTER_DEVICE(env->device);
    EpisodeLogArgs a;
    a.running = running; a.done = done; a.done_all = done_all;
    a.n_user = env->dims.variant == RISVEC_VARIANT_MARL ? env->dims.V : 0;
    a.records = records; a.capacity = capacity; a.count = count;
    const int per = episode_log_envs_per_block(a.n_user);
    k_episode_accumulate<<<(env->dims.E + per - 1) / per, kEpLogThreads, 0, (cudaStream_t)stream>>>(env->dims, env->st,
                                                                                                    a);
    return check_launch(env, "k_episode_accumulate");
}

int risvec_attach_env_params(risvec_env_t* env, const double* table) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (table != nullptr) {
        if (!aligned8(table)) return fail(RISVEC_ERR_INVALID, "the per-env parameter table must be 8-byte aligned");
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, table) != cudaSuccess) {
            cudaGetLastError();
            return fail(RISVEC_ERR_INVALID, "the per-env parameter table is not a CUDA pointer");
        }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
            return fail(RISVEC_ERR_INVALID, "the per-env parameter table must be device memory");
        if (at.device != env->device)
            return fail(RISVEC_ERR_INVALID, "the per-env parameter table is on device %d, the handle on device %d",
                        at.device, env->device);
    }
    env->env_params = table;
    return RISVEC_OK;
}

int risvec_attach_ris_elements(risvec_env_t* env, const int32_t* n_elem) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (n_elem != nullptr) {
        if (((uintptr_t)n_elem) & 3u) return fail(RISVEC_ERR_INVALID, "the per-env RIS size must be 4-byte aligned");
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, n_elem) != cudaSuccess) {
            cudaGetLastError();
            return fail(RISVEC_ERR_INVALID, "the per-env RIS size is not a CUDA pointer");
        }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
            return fail(RISVEC_ERR_INVALID, "the per-env RIS size must be device memory");
        if (at.device != env->device)
            return fail(RISVEC_ERR_INVALID, "the per-env RIS size is on device %d, the handle on device %d", at.device,
                        env->device);
    }
    env->ris_elem = n_elem;
    return RISVEC_OK;
}

int risvec_attach_stats_accumulator(risvec_env_t* env, double* slots) {
    if (!env) return fail(RISVEC_ERR_INVALID, "NULL handle");
    if (((uintptr_t)slots) & 255u) return fail(RISVEC_ERR_INVALID, "the accumulator must be 256-byte aligned");
    env->stats_slots = slots;
    return RISVEC_OK;
}
}  // extern "C"
namespace risvec {
__global__ void k_collect_stats(double* __restrict__ slots, double* __restrict__ out, int accumulate) {
    const int c = threadIdx.x;  // one thread per statistic: the 64 slots are summed in slot order, then cleared
    if (c > RISVEC_NSTAT) return;
    double acc = accumulate ? out[c] : 0.0;
    for (int sl = 0; sl < kRisvecStatSlots; ++sl) {
        acc += slots[sl * 32 + c];
        slots[sl * 32 + c] = 0.0;
    }
    out[c] = acc;
}
}  // namespace risvec
extern "C" {
int risvec_collect_stats(risvec_env_t* env, double* slots, double* out, int accumulate, void* stream) {
    if (!env || !slots || !out) return fail(RISVEC_ERR_INVALID, "NULL argument");
    ENTER_DEVICE(env->device);
    k_collect_stats<<<1, 32, 0, (cudaStream_t)stream>>>(slots, out, accumulate);
    return check_launch(env, "k_collect_stats");
}

// ---- a device buffer other processes of the job can map (CUDA IPC over NVLink peer access)
int risvec_shared_buffer_create(int device, uint64_t bytes, void** dev_ptr, unsigned char ipc_handle[64]) {
    if (!dev_ptr || !ipc_handle || bytes == 0) return fail(RISVEC_ERR_INVALID, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    ENTER_DEVICE(device);
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    CUDA_TRY(cudaMemset(p, 0, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(RISVEC_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(ipc_handle, &h, 64);
    *dev_ptr = p;
    return RISVEC_OK;
}
int risvec_shared_buffer_open(int device, const unsigned char ipc_handle[64], void** dev_ptr) {
    if (!dev_ptr || !ipc_handle) return fail(RISVEC_ERR_INVALID, "bad arguments");
    ENTER_DEVICE(device);
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, 64);
    void* p = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *dev_ptr = p;
    return RISVEC_OK;
}
int risvec_shared_buffer_add(int device, double* dst, const double* src, int n, void* stream) {
    if (!dst || !src || n <= 0) return fail(RISVEC_ERR_INVALID, "bad arguments");
    ENTER_DEVICE(device);
    k_atomic_add_f64<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(dst, src, n);
    CUDA_TRY(cudaGetLastError());
    return RISVEC_OK;
}
int risvec_shared_buffer_close(int device, void* dev_ptr, int owner) {
    if (!dev_ptr) return RISVEC_OK;
    ENTER_DEVICE(device);
    if (owner) CUDA_TRY(cudaFree(dev_ptr));
    else CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
    return RISVEC_OK;
}

int risvec_get_rng_counters(const risvec_env_t* env, uint64_t out[3]) {
    if (!env || !out) return fail(RISVEC_ERR_INVALID, "NULL argument");
    out[0] = env->reset_calls; out[1] = env->mob_calls; out[2] = env->chan_calls;
    return RISVEC_OK;
}
int risvec_set_rng_counters(risvec_env_t* env, const uint64_t in[3]) {
    if (!env || !in) return fail(RISVEC_ERR_INVALID, "NULL argument");
    env->reset_calls = in[0]; env->mob_calls = in[1]; env->chan_calls = in[2];
    return RISVEC_OK;
}
int64_t risvec_launch_count(const risvec_env_t* env) { return env ? env->launches : 0; }
const char* risvec_last_step_kernel(const risvec_env_t* env) { return (env && env->step_kernel) ? env->step_kernel : ""; }

}  // extern "C"
