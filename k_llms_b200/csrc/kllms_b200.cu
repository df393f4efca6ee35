// kllms_b200.cu — C ABI (include/kllms_b200.h) and launchers of the sm_100a consensus kernels.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared -Xcompiler -fPIC
//        (see k_llms_b200/csrc/Makefile; __graft_entry__.build() runs it).
// No torch, no libraries beyond the CUDA runtime; the driver entry point cuTensorMapEncodeTiled is fetched
// through cudaGetDriverEntryPoint so libcuda is not a link-time dependency.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/kllms_b200.h"
#include "kc_internal.h"
#include "kc_common.cuh"
#include "kc_extra.cuh"
#include "kc_medoid.cuh"
#include "kc_numeric.cuh"
#include "kc_push.cuh"
#include "kc_vote.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace

int kc_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

namespace {

#define KC_CUDA(call)                                                                                         \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(KC_ECUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct DeviceInfo {
    int sm_count = 0;
    int cc_major = 0;
};

int device_info(DeviceInfo &info) {
    int dev = 0;
    KC_CUDA(cudaGetDevice(&dev));
    static std::mutex mu;
    static std::vector<DeviceInfo> cache;
    std::lock_guard<std::mutex> lock(mu);
    if ((int)cache.size() <= dev) cache.resize(dev + 1);
    if (cache[dev].sm_count == 0) {
        KC_CUDA(cudaDeviceGetAttribute(&cache[dev].sm_count, cudaDevAttrMultiProcessorCount, dev));
        KC_CUDA(cudaDeviceGetAttribute(&cache[dev].cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    }
    info = cache[dev];
    if (info.cc_major != 10) return fail(KC_ENODEV, "device %d has compute capability %d.x; this library is sm_100a only", dev, info.cc_major);
    return KC_OK;
}

// ---------------------------------------------------------------- TMA descriptor

using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn &fn) {
    static EncodeTiledFn cached = nullptr;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    if (!cached) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        KC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (q != cudaDriverEntryPointSuccess || !p) return fail(KC_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
        cached = reinterpret_cast<EncodeTiledFn>(p);
    }
    fn = cached;
    return KC_OK;
}

// rows of `row_bytes` (a power of two in [32, 512]) viewed as a 2-D int32 tensor whose inner extent is
// min(row_bytes, 128) bytes — the widest span a TMA swizzle mode covers; box = TILE groups.
int make_row_tensor_map(CUtensorMap &map, const void *base, int64_t n_groups, int row_bytes, int tile_groups) {
    EncodeTiledFn encode = nullptr;
    int rc = get_encode_fn(encode);
    if (rc) return rc;
    const int inner_bytes = std::min(row_bytes, 128);
    const int rows_per_group = row_bytes / inner_bytes;
    cuuint64_t dims[2] = {(cuuint64_t)(inner_bytes / 4), (cuuint64_t)n_groups * rows_per_group};
    cuuint64_t strides[1] = {(cuuint64_t)inner_bytes};
    cuuint32_t box[2] = {(cuuint32_t)(inner_bytes / 4), (cuuint32_t)(tile_groups * rows_per_group)};
    cuuint32_t elem_strides[2] = {1, 1};
    const CUtensorMapSwizzle swz = inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                   : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                       : CU_TENSOR_MAP_SWIZZLE_32B;
    CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void *>(base), dims, strides, box, elem_strides,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(KC_ECUDA, "cuTensorMapEncodeTiled failed: CUresult %d", (int)r);
    return KC_OK;
}

template <typename Kernel>
int persistent_grid(Kernel kernel, int threads, size_t smem, int64_t n_tiles, int &grid) {
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return fail(KC_ECUDA, "kernel does not fit on an SM (smem %zu)", smem);
    grid = (int)std::min<int64_t>(n_tiles, (int64_t)info.sm_count * per_sm);  // one wave of resident CTAs
    return KC_OK;
}

// A TMA tile coordinate is int32: launch in slabs of at most this many groups.
constexpr int64_t kMaxGroupsPerLaunch = (int64_t)1 << 28;

// ---------------------------------------------------------------- K1 launchers

kc::FieldMap make_field_map(const int32_t *none_code, int n_fields) {
    kc::FieldMap fm;
    fm.none_code = none_code;
    fm.n_fields = (uint32_t)std::max(n_fields, 1);
    fm.magic = (uint32_t)(((uint64_t)1 << 32) / fm.n_fields + 1);
    return fm;
}

template <int N, int WARPS, int STAGES, bool HAS_NC>
int launch_vote_tma_nc(const int32_t *codes, int64_t G, const int32_t *none_code, int n_fields, int32_t *win, uint32_t *meta,
                       cudaStream_t st, kc::OutRoute mc) {
    auto kernel = kc::vote_tma_kernel<N, WARPS, STAGES, HAS_NC>;
    const size_t smem = (size_t)WARPS * STAGES * 32 * N * 4 + 1024;
    // a slab starts on a record boundary so that (g - g0) % n_fields == g % n_fields
    const int64_t slab = std::max<int64_t>(n_fields, kMaxGroupsPerLaunch / n_fields * n_fields);
    for (int64_t g0 = 0; g0 < G; g0 += slab) {
        const int64_t gs = std::min(slab, G - g0);
        CUtensorMap map;
        int rc = make_row_tensor_map(map, codes + g0 * N, gs, N * 4, 32);
        if (rc) return rc;
        int grid = 0;
        rc = persistent_grid(kernel, WARPS * 32, smem, ((gs + 31) / 32 + WARPS - 1) / WARPS, grid);
        if (rc) return rc;
        kernel<<<grid, WARPS * 32, smem, st>>>(map, (uint32_t)gs, make_field_map(none_code, n_fields), win + g0, meta + g0, mc);
        KC_CUDA(cudaGetLastError());
    }
    return KC_OK;
}

template <int N, int WARPS, int STAGES>
int launch_vote_tma(const int32_t *codes, int64_t G, const int32_t *none_code, int n_fields, int32_t *win, uint32_t *meta,
                    cudaStream_t st, kc::OutRoute mc) {
    if (none_code && n_fields < 60000)
        return launch_vote_tma_nc<N, WARPS, STAGES, true>(codes, G, none_code, n_fields, win, meta, st, mc);
    if (none_code) return fail(KC_EINVAL, "kc_vote_i32: more than 60000 fields with none_code is not supported");
    return launch_vote_tma_nc<N, WARPS, STAGES, false>(codes, G, nullptr, 1, win, meta, st, mc);
}

template <int NP, bool VEC>
int launch_vote_direct(const int32_t *codes, int64_t G, int n, const int32_t *none_code, int n_fields, int32_t *win,
                       uint32_t *meta, cudaStream_t st, kc::OutRoute mc) {
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int threads = 256;
    const int64_t blocks = (G + threads - 1) / threads;
    const int grid = (int)std::min<int64_t>(blocks, (int64_t)info.sm_count * 8);
    const kc::FieldMap fm = make_field_map(none_code, n_fields);
    static const bool prefetch = [] { const char *e = getenv("KC_VOTE_PREFETCH"); return !e || e[0] != '0'; }();
    constexpr bool kCanPrefetch = VEC && NP >= 4 && NP <= 16;
    auto go = [&](auto kernel) -> int {
        kernel<<<grid, threads, 0, st>>>(codes, G, n, fm, win, meta, mc);
        KC_CUDA(cudaGetLastError());
        return KC_OK;
    };
    if (kCanPrefetch && prefetch) return none_code ? go(kc::vote_direct_kernel<NP, VEC, true, kCanPrefetch>) : go(kc::vote_direct_kernel<NP, VEC, false, kCanPrefetch>);
    return none_code ? go(kc::vote_direct_kernel<NP, VEC, true, false>) : go(kc::vote_direct_kernel<NP, VEC, false, false>);
}

// small rows, local results: GPT consecutive groups per thread (kc::vote_multi_kernel); the remainder (< GPT groups) and every
// routed mode go through the one-group-per-thread kernel
template <int NP>
int launch_vote_multi(const int32_t *codes, int64_t G, const int32_t *none_code, int n_fields, int32_t *win, uint32_t *meta,
                      cudaStream_t st) {
    constexpr int GPT = 16 / NP;
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int64_t units = G / GPT;
    if (units > 0) {
        const int threads = 256;
        const int grid = (int)std::min<int64_t>((units + threads - 1) / threads, (int64_t)info.sm_count * 8);
        const kc::FieldMap fm = make_field_map(none_code, n_fields);
        if (none_code) kc::vote_multi_kernel<NP, GPT, true><<<grid, threads, 0, st>>>(codes, units, fm, win, meta);
        else kc::vote_multi_kernel<NP, GPT, false><<<grid, threads, 0, st>>>(codes, units, fm, win, meta);
        KC_CUDA(cudaGetLastError());
    }
    const int64_t done = units * GPT;
    if (done < G) {  // the last few groups: their field phase continues where the units stopped
        kc::OutRoute local{};
        if (!none_code) return launch_vote_direct<NP, true>(codes + done * NP, G - done, NP, nullptr, 1, win + done, meta + done, st, local);
        // rotate the field table so that group `done` sees its own field first: simplest is one group per launch (< GPT of them)
        for (int64_t g = done; g < G; ++g) {
            const int f = (int)(g % n_fields);
            rc = launch_vote_direct<NP, true>(codes + g * NP, 1, NP, none_code + f, 1, win + g, meta + g, st, local);
            if (rc) return rc;
        }
    }
    return KC_OK;
}

template <int NP, bool VEC>
int launch_vote_i8(const int8_t *codes, int64_t G, int n, const int32_t *none_code, int n_fields, int32_t *win, uint32_t *meta,
                   cudaStream_t st) {
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int threads = 256;
    const int grid = (int)std::min<int64_t>((G + threads - 1) / threads, (int64_t)info.sm_count * 8);
    const kc::FieldMap fm = make_field_map(none_code, n_fields);
    if (none_code)
        kc::vote_i8_kernel<NP, VEC, true><<<grid, threads, 0, st>>>(codes, G, n, fm, win, meta, kc::OutRoute{});
    else
        kc::vote_i8_kernel<NP, VEC, false><<<grid, threads, 0, st>>>(codes, G, n, fm, win, meta, kc::OutRoute{});
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

// ---------------------------------------------------------------- K3 launcher

template <int T, int CAP>
static int launch_logprob_tile(const float *d_logprobs, const int64_t *d_offsets, int64_t n_seq, float *d_sum, const DeviceInfo &info,
                               void *stream) {
    // T sequences per tile, their contiguous tokens staged in shared memory (up to CAP floats; longer tiles fall back to
    // the warp-per-sequence loop inside the kernel)
    auto kernel = kc::logprob_sum_tile_kernel<T, CAP>;
    const size_t smem = (size_t)(CAP + 4) * sizeof(float);
    KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, T, smem));
    const int64_t tiles = (n_seq + T - 1) / T;
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)info.sm_count * std::max(per_sm, 1));
    kernel<<<grid, T, smem, static_cast<cudaStream_t>(stream)>>>(d_logprobs, d_offsets, n_seq, d_sum);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

// ---------------------------------------------------------------- K2 launchers

template <int N, int WARPS, int STAGES, int MIN_CTAS = 1>
int launch_numeric_tma(const double *vals, int64_t G, double rel_eps, double abs_eps, double *value, uint32_t *meta,
                       cudaStream_t st, kc::OutRoute mc) {
    auto kernel = kc::numeric_tma_kernel<N, WARPS, STAGES, MIN_CTAS>;
    const size_t smem = (size_t)WARPS * STAGES * 32 * N * 8 + (size_t)WARPS * 32 * N * 8 + 1024;
    for (int64_t g0 = 0; g0 < G; g0 += kMaxGroupsPerLaunch) {
        const int64_t gs = std::min(kMaxGroupsPerLaunch, G - g0);
        CUtensorMap map;
        int rc = make_row_tensor_map(map, vals + g0 * N, gs, N * 8, 32);
        if (rc) return rc;
        int grid = 0;
        rc = persistent_grid(kernel, WARPS * 32, smem, ((gs + 31) / 32 + WARPS - 1) / WARPS, grid);
        if (rc) return rc;
        kernel<<<grid, WARPS * 32, smem, st>>>(map, gs, rel_eps, abs_eps, value + g0, meta + g0, mc);
        KC_CUDA(cudaGetLastError());
    }
    return KC_OK;
}

// fast path in front (kc::numeric_fast), general path for the groups it leaves open; KC_NUM_FAST=0 disables it
template <int N, int WARPS, int STAGES, int MIN_CTAS>
int launch_numeric_tma_fast(const double *vals, int64_t G, double rel_eps, double abs_eps, double *value, uint32_t *meta,
                            cudaStream_t st, kc::OutRoute mc) {
    auto kernel = kc::numeric_tma_fast_kernel<N, WARPS, STAGES, MIN_CTAS>;
    const size_t smem = (size_t)WARPS * STAGES * 32 * N * 8 + (size_t)WARPS * 32 * N * 8 + 1024;
    for (int64_t g0 = 0; g0 < G; g0 += kMaxGroupsPerLaunch) {
        const int64_t gs = std::min(kMaxGroupsPerLaunch, G - g0);
        CUtensorMap map;
        int rc = make_row_tensor_map(map, vals + g0 * N, gs, N * 8, 32);
        if (rc) return rc;
        int grid = 0;
        rc = persistent_grid(kernel, WARPS * 32, smem, ((gs + 31) / 32 + WARPS - 1) / WARPS, grid);
        if (rc) return rc;
        kernel<<<grid, WARPS * 32, smem, st>>>(map, vals + g0 * N, gs, rel_eps, abs_eps, value + g0, meta + g0, mc);
        KC_CUDA(cudaGetLastError());
    }
    return KC_OK;
}

static bool numeric_fast_env() {
    static const bool on = [] { const char *e = getenv("KC_NUM_FAST"); return !(e && e[0] == '0'); }();
    return on;
}

template <int NP, int T>
int launch_numeric_direct(const double *vals, int64_t G, int n, double rel_eps, double abs_eps, double *value,
                          uint32_t *meta, cudaStream_t st, kc::OutRoute mc) {
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    static const bool prefetch_env = [] { const char *e = getenv("KC_NUM_PREFETCH"); return !e || e[0] != '0'; }();
    const bool prefetch = prefetch_env && n == NP && NP >= 4 && NP <= 16;
    const size_t smem = (size_t)NP * T * 8;
    auto launch = [&](auto kernel) -> int {
        KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, T, smem));
        if (per_sm < 1) return fail(KC_ECUDA, "numeric_direct_kernel<%d> does not fit", NP);
        const int64_t blocks = (G + T - 1) / T;
        const int grid = (int)std::min<int64_t>(blocks, (int64_t)info.sm_count * per_sm);
        kernel<<<grid, T, smem, st>>>(vals, G, n, rel_eps, abs_eps, value, meta, mc);
        KC_CUDA(cudaGetLastError());
        return KC_OK;
    };
    if constexpr (NP >= 4 && NP <= 16) {
        if (prefetch) return launch(kc::numeric_direct_kernel<NP, T, true>);
    }
    return launch(kc::numeric_direct_kernel<NP, T, false>);
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// A-B knobs: KC_FORCE_DIRECT=1 / KC_FORCE_TMA=1 route every n through one family of front-ends.
bool force_tma() {
    static const bool v = [] {
        const char *e = getenv("KC_FORCE_TMA");
        return e && e[0] == '1';
    }();
    return v;
}
bool force_direct() {
    static const bool v = [] {
        const char *e = getenv("KC_FORCE_DIRECT");
        return e && e[0] == '1';
    }();
    return v;
}

}  // namespace

// ---------------------------------------------------------------- host-buffer context

namespace {
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t need) {
        if (p && need <= cap) return KC_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        if (cudaMalloc(&p, need) != cudaSuccess) {
            cudaGetLastError();
            return fail(KC_ENOMEM, "cudaMalloc(%zu) failed", need);
        }
        cap = need;
        return KC_OK;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};
struct HostCtx {
    static constexpr int kStreams = 3;
    int device = -1;
    cudaStream_t streams[kStreams] = {};
    DevBuf codes[kStreams], vals[kStreams], win[kStreams], vmeta[kStreams], value[kStreams], nmeta[kStreams], none;
};
std::mutex g_host_mu;
HostCtx g_host[16];

}  // namespace

// ================================================================ C ABI

extern "C" {

int kc_version(void) { return KC_VERSION; }

const char *kc_last_error(void) { return g_err; }

int kc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

int kc_sm_count(int device) {
    int sm = 0;
    KC_CUDA(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
    return sm;
}

int kc_set_device(int device) {
    KC_CUDA(cudaSetDevice(device));
    return KC_OK;
}

int kc_vote_i32(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                int32_t *d_win_code, uint32_t *d_meta, void *stream) {
    return kc_vote_i32_ex(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, KC_OUT_LOCAL, stream);
}

static int make_peer_route(const char *who, int32_t n_peers, const int64_t *peer_delta_bytes, kc::OutRoute &r) {
    if (n_peers < 0 || n_peers > 7) return fail(KC_EINVAL, "%s: n_peers=%d outside [0,7]", who, n_peers);
    if (n_peers > 0 && !peer_delta_bytes) return fail(KC_EINVAL, "%s: NULL peer_delta_bytes", who);
    r = kc::OutRoute{};
    r.mode = KC_OUT_PEERS;
    r.n_peers = n_peers;
    for (int k = 0; k < n_peers; ++k) {
        if (peer_delta_bytes[k] % 8 != 0) return fail(KC_EINVAL, "%s: peer_delta_bytes[%d] is not a multiple of 8", who, k);
        r.delta[k] = (long long)peer_delta_bytes[k];
    }
    return KC_OK;
}

static int vote_i32_routed(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                           int32_t *d_win_code, uint32_t *d_meta, kc::OutRoute mc, void *stream);

int kc_vote_i32_ex(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                   int32_t *d_win_code, uint32_t *d_meta, uint32_t out_mode, void *stream) {
    if (out_mode > KC_OUT_MULTIMEM) return fail(KC_EINVAL, "kc_vote_i32_ex: unknown out_mode %u (peers: kc_vote_i32_peers)", out_mode);
    kc::OutRoute mc{};
    mc.mode = out_mode;
    return vote_i32_routed(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, mc, stream);
}

int kc_vote_i32_peers(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                      int32_t *d_win_code, uint32_t *d_meta, int32_t n_peers, const int64_t *peer_delta_bytes, void *stream) {
    kc::OutRoute mc;
    int rc = make_peer_route("kc_vote_i32_peers", n_peers, peer_delta_bytes, mc);
    if (rc) return rc;
    return vote_i32_routed(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, mc, stream);
}

int kc_vote_i32_peers_packed(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                             int32_t *d_win_code, uint32_t *d_meta, uint32_t *d_packed, int32_t n_peers,
                             const int64_t *peer_delta_bytes, uint32_t *d_overflow, void *stream) {
    if (!d_packed || !d_overflow) return fail(KC_EINVAL, "kc_vote_i32_peers_packed: NULL d_packed / d_overflow");
    kc::OutRoute mc;
    int rc = make_peer_route("kc_vote_i32_peers_packed", n_peers, peer_delta_bytes, mc);
    if (rc) return rc;
    mc.mode = 3u;
    mc.packed = d_packed;
    mc.overflow = d_overflow;
    return vote_i32_routed(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, mc, stream);
}

static int vote_i32_routed(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                           int32_t *d_win_code, uint32_t *d_meta, kc::OutRoute mc, void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_vote_i32: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_groups < 0) return fail(KC_EINVAL, "kc_vote_i32: negative n_groups");
    if (n_groups == 0) return KC_OK;
    if (!d_codes || !d_win_code || !d_meta) return fail(KC_EINVAL, "kc_vote_i32: NULL buffer");
    if (d_none_code && n_fields < 1) return fail(KC_EINVAL, "kc_vote_i32: none_code given but n_fields=%d", n_fields);
    if (!d_none_code) n_fields = 1;
    if (!aligned16(d_codes)) return fail(KC_EINVAL, "kc_vote_i32: d_codes must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // measured on B200 (profiles/README.md): the direct front-end wins up to n = 16, the TMA pipeline from n = 32
    static const bool multi = [] { const char *e = getenv("KC_VOTE_MULTI"); return !e || e[0] != '0'; }();
    if (multi && mc.local() && !force_tma() && (n == 2 || n == 4 || n == 8)) {
        if (n == 2) return launch_vote_multi<2>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st);
        if (n == 4) return launch_vote_multi<4>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st);
        return launch_vote_multi<8>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st);
    }
    if (force_direct() || (!force_tma() && n <= 16)) {
        switch (n) {
            case 1: return launch_vote_direct<1, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 2: return launch_vote_direct<2, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 4: return launch_vote_direct<4, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 8: return launch_vote_direct<8, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 16: return launch_vote_direct<16, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 32: return launch_vote_direct<32, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            case 64: return launch_vote_direct<64, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
            default: break;
        }
    } else
    switch (n) {
        case 1: return launch_vote_direct<1, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        case 2: return launch_vote_direct<2, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        case 4: return launch_vote_direct<4, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        case 8: return launch_vote_tma<8, 8, 4>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        case 16: return launch_vote_tma<16, 8, 4>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st, mc);  // KC_FORCE_TMA only
        case 32: return launch_vote_tma<32, 8, 2>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        case 64: return launch_vote_tma<64, 4, 2>(d_codes, n_groups, d_none_code, n_fields, d_win_code, d_meta, st, mc);
        default: break;
    }
    if (n < 4) return launch_vote_direct<4, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
    if (n < 8) return launch_vote_direct<8, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
    if (n < 16) return launch_vote_direct<16, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
    if (n < 32) return launch_vote_direct<32, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
    return launch_vote_direct<64, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st, mc);
}

int kc_vote_i32_wire(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                     int32_t *d_win_code, uint32_t *d_meta, void *d_wire_words, int32_t wide, int32_t n_peers,
                     const int64_t *peer_delta_bytes, uint32_t *d_overflow, void *stream) {
    if (!d_wire_words || !d_overflow) return fail(KC_EINVAL, "kc_vote_i32_wire: NULL d_wire_words / d_overflow");
    kc::OutRoute mc{};
    if (n_peers) {
        int rc = make_peer_route("kc_vote_i32_wire", n_peers, peer_delta_bytes, mc);
        if (rc) return rc;
    }
    mc.mode = 4u;
    mc.packed = static_cast<uint32_t *>(d_wire_words);
    mc.overflow = d_overflow;
    mc.wire_wide = wide ? 1u : 0u;
    return vote_i32_routed(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, mc, stream);
}

static int fill_push_args(kc::PushArgs &a, const int32_t *d_win_code, const uint32_t *d_vote_meta, int64_t n_vote_groups, const double *d_value,
                          const uint32_t *d_num_meta, int64_t n_num_groups, void *d_wire_votes, void *d_wire_value, void *d_wire_num_meta,
                          int32_t wide, int32_t n_peers, const int64_t *peer_delta_bytes, uint32_t *d_overflow) {
    if (n_vote_groups < 0 || n_num_groups < 0) return fail(KC_EINVAL, "kc_push_results: negative size");
    if (n_vote_groups % 8 || n_num_groups % 8) return fail(KC_EINVAL, "kc_push_results: group counts must be multiples of 8 (whole 16-byte vectors)");
    if (n_peers < 0 || n_peers > 7 || (n_peers && !peer_delta_bytes)) return fail(KC_EINVAL, "kc_push_results: n_peers=%d outside [0,7] or NULL deltas", n_peers);
    if ((n_vote_groups && (((!d_win_code) != (!d_vote_meta)) || !d_wire_votes)) || (n_num_groups && (!d_value || !d_num_meta || !d_wire_value || !d_wire_num_meta)))
        return fail(KC_EINVAL, "kc_push_results: NULL buffer");
    for (const void *p : {(const void *)d_win_code, (const void *)d_vote_meta, (const void *)d_value, (const void *)d_num_meta,
                          (const void *)d_wire_votes, (const void *)d_wire_value, (const void *)d_wire_num_meta})
        if (!aligned16(p)) return fail(KC_EINVAL, "kc_push_results: buffers must be 16-byte aligned");
    a = kc::PushArgs{};
    a.win = d_win_code;
    a.vmeta = d_vote_meta;
    a.gv = n_vote_groups;
    a.value = d_value;
    a.nmeta = d_num_meta;
    a.gx = n_num_groups;
    a.wire_votes = static_cast<uint8_t *>(d_wire_votes);
    a.wire_value = static_cast<uint8_t *>(d_wire_value);
    a.wire_nmeta = static_cast<uint8_t *>(d_wire_num_meta);
    a.n_peers = n_peers;
    for (int k = 0; k < n_peers; ++k) {
        if (peer_delta_bytes[k] % 16 != 0) return fail(KC_EINVAL, "kc_push_results: peer_delta_bytes[%d] is not a multiple of 16", k);
        a.delta[k] = (long long)peer_delta_bytes[k];
    }
    a.wide = wide ? 1 : 0;
    a.overflow = d_overflow;
    return KC_OK;
}

int kc_push_results(const int32_t *d_win_code, const uint32_t *d_vote_meta, int64_t n_vote_groups, const double *d_value,
                    const uint32_t *d_num_meta, int64_t n_num_groups, void *d_wire_votes, void *d_wire_value, void *d_wire_num_meta,
                    int32_t wide, int32_t n_peers, const int64_t *peer_delta_bytes, uint32_t *d_overflow, int32_t max_ctas, void *stream) {
    kc::PushArgs a;
    int rc = fill_push_args(a, d_win_code, d_vote_meta, n_vote_groups, d_value, d_num_meta, n_num_groups, d_wire_votes, d_wire_value,
                            d_wire_num_meta, wide, n_peers, peer_delta_bytes, d_overflow);
    if (rc) return rc;
    if (n_vote_groups == 0 && n_num_groups == 0) return KC_OK;
    DeviceInfo info;
    rc = device_info(info);
    if (rc) return rc;
    const int64_t units = n_vote_groups / (wide ? 4 : 8) + n_num_groups / 2 + n_num_groups / (wide ? 4 : 8);
    int64_t grid = (units + 255) / 256;
    grid = std::min<int64_t>(grid, max_ctas > 0 ? max_ctas : info.sm_count * 2);
    kc::push_kernel<<<(int)std::max<int64_t>(grid, 1), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_vote_i8(const int8_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
               int32_t *d_win_code, uint32_t *d_meta, void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_vote_i8: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_groups < 0) return fail(KC_EINVAL, "kc_vote_i8: negative n_groups");
    if (n_groups == 0) return KC_OK;
    if (!d_codes || !d_win_code || !d_meta) return fail(KC_EINVAL, "kc_vote_i8: NULL buffer");
    if (d_none_code && n_fields < 1) return fail(KC_EINVAL, "kc_vote_i8: none_code given but n_fields=%d", n_fields);
    if (!d_none_code) n_fields = 1;
    if (!aligned16(d_codes)) return fail(KC_EINVAL, "kc_vote_i8: d_codes must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (n) {
        case 4: return launch_vote_i8<4, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
        case 8: return launch_vote_i8<8, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
        case 16: return launch_vote_i8<16, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
        case 32: return launch_vote_i8<32, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
        case 64: return launch_vote_i8<64, true>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
        default: break;
    }
    if (n < 4) return launch_vote_i8<4, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
    if (n < 8) return launch_vote_i8<8, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
    if (n < 16) return launch_vote_i8<16, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
    if (n < 32) return launch_vote_i8<32, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
    return launch_vote_i8<64, false>(d_codes, n_groups, n, d_none_code, n_fields, d_win_code, d_meta, st);
}

int kc_numeric_f64(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                   uint32_t *d_meta, void *stream) {
    return kc_numeric_f64_ex(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, KC_OUT_LOCAL, stream);
}

static int numeric_f64_routed(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                              uint32_t *d_meta, kc::OutRoute mc, void *stream);

int kc_numeric_f64_ex(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                      uint32_t *d_meta, uint32_t out_mode, void *stream) {
    if (out_mode > KC_OUT_MULTIMEM) return fail(KC_EINVAL, "kc_numeric_f64_ex: unknown out_mode %u (peers: kc_numeric_f64_peers)", out_mode);
    kc::OutRoute mc{};
    mc.mode = out_mode;
    return numeric_f64_routed(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, mc, stream);
}

int kc_numeric_f64_peers(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                         uint32_t *d_meta, int32_t n_peers, const int64_t *peer_delta_bytes, void *stream) {
    kc::OutRoute mc;
    int rc = make_peer_route("kc_numeric_f64_peers", n_peers, peer_delta_bytes, mc);
    if (rc) return rc;
    return numeric_f64_routed(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, mc, stream);
}

static int numeric_f64_routed(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                              uint32_t *d_meta, kc::OutRoute mc, void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_numeric_f64: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_groups < 0) return fail(KC_EINVAL, "kc_numeric_f64: negative n_groups");
    if (!(rel_eps >= 0.0) || !(abs_eps >= 0.0)) return fail(KC_EINVAL, "kc_numeric_f64: rel_eps/abs_eps must be >= 0");
    if (n_groups == 0) return KC_OK;
    if (!d_vals || !d_value || !d_meta) return fail(KC_EINVAL, "kc_numeric_f64: NULL buffer");
    if (!aligned16(d_vals)) return fail(KC_EINVAL, "kc_numeric_f64: d_vals must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // The fast kernels store a group's result when it is decided — most lanes at once, the deferred ones later and
    // scattered.  Local stores do not care; multicast stores do (measured at 2 GPUs: K2 0.33 ms with the general
    // kernel's whole-warp stores, 0.57 ms with the fast kernel's), and a fused step is NVLink-bound anyway.
    const bool numeric_fast = numeric_fast_env() && mc.local();  // the fast kernels only have local stores
    // measured on B200: TMA pipeline wins at n = 16 and 32; direct at n <= 8 (tiles too small to prefetch far enough)
    // and at n = 64 (register pressure)
    if (!force_direct() && (force_tma() || n == 16 || n == 32))
        switch (n) {
            case 4: return launch_numeric_tma<4, 8, 2, 3>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
            case 8: return launch_numeric_tma<8, 8, 2, 3>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
            case 16:
                if (numeric_fast) return launch_numeric_tma_fast<16, 4, 1, 6>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
                return launch_numeric_tma<16, 4, 1, 7>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
            case 32:
                if (numeric_fast) return launch_numeric_tma_fast<32, 4, 1, 4>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
                return launch_numeric_tma<32, 4, 1, 4>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
            case 64: return launch_numeric_tma<64, 2, 1, 3>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, st, mc);
            default: break;
        }
    static const bool quads = [] { const char *e = getenv("KC_NUM_QUADS"); return !e || e[0] != '0'; }();
    if (n == 4 && quads && mc.local() && !force_direct() && !force_tma()) {  // the n = 4 pattern analysis, two groups per thread
        DeviceInfo info;
        int rc = device_info(info);
        if (rc) return rc;
        const int64_t units = n_groups / 2;
        if (units > 0) {
            const int grid = (int)std::min<int64_t>((units + 255) / 256, (int64_t)info.sm_count * 8);
            kc::numeric_quads_kernel<<<grid, 256, 0, st>>>(d_vals, units, rel_eps, abs_eps, d_value, d_meta);
            KC_CUDA(cudaGetLastError());
        }
        const int64_t done = units * 2;
        if (done == n_groups) return KC_OK;
        return launch_numeric_direct<4, 128>(d_vals + done * 4, n_groups - done, n, rel_eps, abs_eps, d_value + done, d_meta + done, st, mc);
    }
    if (numeric_fast && !force_direct() && (n == 8 || n == 4)) {
        auto launch_fast = [&](auto kernel, int NP) -> int {
            DeviceInfo info;
            int rc = device_info(info);
            if (rc) return rc;
            const int T = 128;
            const size_t smem = (size_t)T * NP * 8;
            int per_sm = 0;
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, T, smem));
            if (per_sm < 1) return fail(KC_ECUDA, "numeric_direct_fast_kernel<%d> does not fit", NP);
            const int64_t want = (n_groups + T - 1) / T;
            const int grid = (int)std::min<int64_t>(want, (int64_t)info.sm_count * per_sm);
            kernel<<<grid, T, smem, st>>>(d_vals, n_groups, rel_eps, abs_eps, d_value, d_meta, mc);
            KC_CUDA(cudaGetLastError());
            return KC_OK;
        };
        if (n == 8) return launch_fast(kc::numeric_direct_fast_kernel<8, 128>, 8);
        return launch_fast(kc::numeric_direct_fast_kernel<4, 128>, 4);
    }
    static const bool pairs = [] { const char *e = getenv("KC_NUM_PAIRS"); return !e || e[0] != '0'; }();
    if (n == 2 && pairs && mc.local() && !force_direct()) {  // the n = 2 case analysis, four groups per thread; the last < 4 groups below
        DeviceInfo info;
        int rc = device_info(info);
        if (rc) return rc;
        const int64_t units = n_groups / 4;
        if (units > 0) {
            const int grid = (int)std::min<int64_t>((units + 255) / 256, (int64_t)info.sm_count * 8);
            kc::numeric_pairs_kernel<<<grid, 256, 0, st>>>(d_vals, units, rel_eps, abs_eps, d_value, d_meta);
            KC_CUDA(cudaGetLastError());
        }
        const int64_t done = units * 4;
        if (done == n_groups) return KC_OK;
        return launch_numeric_direct<2, 128>(d_vals + done * 2, n_groups - done, n, rel_eps, abs_eps, d_value + done, d_meta + done, st, mc);
    }
    if (n <= 2) return launch_numeric_direct<2, 128>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
    if (n <= 4) return launch_numeric_direct<4, 128>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
    if (n <= 8) return launch_numeric_direct<8, 128>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
    if (n <= 16) return launch_numeric_direct<16, 128>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
    if (n <= 32) return launch_numeric_direct<32, 128>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
    return launch_numeric_direct<64, 64>(d_vals, n_groups, n, rel_eps, abs_eps, d_value, d_meta, st, mc);
}

int kc_confidence_f64(const uint32_t *d_meta, int64_t n_groups, int32_t numeric, const double *d_pvf, double *d_conf,
                      void *stream) {
    if (n_groups < 0) return fail(KC_EINVAL, "kc_confidence_f64: negative n_groups");
    if (n_groups == 0) return KC_OK;
    if (!d_meta || !d_conf) return fail(KC_EINVAL, "kc_confidence_f64: NULL buffer");
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int threads = 256;
    const int grid = (int)std::min<int64_t>((n_groups + threads - 1) / threads, (int64_t)info.sm_count * 8);
    kc::confidence_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(d_meta, n_groups, numeric != 0, d_pvf, d_conf);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_logprob_sum_f32(const float *d_logprobs, const int64_t *d_offsets, int64_t n_seq, float *d_sum, void *stream) {
    if (n_seq < 0) return fail(KC_EINVAL, "kc_logprob_sum_f32: negative n_seq");
    if (n_seq == 0) return KC_OK;
    if (!d_offsets || !d_sum) return fail(KC_EINVAL, "kc_logprob_sum_f32: NULL buffer");
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    static const bool staged = [] { const char *e = getenv("KC_K3_STAGED"); return !e || e[0] != '0'; }();
    if (staged && n_seq >= 4096 && aligned16(d_logprobs)) {
        // 64 sequences per tile, 24 KB of staged tokens: measured best of {128/48 KB, 64/24 KB, 64/16 KB}; 32/12 KB is 3 % faster
        // on config 4 but falls back from 96 tokens per sequence on
        return launch_logprob_tile<64, 6 * 1024>(d_logprobs, d_offsets, n_seq, d_sum, info, stream);
    }
    const int threads = 256;  // 8 warps, one sequence per warp per iteration
    const int64_t warps = n_seq;
    const int grid = (int)std::min<int64_t>((warps + 7) / 8, (int64_t)info.sm_count * 8);
    kc::logprob_sum_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(d_logprobs, d_offsets, n_seq, d_sum);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_weighted_vote_i32(const int32_t *d_codes, const float *d_seq_logprob, int64_t n_records, int32_t n_fields,
                         int32_t n, const int32_t *d_none_code, int32_t *d_win_code, uint32_t *d_meta, float *d_weight,
                         void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_weighted_vote_i32: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_records < 0 || n_fields < 1) return fail(KC_EINVAL, "kc_weighted_vote_i32: bad sizes");
    if (n_records == 0) return KC_OK;
    if (!d_codes || !d_seq_logprob || !d_win_code || !d_meta || !d_weight) return fail(KC_EINVAL, "kc_weighted_vote_i32: NULL buffer");
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int64_t G = n_records * n_fields;
    const int threads = 128;
    const int grid = (int)std::min<int64_t>((G + threads - 1) / threads, (int64_t)info.sm_count * 8);
    const kc::FieldMap fm = make_field_map(d_none_code, n_fields);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    static const bool per_record = [] { const char *e = getenv("KC_K3B_REC"); return !e || e[0] != '0'; }();
    static const bool use_tma = [] { const char *e = getenv("KC_K3B_TMA"); return !e || e[0] != '0'; }();
    if (per_record && use_tma && (n == 32 || n == 64) && n_fields < 60000) {  // rows through K1's warp-private TMA pipelines
        auto launch_tma = [&](auto kernel, int N, int WARPS, int STAGES) -> int {
            const int rec_cap = std::min(32, 31 / n_fields + 2);  // records a tile of 32 groups can span
            const size_t smem = (size_t)WARPS * STAGES * 32 * N * 4 + 1024 + (size_t)WARPS * rec_cap * (N + 1) * 4;
            const int64_t slab = std::max<int64_t>(n_fields, kMaxGroupsPerLaunch / n_fields * n_fields);  // slabs start on record boundaries
            for (int64_t g0 = 0; g0 < G; g0 += slab) {
                const int64_t gs = std::min(slab, G - g0);
                CUtensorMap map;
                int rc2 = make_row_tensor_map(map, d_codes + g0 * N, gs, N * 4, 32);
                if (rc2) return rc2;
                int grid2 = 0;
                rc2 = persistent_grid(kernel, WARPS * 32, smem, ((gs + 31) / 32 + WARPS - 1) / WARPS, grid2);
                if (rc2) return rc2;
                const uint64_t inv_fields = n_fields > 1 ? ~uint64_t(0) / (uint64_t)n_fields + 1 : 0;
                kernel<<<grid2, WARPS * 32, smem, st>>>(map, d_seq_logprob + (g0 / n_fields) * N, (uint32_t)gs, fm, d_none_code != nullptr, rec_cap,
                                                        inv_fields, d_win_code + g0, d_meta + g0, d_weight + g0);
                KC_CUDA(cudaGetLastError());
            }
            return KC_OK;
        };
        static const bool rows = [] { const char *e = getenv("KC_K3B_ROWS"); return !e || e[0] != '0'; }();
        const int rec_cap0 = std::min(32, 31 / n_fields + 2);
        if (rows && n == 32 && rec_cap0 <= 8) {  // weights by a pre-pass, fetched per tile by a bulk copy (n_fields >= 6; n = 64 measured slower)
            auto launch_rows = [&](auto pre_kernel, auto kernel, int N, int WARPS, int STAGES) -> int {
                const int WROW = N + 4;
                float *d_rows = nullptr;
                KC_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&d_rows), (size_t)n_records * WROW * 4, st));
                const int pre_grid = (int)std::min<int64_t>((n_records + 7) / 8, (int64_t)info.sm_count * 8);
                pre_kernel<<<pre_grid, 256, 0, st>>>(d_seq_logprob, n_records, N, WROW, d_rows);
                int rc2 = cudaGetLastError() == cudaSuccess ? KC_OK : fail(KC_ECUDA, "kc_weighted_vote_i32: weight_rows_kernel launch failed");
                const size_t smem = (size_t)WARPS * STAGES * 32 * N * 4 + 1024 + (size_t)WARPS * (STAGES + 1) * rec_cap0 * WROW * 4;
                const int64_t slab = std::max<int64_t>(n_fields, kMaxGroupsPerLaunch / n_fields * n_fields);
                for (int64_t g0 = 0; g0 < G && !rc2; g0 += slab) {
                    const int64_t gs = std::min(slab, G - g0);
                    CUtensorMap map;
                    rc2 = make_row_tensor_map(map, d_codes + g0 * N, gs, N * 4, 32);
                    int grid2 = 0;
                    if (!rc2) rc2 = persistent_grid(kernel, WARPS * 32, smem, ((gs + 31) / 32 + WARPS - 1) / WARPS, grid2);
                    if (rc2) break;
                    const uint64_t inv_fields = n_fields > 1 ? ~uint64_t(0) / (uint64_t)n_fields + 1 : 0;
                    kernel<<<grid2, WARPS * 32, smem, st>>>(map, d_rows + (g0 / n_fields) * WROW, (uint32_t)gs, fm, d_none_code != nullptr, rec_cap0,
                                                            inv_fields, d_win_code + g0, d_meta + g0, d_weight + g0);
                    if (cudaGetLastError() != cudaSuccess) rc2 = fail(KC_ECUDA, "kc_weighted_vote_i32: launch failed");
                }
                cudaFreeAsync(d_rows, st);
                return rc2;
            };
            return launch_rows(kc::weight_rows_kernel, kc::weighted_vote_rows_kernel<32, 8, 2, 3>, 32, 8, 2);
        }
        // measured on B200 (profiles/r2_k3b_variants.txt): n = 32 with 3 CTAs / SM (80 registers) and the logprobs requested a tile ahead;
        // n = 64 (2 x the registers per row) without the prefetch
        if (n == 32) return launch_tma(kc::weighted_vote_tma_kernel<32, 8, 2, 3, true>, 32, 8, 2);
        return launch_tma(kc::weighted_vote_tma_kernel<64, 4, 2, 3, false>, 64, 4, 2);
    }
    if (per_record && n >= 8) {  // weights once per record, one row per thread straight from global memory
        const int max_recs = threads / n_fields + 2;
        auto launch = [&](auto kernel, int NP) -> int {
            const size_t smem = (size_t)max_recs * NP * 4;  // the candidate weights of the tile's records
            KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int per_sm = 1;
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
            const int g2 = (int)std::min<int64_t>((G + threads - 1) / threads, (int64_t)info.sm_count * std::max(per_sm, 1));
            kernel<<<g2, threads, smem, st>>>(d_codes, d_seq_logprob, G, n, fm, d_none_code != nullptr, d_win_code, d_meta, d_weight);
            KC_CUDA(cudaGetLastError());
            return KC_OK;
        };
        if (n <= 8) return launch(kc::weighted_vote_rec_kernel<8, 128>, 8);
        if (n <= 16) return launch(kc::weighted_vote_rec_kernel<16, 128>, 16);
        if (n <= 32) return launch(kc::weighted_vote_rec_kernel<32, 128>, 32);
        return launch(kc::weighted_vote_rec_kernel<64, 128>, 64);
    }
#define KC_WV(NP) kc::weighted_vote_kernel<NP><<<grid, threads, 0, st>>>(d_codes, d_seq_logprob, G, n, fm, d_none_code != nullptr, d_win_code, d_meta, d_weight)
    if (n <= 2) KC_WV(2);
    else if (n <= 4) KC_WV(4);
    else if (n <= 8) KC_WV(8);
    else if (n <= 16) KC_WV(16);
    else if (n <= 32) KC_WV(32);
    else KC_WV(64);
#undef KC_WV
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_candidate_weights_f32(const float *d_seq_logprob, int64_t n_records, int32_t n, float *d_weight, void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_candidate_weights_f32: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_records < 0) return fail(KC_EINVAL, "kc_candidate_weights_f32: negative n_records");
    if (n_records == 0) return KC_OK;
    if (!d_seq_logprob || !d_weight) return fail(KC_EINVAL, "kc_candidate_weights_f32: NULL buffer");
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int grid = (int)std::min<int64_t>((n_records + 7) / 8, (int64_t)info.sm_count * 8);
    kc::weight_rows_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_seq_logprob, n_records, n, n, d_weight);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

static int weighted_vote_groups(const char *what, const void *d_cells, bool i8, int64_t n_groups, int32_t n, const int32_t *d_group_record,
                                const int8_t *d_cand, const float *d_weight, uint32_t *d_meta, float *d_sums, void *stream) {
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "%s: n=%d outside [1,%d]", what, n, KC_MAX_CANDIDATES);
    if (n_groups < 0) return fail(KC_EINVAL, "%s: negative n_groups", what);
    if (n_groups == 0) return KC_OK;
    if (!d_cells || !d_group_record || !d_weight || !d_meta || !d_sums) return fail(KC_EINVAL, "%s: NULL buffer", what);
    if (((uintptr_t)d_sums) & 7) return fail(KC_EINVAL, "%s: d_sums must be 8-byte aligned", what);
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    const int threads = 128;
    const int grid = (int)std::min<int64_t>((n_groups + threads - 1) / threads, (int64_t)info.sm_count * 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float2 *sums = reinterpret_cast<float2 *>(d_sums);
#define KC_WVG(NP)                                                                                                                              \
    do {                                                                                                                                    \
        if (i8)                                                                                                                             \
            kc::weighted_vote_groups_kernel<NP, int8_t><<<grid, threads, 0, st>>>(static_cast<const int8_t *>(d_cells), n_groups, n,     \
                                                                                  d_group_record, d_cand, d_weight, d_meta, sums);      \
        else                                                                                                                                \
            kc::weighted_vote_groups_kernel<NP, int32_t><<<grid, threads, 0, st>>>(static_cast<const int32_t *>(d_cells), n_groups, n,   \
                                                                                   d_group_record, d_cand, d_weight, d_meta, sums);     \
    } while (0)
    if (n <= 16) KC_WVG(16);  // (an 8-cell instance of the int8 kernel spills 16 bytes: the 16-cell one does not)
    else if (n <= 32) KC_WVG(32);
    else KC_WVG(64);
#undef KC_WVG
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_weighted_vote_groups_i8(const int8_t *d_cells, int64_t n_groups, int32_t n, const int32_t *d_group_record, const int8_t *d_cand,
                               const float *d_weight, uint32_t *d_meta, float *d_sums, void *stream) {
    return weighted_vote_groups("kc_weighted_vote_groups_i8", d_cells, true, n_groups, n, d_group_record, d_cand, d_weight, d_meta, d_sums,
                                stream);
}

int kc_weighted_vote_groups_i32(const int32_t *d_cells, int64_t n_groups, int32_t n, const int32_t *d_group_record, const int8_t *d_cand,
                                const float *d_weight, uint32_t *d_meta, float *d_sums, void *stream) {
    return weighted_vote_groups("kc_weighted_vote_groups_i32", d_cells, false, n_groups, n, d_group_record, d_cand, d_weight, d_meta, d_sums,
                                stream);
}

int kc_medoid_str(const uint8_t *d_chars, const int32_t *d_str_off, const int32_t *d_grp_off, int64_t n_groups,
                  int32_t max_group, int32_t *d_best_idx, double *d_best_avg, void *stream) {
    return kc_medoid_str_method(d_chars, d_str_off, d_grp_off, n_groups, max_group, KC_SIM_LEVENSHTEIN, d_best_idx, d_best_avg, stream);
}

int kc_medoid_str_method(const uint8_t *d_chars, const int32_t *d_str_off, const int32_t *d_grp_off, int64_t n_groups,
                         int32_t max_group, int32_t method, int32_t *d_best_idx, double *d_best_avg, void *stream) {
    if (method < KC_SIM_LEVENSHTEIN || method > KC_SIM_HAMMING) return fail(KC_EINVAL, "kc_medoid_str: unknown similarity method %d", method);
    if (n_groups < 0) return fail(KC_EINVAL, "kc_medoid_str: negative n_groups");
    if (max_group < 2 || max_group > kc::kMedoidMaxN)
        return fail(KC_EINVAL, "kc_medoid_str: max_group=%d outside [2,%d]", max_group, kc::kMedoidMaxN);
    if (n_groups == 0) return KC_OK;
    if (!d_chars || !d_str_off || !d_grp_off || !d_best_idx || !d_best_avg) return fail(KC_EINVAL, "kc_medoid_str: NULL buffer");
    DeviceInfo info;
    int rc = device_info(info);
    if (rc) return rc;
    constexpr int WARPS = 4;
    auto kernel = kc::medoid_kernel<WARPS>;
    const size_t per_warp = (kc::MedoidSmem::bytes(max_group) + 15) & ~size_t(15);  // match tables + distances, sized by max_group
    const size_t smem = WARPS * per_warp;
    KC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS * 32, smem));
    const int grid = (int)std::min<int64_t>((n_groups + WARPS - 1) / WARPS, (int64_t)info.sm_count * std::max(per_sm, 1));
    kernel<<<grid, WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(d_chars, d_str_off, d_grp_off, n_groups, max_group,
                                                                         d_best_idx, d_best_avg, method);
    KC_CUDA(cudaGetLastError());
    return KC_OK;
}

int kc_medoid_str_host(const uint8_t *h_chars, int64_t n_chars, const int32_t *h_str_off, const int32_t *h_grp_off, int64_t n_groups,
                       int32_t max_group, int32_t *h_best_idx, double *h_best_avg, int device) {
    if (n_groups < 0 || n_chars < 0) return fail(KC_EINVAL, "kc_medoid_str_host: negative size");
    if (n_groups == 0) return KC_OK;
    if (!h_str_off || !h_grp_off || !h_best_idx || !h_best_avg || (n_chars && !h_chars)) return fail(KC_EINVAL, "kc_medoid_str_host: NULL buffer");
    KC_CUDA(cudaSetDevice(device));
    const int64_t n_str = h_grp_off[n_groups];
    if (n_str < 0 || h_str_off[n_str] != n_chars) return fail(KC_EINVAL, "kc_medoid_str_host: offsets do not add up to n_chars");
    const size_t b_chars = ((size_t)n_chars + 255) & ~size_t(255), b_str = (((size_t)n_str + 1) * 4 + 255) & ~size_t(255),
                 b_grp = (((size_t)n_groups + 1) * 4 + 255) & ~size_t(255), b_idx = ((size_t)n_groups * 4 + 255) & ~size_t(255),
                 b_avg = (size_t)n_groups * 8;
    uint8_t *d = nullptr;
    KC_CUDA(cudaMalloc(&d, b_chars + b_str + b_grp + b_idx + b_avg + 256));
    uint8_t *d_chars = d, *d_str = d + b_chars + 256, *d_grp = d_str + b_str, *d_idx = d_grp + b_grp, *d_avg = d_idx + b_idx;
    int rc = KC_OK;
    cudaStream_t st = nullptr;
    auto guard = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && rc == KC_OK) rc = fail(KC_ECUDA, "kc_medoid_str_host: %s: %s", what, cudaGetErrorString(e));
    };
    guard(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "stream");
    if (n_chars) guard(cudaMemcpyAsync(d_chars, h_chars, (size_t)n_chars, cudaMemcpyHostToDevice, st), "H2D chars");
    guard(cudaMemcpyAsync(d_str, h_str_off, ((size_t)n_str + 1) * 4, cudaMemcpyHostToDevice, st), "H2D str_off");
    guard(cudaMemcpyAsync(d_grp, h_grp_off, ((size_t)n_groups + 1) * 4, cudaMemcpyHostToDevice, st), "H2D grp_off");
    if (rc == KC_OK)
        rc = kc_medoid_str(d_chars, reinterpret_cast<int32_t *>(d_str), reinterpret_cast<int32_t *>(d_grp), n_groups, max_group,
                           reinterpret_cast<int32_t *>(d_idx), reinterpret_cast<double *>(d_avg), st);
    guard(cudaMemcpyAsync(h_best_idx, d_idx, (size_t)n_groups * 4, cudaMemcpyDeviceToHost, st), "D2H idx");
    guard(cudaMemcpyAsync(h_best_avg, d_avg, (size_t)n_groups * 8, cudaMemcpyDeviceToHost, st), "D2H avg");
    if (st) {
        guard(cudaStreamSynchronize(st), "sync");
        cudaStreamDestroy(st);
    }
    cudaFree(d);
    return rc;
}

void *kc_host_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void kc_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ---------------------------------------------------------------- end-to-end with host buffers

static int consensus_host_impl(const void *h_codes_v, int code_bytes, int32_t n_vote_fields, const int32_t *h_none_code,
                               const double *h_vals, int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps,
                               double abs_eps, int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value,
                               uint32_t *h_num_meta, int device, float *device_ms);

int kc_consensus_host(const int32_t *h_codes, int32_t n_vote_fields, const int32_t *h_none_code, const double *h_vals,
                      int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                      int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value, uint32_t *h_num_meta, int device,
                      float *device_ms) {
    return consensus_host_impl(h_codes, 4, n_vote_fields, h_none_code, h_vals, n_num_fields, n_records, n, rel_eps, abs_eps,
                               h_win_code, h_vote_meta, h_value, h_num_meta, device, device_ms);
}

int kc_consensus_host_i8(const int8_t *h_codes, int32_t n_vote_fields, const int32_t *h_none_code, const double *h_vals,
                         int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                         int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value, uint32_t *h_num_meta, int device,
                         float *device_ms) {
    return consensus_host_impl(h_codes, 1, n_vote_fields, h_none_code, h_vals, n_num_fields, n_records, n, rel_eps, abs_eps,
                               h_win_code, h_vote_meta, h_value, h_num_meta, device, device_ms);
}

static int consensus_host_impl(const void *h_codes_v, int code_bytes, int32_t n_vote_fields, const int32_t *h_none_code,
                               const double *h_vals, int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps,
                               double abs_eps, int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value,
                               uint32_t *h_num_meta, int device, float *device_ms) {
    const uint8_t *h_codes = static_cast<const uint8_t *>(h_codes_v);
    if (device_ms) *device_ms = 0.0f;
    if (n < 1 || n > KC_MAX_CANDIDATES) return fail(KC_EINVAL, "kc_consensus_host: n=%d outside [1,%d]", n, KC_MAX_CANDIDATES);
    if (n_records < 0 || n_vote_fields < 0 || n_num_fields < 0) return fail(KC_EINVAL, "kc_consensus_host: negative size");
    if (device < 0 || device >= 16) return fail(KC_EINVAL, "kc_consensus_host: device %d out of range", device);
    if (n_vote_fields > 0 && (!h_codes || !h_win_code || !h_vote_meta)) return fail(KC_EINVAL, "kc_consensus_host: NULL vote buffer");
    if (n_num_fields > 0 && (!h_vals || !h_value || !h_num_meta)) return fail(KC_EINVAL, "kc_consensus_host: NULL numeric buffer");
    if (n_records == 0 || (n_vote_fields == 0 && n_num_fields == 0)) return KC_OK;

    std::lock_guard<std::mutex> lock(g_host_mu);
    int prev = 0;
    KC_CUDA(cudaGetDevice(&prev));
    KC_CUDA(cudaSetDevice(device));
    HostCtx &cx = g_host[device];
    int rc = KC_OK;
    auto finish = [&](int code) {
        cudaSetDevice(prev);
        return code;
    };
    if (cx.device != device) {
        for (auto &s : cx.streams)
            if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return finish(fail(KC_ECUDA, "cudaStreamCreate failed"));
        cx.device = device;
    }
    // chunk: ~48 MiB of input per stream buffer keeps H2D, kernels and D2H of neighbouring chunks overlapped
    const size_t rec_in = (size_t)n * ((size_t)n_vote_fields * code_bytes + (size_t)n_num_fields * 8);
    int64_t chunk = std::max<int64_t>(1024, (int64_t)((48u << 20) / std::max<size_t>(rec_in, 1)));
    chunk = std::min<int64_t>(chunk, n_records);
    chunk = (chunk + 255) / 256 * 256;
    for (int s = 0; s < HostCtx::kStreams && !rc; ++s) {
        if (n_vote_fields) {
            rc = cx.codes[s].reserve((size_t)chunk * n_vote_fields * n * code_bytes);
            if (!rc) rc = cx.win[s].reserve((size_t)chunk * n_vote_fields * 4);
            if (!rc) rc = cx.vmeta[s].reserve((size_t)chunk * n_vote_fields * 4);
        }
        if (n_num_fields && !rc) {
            rc = cx.vals[s].reserve((size_t)chunk * n_num_fields * n * 8);
            if (!rc) rc = cx.value[s].reserve((size_t)chunk * n_num_fields * 8);
            if (!rc) rc = cx.nmeta[s].reserve((size_t)chunk * n_num_fields * 4);
        }
    }
    if (rc) return finish(rc);
    const int32_t *d_none = nullptr;
    if (h_none_code && n_vote_fields) {
        rc = cx.none.reserve((size_t)n_vote_fields * 4);
        if (rc) return finish(rc);
        if (cudaMemcpyAsync(cx.none.p, h_none_code, (size_t)n_vote_fields * 4, cudaMemcpyHostToDevice, cx.streams[0]) != cudaSuccess ||
            cudaStreamSynchronize(cx.streams[0]) != cudaSuccess)
            return finish(fail(KC_ECUDA, "none_code upload failed: %s", cudaGetErrorString(cudaGetLastError())));
        d_none = cx.none.as<int32_t>();
    }
    // device-side timing of the whole call: start on stream 0 before the first copy; stop on stream 0 after it has
    // waited for the other streams' last work
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_join[HostCtx::kStreams] = {};
    if (device_ms) {
        cudaEventCreate(&ev_start);
        cudaEventCreate(&ev_stop);
        for (auto &e : ev_join) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        cudaEventRecord(ev_start, cx.streams[0]);
        for (int s = 1; s < HostCtx::kStreams; ++s) cudaStreamWaitEvent(cx.streams[s], ev_start, 0);  // nothing starts earlier
    }
    int64_t r0 = 0;
    for (int it = 0; r0 < n_records && !rc; ++it, r0 += chunk) {
        const int s = it % HostCtx::kStreams;
        cudaStream_t st = cx.streams[s];
        const int64_t nr = std::min(chunk, n_records - r0);
        cudaError_t e = cudaSuccess;
        nvtxRangePushA("kc_consensus_host: chunk (H2D, K1, K2, D2H)");
        if (n_vote_fields) {
            const int64_t G = nr * n_vote_fields;
            e = cudaMemcpyAsync(cx.codes[s].p, h_codes + (size_t)r0 * n_vote_fields * n * code_bytes, (size_t)G * n * code_bytes,
                                cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                rc = code_bytes == 1
                         ? kc_vote_i8(cx.codes[s].as<int8_t>(), G, n, d_none, n_vote_fields, cx.win[s].as<int32_t>(), cx.vmeta[s].as<uint32_t>(), st)
                         : kc_vote_i32(cx.codes[s].as<int32_t>(), G, n, d_none, n_vote_fields, cx.win[s].as<int32_t>(), cx.vmeta[s].as<uint32_t>(), st);
                if (rc) { nvtxRangePop(); break; }
                e = cudaMemcpyAsync(h_win_code + r0 * n_vote_fields, cx.win[s].as<int32_t>(), (size_t)G * 4, cudaMemcpyDeviceToHost, st);
            }
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(h_vote_meta + r0 * n_vote_fields, cx.vmeta[s].as<uint32_t>(), (size_t)G * 4, cudaMemcpyDeviceToHost, st);
        }
        if (n_num_fields && e == cudaSuccess) {
            const int64_t G = nr * n_num_fields;
            e = cudaMemcpyAsync(cx.vals[s].as<double>(), h_vals + r0 * n_num_fields * n, (size_t)G * n * 8, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                rc = kc_numeric_f64(cx.vals[s].as<double>(), G, n, rel_eps, abs_eps, cx.value[s].as<double>(), cx.nmeta[s].as<uint32_t>(), st);
                if (rc) { nvtxRangePop(); break; }
                e = cudaMemcpyAsync(h_value + r0 * n_num_fields, cx.value[s].as<double>(), (size_t)G * 8, cudaMemcpyDeviceToHost, st);
            }
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(h_num_meta + r0 * n_num_fields, cx.nmeta[s].as<uint32_t>(), (size_t)G * 4, cudaMemcpyDeviceToHost, st);
        }
        nvtxRangePop();
        if (e != cudaSuccess) rc = fail(KC_ECUDA, "kc_consensus_host: %s", cudaGetErrorString(e));
    }
    if (device_ms) {
        for (int s = 1; s < HostCtx::kStreams; ++s) {
            cudaEventRecord(ev_join[s], cx.streams[s]);
            cudaStreamWaitEvent(cx.streams[0], ev_join[s], 0);
        }
        cudaEventRecord(ev_stop, cx.streams[0]);
    }
    for (auto &s : cx.streams) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && !rc) rc = fail(KC_ECUDA, "kc_consensus_host sync: %s", cudaGetErrorString(e));
    }
    if (device_ms) {
        if (!rc) cudaEventElapsedTime(device_ms, ev_start, ev_stop);
        cudaEventDestroy(ev_start);
        cudaEventDestroy(ev_stop);
        for (auto &e : ev_join) cudaEventDestroy(e);
    }
    return finish(rc);
}

}  // extern "C"
