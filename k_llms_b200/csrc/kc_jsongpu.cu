// kc_jsongpu.cu — host side of H1g (kc_jsongpu.cuh): kc_consolidate_json_packed() streams a batch of candidate texts through
// the device JSON path in chunks (H2D -> A0 -> A1 -> K1/K2 -> C0 -> C1 -> D2H, several chunks in flight on their own streams),
// hands the records the device path declined to the host path (kc_consolidate_json), and returns the consensus / likelihoods
// texts as one blob with per-record spans.  Also the kc_debug_jsongpu_* test hooks, which run the SAME phase functions on
// the host so the CPU tests can check the logic against the oracle without a GPU (they are not a product path: the product
// entry needs a device and fails without one).
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_scan.cuh>
#include <nvtx3/nvToolsExt.h>  // header-only; ranges show up in Nsight Systems / ncu --nvtx, cost nothing otherwise

#include "../../include/kllms_b200.h"
#include "kc_internal.h"
#include "kc_jsongpu.cuh"

namespace {

using kc::js::Chunk;
using kc::js::Tok;

struct DBuf {  // grow-only device buffer
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t need) {
        if (p && need <= cap) return KC_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        need += need / 8 + 256;
        if (cudaMalloc(&p, need) != cudaSuccess) {
            cudaGetLastError();
            return kc_fail(KC_ENOMEM, "kc_consolidate_json_packed: cudaMalloc(%zu) failed", need);
        }
        cap = need;
        return KC_OK;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};

struct PBuf {  // grow-only pinned host buffer
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t need) {
        if (p && need <= cap) return KC_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        need += need / 8 + 256;
        if (cudaHostAlloc(&p, need, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            return kc_fail(KC_ENOMEM, "kc_consolidate_json_packed: cudaHostAlloc(%zu) failed", need);
        }
        cap = need;
        return KC_OK;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};

// Everything one in-flight chunk needs on the device.  Workers are pooled per device and reused across calls.
struct Worker {
    int device = -1;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[7] = {};
    DBuf text, off, fcount, slot, status, vbase, xbase, counters, toks, fdesc, piece_c, piece_l, vcells, xcells, win, vmeta, xvalue, xmeta,
        len_c, len_l, out_c, out_l, scan_tmp, mcount, scount, ccount, mchars, mstr_off, mgrp_off, midx, mavg, nest, gpos,
        lp, lp_off, seq_lp, cand_w, vrec, vsums;  // the last six: likelihood-weighted entry only
    PBuf h_small;  // totals and counters (pinned so the small D2H copies are asynchronous)
    PBuf h_scan;   // the scanned record offsets and the statuses of a chunk
    bool busy = false;
    int init(int dev) {
        if (device == dev) return KC_OK;
        KC_CUDA_I(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (auto &e : ev) KC_CUDA_I(cudaEventCreate(&e));
        device = dev;
        return KC_OK;
    }
};

std::mutex g_pool_mu;
std::vector<Worker *> g_workers;  // never freed: device buffers live as long as the process

Worker *acquire_worker(int device) {
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (Worker *w : g_workers)
        if (!w->busy && w->device == device) {
            w->busy = true;
            return w;
        }
    Worker *w = new Worker;
    w->busy = true;
    g_workers.push_back(w);
    return w;
}
void release_worker(Worker *w) {
    std::lock_guard<std::mutex> lock(g_pool_mu);
    w->busy = false;
}

// pinned output blobs are expensive to create (page-locking): recycle them across calls
struct PinnedBlob {
    char *p = nullptr;
    size_t cap = 0;
};
std::vector<PinnedBlob> g_blob_pool;

PinnedBlob acquire_blob(size_t need) {
    {
        std::lock_guard<std::mutex> lock(g_pool_mu);
        int best = -1;
        for (int i = 0; i < (int)g_blob_pool.size(); ++i)
            if (g_blob_pool[i].cap >= need && (best < 0 || g_blob_pool[i].cap < g_blob_pool[best].cap)) best = i;
        if (best >= 0) {
            PinnedBlob b = g_blob_pool[best];
            g_blob_pool.erase(g_blob_pool.begin() + best);
            return b;
        }
    }
    PinnedBlob b;
    void *p = nullptr;
    if (cudaHostAlloc(&p, need, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return b;
    }
    b.p = (char *)p;
    b.cap = need;
    return b;
}
void release_blob(PinnedBlob b) {
    if (!b.p) return;
    std::lock_guard<std::mutex> lock(g_pool_mu);
    // small blobs (single requests, many callers at once) are cheap to keep: up to 64 of them; of the large ones the largest four
    size_t n_small = 0, n_large = 0;
    for (auto &x : g_blob_pool) (x.cap <= ((size_t)4 << 20) ? n_small : n_large)++;
    if (b.cap <= ((size_t)4 << 20) && n_small < 64) {
        g_blob_pool.push_back(b);
        return;
    }
    if (n_large >= 4 || b.cap <= ((size_t)4 << 20)) {
        int smallest = -1;
        for (int i = 0; i < (int)g_blob_pool.size(); ++i)
            if (g_blob_pool[i].cap > ((size_t)4 << 20) && (smallest < 0 || g_blob_pool[i].cap < g_blob_pool[smallest].cap)) smallest = i;
        if (smallest < 0 || g_blob_pool[smallest].cap >= b.cap) {
            cudaFreeHost(b.p);
            return;
        }
        cudaFreeHost(g_blob_pool[smallest].p);
        g_blob_pool.erase(g_blob_pool.begin() + smallest);
    }
    g_blob_pool.push_back(b);
}

int team_size(int n) {
    int t = 2;
    while (t < n && t < 32) t *= 2;
    return t;
}

}  // namespace

struct kc_json_result {
    int64_t R = 0;
    PinnedBlob blob;                   // GPU-written texts (and host-path texts while they fit)
    std::atomic<int64_t> used{0};
    std::vector<int64_t> c_off, c_len, l_off, l_len;
    std::vector<uint8_t> status, why;
    std::string heap;                  // rare: the texts when the host path's share did not fit the pinned blob
    kc_json_stats stats{};
};

namespace {

struct ChunkStage {  // per-chunk device-time split (CUDA events on the chunk's stream)
    float h2d = 0, plan = 0, kernels = 0, emit = 0, d2h = 0;
};

__global__ void rebase_kernel(int64_t *off, int64_t count, int64_t base) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) off[i] -= base;
}

// One chunk on one worker: records [r0, r1) of the batch.  h_lp / h_lp_off non-NULL: the likelihood-weighted vote (K3, the weight
// pre-pass and kc_weighted_vote_groups_i8 in K1's place).
int run_chunk(Worker &w, const char *h_text, const int64_t *h_off, const float *h_lp, const int64_t *h_lp_off, int64_t r0, int64_t r1,
              int32_t n, double rel_eps, double abs_eps, int sm_count, kc_json_result &res, ChunkStage &st) {
    const int64_t Rc = r1 - r0;
    const int64_t b0 = h_off[r0 * n], b1 = h_off[r1 * n];
    const size_t bytes = (size_t)(b1 - b0);
    if (bytes >= ((size_t)1 << 32)) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed: chunk of %zu bytes", bytes);
    cudaStream_t s = w.stream;
    int rc;
#define R_(call)          \
    do {                  \
        rc = (call);      \
        if (rc) return rc; \
    } while (0)
    R_(w.text.reserve(bytes + 16));
    R_(w.off.reserve((size_t)(Rc * n + 1) * 8));
    R_(w.fcount.reserve((size_t)(Rc + 1) * 4));
    R_(w.slot.reserve((size_t)(Rc + 1) * 4));
    R_(w.status.reserve((size_t)Rc));
    R_(w.nest.reserve((size_t)Rc));
    R_(w.vbase.reserve((size_t)Rc * 4));
    R_(w.xbase.reserve((size_t)Rc * 4));
    R_(w.counters.reserve(32));
    R_(w.mcount.reserve((size_t)(Rc + 1) * 4));
    R_(w.scount.reserve((size_t)(Rc + 1) * 4));
    R_(w.ccount.reserve((size_t)(Rc + 1) * 4));
    R_(w.len_c.reserve((size_t)(Rc + 1) * 8));
    R_(w.len_l.reserve((size_t)(Rc + 1) * 8));
    R_(w.h_small.reserve(64));
    R_(w.h_scan.reserve((size_t)(Rc + 1) * 16 + (size_t)Rc));
    size_t tmp_bytes = 0, tmp_bytes32 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const int64_t *)nullptr, (int64_t *)nullptr, (int)(Rc + 1), s);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes32, (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)(Rc + 1), s);
    R_(w.scan_tmp.reserve(std::max(tmp_bytes, tmp_bytes32) + 256));

    Chunk ch{};
    ch.text = w.text.as<uint8_t>();
    ch.off = w.off.as<int64_t>();
    ch.R = (int32_t)Rc;
    ch.n = n;
    ch.fcount = w.fcount.as<uint32_t>();
    ch.slot = w.slot.as<uint32_t>();
    ch.status = w.status.as<uint8_t>();
    ch.nest = w.nest.as<uint8_t>();
    ch.vbase = w.vbase.as<uint32_t>();
    ch.xbase = w.xbase.as<uint32_t>();
    ch.counters = w.counters.as<unsigned long long>();
    ch.mcount = w.mcount.as<uint32_t>();
    ch.scount = w.scount.as<uint32_t>();
    ch.ccount = w.ccount.as<uint32_t>();
    ch.len_c = w.len_c.as<int64_t>();
    ch.len_l = w.len_l.as<int64_t>();

    nvtxRangePushA("kc_json: H2D texts");
    KC_CUDA_I(cudaEventRecord(w.ev[0], s));
    KC_CUDA_I(cudaMemcpyAsync(w.text.p, h_text + b0, bytes, cudaMemcpyHostToDevice, s));
    KC_CUDA_I(cudaMemcpyAsync(w.off.p, h_off + r0 * n, (size_t)(Rc * n + 1) * 8, cudaMemcpyHostToDevice, s));
    const bool weighted = h_lp_off != nullptr;
    const int64_t l0 = weighted ? h_lp_off[r0 * n] : 0, n_tok = weighted ? h_lp_off[r1 * n] - l0 : 0;
    if (weighted) {  // the chunk's token logprobs next to its texts, their offsets rebased to the chunk
        R_(w.lp.reserve((size_t)std::max<int64_t>(n_tok, 4) * 4));
        R_(w.lp_off.reserve((size_t)(Rc * n + 1) * 8));
        R_(w.seq_lp.reserve((size_t)Rc * n * 4));
        R_(w.cand_w.reserve((size_t)Rc * n * 4));
        if (n_tok) KC_CUDA_I(cudaMemcpyAsync(w.lp.p, h_lp + l0, (size_t)n_tok * 4, cudaMemcpyHostToDevice, s));
        KC_CUDA_I(cudaMemcpyAsync(w.lp_off.p, h_lp_off + r0 * n, (size_t)(Rc * n + 1) * 8, cudaMemcpyHostToDevice, s));
        rebase_kernel<<<(int)std::min<int64_t>((Rc * n + 256) / 256, (int64_t)sm_count * 4), 256, 0, s>>>(w.lp_off.as<int64_t>(), Rc * n + 1, l0);
        KC_CUDA_I(cudaGetLastError());
    }
    KC_CUDA_I(cudaEventRecord(w.ev[1], s));
    nvtxRangePop();
    nvtxRangePushA("kc_json: plan (A0 count, A1 scan/type/encode)");

    const int team = team_size(n);
    const int tpw = 32 / team;
    auto grid_for = [&](int64_t threads_needed) {
        const int64_t blocks = (threads_needed + 127) / 128;
        return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)sm_count * 16));
    };
    // A0: fields per record, then their exclusive scan (entry Rc of fcount is 0, so slot[Rc] is the total)
    KC_CUDA_I(cudaMemsetAsync(ch.fcount + Rc, 0, 4, s));
    kc::js::count_kernel<<<grid_for(Rc), 128, 0, s>>>(ch);
    KC_CUDA_I(cudaGetLastError());
    size_t tb = w.scan_tmp.cap;
    KC_CUDA_I(cub::DeviceScan::ExclusiveSum(w.scan_tmp.p, tb, (const uint32_t *)ch.fcount, ch.slot, (int)(Rc + 1), s));
    uint32_t *h_total = w.h_small.as<uint32_t>();
    KC_CUDA_I(cudaMemcpyAsync(h_total, ch.slot + Rc, 4, cudaMemcpyDeviceToHost, s));
    KC_CUDA_I(cudaStreamSynchronize(s));
    const size_t T = *h_total;  // field slots of the chunk
    const size_t Tn = T * (size_t)n;
    R_(w.toks.reserve(std::max<size_t>(Tn, 1) * sizeof(Tok)));
    R_(w.fdesc.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.gpos.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.piece_c.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.piece_l.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.vcells.reserve(std::max<size_t>(Tn, 16)));
    R_(w.xcells.reserve(std::max<size_t>(Tn, 2) * 8));
    R_(w.win.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.vmeta.reserve(std::max<size_t>(T, 1) * 4));
    R_(w.xvalue.reserve(std::max<size_t>(T, 1) * 8));
    R_(w.xmeta.reserve(std::max<size_t>(T, 1) * 4));
    if (weighted) {  // a record has at most one vote group per field slot
        R_(w.vrec.reserve(std::max<size_t>(T, 1) * 4));
        R_(w.vsums.reserve(std::max<size_t>(T, 1) * 8));
        ch.vrec = w.vrec.as<int32_t>();
    }
    ch.toks = w.toks.as<Tok>();
    ch.fdesc = w.fdesc.as<uint32_t>();
    ch.gpos = w.gpos.as<uint32_t>();
    ch.piece_c = w.piece_c.as<uint32_t>();
    ch.piece_l = w.piece_l.as<uint32_t>();
    ch.vcells = w.vcells.as<int8_t>();
    ch.xcells = w.xcells.as<double>();
    ch.vmeta = w.vmeta.as<uint32_t>();
    ch.xvalue = w.xvalue.as<double>();
    ch.xmeta = w.xmeta.as<uint32_t>();
    KC_CUDA_I(cudaMemsetAsync(w.counters.p, 0, 24, s));
    // records declined before slots_phase own no medoid groups
    KC_CUDA_I(cudaMemsetAsync(w.mcount.p, 0, (size_t)(Rc + 1) * 4, s));
    KC_CUDA_I(cudaMemsetAsync(w.scount.p, 0, (size_t)(Rc + 1) * 4, s));
    KC_CUDA_I(cudaMemsetAsync(w.ccount.p, 0, (size_t)(Rc + 1) * 4, s));
    // rows reserved by a record that is declined while encoding stay untouched: give them defined contents
    KC_CUDA_I(cudaMemsetAsync(w.vcells.p, 0xFF, std::max<size_t>(Tn, 16), s));
    KC_CUDA_I(cudaMemsetAsync(w.xcells.p, 0, std::max<size_t>(Tn, 2) * 8, s));
    int64_t gv = 0, gx = 0, gm = 0;
    if (T) {
        const int64_t rounds = (Rc + tpw - 1) / tpw;
        kc::js::plan_kernel<<<grid_for(rounds * 32), 128, 0, s>>>(ch, team);
        KC_CUDA_I(cudaGetLastError());
        unsigned long long *h_cnt = w.h_small.as<unsigned long long>() + 1;
        KC_CUDA_I(cudaMemcpyAsync(h_cnt, w.counters.p, 24, cudaMemcpyDeviceToHost, s));
        KC_CUDA_I(cudaStreamSynchronize(s));
        gv = (int64_t)h_cnt[0];
        gx = (int64_t)h_cnt[1];
        gm = (int64_t)h_cnt[2];
    }
    if (gm) {
        // A2: multi-word string fields -> K4's CSR input.  Sizes by upper bound (no read-back): the normalised characters are a
        // subset of the chunk's text, a group has at most n strings, a record at most fcount groups.
        R_(w.mchars.reserve(bytes + 16));
        R_(w.mstr_off.reserve((Tn + 2) * 4));
        R_(w.mgrp_off.reserve((T + 2) * 4));
        R_(w.midx.reserve((T + 1) * 4));
        R_(w.mavg.reserve((T + 1) * 8));
        ch.mchars = w.mchars.as<uint8_t>();
        ch.mstr_off = w.mstr_off.as<int32_t>();
        ch.mgrp_off = w.mgrp_off.as<int32_t>();
        ch.midx = w.midx.as<int32_t>();
        ch.mavg = w.mavg.as<double>();
        for (uint32_t *cnt : {ch.mcount, ch.scount, ch.ccount}) {
            tb = w.scan_tmp.cap;
            KC_CUDA_I(cub::DeviceScan::ExclusiveSum(w.scan_tmp.p, tb, (const uint32_t *)cnt, cnt, (int)(Rc + 1), s));
        }
        const int64_t rounds = (Rc + tpw - 1) / tpw;
        kc::js::medoid_kernel<<<grid_for(rounds * 32), 128, 0, s>>>(ch, team);
        KC_CUDA_I(cudaGetLastError());
    }
    KC_CUDA_I(cudaEventRecord(w.ev[2], s));
    nvtxRangePop();
    nvtxRangePushA("kc_json: K1 vote + K2 numeric + K4 medoid");
    // K1 / K2 / K4: the same kernels as the columnar path (one "field" per group: local codes, no none_code table)
    if (weighted) {  // K3 -> candidate weights -> the weighted vote (DESIGN.md §5); the logprob sums of the whole chunk are cheap
        R_(kc_logprob_sum_f32(w.lp.as<float>(), w.lp_off.as<int64_t>(), Rc * n, w.seq_lp.as<float>(), s));
        R_(kc_candidate_weights_f32(w.seq_lp.as<float>(), Rc, n, w.cand_w.as<float>(), s));
        if (gv) R_(kc_weighted_vote_groups_i8(ch.vcells, gv, n, ch.vrec, nullptr, w.cand_w.as<float>(), w.vmeta.as<uint32_t>(), w.vsums.as<float>(), s));
        ch.vsums = w.vsums.as<float>();
    } else if (gv) {
        R_(kc_vote_i8(ch.vcells, gv, n, nullptr, 1, w.win.as<int32_t>(), w.vmeta.as<uint32_t>(), s));
    }
    if (gx) R_(kc_numeric_f64(ch.xcells, gx, n, rel_eps, abs_eps, w.xvalue.as<double>(), w.xmeta.as<uint32_t>(), s));
    if (gm) R_(kc_medoid_str(ch.mchars, ch.mstr_off, ch.mgrp_off, gm, std::max(2, n), w.midx.as<int32_t>(), w.mavg.as<double>(), s));
    KC_CUDA_I(cudaEventRecord(w.ev[3], s));
    nvtxRangePop();
    nvtxRangePushA("kc_json: emit (C0 lengths, C1 write)");
    // C0: piece lengths and record lengths, then record offsets in the two output blobs
    KC_CUDA_I(cudaMemsetAsync(ch.len_c + Rc, 0, 8, s));
    KC_CUDA_I(cudaMemsetAsync(ch.len_l + Rc, 0, 8, s));
    {
        const int64_t rounds = (Rc + tpw - 1) / tpw;
        kc::js::len_kernel<<<grid_for(rounds * 32), 128, 0, s>>>(ch, team);
        KC_CUDA_I(cudaGetLastError());
    }
    tb = w.scan_tmp.cap;
    KC_CUDA_I(cub::DeviceScan::ExclusiveSum(w.scan_tmp.p, tb, (const int64_t *)ch.len_c, ch.len_c, (int)(Rc + 1), s));
    tb = w.scan_tmp.cap;
    KC_CUDA_I(cub::DeviceScan::ExclusiveSum(w.scan_tmp.p, tb, (const int64_t *)ch.len_l, ch.len_l, (int)(Rc + 1), s));
    int64_t *h_scan_c = w.h_scan.as<int64_t>(), *h_scan_l = h_scan_c + (Rc + 1);
    uint8_t *h_status = (uint8_t *)(h_scan_l + (Rc + 1));
    KC_CUDA_I(cudaMemcpyAsync(h_scan_c, ch.len_c, (size_t)(Rc + 1) * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_I(cudaMemcpyAsync(h_scan_l, ch.len_l, (size_t)(Rc + 1) * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_I(cudaMemcpyAsync(h_status, ch.status, (size_t)Rc, cudaMemcpyDeviceToHost, s));
    KC_CUDA_I(cudaStreamSynchronize(s));
    const int64_t out_c_bytes = h_scan_c[Rc], out_l_bytes = h_scan_l[Rc];
    R_(w.out_c.reserve((size_t)std::max<int64_t>(out_c_bytes, 1)));
    R_(w.out_l.reserve((size_t)std::max<int64_t>(out_l_bytes, 1)));
    ch.out_c = w.out_c.as<uint8_t>();
    ch.out_l = w.out_l.as<uint8_t>();
    if (out_c_bytes) {
        const int64_t rounds = (Rc + tpw - 1) / tpw;
        kc::js::write_kernel<<<grid_for(rounds * 32), 128, 0, s>>>(ch, team);
        KC_CUDA_I(cudaGetLastError());
    }
    KC_CUDA_I(cudaEventRecord(w.ev[4], s));
    nvtxRangePop();
    nvtxRangePushA("kc_json: D2H texts");
    // the chunk's region of the result blob
    const int64_t need = out_c_bytes + out_l_bytes;
    const int64_t pos = res.used.fetch_add(need);
    if (pos + need > (int64_t)res.blob.cap) {  // the estimate of the output size was too small: leave the chunk to the host path
        res.used.fetch_sub(need);
        for (int64_t r = r0; r < r1; ++r) {
            res.status[(size_t)r] = 1;
            res.why[(size_t)r] = (uint8_t)kc::js::D_TOO_LONG;
        }
        return KC_OK;
    }
    if (out_c_bytes) KC_CUDA_I(cudaMemcpyAsync(res.blob.p + pos, ch.out_c, (size_t)out_c_bytes, cudaMemcpyDeviceToHost, s));
    if (out_l_bytes) KC_CUDA_I(cudaMemcpyAsync(res.blob.p + pos + out_c_bytes, ch.out_l, (size_t)out_l_bytes, cudaMemcpyDeviceToHost, s));
    KC_CUDA_I(cudaEventRecord(w.ev[5], s));
    KC_CUDA_I(cudaStreamSynchronize(s));
    nvtxRangePop();
    for (int64_t i = 0; i < Rc; ++i) {
        const int64_t r = r0 + i;
        res.status[(size_t)r] = h_status[i] ? 1 : 0;
        res.why[(size_t)r] = h_status[i];
        res.c_off[(size_t)r] = pos + h_scan_c[i];
        res.c_len[(size_t)r] = h_scan_c[i + 1] - h_scan_c[i];
        res.l_off[(size_t)r] = pos + out_c_bytes + h_scan_l[i];
        res.l_len[(size_t)r] = h_scan_l[i + 1] - h_scan_l[i];
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, w.ev[0], w.ev[1]); st.h2d += ms;
    cudaEventElapsedTime(&ms, w.ev[1], w.ev[2]); st.plan += ms;
    cudaEventElapsedTime(&ms, w.ev[2], w.ev[3]); st.kernels += ms;
    cudaEventElapsedTime(&ms, w.ev[3], w.ev[4]); st.emit += ms;
    cudaEventElapsedTime(&ms, w.ev[4], w.ev[5]); st.d2h += ms;
#undef R_
    return KC_OK;
}

}  // namespace

namespace {

// kc_consolidate_json_packed (h_lp_off == NULL) and kc_consolidate_json_packed_weighted: one implementation
int consolidate_packed(const char *h_text, const int64_t *h_off, const float *h_lp, const int64_t *h_lp_off, int64_t n_records, int32_t n,
                       double rel_eps, double abs_eps, int device, int32_t threads, uint32_t flags, kc_json_result **out) {
    if (!out) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed: NULL out");
    *out = nullptr;
    if (n < 2 || n > KC_MAX_CANDIDATES) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed: n=%d outside [2,%d]", n, KC_MAX_CANDIDATES);
    if (n_records < 0 || (n_records && (!h_text || !h_off))) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed: bad arguments");
    if (!(rel_eps >= 0.0) || !(abs_eps >= 0.0)) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed: rel_eps/abs_eps must be >= 0");
    const bool weighted = h_lp_off != nullptr;
    int64_t lp_bytes = 0;
    if (weighted && n_records) {
        if (h_lp_off[0] < 0) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed_weighted: negative logprob offset");
        for (int64_t i = 0; i < n_records * n; ++i)
            if (h_lp_off[i + 1] < h_lp_off[i]) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed_weighted: logprob offsets descend at %lld", (long long)i);
        lp_bytes = (h_lp_off[n_records * n] - h_lp_off[0]) * 4;
        if (lp_bytes && !h_lp) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed_weighted: NULL logprobs");
        flags |= KC_JSON_DEVICE_ONLY;  // the host path H1 does not weight: declined records are left to the caller
    }
    const auto t_start = std::chrono::steady_clock::now();
    int prev = 0;
    KC_CUDA_I(cudaGetDevice(&prev));
    KC_CUDA_I(cudaSetDevice(device));
    int sm_count = 0, cc_major = 0;
    KC_CUDA_I(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    KC_CUDA_I(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    if (cc_major != 10) {
        cudaSetDevice(prev);
        return kc_fail(KC_ENODEV, "device %d has compute capability %d.x; this library is sm_100a only", device, cc_major);
    }
    kc_json_result *res = new (std::nothrow) kc_json_result;
    if (!res) return kc_fail(KC_ENOMEM, "kc_consolidate_json_packed: out of memory");
    const int64_t R = n_records;
    res->R = R;
    res->c_off.assign((size_t)R, 0);
    res->c_len.assign((size_t)R, 0);
    res->l_off.assign((size_t)R, 0);
    res->l_len.assign((size_t)R, 0);
    res->status.assign((size_t)R, 1);
    res->why.assign((size_t)R, 0);
    const int64_t total_bytes = R ? h_off[R * n] - h_off[0] : 0;
    // The consensus of a record is about one candidate long and its likelihoods about as long again (numbers can grow:
    // "5" -> "5.0", 17-digit means).  A chunk whose output does not fit what is left is handed to the host path.
    res->blob = acquire_blob((size_t)(total_bytes / n * 3 + (1 << 20)));  // small requests all ask for ~1 MiB: the pool's blobs fit
    if (!res->blob.p) {
        delete res;
        cudaSetDevice(prev);
        return kc_fail(KC_ENOMEM, "kc_consolidate_json_packed: cannot allocate the pinned output blob");
    }
    // chunks of ~chunk_mb of text; records are never split
    size_t chunk_bytes = (size_t)64 << 20;
    if (const char *e = getenv("KC_JSON_CHUNK_MB")) chunk_bytes = (size_t)std::min(1024, std::max(1, atoi(e))) << 20;  // K4's CSR offsets are int32
    std::vector<int64_t> cuts{0};
    {
        int64_t r = 0;
        while (r < R) {
            // records are a few KB: advance by estimate, then adjust
            // the chunk's bytes: its texts, and with weighting its token logprobs
            auto span = [&](int64_t a, int64_t b) -> size_t {
                return (size_t)(h_off[b * n] - h_off[a * n]) + (weighted ? (size_t)(h_lp_off[b * n] - h_lp_off[a * n]) * 4 : 0);
            };
            int64_t lo = r + 1, hi = R;
            while (lo < hi) {  // largest r1 with bytes(r, r1) <= chunk_bytes (at least one record)
                const int64_t mid = lo + (hi - lo + 1) / 2;
                if (span(r, mid) <= chunk_bytes) lo = mid;
                else hi = mid - 1;
            }
            r = lo;
            cuts.push_back(r);
        }
    }
    const int n_chunks = (int)cuts.size() - 1;
    int n_workers = 3;
    if (const char *e = getenv("KC_JSON_STREAMS")) n_workers = std::max(1, std::min(8, atoi(e)));
    n_workers = std::max(1, std::min(n_workers, n_chunks));
    std::vector<Worker *> workers;
    for (int i = 0; i < n_workers; ++i) workers.push_back(acquire_worker(device));
    std::vector<int> rcs((size_t)n_workers, KC_OK);
    std::vector<std::string> errs((size_t)n_workers);
    std::vector<ChunkStage> stages((size_t)n_workers);
    std::atomic<int> next{0};
    auto body = [&](int wi) {
        cudaSetDevice(device);
        Worker &w = *workers[(size_t)wi];
        int rc = w.init(device);
        while (!rc) {
            const int k = next.fetch_add(1);
            if (k >= n_chunks) break;
            rc = run_chunk(w, h_text, h_off, h_lp, h_lp_off, cuts[(size_t)k], cuts[(size_t)k + 1], n, rel_eps, abs_eps, sm_count, *res,
                           stages[(size_t)wi]);
        }
        if (rc) {
            cudaStreamSynchronize(w.stream);
            errs[(size_t)wi] = kc_last_error();
        }
        rcs[(size_t)wi] = rc;
    };
    if (n_workers == 1) {
        body(0);
    } else {
        std::vector<std::thread> pool;
        for (int i = 0; i < n_workers; ++i) pool.emplace_back(body, i);
        for (auto &t : pool) t.join();
    }
    for (Worker *w : workers) release_worker(w);
    int rc = KC_OK;
    for (int i = 0; i < n_workers && !rc; ++i)
        if (rcs[(size_t)i]) rc = kc_fail(rcs[(size_t)i], "%s", errs[(size_t)i].c_str());
    const auto t_gpu = std::chrono::steady_clock::now();
    // the records the device path declined: host path (H1), unless the caller only wants the device path
    int64_t n_declined = 0, n_host = 0;
    if (!rc) {
        std::vector<int64_t> idx;
        for (int64_t r = 0; r < R; ++r)
            if (res->status[(size_t)r]) idx.push_back(r);
        n_declined = (int64_t)idx.size();
        if (!idx.empty() && !(flags & KC_JSON_DEVICE_ONLY)) {
            const int64_t D = (int64_t)idx.size();
            std::vector<const char *> texts((size_t)(D * n));
            std::vector<int64_t> lens((size_t)(D * n));
            for (int64_t i = 0; i < D; ++i)
                for (int32_t c = 0; c < n; ++c) {
                    const int64_t k = idx[(size_t)i] * n + c;
                    texts[(size_t)(i * n + c)] = h_text + h_off[k];
                    lens[(size_t)(i * n + c)] = h_off[k + 1] - h_off[k];
                }
            std::vector<char *> oc((size_t)D, nullptr), ol((size_t)D, nullptr);
            std::vector<uint8_t> hs((size_t)D, 1);
            rc = kc_consolidate_json(texts.data(), lens.data(), D, n, rel_eps, abs_eps, device, threads, oc.data(), ol.data(), hs.data());
            if (!rc) {
                int64_t pos = res->used.load(), extra = 0;
                for (int64_t i = 0; i < D; ++i)
                    if (hs[(size_t)i] == 0) extra += (int64_t)(strlen(oc[(size_t)i]) + strlen(ol[(size_t)i]));
                char *base = res->blob.p;
                if (pos + extra > (int64_t)res->blob.cap) {  // rare: move the texts to the heap (the pinned blob goes back to the pool)
                    res->heap.resize((size_t)(pos + extra));
                    memcpy(&res->heap[0], res->blob.p, (size_t)pos);
                    release_blob(res->blob);
                    res->blob = PinnedBlob{};
                    base = &res->heap[0];
                }
                for (int64_t i = 0; i < D; ++i) {
                    if (hs[(size_t)i] != 0) continue;
                    const int64_t r = idx[(size_t)i];
                    const size_t lc = strlen(oc[(size_t)i]), ll = strlen(ol[(size_t)i]);
                    memcpy(base + pos, oc[(size_t)i], lc);
                    memcpy(base + pos + lc, ol[(size_t)i], ll);
                    res->c_off[(size_t)r] = pos;
                    res->l_off[(size_t)r] = pos + (int64_t)lc;
                    res->c_len[(size_t)r] = (int64_t)lc;
                    res->l_len[(size_t)r] = (int64_t)ll;
                    res->status[(size_t)r] = 2;
                    pos += (int64_t)(lc + ll);
                    ++n_host;
                }
                res->used.store(pos);
            }
            kc_free_strings(oc.data(), D);
            kc_free_strings(ol.data(), D);
        }
    }
    cudaSetDevice(prev);
    if (rc) {
        release_blob(res->blob);
        delete res;
        return rc;
    }
    const auto t_end = std::chrono::steady_clock::now();
    auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    kc_json_stats &s = res->stats;
    s.n_records = R;
    s.n_device = R - n_declined;
    s.n_host = n_host;
    s.n_python = n_declined - n_host;
    s.input_bytes = total_bytes + lp_bytes;
    s.output_bytes = res->used.load();
    s.chunks = n_chunks;
    s.streams = n_workers;
    for (auto &g : stages) {
        s.h2d_ms += g.h2d;
        s.plan_ms += g.plan;
        s.kernel_ms += g.kernels;
        s.emit_ms += g.emit;
        s.d2h_ms += g.d2h;
    }
    s.device_path_wall_ms = ms(t_start, t_gpu);
    s.host_path_wall_ms = ms(t_gpu, t_end);
    s.wall_ms = ms(t_start, t_end);
    *out = res;
    return KC_OK;
}

}  // namespace

extern "C" {

int kc_consolidate_json_packed(const char *h_text, const int64_t *h_off, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                               int device, int32_t threads, uint32_t flags, kc_json_result **out) {
    return consolidate_packed(h_text, h_off, nullptr, nullptr, n_records, n, rel_eps, abs_eps, device, threads, flags, out);
}

int kc_consolidate_json_packed_weighted(const char *h_text, const int64_t *h_off, const float *h_lp, const int64_t *h_lp_off,
                                        int64_t n_records, int32_t n, double rel_eps, double abs_eps, int device, int32_t threads,
                                        uint32_t flags, kc_json_result **out) {
    if (n_records > 0 && !h_lp_off) return kc_fail(KC_EINVAL, "kc_consolidate_json_packed_weighted: NULL logprob offsets");
    return consolidate_packed(h_text, h_off, h_lp, h_lp_off, n_records, n, rel_eps, abs_eps, device, threads, flags, out);
}

int kc_json_result_view(kc_json_result *res, const char **text, const int64_t **content_off, const int64_t **content_len,
                        const int64_t **likelihoods_off, const int64_t **likelihoods_len, const uint8_t **status, const uint8_t **why,
                        kc_json_stats *stats) {
    if (!res) return kc_fail(KC_EINVAL, "kc_json_result_view: NULL result");
    if (text) *text = res->blob.p ? res->blob.p : res->heap.data();
    if (content_off) *content_off = res->c_off.data();
    if (content_len) *content_len = res->c_len.data();
    if (likelihoods_off) *likelihoods_off = res->l_off.data();
    if (likelihoods_len) *likelihoods_len = res->l_len.data();
    if (status) *status = res->status.data();
    if (why) *why = res->why.data();
    if (stats) *stats = res->stats;
    return KC_OK;
}

void kc_json_result_free(kc_json_result *res) {
    if (!res) return;
    release_blob(res->blob);
    delete res;
}

// ---------------------------------------------------------------- test hooks: the device phases, run on the host

struct kc_debug_jsongpu {
    std::vector<int64_t> off;
    std::vector<uint8_t> text;
    int32_t n = 0;
    int64_t R = 0;
    std::vector<uint32_t> fcount, slot, fdesc, gpos, vbase, xbase, piece_c, piece_l;
    std::vector<uint8_t> status, nest;
    std::vector<Tok> toks;
    unsigned long long counters[3] = {0, 0, 0};
    std::vector<uint32_t> mcount, scount, ccount;
    std::vector<uint8_t> mchars;
    std::vector<int32_t> mstr_off, mgrp_off;
    std::vector<int8_t> vcells;
    std::vector<int32_t> vrec;
    std::vector<double> xcells;
    std::vector<int64_t> len_c, len_l;
    std::vector<uint8_t> out_c, out_l;
    Chunk ch{};
};

int kc_debug_jsongpu_plan(const char *h_text, const int64_t *h_off, int64_t n_records, int32_t n, kc_debug_jsongpu **out) {
    if (!h_text || !h_off || !out || n < 2 || n > KC_MAX_CANDIDATES || n_records < 0) return KC_EINVAL;
    kc_debug_jsongpu *h = new kc_debug_jsongpu;
    const int64_t R = n_records;
    h->R = R;
    h->n = n;
    h->off.assign(h_off, h_off + R * n + 1);
    h->text.assign((const uint8_t *)h_text + h_off[0], (const uint8_t *)h_text + h_off[R * n]);
    h->fcount.assign((size_t)R + 1, 0);
    h->slot.assign((size_t)R + 1, 0);
    h->status.assign((size_t)R, 0);
    h->nest.assign((size_t)R, 0);
    h->vbase.assign((size_t)R, 0);
    h->xbase.assign((size_t)R, 0);
    h->len_c.assign((size_t)R + 1, 0);
    h->len_l.assign((size_t)R + 1, 0);
    h->mcount.assign((size_t)R + 1, 0);
    h->scount.assign((size_t)R + 1, 0);
    h->ccount.assign((size_t)R + 1, 0);
    Chunk &ch = h->ch;
    ch.text = h->text.data();
    ch.off = h->off.data();
    ch.R = (int32_t)R;
    ch.n = n;
    ch.fcount = h->fcount.data();
    ch.slot = h->slot.data();
    ch.status = h->status.data();
    ch.nest = h->nest.data();
    ch.vbase = h->vbase.data();
    ch.xbase = h->xbase.data();
    ch.counters = h->counters;
    ch.mcount = h->mcount.data();
    ch.scount = h->scount.data();
    ch.ccount = h->ccount.data();
    ch.len_c = h->len_c.data();
    ch.len_l = h->len_l.data();
    for (int32_t r = 0; r < R; ++r) kc::js::count_record(ch, r);
    for (int64_t r = 0; r < R; ++r) h->slot[(size_t)r + 1] = h->slot[(size_t)r] + h->fcount[(size_t)r];
    const size_t T = h->slot[(size_t)R];
    h->toks.assign(std::max<size_t>(T * n, 1), Tok{});
    h->fdesc.assign(std::max<size_t>(T, 1), 0);
    h->gpos.assign(std::max<size_t>(T, 1), 0);
    h->piece_c.assign(std::max<size_t>(T, 1), 0);
    h->piece_l.assign(std::max<size_t>(T, 1), 0);
    h->vcells.assign(std::max<size_t>(T * n, 16), (int8_t)-1);
    h->xcells.assign(std::max<size_t>(T * n, 2), 0.0);
    h->vrec.assign(std::max<size_t>(T, 1), 0);
    ch.vrec = h->vrec.data();  // written by slots_phase; only the weighted emit reads what it says
    ch.toks = h->toks.data();
    ch.fdesc = h->fdesc.data();
    ch.gpos = h->gpos.data();
    ch.piece_c = h->piece_c.data();
    ch.piece_l = h->piece_l.data();
    ch.vcells = h->vcells.data();
    ch.xcells = h->xcells.data();
    const int team = team_size(n);
    for (int32_t r = 0; r < R; ++r) {
        for (int lane = 0; lane < team; ++lane) kc::js::parse_phase(ch, r, lane, team);
        for (int lane = 0; lane < team; ++lane) kc::js::type_phase(ch, r, lane, team);
        for (int lane = 0; lane < team; ++lane) kc::js::order_phase(ch, r, lane, team);
        kc::js::slots_phase(ch, r);
        for (int lane = 0; lane < team; ++lane) kc::js::encode_phase(ch, r, lane, team);
    }
    for (std::vector<uint32_t> *cnt : {&h->mcount, &h->scount, &h->ccount}) {  // exclusive scans, in place
        uint32_t acc = 0;
        for (auto &x : *cnt) {
            const uint32_t v = x;
            x = acc;
            acc += v;
        }
    }
    h->mchars.assign((size_t)h->ccount[(size_t)R] + 1, 0);
    h->mstr_off.assign((size_t)h->scount[(size_t)R] + 1, 0);
    h->mgrp_off.assign((size_t)h->mcount[(size_t)R] + 1, 0);
    ch.mchars = h->mchars.data();
    ch.mstr_off = h->mstr_off.data();
    ch.mgrp_off = h->mgrp_off.data();
    for (int32_t r = 0; r < R; ++r)
        for (int lane = 0; lane < team; ++lane) kc::js::medoid_phase(ch, r, lane, team);
    *out = h;
    return KC_OK;
}

// the medoid groups of the planned batch in kc_medoid_str's CSR form, and where the test puts K4's results
int kc_debug_jsongpu_medoid_inputs(const kc_debug_jsongpu *h, const uint8_t **chars, const int32_t **str_off, const int32_t **grp_off,
                                   int64_t *n_groups) {
    if (!h) return KC_EINVAL;
    if (chars) *chars = h->mchars.data();
    if (str_off) *str_off = h->mstr_off.data();
    if (grp_off) *grp_off = h->mgrp_off.data();
    if (n_groups) *n_groups = (int64_t)h->counters[2];
    return KC_OK;
}

int kc_debug_jsongpu_set_medoid(kc_debug_jsongpu *h, const int32_t *medoid_idx, const double *medoid_avg) {
    if (!h) return KC_EINVAL;
    h->ch.midx = medoid_idx;  // must stay alive until kc_debug_jsongpu_emit has returned
    h->ch.mavg = medoid_avg;
    return KC_OK;
}

int kc_debug_jsongpu_inputs(const kc_debug_jsongpu *h, const int8_t **vote_cells, int64_t *n_vote_groups, const double **num_cells,
                            int64_t *n_num_groups, const uint8_t **status) {
    if (!h) return KC_EINVAL;
    if (vote_cells) *vote_cells = h->vcells.data();
    if (n_vote_groups) *n_vote_groups = (int64_t)h->counters[0];
    if (num_cells) *num_cells = h->xcells.data();
    if (n_num_groups) *n_num_groups = (int64_t)h->counters[1];
    if (status) *status = h->status.data();
    return KC_OK;
}

int kc_debug_jsongpu_emit(kc_debug_jsongpu *h, const uint32_t *vote_meta, const double *num_value, const uint32_t *num_meta,
                          const char **content, const int64_t **content_off, const char **likelihoods, const int64_t **likelihoods_off) {
    if (!h) return KC_EINVAL;
    Chunk &ch = h->ch;
    ch.vmeta = vote_meta;
    ch.xvalue = num_value;
    ch.xmeta = num_meta;
    const int64_t R = h->R;
    const int team = team_size(h->n);
    for (int32_t r = 0; r < R; ++r) {
        for (int lane = 0; lane < team; ++lane) kc::js::len_phase(ch, r, lane, team);
        kc::js::offsets_phase(ch, r);
    }
    int64_t ac = 0, al = 0;
    for (int64_t r = 0; r <= R; ++r) {  // exclusive scans, in place
        const int64_t c = r < R ? h->len_c[(size_t)r] : 0, l = r < R ? h->len_l[(size_t)r] : 0;
        h->len_c[(size_t)r] = ac;
        h->len_l[(size_t)r] = al;
        ac += c;
        al += l;
    }
    h->out_c.assign((size_t)std::max<int64_t>(ac, 1), 0);
    h->out_l.assign((size_t)std::max<int64_t>(al, 1), 0);
    ch.out_c = h->out_c.data();
    ch.out_l = h->out_l.data();
    for (int32_t r = 0; r < R; ++r)
        for (int lane = 0; lane < team; ++lane) kc::js::write_phase(ch, r, lane, team);
    if (content) *content = (const char *)h->out_c.data();
    if (content_off) *content_off = h->len_c.data();
    if (likelihoods) *likelihoods = (const char *)h->out_l.data();
    if (likelihoods_off) *likelihoods_off = h->len_l.data();
    return KC_OK;
}

// the record of every vote group (what kc_weighted_vote_groups_i8 takes as d_group_record)
int kc_debug_jsongpu_vote_records(const kc_debug_jsongpu *h, const int32_t **vote_records) {
    if (!h || !vote_records) return KC_EINVAL;
    *vote_records = h->vrec.data();
    return KC_OK;
}

// kc_debug_jsongpu_emit with the weighted vote's (W_win, W_present) per vote group: the confidences of the weighted entry
int kc_debug_jsongpu_emit_weighted(kc_debug_jsongpu *h, const uint32_t *vote_meta, const float *vote_sums, const double *num_value,
                                   const uint32_t *num_meta, const char **content, const int64_t **content_off, const char **likelihoods,
                                   const int64_t **likelihoods_off) {
    if (!h || !vote_sums) return KC_EINVAL;
    h->ch.vsums = vote_sums;
    const int rc = kc_debug_jsongpu_emit(h, vote_meta, num_value, num_meta, content, content_off, likelihoods, likelihoods_off);
    h->ch.vsums = nullptr;
    return rc;
}

void kc_debug_jsongpu_free(kc_debug_jsongpu *h) { delete h; }

// float(text) and float.__repr__ as the device code computes them (batch test hooks)
int kc_debug_parse_doubles(const char *text, const int64_t *off, int64_t count, double *out, uint8_t *ok) {
    if (!text || !off || !out || !ok) return KC_EINVAL;
    for (int64_t i = 0; i < count; ++i) {
        double v = 0.0;
        ok[i] = kc::js::to_double((const uint8_t *)text + off[i], (uint32_t)(off[i + 1] - off[i]), v) ? 1 : 0;
        out[i] = v;
    }
    return KC_OK;
}

int kc_debug_float_reprs(const double *xs, int64_t count, char *out /* [count][32] */, int32_t *lens) {
    if (!xs || !out || !lens) return KC_EINVAL;
    for (int64_t i = 0; i < count; ++i) {
        kc::js::Sink s{(uint8_t *)out + i * 32, 0};
        kc::js::float_repr(xs[i], s);
        lens[i] = (int32_t)s.n;
    }
    return KC_OK;
}

int kc_debug_round5(const double *xs, int64_t count, double *out) {
    if (!xs || !out) return KC_EINVAL;
    for (int64_t i = 0; i < count; ++i) out[i] = kc::js::py_round5(xs[i]);
    return KC_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- bench / test input: schema S32 as candidate texts

namespace {

struct SplitMix {
    uint64_t s;
    uint64_t next() {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
};

// One record of schema S32 (SURVEY.md §8d; same distribution as k_llms_b200/synth.py): n candidate texts exactly as
// json.dumps(dict) prints them.  f00-f15 string-enum (8 words, 4 spellings that sanitise alike), f16-f23 bool, f24-f29 int in
// [1, 1e6), f30-f31 float U(1, 1e4); per field a truth, each candidate copies it w.p. p_agree, then is None w.p. p_none.
void s32_record(uint64_t seed, int64_t r, int32_t n, kc::js::Sink &o, int64_t *off /* n+1 entries, relative to o.n at entry */) {
    static const char *vocab[8] = {"alpha", "Bravo", "charlie", "DELTA", "echo", "foxtrot", "golf", "Hotel"};
    SplitMix g{seed * 0x9E3779B97F4A7C15ull + (uint64_t)r * 0xD1B54A32D192ED03ull + 1};
    const double p_agree = 0.8, p_none = 0.05;
    int32_t truth_code[24];
    double truth_num[8];
    for (int f = 0; f < 24; ++f) truth_code[f] = (int32_t)(g.uni() * (f < 16 ? 8 : 2));
    for (int f = 0; f < 8; ++f) truth_num[f] = f < 6 ? (double)(int64_t)(1 + g.uni() * (1e6 - 1)) : 1.0 + g.uni() * (1e4 - 1.0);
    const int64_t base = o.n;
    for (int32_t c = 0; c < n; ++c) {
        off[c] = o.n - base;
        o.put('{');
        for (int f = 0; f < 32; ++f) {
            if (f) o.lit(", ");
            o.lit("\"f");
            o.put((uint8_t)('0' + f / 10));
            o.put((uint8_t)('0' + f % 10));
            o.lit("\": ");
            const bool agree = g.uni() < p_agree, none = g.uni() < p_none;
            if (f < 24) {
                const int32_t draw = (int32_t)(g.uni() * (f < 16 ? 8 : 2));
                const int32_t k = agree ? truth_code[f] : draw;
                if (none) {
                    o.lit("null");
                } else if (f >= 16) {
                    o.lit(k ? "true" : "false");
                } else {
                    const char *w = vocab[k];
                    const int variant = (int)((r + c + f) & 3);
                    o.put('"');
                    if (variant == 3) o.put(' ');
                    for (const char *q = w; *q; ++q) {
                        char ch = *q;
                        if (variant == 1 && ch >= 'a' && ch <= 'z') ch = (char)(ch - 32);
                        if (variant == 2 && ch >= 'A' && ch <= 'Z') ch = (char)(ch + 32);
                        o.put((uint8_t)ch);
                    }
                    if (variant == 2) o.put('!');
                    o.put('"');
                }
            } else {
                const int k = f - 24;
                const double draw = k < 6 ? (double)(int64_t)(1 + g.uni() * (1e6 - 1)) : 1.0 + g.uni() * (1e4 - 1.0);
                const double v = agree ? truth_num[k] : draw;
                if (none) {
                    o.lit("null");
                } else if (k < 6) {
                    char buf[24];
                    const int len = snprintf(buf, sizeof buf, "%lld", (long long)v);
                    o.put((const uint8_t *)buf, (uint32_t)len);
                } else {
                    kc::js::float_repr(v, o);
                }
            }
        }
        o.put('}');
    }
    off[n] = o.n - base;
}

}  // namespace

extern "C" int kc_debug_s32_texts(uint64_t seed, int64_t n_records, int32_t n, int32_t threads, char *out, int64_t cap, int64_t *off) {
    if (n_records < 0 || n < 1 || n > KC_MAX_CANDIDATES || !off) return KC_EINVAL;
    if (threads <= 0) threads = (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    const int64_t R = n_records;
    const bool write = out != nullptr;
    // pass 1 (out == NULL): lengths -> off[] (absolute, off[0] = 0); pass 2: the texts, at the offsets pass 1 left in off[]
    std::atomic<int64_t> next{0};
    std::atomic<int> bad{0};
    auto body = [&] {
        std::vector<int64_t> rel((size_t)n + 1);
        for (;;) {
            const int64_t b = next.fetch_add(1024);
            if (b >= R) return;
            const int64_t e = std::min(R, b + 1024);
            for (int64_t r = b; r < e; ++r) {
                if (!write) {
                    kc::js::Sink s{nullptr, 0};
                    s32_record(seed, r, n, s, rel.data());
                    for (int32_t c = 0; c < n; ++c) off[r * n + c + 1] = rel[(size_t)c + 1] - rel[(size_t)c];  // lengths for now
                } else {
                    if (off[(r + 1) * n] > cap) {
                        bad = 1;
                        return;
                    }
                    kc::js::Sink s{(uint8_t *)out + off[r * n], 0};
                    s32_record(seed, r, n, s, rel.data());
                }
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t) pool.emplace_back(body);
    for (auto &t : pool) t.join();
    if (!write) {
        off[0] = 0;
        for (int64_t i = 1; i <= R * n; ++i) off[i] += off[i - 1];
    }
    return bad ? KC_EINVAL : KC_OK;
}
