// msfm_multi.cc — implementation of include/msfm_multi.h: one host process, all GPUs of the box.
//
//   * one single-GPU context (msfm_api.cu) per device, all with the same table layout: every device reserves every image
//     in the same order, so an image occupies the same arena rows everywhere and replication is a plain range copy;
//   * NCCL (ncclCommInitAll, one communicator per device, grouped ncclBroadcast per owner block) forwards freshly packed
//     rows + column keys over NVLink into the other devices' tables; NCCL is resolved with dlopen at run time, so the
//     library has no link-time dependency on it and a process that already carries torch's NCCL shares that copy;
//   * the pair list is sharded by msfm_sched_shard, one host thread per device runs the single-GPU matcher into
//     page-locked blocks, the lists are stitched into the caller's msfm_result in the caller's pair order.
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>

#include "../../include/msfm_multi.h"
#include "msfm_internal.h"

namespace {

// ---------------------------------------------------------------------------------------------------- NCCL via dlopen
// Prototypes restated from nccl.h (2.x ABI: ncclResult_t and ncclDataType_t are ints, ncclComm_t an opaque pointer).
typedef void *nccl_comm_t;
struct NcclApi {
    void *handle = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    int (*CommInitAll)(nccl_comm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    std::string error;
    bool ok = false;
};
constexpr int kNcclUint8 = 1;  // ncclUint8

NcclApi &nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            api.handle = dlopen(name, RTLD_NOW | RTLD_LOCAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            api.error = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "not found");
            return;
        }
        auto sym = [&](const char *n) { return dlsym(api.handle, n); };
        api.GetErrorString = reinterpret_cast<const char *(*)(int)>(sym("ncclGetErrorString"));
        api.CommInitAll = reinterpret_cast<int (*)(nccl_comm_t *, int, const int *)>(sym("ncclCommInitAll"));
        api.CommDestroy = reinterpret_cast<int (*)(nccl_comm_t)>(sym("ncclCommDestroy"));
        api.GroupStart = reinterpret_cast<int (*)()>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<int (*)()>(sym("ncclGroupEnd"));
        api.Broadcast = reinterpret_cast<int (*)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t)>(sym("ncclBroadcast"));
        api.ok = api.GetErrorString && api.CommInitAll && api.CommDestroy && api.GroupStart && api.GroupEnd && api.Broadcast;
        if (!api.ok) api.error = "libnccl.so.2 lacks a required symbol";
    });
    return api;
}

// Page-locked result block of one device: the match lists of consecutive batches, back to back.
struct Block {
    int32_t (*m)[2] = nullptr;
    uint8_t *g = nullptr;
    int64_t cap = 0, used = 0;
};
struct Segment {  // one batch: local match indices [first, first + n) live at m / g
    int64_t first, n;
    int32_t (*m)[2];
    uint8_t *g;
};
constexpr int64_t kBlockEntries = 4ll << 20;  // 32 MiB of matches + 4 MiB of flags

struct DeviceSlot {
    int device = 0;
    msfm_ctx *ctx = nullptr;
    nccl_comm_t comm = nullptr;
    cudaStream_t main_stream = nullptr, upload_stream = nullptr;
    std::vector<cudaEvent_t> event_pool;
    uint8_t *desc = nullptr;
    int32_t *norms = nullptr;
    std::vector<Block> blocks;
    std::vector<Segment> segments;
    // per match call
    std::vector<msfm_pair> pairs;
    std::vector<int64_t> pair_index, offsets;
    std::vector<int32_t> ok;
    msfm_status status = MSFM_OK;
    std::string err;
    bool want_good = false;
};

int sink_fn(void *user, int64_t first, int64_t n, int32_t (**m)[2], uint8_t **g) {
    DeviceSlot *d = static_cast<DeviceSlot *>(user);
    Block *b = nullptr;
    for (Block &x : d->blocks)
        if (x.cap - x.used >= n) { b = &x; break; }
    if (!b) {
        Block nb;
        nb.cap = std::max(n, kBlockEntries);
        if (cudaHostAlloc(reinterpret_cast<void **>(&nb.m), (size_t)nb.cap * 8, cudaHostAllocPortable) != cudaSuccess) return 1;
        if (cudaHostAlloc(reinterpret_cast<void **>(&nb.g), (size_t)nb.cap, cudaHostAllocPortable) != cudaSuccess) {
            cudaFreeHost(nb.m);
            return 1;
        }
        d->blocks.push_back(nb);
        b = &d->blocks.back();
    }
    *m = b->m + b->used;
    *g = d->want_good ? b->g + b->used : nullptr;
    d->segments.push_back({first, n, *m, b->g + b->used});
    b->used += n;
    return 0;
}

}  // namespace

// A staged group whose rows sit on their owner devices only: the broadcast to the other devices is issued lazily, between
// two matching launches (see flush_pending).
struct ArenaRange { int64_t off, rows; int owner; };
struct PendingGroup {
    uint64_t serial;
    std::vector<ArenaRange> ranges;
    std::vector<cudaEvent_t> uploaded;  // per device: recorded on its upload stream after the group's uploads / reserves
};

struct msfm_multi {
    std::vector<DeviceSlot> dev;
    std::vector<int32_t> rows;  // per image id; -1 = not staged
    std::vector<uint64_t> group_of;  // per image id: serial of the staging group that brought it
    std::vector<PendingGroup> pending;
    uint64_t next_serial = 1;
    int32_t max_images = 0;
    std::string err;
    std::mutex mu;
    msfm_multi_timing timing{};
};

namespace {

msfm_status mfail(msfm_multi *mm, msfm_status st, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (mm) mm->err = buf;
    return st;
}

#define MM_CUDA(mm, call)                                                                                                    \
    do {                                                                                                                     \
        cudaError_t e__ = (call);                                                                                            \
        if (e__ != cudaSuccess) return mfail(mm, MSFM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
#define MM_NCCL(mm, call)                                                                                                    \
    do {                                                                                                                     \
        int r__ = (call);                                                                                                    \
        if (r__ != 0) return mfail(mm, MSFM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, nccl().GetErrorString(r__), __FILE__, __LINE__); \
    } while (0)
#define MM_CTX(mm, d, call)                                                                                                  \
    do {                                                                                                                     \
        msfm_status s__ = (call);                                                                                            \
        if (s__ != MSFM_OK) return mfail(mm, s__, "device %d: %s", (d).device, msfm_last_error((d).ctx));                    \
    } while (0)

// Stage one group.  `upload` enqueues the owner's part on device slot d for the images [a, b) of the call.
template <class UploadRun>
msfm_status stage_group(msfm_multi *mm, int32_t n, const int32_t *ids, const int32_t *rows, UploadRun upload) {
    const int W = (int)mm->dev.size();
    if (n < 0 || (n > 0 && (!ids || !rows))) return mfail(mm, MSFM_ERR_INVALID_ARG, "null argument");
    for (int32_t i = 0; i < n; ++i) {
        if (ids[i] < 0 || ids[i] >= mm->max_images) return mfail(mm, MSFM_ERR_INVALID_ARG, "image id %d outside [0, %d)", ids[i], mm->max_images);
        if (mm->rows[ids[i]] >= 0) return mfail(mm, MSFM_ERR_EXISTS, "image id %d already staged", ids[i]);
    }
    if (n == 0) return MSFM_OK;
    std::vector<int32_t> owner((size_t)n);
    msfm_sched_image_owner(n, W, owner.data());
    struct Run { int32_t a, b, owner; };
    std::vector<Run> runs;
    for (int32_t i = 0; i < n; ++i) {
        if (runs.empty() || runs.back().owner != owner[i]) runs.push_back({i, i + 1, owner[i]});
        else runs.back().b = i + 1;
    }
    // identical allocation order on every device => identical arena offsets
    std::vector<cudaEvent_t> uploaded;
    for (int d = 0; d < W; ++d) {
        DeviceSlot &ds = mm->dev[d];
        for (const Run &r : runs) {
            if (r.owner == d) MM_CTX(mm, ds, upload(ds, r.a, r.b));
            else MM_CTX(mm, ds, msfm_reserve_batch_async(ds.ctx, r.b - r.a, ids + r.a, rows + r.a, nullptr));
        }
        if (W > 1) {
            MM_CUDA(mm, cudaSetDevice(ds.device));
            cudaEvent_t ev = nullptr;
            if (!ds.event_pool.empty()) { ev = ds.event_pool.back(); ds.event_pool.pop_back(); }
            else MM_CUDA(mm, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            MM_CUDA(mm, cudaEventRecord(ev, ds.upload_stream));  // packed rows / pad rows / tensor maps of this group
            uploaded.push_back(ev);
        }
    }
    const uint64_t serial = mm->next_serial++;
    if (W > 1) {
        // the broadcast itself is issued lazily (flush_pending): one range per owner block and arena, adjacent images coalesced
        PendingGroup pg;
        pg.serial = serial;
        pg.uploaded = uploaded;
        for (const Run &r : runs)
            for (int32_t i = r.a; i < r.b; ++i) {
                int32_t rr = 0;
                int64_t off = 0;
                MM_CTX(mm, mm->dev[0], msfm_image_info(mm->dev[0].ctx, ids[i], &rr, &off));
                const int64_t padded = ((int64_t)std::max(rr, 1) + 255) / 256 * 256;
                if (!pg.ranges.empty() && pg.ranges.back().owner == r.owner && pg.ranges.back().off + pg.ranges.back().rows == off) pg.ranges.back().rows += padded;
                else pg.ranges.push_back({off, padded, r.owner});
            }
        mm->pending.push_back(pg);
    }
    for (int32_t i = 0; i < n; ++i) {
        mm->rows[ids[i]] = rows[i];
        mm->group_of[ids[i]] = serial;
    }
    return MSFM_OK;
}

// Replicate the staged groups up to `serial` on every device: grouped ncclBroadcast per owner block (descriptor rows and
// side words), queued on each device's MAIN stream behind the group's uploads.  Running the collective on the stream the
// matching launches use keeps it BETWEEN launches: the matching kernel is persistent (one CTA per SM, statically
// partitioned work), and a collective kernel parked on a few SMs while a peer device is still matching would stall the
// CTAs that cannot be placed next to it.
msfm_status flush_pending(msfm_multi *mm, uint64_t serial) {
    const int W = (int)mm->dev.size();
    size_t done = 0;
    for (PendingGroup &pg : mm->pending) {
        if (pg.serial > serial) break;
        for (int d = 0; d < W; ++d) {
            MM_CUDA(mm, cudaSetDevice(mm->dev[d].device));
            MM_CUDA(mm, cudaStreamWaitEvent(mm->dev[d].main_stream, pg.uploaded[d], 0));
            mm->dev[d].event_pool.push_back(pg.uploaded[d]);
        }
        NcclApi &nc = nccl();
        MM_NCCL(mm, nc.GroupStart());
        for (const ArenaRange &rg : pg.ranges)
            for (int d = 0; d < W; ++d) {
                DeviceSlot &ds = mm->dev[d];
                MM_NCCL(mm, nc.Broadcast(ds.desc + rg.off * MSFM_DIM, ds.desc + rg.off * MSFM_DIM, (size_t)rg.rows * MSFM_DIM, kNcclUint8, rg.owner, ds.comm, ds.main_stream));
                MM_NCCL(mm, nc.Broadcast(ds.norms + rg.off, ds.norms + rg.off, (size_t)rg.rows * 4, kNcclUint8, rg.owner, ds.comm, ds.main_stream));
            }
        MM_NCCL(mm, nc.GroupEnd());
        for (const ArenaRange &rg : pg.ranges) mm->timing.bytes_broadcast += rg.rows * (MSFM_DIM + 4);
        ++done;
    }
    mm->pending.erase(mm->pending.begin(), mm->pending.begin() + done);
    return MSFM_OK;
}

}  // namespace

extern "C" {

msfm_status msfm_multi_create(const msfm_multi_config *cfg, msfm_multi **out) {
    if (!cfg || !out) return MSFM_ERR_INVALID_ARG;
    *out = nullptr;
    if (cfg->n_devices < 1 || cfg->n_devices > 64 || cfg->max_images <= 0 || cfg->arena_rows <= 0) return MSFM_ERR_INVALID_ARG;
    for (int32_t r : cfg->reserved)
        if (r) return MSFM_ERR_INVALID_ARG;
    if (cfg->n_devices > 1 && !nccl().ok) {
        fprintf(stderr, "[msfm_multi] %s\n", nccl().error.c_str());
        return MSFM_ERR_UNSUPPORTED;
    }
    msfm_multi *mm = new (std::nothrow) msfm_multi();
    if (!mm) return MSFM_ERR_OUT_OF_MEMORY;
    mm->max_images = cfg->max_images;
    mm->rows.assign((size_t)cfg->max_images, -1);
    mm->group_of.assign((size_t)cfg->max_images, 0);
    mm->dev.resize((size_t)cfg->n_devices);
    auto bail = [&](msfm_status st) {
        msfm_multi_destroy(mm);
        return st;
    };
    std::vector<int> devlist;
    for (int32_t k = 0; k < cfg->n_devices; ++k) {
        DeviceSlot &ds = mm->dev[k];
        ds.device = cfg->devices ? cfg->devices[k] : k;
        devlist.push_back(ds.device);
        msfm_config c;
        memset(&c, 0, sizeof c);
        c.device = ds.device;
        c.max_images = cfg->max_images;
        c.arena_rows = cfg->arena_rows;
        const msfm_status st = msfm_create(&c, &ds.ctx);
        if (st != MSFM_OK) return bail(st);
        void *dp = nullptr, *np = nullptr, *us = nullptr, *ms = nullptr;
        msfm_table_ptrs(ds.ctx, &dp, &np, nullptr, nullptr);
        msfm_get_upload_stream(ds.ctx, &us);
        msfm_get_stream(ds.ctx, &ms);
        ds.desc = static_cast<uint8_t *>(dp);
        ds.norms = static_cast<int32_t *>(np);
        ds.upload_stream = static_cast<cudaStream_t>(us);
        ds.main_stream = static_cast<cudaStream_t>(ms);
    }
    if (cfg->n_devices > 1) {
        std::vector<nccl_comm_t> comms((size_t)cfg->n_devices, nullptr);
        const int r = nccl().CommInitAll(comms.data(), cfg->n_devices, devlist.data());
        if (r != 0) {
            fprintf(stderr, "[msfm_multi] ncclCommInitAll failed: %s\n", nccl().GetErrorString(r));
            return bail(MSFM_ERR_CUDA);
        }
        for (int32_t k = 0; k < cfg->n_devices; ++k) mm->dev[k].comm = comms[k];
    }
    mm->timing.n_devices = cfg->n_devices;
    *out = mm;
    return MSFM_OK;
}

msfm_status msfm_multi_destroy(msfm_multi *mm) {
    if (!mm) return MSFM_OK;
    for (DeviceSlot &ds : mm->dev) {
        cudaSetDevice(ds.device);
        if (ds.main_stream) cudaStreamSynchronize(ds.main_stream);
    }
    for (PendingGroup &pg : mm->pending)
        for (size_t d = 0; d < pg.uploaded.size() && d < mm->dev.size(); ++d) mm->dev[d].event_pool.push_back(pg.uploaded[d]);
    for (DeviceSlot &ds : mm->dev) {
        cudaSetDevice(ds.device);
        if (ds.comm) nccl().CommDestroy(ds.comm);
        for (cudaEvent_t e : ds.event_pool) cudaEventDestroy(e);
        if (ds.ctx) msfm_destroy(ds.ctx);
        for (Block &b : ds.blocks) {
            cudaFreeHost(b.m);
            cudaFreeHost(b.g);
        }
    }
    delete mm;
    return MSFM_OK;
}

const char *msfm_multi_last_error(const msfm_multi *mm) { return mm ? mm->err.c_str() : "null context"; }
int32_t msfm_multi_device_count(const msfm_multi *mm) { return mm ? (int32_t)mm->dev.size() : 0; }
msfm_ctx *msfm_multi_context(msfm_multi *mm, int32_t k) { return (mm && k >= 0 && k < (int32_t)mm->dev.size()) ? mm->dev[k].ctx : nullptr; }

msfm_status msfm_multi_upload_u8(msfm_multi *mm, int32_t n, const int32_t *image_ids, const uint8_t *const *descs, const int32_t *rows) {
    if (!mm) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(mm->mu);
    if (n > 0 && !descs) return mfail(mm, MSFM_ERR_INVALID_ARG, "null descriptors");
    return stage_group(mm, n, image_ids, rows, [&](DeviceSlot &ds, int32_t a, int32_t b) {
        return msfm_upload_u8_batch_async(ds.ctx, b - a, image_ids + a, descs + a, rows + a, nullptr);
    });
}

msfm_status msfm_multi_upload_f32(msfm_multi *mm, int32_t n, const int32_t *image_ids, const float *const *descs, const int32_t *rows,
                                  float scale) {
    if (!mm) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(mm->mu);
    if (n > 0 && !descs) return mfail(mm, MSFM_ERR_INVALID_ARG, "null descriptors");
    return stage_group(mm, n, image_ids, rows, [&](DeviceSlot &ds, int32_t a, int32_t b) {
        return msfm_upload_f32_batch_async(ds.ctx, b - a, image_ids + a, descs + a, rows + a, scale);
    });
}

msfm_status msfm_multi_sync(msfm_multi *mm) {
    if (!mm) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(mm->mu);
    const msfm_status st = flush_pending(mm, ~0ull);  // every staged group is replicated
    if (st != MSFM_OK) return st;
    for (DeviceSlot &ds : mm->dev) MM_CTX(mm, ds, msfm_sync(ds.ctx));  // upload streams and main streams (the collectives)
    return MSFM_OK;
}

msfm_status msfm_multi_release_all(msfm_multi *mm) {
    if (!mm) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(mm->mu);
    const msfm_status st = flush_pending(mm, ~0ull);  // keeps the devices' collective sequences in step
    if (st != MSFM_OK) return st;
    for (DeviceSlot &ds : mm->dev) MM_CTX(mm, ds, msfm_sync(ds.ctx));
    for (DeviceSlot &ds : mm->dev) MM_CTX(mm, ds, msfm_release_all(ds.ctx));
    std::fill(mm->rows.begin(), mm->rows.end(), -1);
    mm->timing.bytes_broadcast = 0;
    return MSFM_OK;
}

msfm_status msfm_multi_match_pairs(msfm_multi *mm, const msfm_pair *pairs, int64_t n_pairs, const msfm_params *params, msfm_result *out) {
    if (!mm) return MSFM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(mm->mu);
    if (n_pairs < 0 || (n_pairs > 0 && !pairs) || !params || !out || !out->offsets || !out->ok || (!out->matches && out->match_capacity > 0))
        return mfail(mm, MSFM_ERR_INVALID_ARG, "null pair list / params / result buffers or negative n_pairs");
    const auto t0 = std::chrono::steady_clock::now();
    const int W = (int)mm->dev.size();
    for (int64_t i = 0; i < n_pairs; ++i)
        for (int32_t id : {pairs[i].ref, pairs[i].query})
            if (id < 0 || id >= mm->max_images || mm->rows[id] < 0) return mfail(mm, MSFM_ERR_NOT_FOUND, "pair %lld names image %d, which is not staged", (long long)i, id);
    // replicate what the pair list needs: the staged groups up to the newest one it touches (later groups stay in flight)
    uint64_t need = 0;
    for (int64_t i = 0; i < n_pairs; ++i) need = std::max(need, std::max(mm->group_of[pairs[i].ref], mm->group_of[pairs[i].query]));
    if (W > 1) {
        const msfm_status fst = flush_pending(mm, need);
        if (fst != MSFM_OK) return fst;
    }
    // rows of unstaged images are irrelevant to the scheduler (no pair names them)
    std::vector<int32_t> rows(mm->rows);
    for (int32_t &r : rows) r = std::max(r, 0);
    std::vector<int32_t> worker((size_t)std::max<int64_t>(n_pairs, 1));
    if (msfm_sched_shard(pairs, n_pairs, rows.data(), mm->max_images, W, worker.data(), nullptr) != 0)
        return mfail(mm, MSFM_ERR_INVALID_ARG, "msfm_sched_shard rejected the pair list");
    for (DeviceSlot &ds : mm->dev) {
        ds.pairs.clear();
        ds.pair_index.clear();
        ds.segments.clear();
        for (Block &b : ds.blocks) b.used = 0;
        ds.status = MSFM_OK;
        ds.want_good = out->good != nullptr;
    }
    for (int64_t i = 0; i < n_pairs; ++i) {
        DeviceSlot &ds = mm->dev[worker[i]];
        ds.pairs.push_back(pairs[i]);
        ds.pair_index.push_back(i);
    }
    // ---- match: one host thread per device, no data-path collective
    auto run_device = [&](DeviceSlot &ds) {
        ds.offsets.assign(ds.pairs.size() + 1, 0);
        ds.ok.assign(std::max<size_t>(ds.pairs.size(), 1), 0);
        ds.status = msfm_internal_match_pairs_sink(ds.ctx, ds.pairs.data(), (int64_t)ds.pairs.size(), params, ds.offsets.data(), ds.ok.data(),
                                                   ds.want_good ? 1 : 0, sink_fn, &ds);
        if (ds.status != MSFM_OK) ds.err = msfm_last_error(ds.ctx);
    };
    {
        std::vector<std::thread> threads;
        for (int d = 1; d < W; ++d) threads.emplace_back(run_device, std::ref(mm->dev[d]));
        run_device(mm->dev[0]);
        for (std::thread &t : threads) t.join();
    }
    for (DeviceSlot &ds : mm->dev)
        if (ds.status != MSFM_OK) return mfail(mm, ds.status, "device %d: %s", ds.device, ds.err.c_str());
    // ---- gather: global offsets, then every device's lists to their places in the caller's pair order
    const auto t1 = std::chrono::steady_clock::now();
    out->offsets[0] = 0;
    for (DeviceSlot &ds : mm->dev)
        for (size_t k = 0; k < ds.pairs.size(); ++k) {
            out->offsets[ds.pair_index[k] + 1] = ds.offsets[k + 1] - ds.offsets[k];  // counts first
            out->ok[ds.pair_index[k]] = ds.ok[k];
        }
    for (int64_t p = 0; p < n_pairs; ++p) out->offsets[p + 1] += out->offsets[p];
    if (out->offsets[n_pairs] > out->match_capacity)
        return mfail(mm, MSFM_ERR_CAPACITY, "match buffer too small: need %lld entries, capacity %lld", (long long)out->offsets[n_pairs], (long long)out->match_capacity);
    auto scatter_device = [&](DeviceSlot &ds) {
        size_t k = 0;
        for (const Segment &sg : ds.segments) {  // a batch holds whole pairs, in local order
            // consecutive local pairs that are also consecutive in the caller's list (a run sharing the reference image)
            // are contiguous on both sides: one copy per run
            while (k < ds.pairs.size() && ds.offsets[k + 1] <= sg.first + sg.n) {
                size_t e = k + 1;
                while (e < ds.pairs.size() && ds.offsets[e + 1] <= sg.first + sg.n && ds.pair_index[e] == ds.pair_index[e - 1] + 1) ++e;
                const int64_t a = ds.offsets[k], cnt = ds.offsets[e] - a;
                if (cnt > 0) {
                    const int64_t dst = out->offsets[ds.pair_index[k]];
                    memcpy(out->matches + dst, sg.m + (a - sg.first), (size_t)cnt * 8);
                    if (out->good) memcpy(out->good + dst, sg.g + (a - sg.first), (size_t)cnt);
                }
                k = e;
            }
        }
    };
    {
        std::vector<std::thread> threads;
        for (int d = 1; d < W; ++d) threads.emplace_back(scatter_device, std::ref(mm->dev[d]));
        scatter_device(mm->dev[0]);
        for (std::thread &t : threads) t.join();
    }
    const auto t2 = std::chrono::steady_clock::now();
    mm->timing.wall_ms = std::chrono::duration<float, std::milli>(t2 - t0).count();
    mm->timing.stitch_ms = std::chrono::duration<float, std::milli>(t2 - t1).count();
    mm->timing.device_ms_max = 0.f;
    mm->timing.int8_ops = 0;
    for (DeviceSlot &ds : mm->dev) {
        msfm_timing t;
        if (msfm_last_timing(ds.ctx, &t) == MSFM_OK && !ds.pairs.empty()) {
            mm->timing.device_ms_max = std::max(mm->timing.device_ms_max, t.total_ms);
            mm->timing.int8_ops += t.int8_ops;
        }
    }
    return MSFM_OK;
}

msfm_status msfm_multi_last_timing(const msfm_multi *mm, msfm_multi_timing *out, msfm_timing *per_device) {
    if (!mm || !out) return MSFM_ERR_INVALID_ARG;
    *out = mm->timing;
    if (per_device)
        for (size_t d = 0; d < mm->dev.size(); ++d) msfm_last_timing(mm->dev[d].ctx, per_device + d);
    return MSFM_OK;
}

}  // extern "C"
