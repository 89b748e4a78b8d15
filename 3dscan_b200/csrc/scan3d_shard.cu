// scan3d_shard.cu -- host side of the row-sharded mode (include/scan3d_shard.h): a POSIX shared-memory board for the
// per-scan control words (counts, "pushed", "released") of the processes of one node, CUDA IPC for root's output
// blocks, copy-engine pushes over NVLink for the data.  No kernel is launched here.
#include <fcntl.h>
#include <sched.h>
#include <stdio.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

#include <atomic>
#include <new>
#include <string>

#include "../../include/scan3d_shard.h"
#include "scan3d_internal.h"

namespace {

constexpr int MAX_WORLD = 16, MAX_SLOTS = 4;
constexpr uint64_t MAGIC = 0x5343414e33445348ull;   // "SCAN3DSH"

struct SlotBoard {
    std::atomic<uint64_t> count[MAX_WORLD];    // seq << 32 | points of that rank in scan number seq of this slot
    std::atomic<uint64_t> pushed[MAX_WORLD];   // seq: that rank's points of scan seq have landed in root's block
    std::atomic<uint64_t> released;            // seq: root has consumed the cloud of scan seq
};
struct Board {
    std::atomic<uint64_t> magic;               // set last by root
    std::atomic<int> joined, left;
    int world, slots;
    uint8_t handle[MAX_SLOTS][64];             // CUDA IPC handles of root's output blocks
    SlotBoard slot[MAX_SLOTS];
};

thread_local std::string g_shard_error;

double now_s()
{
    timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return t.tv_sec + 1e-9 * t.tv_nsec;
}

}  // namespace

struct scan3d_shard {
    std::string name, err;
    int rank = 0, world = 1, device = 0, slots = 0;
    int64_t capacity = 0;
    Board* board = nullptr;
    void* block[MAX_SLOTS] = {};       // root: owned; others: IPC mapping (host mode: all ranks map one shared segment)
    bool host_mode = false;            // device < 0: no GPU anywhere, the blocks live in shared memory (CPU tests of the protocol)
    void* host_blocks = nullptr;
    size_t host_bytes = 0;
    uint64_t seq[MAX_SLOTS] = {};      // gathers done on each slot
    uint32_t* h_count = nullptr;       // pinned
    double timeout_s = 60.0;
};

static int sfail(scan3d_shard* sh, int code, const std::string& msg)
{
    if (sh) sh->err = msg;
    else g_shard_error = msg;
    return code;
}

// spin (politely) until pred() or the timeout
template <class F>
static bool wait_for(scan3d_shard* sh, F pred)
{
    const double t0 = now_s();
    for (int spins = 0; !pred(); spins++) {
        if (spins > 2000) sched_yield();
        if ((spins & 1023) == 1023 && now_s() - t0 > sh->timeout_s) return false;
    }
    return true;
}

extern "C" {

const char* scan3d_shard_last_error(const scan3d_shard* sh) { return sh ? sh->err.c_str() : g_shard_error.c_str(); }

int scan3d_shard_create(const char* name, int rank, int world, int device, int64_t capacity_points, int slots, scan3d_shard** out)
{
    if (!out) return sfail(nullptr, SCAN3D_ERR_ARG, "null out pointer");
    *out = nullptr;
    if (!name || !*name || world < 1 || world > MAX_WORLD || rank < 0 || rank >= world || slots < 1 || slots > MAX_SLOTS ||
        capacity_points < 1)
        return sfail(nullptr, SCAN3D_ERR_ARG, "scan3d_shard_create: bad argument (world <= 16, slots <= 4)");
    const bool host_mode = device < 0;
    if (!host_mode && cudaSetDevice(device) != cudaSuccess) return sfail(nullptr, SCAN3D_ERR_CUDA, "cudaSetDevice failed");
    scan3d_shard* sh = new (std::nothrow) scan3d_shard();
    if (!sh) return sfail(nullptr, SCAN3D_ERR_CUDA, "out of host memory");
    sh->host_mode = host_mode;
    sh->name = std::string("/scan3d_") + name;
    sh->rank = rank; sh->world = world; sh->device = device; sh->slots = slots; sh->capacity = capacity_points;
    auto bail = [&](int code, const std::string& msg) {
        g_shard_error = msg;
        scan3d_shard_destroy(sh);
        return code;
    };
    // ---- the board: root creates and initialises it, the others wait for the magic word
    int fd = -1;
    if (rank == 0) {
        shm_unlink(sh->name.c_str());     // a stale board of a crashed job with the same name
        fd = shm_open(sh->name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
        if (fd < 0 || ftruncate(fd, sizeof(Board)) != 0) return bail(SCAN3D_ERR_IO, "cannot create the shared-memory board " + sh->name);
    } else {
        const double t0 = now_s();
        while ((fd = shm_open(sh->name.c_str(), O_RDWR, 0600)) < 0) {
            if (now_s() - t0 > sh->timeout_s) return bail(SCAN3D_ERR_IO, "the shared-memory board " + sh->name + " never appeared (is rank 0 up?)");
            usleep(1000);
        }
        struct stat st;
        const double t1 = now_s();
        while (fstat(fd, &st) == 0 && (size_t)st.st_size < sizeof(Board)) {
            if (now_s() - t1 > sh->timeout_s) { close(fd); return bail(SCAN3D_ERR_IO, "the shared-memory board was never sized"); }
            usleep(1000);
        }
    }
    void* p = mmap(nullptr, sizeof(Board), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) return bail(SCAN3D_ERR_IO, "mmap of the shared-memory board failed");
    sh->board = static_cast<Board*>(p);
    Board* b = sh->board;
    if (!host_mode && cudaHostAlloc((void**)&sh->h_count, 64, cudaHostAllocDefault) != cudaSuccess) return bail(SCAN3D_ERR_CUDA, "cudaHostAlloc failed");
    if (host_mode) {
        // the output blocks of the GPU-less mode: a second shared segment every rank maps
        const std::string bn = sh->name + "_blk";
        sh->host_bytes = (size_t)slots * capacity_points * 12;
        int bfd = -1;
        if (rank == 0) {
            shm_unlink(bn.c_str());
            bfd = shm_open(bn.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
            if (bfd < 0 || ftruncate(bfd, sh->host_bytes) != 0) return bail(SCAN3D_ERR_IO, "cannot create the shared output blocks");
        } else {
            if (!wait_for(sh, [&] { return b->magic.load(std::memory_order_acquire) == MAGIC; }))
                return bail(SCAN3D_ERR_IO, "the shared-memory board was never initialised");
            bfd = shm_open(bn.c_str(), O_RDWR, 0600);
            if (bfd < 0) return bail(SCAN3D_ERR_IO, "cannot open the shared output blocks");
        }
        sh->host_blocks = mmap(nullptr, sh->host_bytes, PROT_READ | PROT_WRITE, MAP_SHARED, bfd, 0);
        close(bfd);
        if (sh->host_blocks == MAP_FAILED) { sh->host_blocks = nullptr; return bail(SCAN3D_ERR_IO, "mmap of the shared output blocks failed"); }
        for (int s = 0; s < slots; s++) sh->block[s] = static_cast<uint8_t*>(sh->host_blocks) + (size_t)s * capacity_points * 12;
    }
    if (rank == 0) {
        memset((void*)b, 0, sizeof(Board));
        b->world = world; b->slots = slots;
        for (int s = 0; s < slots && !host_mode; s++) {
            if (scan3d_peer_alloc(device, capacity_points * 12, &sh->block[s], b->handle[s]) != SCAN3D_OK)
                return bail(SCAN3D_ERR_CUDA, "cannot allocate / export an output block");
        }
        b->joined.store(1, std::memory_order_relaxed);
        b->magic.store(MAGIC, std::memory_order_release);
    } else {
        if (!wait_for(sh, [&] { return b->magic.load(std::memory_order_acquire) == MAGIC; }))
            return bail(SCAN3D_ERR_IO, "the shared-memory board was never initialised");
        if (b->world != world || b->slots != slots) return bail(SCAN3D_ERR_ARG, "ranks disagree about world size / slots");
        for (int s = 0; s < slots && !host_mode; s++)
            if (scan3d_peer_open(device, b->handle[s], &sh->block[s]) != SCAN3D_OK)
                return bail(SCAN3D_ERR_CUDA, "cannot map root's output block (no peer access between the GPUs?)");
        b->joined.fetch_add(1, std::memory_order_acq_rel);
    }
    if (!wait_for(sh, [&] { return b->joined.load(std::memory_order_acquire) == world; }))
        return bail(SCAN3D_ERR_IO, "not every rank joined the row-shard group");
    *out = sh;
    return SCAN3D_OK;
}

int scan3d_shard_destroy(scan3d_shard* sh)
{
    if (!sh) return SCAN3D_OK;
    if (!sh->host_mode) {
        cudaSetDevice(sh->device);
        cudaDeviceSynchronize();
    }
    Board* b = sh->board;
    if (b && b->magic.load(std::memory_order_acquire) == MAGIC) {
        // nobody unmaps / frees while another rank may still be pushing into the blocks
        b->left.fetch_add(1, std::memory_order_acq_rel);
        wait_for(sh, [&] { return b->left.load(std::memory_order_acquire) >= sh->world; });
    }
    for (int s = 0; s < sh->slots && !sh->host_mode; s++)
        if (sh->block[s]) {
            if (sh->rank == 0) scan3d_peer_free(sh->device, sh->block[s]);
            else scan3d_peer_close(sh->device, sh->block[s]);
        }
    if (sh->h_count) cudaFreeHost(sh->h_count);
    if (sh->host_blocks) munmap(sh->host_blocks, sh->host_bytes);
    if (b) munmap((void*)b, sizeof(Board));
    if (sh->rank == 0) {
        shm_unlink(sh->name.c_str());
        if (sh->host_mode) shm_unlink((sh->name + "_blk").c_str());
    }
    delete sh;
    return SCAN3D_OK;
}

int scan3d_shard_bind(scan3d_shard* sh, int slot, scan3d_ctx* ctx)
{
    if (!sh || !ctx || slot < 0 || slot >= sh->slots) return sfail(sh, SCAN3D_ERR_ARG, "scan3d_shard_bind: bad argument");
    if (sh->rank != 0) return SCAN3D_OK;
    if (scan3d_set_points_buffer(ctx, sh->block[slot], sh->capacity) != SCAN3D_OK)
        return sfail(sh, SCAN3D_ERR_ARG, std::string("scan3d_set_points_buffer: ") + scan3d_last_error(ctx));
    return SCAN3D_OK;
}

void* scan3d_shard_output(scan3d_shard* sh, int slot)
{
    return (sh && sh->rank == 0 && slot >= 0 && slot < sh->slots) ? sh->block[slot] : nullptr;
}

int scan3d_shard_release(scan3d_shard* sh, int slot)
{
    if (!sh || slot < 0 || slot >= sh->slots) return sfail(sh, SCAN3D_ERR_ARG, "scan3d_shard_release: bad argument");
    if (sh->rank == 0) sh->board->slot[slot].released.store(sh->seq[slot], std::memory_order_release);
    return SCAN3D_OK;
}

// the protocol of one scan on one slot; src = this rank's points (device memory, or host memory in the GPU-less mode)
static int gather_impl(scan3d_shard* sh, int slot, uint64_t mine, const float* src, cudaStream_t stream, int64_t* total_points,
                       int64_t* counts)
{
    SlotBoard& sb = sh->board->slot[slot];
    const uint64_t q = ++sh->seq[slot];
    sb.count[sh->rank].store((q << 32) | mine, std::memory_order_release);
    // the counts this rank needs: the lower ranks' (its base offset); root needs them all (the total)
    const int need = sh->rank == 0 ? sh->world : sh->rank;
    uint64_t c[MAX_WORLD] = {};
    for (int i = 0; i < sh->world; i++) {
        if (i >= need && !counts && !total_points) break;
        uint64_t w = 0;
        if (!wait_for(sh, [&] { w = sb.count[i].load(std::memory_order_acquire); return (w >> 32) >= q; }))
            return sfail(sh, SCAN3D_ERR_IO, "timed out waiting for rank " + std::to_string(i) + "'s point count");
        c[i] = w & 0xffffffffull;
    }
    uint64_t base = 0, total = 0;
    for (int i = 0; i < sh->world; i++) {
        if (i < sh->rank) base += c[i];
        total += c[i];
        if (counts) counts[i] = (int64_t)c[i];
    }
    if (total_points) *total_points = (int64_t)total;
    if (sh->rank > 0) {
        // push: one copy-engine transfer to the final place in root's block -- once root has released the cloud that
        // lived there before (scan q - 1 of this slot)
        if (base + mine > (uint64_t)sh->capacity) return sfail(sh, SCAN3D_ERR_ARG, "more points than the block holds");
        if (!wait_for(sh, [&] { return sb.released.load(std::memory_order_acquire) + 1 >= q; }))
            return sfail(sh, SCAN3D_ERR_IO, "timed out waiting for root to release the slot's previous cloud");
        if (mine) {
            float* dst = static_cast<float*>(sh->block[slot]) + 3 * base;
            if (sh->host_mode) {
                memcpy(dst, src, (size_t)mine * 12);
            } else {
                cudaError_t e = cudaMemcpyAsync(dst, src, (size_t)mine * 12, cudaMemcpyDeviceToDevice, stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
                if (e != cudaSuccess) return sfail(sh, SCAN3D_ERR_CUDA, std::string("push over NVLink: ") + cudaGetErrorString(e));
            }
        }
        sb.pushed[sh->rank].store(q, std::memory_order_release);
    } else {
        // root: its own points are in place already; wait for the others'
        for (int i = 1; i < sh->world; i++)
            if (!wait_for(sh, [&] { return sb.pushed[i].load(std::memory_order_acquire) >= q; }))
                return sfail(sh, SCAN3D_ERR_IO, "timed out waiting for rank " + std::to_string(i) + "'s points");
    }
    return SCAN3D_OK;
}

int scan3d_shard_gather(scan3d_shard* sh, int slot, scan3d_ctx* ctx, int64_t* total_points, int64_t* counts)
{
    if (!sh || !ctx || slot < 0 || slot >= sh->slots || sh->host_mode) return sfail(sh, SCAN3D_ERR_ARG, "scan3d_shard_gather: bad argument");
    if (cudaSetDevice(sh->device) != cudaSuccess) return sfail(sh, SCAN3D_ERR_CUDA, "cudaSetDevice failed");
    if (!ctx->results.has(s3d::POINTS)) return sfail(sh, SCAN3D_ERR_STATE, "scan3d_shard_gather before the ctx's reconstruction");
    // this rank's count (waits for its reconstruction)
    cudaError_t e = cudaMemcpyAsync(sh->h_count, ctx->d_count, 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return sfail(sh, SCAN3D_ERR_CUDA, std::string("count read-back: ") + cudaGetErrorString(e));
    return gather_impl(sh, slot, *sh->h_count, ctx->pts_ext ? ctx->pts_ext : ctx->pts, ctx->stream, total_points, counts);
}

/* The same protocol without any GPU (group created with device < 0: the blocks live in shared memory): this rank's
 * points come from host memory; root's own points must be copied by the caller to scan3d_shard_output(slot) before
 * the call.  Exists so that the ordering logic (counts, base offsets, slot reuse) can be tested on a CPU-only box. */
int scan3d_shard_gather_host(scan3d_shard* sh, int slot, const float* points_host, int64_t count, int64_t* total_points, int64_t* counts)
{
    if (!sh || slot < 0 || slot >= sh->slots || !sh->host_mode || count < 0 || (count && !points_host))
        return sfail(sh, SCAN3D_ERR_ARG, "scan3d_shard_gather_host: bad argument (host-mode groups only)");
    return gather_impl(sh, slot, (uint64_t)count, points_host, nullptr, total_points, counts);
}

}  // extern "C"
