// bmx_exchange.cu -- the exchange step of the sharded scan, inside the library, over NVLink peer memory.
//
// The reference has one device (BoyreMoore/BoyreMoore/BoyreMoore.cpp:217-219) and splits its text into word
// ranges WITHOUT overlap (:119-141), so it has nothing to exchange.  The sharded scan (SURVEY 8e) does: every
// rank must learn the global hit count and rank `dst` must receive the concatenation of the per-shard position
// lists (rank order == ascending order).  Round 1 did that with one NCCL all-gather per step through
// torch.distributed; its kernel had to wait for SMs behind the persistent scan grid and its completion needed a
// host synchronisation per step.  Here the step is two tiny kernels and no host involvement:
//
//   post     (stream-ordered behind the scan of step q on rank r)  stores {count, held, sent} into the mailbox
//            slot [q % depth][r] of EVERY rank and the first head_cap positions into rank dst's mailbox, through
//            peer pointers (NVLink P2P stores; cudaIpc mappings when the ranks are processes), then publishes
//            the step number with st.release.sys.  Lists longer than head_cap (dense texts) put their tail into
//            the per-source tail areas of dst (two per source, alternating).
//   collect  (any later point of the same stream) waits for the world's step numbers with ld.acquire.sys, sums
//            the counts, concatenates the lists on dst, writes {total, per-rank counts, list length} into a
//            host-mapped result ring and returns one credit (ack) to every source, which is what lets a source
//            reuse the slot depth steps later.
//
// Nothing here waits for the host and the host waits for nothing: bmx_exchange_wait() polls the result ring
// in pinned memory.  A rank never waits for another rank's *scan*, only (in collect) for its post, and a
// caller that collects step q-1 after posting step q hides even that.  Every device-side wait has a timeout
// (BMX_XCHG_TIMEOUT_MS, default 20 s) that turns a dead peer into an error status instead of a hung GPU.
#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "bmx_ctx.h"

namespace bmx {

constexpr int kMaxRanks = 16;
constexpr int kXchgThreads = 256;
constexpr int kTailBlocks = 32;      // blocks of the post kernel that ship a list's tail
constexpr int kCollectBlocks = 16;   // blocks of the collect kernel on dst
constexpr unsigned long long kTailDepth = 2;   // tail areas per source on dst

struct XHdr {  // one per (slot, source) in every mailbox; seq is stored last (release)
    unsigned long long seq, count, held, sent;
};
struct XResult {  // host-mapped ring, one per slot; seq is stored last (release)
    unsigned long long seq, total, gathered, status;
    unsigned long long counts[kMaxRanks];
};

struct XArgs {
    unsigned char *mb[kMaxRanks];  // mailbox base of every rank as seen from this device ([rank] = own)
    int rank, world, dst, depth;
    unsigned long long seq;
    long long head_cap, tail_cap;
    size_t off_ack, off_tdone, off_head, off_tail;  // the header ring sits at offset 0
    unsigned long long timeout_ns;
    uint32_t *local;  // [0] tail blocks done, [1] collect blocks done, [2] sticky error bits
    // post
    const unsigned long long *count;
    const int64_t *pos;
    long long pos_cap;
    // collect
    int64_t *out;
    long long out_cap;
    XResult *res;
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.sys.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.sys.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.sys.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Waits until *p >= want (step numbers only grow).  false = timed out.
__device__ __noinline__ bool spin_until_ge(const unsigned long long *p, unsigned long long want, unsigned long long timeout_ns)
{
    unsigned long long t0 = 0;
    for (uint32_t it = 1;; ++it) {
        if (ld_acquire_sys(p) >= want) return true;
        if ((it & 63u) == 0u) {
            const unsigned long long now = global_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > timeout_ns) return false;
            __nanosleep(100);
        }
    }
}

__device__ __forceinline__ XHdr *x_hdr(unsigned char *mb, const XArgs &A, uint32_t slot, int src)
{
    return reinterpret_cast<XHdr *>(mb) + (size_t)slot * A.world + src;
}
__device__ __forceinline__ unsigned long long *x_ack(unsigned char *mb, const XArgs &A)
{
    return reinterpret_cast<unsigned long long *>(mb + A.off_ack);
}
__device__ __forceinline__ unsigned long long *x_tdone(unsigned char *mb, const XArgs &A, uint32_t tslot)
{
    return reinterpret_cast<unsigned long long *>(mb + A.off_tdone) + (size_t)tslot * A.world;
}
__device__ __forceinline__ int64_t *x_head(unsigned char *mb, const XArgs &A, uint32_t slot, int src)
{
    return reinterpret_cast<int64_t *>(mb + A.off_head) + ((size_t)slot * A.world + src) * (size_t)A.head_cap;
}
__device__ __forceinline__ int64_t *x_tail(unsigned char *mb, const XArgs &A, uint32_t tslot, int src)
{
    return reinterpret_cast<int64_t *>(mb + A.off_tail) + ((size_t)tslot * A.world + src) * (size_t)A.tail_cap;
}

// Block 0: credit check, head of the list -> dst, header -> everyone.  Blocks 1..: tail of a long list -> dst.
__global__ void __launch_bounds__(kXchgThreads) xchg_post_kernel(const __grid_constant__ XArgs A)
{
    const int tid = threadIdx.x;
    const unsigned long long c = *A.count;  // the scan and its expand kernel are complete: stream order
    const long long held = A.pos ? ((long long)c < A.pos_cap ? (long long)c : A.pos_cap) : 0;
    const long long room = A.head_cap + A.tail_cap;
    const long long sent = held < room ? held : room;
    const uint32_t slot = (uint32_t)(A.seq % (unsigned long long)A.depth);
    unsigned char *me = A.mb[A.rank];

    if (blockIdx.x == 0) {
        // ring credit: every receiver has consumed the step that used this slot before
        bool good = true;
        if (tid < A.world && A.seq > (unsigned long long)A.depth)
            good = spin_until_ge(x_ack(me, A) + tid, A.seq - (unsigned long long)A.depth, A.timeout_ns);
        if (!__syncthreads_and(good) && tid == 0) atomicOr(A.local + 2, 1u);
        const long long n_head = sent < A.head_cap ? sent : A.head_cap;
        int64_t *hd = x_head(A.mb[A.dst], A, slot, A.rank);
        for (long long i = tid; i < n_head; i += kXchgThreads) hd[i] = A.pos[i];
        __threadfence_system();
        __syncthreads();
        if (tid < A.world) {
            XHdr *h = x_hdr(A.mb[tid], A, slot, A.rank);
            st_relaxed_sys(&h->count, c);
            st_relaxed_sys(&h->held, (unsigned long long)held);
            st_relaxed_sys(&h->sent, (unsigned long long)sent);
            __threadfence_system();
            st_release_sys(&h->seq, A.seq);
        }
        return;
    }
    if (sent <= A.head_cap) return;
    // the tail area of dst is double-buffered (kTailDepth): dst must have consumed the step before the previous one.
    // (Single buffering would deadlock a caller that collects step q-1 BEHIND post q on dst's own stream.)
    __shared__ int s_good;
    const uint32_t tslot = (uint32_t)(A.seq % kTailDepth);
    if (tid == 0) s_good = A.seq <= kTailDepth || spin_until_ge(x_ack(me, A) + A.dst, A.seq - kTailDepth, A.timeout_ns) ? 1 : 0;
    __syncthreads();
    if (!s_good && tid == 0) atomicOr(A.local + 2, 2u);
    int64_t *tl = x_tail(A.mb[A.dst], A, tslot, A.rank);
    const long long n_tail = sent - A.head_cap;
    const long long stride = (long long)(gridDim.x - 1) * kXchgThreads;
    for (long long i = (long long)(blockIdx.x - 1) * kXchgThreads + tid; i < n_tail; i += stride) tl[i] = A.pos[A.head_cap + i];
    __threadfence_system();
    __syncthreads();
    if (tid == 0 && atomicAdd(A.local + 0, 1u) == gridDim.x - 2) {  // the last tail block publishes
        A.local[0] = 0u;
        __threadfence_system();
        st_release_sys(x_tdone(A.mb[A.dst], A, tslot) + A.rank, A.seq);
    }
}

// Every rank: wait for the world's headers of this step, total = sum of counts.  dst: concatenate the lists.
// The gathered list is always a PREFIX of the global ascending list: it stops behind the first rank that
// could not ship its whole list (capacity of its own buffer, or of head + tail).
__global__ void __launch_bounds__(kXchgThreads) xchg_collect_kernel(const __grid_constant__ XArgs A)
{
    __shared__ unsigned long long s_count[kMaxRanks], s_sent[kMaxRanks], s_take[kMaxRanks], s_off[kMaxRanks];
    __shared__ unsigned long long s_total, s_len;
    __shared__ int s_last;
    const int tid = threadIdx.x;
    const uint32_t slot = (uint32_t)(A.seq % (unsigned long long)A.depth);
    unsigned char *me = A.mb[A.rank];
    const bool gather = A.rank == A.dst && A.out != nullptr;

    bool good = true;
    if (tid < A.world) {
        XHdr *h = x_hdr(me, A, slot, tid);
        good = spin_until_ge(&h->seq, A.seq, A.timeout_ns);
        s_count[tid] = ld_relaxed_sys(&h->count);
        s_sent[tid] = ld_relaxed_sys(&h->sent);
        if (gather && (long long)s_sent[tid] > A.head_cap)
            good = good && spin_until_ge(x_tdone(me, A, (uint32_t)(A.seq % kTailDepth)) + tid, A.seq, A.timeout_ns);
    }
    if (!__syncthreads_and(good) && tid == 0) atomicOr(A.local + 2, 4u);
    if (tid == 0) {
        unsigned long long off = 0, total = 0;
        bool complete = true;
        for (int r = 0; r < A.world; ++r) {
            total += s_count[r];
            const unsigned long long take = complete ? s_sent[r] : 0ull;
            s_off[r] = off;
            s_take[r] = take;
            off += take;
            if (s_sent[r] != s_count[r]) complete = false;
        }
        s_total = total;
        s_len = off;
    }
    __syncthreads();
    if (gather) {
        const long long stride = (long long)gridDim.x * kXchgThreads;
        for (int r = 0; r < A.world; ++r) {
            const long long take = (long long)s_take[r], base = (long long)s_off[r];
            const int64_t *hd = x_head(me, A, slot, r), *tl = x_tail(me, A, (uint32_t)(A.seq % kTailDepth), r);
            for (long long i = (long long)blockIdx.x * kXchgThreads + tid; i < take && base + i < A.out_cap; i += stride)
                A.out[base + i] = __ldcv(i < A.head_cap ? hd + i : tl + (i - A.head_cap));  // written by a peer: bypass L1
        }
    }
    // the block that finishes last reports to the host and returns the credits
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(A.local + 1, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    if (!s_last) return;
    if (tid == 0) {
        A.local[1] = 0u;
        XResult *R = A.res + slot;
        R->total = s_total;
        R->gathered = gather ? (s_len < (unsigned long long)A.out_cap ? s_len : (unsigned long long)A.out_cap) : 0ull;
        R->status = (unsigned long long)atomicOr(A.local + 2, 0u);
        for (int r = 0; r < A.world; ++r) R->counts[r] = s_count[r];
        __threadfence_system();
        st_release_sys(&R->seq, A.seq);
    }
    if (tid < A.world) st_release_sys(x_ack(A.mb[tid], A) + A.rank, A.seq);  // credit: slot (and tail area) may be reused
}

}  // namespace bmx

using namespace bmx;

struct bmx_exchange {
    int device = 0, rank = 0, world = 1, dst = 0, depth = 4;
    int64_t head_cap = 0, tail_cap = 0;
    size_t off_ack = 0, off_tdone = 0, off_head = 0, off_tail = 0, bytes = 0;
    unsigned char *mailbox = nullptr;
    unsigned char *peer[kMaxRanks] = {};
    bool peer_ipc[kMaxRanks] = {};
    uint32_t *d_local = nullptr;
    XResult *h_res = nullptr, *d_res = nullptr;
    uint64_t posted = 0, collected = 0;
    bool connected = false;
    unsigned long long timeout_ns = 20ull * 1000 * 1000 * 1000;
};

static XArgs make_args(const bmx_exchange *x, uint64_t seq)
{
    XArgs a{};
    for (int r = 0; r < x->world; ++r) a.mb[r] = x->peer[r];
    a.rank = x->rank;
    a.world = x->world;
    a.dst = x->dst;
    a.depth = x->depth;
    a.seq = seq;
    a.head_cap = x->head_cap;
    a.tail_cap = x->tail_cap;
    a.off_ack = x->off_ack;
    a.off_tdone = x->off_tdone;
    a.off_head = x->off_head;
    a.off_tail = x->off_tail;
    a.timeout_ns = x->timeout_ns;
    a.local = x->d_local;
    a.res = x->d_res;
    return a;
}

extern "C" {

int bmx_exchange_create(int device, int rank, int world, int dst, int64_t head_cap, int64_t tail_cap, int depth,
                        bmx_exchange **out)
{
    if (!out) return fail(BMX_E_BADARG, "bmx_exchange_create: out is NULL");
    *out = nullptr;
    if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world || dst < 0 || dst >= world)
        return fail(BMX_E_BADARG, "bmx_exchange_create: rank %d / dst %d / world %d (1..%d)", rank, dst, world, kMaxRanks);
    if (head_cap < 0 || tail_cap < 0 || depth < 2 || depth > 64)
        return fail(BMX_E_BADARG, "bmx_exchange_create: head_cap/tail_cap >= 0 and 2 <= depth <= 64 required");
    if (int rc = check_device(device)) return rc;
    BMX_CUDA(cudaSetDevice(device));
    bmx_exchange *x = new (std::nothrow) bmx_exchange();
    if (!x) return fail(BMX_E_NOMEM, "out of host memory");
    x->device = device;
    x->rank = rank;
    x->world = world;
    x->dst = dst;
    x->depth = depth;
    x->head_cap = head_cap;
    x->tail_cap = tail_cap;
    if (const int ms = env_int("BMX_XCHG_TIMEOUT_MS", 0); ms > 0) x->timeout_ns = (unsigned long long)ms * 1000000ull;
    // the same offsets on every rank (a writer computes addresses inside dst's mailbox from them); only dst
    // backs the list areas with memory
    auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
    x->off_ack = align(sizeof(XHdr) * (size_t)depth * world);
    x->off_tdone = x->off_ack + align(8 * (size_t)world);
    x->off_head = x->off_tdone + align(8 * (size_t)world * kTailDepth);
    x->off_tail = x->off_head + align(8 * (size_t)depth * world * (size_t)head_cap);
    x->bytes = rank == dst ? x->off_tail + align(8 * (size_t)world * (size_t)tail_cap * kTailDepth) : x->off_head;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&x->mailbox), x->bytes);  // plain cudaMalloc: IPC-exportable
    if (e == cudaSuccess) e = cudaMemset(x->mailbox, 0, std::min(x->bytes, x->off_head));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&x->d_local), 64);
    if (e == cudaSuccess) e = cudaMemset(x->d_local, 0, 64);
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&x->h_res), sizeof(XResult) * (size_t)depth, cudaHostAllocMapped);
    if (e == cudaSuccess) {
        memset(x->h_res, 0, sizeof(XResult) * (size_t)depth);
        e = cudaHostGetDevicePointer(reinterpret_cast<void **>(&x->d_res), x->h_res, 0);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        bmx_exchange_destroy(x);
        return fail(e == cudaErrorMemoryAllocation ? BMX_E_NOMEM : BMX_E_CUDA, "bmx_exchange_create: %s", cudaGetErrorString(e));
    }
    x->peer[rank] = x->mailbox;
    x->connected = world == 1;
    *out = x;
    return BMX_OK;
}

void bmx_exchange_destroy(bmx_exchange *x)
{
    if (!x) return;
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < x->world; ++r)
        if (x->peer_ipc[r] && x->peer[r]) cudaIpcCloseMemHandle(x->peer[r]);
    if (x->mailbox) cudaFree(x->mailbox);
    if (x->d_local) cudaFree(x->d_local);
    if (x->h_res) cudaFreeHost(x->h_res);
    (void)cudaGetLastError();
    delete x;
}

int bmx_exchange_handle(bmx_exchange *x, void *handle_out)
{
    if (!x || !handle_out) return fail(BMX_E_BADARG, "bmx_exchange_handle: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == BMX_EXCHANGE_HANDLE_BYTES, "handle size");
    BMX_CUDA(cudaSetDevice(x->device));
    cudaIpcMemHandle_t h;
    BMX_CUDA(cudaIpcGetMemHandle(&h, x->mailbox));
    memcpy(handle_out, &h, sizeof h);
    return BMX_OK;
}

int bmx_exchange_connect(bmx_exchange *x, const void *handles)
{
    if (!x || (!handles && x->world > 1)) return fail(BMX_E_BADARG, "bmx_exchange_connect: NULL argument");
    BMX_CUDA(cudaSetDevice(x->device));
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank || x->peer[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const unsigned char *>(handles) + (size_t)r * sizeof h, sizeof h);
        void *p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(BMX_E_EXCHANGE, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
        }
        x->peer[r] = static_cast<unsigned char *>(p);
        x->peer_ipc[r] = true;
    }
    x->connected = true;
    return BMX_OK;
}

int bmx_exchange_connect_local(bmx_exchange *const *all, int world)
{
    if (!all || world < 1 || world > kMaxRanks) return fail(BMX_E_BADARG, "bmx_exchange_connect_local: bad argument");
    for (int r = 0; r < world; ++r)
        if (!all[r] || all[r]->world != world || all[r]->rank != r)
            return fail(BMX_E_BADARG, "bmx_exchange_connect_local: entry %d is not rank %d of a world of %d", r, r, world);
    ScopedDevice keep;
    for (int a = 0; a < world; ++a) {
        BMX_CUDA(cudaSetDevice(all[a]->device));
        for (int b = 0; b < world; ++b) {
            if (all[b]->device != all[a]->device) {
                int can = 0;
                BMX_CUDA(cudaDeviceCanAccessPeer(&can, all[a]->device, all[b]->device));
                if (!can) return fail(BMX_E_EXCHANGE, "device %d cannot access device %d", all[a]->device, all[b]->device);
                const cudaError_t e = cudaDeviceEnablePeerAccess(all[b]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                    return fail(BMX_E_EXCHANGE, "cudaDeviceEnablePeerAccess(%d -> %d): %s", all[a]->device, all[b]->device, cudaGetErrorString(e));
                (void)cudaGetLastError();
            }
            all[a]->peer[b] = all[b]->mailbox;
        }
        all[a]->connected = true;
    }
    return BMX_OK;
}

int bmx_exchange_post(bmx_exchange *x, bmx_scanner *s, void *stream, uint64_t *seq_out)
{
    if (!x || !s) return fail(BMX_E_BADARG, "bmx_exchange_post: NULL argument");
    if (!x->connected) return fail(BMX_E_BADARG, "bmx_exchange_post: exchange is not connected");
    if (s->device != x->device) return fail(BMX_E_BADARG, "bmx_exchange_post: scanner on device %d, exchange on %d", s->device, x->device);
    if (x->posted - x->collected >= (uint64_t)x->depth - 1)
        return fail(BMX_E_BADARG, "bmx_exchange_post: %llu steps posted but not collected (depth %d)",
                    (unsigned long long)(x->posted - x->collected), x->depth);
    if (x->tail_cap > 0 && x->posted - x->collected >= kTailDepth)
        return fail(BMX_E_BADARG, "bmx_exchange_post: with a tail area at most %d steps may be posted and not collected", (int)kTailDepth);
    BMX_CUDA(cudaSetDevice(x->device));
    XArgs a = make_args(x, x->posted + 1);
    a.count = result_slot(s);
    a.pos = s->positions ? s->d_pos_out : nullptr;
    a.pos_cap = s->positions ? s->pos_cap : 0;
    const int grid = 1 + (s->positions && s->pos_cap > x->head_cap && x->tail_cap > 0 ? kTailBlocks : 0);
    xchg_post_kernel<<<grid, kXchgThreads, 0, static_cast<cudaStream_t>(stream)>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "exchange post launch: %s", cudaGetErrorString(e));
    x->posted += 1;
    if (seq_out) *seq_out = x->posted;
    return BMX_OK;
}

int bmx_exchange_collect(bmx_exchange *x, int64_t *d_out, int64_t out_cap, void *stream, uint64_t *seq_out)
{
    if (!x || out_cap < 0) return fail(BMX_E_BADARG, "bmx_exchange_collect: bad argument");
    if (x->collected >= x->posted) return fail(BMX_E_BADARG, "bmx_exchange_collect: nothing posted");
    BMX_CUDA(cudaSetDevice(x->device));
    XArgs a = make_args(x, x->collected + 1);
    a.out = x->rank == x->dst ? d_out : nullptr;
    a.out_cap = a.out ? out_cap : 0;
    const int grid = a.out ? kCollectBlocks : 1;
    xchg_collect_kernel<<<grid, kXchgThreads, 0, static_cast<cudaStream_t>(stream)>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "exchange collect launch: %s", cudaGetErrorString(e));
    x->collected += 1;
    if (seq_out) *seq_out = x->collected;
    return BMX_OK;
}

int bmx_exchange_wait(bmx_exchange *x, uint64_t seq, uint64_t *total_out, uint64_t *counts_out, int64_t *gathered_out)
{
    if (!x || seq == 0 || seq > x->collected) return fail(BMX_E_BADARG, "bmx_exchange_wait: step %llu was not collected", (unsigned long long)seq);
    volatile XResult *R = x->h_res + (seq % (uint64_t)x->depth);
    const auto t0 = std::chrono::steady_clock::now();
    const double limit_s = (double)x->timeout_ns * 1e-9 * 2.0 + 5.0;
    for (uint32_t it = 1;; ++it) {
        const unsigned long long have = __atomic_load_n(const_cast<unsigned long long *>(&R->seq), __ATOMIC_ACQUIRE);
        if (have >= seq) {
            if (have != seq)
                return fail(BMX_E_BADARG, "bmx_exchange_wait: the result of step %llu was overwritten by step %llu (wait within depth steps)",
                            (unsigned long long)seq, have);
            break;
        }
        if ((it & 1023u) == 0u) {
            // a failed kernel never writes its result: notice that instead of spinning forever
            if (cudaPeekAtLastError() != cudaSuccess) return fail(BMX_E_CUDA, "bmx_exchange_wait: %s", cudaGetErrorString(cudaGetLastError()));
            if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > limit_s)
                return fail(BMX_E_EXCHANGE, "bmx_exchange_wait: step %llu did not complete within %.0f s", (unsigned long long)seq, limit_s);
            sched_yield();
        }
    }
    if (R->status != 0)
        return fail(BMX_E_EXCHANGE, "exchange step %llu timed out on the device (status bits %llu: 1 ring credit, 2 tail credit, 4 peer post)",
                    (unsigned long long)seq, (unsigned long long)R->status);
    if (total_out) *total_out = R->total;
    if (gathered_out) *gathered_out = (int64_t)R->gathered;
    if (counts_out)
        for (int r = 0; r < x->world; ++r) counts_out[r] = R->counts[r];
    return BMX_OK;
}

}  // extern "C"
