// exchange.cu -- the one exchange step of a sharded string operation (SURVEY 8e, K7), done by the GPUs themselves over NVLink peer
// memory: no NCCL call, no host round trip, one kernel launch per exchange.
//
// What crosses the link is tiny (one boolean LWE block per rank for eq / contains, one sign block for lt / le / gt / ge, 1 + index
// blocks for find: 16 KiB each), so the cost of a collective library call is all launch latency and host synchronisation.  Here every
// rank owns a symmetric buffer (cudaMalloc + CUDA IPC handle, opened by every peer):
//
//     [ flags: world x u64 | pad | send rows, epoch parity 0 | send rows, epoch parity 1 ]
//
// A rank's last tree level writes its result rows straight into its own send area (tfhe_b200_program_run_device with d_outputs =
// tfhe_b200_exchange_send_rows).  The exchange kernel then
//   1. publishes: __threadfence_system, st.release.sys of the epoch number into flag[my rank] of every peer's buffer (NVLink stores);
//   2. waits: every CTA spins (ld.acquire.sys, bounded) until all `world` local flags have reached the epoch;
//   3. pulls: 16-byte ld.relaxed.sys loads from every peer's send area (NVLink P2P reads, L1 bypassed) and either concatenates them
//      (all-gather) or adds them word-wise modulo 2^64 (all-reduce: u64 wrap-around addition of LWE words IS the homomorphic addition,
//      lwe_linear_algebra.rs:27-41), writing the result where the finishing program reads its inputs.
// Send areas are double-buffered by epoch parity: a rank can only be one exchange ahead of its slowest peer (it needs that peer's
// flag to finish an exchange, and the peer raises flag e+1 only after its own exchange-e kernel has completed in stream order), so
// epoch e+2 never overwrites rows that a peer is still reading for epoch e.
// A peer that never arrives turns into a launch failure after ~20 s (__trap), never into a hung GPU.
// The scatter kernels below use the same publish / wait steps after every split level of a sharded program (tfhe_b200_program_run_sharded):
// every rank pulls every rank's PBS share and writes each row to its own arena slot.
#include "ctx.h"

#include <memory>

using tbc::DevBuf;
using tbc::DeviceGuard;
using tbc::fail;

namespace {

constexpr int kMaxWorld = 64;
constexpr long long kSpinLimitCycles = 40000000000LL;   // ~20 s at 1.9 GHz

__device__ __forceinline__ void st_release_sys(uint64_t *p, uint64_t v) { asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ ulonglong2 ld_relaxed_sys_v2(const ulonglong2 *p) {
    ulonglong2 v;
    asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint64_t ld_relaxed_sys(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// steps 1 and 2 of every exchange kernel; on return every peer's rows of `epoch` are readable by this CTA
__device__ __forceinline__ void publish_and_wait(void *const *__restrict__ peers, uint32_t rank, uint32_t world, uint64_t epoch) {
    // 1. publish (one CTA): everything the previous kernels of this stream wrote to my send area is visible system-wide first
    if (blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();
        st_release_sys(reinterpret_cast<uint64_t *>(peers[threadIdx.x]) + rank, epoch);
    }
    // 2. wait for every rank's flag in MY buffer
    if (threadIdx.x < world) {
        const uint64_t *flag = reinterpret_cast<const uint64_t *>(peers[rank]) + threadIdx.x;
        const long long t0 = clock64();
        while (ld_acquire_sys(flag) < epoch)
            if (clock64() - t0 > kSpinLimitCycles) __trap();
    }
    __syncthreads();
}

// words16 = number of 16-byte units per rank (rows * lwe_len words rounded up to even, / 2); out is 16-byte aligned
__device__ __forceinline__ void exchange_body(void *const *__restrict__ peers, uint32_t rank, uint32_t world, uint64_t epoch, size_t flags_bytes,
                                              size_t area_bytes, size_t words16, int reduce, ulonglong2 *__restrict__ out) {
    publish_and_wait(peers, rank, world, epoch);
    // 3. pull
    const size_t off = flags_bytes + (size_t)(epoch & 1) * area_bytes;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < words16; i += stride) {
        if (reduce) {
            ulonglong2 acc = make_ulonglong2(0, 0);
            for (uint32_t r = 0; r < world; ++r) {
                const ulonglong2 v = ld_relaxed_sys_v2(reinterpret_cast<const ulonglong2 *>(static_cast<const char *>(peers[r]) + off) + i);
                acc.x += v.x; acc.y += v.y;
            }
            out[i] = acc;
        } else {
            for (uint32_t r = 0; r < world; ++r)
                out[(size_t)r * words16 + i] = ld_relaxed_sys_v2(reinterpret_cast<const ulonglong2 *>(static_cast<const char *>(peers[r]) + off) + i);
        }
    }
}

__global__ void __launch_bounds__(256)
exchange_kernel(void *const *__restrict__ peers, uint32_t rank, uint32_t world, uint64_t epoch, size_t flags_bytes, size_t area_bytes,
                size_t words16, int reduce, ulonglong2 *__restrict__ out) {
    exchange_body(peers, rank, world, epoch, flags_bytes, area_bytes, words16, reduce, out);
}

// Several ranks on ONE GPU (one process driving all of them: the single-GPU tests).  Kernels that wait on one another must not be
// separate launches on one device -- nothing guarantees that they run at the same time -- so the ranks' exchanges run as ONE cooperative
// launch, blockIdx.y = rank, every rank executing exactly the code of the multi-GPU kernel on its own buffers.
struct GroupRank { void *const *peers; ulonglong2 *out; uint64_t epoch; };
__global__ void __launch_bounds__(256)
exchange_group_kernel(const GroupRank *__restrict__ ranks, uint32_t world, size_t flags_bytes, size_t area_bytes, size_t words16, int reduce) {
    const GroupRank g = ranks[blockIdx.y];
    exchange_body(g.peers, blockIdx.y, world, g.epoch, flags_bytes, area_bytes, words16, reduce, g.out);
}

// ---- scatter: the exchange after a split level of a sharded program (tfhe_b200_program_run_sharded*) ----------------------------------
// Rank r's PBS share of a level of w jobs, rows [lo_r, hi_r) of tbc::shard_range, sits contiguously in r's send area; every rank pulls
// every share (its own included) and writes job g's row to ITS arena row out_slot[g].  Rows are k*N+1 words, an odd count at every
// parameter set, so a row and the arena slot it goes to need not share their 16-byte alignment: 8-byte loads and stores, kUnroll of them
// in flight per thread (peer loads take a NVLink round trip).
// The double buffer still holds with one exchange after every split level: whatever runs between two exchanges (the next levels' linear,
// keyswitch and PBS kernels, or nothing for a rank with an empty share), a rank finishes exchange e + 1 only once every peer has raised
// flag e + 1, which a peer does only after its exchange-e kernel -- the last reader of the epoch-e rows -- has completed in stream order.
// So the PBS of the level after exchange e + 1 may overwrite the parity-e send area.  The epochs stay in step because every rank runs
// an exchange after every split level, with or without a share: the plan depends only on (program, world, min_shard_width).
constexpr int kUnroll = 8;

__device__ __forceinline__ void scatter_body(void *const *__restrict__ peers, uint32_t rank, uint32_t world, uint64_t epoch, size_t flags_bytes,
                                             size_t area_bytes, size_t lwe_len, uint32_t w, const uint32_t *__restrict__ out_slot,
                                             uint64_t *__restrict__ arena) {
    publish_and_wait(peers, rank, world, epoch);
    const size_t off = flags_bytes + (size_t)(epoch & 1) * area_bytes;
    const uint32_t base = w / world, rem = w % world, big = rem * (base + 1);   // jobs [0, big) belong to the ranks with base + 1 jobs
    for (uint32_t g = blockIdx.x; g < w; g += gridDim.x) {
        const uint32_t r = g < big ? g / (base + 1) : rem + (g - big) / base;
        size_t lo, hi;
        tbc::shard_range(w, r, world, lo, hi);
        const uint64_t *src = reinterpret_cast<const uint64_t *>(static_cast<const char *>(peers[r]) + off) + (g - lo) * lwe_len;
        uint64_t *dst = arena + (size_t)out_slot[g] * lwe_len;
        for (size_t j0 = threadIdx.x; j0 < lwe_len; j0 += (size_t)kUnroll * blockDim.x) {
            uint64_t v[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = j0 + (size_t)u * blockDim.x;
                if (j < lwe_len) v[u] = ld_relaxed_sys(src + j);
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = j0 + (size_t)u * blockDim.x;
                if (j < lwe_len) dst[j] = v[u];
            }
        }
    }
}

__global__ void __launch_bounds__(256)
scatter_kernel(void *const *__restrict__ peers, uint32_t rank, uint32_t world, uint64_t epoch, size_t flags_bytes, size_t area_bytes,
               size_t lwe_len, uint32_t w, const uint32_t *__restrict__ out_slot, uint64_t *__restrict__ arena) {
    scatter_body(peers, rank, world, epoch, flags_bytes, area_bytes, lwe_len, w, out_slot, arena);
}

// several ranks on one GPU: one cooperative launch, blockIdx.y = rank, as exchange_group_kernel.  The per-rank arguments travel by value
// (64 x 32 bytes fit the kernel parameter space), so a launch needs no upload and no synchronisation.
struct ScatterRank { void *const *peers; const uint32_t *out_slot; uint64_t *arena; uint64_t epoch; };
struct ScatterGroup { ScatterRank r[kMaxWorld]; };
__global__ void __launch_bounds__(256)
scatter_group_kernel(const ScatterGroup g, uint32_t world, size_t flags_bytes, size_t area_bytes, size_t lwe_len, uint32_t w) {
    const ScatterRank &m = g.r[blockIdx.y];
    scatter_body(m.peers, blockIdx.y, world, m.epoch, flags_bytes, area_bytes, lwe_len, w, m.out_slot, m.arena);
}

size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int run_exchange(tfhe_b200_exchange *ex, uint32_t rows, uint64_t *d_out, void *stream, int reduce) {
    if (!ex || !d_out) return fail("null argument");
    if (!ex->attached) return fail("exchange: peers not attached yet (tfhe_b200_exchange_attach)");
    if (ex->shares_device) return fail("exchange: ranks that share a GPU must use tfhe_b200_exchange_group_run (kernels that wait on one another cannot be separate launches on one device)");
    if (rows == 0 || rows > ex->max_rows) return fail("exchange: row count outside [1, max_rows]");
    if ((reinterpret_cast<uintptr_t>(d_out) & 15) != 0) return fail("exchange: output buffer must be 16-byte aligned");
    std::lock_guard<std::mutex> lk(ex->ctx->mu);
    DeviceGuard g(ex->device);
    cudaStream_t s = stream ? (cudaStream_t)stream : ex->ctx->stream;
    const size_t words = (size_t)rows * ex->lwe_len, words16 = (words + 1) / 2;
    ex->epoch += 1;
    const int blocks = (int)std::min<size_t>((size_t)ex->ctx->sms, (words16 + 255) / 256);
    exchange_kernel<<<blocks, 256, 0, s>>>((void *const *)ex->d_peers.p, ex->rank, ex->world, ex->epoch, ex->flags_bytes, ex->area_bytes, words16,
                                           reduce, reinterpret_cast<ulonglong2 *>(d_out));
    TB_CUDA(cudaGetLastError());
    ex->ctx->launches += 1;
    return 0;
}

}  // namespace

namespace tbc {

int exchange_scatter(tfhe_b200_exchange *ex, uint32_t w, const uint32_t *out_slot, uint64_t *arena, cudaStream_t s) {
    ex->epoch += 1;
    const int blocks = (int)std::max<uint32_t>(1, std::min<uint32_t>((uint32_t)ex->ctx->sms, w));
    scatter_kernel<<<blocks, 256, 0, s>>>((void *const *)ex->d_peers.p, ex->rank, ex->world, ex->epoch, ex->flags_bytes, ex->area_bytes,
                                          ex->lwe_len, w, out_slot, arena);
    TB_CUDA(cudaGetLastError());
    ex->ctx->launches += 1;
    return 0;
}

int exchange_scatter_group(tfhe_b200_exchange *const *group, uint32_t world, uint32_t w, const uint32_t *const *out_slots,
                           uint64_t *const *arenas, cudaStream_t s) {
    tfhe_b200_exchange *lead = group[0];
    ScatterGroup g{};
    for (uint32_t r = 0; r < world; ++r) {
        group[r]->epoch += 1;
        g.r[r] = ScatterRank{(void *const *)group[r]->d_peers.p, out_slots[r], arenas[r], group[r]->epoch};
    }
    const unsigned bx = std::max<unsigned>(1, std::min<unsigned>((unsigned)lead->ctx->sms / world, w));
    void *args[] = {(void *)&g, (void *)&world, (void *)&lead->flags_bytes, (void *)&lead->area_bytes, (void *)&lead->lwe_len, (void *)&w};
    TB_CUDA(cudaLaunchCooperativeKernel((const void *)scatter_group_kernel, dim3(bx, world), dim3(256), args, 0, s));
    lead->ctx->launches += 1;
    return 0;
}

}  // namespace tbc

extern "C" {

/* Symmetric exchange buffer of rank `rank` out of `world` ranks (one process per GPU), sized for `max_rows` LWE rows per rank per
 * exchange.  Replaces the CPU reference's shared-memory hand-over at the narrow end of a rayon reduction (e.g. the last levels of
 * are_all_comparisons_block_true, integer/server_key/radix_parallel/scalar_comparison.rs:147-240) when the wide levels are sharded. */
int tfhe_b200_exchange_create(tfhe_b200_ctx *c, uint32_t rank, uint32_t world, uint32_t max_rows, tfhe_b200_exchange **out) {
    if (!out) return fail("null out pointer");
    *out = nullptr;
    if (!c) return fail("null context");
    if (world < 1 || world > kMaxWorld || rank >= world) return fail("exchange: need 1 <= world <= 64 and rank < world");
    if (max_rows < 1) return fail("exchange: max_rows must be >= 1");
    DeviceGuard g(c->device);
    auto ex = std::make_unique<tfhe_b200_exchange>();
    ex->ctx = c; ex->device = c->device; ex->rank = rank; ex->world = world; ex->max_rows = max_rows;
    ex->lwe_len = c->big_len();
    ex->flags_bytes = round_up((size_t)world * 8, 256);
    ex->area_bytes = round_up((size_t)max_rows * ex->lwe_len * 8 + 16, 256);
    TB_CUDA(ex->local.reserve(ex->flags_bytes + 2 * ex->area_bytes));
    TB_CUDA(cudaMemset(ex->local.p, 0, ex->flags_bytes + 2 * ex->area_bytes));
    TB_CUDA(cudaDeviceSynchronize());
    ex->peer.assign(world, nullptr);
    ex->opened.assign(world, false);
    ex->peer[rank] = ex->local.p;
    TB_CUDA(ex->d_peers.reserve((size_t)world * sizeof(void *)));
    if (world == 1) {
        TB_CUDA(cudaMemcpy(ex->d_peers.p, ex->peer.data(), sizeof(void *), cudaMemcpyHostToDevice));
        ex->attached = true;
    }
    *out = ex.release();
    return 0;
}

/* The 64-byte CUDA IPC handle of this rank's buffer, to be handed to every peer process (any transport: the Python driver uses
 * torch.distributed.all_gather). */
int tfhe_b200_exchange_handle(tfhe_b200_exchange *ex, uint8_t handle[64]) {
    if (!ex || !handle) return fail("null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    DeviceGuard g(ex->device);
    cudaIpcMemHandle_t h;
    TB_CUDA(cudaIpcGetMemHandle(&h, ex->local.p));
    std::memcpy(handle, &h, 64);
    return 0;
}

/* handles: world x 64 bytes in rank order (this rank's own entry is ignored).  Maps every peer's buffer into this process. */
int tfhe_b200_exchange_attach(tfhe_b200_exchange *ex, const uint8_t *handles) {
    if (!ex || !handles) return fail("null argument");
    if (ex->attached) return fail("exchange: already attached");
    DeviceGuard g(ex->device);
    for (uint32_t r = 0; r < ex->world; ++r) {
        if (r == ex->rank) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, handles + (size_t)r * 64, 64);
        void *p = nullptr;
        TB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ex->peer[r] = p;
        ex->opened[r] = true;
    }
    TB_CUDA(cudaMemcpy(ex->d_peers.p, ex->peer.data(), (size_t)ex->world * sizeof(void *), cudaMemcpyHostToDevice));
    ex->attached = true;
    return 0;
}

/* Same-process variant (one process driving several GPUs, and the single-GPU tests): peers[r] = the tfhe_b200_exchange of rank r. */
int tfhe_b200_exchange_attach_local(tfhe_b200_exchange *ex, tfhe_b200_exchange *const *peers) {
    if (!ex || !peers) return fail("null argument");
    if (ex->attached) return fail("exchange: already attached");
    DeviceGuard g(ex->device);
    for (uint32_t r = 0; r < ex->world; ++r) {
        if (r == ex->rank) continue;
        if (!peers[r] || peers[r]->world != ex->world || peers[r]->rank != r || peers[r]->max_rows != ex->max_rows)
            return fail("exchange: peer " + std::to_string(r) + " does not match");
        if (peers[r]->device == ex->device) ex->shares_device = true;
        if (peers[r]->device != ex->device) {
            int can = 0;
            TB_CUDA(cudaDeviceCanAccessPeer(&can, ex->device, peers[r]->device));
            if (!can) return fail("exchange: no peer access between the two devices");
            cudaError_t e = cudaDeviceEnablePeerAccess(peers[r]->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else TB_CUDA(e);
        }
        ex->peer[r] = peers[r]->local.p;
    }
    TB_CUDA(cudaMemcpy(ex->d_peers.p, ex->peer.data(), (size_t)ex->world * sizeof(void *), cudaMemcpyHostToDevice));
    ex->attached = true;
    return 0;
}

/* Device pointer of the send area of the NEXT exchange: max_rows x (k*N+1) words.  The rows must be written by work enqueued on the
 * stream the exchange is then called with (e.g. tfhe_b200_program_run_device(..., d_outputs = this pointer, stream)). */
int tfhe_b200_exchange_send_rows(tfhe_b200_exchange *ex, uint64_t **d_rows) {
    if (!ex || !d_rows) return fail("null argument");
    *d_rows = tbc::exchange_next_send_area(ex);
    return 0;
}

/* d_out: world x rows x (k*N+1) words, rank order (16-byte aligned; rows * (k*N+1) odd: each rank's part is padded to an even word
 * count, see tfhe_b200_exchange_gather_stride). */
int tfhe_b200_exchange_all_gather(tfhe_b200_exchange *ex, uint32_t rows, uint64_t *d_out, void *cuda_stream) {
    return run_exchange(ex, rows, d_out, cuda_stream, 0);
}
/* words between two ranks' parts in the all-gather output (rows * (k*N+1) rounded up to an even count: 16-byte transfers) */
size_t tfhe_b200_exchange_gather_stride(const tfhe_b200_exchange *ex, uint32_t rows) {
    return ex ? (((size_t)rows * ex->lwe_len + 1) / 2) * 2 : 0;
}
/* d_out: rows x (k*N+1) words (+ one pad word if that count is odd) = sum over ranks modulo 2^64, i.e. the homomorphic sum. */
int tfhe_b200_exchange_all_reduce_sum(tfhe_b200_exchange *ex, uint32_t rows, uint64_t *d_out, void *cuda_stream) {
    return run_exchange(ex, rows, d_out, cuda_stream, 1);
}

/* One process, several ranks on the same GPU: performs the exchange of EVERY rank of `group` (rank order) in one cooperative launch
 * on `cuda_stream`; d_outs[r] is rank r's output as in all_gather / all_reduce_sum.  The caller orders the stream after every rank's
 * producer work. */
int tfhe_b200_exchange_group_run(tfhe_b200_exchange *const *group, uint32_t world, uint32_t rows, uint64_t *const *d_outs, int reduce,
                                 void *cuda_stream) {
    if (!group || !d_outs || world < 1) return fail("null argument");
    tfhe_b200_exchange *lead = group[0];
    if (!lead) return fail("null exchange");
    for (uint32_t r = 0; r < world; ++r) {
        tfhe_b200_exchange *ex = group[r];
        if (!ex || !ex->attached || ex->world != world || ex->rank != r || ex->device != lead->device || ex->max_rows != lead->max_rows)
            return fail("exchange group: rank " + std::to_string(r) + " does not belong to this single-GPU group");
        if (!d_outs[r] || (reinterpret_cast<uintptr_t>(d_outs[r]) & 15) != 0) return fail("exchange group: outputs must be 16-byte aligned");
    }
    if (rows == 0 || rows > lead->max_rows) return fail("exchange: row count outside [1, max_rows]");
    DeviceGuard g(lead->device);
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : lead->ctx->stream;
    std::vector<GroupRank> h(world);
    for (uint32_t r = 0; r < world; ++r) {
        group[r]->epoch += 1;
        h[r] = GroupRank{(void *const *)group[r]->d_peers.p, reinterpret_cast<ulonglong2 *>(d_outs[r]), group[r]->epoch};
    }
    TB_CUDA(lead->d_group.reserve_on(world * sizeof(GroupRank), s));
    TB_CUDA(cudaMemcpyAsync(lead->d_group.p, h.data(), world * sizeof(GroupRank), cudaMemcpyHostToDevice, s));
    TB_CUDA(cudaStreamSynchronize(s));      // h goes out of scope (test path: a synchronisation here is harmless)
    const size_t words = (size_t)rows * lead->lwe_len;
    size_t words16 = (words + 1) / 2;
    const GroupRank *d_ranks = (const GroupRank *)lead->d_group.p;
    int reduce_i = reduce;
    const unsigned bx = (unsigned)std::max<size_t>(1, std::min<size_t>((size_t)lead->ctx->sms / world, (words16 + 255) / 256));
    void *args[] = {(void *)&d_ranks, (void *)&world, (void *)&lead->flags_bytes, (void *)&lead->area_bytes, (void *)&words16, (void *)&reduce_i};
    TB_CUDA(cudaLaunchCooperativeKernel((const void *)exchange_group_kernel, dim3(bx, world), dim3(256), args, 0, s));
    lead->ctx->launches += 1;
    return 0;
}

int tfhe_b200_exchange_destroy(tfhe_b200_exchange *ex) {
    if (!ex) return 0;
    DeviceGuard g(ex->device);
    cudaDeviceSynchronize();
    for (uint32_t r = 0; r < ex->world; ++r)
        if (ex->opened[r] && ex->peer[r]) cudaIpcCloseMemHandle(ex->peer[r]);
    delete ex;
    return 0;
}

}  // extern "C"
