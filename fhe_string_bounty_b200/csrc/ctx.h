// ctx.h -- the opaque context behind tfhe_b200_ctx, shared by c_api.cu and host_api.cu.
#pragma once
#include "../../include/tfhe_b200.h"
#include "fft_core.cuh"
#include "fft16_core.cuh"
#include "fft8_core.cuh"
#include "kernels.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace tbc {

int fail(const std::string &msg);   // records the thread-local error string, returns 1

#define TB_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return tbc::fail(std::string(#expr) + ": " + cudaGetErrorString(e__));                 \
    } while (0)

struct DevBuf {   // owning device allocation; freed on scope exit (error paths included).  The owner sets the device first.
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    // stream-ordered growth for the per-call scratch of the device entry points: cudaFree would synchronise the whole device (and, with
    // several ranks driven by one process, wait for a peer's exchange kernel that itself waits for this rank)
    cudaError_t reserve_on(size_t bytes, cudaStream_t s) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFreeAsync(p, s); if (e != cudaSuccess) return e; }
        p = nullptr; cap = 0;
        cudaError_t e = cudaMallocAsync(&p, bytes, s);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace tbc

struct tfhe_b200_ctx {
    uint64_t id = 0;      // unique per process: programs remember the id of the context they are bound to, not its address
    int device = 0;
    tfhe_b200_params p{};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    bool timed = false;
    // keys
    tbc::DevBuf ksk_packed, ksk_colsum, ksk_planes, ks_digits, bskf, bskf8, tbl16, tbl8, tw_generic, roots, luts;
    int ks_kernel = 2;    // 2: tcgen05 GEMM (keyswitch_tc.cu), 1: mma.sync GEMM (keyswitch_mma.cu), 0: IMAD GEMM (keyswitch.cu); env TFHE_B200_KS_KERNEL=tc|mma|imad
    uint32_t n_luts = 0;
    bool have_ksk = false, have_bsk = false;
    int narrow_kernel = 8;   // classic PBS, levels of <= 2 * SM count ciphertexts: 8 = pbs_v8.cu (8 FFT points per thread, 8 warps per ciphertext; keeps a second copy of the Fourier key in its own layout), 0 = the 1- / 2-ciphertext instances of pbs_v4.cu; env TFHE_B200_NARROW_KERNEL
    bool generic = false;    // parameter sets outside N = 2048, k = 1, l = 1 (or TFHE_B200_PBS_KERNEL=generic): pbs_generic.cu, no fused modulus switch
    int log2_q = 64;         // ciphertext modulus 2^log2_q; < 64: PBS outputs are rounded to multiples of 2^(64 - log2_q) (bootstrap.rs:318-330)
    int sms = 148;
    bool tuned512 = false;   // N = 512, k = 3, one level: pbs_n512.cu serves batches of at least tuned512_min ciphertexts (key copy in bskf8, table in tbl16)
    bool tuned8192 = false;  // N = 8192, k = 1, two levels: pbs_n8192.cu (one ciphertext per two-SM cluster; key copy in bskf8, table in tbl16)
    int tuned512_min = 0;    // 0 = default (SM count); smaller batches stay on the generic kernel
    int narrow_cluster = 1;  // classic levels of at most SM count / 2 ciphertexts: one ciphertext per two-SM cluster (pbs_classic_kernel_v8x2)
    int narrow_max = 0;      // widest level the narrow kernel takes (0 = 2 * SM count); env TFHE_B200_NARROW_MAX
    // staging for the host-pointer entry points
    tbc::DevBuf d_in, d_small, d_out, d_idx;
    // two copy/compute lanes for the host-buffer KS-PBS entry point: H2D of chunk k+1 and D2H of chunk k-1 overlap the
    // kernels of chunk k, and the tail wave of one chunk overlaps the head of the next
    struct Lane { cudaStream_t s = nullptr; tbc::DevBuf in, small, out, idx, digits; };
    Lane lane[2];
    uint64_t launches = 0;
    std::mutex mu;

    size_t big_len() const { return (size_t)p.glwe_dim * p.poly_size + 1; }
    size_t small_len() const { return (size_t)p.lwe_dim + 1; }
    size_t lut_len() const { return (size_t)(p.glwe_dim + 1) * p.poly_size; }
};

namespace tbc {
// shared launch helpers (c_api.cu)
// fused = the keyswitch epilogue applies the PBS modulus switch and writes u16 values; the PBS then reads u16 (classic PBS on
// the tensor-core keyswitch + v3 kernel only; fused_supported() says whether the context can do it)
bool fused_supported(const tfhe_b200_ctx *c);
int do_keyswitch(tfhe_b200_ctx *c, const uint64_t *d_in, uint64_t *d_small, size_t batch, cudaStream_t s,
                 const uint32_t *in_slot = nullptr, DevBuf *digits = nullptr, bool fused = false);
int do_pbs(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, const uint64_t *d_luts, uint64_t *d_out, size_t batch,
           uint32_t n_iters, cudaStream_t s, const uint32_t *out_slot = nullptr, bool fused = false);

// rank r's PBS jobs [lo, hi) of a split level of w jobs: contiguous and balanced, the first w % world ranks take one more
// (multi_gpu.shard_range; the scatter kernel inverts it on the device)
__host__ __device__ inline void shard_range(size_t w, uint32_t r, uint32_t world, size_t &lo, size_t &hi) {
    const size_t base = w / world, rem = w % world;
    lo = r * base + (r < rem ? r : rem);
    hi = lo + base + (r < rem ? 1 : 0);
}
}  // namespace tbc

// the symmetric exchange buffer of one rank (csrc/exchange.cu); here so that the program executor (host_api.cu) can validate it
struct tfhe_b200_exchange {
    tfhe_b200_ctx *ctx = nullptr;
    int device = 0;
    uint32_t rank = 0, world = 1, max_rows = 0;
    size_t lwe_len = 0, flags_bytes = 0, area_bytes = 0;
    tbc::DevBuf local;                         // the symmetric buffer of this rank
    std::vector<void *> peer;                  // peer[r] = rank r's buffer as mapped into this process (peer[rank] = local.p)
    std::vector<bool> opened;                  // mapped through cudaIpcOpenMemHandle (must be closed)
    tbc::DevBuf d_peers;                       // device copy of `peer`
    tbc::DevBuf d_group;                       // per-rank arguments of a single-GPU group launch
    uint64_t epoch = 0;
    bool attached = false;
    bool shares_device = false;                // some peer lives on this very GPU: only tfhe_b200_exchange_group_run may run the exchange
};

namespace tbc {
// send area of the NEXT exchange of `ex`
inline uint64_t *exchange_next_send_area(const tfhe_b200_exchange *ex) {
    return reinterpret_cast<uint64_t *>(static_cast<char *>(ex->local.p) + ex->flags_bytes + (size_t)((ex->epoch + 1) & 1) * ex->area_bytes);
}
// The scatter exchange after a split level of w PBS jobs (csrc/exchange.cu): every rank's share (shard_range) is pulled from that rank's
// send area and row i of rank r's share lands in arena row out_slot[lo_r + i].  No validation and no locking: the caller holds the
// context's mutex and has checked the exchange.  exchange_scatter: one rank of a one-process-per-GPU world; exchange_scatter_group: all
// `world` ranks of one GPU in one cooperative launch (arenas[r] / out_slots[r] are rank r's).
int exchange_scatter(tfhe_b200_exchange *ex, uint32_t w, const uint32_t *out_slot, uint64_t *arena, cudaStream_t s);
int exchange_scatter_group(tfhe_b200_exchange *const *group, uint32_t world, uint32_t w, const uint32_t *const *out_slots,
                           uint64_t *const *arenas, cudaStream_t s);
}  // namespace tbc
