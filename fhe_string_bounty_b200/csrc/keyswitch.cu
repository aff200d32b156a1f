// keyswitch.cu -- batched LWE keyswitch (big key -> small key) for sm_100a.
//
// Replaces core_crypto/algorithms/lwe_keyswitch.rs:96-170 (+ the signed decomposition of
// commons/math/decomposition/{decomposer.rs:98-152, iter.rs:37-50,120-127} and
// slice_algorithms.rs:363-461) for a whole batch at once:
//     out[b] = (0, ..., 0, body_b) - sum_{i < kN} sum_{lvl} digit(a_{b,i})[lvl] * KSK[i][lvl][.]
// i.e. an integer GEMM  D[batch x (kN*l)] * KSK[(kN*l) x (n+1)]  in wrapping u64 arithmetic, so the
// keyswitch key is streamed once per 64-ciphertext tile instead of once per ciphertext.
//
// Exactness: wrapping u64 sums are associative, so any summation order is bit-identical to the reference.
// Signed digits d in [-B/2, B/2] are applied as d' = d + B/2 >= 0 (one mad.wide.u32 + one mad.lo.u32 per
// u64 MAC) and the bias B/2 * sum_r KSK[r][j] is added back from a column sum computed at key upload.
#include "kernels.h"

namespace tbks {

constexpr int TILE_B = 64;     // ciphertexts per CTA
constexpr int TILE_J = 128;    // output columns per CTA
constexpr int CH_I = 8;        // input mask elements per pipeline stage
constexpr int THREADS = 256;   // 8 ciphertext groups (8 cts each) x 32 column groups (4 cols each)

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ksk_packed: [kN*level rows][ldk columns] (rows padded to ldk = multiple of TILE_J, zero filled)
// colsum:     [ldk]  = sum over rows (wrapping)
__global__ void __launch_bounds__(THREADS, 2)
keyswitch_kernel(const uint64_t *__restrict__ lwe_in,     // [batch][in_dim + 1], or an arena indexed by in_slot
                 const uint32_t *__restrict__ in_slot,    // nullptr, or arena slot of each batch element
                 const uint64_t *__restrict__ ksk_packed, const uint64_t *__restrict__ colsum,
                 uint64_t *__restrict__ lwe_out,          // [batch][n + 1]
                 int batch, int in_dim, int n, int ldk, int base_log, int level) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int rows_per_stage = CH_I * level;
    uint64_t *ks[2];
    uint8_t *dg[2];
    ks[0] = reinterpret_cast<uint64_t *>(smem);
    ks[1] = ks[0] + (size_t)rows_per_stage * TILE_J;
    dg[0] = reinterpret_cast<uint8_t *>(ks[1] + (size_t)rows_per_stage * TILE_J);
    dg[1] = dg[0] + rows_per_stage * TILE_B;

    const int tid = threadIdx.x;
    const int tb = tid >> 5;        // ciphertext group: cts tb*8 .. tb*8+7 of the tile
    const int tj = tid & 31;        // column group: cols tj*4 .. tj*4+3 of the tile
    const int b0 = blockIdx.x * TILE_B;
    const int j0 = blockIdx.y * TILE_J;
    const int n_stages = in_dim / CH_I;

    uint64_t acc[8][4];
#pragma unroll
    for (int x = 0; x < 8; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = 0;

    const uint32_t mod_b_mask = (1u << base_log) - 1u;
    const uint32_t half_b = 1u << (base_log - 1);
    const int total_bits = base_log * level;

    auto load_stage = [&](int st, int buf) {
        // KSK rows [st*rows_per_stage, +rows_per_stage), columns [j0, j0 + TILE_J): 16-byte cp.async
        const uint64_t *src = ksk_packed + (size_t)st * rows_per_stage * ldk + j0;
        const int chunks = rows_per_stage * (TILE_J / 2);
        for (int c = tid; c < chunks; c += THREADS) {
            const int r = c / (TILE_J / 2), q = c % (TILE_J / 2);
            cp_async16(ks[buf] + (size_t)r * TILE_J + q * 2, src + (size_t)r * ldk + q * 2);
        }
        cp_async_commit();
        // digits of the 64 x CH_I mask elements of this stage (decomposer.rs:98-152, iter.rs:120-127)
        for (int e = tid; e < TILE_B * CH_I; e += THREADS) {
            const int cl = e / CH_I, ii = e % CH_I;
            const int b = b0 + cl;
            uint64_t x = 0;
            if (b < batch) x = __ldg(lwe_in + (size_t)(in_slot ? in_slot[b] : b) * (in_dim + 1) + st * CH_I + ii);
            // closest_representable(x) >> (64 - total_bits), kept modulo 2^total_bits
            uint32_t state = (uint32_t)(((x >> (63 - total_bits)) + 1) >> 1) & ((1u << total_bits) - 1u);
            for (int lv = 0; lv < level; ++lv) {   // yields level `level` first == KSK row order
                const uint32_t res = state & mod_b_mask;
                state >>= base_log;
                uint32_t carry = ((res - 1u) | state) & res;
                carry >>= base_log - 1;
                state += carry;
                // digit = res - carry*B in [-B/2, B/2]; store digit + B/2 in [0, B]
                dg[buf][(ii * level + lv) * TILE_B + cl] = (uint8_t)(res + half_b - (carry << base_log));
            }
        }
    };

    load_stage(0, 0);
    for (int st = 0; st < n_stages; ++st) {
        const int buf = st & 1;
        if (st + 1 < n_stages) {
            load_stage(st + 1, buf ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const uint64_t *kt = ks[buf];
        const uint8_t *dt = dg[buf];
        for (int r = 0; r < rows_per_stage; ++r) {
            const uint2 dpack = *reinterpret_cast<const uint2 *>(dt + r * TILE_B + tb * 8);
            const ulonglong2 k01 = *reinterpret_cast<const ulonglong2 *>(kt + r * TILE_J + tj * 4);
            const ulonglong2 k23 = *reinterpret_cast<const ulonglong2 *>(kt + r * TILE_J + tj * 4 + 2);
            const uint64_t kv[4] = {k01.x, k01.y, k23.x, k23.y};
#pragma unroll
            for (int x = 0; x < 8; ++x) {
                const uint32_t d = ((x < 4 ? dpack.x : dpack.y) >> (8 * (x & 3))) & 0xffu;
#pragma unroll
                for (int y = 0; y < 4; ++y) {
                    const uint32_t klo = (uint32_t)kv[y], khi = (uint32_t)(kv[y] >> 32);
                    uint64_t a = acc[x][y];
                    a += (uint64_t)d * (uint64_t)klo;             // mad.wide.u32
                    a += (uint64_t)(d * khi) << 32;               // mad.lo.u32 on the high word
                    acc[x][y] = a;
                }
            }
        }
        __syncthreads();
    }

    // out = body * [j == n] + B/2 * colsum[j] - sum d' * K      (lwe_keyswitch.rs:144-147,161-168)
#pragma unroll
    for (int x = 0; x < 8; ++x) {
        const int b = b0 + tb * 8 + x;
        if (b >= batch) continue;
        const uint64_t body = __ldg(lwe_in + (size_t)(in_slot ? in_slot[b] : b) * (in_dim + 1) + in_dim);
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int j = j0 + tj * 4 + y;
            if (j > n) continue;
            uint64_t v = (uint64_t)half_b * __ldg(colsum + j) - acc[x][y];
            if (j == n) v += body;
            lwe_out[(size_t)b * (n + 1) + j] = v;
        }
    }
}

// one-time repack of the reference-layout KSK [rows][n+1] into [rows][ldk] + column sums
__global__ void ksk_pack_kernel(const uint64_t *__restrict__ ksk, uint64_t *__restrict__ packed, int rows, int n1, int ldk) {
    const size_t total = (size_t)rows * ldk;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / ldk;
        const int j = (int)(e % ldk);
        packed[e] = j < n1 ? ksk[r * n1 + j] : 0;
    }
}

__global__ void ksk_colsum_kernel(const uint64_t *__restrict__ packed, uint64_t *__restrict__ colsum, int rows, int ldk) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ldk) return;
    uint64_t s = 0;
    for (int r = 0; r < rows; ++r) s += packed[(size_t)r * ldk + j];
    colsum[j] = s;
}

static size_t ks_smem_bytes(int level) {
    const size_t rows = (size_t)CH_I * level;
    return 2 * (rows * TILE_J * sizeof(uint64_t) + rows * TILE_B);
}

}  // namespace tbks

namespace tbk {

int ks_padded_cols(int n) { return ((n + 1 + tbks::TILE_J - 1) / tbks::TILE_J) * tbks::TILE_J; }

int ks_max_level() {
    int level = 1;
    while (tbks::ks_smem_bytes(level + 1) <= 227 * 1024) ++level;
    return level;                                   // 13: 17 408 bytes per level
}

// The limit is a property of the kernel on the current device, shared by every context of the process: it is set to what the largest
// supported level count needs, so that a context created later (with fewer levels) cannot lower it below an earlier context's launch.
cudaError_t ks_configure() {
    return cudaFuncSetAttribute(tbks::keyswitch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)tbks::ks_smem_bytes(ks_max_level()));
}

cudaError_t launch_ksk_pack(const uint64_t *ksk, uint64_t *packed, uint64_t *colsum, int rows, int n, cudaStream_t stream) {
    const int ldk = ks_padded_cols(n);
    tbks::ksk_pack_kernel<<<1024, 256, 0, stream>>>(ksk, packed, rows, n + 1, ldk);
    tbks::ksk_colsum_kernel<<<(ldk + 127) / 128, 128, 0, stream>>>(packed, colsum, rows, ldk);
    return cudaGetLastError();
}

cudaError_t launch_keyswitch(const uint64_t *lwe_in, const uint32_t *in_slot, const uint64_t *ksk_packed, const uint64_t *colsum, uint64_t *lwe_out,
                             int batch, int in_dim, int n, int base_log, int level, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    const int ldk = ks_padded_cols(n);
    dim3 grid((batch + tbks::TILE_B - 1) / tbks::TILE_B, ldk / tbks::TILE_J);
    tbks::keyswitch_kernel<<<grid, tbks::THREADS, tbks::ks_smem_bytes(level), stream>>>(
        lwe_in, in_slot, ksk_packed, colsum, lwe_out, batch, in_dim, n, ldk, base_log, level);
    return cudaGetLastError();
}

}  // namespace tbk
