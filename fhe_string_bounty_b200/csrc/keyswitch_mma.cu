// keyswitch_mma.cu -- batched LWE keyswitch on the tensor cores.
//
// Same result, bit for bit, as keyswitch.cu / core_crypto/algorithms/lwe_keyswitch.rs:96-170: the keyswitch IS a dense
// integer GEMM  out[b][j] = body_b*[j==n] - sum_r digit[b][r] * KSK[r][j]  (r = mask element x level) in Z/2^64.  The
// u64 key is split into its 8 byte planes, the signed digits are biased to unsigned bytes (d' = d + B/2), and
//     S_p[b][j] = sum_r d'[b][r] * byte_p(KSK[r][j])            (u8 x u8 -> s32, wrapping; < 2^32, u32 zero-extended: exact)
// S_p <= K * B * 255 with d' <= B = 2^base_log; the worst accepted shape, kN = 32768 at (base_log, level) = (7, 4), bounds it by
// 4.28e9 (4.25e9 reachable), above 2^31: the epilogue reads each plane sum as a u32.
// runs as 8 interleaved int8 GEMM columns on mma.sync.m16n8k32 (one n8 tile = the 8 planes of one KSK column), then
//     sum_r d' * KSK = sum_p S_p << 8p  (mod 2^64),    out = body*[j==n] + B/2 * colsum[j] - that.
// Two kernels: ks_digits_kernel writes the digit matrix once (decomposer.rs:98-152, iter.rs:120-127), ks_mma_kernel is a
// cp.async-pipelined tiled GEMM with ldmatrix fragment loads and a quad-shuffle epilogue.
#include "kernels.h"

namespace tbkm {

constexpr int BM = 64, BN = 128;          // CTA tile: 64 ciphertexts x 128 GEMM columns (= 16 KSK columns x 8 planes)
constexpr int THREADS = 256;              // 8 warps as 2 (M) x 4 (N); warp tile 32 x 32
constexpr int STAGES = 3;
constexpr int PAD = 16;                   // bytes of row padding in shared memory (conflict-free ldmatrix)

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void *p) {
    unsigned s = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(s));
}
__device__ __forceinline__ void mma_u8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// digits[b][i*level + lv] = signed digit + B/2 (level `level` first, the KSK row order); rows b >= batch are zero
__global__ void __launch_bounds__(256)
ks_digits_kernel(const uint64_t *__restrict__ lwe_in, const uint32_t *__restrict__ in_slot, uint8_t *__restrict__ digits,
                 int batch, int batch_pad, int in_dim, int base_log, int level) {
    const int K = in_dim * level;
    const uint32_t mod_b_mask = (1u << base_log) - 1u, half_b = 1u << (base_log - 1);
    const int total_bits = base_log * level;
    const size_t total = (size_t)batch_pad * in_dim;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / in_dim), i = (int)(e % in_dim);
        uint8_t *dst = digits + (size_t)b * K + (size_t)i * level;
        if (b >= batch) {
            for (int lv = 0; lv < level; ++lv) dst[lv] = 0;
            continue;
        }
        const uint64_t x = __ldg(lwe_in + (size_t)(in_slot ? in_slot[b] : b) * (in_dim + 1) + i);
        uint32_t state = (uint32_t)(((x >> (63 - total_bits)) + 1) >> 1) & ((1u << total_bits) - 1u);
        for (int lv = 0; lv < level; ++lv) {
            const uint32_t res = state & mod_b_mask;
            state >>= base_log;
            uint32_t carry = ((res - 1u) | state) & res;
            carry >>= base_log - 1;
            state += carry;
            dst[lv] = (uint8_t)(res + half_b - (carry << base_log));
        }
    }
}

// bmat[n = j*8 + p][k] = byte p of ksk_packed[k][j]      (k contiguous: the "col" operand of mma.row.col)
__global__ void ksk_planes_kernel(const uint64_t *__restrict__ packed, uint8_t *__restrict__ bmat, int rows, int ldk) {
    const size_t total = (size_t)rows * ldk;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const size_t k = e / ldk;
        const int j = (int)(e % ldk);
        const uint64_t v = packed[e];
#pragma unroll
        for (int p = 0; p < 8; ++p) bmat[((size_t)j * 8 + p) * rows + k] = (uint8_t)(v >> (8 * p));
    }
}

template <int KSTEP>   // bytes of K per pipeline stage = 32 mask elements x level
__global__ void __launch_bounds__(THREADS, 2)
ks_mma_kernel(const uint8_t *__restrict__ digits, const uint8_t *__restrict__ bmat, const uint64_t *__restrict__ colsum,
              const uint64_t *__restrict__ lwe_in, const uint32_t *__restrict__ in_slot, uint64_t *__restrict__ lwe_out,
              int batch, int in_dim, int n, int K, int half_b, int ms_shift) {
    constexpr int LD = KSTEP + PAD;
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned char *As = smem;                              // [STAGES][BM][LD]
    unsigned char *Bs = smem + (size_t)STAGES * BM * LD;   // [STAGES][BN][LD]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wm = warp & 1, wn = warp >> 1;               // warp tile origin: rows wm*32, cols wn*32
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int n_stages = K / KSTEP;

    auto load_stage = [&](int st, int buf) {
        constexpr int CH = KSTEP / 16;                     // 16-byte chunks per row
        const uint8_t *ga = digits + (size_t)m0 * K + (size_t)st * KSTEP;
        const uint8_t *gb = bmat + (size_t)n0 * K + (size_t)st * KSTEP;
        for (int c = tid; c < (BM + BN) * CH; c += THREADS) {
            const int row = c / CH, q = c % CH;
            if (row < BM) cp_async16(As + ((size_t)buf * BM + row) * LD + q * 16, ga + (size_t)row * K + q * 16);
            else cp_async16(Bs + ((size_t)buf * BN + (row - BM)) * LD + q * 16, gb + (size_t)(row - BM) * K + q * 16);
        }
        cp_async_commit();
    };

    int acc[2][4][4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[a][b][c] = 0;

    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < n_stages) load_stage(s, s); else cp_async_commit();
    }
    for (int st = 0; st < n_stages; ++st) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        if (st + STAGES - 1 < n_stages) load_stage(st + STAGES - 1, (st + STAGES - 1) % STAGES); else cp_async_commit();
        const unsigned char *at = As + (size_t)(st % STAGES) * BM * LD;
        const unsigned char *bt = Bs + (size_t)(st % STAGES) * BN * LD;
#pragma unroll
        for (int kk = 0; kk < KSTEP; kk += 32) {
            uint32_t af[2][4], bf[2][4];
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) {
                // four 8x8 b16 matrices: (rows 0-7, bytes 0-15), (rows 8-15, bytes 0-15), (rows 0-7, 16-31), (rows 8-15, 16-31)
                const int row = wm * 32 + mi * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                ldmatrix_x4(af[mi], at + (size_t)row * LD + kk + (lane >> 4) * 16);
            }
#pragma unroll
            for (int nj = 0; nj < 2; ++nj) {
                // two n8 tiles at once: (n 0-7, k 0-15), (n 0-7, k 16-31), (n 8-15, k 0-15), (n 8-15, k 16-31)
                const int nrow = wn * 32 + nj * 16 + (lane & 7) + (lane >> 4) * 8;
                ldmatrix_x4(bf[nj], bt + (size_t)nrow * LD + kk + ((lane >> 3) & 1) * 16);
            }
#pragma unroll
            for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) mma_u8(acc[mi][ni], af[mi], bf[ni >> 1][(ni & 1) * 2], bf[ni >> 1][(ni & 1) * 2 + 1]);
        }
    }

    // epilogue: n8 tile = the 8 byte planes of KSK column j; thread (g = lane/4, t = lane%4) holds planes 2t, 2t+1 of rows g, g+8
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            const int j = (n0 + wn * 32 + ni * 8) >> 3;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint64_t v = ((uint64_t)(uint32_t)acc[mi][ni][2 * h] << (16 * t)) + ((uint64_t)(uint32_t)acc[mi][ni][2 * h + 1] << (16 * t + 8));
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                const int b = m0 + wm * 32 + mi * 16 + g + 8 * h;
                if (t == 0 && b < batch && j <= n) {
                    uint64_t o = (uint64_t)half_b * __ldg(colsum + j) - v;
                    if (j == n) o += __ldg(lwe_in + (size_t)(in_slot ? in_slot[b] : b) * (in_dim + 1) + in_dim);
                    if (ms_shift) {
                        // fused fast_pbs_modulus_switch (fft_impl/common.rs:26-43): the blind rotation only needs round(x / 2^(64 - log2(2N)))
                        reinterpret_cast<uint16_t *>(lwe_out)[(size_t)b * (n + 1) + j] = (uint16_t)(((o >> ms_shift) + 1) >> 1);
                    } else {
                        lwe_out[(size_t)b * (n + 1) + j] = o;
                    }
                }
            }
        }
}

template <int KSTEP>
static cudaError_t launch_mma(const uint8_t *digits, const uint8_t *bmat, const uint64_t *colsum, const uint64_t *lwe_in,
                              const uint32_t *in_slot, uint64_t *lwe_out, int batch, int in_dim, int n, int K, int ldk, int half_b,
                              int ms_shift, cudaStream_t stream) {
    const size_t smem = (size_t)STAGES * (BM + BN) * (KSTEP + PAD);
    // function attributes are per device: set on every launch (microseconds) rather than caching a process-wide flag
    cudaError_t e = cudaFuncSetAttribute(ks_mma_kernel<KSTEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid((batch + BM - 1) / BM, (ldk * 8) / BN);
    ks_mma_kernel<KSTEP><<<grid, THREADS, smem, stream>>>(digits, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, half_b, ms_shift);
    return cudaGetLastError();
}

}  // namespace tbkm

namespace tbk {

bool ks_mma_supported(int level) { return level >= 1 && level <= 7; }

cudaError_t launch_ksk_planes(const uint64_t *packed, uint8_t *bmat, int rows, int ldk, cudaStream_t stream) {
    tbkm::ksk_planes_kernel<<<2048, 256, 0, stream>>>(packed, bmat, rows, ldk);
    return cudaGetLastError();
}

cudaError_t launch_ks_digits(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits, int batch, int batch_pad, int in_dim,
                             int base_log, int level, cudaStream_t stream) {
    const size_t total = (size_t)batch_pad * in_dim;
    const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    tbkm::ks_digits_kernel<<<blocks, 256, 0, stream>>>(lwe_in, in_slot, digits, batch, batch_pad, in_dim, base_log, level);
    return cudaGetLastError();
}

cudaError_t launch_keyswitch_mma(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits_scratch, const uint8_t *bmat,
                                 const uint64_t *colsum, uint64_t *lwe_out, int batch, int in_dim, int n, int base_log, int level,
                                 int ms_log2_2n, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    const int ldk = ks_padded_cols(n);
    const int K = in_dim * level;
    const int batch_pad = ((batch + tbkm::BM - 1) / tbkm::BM) * tbkm::BM;
    cudaError_t e = launch_ks_digits(lwe_in, in_slot, digits_scratch, batch, batch_pad, in_dim, base_log, level, stream);
    if (e != cudaSuccess) return e;
    const int half_b = 1 << (base_log - 1);
    const int ms_shift = ms_log2_2n ? 64 - ms_log2_2n - 1 : 0;   // 0: raw u64 output; else u16 round(x / 2^(64 - log2(2N)))
    switch (level) {
        case 1: return tbkm::launch_mma<32>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 2: return tbkm::launch_mma<64>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 3: return tbkm::launch_mma<96>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 4: return tbkm::launch_mma<128>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 5: return tbkm::launch_mma<160>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 6: return tbkm::launch_mma<192>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        case 7: return tbkm::launch_mma<224>(digits_scratch, bmat, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, ldk, half_b, ms_shift, stream);
        default: return cudaErrorInvalidValue;
    }
}

size_t ks_mma_digits_bytes(int batch, int in_dim, int level) {
    const size_t batch_pad = ((size_t)(batch + tbkm::BM - 1) / tbkm::BM) * tbkm::BM;
    return batch_pad * (size_t)in_dim * level;
}

}  // namespace tbk
