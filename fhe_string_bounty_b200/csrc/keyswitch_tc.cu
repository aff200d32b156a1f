// keyswitch_tc.cu -- the keyswitch GEMM on the 5th-generation tensor cores: tcgen05.mma kind::i8, operands staged by TMA, accumulators in
// Tensor Memory.  Same arithmetic, bit for bit, as keyswitch_mma.cu (the mma.sync version, kept as the A/B reference) and as
// core_crypto/algorithms/lwe_keyswitch.rs:96-170:
//     S_p[b][j] = sum_r d'[b][r] * byte_p(KSK[r][j])      u8 x u8 -> s32 accumulator, read back as u32 and zero-extended: exact, since
//                                                          S_p <= K * B * 255 < 2^32 for every accepted shape (d' <= B = 2^base_log; worst
//                                                          kN = 32768 at (base_log, level) = (7, 4): 4.28e9 bound, 4.25e9 reachable)
//     out[b][j] = body_b * [j == n] + B/2 * colsum[j] - sum_p S_p << 8p          (mod 2^64)
// with d' = signed digit + B/2 written once per batch by ks_digits_kernel, and the key split into its 8 byte planes at upload
// (bmat[n = 8 j + p][k], k contiguous): both operands are K-major byte matrices, exactly what the tensor core wants.
//
// One CTA computes a 128 (ciphertexts) x 256 (= 32 KSK columns x 8 planes) tile of the s32 accumulator:
//   warp 4, one lane   TMA producer: per K block of 128 bytes one 128 x 128 box of digits and one 256 x 128 box of key planes
//                      (cp.async.bulk.tensor.2d, SWIZZLE_128B) into a 4-stage ring, mbarrier expect-tx;
//   warp 5, one lane   MMA issuer: 4 x tcgen05.mma.cta_group::1.kind::i8 (M 128, N 256, K 32) per stage on shared-memory descriptors,
//                      tcgen05.commit hands the stage back to the producer and, after the last K block, the accumulator to the epilogue;
//   warps 0-3          epilogue: tcgen05.ld of the thread's own row (TMEM lane = ciphertext), 8 planes -> one u64, bias, body, optional
//                      fused fast_pbs_modulus_switch (fft_impl/common.rs:26-43), store.
// The GEMM is L2-bandwidth bound, not tensor bound (a 128 x 256 tile streams 3.9 MB of operands for 335 M MACs).  Tile order: blockIdx.x
// walks the key's column tiles, so a wave of CTAs works on ~6 digit tiles (8 MB) against the whole key (63 MB): both stay in the 126 MB L2
// (with the digit tiles in x, ncu showed 970 MB of DRAM reads per 8192 ciphertexts against 147 MB of operands).
#include <cuda.h>

#include "kernels.h"
#include "ring_helpers.cuh"

namespace tbtc {
using namespace tbr;

constexpr int BM = 128, BN = 256, BK = 128, STAGES = 4, UMMA_K = 32;
constexpr int A_BYTES = BM * BK, B_BYTES = BN * BK, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 192;
constexpr int TMEM_COLS = 256;

struct Smem {
    uint8_t a[STAGES][A_BYTES];        // 1024-byte aligned tiles (SWIZZLE_128B atoms are 8 rows x 128 bytes)
    uint8_t b[STAGES][B_BYTES];
    unsigned long long full[STAGES], empty[STAGES], accum;
    uint32_t tmem_base;
};

__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, void *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
// shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp, SmemDescriptor): K-major operand, SWIZZLE_128B, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor (InstrDescriptor): D = S32, A = B = unsigned 8 bit, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(da), "l"(db),
        "r"(kIdesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(void *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
ks_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const uint64_t *__restrict__ colsum,
             const uint64_t *__restrict__ lwe_in, const uint32_t *__restrict__ in_slot, uint64_t *__restrict__ lwe_out, int batch, int in_dim,
             int n, int K, int half_b, int ms_shift) {
    extern __shared__ unsigned char smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;      // x = column tile: the CTAs of a wave share few digit tiles and sweep the whole key (L2 resident)
    const int num_kb = K / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
        mbar_init(&sm.accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = sm.tmem_base;

    if (warp == 4) {
        if (lane == 0) {       // ---- TMA producer ----
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
                mbar_wait(&sm.empty[s], ph ^ 1u);              // first pass: the slot has never been used (parity trick)
                mbar_expect_tx(&sm.full[s], STAGE_BYTES);
                tma_load_2d(sm.a[s], &map_a, kb * BK, m0, &sm.full[s]);
                tma_load_2d(sm.b[s], &map_b, kb * BK, n0, &sm.full[s]);
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {       // ---- MMA issuer ----
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
                mbar_wait(&sm.full[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t da = umma_desc(smem_u32(sm.a[s])), db = umma_desc(smem_u32(sm.b[s]));
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k)          // 32 bytes further along K inside the 128-byte swizzle row: +2 in units of 16 bytes
                    umma_i8(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), (uint32_t)((kb | k) != 0));
                umma_commit(&sm.empty[s]);                      // the stage is free once these MMAs have read it
            }
            umma_commit(&sm.accum);                             // the accumulator is complete once every MMA has retired
        }
    } else {                   // ---- epilogue: warp w owns TMEM lanes 32 w .. 32 w + 31 = ciphertexts m0 + 32 w + lane ----
        mbar_wait(&sm.accum, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int b = m0 + warp * 32 + lane;
        const uint64_t body = b < batch ? __ldg(lwe_in + (size_t)(in_slot ? in_slot[b] : b) * (in_dim + 1) + in_dim) : 0;
#pragma unroll 1
        for (int c = 0; c < BN / 16; ++c) {                     // 16 accumulator columns = the 8 planes of two KSK columns
            uint32_t v[16];
            tmem_ld16(tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(16 * c), v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = (n0 >> 3) + 2 * c + h;
                uint64_t sum = 0;
#pragma unroll
                for (int p = 0; p < 8; ++p) sum += (uint64_t)v[8 * h + p] << (8 * p);
                if (b < batch && j <= n) {
                    uint64_t o = (uint64_t)half_b * __ldg(colsum + j) - sum;
                    if (j == n) o += body;
                    if (ms_shift) reinterpret_cast<uint16_t *>(lwe_out)[(size_t)b * (n + 1) + j] = (uint16_t)(((o >> ms_shift) + 1) >> 1);
                    else lwe_out[(size_t)b * (n + 1) + j] = o;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
}

using EncodeTiled = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                 const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiled encode_tiled_fn() {
    static EncodeTiled fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiled>(p);
    }();
    return fn;
}

// byte matrix [rows][K] (K contiguous) -> tensor map with boxes of box_rows x 128 bytes, 128-byte swizzle
static bool make_map(CUtensorMap *map, const void *base, uint64_t rows, uint64_t K, uint32_t box_rows) {
    EncodeTiled enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t dims[2] = {K, rows}, strides[1] = {K};
    const cuuint32_t box[2] = {(cuuint32_t)BK, box_rows}, estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tbtc

namespace tbk {

bool ks_tc_supported(int in_dim, int level) { return level >= 1 && level <= 7 && (in_dim * level) % tbtc::BK == 0 && tbtc::encode_tiled_fn() != nullptr; }

size_t ks_tc_digits_bytes(int batch, int in_dim, int level) {
    const size_t batch_pad = ((size_t)(batch + tbtc::BM - 1) / tbtc::BM) * tbtc::BM;
    return batch_pad * (size_t)in_dim * level;
}

// digits: scratch of ks_tc_digits_bytes() bytes (written here by ks_digits_kernel of keyswitch_mma.cu); bmat: the key's byte planes
cudaError_t launch_keyswitch_tc(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits_scratch, const uint8_t *bmat,
                                const uint64_t *colsum, uint64_t *lwe_out, int batch, int in_dim, int n, int base_log, int level,
                                int ms_log2_2n, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    const int ldk = ks_padded_cols(n);
    const int K = in_dim * level;
    const int batch_pad = ((batch + tbtc::BM - 1) / tbtc::BM) * tbtc::BM;
    cudaError_t e = launch_ks_digits(lwe_in, in_slot, digits_scratch, batch, batch_pad, in_dim, base_log, level, stream);
    if (e != cudaSuccess) return e;
    CUtensorMap map_a, map_b;
    if (!tbtc::make_map(&map_a, digits_scratch, (uint64_t)batch_pad, (uint64_t)K, tbtc::BM) ||
        !tbtc::make_map(&map_b, bmat, (uint64_t)ldk * 8, (uint64_t)K, tbtc::BN))
        return cudaErrorInvalidValue;
    const size_t smem = sizeof(tbtc::Smem) + 1024;
    e = cudaFuncSetAttribute(tbtc::ks_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int half_b = 1 << (base_log - 1);
    const int ms_shift = ms_log2_2n ? 64 - ms_log2_2n - 1 : 0;
    dim3 grid((ldk * 8) / tbtc::BN, batch_pad / tbtc::BM);
    tbtc::ks_tc_kernel<<<grid, tbtc::THREADS, smem, stream>>>(map_a, map_b, colsum, lwe_in, in_slot, lwe_out, batch, in_dim, n, K, half_b, ms_shift);
    return cudaGetLastError();
}

}  // namespace tbk
