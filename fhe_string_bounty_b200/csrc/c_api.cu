// c_api.cu -- extern "C" boundary of libtfhe_b200.so (see include/tfhe_b200.h for the reference
// interfaces each entry point replaces).  Plain pointers and sizes only; no torch types.
#include "ctx.h"

#include <atomic>
#include <memory>
#include "host/wire.h"
#include <chrono>

namespace {
thread_local std::string g_last_error;
}

namespace tbc {
int fail(const std::string &msg) {
    g_last_error = msg;
    return 1;
}
}  // namespace tbc

using tbc::DevBuf;
using tbc::DeviceGuard;
using tbc::fail;

namespace {

int check_params(const tfhe_b200_params &p) {
    // N = 2048, k = 1, one PBS level: the specialised kernels; every other (N, k) of shortint/parameters/mod.rs and any
    // level count: pbs_generic.cu (classic PBS only)
    const bool tuned = p.poly_size == (uint32_t)tb::kN && p.glwe_dim == 1 && p.pbs_level == 1;
    if (!tuned) {
        if (!tbk::pbs_generic_supported((int)p.poly_size, (int)p.glwe_dim))
            return fail("unsupported (poly_size, glwe_dim): supported pairs are (256,5) (512,3) (512,2) (1024,2) (2048,1) (4096,1) (8192,1) (16384,1) (32768,1)");
        if (p.pbs_level < 1 || p.pbs_level > 8 || p.pbs_base_log * p.pbs_level > 52) return fail("unsupported pbs_level / pbs_base_log");
        if (p.grouping_factor != 0 && p.poly_size > 8192) return fail("multi-bit PBS needs poly_size <= 8192");
    }
    if (p.pbs_base_log < 2 || p.pbs_base_log > 30) return fail("unsupported pbs_base_log");
    if (p.ks_level < 1 || p.ks_base_log < 2 || p.ks_base_log > 7 || p.ks_base_log * p.ks_level > 31)
        return fail("unsupported keyswitch decomposition");
    if ((int)p.ks_level > tbk::ks_max_level())    // the IMAD kernel (the only one above 7 levels) stages 8 * ks_level key rows per step
        return fail("unsupported ks_level " + std::to_string(p.ks_level) + ": at most " + std::to_string(tbk::ks_max_level()) +
                    " levels (the keyswitch's shared-memory stages need 17 408 bytes per level, 227 KB per block)");
    if (p.lwe_dim < 1 || p.lwe_dim > 4096) return fail("unsupported lwe_dim");
    if (p.grouping_factor != 0 && p.grouping_factor != 2 && p.grouping_factor != 3)
        return fail("unsupported grouping_factor (0 = classic, 2 or 3 = multi-bit)");
    if (p.grouping_factor != 0 && p.lwe_dim % p.grouping_factor != 0) return fail("multi-bit: lwe_dim must be a multiple of the grouping factor");
    return 0;
}

}  // namespace

namespace tbc {

// How a tree level of `batch` ciphertexts of the headline set is cut into launches.  Wave times in ms, measured on B200 with
// scripts/level_width_probe.py (n = 742): a wave of 4 per SM 7.2, of 3 per SM 5.49, the narrow kernels 4.37 (<= 2 per SM), 2.75 (<= 1
// per SM) and 1.84 (<= 1 per two-SM cluster).  Only their ratios matter.  narrow = the widest tail the narrow kernels may take (0: none,
// then everything goes to pbs_v4.cu and its launcher picks the instance from the batch size).
struct LevelPlan { size_t four_per_sm, three_per_sm, tail; bool auto_instance; };
LevelPlan plan_classic_level(size_t batch, size_t sms, size_t narrow, bool cluster) {
    if (narrow == 0) return {batch, 0, 0, true};
    const double c4 = 7.2, c3 = 5.49, c2 = 4.37, c1 = 2.75, cx = 1.84;
    const size_t w4 = 4 * sms, w3 = 3 * sms;
    LevelPlan best{batch, 0, 0, false};
    double best_cost = 1e30;
    for (size_t a = 0; a * w4 < batch + w4; ++a) {
        for (size_t b = 0; b <= 3; ++b) {
            const size_t n4 = a * w4 < batch ? a * w4 : batch, left = batch - n4, n3 = b * w3 < left ? b * w3 : left, r = left - n3;
            if ((a && n4 <= (a - 1) * w4) || (b && n3 <= (b - 1) * w3)) continue;      // an empty wave
            double cost = a * c4 + b * c3;
            if (r > narrow || r > 2 * sms) continue;
            if (r) cost += (cluster && r <= sms / 2) ? cx : r <= sms ? c1 : c2;
            cost += 0.02 * ((a != 0) + (b != 0) + (r != 0));                          // ties: fewer launches
            if (cost < best_cost) { best_cost = cost; best = {n4, n3, r, false}; }
        }
    }
    return best;
}

bool fused_supported(const tfhe_b200_ctx *c) { return c->ks_kernel >= 1 && c->p.grouping_factor == 0 && !c->generic; }

int do_keyswitch(tfhe_b200_ctx *c, const uint64_t *d_in, uint64_t *d_small, size_t batch, cudaStream_t s, const uint32_t *in_slot,
                 DevBuf *digits, bool fused) {
    if (fused && !fused_supported(c)) return fail("internal: fused keyswitch requested on an unsupported configuration");
    if (!digits) digits = &c->ks_digits;
    if (!c->have_ksk) return fail("keyswitch key not uploaded");
    if (c->ks_kernel == 2) {   // tcgen05.mma kind::i8 (keyswitch_tc.cu)
        TB_CUDA(digits->reserve_on(tbk::ks_tc_digits_bytes((int)batch, (int)(c->p.glwe_dim * c->p.poly_size), (int)c->p.ks_level), s));
        TB_CUDA(tbk::launch_keyswitch_tc(d_in, in_slot, (uint8_t *)digits->p, (const uint8_t *)c->ksk_planes.p,
                                         (const uint64_t *)c->ksk_colsum.p, d_small, (int)batch, (int)(c->p.glwe_dim * c->p.poly_size),
                                         (int)c->p.lwe_dim, (int)c->p.ks_base_log, (int)c->p.ks_level, fused ? tb::kLogN + 1 : 0, s));
        c->launches += 2;
        return 0;
    }
    if (c->ks_kernel == 1) {
        TB_CUDA(digits->reserve_on(tbk::ks_mma_digits_bytes((int)batch, (int)(c->p.glwe_dim * c->p.poly_size), (int)c->p.ks_level), s));
        TB_CUDA(tbk::launch_keyswitch_mma(d_in, in_slot, (uint8_t *)digits->p, (const uint8_t *)c->ksk_planes.p,
                                          (const uint64_t *)c->ksk_colsum.p, d_small, (int)batch, (int)(c->p.glwe_dim * c->p.poly_size),
                                          (int)c->p.lwe_dim, (int)c->p.ks_base_log, (int)c->p.ks_level, fused ? tb::kLogN + 1 : 0, s));
        c->launches += 2;
        return 0;
    }
    TB_CUDA(tbk::launch_keyswitch(d_in, in_slot, (const uint64_t *)c->ksk_packed.p, (const uint64_t *)c->ksk_colsum.p, d_small,
                                  (int)batch, (int)(c->p.glwe_dim * c->p.poly_size), (int)c->p.lwe_dim,
                                  (int)c->p.ks_base_log, (int)c->p.ks_level, s));
    c->launches += 1;
    return 0;
}

static int do_pbs_kernels(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, const uint64_t *d_luts, uint64_t *d_out, size_t batch,
                          uint32_t n_iters, cudaStream_t s, const uint32_t *out_slot, bool fused);

int do_pbs(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, const uint64_t *d_luts, uint64_t *d_out, size_t batch,
           uint32_t n_iters, cudaStream_t s, const uint32_t *out_slot, bool fused) {
    if (do_pbs_kernels(c, d_small, d_idx, d_luts, d_out, batch, n_iters, s, out_slot, fused)) return 1;
    if (c->log2_q < 64 && batch) {
        TB_CUDA(tbk::launch_round_pow2(d_out, out_slot, (int)batch, (int)c->p.poly_size, (int)c->big_len(), c->log2_q, s));
        c->launches += 1;
    }
    return 0;
}

static int do_pbs_kernels(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, const uint64_t *d_luts, uint64_t *d_out, size_t batch,
                          uint32_t n_iters, cudaStream_t s, const uint32_t *out_slot, bool fused) {
    if (fused && !fused_supported(c)) return fail("internal: fused PBS input requested on an unsupported configuration");
    if (!c->have_bsk) return fail("bootstrap key not uploaded");
    if (!d_luts) return fail("no lookup tables uploaded");
    if (c->tuned512 && batch >= (size_t)(c->tuned512_min ? c->tuned512_min : c->sms)) {
        TB_CUDA(tbk::launch_pbs_n512(d_small, d_idx, d_luts, c->bskf8.p, c->tbl16.p, d_out, out_slot, (int)batch, (int)c->p.lwe_dim,
                                     (int)c->p.pbs_base_log, (int)(n_iters < c->p.lwe_dim ? n_iters : c->p.lwe_dim), s));
        c->launches += 1;
        return 0;
    }
    if (c->tuned8192) {
        TB_CUDA(tbk::launch_pbs_n8192(d_small, d_idx, d_luts, c->bskf8.p, c->tbl16.p, d_out, out_slot, (int)batch, (int)c->p.lwe_dim,
                                      (int)c->p.pbs_base_log, (int)(n_iters < c->p.lwe_dim ? n_iters : c->p.lwe_dim), (int)c->p.lwe_dim, s));
        c->launches += 1;
        return 0;
    }
    if (c->generic) {
        const uint32_t steps = c->p.grouping_factor ? c->p.lwe_dim / c->p.grouping_factor : c->p.lwe_dim;
        TB_CUDA(tbk::launch_pbs_generic(d_small, d_idx, d_luts, c->bskf.p, c->tw_generic.p, d_out, out_slot, (int)batch, (int)c->p.lwe_dim,
                                        (int)c->p.poly_size, (int)c->p.glwe_dim, (int)c->p.pbs_base_log, (int)c->p.pbs_level,
                                        (int)c->p.grouping_factor, (int)(n_iters < steps ? n_iters : steps), s));
        c->launches += 1;
        return 0;
    }
    if (c->p.grouping_factor == 3) {
        const uint32_t groups = c->p.lwe_dim / 3;
        // whole waves of 3 ciphertexts per SM, then the remainder on the 1- / 2-ciphertext instances if it fits them (the launcher
        // picks the instance from the batch size); a remainder or a whole level of at most one ciphertext per SM runs on the
        // 8-points-per-thread kernel pbs_multibit_v8.cu
        const size_t wave = (size_t)3 * c->sms, rem = batch % wave;
        const size_t tail = batch <= (size_t)2 * c->sms ? batch : (rem != 0 && rem <= (size_t)2 * c->sms) ? rem : 0, wide = batch - tail;
        const int steps = (int)(n_iters < groups ? n_iters : groups);
        if (wide) {
            TB_CUDA(tbk::launch_pbs_multibit_v4(d_small, d_idx, d_luts, c->bskf.p, c->tbl16.p, c->roots.p, d_out, out_slot, (int)wide,
                                                (int)c->p.lwe_dim, (int)c->p.pbs_base_log, steps, s));
            c->launches += 1;
        }
        if (tail) {
            const uint64_t *t_small = d_small + wide * (size_t)(c->p.lwe_dim + 1);
            uint64_t *t_out = out_slot ? d_out : d_out + wide * ((size_t)c->p.glwe_dim * c->p.poly_size + 1);
            if (c->narrow_kernel == 8 && tail <= (size_t)(c->narrow_max ? c->narrow_max : c->sms))
                TB_CUDA(tbk::launch_pbs_multibit_v8(t_small, d_idx ? d_idx + wide : nullptr, d_luts, c->bskf8.p, c->tbl8.p, c->roots.p, t_out,
                                                    out_slot ? out_slot + wide : nullptr, (int)tail, (int)c->p.lwe_dim,
                                                    (int)c->p.pbs_base_log, steps, c->narrow_cluster ? c->sms / 2 : 0, s));
            else
                TB_CUDA(tbk::launch_pbs_multibit_v4(t_small, d_idx ? d_idx + wide : nullptr, d_luts, c->bskf.p, c->tbl16.p, c->roots.p, t_out,
                                                    out_slot ? out_slot + wide : nullptr, (int)tail, (int)c->p.lwe_dim,
                                                    (int)c->p.pbs_base_log, steps, s));
            c->launches += 1;
        }
        return 0;
    }
    {
        // A level is cut into at most three launches over contiguous ranges: whole waves of 4 ciphertexts per SM (pbs_v4.cu), waves of 3
        // per SM (the same kernel's 152-register instance), and a tail of at most 2 per SM on the narrow-level kernels (pbs_v8.cu);
        // plan_classic_level picks the cheapest cut from the measured wave times.
        const size_t narrow = c->narrow_kernel == 8 ? (size_t)(c->narrow_max ? c->narrow_max : 2 * c->sms) : 0;
        const LevelPlan plan = plan_classic_level(batch, (size_t)c->sms, narrow, c->narrow_cluster != 0);
        const size_t in_stride = (size_t)(c->p.lwe_dim + 1) * (fused ? 2 : 8), out_stride = (size_t)c->p.glwe_dim * c->p.poly_size + 1;
        size_t done = 0;
        auto wide_launch = [&](size_t count, int cts) -> int {
            const uint64_t *w_small = reinterpret_cast<const uint64_t *>(reinterpret_cast<const char *>(d_small) + done * in_stride);
            TB_CUDA(tbk::launch_pbs_classic_v4(w_small, d_idx ? d_idx + done : nullptr, d_luts, c->bskf.p, c->tbl16.p,
                                               out_slot ? d_out : d_out + done * out_stride, out_slot ? out_slot + done : nullptr, (int)count,
                                               (int)c->p.lwe_dim, (int)c->p.pbs_base_log, (int)n_iters, fused ? 1 : 0, cts, s));
            c->launches += 1;
            done += count;
            return 0;
        };
        if (plan.four_per_sm && wide_launch(plan.four_per_sm, plan.auto_instance ? 0 : 4)) return -1;
        if (plan.three_per_sm && wide_launch(plan.three_per_sm, 3)) return -1;
        if (plan.tail) {
            const uint64_t *t_small = reinterpret_cast<const uint64_t *>(reinterpret_cast<const char *>(d_small) + done * in_stride);
            TB_CUDA(tbk::launch_pbs_classic_v8(t_small, d_idx ? d_idx + done : nullptr, d_luts, c->bskf8.p, c->tbl8.p,
                                               out_slot ? d_out : d_out + done * out_stride, out_slot ? out_slot + done : nullptr, (int)plan.tail,
                                               (int)c->p.lwe_dim, (int)c->p.pbs_base_log, (int)n_iters, fused ? 1 : 0,
                                               c->narrow_cluster ? c->sms / 2 : 0, s));
            c->launches += 1;
        }
        return 0;
    }
}

}  // namespace tbc

using tbc::do_keyswitch;

static int do_pbs(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, uint64_t *d_out, size_t batch, uint32_t n_iters,
                  cudaStream_t s) {
    return tbc::do_pbs(c, d_small, d_idx, c->n_luts ? (const uint64_t *)c->luts.p : nullptr, d_out, batch, n_iters, s, nullptr);
}

extern "C" {

const char *tfhe_b200_last_error(void) { return g_last_error.c_str(); }
const char *tfhe_b200_version(void) { return "tfhe_b200 0.3 (sm_100a; classic + multi-bit(g=3) KS-PBS tuned for N=2048, k=1, l=1; classic KS-PBS for every (N, k, l) of shortint/parameters/mod.rs)"; }

int tfhe_b200_ctx_create(int cuda_device, const tfhe_b200_params *params, tfhe_b200_ctx **out) {
    if (!out) return fail("null out pointer");
    *out = nullptr;
    if (!params) return fail("null params");
    if (check_params(*params)) return 1;
    int count = 0;
    TB_CUDA(cudaGetDeviceCount(&count));
    if (cuda_device < 0 || cuda_device >= count) return fail("no such CUDA device (this engine has no CPU fallback)");
    DeviceGuard g(cuda_device);
    static std::atomic<uint64_t> next_id{1};
    // every early return below (TB_CUDA) destroys the half-built context: streams, events and buffers do not leak
    std::unique_ptr<tfhe_b200_ctx, int (*)(tfhe_b200_ctx *)> guard(new tfhe_b200_ctx(), tfhe_b200_ctx_destroy);
    tfhe_b200_ctx *c = guard.get();
    c->id = next_id.fetch_add(1);
    c->device = cuda_device;
    c->p = *params;
    TB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (auto &e : c->ev) TB_CUDA(cudaEventCreate(&e));
    for (auto &L : c->lane) TB_CUDA(cudaStreamCreateWithFlags(&L.s, cudaStreamNonBlocking));
    if (const char *e = std::getenv("TFHE_B200_KS_KERNEL")) c->ks_kernel = (e[0] == 'i') ? 0 : (e[0] == 'm') ? 1 : 2;   // imad / mma / tc
    if (c->ks_kernel == 2 && !tbk::ks_tc_supported((int)(params->glwe_dim * params->poly_size), (int)params->ks_level)) c->ks_kernel = 1;
    if (!tbk::ks_mma_supported((int)params->ks_level)) c->ks_kernel = 0;
    c->generic = !(params->poly_size == (uint32_t)tb::kN && params->glwe_dim == 1 && params->pbs_level == 1) || params->grouping_factor == 2;
    if (const char *e = std::getenv("TFHE_B200_PBS_KERNEL")) if (e[0] == 'g') c->generic = true;
    if (c->generic) {   // twist table of pbs_generic.cu: exp(i*pi*j/N), j < N/2 (fft/mod.rs:58-69)
        const size_t M = params->poly_size / 2;
        std::vector<double> tw(2 * M);
        const long double pi = 3.14159265358979323846264338327950288L;
        for (size_t j = 0; j < M; ++j) { tw[2 * j] = (double)cosl(pi * j / (long double)params->poly_size); tw[2 * j + 1] = (double)sinl(pi * j / (long double)params->poly_size); }
        TB_CUDA(c->tw_generic.reserve(tw.size() * 8));
        TB_CUDA(cudaMemcpy(c->tw_generic.p, tw.data(), tw.size() * 8, cudaMemcpyHostToDevice));
    }
    c->tuned512 = c->generic && tbk::pbs_n512_supported((int)params->poly_size, (int)params->glwe_dim, (int)params->pbs_level, (int)params->grouping_factor);
    if (const char *e = std::getenv("TFHE_B200_TUNED512")) if (e[0] == '0') c->tuned512 = false;
    if (c->tuned512) TB_CUDA(tbk::pbs_n512_configure());
    c->tuned8192 = c->generic && tbk::pbs_n8192_supported((int)params->poly_size, (int)params->glwe_dim, (int)params->pbs_level, (int)params->pbs_base_log,
                                                              (int)params->grouping_factor);
    if (const char *e = std::getenv("TFHE_B200_TUNED8192")) if (e[0] == '0') c->tuned8192 = false;
    if (c->tuned8192) TB_CUDA(tbk::pbs_n8192_configure());
    TB_CUDA(tbk::pbs_v4_configure());
    TB_CUDA(tbk::pbs_v8_configure());
    if (const char *e = std::getenv("TFHE_B200_NARROW_KERNEL")) c->narrow_kernel = (e[0] == '8') ? 8 : 0;
    if (const char *e = std::getenv("TFHE_B200_NARROW_CLUSTER")) c->narrow_cluster = (e[0] == '0') ? 0 : 1;
    if (const char *e = std::getenv("TFHE_B200_NARROW_MAX")) c->narrow_max = atoi(e);
    TB_CUDA(cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, cuda_device));
    TB_CUDA(tbk::pbs_multibit_v4_configure());
    TB_CUDA(tbk::pbs_multibit_v8_configure());
    {   // roots[e] = exp(i*pi*e/2048): monomial spectra of the multi-bit combine
        std::vector<double> r(2 * 4096);
        const long double pi = 3.14159265358979323846264338327950288L;
        for (int e = 0; e < 4096; ++e) { r[2 * e] = (double)cosl(pi * e / 2048.0L); r[2 * e + 1] = (double)sinl(pi * e / 2048.0L); }
        TB_CUDA(c->roots.reserve(r.size() * 8));
        TB_CUDA(cudaMemcpy(c->roots.p, r.data(), r.size() * 8, cudaMemcpyHostToDevice));
    }
    TB_CUDA(tbk::ks_configure());
    // twiddle tables of the 16- and 8-points-per-thread FFTs
    std::vector<double> tbl16(c->tuned8192 ? 2 * 4352 : 2 * (tb::kM + 64));
    if (c->tuned8192) tbk::pbs_n8192_make_table(tbl16.data());
    else if (c->tuned512) tbk::pbs_n512_make_table(tbl16.data());      // this context never runs the N = 2048 kernels: the buffer holds pbs_n512.cu's table
    else tb16_make_tables(tbl16.data(), tbl16.data() + 2 * tb::kM);
    TB_CUDA(c->tbl16.reserve(tbl16.size() * sizeof(double)));
    TB_CUDA(cudaMemcpyAsync(c->tbl16.p, tbl16.data(), tbl16.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    std::vector<double> tbl8(2 * 24 * 128);
    tb8_make_tables(tbl8.data());
    TB_CUDA(c->tbl8.reserve(tbl8.size() * sizeof(double)));
    TB_CUDA(cudaMemcpyAsync(c->tbl8.p, tbl8.data(), tbl8.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    TB_CUDA(cudaStreamSynchronize(c->stream));
    *out = guard.release();
    return 0;
}

int tfhe_b200_set_ciphertext_modulus_log2(tfhe_b200_ctx *c, uint32_t log2_q) {
    if (!c) return fail("null context");
    if (log2_q < 2 || log2_q > 64) return fail("ciphertext modulus must be 2^2 ... 2^64");
    std::lock_guard<std::mutex> lk(c->mu);
    c->log2_q = (int)log2_q;
    return 0;
}

void tfhe_b200_plan_classic_level(size_t batch, uint32_t sms, size_t narrow_max, int cluster, size_t counts[3]) {
    const tbc::LevelPlan plan = tbc::plan_classic_level(batch, sms, narrow_max, cluster != 0);
    counts[0] = plan.four_per_sm; counts[1] = plan.three_per_sm; counts[2] = plan.tail;
}

int tfhe_b200_set_tuning(tfhe_b200_ctx *c, const char *key, int value) {
    if (!c || !key) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    const std::string k(key);
    if (k == "narrow_kernel") {
        if (value != 0 && value != 8) return fail("narrow_kernel must be 0 or 8");
        c->narrow_kernel = value;
    } else if (k == "narrow_max") {
        if (value < 0) return fail("narrow_max must be >= 0");
        c->narrow_max = value;
    } else if (k == "tuned8192") {
        if (value != 0 && value != 1) return fail("tuned8192 must be 0 or 1");
        if (value == 1 && !(c->bskf8.p && tbk::pbs_n8192_supported((int)c->p.poly_size, (int)c->p.glwe_dim, (int)c->p.pbs_level,
                                                                        (int)c->p.pbs_base_log, (int)c->p.grouping_factor)))
            return fail("tuned8192: not this parameter shape, or the key was uploaded without the tuned copy");
        c->tuned8192 = value;
    } else if (k == "tuned512_min") {
        if (value < 0) return fail("tuned512_min must be >= 0");
        c->tuned512_min = value;
    } else if (k == "narrow_cluster") {
        if (value != 0 && value != 1) return fail("narrow_cluster must be 0 or 1");
        c->narrow_cluster = value;
    } else if (k == "ks_kernel") {
        if (value < 0 || value > 2) return fail("ks_kernel must be 0 (IMAD), 1 (tensor cores, mma.sync) or 2 (tensor cores, tcgen05)");
        if (value >= 1 && !tbk::ks_mma_supported((int)c->p.ks_level)) return fail("tensor-core keyswitch does not support this level count");
        if (value == 2 && !tbk::ks_tc_supported((int)(c->p.glwe_dim * c->p.poly_size), (int)c->p.ks_level))
            return fail("tcgen05 keyswitch: glwe_dim * poly_size * ks_level must be a multiple of 128 (and the driver must export cuTensorMapEncodeTiled)");
        if (value >= 1 && c->have_ksk && !c->ksk_planes.p) return fail("the keyswitch key was uploaded for the IMAD kernel only: upload it again after selecting ks_kernel = 1");
        c->ks_kernel = value;
    } else
        return fail("unknown tuning key '" + k + "'");
    return 0;
}

int tfhe_b200_ctx_destroy(tfhe_b200_ctx *c) {
    if (!c) return 0;
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    for (DevBuf *b : {&c->ksk_packed, &c->ksk_colsum, &c->ksk_planes, &c->ks_digits, &c->bskf, &c->bskf8, &c->tbl16, &c->tbl8, &c->tw_generic, &c->roots, &c->luts, &c->d_in, &c->d_small, &c->d_out, &c->d_idx})
        b->release();
    for (auto &e : c->ev) if (e) cudaEventDestroy(e);
    for (auto &L : c->lane) {
        if (L.s) { cudaStreamSynchronize(L.s); cudaStreamDestroy(L.s); }
        for (DevBuf *b : {&L.in, &L.small, &L.out, &L.idx, &L.digits}) b->release();
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

// raw (standard-layout) keys already in device memory -> the engine's own layouts
static int finish_ksk(tfhe_b200_ctx *c, const tbc::DevBuf &raw) {
    const size_t rows = (size_t)c->p.glwe_dim * c->p.poly_size * c->p.ks_level;
    const int ldk = tbk::ks_padded_cols((int)c->p.lwe_dim);
    TB_CUDA(c->ksk_packed.reserve(rows * ldk * 8));
    TB_CUDA(c->ksk_colsum.reserve((size_t)ldk * 8));
    TB_CUDA(tbk::launch_ksk_pack((const uint64_t *)raw.p, (uint64_t *)c->ksk_packed.p, (uint64_t *)c->ksk_colsum.p, (int)rows,
                                 (int)c->p.lwe_dim, c->stream));
    c->launches += 2;
    if (c->ks_kernel >= 1) {
        TB_CUDA(c->ksk_planes.reserve(rows * (size_t)ldk * 8));
        TB_CUDA(tbk::launch_ksk_planes((const uint64_t *)c->ksk_packed.p, (uint8_t *)c->ksk_planes.p, (int)rows, ldk, c->stream));
        c->launches += 1;
    }
    TB_CUDA(cudaStreamSynchronize(c->stream));
    c->have_ksk = true;
    return 0;
}

static size_t bsk_poly_count(const tfhe_b200_ctx *c) {
    const size_t k1 = c->p.glwe_dim + 1;
    const size_t n_ggsw = c->p.grouping_factor ? (size_t)(c->p.lwe_dim / c->p.grouping_factor) << c->p.grouping_factor : c->p.lwe_dim;
    return n_ggsw * c->p.pbs_level * k1 * k1;
}

static int finish_bsk(tfhe_b200_ctx *c, const tbc::DevBuf &raw) {
    const size_t n_polys = bsk_poly_count(c);
    TB_CUDA(c->bskf.reserve(n_polys * (c->p.poly_size / 2) * sizeof(double) * 2));
    if (c->generic) {
        TB_CUDA(tbk::launch_bsk_convert_generic((const uint64_t *)raw.p, c->bskf.p, c->tw_generic.p, n_polys, (int)c->p.poly_size, c->stream));
        if (c->tuned8192) {    // second copy of the key, per output polynomial, in pbs_n8192.cu's ring order
            TB_CUDA(c->bskf8.reserve(n_polys * (c->p.poly_size / 2) * sizeof(double) * 2));
            TB_CUDA(tbk::launch_bsk_convert_n8192((const uint64_t *)raw.p, c->bskf8.p, c->tbl16.p, (int)c->p.lwe_dim, c->stream));
            c->launches += 1;
        }
        if (c->tuned512) {     // second copy of the key in pbs_n512.cu's ring order
            TB_CUDA(c->bskf8.reserve(n_polys * (c->p.poly_size / 2) * sizeof(double) * 2));
            TB_CUDA(tbk::launch_bsk_convert_n512((const uint64_t *)raw.p, c->bskf8.p, c->tbl16.p, (int)n_polys, c->stream));
            c->launches += 1;
        }
    } else if (c->p.grouping_factor == 3) {
        TB_CUDA(tbk::launch_bsk_convert_multibit_v4((const uint64_t *)raw.p, c->bskf.p, c->tbl16.p, (int)n_polys, c->stream));
        // second copy of the key for the narrow-level kernel (always built: the narrow-kernel choice can change per context at run time)
        TB_CUDA(c->bskf8.reserve(n_polys * tb::kM * sizeof(double) * 2));
        TB_CUDA(tbk::launch_bsk_convert_multibit_v8((const uint64_t *)raw.p, c->bskf8.p, c->tbl8.p, (int)n_polys, c->stream));
        c->launches += 1;
    } else {
        TB_CUDA(tbk::launch_bsk_convert_v4((const uint64_t *)raw.p, c->bskf.p, c->tbl16.p, (int)n_polys, c->stream));
        // second copy of the key, in the narrow-level kernel's (thread, register) order
        TB_CUDA(c->bskf8.reserve(n_polys * tb::kM * sizeof(double) * 2));
        TB_CUDA(tbk::launch_bsk_convert_v8((const uint64_t *)raw.p, c->bskf8.p, c->tbl8.p, (int)n_polys, c->stream));
        c->launches += 1;
    }
    c->launches += 1;
    TB_CUDA(cudaStreamSynchronize(c->stream));
    c->have_bsk = true;
    return 0;
}

int tfhe_b200_upload_ksk(tfhe_b200_ctx *c, const uint64_t *ksk, size_t len) {
    if (!c || !ksk) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    const size_t rows = (size_t)c->p.glwe_dim * c->p.poly_size * c->p.ks_level;
    if (len != rows * (c->p.lwe_dim + 1)) return fail("keyswitch key length does not match the parameters");
    DevBuf raw;
    TB_CUDA(raw.reserve(len * 8));
    TB_CUDA(cudaMemcpyAsync(raw.p, ksk, len * 8, cudaMemcpyHostToDevice, c->stream));
    const int rc = finish_ksk(c, raw);
    raw.release();
    return rc;
}

int tfhe_b200_upload_bsk_std(tfhe_b200_ctx *c, const uint64_t *bsk, size_t len) {
    if (!c || !bsk) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    if (len != bsk_poly_count(c) * c->p.poly_size) return fail("bootstrap key length does not match the parameters");
    DevBuf raw;
    TB_CUDA(raw.reserve(len * 8));
    TB_CUDA(cudaMemcpyAsync(raw.p, bsk, len * 8, cudaMemcpyHostToDevice, c->stream));
    const int rc = finish_bsk(c, raw);
    raw.release();
    return rc;
}

// seeded keys: bodies from the host, masks re-drawn on the device from the compression seed (seeded.cu)
static int upload_seeded(tfhe_b200_ctx *c, const uint8_t *seed, const uint64_t *bodies, size_t len, bool is_bsk) {
    if (!c || !seed || !bodies) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    size_t n_rows, mask_len, body_len;
    if (is_bsk) {
        n_rows = bsk_poly_count(c) / (c->p.glwe_dim + 1);          // GLWE rows
        mask_len = (size_t)c->p.glwe_dim * c->p.poly_size;
        body_len = c->p.poly_size;
    } else {
        n_rows = (size_t)c->p.glwe_dim * c->p.poly_size * c->p.ks_level;   // LWE rows
        mask_len = c->p.lwe_dim;
        body_len = 1;
    }
    if (len != n_rows * body_len) return fail(is_bsk ? "seeded bootstrap key length does not match the parameters"
                                                     : "seeded keyswitch key length does not match the parameters");
    const bool trace = std::getenv("TFHE_B200_TRACE") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    const auto t0 = now();
    DevBuf d_bodies, raw;
    TB_CUDA(d_bodies.reserve(len * 8));
    TB_CUDA(raw.reserve(n_rows * (mask_len + body_len) * 8));
    const auto t1 = now();
    TB_CUDA(cudaMemcpyAsync(d_bodies.p, bodies, len * 8, cudaMemcpyHostToDevice, c->stream));
    const auto t2 = now();
    TB_CUDA(tbk::launch_seeded_expand(seed, (uint64_t *)raw.p, (const uint64_t *)d_bodies.p, n_rows, (uint32_t)mask_len, (uint32_t)body_len,
                                      c->stream));
    c->launches += 1;
    if (trace) cudaStreamSynchronize(c->stream);
    const auto t3 = now();
    const int rc = is_bsk ? finish_bsk(c, raw) : finish_ksk(c, raw);
    const auto t4 = now();
    d_bodies.release();
    raw.release();
    const auto t5 = now();
    if (trace) fprintf(stderr, "[tfhe_b200] upload_seeded(%s): alloc %.2f ms, h2d %.2f, expand %.2f, finish %.2f, free %.2f\n", is_bsk ? "bsk" : "ksk",
                       ms(t0, t1), ms(t1, t2), ms(t2, t3), ms(t3, t4), ms(t4, t5));
    return rc;
}

int tfhe_b200_upload_seeded_ksk(tfhe_b200_ctx *c, const uint8_t seed[16], const uint64_t *bodies, size_t len) {
    return upload_seeded(c, seed, bodies, len, false);
}
int tfhe_b200_upload_seeded_bsk(tfhe_b200_ctx *c, const uint8_t seed[16], const uint64_t *bodies, size_t len) {
    return upload_seeded(c, seed, bodies, len, true);
}

// ---- tfhe-rs wire format (host/wire.h) ----------------------------------------------------------------------------------
static void fill_wire_view(const tbw::ServerKeyView &v, tfhe_b200_wire_server_key *out) {
    std::memset(out, 0, sizeof(*out));
    out->params.lwe_dim = v.lwe_dim; out->params.glwe_dim = v.glwe_dim; out->params.poly_size = v.poly_size;
    out->params.pbs_base_log = v.pbs_base_log; out->params.pbs_level = v.pbs_level;
    out->params.ks_base_log = v.ks_base_log; out->params.ks_level = v.ks_level;
    out->params.grouping_factor = v.grouping_factor; out->params.msg_mod = v.msg_mod; out->params.carry_mod = v.carry_mod;
    out->pbs_order = v.pbs_order; out->deterministic_execution = v.deterministic; out->max_degree = v.max_degree;
    std::memcpy(out->ksk_seed, v.ksk_seed, 16); std::memcpy(out->bsk_seed, v.bsk_seed, 16);
    out->ksk_byte_offset = v.ksk_off; out->ksk_words = v.ksk_len; out->bsk_byte_offset = v.bsk_off; out->bsk_words = v.bsk_len;
}

int tfhe_b200_wire_parse_compressed_server_key(const uint8_t *bytes, size_t len, tfhe_b200_wire_server_key *out) {
    if (!bytes || !out) return fail("null argument");
    try {
        fill_wire_view(tbw::parse_compressed_server_key(bytes, len), out);
    } catch (const std::exception &e) {
        return fail(e.what());
    }
    return 0;
}

int tfhe_b200_load_compressed_server_key(tfhe_b200_ctx *c, const uint8_t *bytes, size_t len) {
    if (!c || !bytes) return fail("null argument");
    tbw::ServerKeyView v;
    try {
        v = tbw::parse_compressed_server_key(bytes, len);
    } catch (const std::exception &e) {
        return fail(e.what());
    }
    const tfhe_b200_params &p = c->p;
    if (v.lwe_dim != p.lwe_dim || v.glwe_dim != p.glwe_dim || v.poly_size != p.poly_size || v.pbs_base_log != p.pbs_base_log ||
        v.pbs_level != p.pbs_level || v.ks_base_log != p.ks_base_log || v.ks_level != p.ks_level ||
        v.grouping_factor != p.grouping_factor || v.msg_mod != p.msg_mod || v.carry_mod != p.carry_mod)
        return fail("serialized server key does not match the context's parameter set");
    // the u64 arrays sit at arbitrary byte offsets inside the blob: copy them out to aligned storage first
    std::vector<uint64_t> ksk(v.ksk_len), bsk(v.bsk_len);
    std::memcpy(ksk.data(), bytes + v.ksk_off, v.ksk_len * 8);
    std::memcpy(bsk.data(), bytes + v.bsk_off, v.bsk_len * 8);
    if (int rc = tfhe_b200_upload_seeded_ksk(c, v.ksk_seed, ksk.data(), ksk.size())) return rc;
    return tfhe_b200_upload_seeded_bsk(c, v.bsk_seed, bsk.data(), bsk.size());
}

int tfhe_b200_wire_read_ciphertexts(const uint8_t *bytes, size_t len, int is_radix, uint64_t *lwe_out, size_t lwe_cap_words,
                                    uint64_t *meta_out, size_t *n_cts, size_t *lwe_len) {
    if (!bytes || !n_cts || !lwe_len) return fail("null argument");
    std::vector<uint64_t> lwe;
    std::vector<tbw::CiphertextMeta> meta;
    size_t ll = 0;
    try {
        tbw::parse_ciphertexts(bytes, len, is_radix != 0, lwe, ll, meta);
    } catch (const std::exception &e) {
        return fail(e.what());
    }
    *n_cts = meta.size();
    *lwe_len = ll;
    if (!lwe_out) return 0;                       // size query
    if (lwe_cap_words < lwe.size()) return fail("output buffer too small for the serialized ciphertexts");
    std::memcpy(lwe_out, lwe.data(), lwe.size() * 8);
    if (meta_out)
        for (size_t i = 0; i < meta.size(); ++i) {
            meta_out[5 * i] = meta[i].degree; meta_out[5 * i + 1] = meta[i].noise_level; meta_out[5 * i + 2] = meta[i].msg_mod;
            meta_out[5 * i + 3] = meta[i].carry_mod; meta_out[5 * i + 4] = meta[i].pbs_order;
        }
    return 0;
}

int tfhe_b200_wire_write_ciphertexts(const uint64_t *lwe, size_t lwe_len, const uint64_t *meta, size_t n_cts, int is_radix,
                                     uint8_t *out, size_t out_cap, size_t *out_len) {
    if (!lwe || !meta || !out_len || lwe_len == 0) return fail("null argument");
    if (!is_radix && n_cts != 1) return fail("a single shortint::Ciphertext holds exactly one LWE ciphertext");
    std::vector<tbw::CiphertextMeta> m(n_cts);
    for (size_t i = 0; i < n_cts; ++i) {
        m[i].degree = meta[5 * i]; m[i].noise_level = meta[5 * i + 1]; m[i].msg_mod = meta[5 * i + 2];
        m[i].carry_mod = meta[5 * i + 3]; m[i].pbs_order = (uint32_t)meta[5 * i + 4];
    }
    const std::vector<uint8_t> b = tbw::write_ciphertexts(lwe, lwe_len, m.data(), n_cts, is_radix != 0);
    *out_len = b.size();
    if (!out) return 0;                           // size query
    if (out_cap < b.size()) return fail("output buffer too small for the serialized ciphertexts");
    std::memcpy(out, b.data(), b.size());
    return 0;
}

int tfhe_b200_upload_luts(tfhe_b200_ctx *c, const uint64_t *luts, uint32_t n_luts) {
    if (!c || !luts || n_luts == 0) return fail("null or empty lookup-table set");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    const size_t bytes = (size_t)n_luts * c->lut_len() * 8;
    TB_CUDA(cudaStreamSynchronize(c->stream));
    TB_CUDA(c->luts.reserve(bytes));
    TB_CUDA(cudaMemcpyAsync(c->luts.p, luts, bytes, cudaMemcpyHostToDevice, c->stream));
    TB_CUDA(cudaStreamSynchronize(c->stream));
    c->n_luts = n_luts;
    return 0;
}

int tfhe_b200_synchronize(tfhe_b200_ctx *c) {
    if (!c) return fail("null context");
    DeviceGuard g(c->device);
    TB_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- device-buffer entry points -----------------------------------------------------------------

int tfhe_b200_keyswitch_batch_device(tfhe_b200_ctx *c, const uint64_t *d_in, uint64_t *d_small, size_t batch, void *stream) {
    if (!c || (batch && (!d_in || !d_small))) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);   // the digit scratch buffer is per context
    DeviceGuard g(c->device);
    return do_keyswitch(c, d_in, d_small, batch, stream ? (cudaStream_t)stream : c->stream);
}

int tfhe_b200_pbs_batch_device(tfhe_b200_ctx *c, const uint64_t *d_small, const uint32_t *d_idx, uint64_t *d_out, size_t batch,
                               void *stream) {
    if (!c || (batch && (!d_small || !d_out))) return fail("null argument");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    return do_pbs(c, d_small, d_idx, d_out, batch, c->p.lwe_dim, stream ? (cudaStream_t)stream : c->stream);
}

int tfhe_b200_ks_pbs_batch_device(tfhe_b200_ctx *c, const uint64_t *d_in, const uint32_t *d_idx, uint64_t *d_out, size_t batch,
                                  void *stream) {
    if (!c || (batch && (!d_in || !d_out))) return fail("null argument");
    if (batch == 0) return 0;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    TB_CUDA(c->d_small.reserve_on(batch * c->small_len() * 8, s));
    TB_CUDA(cudaEventRecord(c->ev[0], s));
    const bool fused = tbc::fused_supported(c);
    if (tbc::do_keyswitch(c, d_in, (uint64_t *)c->d_small.p, batch, s, nullptr, nullptr, fused)) return 1;
    TB_CUDA(cudaEventRecord(c->ev[1], s));
    if (c->n_luts == 0) return fail("no lookup tables uploaded");
    if (tbc::do_pbs(c, (const uint64_t *)c->d_small.p, d_idx, (const uint64_t *)c->luts.p, d_out, batch, c->p.lwe_dim, s, nullptr, fused)) return 1;
    TB_CUDA(cudaEventRecord(c->ev[2], s));
    c->timed = true;
    return 0;
}

// ---- host-buffer entry points ---------------------------------------------------------------------

// a LUT index past the uploaded table would be an out-of-bounds device read: reject it where the indices are host-visible
static int check_lut_indices(const tfhe_b200_ctx *c, const uint32_t *idx, size_t batch) {
    if (!idx) return 0;
    for (size_t i = 0; i < batch; ++i)
        if (idx[i] >= c->n_luts)
            return fail("lut_idx[" + std::to_string(i) + "] = " + std::to_string(idx[i]) + " but only " + std::to_string(c->n_luts) + " lookup tables are uploaded");
    return 0;
}

int tfhe_b200_keyswitch_batch(tfhe_b200_ctx *c, const uint64_t *in, uint64_t *out, size_t batch) {
    if (!c || (batch && (!in || !out))) return fail("null argument");
    if (batch == 0) return 0;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    TB_CUDA(c->d_in.reserve(batch * c->big_len() * 8));
    TB_CUDA(c->d_small.reserve(batch * c->small_len() * 8));
    TB_CUDA(cudaMemcpyAsync(c->d_in.p, in, batch * c->big_len() * 8, cudaMemcpyHostToDevice, c->stream));
    if (do_keyswitch(c, (const uint64_t *)c->d_in.p, (uint64_t *)c->d_small.p, batch, c->stream)) return 1;
    TB_CUDA(cudaMemcpyAsync(out, c->d_small.p, batch * c->small_len() * 8, cudaMemcpyDeviceToHost, c->stream));
    TB_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

static int pbs_host(tfhe_b200_ctx *c, const uint64_t *in, const uint32_t *idx, uint64_t *out, size_t batch, uint32_t n_iters) {
    if (!c || (batch && (!in || !out))) return fail("null argument");
    if (batch == 0) return 0;
    if (n_iters > c->p.lwe_dim) return fail("n_iters exceeds lwe_dim");
    std::lock_guard<std::mutex> lk(c->mu);
    if (check_lut_indices(c, idx, batch)) return 1;
    DeviceGuard g(c->device);
    TB_CUDA(c->d_small.reserve(batch * c->small_len() * 8));
    TB_CUDA(c->d_out.reserve(batch * c->big_len() * 8));
    TB_CUDA(cudaMemcpyAsync(c->d_small.p, in, batch * c->small_len() * 8, cudaMemcpyHostToDevice, c->stream));
    const uint32_t *d_idx = nullptr;
    if (idx) {
        TB_CUDA(c->d_idx.reserve(batch * 4));
        TB_CUDA(cudaMemcpyAsync(c->d_idx.p, idx, batch * 4, cudaMemcpyHostToDevice, c->stream));
        d_idx = (const uint32_t *)c->d_idx.p;
    }
    if (do_pbs(c, (const uint64_t *)c->d_small.p, d_idx, (uint64_t *)c->d_out.p, batch, n_iters, c->stream)) return 1;
    TB_CUDA(cudaMemcpyAsync(out, c->d_out.p, batch * c->big_len() * 8, cudaMemcpyDeviceToHost, c->stream));
    TB_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

int tfhe_b200_pbs_batch(tfhe_b200_ctx *c, const uint64_t *in, const uint32_t *idx, uint64_t *out, size_t batch) {
    if (!c) return fail("null context");
    return pbs_host(c, in, idx, out, batch, c->p.lwe_dim);
}

int tfhe_b200_pbs_batch_partial(tfhe_b200_ctx *c, const uint64_t *in, const uint32_t *idx, uint64_t *out, size_t batch,
                                uint32_t n_iters) {
    return pbs_host(c, in, idx, out, batch, n_iters);
}

int tfhe_b200_ks_pbs_batch(tfhe_b200_ctx *c, const uint64_t *in, const uint32_t *idx, uint64_t *out, size_t batch) {
    if (!c || (batch && (!in || !out))) return fail("null argument");
    if (batch == 0) return 0;
    if (!c->have_ksk) return fail("keyswitch key not uploaded");
    if (!c->have_bsk) return fail("bootstrap key not uploaded");
    if (c->n_luts == 0) return fail("no lookup tables uploaded");
    std::lock_guard<std::mutex> lk(c->mu);
    if (check_lut_indices(c, idx, batch)) return 1;
    DeviceGuard g(c->device);
    // chunks of whole waves (classic: 4 ciphertexts per SM x 4 waves; multi-bit: 3 per SM x 5 waves), alternating between two lanes
    // (stream + staging buffers)
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    const size_t chunk = std::min<size_t>(batch, c->p.grouping_factor ? (size_t)sms * 3 * 5 : (size_t)sms * 4 * 4);
    const size_t L = c->big_len();
    for (auto &ln : c->lane) {
        TB_CUDA(ln.in.reserve(chunk * L * 8));
        TB_CUDA(ln.out.reserve(chunk * L * 8));
        TB_CUDA(ln.small.reserve(chunk * c->small_len() * 8));
        if (idx) TB_CUDA(ln.idx.reserve(chunk * 4));
        if (batch <= chunk) break;   // a single chunk only needs lane 0
    }
    size_t k = 0;
    for (size_t off = 0; off < batch; off += chunk, ++k) {
        tfhe_b200_ctx::Lane &ln = c->lane[k & 1];
        const size_t n = std::min(chunk, batch - off);
        TB_CUDA(cudaMemcpyAsync(ln.in.p, in + off * L, n * L * 8, cudaMemcpyHostToDevice, ln.s));
        if (idx) TB_CUDA(cudaMemcpyAsync(ln.idx.p, idx + off, n * 4, cudaMemcpyHostToDevice, ln.s));
        const bool fused = tbc::fused_supported(c);
        if (tbc::do_keyswitch(c, (const uint64_t *)ln.in.p, (uint64_t *)ln.small.p, n, ln.s, nullptr, &ln.digits, fused)) return 1;
        if (tbc::do_pbs(c, (const uint64_t *)ln.small.p, idx ? (const uint32_t *)ln.idx.p : nullptr, (const uint64_t *)c->luts.p,
                        (uint64_t *)ln.out.p, n, c->p.lwe_dim, ln.s, nullptr, fused))
            return 1;
        TB_CUDA(cudaMemcpyAsync(out + off * L, ln.out.p, n * L * 8, cudaMemcpyDeviceToHost, ln.s));
    }
    TB_CUDA(cudaStreamSynchronize(c->lane[0].s));
    if (k > 1) TB_CUDA(cudaStreamSynchronize(c->lane[1].s));
    return 0;
}

/* PBS -> KS order (PBSOrder::BootstrapKeyswitch, shortint/server_key/mod.rs:859-932): ciphertexts live under the SMALL key */
int tfhe_b200_pbs_ks_batch(tfhe_b200_ctx *c, const uint64_t *in, const uint32_t *idx, uint64_t *out, size_t batch) {
    if (!c || (batch && (!in || !out))) return fail("null argument");
    if (batch == 0) return 0;
    if (c->n_luts == 0) return fail("no lookup tables uploaded");
    std::lock_guard<std::mutex> lk(c->mu);
    if (check_lut_indices(c, idx, batch)) return 1;
    DeviceGuard g(c->device);
    cudaStream_t s = c->stream;
    TB_CUDA(c->d_small.reserve(batch * c->small_len() * 8));
    TB_CUDA(c->d_out.reserve(batch * c->big_len() * 8));
    TB_CUDA(c->d_in.reserve(batch * c->small_len() * 8));
    TB_CUDA(cudaMemcpyAsync(c->d_small.p, in, batch * c->small_len() * 8, cudaMemcpyHostToDevice, s));
    const uint32_t *d_idx = nullptr;
    if (idx) {
        TB_CUDA(c->d_idx.reserve(batch * 4));
        TB_CUDA(cudaMemcpyAsync(c->d_idx.p, idx, batch * 4, cudaMemcpyHostToDevice, s));
        d_idx = (const uint32_t *)c->d_idx.p;
    }
    if (tbc::do_pbs(c, (const uint64_t *)c->d_small.p, d_idx, (const uint64_t *)c->luts.p, (uint64_t *)c->d_out.p, batch, c->p.lwe_dim, s,
                    nullptr))
        return 1;
    if (tbc::do_keyswitch(c, (const uint64_t *)c->d_out.p, (uint64_t *)c->d_in.p, batch, s)) return 1;
    TB_CUDA(cudaMemcpyAsync(out, c->d_in.p, batch * c->small_len() * 8, cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaStreamSynchronize(s));
    return 0;
}

// ---- instrumentation --------------------------------------------------------------------------------

uint64_t tfhe_b200_kernel_launches(const tfhe_b200_ctx *c) { return c ? c->launches : 0; }

int tfhe_b200_time_last_kernels(tfhe_b200_ctx *c, float *ks_ms, float *pbs_ms) {
    if (!c || !c->timed) return fail("no timed ks_pbs call yet");
    DeviceGuard g(c->device);
    TB_CUDA(cudaEventSynchronize(c->ev[2]));
    if (ks_ms) TB_CUDA(cudaEventElapsedTime(ks_ms, c->ev[0], c->ev[1]));
    if (pbs_ms) TB_CUDA(cudaEventElapsedTime(pbs_ms, c->ev[1], c->ev[2]));
    return 0;
}

int tfhe_b200_probe_fp64_tflops(int cuda_device, double *tflops) {
    if (!tflops) return fail("null argument");
    *tflops = 0.0;
    int count = 0;
    TB_CUDA(cudaGetDeviceCount(&count));
    if (cuda_device < 0 || cuda_device >= count) return fail("no such CUDA device");
    DeviceGuard g(cuda_device);
    cudaDeviceProp prop;
    TB_CUDA(cudaGetDeviceProperties(&prop, cuda_device));
    double *sink = nullptr;
    TB_CUDA(cudaMalloc(&sink, 8));
    cudaEvent_t a, b;
    TB_CUDA(cudaEventCreate(&a));
    TB_CUDA(cudaEventCreate(&b));
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    TB_CUDA(tbk::launch_fp64_peak(sink, blocks, 256, nullptr));   // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        TB_CUDA(cudaEventRecord(a));
        TB_CUDA(tbk::launch_fp64_peak(sink, blocks, iters, nullptr));
        TB_CUDA(cudaEventRecord(b));
        TB_CUDA(cudaEventSynchronize(b));
        float ms = 0;
        TB_CUDA(cudaEventElapsedTime(&ms, a, b));
        if (ms < best) best = ms;
    }
    const double flops = 2.0 * 64.0 * (double)iters * 256.0 * (double)blocks;  // 64 FMA per thread-iteration
    *tflops = flops / (best * 1e-3) / 1e12;
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(sink);
    return 0;
}

}  // extern "C"
