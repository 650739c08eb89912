// DEV SIMULATION of the device code for the CPU ("not gpu") test-suite.
//
// Compiles the very same headers the CUDA kernels are built from (zkvm_pairings_b200/csrc/*.cuh)
// as plain C++ (the PTX carry flag emulated), so the limb-level Montgomery arithmetic, its operand
// bounds (ZKP_SIM_ASSERT aborts on a violation), the tower and the pairing control flow can be
// checked against the oracle without a GPU.  The two lanes that share one pairing on the device are two host threads in
// lock-step here; the shfl.xor exchange is a two-party rendezvous.  TEST INFRASTRUCTURE ONLY: built
// into tests/host_sim/libzkpair_sim*.so, never linked into or loaded by libzkpair.so / the
// zkvm_pairings_b200 package, and not a CPU fallback (the product path raises when the CUDA
// library or a GPU is missing).
#define ZKP_HOST_SIM 1
#include <stddef.h>
#include <string.h>

#include <atomic>
#include <thread>

#include "../../zkvm_pairings_b200/csrc/ops.cuh"
#include "../device_harness/bodies.cuh"

namespace zkp {
thread_local int zkp_sim_par = 0;
thread_local unsigned long long zkp_sim_macs = 0;
static std::atomic<unsigned long long> g_macs{0};
static std::atomic<int> g_arrived{0};
static std::atomic<int> g_phase{0};
static unsigned char g_slot[2][512];
static void pair_barrier() {
    int ph = g_phase.load(std::memory_order_acquire);
    if (g_arrived.fetch_add(1, std::memory_order_acq_rel) == 1) {
        g_arrived.store(0, std::memory_order_relaxed);
        g_phase.store(ph + 1, std::memory_order_release);
    } else {
        int spins = 0;
        while (g_phase.load(std::memory_order_acquire) == ph)
            if (++spins > 2000) std::this_thread::yield();
    }
}
void zkp_sim_xchg(void *buf, unsigned long bytes) {
    memcpy(g_slot[zkp_sim_par], buf, bytes);
    pair_barrier();
    memcpy(buf, g_slot[zkp_sim_par ^ 1], bytes);
    pair_barrier();
}
uint32_t zkp_sim_word_xchg(uint32_t v) {
    zkp_sim_xchg(&v, sizeof v);
    return v;
}
}  // namespace zkp

using namespace zkp;

// run f() on both lanes of a pair (this thread = even lane, a helper thread = odd lane)
template <class F>
static void run_pair(F f) {
    std::thread odd([&]() {
        zkp_sim_par = 1;
        zkp_sim_macs = 0;
        f();
        g_macs += zkp_sim_macs;
    });
    zkp_sim_par = 0;
    zkp_sim_macs = 0;
    f();
    g_macs += zkp_sim_macs;
    odd.join();
}

extern "C" {
int sim_tower_op(int op, const uint64_t *a, const uint64_t *b, uint64_t *out, uint8_t *status, size_t n) {
    int na, nb, nr;
    tower_op_shape(op, na, nb, nr);
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            uint8_t s = tower_op_one(op, a + 6 * na * i, b ? b + 6 * nb * i : nullptr, out + 6 * nr * i);
            if (status && lane_par() == 0) status[i] = s;
        }
    });
    return 0;
}
int sim_pairing(int mode, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                size_t n, int k, const uint64_t *in12, uint64_t *out, uint8_t *is_one) {
    std::atomic<int> bad{0};
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            size_t e = i * (size_t)k;
            if (pairing_one<8>(mode, g1 ? g1 + 12 * e : nullptr, g1inf ? g1inf + e : nullptr, g2 ? g2 + 24 * e : nullptr,
                               g2inf ? g2inf + e : nullptr, k, in12 ? in12 + 72 * i : nullptr, out + 72 * i,
                               is_one ? is_one + i : nullptr))
                bad.store(1);
        }
    });
    return bad.load() ? -1 : 0;
}
// prepared G2 line tables (SURVEY 8f-4): same blob layout as the GPU kernel k_g2_prepare
void sim_g2_prepare(const uint64_t *g2, size_t n, uint64_t *out) {
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            bool bad = false;
            G2A q;
            load_g2(q, g2 + 24 * i, bad);
            g2_prepare(q, (Fp *)out + i * (ZKP_LINE_STEPS * 3 * 2) + lane_par());
        }
    });
}
// n checks of k pairs, the last kf of them from the tables `tab`; full pairing (mode 3)
int sim_pairing_prepared(const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf, size_t n, int k,
                         const uint64_t *tab, const uint8_t *tabinf, int kf, uint64_t *out, uint8_t *is_one) {
    std::atomic<int> anybad{0};
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            bool bad = false;
            Fp12 f;
            size_t e = i * (size_t)k, e2 = i * (size_t)(k - kf);
            pairing_front<8>(f, bad, 3, g1 + 12 * e, g1inf ? g1inf + e : nullptr, g2 ? g2 + 24 * e2 : nullptr,
                             g2inf ? g2inf + e2 : nullptr, k, nullptr, (const Fp *)tab, tabinf, kf);
            final_exponentiation(f, f);
            bool one = store_fp12(out + 72 * i, f);
            if (is_one && lane_par() == 0) is_one[i] = one ? 1 : 0;
            if (lane_or(bad)) anybad.store(1);
        }
    });
    return anybad.load() ? -1 : 0;
}
// group-level ops of ops.cuh (SURVEY 8f): gop 0/1 = G1/G2 validity, 2/3 = G1/G2 scalar multiplication
int sim_group_op(int gop, const uint64_t *pts, const uint8_t *inf, const uint64_t *scalars, uint64_t *out, uint8_t *flag, size_t n) {
    std::atomic<int> anybad{0};
    const int w = (gop & 1) ? 24 : 12;
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            bool bad = false;
            uint8_t is_inf = inf ? inf[i] : 0, f = 0;
            switch (gop) {
                case GOP_G1_CHECK: f = g1_check_one(pts + w * i, is_inf, bad); break;
                case GOP_G2_CHECK: f = g2_check_one(pts + w * i, is_inf, bad); break;
                case GOP_G1_MUL: g1_mul_one(pts + w * i, is_inf, scalars + 4 * i, out + w * i, flag + i, bad); break;
                default: g2_mul_one(pts + w * i, is_inf, scalars + 4 * i, out + w * i, flag + i, bad); break;
            }
            if (lane_or(bad)) anybad.store(1);
            if (gop <= GOP_G2_CHECK && lane_par() == 0) flag[i] = f;
        }
    });
    return anybad.load() ? -1 : 0;
}
// element-wise affine addition (gop 4 = G1, 5 = G2): out = a + b, flag bit0 identity, bit1 undefined in the reference
int sim_group_add(int gop, const uint64_t *a, const uint8_t *ainf, const uint64_t *b, const uint8_t *binf, uint64_t *out, uint8_t *flag, size_t n) {
    std::atomic<int> anybad{0};
    const int w = (gop & 1) ? 24 : 12;
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            bool bad = false;
            uint8_t ia = ainf ? ainf[i] : 0, ib = binf ? binf[i] : 0;
            if (gop == GOP_G1_ADD) g1_add_one(a + w * i, ia, b + w * i, ib, out + w * i, flag + i, bad);
            else g2_add_one(a + w * i, ia, b + w * i, ib, out + w * i, flag + i, bad);
            if (lane_or(bad)) anybad.store(1);
        }
    });
    return anybad.load() ? -1 : 0;
}
// Montgomery-trick batch inversion of pairing.cuh (one simulated thread, runs of `run` elements)
void sim_batch_inv(const uint64_t *in, uint64_t *out, size_t n, int run) {
    zkp_sim_par = 0;
    bool bad = false;
    for (size_t lo = 0; lo < n; lo += run) {
        int cnt = (int)(n - lo < (size_t)run ? n - lo : run);
        Fp v[64], pre[64];
        for (int i = 0; i < cnt; i++) v[i] = load_fp(in + 6 * (lo + i), bad);
        fp_batch_inv(v, pre, cnt);
        for (int i = 0; i < cnt; i++) store_fp(out + 6 * (lo + i), v[i], nullptr);
    }
}
// Bound check of the Fp6-level bodies (in particular of their lazy-reduction forms, -DZKP_LAZY): every Montgomery
// representative of an operand may lie anywhere in [0, 2p]; the recombined unreduced values are multilinear in them, so
// their extremes are reached at the vertices of that box.  Runs fp6_mul (what = 0, 2^12 vertices), fp6_mul_by_01 (1, 2^10)
// and fp4_square (2, 2^4) with every operand within 2^20 of 0 or of 2p and compares with the schoolbook formulas on
// reduced Fp2 products; the ZKP_SIM_ASSERTs inside abort on a bound violation.  Returns the number of mismatches.
static Fp vertex_fp(unsigned combo, int operand, int what) {
    int bit = 2 * operand + lane_par();
    uint32_t d = (uint32_t)(splitmix64_at(0xB0DD + what, (uint64_t)combo * 64 + bit) & 0xfffff);
    Fp r = ((combo >> bit) & 1) ? fp_const(ZKP_2P) : fp_zero();
    if ((combo >> bit) & 1) r.l[0] -= d;   // 2p - d (the low word of 2p is 0xffff5556: no borrow)
    else r.l[0] = d;
    return r;
}
static bool same_fp2(const Fp2 &x, const Fp2 &y) {
    uint32_t a[ZKP_NL], b[ZKP_NL];
    fp_to_words(a, x.c);
    fp_to_words(b, y.c);
    return lane_and(memcmp(a, b, sizeof a) == 0);
}
int sim_vertex_check(int what) {
    std::atomic<int> bad{0};
    const unsigned combos = what == 0 ? 1u << 12 : what == 1 ? 1u << 10 : 1u << 4;
    run_pair([&]() {
        for (unsigned c = 0; c < combos; c++) {
            Fp2 v[6];
            for (int k = 0; k < 6; k++) v[k].c = vertex_fp(c, k, what);
            if (what == 0) {
                Fp6 a = {v[0], v[1], v[2]}, b = {v[3], v[4], v[5]}, r;
                fp6_mul(r, a, b);
                Fp2 e0 = fp2_add(fp2_mul(a.c0, b.c0), fp2_mul_nr(fp2_add(fp2_mul(a.c1, b.c2), fp2_mul(a.c2, b.c1))));
                Fp2 e1 = fp2_add(fp2_add(fp2_mul(a.c0, b.c1), fp2_mul(a.c1, b.c0)), fp2_mul_nr(fp2_mul(a.c2, b.c2)));
                Fp2 e2 = fp2_add(fp2_add(fp2_mul(a.c0, b.c2), fp2_mul(a.c1, b.c1)), fp2_mul(a.c2, b.c0));
                if (!(same_fp2(r.c0, e0) & same_fp2(r.c1, e1) & same_fp2(r.c2, e2))) bad++;
            } else if (what == 1) {
                Fp6 a = {v[0], v[1], v[2]}, r;
                fp6_mul_by_01(r, a, v[3], v[4]);
                Fp2 e0 = fp2_add(fp2_mul(a.c0, v[3]), fp2_mul_nr(fp2_mul(a.c2, v[4])));
                Fp2 e1 = fp2_add(fp2_mul(a.c0, v[4]), fp2_mul(a.c1, v[3]));
                Fp2 e2 = fp2_add(fp2_mul(a.c1, v[4]), fp2_mul(a.c2, v[3]));
                if (!(same_fp2(r.c0, e0) & same_fp2(r.c1, e1) & same_fp2(r.c2, e2))) bad++;
            } else {
                Fp2 c0, c1;
                fp4_square(c0, c1, v[0], v[1]);
                Fp2 e0 = fp2_add(fp2_mul(v[0], v[0]), fp2_mul_nr(fp2_mul(v[1], v[1])));
                Fp2 e1 = fp2_dbl(fp2_mul(v[0], v[1]));
                if (!(same_fp2(c0, e0) & same_fp2(c1, e1))) bad++;
            }
        }
    });
    return bad.load();
}
// the bodies of tests/device_harness/bodies.cuh on raw representatives, n elements of BODY_U64 u64: the same
// computation as the device harness (harness_run), representative for representative
void sim_body(int body, const uint64_t *in, uint64_t *out, size_t n) {
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) body_one(body, in + i * BODY_U64, out + i * BODY_U64, true);
    });
}
// wide MACs executed by both lanes since the last call (boundary conversions included)
uint64_t sim_take_mac_count() { return g_macs.exchange(0); }
uint64_t sim_splitmix64_at(uint64_t seed, uint64_t idx) { return splitmix64_at(seed, idx); }
void sim_gen_points(const uint64_t *k1, const uint64_t *k2, size_t n, uint64_t *g1, uint8_t *g1inf, uint64_t *g2, uint8_t *g2inf) {
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            gen_g1_one(k1[i], g1 + 12 * i, g1inf + i);
            gen_g2_one(k2[i], g2 + 24 * i, g2inf + i);
        }
    });
}
}
