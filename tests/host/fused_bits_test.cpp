// CPU check of the bit helpers the fused multi-k sketch loop and its start-bitmap pass are built from
// (sourmash_rust_b200/csrc/kmer_bits.cuh):
//   * dilate_words<KA, KB, KC> (one doubling chain for every k-size) against dilate_word, which
//     tests/host/tile_views_test.cpp checks against the bit-by-bit definition;
//   * FusedGeom<KA, KB, KC>::split (every k-size's end-aligned 2-bit words from one forward and one
//     reverse-complement extraction) against extract2_end<K> at the same window, with the addressing the
//     kernel uses (sketch.cu: kmer_loop, kmer_loop_fused).
// Built and run by tests/test_host_fused_bits.py (no GPU needed).
#include <cstdio>
#include <vector>

#include "../../sourmash_rust_b200/csrc/kmer_bits.cuh"

using namespace smb200;

static uint64_t rng_state = 0x5EED5EEDull;
static uint32_t rnd32() {
    uint64_t z = (rng_state += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return (uint32_t)(z ^ (z >> 31));
}

template <int KA, int KB, int KC>
static int dilate_all(int trials) {
    int fails = 0;
    const int Ks[3] = {KA, KB, KC};
    for (int t = 0; t < trials; t++) {
        uint32_t in[3];
        for (int j = 0; j < 3; j++) {
            in[j] = rnd32();
            if (t % 3) in[j] &= rnd32();   // sparse bits, as in a mostly valid tile
            if (t % 5 == 0) in[j] &= rnd32() & rnd32();
            if (t % 7 == 1) in[j] = 0;
        }
        for (uint32_t d = 0; d <= 1; d++) {
            uint32_t out[3];
            dilate_words<KA, KB, KC>(in[0], in[1], in[2], d, out);
            for (int j = 0; j < 3; j++) {
                if (!Ks[j]) continue;
                const uint32_t want = dilate_word(in[0], in[1], in[2], Ks[j] - (int)d);
                if (out[j] != want) {
                    if (fails++ < 5) printf("dilate_words<%d,%d,%d> k=%d d=%u: %08x vs %08x\n", KA, KB, KC, Ks[j], d, out[j], want);
                }
            }
        }
    }
    return fails;
}

// one k-size of the fused launch at every window start i of a tile of B bases: split<K> of the shared words against
// extract2_end<K> addressed as kmer_loop addresses it
template <int KA, int KB, int KC, int K>
static int split_one(const uint32_t *f2, const uint32_t *r2, int B, int tile) {
    using FG = FusedGeom<KA, KB, KC>;
    constexpr int NE = KmerGeom<K>::NE;
    int fails = 0;
    for (int i = 0; i < tile; i++) {
        uint32_t F[FG::NF], R[FG::NR];
        const int ef0 = i + FG::KM - 16 * FG::NF, er0 = B - i - 16 * FG::NR;
        funnel_words<FG::NF>(f2 + (ef0 >> 4), (uint32_t)ef0 * 2u, F);
        funnel_words<FG::NR>(r2 + (er0 >> 4), (uint32_t)er0 * 2u, R);
        uint32_t ef[NE], er[NE], wf[NE], wr[NE];
        FG::template split<K>(F, R, ef, er);
        const int kf = i + K - 16 * NE, kr = (B - K - i) + K - 16 * NE;
        extract2_end<K>(f2 + (kf >> 4), (uint32_t)kf * 2u, wf);
        extract2_end<K>(r2 + (kr >> 4), (uint32_t)kr * 2u, wr);
        for (int j = 0; j < NE; j++) {
            if (ef[j] != wf[j] || er[j] != wr[j]) {
                if (fails++ < 5) printf("split<%d> of <%d,%d,%d> at window %d word %d\n", K, KA, KB, KC, i, j);
            }
        }
    }
    return fails;
}

template <int KA, int KB, int KC>
static int split_all(int tile) {
    using FG = FusedGeom<KA, KB, KC>;
    const int B = tile + ((FG::KM - 1 + 15) / 16) * 16;
    constexpr int PAD = 4;  // words in front of each stream, as SK_PAD2 (extraction reaches up to 64 bases back)
    static_assert(16 * FG::NF - FG::KM <= 16 * PAD, "pad");
    std::vector<uint32_t> f2(PAD + B / 16 + 2), r2(PAD + B / 16 + 2);
    for (auto &x : f2) x = rnd32();
    for (auto &x : r2) x = rnd32();
    int fails = split_one<KA, KB, KC, KA>(f2.data() + PAD, r2.data() + PAD, B, tile);
    if constexpr (KB != 0) fails += split_one<KA, KB, KC, KB>(f2.data() + PAD, r2.data() + PAD, B, tile);
    if constexpr (KC != 0) fails += split_one<KA, KB, KC, KC>(f2.data() + PAD, r2.data() + PAD, B, tile);
    return fails;
}

int main() {
    int fails = 0;
    // the fast-path forms, and k-sizes at the ends of what the helpers accept
    fails += dilate_all<21, 31, 51>(2000);
    fails += dilate_all<21, 31, 0>(500);
    fails += dilate_all<21, 51, 0>(500);
    fails += dilate_all<31, 51, 0>(500);
    fails += dilate_all<21, 0, 0>(500);
    fails += dilate_all<31, 0, 0>(500);
    fails += dilate_all<51, 0, 0>(500);
    fails += dilate_all<3, 33, 63>(2000);
    fails += dilate_all<5, 17, 0>(500);
    fails += split_all<21, 31, 51>(4096);
    fails += split_all<21, 31, 0>(4096);
    fails += split_all<21, 51, 0>(4096);
    fails += split_all<31, 51, 0>(4096);
    fails += split_all<3, 17, 63>(1024);
    fails += split_all<15, 33, 0>(1024);
    printf(fails ? "FAILED %d\n" : "OK\n", fails);
    return fails ? 1 : 0;
}
