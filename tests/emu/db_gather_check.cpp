// test-only: the gather of a resident database's subjects by caller id (csrc/kern_util.cuh) on the CPU, with the
// kernel sources compiled under -DPSB_EMULATE.  Random subjects are packed by pack_db_kernel at 2, 3 and 5 bit in a
// random storage order, invert_perm_kernel inverts that order, and unpack_db_kernel gathers caller-order ids through
// it: the output must be mapper[raw] byte for byte.
// usage: db_gather_check seed bits n_subjects
#define PSB_EMULATE 1
#include "../../parasail_rs_b200/csrc/kern_util.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <random>
#include <vector>

using namespace psb;

int main(int argc, char **argv) {
    if (argc < 4) return 2;
    const unsigned seed = (unsigned)std::atoi(argv[1]);
    const int bits = std::atoi(argv[2]);
    const long long n = std::atoll(argv[3]);
    const int rpw = residues_per_word(bits);
    const int size = bits == 2 ? 4 : (bits == 3 ? 8 : 32);   // the largest alphabet each width holds
    std::mt19937_64 rng(seed);

    // raw residues: letters 'A'.. of the alphabet in both cases plus unknown bytes; the mapper sends every byte to a
    // code below `size`, as a matrix's mapper does
    uint8_t mapper[256];
    for (int b = 0; b < 256; ++b) mapper[b] = (uint8_t)(size - 1);
    for (int c = 0; c < size - 1; ++c) mapper['A' + c] = mapper['a' + c] = (uint8_t)c;
    unsigned lut[64];
    for (int i = 0; i < 64; ++i)
        lut[i] = (unsigned)mapper[4 * i] | ((unsigned)mapper[4 * i + 1] << 8) | ((unsigned)mapper[4 * i + 2] << 16) | ((unsigned)mapper[4 * i + 3] << 24);

    // lengths: one-residue subjects, exact multiples of residues-per-word, one off either side, and random ones
    std::vector<long long> len(n);
    for (long long i = 0; i < n; ++i) {
        const int kind = (int)(i % 5);
        if (kind == 0) len[i] = 1;
        else if (kind == 1) len[i] = rpw * (1 + (long long)(rng() % 8));
        else if (kind == 2) len[i] = rpw * (1 + (long long)(rng() % 8)) + 1;
        else if (kind == 3) len[i] = rpw * (1 + (long long)(rng() % 8)) - 1;
        else len[i] = 1 + (long long)(rng() % 700);
    }
    std::vector<long long> raw_off(n + 1, 0);
    for (long long i = 0; i < n; ++i) raw_off[i + 1] = raw_off[i] + len[i];
    std::vector<uint8_t> raw(raw_off[n]);
    for (auto &x : raw) {
        const unsigned r = (unsigned)(rng() % 64);
        x = r < 60 ? (uint8_t)((r & 1 ? 'a' : 'A') + (r >> 1) % (size - 1)) : (uint8_t)("?*#\x7f"[r - 60]);
    }

    // storage order: a random permutation (sorted position -> caller id), word offsets in that order
    std::vector<int> perm(n);
    std::iota(perm.begin(), perm.end(), 0);
    std::shuffle(perm.begin(), perm.end(), rng);
    std::vector<long long> word_off(n + 1, 0);
    for (long long s = 0; s < n; ++s) word_off[s + 1] = word_off[s] + (len[perm[s]] + rpw - 1) / rpw;
    std::vector<unsigned> words(word_off[n] + 16, 0xdeadbeefu);

    PackParams pp;
    pp.raw = raw.data(); pp.raw_off = raw_off.data(); pp.raw_base = 0; pp.perm = perm.data();
    pp.word_off = word_off.data(); pp.words = words.data(); pp.n = n; pp.bits = bits;
    std::memcpy(pp.lut, lut, sizeof(lut));
    emu::launch(3, 256, [&]() { pack_db_kernel(pp); });

    std::vector<int> inv(n, -1);
    emu::launch(2, 0, [&]() { invert_perm_kernel(perm.data(), n, inv.data()); });
    for (long long s = 0; s < n; ++s)
        if (inv[perm[s]] != s) { std::printf("inverse permutation wrong at %lld\n", s); return 1; }

    // caller ids: first, last, repeats, then random
    std::vector<int> ids = {0, (int)(n - 1), 0, (int)(n - 1), (int)(n / 2), (int)(n / 2)};
    for (int t = 0; t < 300; ++t) ids.push_back((int)(rng() % n));
    const long long m = (long long)ids.size();
    std::vector<long long> out_off(m + 1, 0);
    for (long long i = 0; i < m; ++i) out_off[i + 1] = out_off[i] + len[ids[i]];
    // outputs written through a pointer biased by a base offset, as a pass of psb_db_align does
    const long long base = 12345;
    for (auto &o : out_off) o += base;
    std::vector<uint8_t> out(out_off[m] - base, 0xee);
    UnpackParams u;
    u.words = words.data(); u.word_off = word_off.data(); u.ids = ids.data(); u.inv_perm = inv.data();
    u.out_off = out_off.data(); u.out = out.data() - base; u.n = m; u.bits = bits;
    emu::launch(4, 0, [&]() { unpack_db_kernel(u); });
    for (long long i = 0; i < m; ++i) {
        const long long id = ids[i];
        for (long long c = 0; c < len[id]; ++c) {
            const uint8_t want = mapper[raw[raw_off[id] + c]], got = out[out_off[i] - base + c];
            if (got != want) {
                std::printf("mismatch: row %lld (id %lld, length %lld) residue %lld: got %d, expected %d\n", i, id, len[id], c, got, want);
                return 1;
            }
        }
    }

    // NULL inv_perm keeps the old meaning: ids are sorted positions
    std::vector<int> spos = {0, (int)(n - 1), (int)(n / 3)};
    std::vector<long long> soff(4, 0);
    for (int i = 0; i < 3; ++i) soff[i + 1] = soff[i] + len[perm[spos[i]]];
    std::vector<uint8_t> sout(soff[3], 0xee);
    UnpackParams v = u;
    v.ids = spos.data(); v.inv_perm = nullptr; v.out_off = soff.data(); v.out = sout.data(); v.n = 3;
    emu::launch(1, 0, [&]() { unpack_db_kernel(v); });
    for (int i = 0; i < 3; ++i) {
        const long long id = perm[spos[i]];
        for (long long c = 0; c < len[id]; ++c)
            if (sout[soff[i] + c] != mapper[raw[raw_off[id] + c]]) { std::printf("sorted-position gather wrong at row %d\n", i); return 1; }
    }
    std::printf("ok bits %d: %lld subjects, %lld gathered, %lld residues\n", bits, n, m, out_off[m] - base);
    return 0;
}
