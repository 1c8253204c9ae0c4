// compact_demo.cpp -- a 32-bit SIMD ripple-carry adder over 1024 lanes whose every carry is one compacting gate:
// C = CiphertextArray::compactSumOfProducts({{X, Y}, {T, C}}) keeps only the blocks with at least D set bits, so the
// carry stays a few dozen blocks per lane where the uncompacted carry of bit i holds 2^(i+1) - 1.  Checks that the
// decrypted sums and the final carry are those of x + y in every lane, that the carry stays small, that compact() of an
// uncompacted carry equals the compacting gate, that a scalar Ciphertext chain compacted with Ciphertext::compact()
// decrypts right after every step, and that the error cases throw.
#include "certFHE.h"

#include <algorithm>
#include <cstdlib>
#include <iostream>
#include <vector>

using namespace certFHE;

static int failures = 0;

static void expect(bool ok, const std::string &what) {
    if (!ok) {
        ++failures;
        std::cout << "FAILED: " << what << std::endl;
    }
}

static bool same_words(const Ciphertext &a, const Ciphertext &b) {
    if (a.getLen() != b.getLen()) return false;
    const uint64_t *x = a.getValues(), *y = b.getValues();
    for (uint64_t i = 0; i < a.getLen(); ++i)
        if (x[i] != y[i]) return false;
    return true;
}

int main() {
    Library::initializeLibrary();
    srand(2718);
    const uint64_t lanes = 1024, bits = 32;
    Context ctx(1247, 16);
    SecretKey sk(ctx);
    std::vector<uint64_t> x(lanes), y(lanes);
    // element i*lanes + l: bit i of x in lane l; then the bits of y the same way
    std::vector<unsigned char> plain(2 * bits * lanes);
    for (uint64_t l = 0; l < lanes; ++l) {
        x[l] = ((uint64_t)rand() << 16 ^ (uint64_t)rand()) & 0xffffffffull;
        y[l] = ((uint64_t)rand() << 16 ^ (uint64_t)rand()) & 0xffffffffull;
        for (uint64_t i = 0; i < bits; ++i) {
            plain[i * lanes + l] = (unsigned char)((x[l] >> i) & 1u);
            plain[(bits + i) * lanes + l] = (unsigned char)((y[l] >> i) & 1u);
        }
    }
    CiphertextArray all = sk.encryptArray(plain.data(), plain.size(), 161803);
    auto bit_row = [&](uint64_t row) {
        std::vector<uint64_t> idx(lanes);
        for (uint64_t l = 0; l < lanes; ++l) idx[l] = row * lanes + l;
        return all.gather(idx);
    };

    // s_i = x_i + y_i + c; the carry c' = x_i*y_i + (x_i + y_i)*c, compacted in the same call
    std::vector<CiphertextArray> S;
    CiphertextArray X0 = bit_row(0), Y0 = bit_row(bits);
    S.push_back(X0 + Y0);
    CiphertextArray C = CiphertextArray::compactSumOfProducts({{X0, Y0}});
    uint64_t most = C.getOffsets().back();
    for (uint64_t i = 1; i < bits; ++i) {
        CiphertextArray X = bit_row(i), Y = bit_row(bits + i);
        CiphertextArray T = X + Y;
        S.push_back(T + C);
        if (i == 8) {   // compact() of the uncompacted gate is the compacting gate, word for word
            CiphertextArray U = CiphertextArray::sumOfProducts({{X, Y}, {T, C}});
            CiphertextArray V = CiphertextArray::compactSumOfProducts({{X, Y}, {T, C}});
            CiphertextArray W = U.compact();
            expect(W.getOffsets() == V.getOffsets(), "compact() and compactSumOfProducts offsets differ");
            for (uint64_t q = 0; q < 16; ++q) {
                const uint64_t l = (q * 613 + 5) % lanes;
                expect(same_words(W.get(l), V.get(l)), "lane " + to_string(l) + ": compacted words differ");
            }
            expect(V.getOffsets().back() < U.getOffsets().back(), "the filter dropped nothing");
        }
        C = CiphertextArray::compactSumOfProducts({{X, Y}, {T, C}});
        most = std::max<uint64_t>(most, C.getOffsets().back());
    }
    expect(most < 512 * lanes, "a carry holds " + to_string(most) + " blocks over " + to_string(lanes) + " lanes");
    std::vector<unsigned char> dec(lanes);
    std::vector<uint64_t> got(lanes, 0);
    for (uint64_t i = 0; i < bits; ++i) {
        sk.decryptArray(S[i], dec.data());
        for (uint64_t l = 0; l < lanes; ++l) got[l] |= (uint64_t)dec[l] << i;
    }
    sk.decryptArray(C, dec.data());
    uint64_t wrong = 0;
    for (uint64_t l = 0; l < lanes; ++l) {
        const uint64_t want = x[l] + y[l];
        if (got[l] != (want & 0xffffffffull) || dec[l] != (want >> 32)) ++wrong;
    }
    expect(wrong == 0, "decrypted sum or carry differs in " + to_string(wrong) + " lanes");

    // a scalar chain acc = acc * Enc(a) + Enc(b), compacted after every step
    unsigned char want = (unsigned char)(rand() & 1);
    Plaintext p0(want);
    Ciphertext acc = sk.encrypt(p0);
    for (int step = 0; step < 12; ++step) {
        const unsigned char a = (unsigned char)(rand() & 1), b = (unsigned char)(rand() & 1);
        Plaintext pa(a), pb(b);
        Ciphertext ca = sk.encrypt(pa), cb = sk.encrypt(pb);
        Ciphertext next = acc * ca + cb;
        Ciphertext small = next.compact();
        want = (unsigned char)((want & a) ^ b);
        expect(small.getBlocks() <= next.getBlocks(), "compact() grew a ciphertext");
        expect(sk.decrypt(small).getValue() == want, "scalar chain: step " + to_string(step) + " decrypts wrong");
        expect(sk.decrypt(next).getValue() == want, "scalar chain: step " + to_string(step) + " (uncompacted) wrong");
        acc = small;
    }

    // argument errors throw certFHE::Error
    int thrown = 0;
    try {
        CiphertextArray::compactSumOfProducts({});
    } catch (const Error &) {
        ++thrown;
    }
    try {
        CiphertextArray::compactSumOfProducts({{X0, Y0}}, {all});
    } catch (const Error &) {
        ++thrown;
    }
    try {
        Context ctx2(64, 4);
        SecretKey sk2(ctx2);
        CiphertextArray Z = sk2.encryptArray(plain.data(), lanes, 5);
        CiphertextArray::compactSumOfProducts({{X0, Y0}}, {Z});
    } catch (const Error &) {
        ++thrown;
    }
    expect(thrown == 3, "argument errors: " + to_string(thrown) + " of 3 threw");

    if (failures) {
        std::cout << "compact_demo: " << failures << " checks failed" << std::endl;
        return 1;
    }
    std::cout << "compact_demo: 32-bit adder over " << lanes
              << " lanes with compactSumOfProducts carries: all checks passed (at most " << most << " carry blocks, "
              << C.getOffsets().back() << " in the last carry)" << std::endl;
    return 0;
}
