// array_demo.cpp -- an 8-bit SIMD ripple-carry adder over many lanes, evaluated twice: on CiphertextArrays (one call,
// and one kernel launch for the small elements, per gate layer) and with plain Ciphertext operators lane by lane.
// Checks that the decrypted sums and carries are (x + y) mod 256 and the carry of every lane, and that sampled lanes
// hold the same words both ways.
#include "certFHE.h"

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
    srand(12345);
    const uint64_t lanes = 1024, bits = 8;
    Context ctx(1247, 16);
    SecretKey sk(ctx);
    std::vector<unsigned> x(lanes), y(lanes);
    // element i*lanes + l: bit i of x in lane l; then the bits of y the same way
    std::vector<unsigned char> plain(2 * bits * lanes);
    for (uint64_t l = 0; l < lanes; ++l) {
        x[l] = (unsigned)rand() & 255u;
        y[l] = (unsigned)rand() & 255u;
        for (uint64_t i = 0; i < bits; ++i) {
            plain[i * lanes + l] = (unsigned char)((x[l] >> i) & 1u);
            plain[(bits + i) * lanes + l] = (unsigned char)((y[l] >> i) & 1u);
        }
    }
    CiphertextArray all = sk.encryptArray(plain.data(), plain.size(), 777);
    auto bit_row = [&](uint64_t row) {
        std::vector<uint64_t> idx(lanes);
        for (uint64_t l = 0; l < lanes; ++l) idx[l] = row * lanes + l;
        return all.gather(idx);
    };

    // arrays: s_i = x_i + y_i + c, c' = x_i*y_i + (x_i + y_i)*c
    std::vector<CiphertextArray> S;
    CiphertextArray X0 = bit_row(0), Y0 = bit_row(bits);
    S.push_back(X0 + Y0);
    CiphertextArray C = X0 * Y0;
    for (uint64_t i = 1; i < bits; ++i) {
        CiphertextArray X = bit_row(i), Y = bit_row(bits + i);
        CiphertextArray T = X + Y;
        S.push_back(T + C);
        C = X * Y + T * C;
    }
    std::vector<unsigned char> dec(lanes);
    std::vector<unsigned> got(lanes, 0);
    for (uint64_t i = 0; i < bits; ++i) {
        sk.decryptArray(S[i], dec.data());
        for (uint64_t l = 0; l < lanes; ++l) got[l] |= (unsigned)dec[l] << i;
    }
    sk.decryptArray(C, dec.data());
    uint64_t wrong = 0;
    for (uint64_t l = 0; l < lanes; ++l) {
        const unsigned want = x[l] + y[l];
        if (got[l] != (want & 255u) || dec[l] != (want >> 8)) ++wrong;
    }
    expect(wrong == 0, "decrypted sum or carry differs in " + to_string(wrong) + " lanes");

    // the same circuit with plain Ciphertext operators on 16 lanes
    for (uint64_t q = 0; q < 16; ++q) {
        const uint64_t l = (q * 977) % lanes;
        Ciphertext xs = all.get(l), ys = all.get(bits * lanes + l);
        Ciphertext s = xs + ys, c = xs * ys;
        expect(same_words(s, S[0].get(l)), "lane " + to_string(l) + " bit 0: words differ");
        for (uint64_t i = 1; i < bits; ++i) {
            Ciphertext xi = all.get(i * lanes + l), yi = all.get((bits + i) * lanes + l);
            Ciphertext t = xi + yi;
            s = t + c;
            c = xi * yi + t * c;
            expect(same_words(s, S[i].get(l)), "lane " + to_string(l) + " bit " + to_string(i) + ": words differ");
            expect(sk.decrypt(s).getValue() == ((x[l] + y[l]) >> i & 1u), "lane " + to_string(l) + " plain decrypt");
        }
        expect(same_words(c, C.get(l)), "lane " + to_string(l) + " carry: words differ");
    }
    if (failures) {
        std::cout << "array_demo: " << failures << " checks failed" << std::endl;
        return 1;
    }
    std::cout << "array_demo: 8-bit adder over " << lanes << " lanes on CiphertextArray: all checks passed (carry "
              << C.getBlocks(0) << " blocks per lane)" << std::endl;
    return 0;
}
