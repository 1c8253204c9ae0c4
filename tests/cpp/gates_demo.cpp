// gates_demo.cpp -- the 8-bit SIMD ripple-carry adder of array_demo.cpp with every carry one gate call:
// C = CiphertextArray::sumOfProducts({{X, Y}, {T, C}}) (one call, every word of the new carry written once) instead of
// X * Y + T * C (three calls).  Checks that the decrypted sums and carries are (x + y) mod 256 and the carry of every
// lane, that every carry holds the same words both ways on sampled lanes, and that the error cases throw.
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
    srand(4242);
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
    CiphertextArray all = sk.encryptArray(plain.data(), plain.size(), 31337);
    auto bit_row = [&](uint64_t row) {
        std::vector<uint64_t> idx(lanes);
        for (uint64_t l = 0; l < lanes; ++l) idx[l] = row * lanes + l;
        return all.gather(idx);
    };

    // s_i = x_i + y_i + c; the carry c' = x_i*y_i + (x_i + y_i)*c as one gate, and as three operator calls
    std::vector<CiphertextArray> S;
    CiphertextArray X0 = bit_row(0), Y0 = bit_row(bits);
    S.push_back(X0 + Y0);
    CiphertextArray C = CiphertextArray::sumOfProducts({{X0, Y0}});
    CiphertextArray Cops = X0 * Y0;
    std::vector<CiphertextArray> carries(1, C), carries_ops(1, Cops);
    for (uint64_t i = 1; i < bits; ++i) {
        CiphertextArray X = bit_row(i), Y = bit_row(bits + i);
        CiphertextArray T = X + Y;
        S.push_back(T + C);
        C = CiphertextArray::sumOfProducts({{X, Y}, {T, C}});
        Cops = X * Y + T * Cops;
        carries.push_back(C);
        carries_ops.push_back(Cops);
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

    // the carries of the gate form and of the operator form, word for word on 16 lanes
    for (uint64_t i = 0; i < bits; ++i) {
        expect(carries[i].getOffsets() == carries_ops[i].getOffsets(), "bit " + to_string(i) + ": carry offsets differ");
        for (uint64_t q = 0; q < 16; ++q) {
            const uint64_t l = (q * 977 + i) % lanes;
            expect(same_words(carries[i].get(l), carries_ops[i].get(l)),
                   "lane " + to_string(l) + " bit " + to_string(i) + ": carry words differ");
        }
    }

    // argument errors throw certFHE::Error
    int thrown = 0;
    try {
        CiphertextArray::sumOfProducts({});
    } catch (const Error &) {
        ++thrown;
    }
    try {
        CiphertextArray::sumOfProducts({{X0, Y0}}, {all});
    } catch (const Error &) {
        ++thrown;
    }
    try {
        Context ctx2(64, 4);
        SecretKey sk2(ctx2);
        CiphertextArray Z = sk2.encryptArray(plain.data(), lanes, 5);
        CiphertextArray::sumOfProducts({{X0, Y0}}, {Z});
    } catch (const Error &) {
        ++thrown;
    }
    expect(thrown == 3, "argument errors: " + to_string(thrown) + " of 3 threw");

    if (failures) {
        std::cout << "gates_demo: " << failures << " checks failed" << std::endl;
        return 1;
    }
    std::cout << "gates_demo: 8-bit adder over " << lanes
              << " lanes with one sumOfProducts call per carry: all checks passed (carry " << C.getBlocks(0)
              << " blocks per lane)" << std::endl;
    return 0;
}
