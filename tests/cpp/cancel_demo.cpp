// cancel_demo.cpp -- a 5-bit SIMD multiplier (product mod 32) over 1024 lanes whose every sum and carry is one
// compacting gate followed by CiphertextArray::cancel(): a circuit that reuses its inputs produces the same monomial
// along several paths, and cancellation keeps one block per monomial of odd coefficient.  Checks that every lane
// decrypts to x*y mod 32, that output bit i holds at most 1, 2, 4, 10, 26 blocks per lane (exactly that many in the
// lanes whose inputs all encrypt 1), that a scalar Ciphertext x*x cancels to x and x + x to nothing, and that the
// decryption of a cancelled chain stays right.
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

typedef std::vector<std::pair<CiphertextArray, CiphertextArray>> Products;

static CiphertextArray gate(const Products &products, const std::vector<CiphertextArray> &terms) {
    return CiphertextArray::compactSumOfProducts(products, terms).cancel();
}

int main() {
    Library::initializeLibrary();
    srand(31415);
    const uint64_t lanes = 1024, bits = 5;
    Context ctx(1247, 16);
    SecretKey sk(ctx);
    std::vector<uint64_t> x(lanes), y(lanes);
    std::vector<unsigned char> plain(2 * bits * lanes);
    for (uint64_t l = 0; l < lanes; ++l) {
        x[l] = l % 8 == 0 ? 31 : (uint64_t)rand() % 32;   // every eighth lane: all inputs encrypt 1
        y[l] = l % 8 == 0 ? 31 : (uint64_t)rand() % 32;
        for (uint64_t i = 0; i < bits; ++i) {
            plain[i * lanes + l] = (unsigned char)((x[l] >> i) & 1u);
            plain[(bits + i) * lanes + l] = (unsigned char)((y[l] >> i) & 1u);
        }
    }
    CiphertextArray all = sk.encryptArray(plain.data(), plain.size(), 27182);
    std::vector<CiphertextArray> X, Y;
    for (uint64_t r = 0; r < 2 * bits; ++r) {
        std::vector<uint64_t> idx(lanes);
        for (uint64_t l = 0; l < lanes; ++l) idx[l] = r * lanes + l;
        (r < bits ? X : Y).push_back(all.gather(idx));
    }

    // schoolbook rows, ripple-carry adds: s = a + b + c, c' = a*b + a*c + b*c over the operands that are not zero
    std::vector<std::vector<CiphertextArray>> acc(bits);   // an empty vector: the bit is zero (no blocks)
    for (uint64_t j = 0; j < bits; ++j) {
        std::vector<std::vector<CiphertextArray>> pp(bits);
        for (uint64_t i = 0; i + j < bits; ++i) pp[i + j].push_back(gate({{X[i], Y[j]}}, {}));
        std::vector<CiphertextArray> c;
        std::vector<std::vector<CiphertextArray>> out(bits);
        for (uint64_t k = 0; k < bits; ++k) {
            std::vector<CiphertextArray> ops;
            for (const auto *v : {&acc[k], &pp[k], &c})
                if (!v->empty()) ops.push_back(v->front());
            if (!ops.empty()) out[k].push_back(gate({}, ops));
            Products prods;
            for (size_t p = 0; p < ops.size(); ++p)
                for (size_t q = p + 1; q < ops.size(); ++q) prods.push_back({ops[p], ops[q]});
            c.clear();
            if (!prods.empty()) c.push_back(gate(prods, {}));
        }
        acc = out;
    }

    const uint64_t bound[5] = {1, 2, 4, 10, 26};   // monomials of odd coefficient of product bit i
    std::vector<uint64_t> got(lanes, 0);
    std::vector<unsigned char> dec(lanes);
    uint64_t most = 0;
    for (uint64_t i = 0; i < bits; ++i) {
        expect(!acc[i].empty(), "product bit " + to_string(i) + " is missing");
        if (acc[i].empty()) continue;
        const CiphertextArray &P = acc[i].front();
        sk.decryptArray(P, dec.data());
        for (uint64_t l = 0; l < lanes; ++l) {
            got[l] |= (uint64_t)dec[l] << i;
            const uint64_t held = P.getBlocks(l);
            most = std::max(most, held);
            expect(held <= bound[i], "bit " + to_string(i) + ", lane " + to_string(l) + ": " + to_string(held) + " blocks");
            if (l % 8 == 0)
                expect(held == bound[i], "bit " + to_string(i) + ", all-ones lane " + to_string(l) + ": " +
                                             to_string(held) + " blocks");
        }
    }
    uint64_t wrong = 0;
    for (uint64_t l = 0; l < lanes; ++l) wrong += got[l] != ((x[l] * y[l]) & 31u);
    expect(wrong == 0, "decrypted product differs in " + to_string(wrong) + " lanes");

    // scalar Ciphertext: x*x -> x, x + x -> nothing, cancel() of distinct blocks is the identity
    const unsigned char one = 1, zero = 0;
    Plaintext p1(one), p0(zero);
    Ciphertext cx = sk.encrypt(p1) + sk.encrypt(p0) + sk.encrypt(p1);
    expect(same_words((cx * cx).cancel(), cx), "x*x does not cancel to x");
    expect((cx + cx).cancel().getBlocks() == 0, "x + x does not cancel to nothing");
    expect(same_words(cx.cancel(), cx), "cancel() changed a ciphertext of distinct blocks");
    // a chain c = c * Enc(a) + c * Enc(b) + c * c, cancelled after every step (c * c cancels to c)
    unsigned char want = 1;
    Ciphertext chain = sk.encrypt(p1);
    for (int step = 0; step < 6; ++step) {
        const unsigned char a = (unsigned char)(rand() & 1), b = (unsigned char)(rand() & 1);
        Plaintext pa(a), pb(b);
        Ciphertext ca = sk.encrypt(pa), cb = sk.encrypt(pb);
        Ciphertext next = chain * ca + chain * cb + chain * chain;
        Ciphertext small = next.cancel();
        want = (unsigned char)((want & a) ^ (want & b) ^ want);
        expect(small.getBlocks() <= next.getBlocks(), "cancel() grew a ciphertext");
        expect(sk.decrypt(small).getValue() == want, "scalar chain: step " + to_string(step) + " decrypts wrong");
        chain = small;
    }

    if (failures) {
        std::cout << "cancel_demo: " << failures << " checks failed" << std::endl;
        return 1;
    }
    std::cout << "cancel_demo: 5-bit multiplier over " << lanes
              << " lanes with cancelled gates: all checks passed (at most " << most << " blocks per lane in a product bit)"
              << std::endl;
    return 0;
}
