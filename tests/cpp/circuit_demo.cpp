// circuit_demo.cpp -- whole circuits through certFHE::Circuit, every lane in one call: a 16-bit ripple-carry adder over
// 1024 lanes (compacted gates) and a 5-bit multiplier mod 2^5 over 1024 lanes (compacted and cancelled gates, one lane
// in eight with all-ones inputs).  Checks the decrypted outputs against x + y and x * y in every lane, that a tiny lane
// capacity sends every lane down the gate-by-gate path with the same words, and that bad netlists throw.
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

static bool same_array(const CiphertextArray &a, const CiphertextArray &b) {
    if (a.getOffsets() != b.getOffsets()) return false;
    for (uint64_t k = 0; k < a.size(); ++k) {
        const Ciphertext x = a.get(k), y = b.get(k);
        const uint64_t *p = x.getValues(), *q = y.getValues();
        for (uint64_t i = 0; i < x.getLen(); ++i)
            if (p[i] != q[i]) return false;
    }
    return true;
}

// Encrypts bit i of x (rows 0 .. bits-1) and of y (rows bits .. 2 bits-1) of every lane; returns the 2 bits rows.
static std::vector<CiphertextArray> encrypt_rows(SecretKey &sk, const std::vector<uint64_t> &x,
                                                 const std::vector<uint64_t> &y, uint64_t bits, uint64_t seed) {
    const uint64_t lanes = x.size();
    std::vector<unsigned char> plain(2 * bits * lanes);
    for (uint64_t l = 0; l < lanes; ++l)
        for (uint64_t i = 0; i < bits; ++i) {
            plain[i * lanes + l] = (unsigned char)((x[l] >> i) & 1u);
            plain[(bits + i) * lanes + l] = (unsigned char)((y[l] >> i) & 1u);
        }
    CiphertextArray all = sk.encryptArray(plain.data(), plain.size(), seed);
    std::vector<CiphertextArray> rows;
    for (uint64_t r = 0; r < 2 * bits; ++r) {
        std::vector<uint64_t> idx(lanes);
        for (uint64_t l = 0; l < lanes; ++l) idx[l] = r * lanes + l;
        rows.push_back(all.gather(idx));
    }
    return rows;
}

static std::vector<uint64_t> decrypt_word(SecretKey &sk, const std::vector<CiphertextArray> &bits) {
    std::vector<uint64_t> v(bits[0].size(), 0);
    std::vector<unsigned char> b(v.size());
    for (size_t i = 0; i < bits.size(); ++i) {
        sk.decryptArray(bits[i], b.data());
        for (size_t l = 0; l < v.size(); ++l) v[l] |= (uint64_t)(b[l] & 1u) << i;
    }
    return v;
}

int main() {
    Library::initializeLibrary();
    srand(1618);
    const uint64_t lanes = 1024;
    Context ctx(1247, 16);
    SecretKey sk(ctx);

    // 16-bit adder: s_i = x_i + y_i + c, c' = x_i*y_i + (x_i + y_i)*c; outputs s_0 .. s_15 and the final carry
    {
        const uint32_t bits = 16;
        std::vector<uint64_t> x(lanes), y(lanes);
        for (uint64_t l = 0; l < lanes; ++l) {
            x[l] = (uint64_t)rand() & 0xffff;
            y[l] = (uint64_t)rand() & 0xffff;
        }
        std::vector<CiphertextArray> in = encrypt_rows(sk, x, y, bits, 271828);
        Circuit add(2 * bits);
        std::vector<uint32_t> outs;
        outs.push_back(add.gate({}, {0, bits}));
        uint32_t c = add.gate({{0, bits}});
        for (uint32_t i = 1; i < bits; ++i) {
            const uint32_t t = add.gate({}, {i, bits + i});
            outs.push_back(add.gate({}, {t, c}));
            c = add.gate({{i, bits + i}, {t, c}});
        }
        outs.push_back(c);
        std::vector<CiphertextArray> s = add.evaluate(in, outs);
        expect(s.size() == bits + 1, "adder: wrong number of outputs");
        std::vector<uint64_t> got = decrypt_word(sk, s);
        for (uint64_t l = 0; l < lanes; ++l)
            if (got[l] != x[l] + y[l]) {
                expect(false, "adder: lane " + to_string(l) + " decrypts to " + to_string(got[l]));
                break;
            }
        std::cout << "adder: " << add.lastFallback() << " fallback lanes" << std::endl;
        // every lane gate by gate: the same words and offsets
        std::vector<CiphertextArray> f = add.evaluate(in, outs, -1, false, 1);
        expect(add.lastFallback() == lanes, "adder: lane capacity 1 did not send every lane to the fallback");
        for (size_t j = 0; j < outs.size(); ++j)
            expect(same_array(s[j], f[j]), "adder: output " + to_string(j) + " differs on the gate-by-gate path");
    }

    // 5-bit multiplier mod 2^5: schoolbook rows added with ripple carries, every gate compacted and cancelled
    {
        const uint32_t bits = 5;
        std::vector<uint64_t> x(lanes), y(lanes);
        for (uint64_t l = 0; l < lanes; ++l) {
            x[l] = l % 8 == 0 ? 31 : (uint64_t)rand() & 31;
            y[l] = l % 8 == 0 ? 31 : (uint64_t)rand() & 31;
        }
        std::vector<CiphertextArray> in = encrypt_rows(sk, x, y, bits, 314159);
        Circuit mul(2 * bits);
        const int64_t none = -1;   // an all-zero bit: no wire
        std::vector<int64_t> acc(bits, none);
        for (uint32_t j = 0; j < bits; ++j) {
            std::vector<int64_t> pp(bits, none);
            for (uint32_t i = 0; i + j < bits; ++i) pp[i + j] = mul.gate({{i, bits + j}});
            int64_t c = none;
            std::vector<int64_t> next(bits, none);
            for (uint32_t k = 0; k < bits; ++k) {
                std::vector<uint32_t> ops;
                for (int64_t w : {acc[k], pp[k], c})
                    if (w != none) ops.push_back((uint32_t)w);
                next[k] = ops.empty() ? none : (int64_t)mul.gate({}, ops);
                std::vector<std::pair<uint32_t, uint32_t>> prods;
                for (size_t p = 0; p < ops.size(); ++p)
                    for (size_t q = p + 1; q < ops.size(); ++q) prods.push_back({ops[p], ops[q]});
                c = prods.empty() ? none : (int64_t)mul.gate(prods);
            }
            acc = next;
        }
        std::vector<uint32_t> outs;
        for (int64_t w : acc) outs.push_back((uint32_t)w);
        std::vector<CiphertextArray> p = mul.evaluate(in, outs, -1, true);
        std::vector<uint64_t> got = decrypt_word(sk, p);
        for (uint64_t l = 0; l < lanes; ++l)
            if (got[l] != (x[l] * y[l]) % 32) {
                expect(false, "multiplier: lane " + to_string(l) + " decrypts to " + to_string(got[l]));
                break;
            }
        std::cout << "multiplier: " << mul.wires() << " wires, " << mul.lastFallback() << " fallback lanes" << std::endl;
    }

    // bad netlists and arguments throw
    Circuit bad(2);
    bool threw = false;
    try {
        bad.gate({{0, 2}});
    } catch (const Error &) {
        threw = true;
    }
    expect(threw, "an operand that is not an earlier wire did not throw");
    threw = false;
    try {
        bad.gate({}, {});
    } catch (const Error &) {
        threw = true;
    }
    expect(threw, "a gate without operands did not throw");

    if (failures) {
        std::cout << "circuit_demo: " << failures << " failures" << std::endl;
        return 1;
    }
    std::cout << "circuit_demo: 16-bit adder and 5-bit multiplier over 1024 lanes as circuits: all checks passed"
              << std::endl;
    return 0;
}
