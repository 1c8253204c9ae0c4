// uint_demo.cpp -- encrypted integers through the C++ drop-in: SecretKey::encryptUInt of random 8-bit values over 4096
// lanes, every UIntCircuit operation evaluated in one call (and the 5-bit composite min(a + b, c) - a with lt(a + b, c)),
// the eager EncryptedUInt operators, SecretKey::decryptUInt, each checked against the same arithmetic on the host, and
// the error cases that throw certFHE::Error.
#include "certFHE.h"

#include <algorithm>
#include <cstdlib>
#include <iostream>
#include <vector>

using namespace certFHE;
typedef UIntCircuit::UInt UInt;

static int failures = 0;

static void expect(bool ok, const std::string &what) {
    if (!ok) {
        ++failures;
        std::cout << "FAILED: " << what << std::endl;
    }
}

template <typename F>
static void expect_throw(F f, const std::string &what) {
    try {
        f();
        expect(false, what + " did not throw");
    } catch (const Error &) {
    }
}

int main() {
    Library::initializeLibrary();
    srand(4242);
    const uint64_t n = 4096;
    const uint32_t W = 8;
    const uint64_t m = (1u << W) - 1;
    Context ctx(1247, 16);
    SecretKey sk(ctx);
    std::vector<uint64_t> a(n), b(n), c(n), ones(n, 1), got(n);
    for (uint64_t k = 0; k < n; ++k) {
        a[k] = (uint64_t)rand() & m;
        b[k] = k < 64 ? a[k] : (uint64_t)rand() & m;
        c[k] = (uint64_t)rand() & m;
    }
    EncryptedUInt A = sk.encryptUInt(a.data(), n, W, 11), B = sk.encryptUInt(b.data(), n, W, 12);
    std::vector<unsigned char> onebits(n, 1);
    CiphertextArray one = sk.encryptArray(onebits.data(), n, 14);

    sk.decryptUInt(A, got.data());
    expect(got == a, "decryptUInt(encryptUInt(a))");

    // every operation of the table, one evaluate() call each
    struct Op {
        const char *name;
        UInt (UIntCircuit::*f)(const UInt &, const UInt &);
        uint64_t (*ref)(uint64_t, uint64_t);
        bool one;
    };
    const Op ops[] = {
        {"add", &UIntCircuit::add, [](uint64_t x, uint64_t y) -> uint64_t { return (x + y) & 255; }, false},
        {"sub", &UIntCircuit::sub, [](uint64_t x, uint64_t y) -> uint64_t { return (x - y) & 255; }, false},
        {"mul", &UIntCircuit::mul, [](uint64_t x, uint64_t y) -> uint64_t { return (x * y) & 255; }, false},
        {"lt", &UIntCircuit::lt, [](uint64_t x, uint64_t y) -> uint64_t { return x < y; }, false},
        {"gt", &UIntCircuit::gt, [](uint64_t x, uint64_t y) -> uint64_t { return x > y; }, false},
        {"ne", &UIntCircuit::ne, [](uint64_t x, uint64_t y) -> uint64_t { return x != y; }, false},
        {"eq", &UIntCircuit::eq, [](uint64_t x, uint64_t y) -> uint64_t { return x == y; }, true},
        {"le", &UIntCircuit::le, [](uint64_t x, uint64_t y) -> uint64_t { return x <= y; }, true},
        {"ge", &UIntCircuit::ge, [](uint64_t x, uint64_t y) -> uint64_t { return x >= y; }, true},
        {"min", &UIntCircuit::min, [](uint64_t x, uint64_t y) -> uint64_t { return std::min(x, y); }, false},
        {"max", &UIntCircuit::max, [](uint64_t x, uint64_t y) -> uint64_t { return std::max(x, y); }, false},
        {"and", &UIntCircuit::and_, [](uint64_t x, uint64_t y) -> uint64_t { return x & y; }, false},
        {"xor", &UIntCircuit::xor_, [](uint64_t x, uint64_t y) -> uint64_t { return x ^ y; }, false},
        {"or", &UIntCircuit::or_, [](uint64_t x, uint64_t y) -> uint64_t { return x | y; }, false},
    };
    for (const Op &op : ops) {
        UIntCircuit u(W, 2, op.one);
        const UInt r = (u.*op.f)(u.inputs()[0], u.inputs()[1]);
        EncryptedUInt x = u.evaluate({A, B}, {r}, -1, true, 0, op.one ? &one : nullptr)[0];
        sk.decryptUInt(x, got.data());
        bool ok = true;
        for (uint64_t k = 0; k < n; ++k) ok = ok && got[k] == op.ref(a[k], b[k]);
        expect(ok, std::string("UIntCircuit::") + op.name);
    }

    // min(a + b, c) - a and lt(a + b, c) in one call, on 5-bit values: a composition of comparisons holds the monomials
    // of its algebraic normal form, which grow about threefold per bit and per operand
    {
        const uint32_t W5 = 5;
        const uint64_t m5 = (1u << W5) - 1;
        std::vector<uint64_t> a5(n), b5(n), c5(n), lt(n);
        for (uint64_t k = 0; k < n; ++k) {
            a5[k] = a[k] & m5;
            b5[k] = b[k] & m5;
            c5[k] = c[k] & m5;
        }
        EncryptedUInt A5 = sk.encryptUInt(a5.data(), n, W5, 21), B5 = sk.encryptUInt(b5.data(), n, W5, 22),
                      C5 = sk.encryptUInt(c5.data(), n, W5, 23);
        UIntCircuit u(W5, 3);
        const UInt s = u.add(u.inputs()[0], u.inputs()[1]);
        std::vector<EncryptedUInt> r =
            u.evaluate({A5, B5, C5}, {u.sub(u.min(s, u.inputs()[2]), u.inputs()[0]), u.lt(s, u.inputs()[2])}, -1, true);
        sk.decryptUInt(r[0], got.data());
        sk.decryptUInt(r[1], lt.data());
        bool ok = true;
        for (uint64_t k = 0; k < n; ++k) {
            const uint64_t sum = (a5[k] + b5[k]) & m5;
            ok = ok && got[k] == ((std::min(sum, c5[k]) - a5[k]) & m5) && lt[k] == (sum < c5[k] ? 1u : 0u);
        }
        expect(ok, "composite min(a + b, c) - a, lt(a + b, c)");
    }

    // eager operators
    {
        EncryptedUInt lt = A < B;
        expect(lt.width() == 1, "a < b is one bit");
        std::vector<EncryptedUInt> xs = {A + B, A - B, A * B, lt, A > B, A & B, A ^ B, A | B,
                                         EncryptedUInt::select(lt, A, B)};
        uint64_t (*refs[])(uint64_t, uint64_t) = {
            [](uint64_t x, uint64_t y) -> uint64_t { return (x + y) & 255; },
            [](uint64_t x, uint64_t y) -> uint64_t { return (x - y) & 255; },
            [](uint64_t x, uint64_t y) -> uint64_t { return (x * y) & 255; },
            [](uint64_t x, uint64_t y) -> uint64_t { return x < y; },
            [](uint64_t x, uint64_t y) -> uint64_t { return x > y; },
            [](uint64_t x, uint64_t y) -> uint64_t { return x & y; },
            [](uint64_t x, uint64_t y) -> uint64_t { return x ^ y; },
            [](uint64_t x, uint64_t y) -> uint64_t { return x | y; },
            [](uint64_t x, uint64_t y) -> uint64_t { return std::min(x, y); },
        };
        for (size_t i = 0; i < xs.size(); ++i) {
            sk.decryptUInt(xs[i], got.data());
            bool ok = true;
            for (uint64_t k = 0; k < n; ++k) ok = ok && got[k] == refs[i](a[k], b[k]);
            expect(ok, "eager operator " + std::to_string(i));
        }
    }

    // errors
    {
        UIntCircuit u(W, 2);
        expect_throw([&]() { u.eq(u.inputs()[0], u.inputs()[1]); }, "eq without one");
        expect_throw([&]() { u.invert(u.inputs()[0]); }, "invert without one");
        expect_throw([&]() { u.evaluate({A}, {u.inputs()[0]}); }, "evaluate with a missing operand");
        expect_throw([&]() { u.evaluate({A, B}, {u.inputs()[0]}, -1, false, 0, &one); }, "one given to a plain circuit");
        UIntCircuit narrow(4, 2);
        expect_throw([&]() { narrow.evaluate({A, B}, {narrow.inputs()[0]}); }, "an 8-bit operand in a 4-bit circuit");
        expect_throw([&]() { UIntCircuit(0, 1); }, "width 0");
        std::vector<uint64_t> big(1, 256);
        expect_throw([&]() { sk.encryptUInt(big.data(), 1, 8, 1); }, "a value that does not fit");
        Context other(64, 4);
        SecretKey sk2(other);
        EncryptedUInt Z = sk2.encryptUInt(a.data(), 16, W, 1);
        expect_throw([&]() { A + Z; }, "operands of different sizes and contexts");
    }

    if (failures) {
        std::cout << "uint_demo: " << failures << " checks failed" << std::endl;
        return 1;
    }
    std::cout << "uint_demo: all checks passed" << std::endl;
    return 0;
}
