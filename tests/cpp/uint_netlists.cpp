// uint_netlists.cpp -- host only: prints the flat netlist certFHE::UIntCircuit builds for every integer operation, one
// line per operation ("op n_inputs gates... -> result wires"), in the order and format of python_netlists() in
// tests/test_uint_cpu.py, which checks that both builders emit the same netlists.  Building a netlist touches no device.
#include "certFHE.h"

#include <cstdio>
#include <cstdlib>
#include <string>

using namespace certFHE;
typedef UIntCircuit::UInt UInt;

namespace {

void print(const char *op, const UIntCircuit &c, const UInt &r) {
    std::string line = std::string(op) + " " + std::to_string(c.circuit().inputCount());
    for (uint32_t g : c.circuit().getNetlist()) line += " " + std::to_string(g);
    line += " ->";
    for (uint32_t w : r) line += " " + std::to_string(w);
    std::printf("%s\n", line.c_str());
}

typedef UInt (UIntCircuit::*Binary)(const UInt &, const UInt &);

void binary(const char *op, Binary f, uint32_t W, bool one) {
    UIntCircuit c(W, 2, one);
    const UInt r = (c.*f)(c.inputs()[0], c.inputs()[1]);
    print(op, c, r);
}

}  // namespace

int main(int argc, char **argv) {
    const uint32_t W = argc > 1 ? (uint32_t)std::atoi(argv[1]) : 8;
    // sorted by name, as the Python side lists them
    binary("add", &UIntCircuit::add, W, false);
    binary("and", &UIntCircuit::and_, W, false);
    binary("eq", &UIntCircuit::eq, W, true);
    binary("ge", &UIntCircuit::ge, W, true);
    binary("gt", &UIntCircuit::gt, W, false);
    binary("le", &UIntCircuit::le, W, true);
    binary("lt", &UIntCircuit::lt, W, false);
    binary("max", &UIntCircuit::max, W, false);
    binary("min", &UIntCircuit::min, W, false);
    binary("mul", &UIntCircuit::mul, W, false);
    binary("ne", &UIntCircuit::ne, W, false);
    binary("or", &UIntCircuit::or_, W, false);
    binary("sub", &UIntCircuit::sub, W, false);
    binary("xor", &UIntCircuit::xor_, W, false);
    {
        UIntCircuit c(W, 1, true);
        const UInt r = c.invert(c.inputs()[0]);
        print("invert", c, r);
    }
    {
        UIntCircuit c(W, 1);
        const UInt r = c.neg(c.inputs()[0]);
        print("neg", c, r);
    }
    {
        UIntCircuit c(W, 1);
        const UInt r = c.shl(c.inputs()[0], 3);
        print("shl3", c, r);
    }
    {
        UIntCircuit c(W, 1);
        const UInt r = c.shr(c.inputs()[0], 2);
        print("shr2", c, r);
    }
    {
        UIntCircuit c(W, 3);
        const UInt r = c.select(UInt(1, c.inputs()[0][0]), c.inputs()[1], c.inputs()[2]);
        print("select", c, r);
    }
    // the NOT-based operations refuse a circuit without `one`
    UIntCircuit plain(W, 2);
    try {
        plain.eq(plain.inputs()[0], plain.inputs()[1]);
        std::printf("FAIL: eq without one did not throw\n");
        return 1;
    } catch (const Error &) {
    }
    return 0;
}
