// uint_types.cpp -- encrypted integers over the C ABI (include/csgn.h, "encrypted integers"):
//   SecretKey::encryptUInt / decryptUInt -> csgn_encrypt_uint / csgn_decrypt_uint (one launch each)
//   UIntCircuit                           -> integer netlists, one csgn_seg_circuit call per evaluate()
//   EncryptedUInt operators              -> a one-operation UIntCircuit each
// The netlists are those of csgn_b200/engine.py's UIntCircuit, wire for wire (tests/test_uint_cpu.py compares them).
#include "certFHE.h"
#include "engine_glue.h"

namespace certFHE {

namespace {

void check_width(uint32_t width, const char *who) {
    if (width < 1 || width > 64) throw Error(std::string(who) + ": width " + to_string(width) + " outside 1..64");
}

}  // namespace

// ---- EncryptedUInt --------------------------------------------------------------------------------------------------
EncryptedUInt::EncryptedUInt(const std::vector<CiphertextArray> &p) : planes(p) {
    if (planes.empty()) throw Error("EncryptedUInt: no bit planes");
    check_width((uint32_t)planes.size(), "EncryptedUInt");
    for (size_t j = 1; j < planes.size(); ++j) {
        if (planes[j].size() != planes[0].size()) throw Error("EncryptedUInt: bit planes of different sizes");
        if (planes[j].getContext().getN() != planes[0].getContext().getN() ||
            planes[j].getContext().getD() != planes[0].getContext().getD())
            throw Error("EncryptedUInt: bit planes of different contexts");
    }
}

namespace {

typedef UIntCircuit::UInt (UIntCircuit::*BinaryOp)(const UIntCircuit::UInt &, const UIntCircuit::UInt &);

EncryptedUInt apply(BinaryOp op, const EncryptedUInt &a, const EncryptedUInt &b) {
    UIntCircuit c(std::max(a.width(), b.width()), 2);
    const UIntCircuit::UInt r = (c.*op)(c.inputs()[0], c.inputs()[1]);
    return c.evaluate({a, b}, {r}, -1, true)[0];
}

}  // namespace

EncryptedUInt EncryptedUInt::operator+(const EncryptedUInt &b) const { return apply(&UIntCircuit::add, *this, b); }
EncryptedUInt EncryptedUInt::operator-(const EncryptedUInt &b) const { return apply(&UIntCircuit::sub, *this, b); }
EncryptedUInt EncryptedUInt::operator*(const EncryptedUInt &b) const { return apply(&UIntCircuit::mul, *this, b); }
EncryptedUInt EncryptedUInt::operator<(const EncryptedUInt &b) const { return apply(&UIntCircuit::lt, *this, b); }
EncryptedUInt EncryptedUInt::operator>(const EncryptedUInt &b) const { return apply(&UIntCircuit::gt, *this, b); }
EncryptedUInt EncryptedUInt::operator&(const EncryptedUInt &b) const { return apply(&UIntCircuit::and_, *this, b); }
EncryptedUInt EncryptedUInt::operator^(const EncryptedUInt &b) const { return apply(&UIntCircuit::xor_, *this, b); }
EncryptedUInt EncryptedUInt::operator|(const EncryptedUInt &b) const { return apply(&UIntCircuit::or_, *this, b); }

EncryptedUInt EncryptedUInt::select(const EncryptedUInt &c, const EncryptedUInt &x, const EncryptedUInt &y) {
    if (c.width() != 1) throw Error("EncryptedUInt::select: the condition has " + to_string(c.width()) + " bits, not 1");
    UIntCircuit u(std::max(x.width(), y.width()), 3);
    const UIntCircuit::UInt s(1, u.inputs()[0][0]);
    return u.evaluate({c, x, y}, {u.select(s, u.inputs()[1], u.inputs()[2])}, -1, true)[0];
}

// ---- UIntCircuit: wires and gates -------------------------------------------------------------------------------------
UIntCircuit::UIntCircuit(uint32_t width, uint32_t n_operands, bool one)
    : w(width), operands(n_operands), has_one(one), one_w(n_operands * width), zero_w(n_operands * width + (one ? 1 : 0)),
      c((check_width(width, "UIntCircuit"), zero_w + 1)) {
    for (uint32_t i = 0; i < operands; ++i) {
        UInt x(w);
        for (uint32_t j = 0; j < w; ++j) x[j] = i * w + j;
        in.push_back(x);
    }
}

uint32_t UIntCircuit::gate(std::vector<std::pair<uint32_t, uint32_t>> products, std::vector<uint32_t> terms) {
    std::vector<uint32_t> t;
    for (uint32_t x : terms)
        if (x != zero_w) t.push_back(x);
    std::vector<std::pair<uint32_t, uint32_t>> p;
    for (const auto &pr : products) {
        if (pr.first == zero_w || pr.second == zero_w) continue;
        if (has_one && pr.first == one_w) t.push_back(pr.second);
        else if (has_one && pr.second == one_w) t.push_back(pr.first);
        else p.push_back(pr);
    }
    if (p.empty() && t.empty()) return zero_w;
    if (p.empty() && t.size() == 1) return t[0];
    return c.gate(p, t);
}

uint32_t UIntCircuit::notw(uint32_t x) {
    if (!has_one) throw Error("UIntCircuit: NOT needs the `one` input: build the circuit with one = true");
    return gate({}, {x, one_w});
}

void UIntCircuit::pair(UInt &a, UInt &b) const {
    const size_t n = std::max(a.size(), b.size());
    a.resize(n, zero_w);
    b.resize(n, zero_w);
}

// borrow of a - b - r: a*b + t*r + b + r with t = a + b, which is (not a and b) or (not (a xor b) and r)
uint32_t UIntCircuit::borrow(uint32_t a, uint32_t b, uint32_t r, uint32_t t) { return gate({{a, b}, {t, r}}, {b, r}); }

// ---- UIntCircuit: operations ------------------------------------------------------------------------------------------
UIntCircuit::UInt UIntCircuit::add(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0, out;
    pair(a, b);
    uint32_t carry = zero_w;
    for (size_t i = 0; i < a.size(); ++i) {
        const uint32_t t = gate({}, {a[i], b[i]});
        out.push_back(gate({}, {t, carry}));
        if (i + 1 < a.size()) carry = gate({{a[i], b[i]}, {t, carry}}, {});
    }
    return out;
}

UIntCircuit::UInt UIntCircuit::sub(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0, out;
    pair(a, b);
    uint32_t r = zero_w;
    for (size_t i = 0; i < a.size(); ++i) {
        const uint32_t t = gate({}, {a[i], b[i]});
        out.push_back(gate({}, {t, r}));
        if (i + 1 < a.size()) r = borrow(a[i], b[i], r, t);
    }
    return out;
}

UIntCircuit::UInt UIntCircuit::neg(const UInt &a) { return sub(UInt(a.size(), zero_w), a); }

UIntCircuit::UInt UIntCircuit::lt(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0;
    pair(a, b);
    uint32_t r = zero_w;
    for (size_t i = 0; i < a.size(); ++i) {
        const uint32_t t = r != zero_w ? gate({}, {a[i], b[i]}) : zero_w;
        r = borrow(a[i], b[i], r, t);
    }
    return UInt(1, r);
}

UIntCircuit::UInt UIntCircuit::gt(const UInt &a, const UInt &b) { return lt(b, a); }

UIntCircuit::UInt UIntCircuit::ne(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0;
    pair(a, b);
    uint32_t o = zero_w;
    for (size_t i = 0; i < a.size(); ++i) {
        const uint32_t t = gate({}, {a[i], b[i]});
        o = o == zero_w ? t : gate({{o, t}}, {o, t});
    }
    return UInt(1, o);
}

UIntCircuit::UInt UIntCircuit::eq(const UInt &a, const UInt &b) { return UInt(1, notw(ne(a, b)[0])); }
UIntCircuit::UInt UIntCircuit::le(const UInt &a, const UInt &b) { return UInt(1, notw(gt(a, b)[0])); }
UIntCircuit::UInt UIntCircuit::ge(const UInt &a, const UInt &b) { return UInt(1, notw(lt(a, b)[0])); }

UIntCircuit::UInt UIntCircuit::invert(const UInt &a) {
    UInt out;
    for (uint32_t x : a) out.push_back(notw(x));
    return out;
}

UIntCircuit::UInt UIntCircuit::select(const UInt &s, const UInt &x0, const UInt &y0) {
    if (s.size() != 1) throw Error("UIntCircuit::select: the condition has " + to_string(s.size()) + " bits, not 1");
    UInt x = x0, y = y0, out;
    pair(x, y);
    for (size_t i = 0; i < x.size(); ++i) out.push_back(gate({{s[0], x[i]}, {s[0], y[i]}}, {y[i]}));
    return out;
}

UIntCircuit::UInt UIntCircuit::min(const UInt &a, const UInt &b) { return select(lt(a, b), a, b); }
UIntCircuit::UInt UIntCircuit::max(const UInt &a, const UInt &b) { return select(lt(a, b), b, a); }

// schoolbook rows a*b_j shifted by j, each added to the accumulator with ripple carries (a column of three addends
// carries their majority, of two their product)
UIntCircuit::UInt UIntCircuit::mul(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0;
    pair(a, b);
    const size_t W = a.size();
    UInt acc(W, zero_w);
    for (size_t j = 0; j < W; ++j) {
        UInt pp(j, zero_w), out;
        for (size_t i = 0; i + j < W; ++i) pp.push_back(gate({{a[i], b[j]}}, {}));
        uint32_t carry = zero_w;
        for (size_t k = 0; k < W; ++k) {
            std::vector<uint32_t> ops;
            for (uint32_t x : {acc[k], pp[k], carry})
                if (x != zero_w) ops.push_back(x);
            out.push_back(gate({}, ops));
            std::vector<std::pair<uint32_t, uint32_t>> prods;
            for (size_t p = 0; p < ops.size(); ++p)
                for (size_t q = p + 1; q < ops.size(); ++q) prods.push_back({ops[p], ops[q]});
            carry = !prods.empty() && k + 1 < W ? gate(prods, {}) : zero_w;
        }
        acc = out;
    }
    return acc;
}

UIntCircuit::UInt UIntCircuit::and_(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0, out;
    pair(a, b);
    for (size_t i = 0; i < a.size(); ++i) out.push_back(gate({{a[i], b[i]}}, {}));
    return out;
}

UIntCircuit::UInt UIntCircuit::xor_(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0, out;
    pair(a, b);
    for (size_t i = 0; i < a.size(); ++i) out.push_back(gate({}, {a[i], b[i]}));
    return out;
}

UIntCircuit::UInt UIntCircuit::or_(const UInt &a0, const UInt &b0) {
    UInt a = a0, b = b0, out;
    pair(a, b);
    for (size_t i = 0; i < a.size(); ++i) out.push_back(gate({{a[i], b[i]}}, {a[i], b[i]}));
    return out;
}

UIntCircuit::UInt UIntCircuit::shl(const UInt &a, uint32_t k) {
    UInt out(std::min<size_t>(k, a.size()), zero_w);
    for (size_t i = 0; out.size() < a.size(); ++i) out.push_back(a[i]);
    return out;
}

UIntCircuit::UInt UIntCircuit::shr(const UInt &a, uint32_t k) {
    UInt out;
    for (size_t i = k; i < a.size(); ++i) out.push_back(a[i]);
    out.resize(a.size(), zero_w);
    return out;
}

// ---- UIntCircuit: evaluation ------------------------------------------------------------------------------------------
std::vector<EncryptedUInt> UIntCircuit::evaluate(const std::vector<EncryptedUInt> &ops, const std::vector<UInt> &results,
                                                 int64_t minBits, bool cancel, uint64_t laneCapacity,
                                                 const CiphertextArray *one) {
    if (ops.size() != operands)
        throw Error("UIntCircuit::evaluate: the circuit has " + to_string(operands) + " operands, got " +
                    to_string(ops.size()));
    if ((one != nullptr) != has_one) throw Error("UIntCircuit::evaluate: `one` given to a circuit built without it, or missing");
    const CiphertextArray &first = one ? *one : ops.at(0).getPlanes()[0];
    const uint64_t n = first.size();
    const Context ctx = first.getContext();
    csgn_buf *empty = nullptr;
    glue::check(csgn_buf_alloc(0, csgn_words_per_block(ctx.getN()), &empty), "csgn_buf_alloc");
    const CiphertextArray zero(empty, std::vector<uint64_t>(n + 1, 0), ctx);
    std::vector<CiphertextArray> inputs;
    for (const EncryptedUInt &x : ops) {
        if (x.width() > w)
            throw Error("UIntCircuit::evaluate: an operand of " + to_string(x.width()) + " bits in a " + to_string(w) +
                        "-bit circuit");
        for (const CiphertextArray &p : x.getPlanes()) inputs.push_back(p);
        for (uint32_t j = x.width(); j < w; ++j) inputs.push_back(zero);
    }
    if (one) inputs.push_back(*one);
    inputs.push_back(zero);
    std::vector<uint32_t> flat;
    for (const UInt &r : results) {
        if (r.empty()) throw Error("UIntCircuit::evaluate: a result has no bits");
        flat.insert(flat.end(), r.begin(), r.end());
    }
    std::vector<CiphertextArray> arrs = c.evaluate(inputs, flat, minBits, cancel, laneCapacity);
    std::vector<EncryptedUInt> out;
    size_t at = 0;
    for (const UInt &r : results) {
        out.push_back(EncryptedUInt(std::vector<CiphertextArray>(arrs.begin() + at, arrs.begin() + at + r.size())));
        at += r.size();
    }
    return out;
}

// ---- SecretKey ----------------------------------------------------------------------------------------------------
EncryptedUInt SecretKey::encryptUInt(const uint64_t *values, uint64_t n, uint32_t width, uint64_t seed) {
    check_width(width, "SecretKey::encryptUInt");
    if (!device_key) {
        glue::ensure_engine();
        glue::check(csgn_key_create(certFHEContext->getN(), s, (uint32_t)length, &device_key), "csgn_key_create");
    }
    std::vector<csgn_buf *> bufs(width, nullptr);
    glue::check(csgn_encrypt_uint(device_key, values, n, width, 0, seed, bufs.data()), "csgn_encrypt_uint");
    std::vector<uint64_t> off(n + 1);
    for (uint64_t k = 0; k <= n; ++k) off[k] = k;
    std::vector<CiphertextArray> planes;
    for (csgn_buf *b : bufs) planes.push_back(CiphertextArray(b, off, *certFHEContext));
    return EncryptedUInt(planes);
}

void SecretKey::decryptUInt(const EncryptedUInt &x, uint64_t *values) {
    if (!device_key) {
        glue::ensure_engine();
        glue::check(csgn_key_create(certFHEContext->getN(), s, (uint32_t)length, &device_key), "csgn_key_create");
    }
    std::vector<const csgn_buf *> planes;
    std::vector<const uint64_t *> offs;
    for (const CiphertextArray &p : x.getPlanes()) {
        planes.push_back(p.deviceBuffer());
        offs.push_back(p.getOffsets().data());
    }
    glue::check(csgn_decrypt_uint(planes.data(), offs.data(), x.width(), x.size(), device_key, values),
                "csgn_decrypt_uint");
}

}  // namespace certFHE
