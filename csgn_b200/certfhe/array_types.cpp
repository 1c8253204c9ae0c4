// array_types.cpp -- CiphertextArray and the array members of SecretKey over the C ABI's ciphertext arrays
// (include/csgn.h): each operation is ONE call, which makes one kernel launch for all small elements.
//   CiphertextArray(vector)   -> csgn_concat_n
//   operator* / operator+     -> csgn_seg_mul / csgn_seg_concat
//   sumOfProducts             -> csgn_seg_mul_sum
//   compactSumOfProducts, compact, Ciphertext::compact -> csgn_seg_mul_sum_compact (min_bits = D)
//   cancel, Ciphertext::cancel -> csgn_seg_cancel
//   gather                    -> csgn_seg_gather
//   applyPermutation          -> csgn_permute on the storage (a permutation acts on every block by itself)
//   encryptArray / decryptArray -> csgn_encrypt_batch / csgn_seg_decrypt
#include "certFHE.h"
#include "engine_glue.h"

namespace certFHE {

namespace {

std::shared_ptr<csgn_buf> adopt(csgn_buf *b) {
    return std::shared_ptr<csgn_buf>(b, [](csgn_buf *p) { csgn_buf_free(p); });
}

Context first_context(const std::vector<Ciphertext> &elements) {
    if (elements.empty()) throw Error("CiphertextArray: no elements");
    return elements[0].getContext();
}

}  // namespace

CiphertextArray::CiphertextArray(csgn_buf *buf, const std::vector<uint64_t> &off, const Context &ctx)
    : storage(adopt(buf)), offsets(off), context(ctx) {}

CiphertextArray::CiphertextArray(const std::vector<Ciphertext> &elements) : context(first_context(elements)) {
    std::vector<const csgn_buf *> parts;
    offsets.assign(1, 0);
    for (size_t i = 0; i < elements.size(); ++i) {
        const Ciphertext &c = elements[i];
        if (c.isSharded()) throw Error("CiphertextArray: element " + to_string(i) + " is sharded");
        const csgn_buf *b = c.deviceBuffer();   // writes a pending product; csgn_concat_n makes a lazy sum dense
        if (b) parts.push_back(b);
        offsets.push_back(offsets.back() + (b ? csgn_buf_blocks(b) : 0));
    }
    if (parts.empty()) throw Error("CiphertextArray: every element is empty");
    csgn_buf *out = nullptr;
    glue::check(csgn_concat_n(parts.data(), parts.size(), &out), "csgn_concat_n");
    storage = adopt(out);
}

uint64_t CiphertextArray::size() const { return offsets.size() - 1; }

uint64_t CiphertextArray::getBlocks(uint64_t k) const {
    if (k >= size()) throw Error("CiphertextArray::getBlocks: element " + to_string(k) + " of " + to_string(size()));
    return offsets[k + 1] - offsets[k];
}

Ciphertext CiphertextArray::get(uint64_t k) const {
    const uint64_t n = getBlocks(k);
    csgn_buf *b = nullptr;
    glue::check(csgn_buf_slice(storage.get(), offsets[k], n, &b), "csgn_buf_slice");
    Ciphertext out;
    out.certFHEcontext = new Context(context);
    out.dev = adopt(b);
    return out;
}

Context CiphertextArray::getContext() const { return context; }

const std::vector<uint64_t> &CiphertextArray::getOffsets() const { return offsets; }

const csgn_buf *CiphertextArray::deviceBuffer() const { return storage.get(); }

CiphertextArray CiphertextArray::operator*(const CiphertextArray &c) const {
    if (c.size() != size()) throw Error("CiphertextArray::operator*: arrays of " + to_string(size()) + " and " +
                                        to_string(c.size()) + " elements");
    std::vector<uint64_t> off(size() + 1);
    csgn_buf *out = nullptr;
    glue::check(csgn_seg_mul(storage.get(), offsets.data(), c.storage.get(), c.offsets.data(), size(), off.data(), &out),
                "csgn_seg_mul");
    return CiphertextArray(out, off, context);
}

CiphertextArray CiphertextArray::operator+(const CiphertextArray &c) const {
    if (c.size() != size()) throw Error("CiphertextArray::operator+: arrays of " + to_string(size()) + " and " +
                                        to_string(c.size()) + " elements");
    std::vector<uint64_t> off(size() + 1);
    csgn_buf *out = nullptr;
    glue::check(csgn_seg_concat(storage.get(), offsets.data(), c.storage.get(), c.offsets.data(), size(), off.data(),
                                &out),
                "csgn_seg_concat");
    return CiphertextArray(out, off, context);
}

CiphertextArray CiphertextArray::gate(const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products,
                                      const std::vector<CiphertextArray> &terms, bool compact) {
    const std::string who = compact ? "CiphertextArray::compactSumOfProducts" : "CiphertextArray::sumOfProducts";
    std::vector<const CiphertextArray *> all;
    for (size_t i = 0; i < products.size(); ++i) {
        all.push_back(&products[i].first);
        all.push_back(&products[i].second);
    }
    for (size_t i = 0; i < terms.size(); ++i) all.push_back(&terms[i]);
    if (all.empty()) throw Error(who + ": no products and no terms");
    const CiphertextArray &x0 = *all[0];
    for (size_t i = 1; i < all.size(); ++i) {
        if (all[i]->size() != x0.size())
            throw Error(who + ": arrays of " + to_string(x0.size()) + " and " +
                        to_string(all[i]->size()) + " elements");
        if (all[i]->context.getN() != x0.context.getN() || all[i]->context.getD() != x0.context.getD())
            throw Error(who + ": arrays of different contexts");
    }
    std::vector<const csgn_buf *> a, b, c;
    std::vector<const uint64_t *> ao, bo, co;
    for (size_t i = 0; i < products.size(); ++i) {
        a.push_back(products[i].first.storage.get());
        ao.push_back(products[i].first.offsets.data());
        b.push_back(products[i].second.storage.get());
        bo.push_back(products[i].second.offsets.data());
    }
    for (size_t i = 0; i < terms.size(); ++i) {
        c.push_back(terms[i].storage.get());
        co.push_back(terms[i].offsets.data());
    }
    std::vector<uint64_t> off(x0.size() + 1);
    csgn_buf *out = nullptr;
    if (compact)
        glue::check(csgn_seg_mul_sum_compact(a.data(), ao.data(), b.data(), bo.data(), (uint32_t)products.size(),
                                             c.data(), co.data(), (uint32_t)terms.size(), x0.size(),
                                             (uint32_t)x0.context.getD(), off.data(), &out),
                    "csgn_seg_mul_sum_compact");
    else
        glue::check(csgn_seg_mul_sum(a.data(), ao.data(), b.data(), bo.data(), (uint32_t)products.size(), c.data(),
                                     co.data(), (uint32_t)terms.size(), x0.size(), off.data(), &out),
                    "csgn_seg_mul_sum");
    return CiphertextArray(out, off, x0.context);
}

CiphertextArray CiphertextArray::sumOfProducts(const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products,
                                               const std::vector<CiphertextArray> &terms) {
    return gate(products, terms, false);
}

CiphertextArray CiphertextArray::compactSumOfProducts(
    const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products, const std::vector<CiphertextArray> &terms) {
    return gate(products, terms, true);
}

CiphertextArray CiphertextArray::compact() const { return gate({}, {*this}, true); }

CiphertextArray CiphertextArray::cancel() const {
    std::vector<uint64_t> off(size() + 1);
    csgn_buf *out = nullptr;
    glue::check(csgn_seg_cancel(storage.get(), offsets.data(), size(), off.data(), &out), "csgn_seg_cancel");
    return CiphertextArray(out, off, context);
}


CiphertextArray CiphertextArray::gather(const std::vector<uint64_t> &idx) const {
    std::vector<uint64_t> off(idx.size() + 1);
    csgn_buf *out = nullptr;
    glue::check(csgn_seg_gather(storage.get(), offsets.data(), size(), idx.data(), idx.size(), off.data(), &out),
                "csgn_seg_gather");
    return CiphertextArray(out, off, context);
}

CiphertextArray CiphertextArray::applyPermutation(const Permutation &permutation) const {
    csgn_buf *out = nullptr;
    if (csgn_buf_blocks(storage.get()) == 0)
        glue::check(csgn_buf_clone(storage.get(), &out), "csgn_buf_clone");
    else
        glue::check(csgn_permute(storage.get(), permutation.deviceMap(context.getN()), 0, &out), "csgn_permute");
    return CiphertextArray(out, offsets, context);
}

Ciphertext Ciphertext::compact() const {
    const csgn_buf *b = deviceBuffer();   // writes a pending product; the call makes a lazy sum dense
    if (!b) return *this;
    if (!certFHEcontext) throw Error("Ciphertext::compact: no context");
    const csgn_buf *one[1] = {b};
    const uint64_t off[2] = {0, csgn_buf_blocks(b)};
    const uint64_t *offs[1] = {off};
    uint64_t out_off[2];
    csgn_buf *res = nullptr;
    glue::check(csgn_seg_mul_sum_compact(nullptr, nullptr, nullptr, nullptr, 0, one, offs, 1, 1,
                                         (uint32_t)certFHEcontext->getD(), out_off, &res),
                "csgn_seg_mul_sum_compact");
    Ciphertext out;
    out.certFHEcontext = new Context(*certFHEcontext);
    out.dev = adopt(res);
    out.sharded = sharded;
    return out;
}

Ciphertext Ciphertext::cancel() const {
    const csgn_buf *b = deviceBuffer();   // writes a pending product; the call makes a lazy sum dense
    if (!b) return *this;
    if (!certFHEcontext) throw Error("Ciphertext::cancel: no context");
    const uint64_t off[2] = {0, csgn_buf_blocks(b)};
    uint64_t out_off[2];
    csgn_buf *res = nullptr;
    glue::check(csgn_seg_cancel(b, off, 1, out_off, &res), "csgn_seg_cancel");
    Ciphertext out;
    out.certFHEcontext = new Context(*certFHEcontext);
    out.dev = adopt(res);
    out.sharded = sharded;
    return out;
}

Circuit::Circuit(uint32_t inputs) : inputs(inputs) {
    if (inputs == 0) throw Error("Circuit: a circuit needs at least one input");
}

uint32_t Circuit::gate(const std::vector<std::pair<uint32_t, uint32_t>> &products, const std::vector<uint32_t> &terms) {
    if (products.empty() && terms.empty()) throw Error("Circuit::gate: no products and no terms");
    const uint32_t own = wires();
    for (const auto &pr : products)
        if (pr.first >= own || pr.second >= own) throw Error("Circuit::gate: an operand is not an earlier wire");
    for (uint32_t w : terms)
        if (w >= own) throw Error("Circuit::gate: a term is not an earlier wire");
    netlist.push_back((uint32_t)products.size());
    netlist.push_back((uint32_t)terms.size());
    for (const auto &pr : products) {
        netlist.push_back(pr.first);
        netlist.push_back(pr.second);
    }
    netlist.insert(netlist.end(), terms.begin(), terms.end());
    return inputs + gates++;
}

std::vector<CiphertextArray> Circuit::evaluate(const std::vector<CiphertextArray> &in,
                                               const std::vector<uint32_t> &outputs, int64_t minBits, bool cancel,
                                               uint64_t laneCapacity) {
    if (in.size() != inputs) throw Error("Circuit::evaluate: wrong number of input arrays");
    if (outputs.empty()) throw Error("Circuit::evaluate: no outputs");
    const uint64_t n = in[0].size();
    const Context &ctx = in[0].context;
    std::vector<const csgn_buf *> bufs;
    std::vector<const uint64_t *> offs;
    for (const CiphertextArray &x : in) {
        if (x.size() != n) throw Error("Circuit::evaluate: input arrays of different sizes");
        if (x.context.getN() != ctx.getN() || x.context.getD() != ctx.getD())
            throw Error("Circuit::evaluate: input arrays of different contexts");
        bufs.push_back(x.storage.get());
        offs.push_back(x.offsets.data());
    }
    for (uint32_t w : outputs)
        if (w >= wires()) throw Error("Circuit::evaluate: an output is not a wire of the circuit");
    if (minBits > 64 * (int64_t)csgn_words_per_block(ctx.getN())) throw Error("Circuit::evaluate: minBits out of range");
    const uint32_t mb = minBits < 0 ? (uint32_t)ctx.getD() : (uint32_t)minBits;
    std::vector<std::vector<uint64_t>> off(outputs.size(), std::vector<uint64_t>(n + 1));
    std::vector<uint64_t *> off_p;
    for (auto &o : off) off_p.push_back(o.data());
    std::vector<csgn_buf *> res(outputs.size(), nullptr);
    glue::check(csgn_seg_circuit(bufs.data(), offs.data(), inputs, n, netlist.data(), netlist.size(), gates,
                                 outputs.data(), (uint32_t)outputs.size(), mb, cancel ? 1 : 0, laneCapacity,
                                 off_p.data(), res.data(), &fallback),
                "csgn_seg_circuit");
    std::vector<CiphertextArray> out;
    for (size_t j = 0; j < outputs.size(); ++j) out.push_back(CiphertextArray(res[j], off[j], ctx));
    return out;
}

CiphertextArray SecretKey::encryptArray(const unsigned char *bits, uint64_t n, uint64_t seed) {
    if (!device_key) {
        glue::ensure_engine();
        glue::check(csgn_key_create(certFHEContext->getN(), s, (uint32_t)length, &device_key), "csgn_key_create");
    }
    csgn_buf *buf = nullptr;
    glue::check(csgn_encrypt_batch(device_key, bits, n, 0, seed, &buf), "csgn_encrypt_batch");
    std::vector<uint64_t> off(n + 1);
    for (uint64_t k = 0; k <= n; ++k) off[k] = k;
    return CiphertextArray(buf, off, *certFHEContext);
}

void SecretKey::decryptArray(const CiphertextArray &array, unsigned char *bits) {
    if (!device_key) {
        glue::ensure_engine();
        glue::check(csgn_key_create(certFHEContext->getN(), s, (uint32_t)length, &device_key), "csgn_key_create");
    }
    glue::check(csgn_seg_decrypt(array.deviceBuffer(), array.getOffsets().data(), array.size(), device_key, bits, nullptr),
                "csgn_seg_decrypt");
}

}  // namespace certFHE
