// dropin_golden.cpp -- the certFHE drop-in driven through its public class API on the inputs of the stored
// reference cases (tests/golden/csgn_golden.json, written by the unmodified reference); tests/test_cpp_dropin.py
// compares what this prints with the stored outputs.
//
//   dropin_golden host   Context, Permutation generation in rand() order, inverse, composition, SecretKey
//                        setKey / applyPermutation / size: host-side classes only, no GPU
//   dropin_golden all    also encrypt in rand() order, Ciphertext operator* / operator+, getBitlen, size(),
//                        SecretKey::decrypt, applyPermutation (reference-strict and every block): needs the GPU
//
// stdin: the number of cases, then per case "N D seed na nb", na bits, nb bits, D key positions.
// stdout: one "name value..." line per observable; words as 16 hex digits each, lists as decimal.
#include "certFHE.h"

#include <cstdio>
#include <cstring>
#include <iostream>
#include <string>
#include <vector>

using namespace certFHE;

static void hex(const char *name, const uint64_t *v, uint64_t n) {
    printf("%s ", name);
    for (uint64_t i = 0; i < n; ++i) printf("%016llx", (unsigned long long)v[i]);
    printf("\n");
}

static void dec(const char *name, const uint64_t *v, uint64_t n) {
    printf("%s", name);
    for (uint64_t i = 0; i < n; ++i) printf(" %llu", (unsigned long long)v[i]);
    printf("\n");
}

static std::vector<uint64_t> canonical_bitlen(uint64_t N, uint64_t n_words) {
    const uint64_t L = N / 64 + (N % 64 ? 1 : 0), rem = N % 64;
    std::vector<uint64_t> bl(n_words);
    for (uint64_t i = 0; i < n_words; ++i) bl[i] = ((i % L) + 1 == L && rem) ? rem : 64;
    return bl;
}

static Ciphertext from_words(const std::vector<uint64_t> &w, uint64_t N, const Context &ctx) {
    std::vector<uint64_t> bl = canonical_bitlen(N, w.size());
    return Ciphertext(w.data(), bl.data(), w.size(), ctx);
}

int main(int argc, char **argv) {
    const bool all = argc > 1 && std::string(argv[1]) == "all";
    if (all) Library::initializeLibrary();
    int cases = 0;
    std::cin >> cases;
    for (int c = 0; c < cases; ++c) {
        uint64_t N, D, seed, na, nb;
        std::cin >> N >> D >> seed >> na >> nb;
        std::vector<int> bits_a(na), bits_b(nb);
        for (auto &x : bits_a) std::cin >> x;
        for (auto &x : bits_b) std::cin >> x;
        std::vector<uint64_t> key(D);
        for (auto &x : key) std::cin >> x;
        if (!std::cin) {
            fprintf(stderr, "dropin_golden: malformed input in case %d\n", c);
            return 2;
        }
        printf("case %d\n", c);
        Context ctx(N, D);
        const uint64_t L = ctx.getDefaultN();
        const uint64_t cx[4] = {ctx.getN(), ctx.getD(), ctx.getS(), L};
        dec("context", cx, 4);
        SecretKey sk(ctx);
        sk.setKey(key.data(), D);
        printf("sk_size %ld\n", (long)sk.size());

        std::vector<uint64_t> a, b;
        if (all) {                               // the reference cases encrypt after srand(seed) and srand(seed + 1)
            for (int half = 0; half < 2; ++half) {
                srand((unsigned)(seed + half));
                std::vector<uint64_t> &out = half ? b : a;
                for (int bit : half ? bits_b : bits_a) {
                    Plaintext p(bit);
                    Ciphertext e = sk.encrypt(p);
                    out.insert(out.end(), e.getValues(), e.getValues() + e.getLen());
                }
            }
            hex("enc_a", a.data(), a.size());
            hex("enc_b", b.data(), b.size());
        }

        srand((unsigned)(seed + 2));
        Permutation perm(N);
        Permutation inv = perm.getInverse();
        Permutation ident = perm + inv;
        dec("perm", perm.getPermutation(), perm.getLength());
        dec("perm_inverse", inv.getPermutation(), inv.getLength());
        dec("perm_compose", ident.getPermutation(), ident.getLength());
        SecretKey pkey = sk.applyPermutation(perm);
        dec("permuted_key", pkey.getKey(), pkey.getLength());
        if (!all) continue;

        Ciphertext A = from_words(a, N, ctx), B = from_words(b, N, ctx);
        Ciphertext prod = A * B, summ = A + B;
        hex("mul", prod.getValues(), prod.getLen());
        hex("mul_bitlen", prod.getBitlen(), prod.getLen());
        hex("add", summ.getValues(), summ.getLen());
        hex("add_bitlen", summ.getBitlen(), summ.getLen());
        printf("dec %d %d %d %d\n", sk.decrypt(A).getValue(), sk.decrypt(B).getValue(), sk.decrypt(prod).getValue(),
               sk.decrypt(summ).getValue());
        Library::setStrictReferencePermutation(true);      // the reference's result: block 0 permuted
        Ciphertext strict = A.applyPermutation(perm);
        Library::setStrictReferencePermutation(false);
        hex("permute_strict", strict.getValues(), strict.getLen());
        dec("permute_strict_bitlen", strict.getBitlen(), strict.getLen());
        Ciphertext each = A.applyPermutation(perm);
        hex("permute_each_block", each.getValues(), each.getLen());
        printf("dec_permuted %d\n", pkey.decrypt(each).getValue());
        Ciphertext one = from_words(std::vector<uint64_t>(a.begin(), a.begin() + L), N, ctx);
        printf("ct_size_one_block %ld\n", (long)one.size());
    }
    fflush(stdout);
    return 0;
}
