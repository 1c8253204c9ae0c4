// accept_demos.cpp -- acceptance run of the certFHE API on the GPU engine.
//
// Walks the same three user journeys as the reference's demo programs
// (reference tests/basic_operations.cpp, tests/permutations.cpp, tests/timings.cpp)
// but, unlike them, ASSERTS the outcome: every decrypted bit, the size() figures the
// timing demo prints (352 / 672 / 352 / 144 bytes), and the scheme's homomorphic
// identities on random circuits.  Exit status 0 = all good.
#include "certFHE.h"

#include <cstdio>
#include <cstdlib>
#include <sstream>
#include <string>
#include <vector>

#include <unistd.h>

using namespace certFHE;

static int failures = 0;

// the files this program writes go to a fresh directory under $TMPDIR (default /tmp), so that runs by several users or
// at the same time never meet each other's files
static std::string scratch;
static std::string scratch_file(const char *name) {
    if (scratch.empty()) {
        const char *base = getenv("TMPDIR");
        std::string tmpl = std::string(base && *base ? base : "/tmp") + "/csgn_accept_XXXXXX";
        std::vector<char> buf(tmpl.begin(), tmpl.end());
        buf.push_back('\0');
        if (!mkdtemp(buf.data())) {
            perror("mkdtemp");
            exit(2);
        }
        scratch = buf.data();
    }
    return scratch + "/" + name;
}

#define EXPECT(cond)                                                            \
    do {                                                                        \
        if (!(cond)) {                                                          \
            std::cerr << "FAILED " << __FILE__ << ":" << __LINE__ << "  " #cond << std::endl; \
            ++failures;                                                         \
        }                                                                       \
    } while (0)

static void basic_operations() {
    Context context(1247, 16);
    SecretKey seckey(context);
    Plaintext p1(1), p0(0);
    Ciphertext c1 = seckey.encrypt(p1);
    Ciphertext c0 = seckey.encrypt(p0);
    Ciphertext added, multiplied;
    added = c1 + c0;
    multiplied = c1 * c0;
    Plaintext dec_addition = seckey.decrypt(added);
    Plaintext dec_multiplied = seckey.decrypt(multiplied);
    std::cout << "Dec ( Enc (1) + Enc (0) ) = " << dec_addition << std::endl;
    std::cout << "Dec ( Enc (1) * Enc (0) ) = " << dec_multiplied << std::endl;
    EXPECT(dec_addition.getValue() == 1);
    EXPECT(dec_multiplied.getValue() == 0);
    // an assigned-into object keeps a usable context (the reference loses it here)
    Ciphertext again = added * multiplied;
    EXPECT(seckey.decrypt(again).getValue() == 0);
    EXPECT(again.getLen() == 2 * 1 * context.getDefaultN());
}

static void permutations() {
    Context context(1247, 16);
    SecretKey seckey(context);
    Plaintext p1(1);
    Ciphertext c1 = seckey.encrypt(p1);
    Permutation permutation(context);
    SecretKey permutedSecretKey = seckey.applyPermutation(permutation);
    Ciphertext permutedCiphertext = c1.applyPermutation(permutation);
    Plaintext decrypted = permutedSecretKey.decrypt(permutedCiphertext);
    std::cout << " Dec ( Enc ( 1 ) ) = " << decrypted << endl;
    EXPECT(decrypted.getValue() == 1);
    Permutation inversePermutation = permutation.getInverse();
    Permutation identityPermutation;
    identityPermutation = permutation + inversePermutation;
    EXPECT(identityPermutation.getLength() == 1247);
    for (uint64_t i = 0; i < identityPermutation.getLength(); ++i) EXPECT(identityPermutation.getPermutation()[i] == i);
    // and back again with the inverse
    Ciphertext back = permutedCiphertext.applyPermutation(inversePermutation);
    EXPECT(memcmp(back.getValues(), c1.getValues(), c1.getLen() * 8) == 0);
    Permutation mismatched(7);
    EXPECT((permutation + mismatched).getLength() == 0);  // soft failure, as in the reference
}

static void timings_and_sizes() {
    Context context(1247, 16);
    std::ostringstream os;
    os << context;
    EXPECT(os.str() == "N= 1247\nD= 16\nS= 38\n");
    Timer t1("Key generation ");
    t1.start();
    SecretKey seckey(context);
    EXPECT(t1.stopAndPrint() >= 0.0);
    Plaintext p1(1);
    Ciphertext c1 = seckey.encrypt(p1);
    Ciphertext added, multiplicated;
    added = c1 + c1;
    multiplicated = c1 * c1;
    std::cout << "Secret key size: " << seckey.size() << " bytes" << endl;
    std::cout << "Fresh ciphertext size: " << c1.size() << " bytes" << endl;
    std::cout << "After multiplication ciphertext size: " << multiplicated.size() << " bytes" << endl;
    std::cout << "After addition ciphertext size: " << added.size() << " bytes" << endl;
    EXPECT(seckey.size() == 144);
    EXPECT(c1.size() == 352);
    EXPECT(multiplicated.size() == 352);
    EXPECT(added.size() == 672);
    EXPECT(seckey.decrypt(added).getValue() == 0);          // 1 xor 1
    EXPECT(seckey.decrypt(multiplicated).getValue() == 1);  // 1 and 1
}

// Random depth-2 circuits: Dec(sum_i a_i * sum_j b_j + c) == (xor a) & (xor b) ^ c
static void random_circuits(uint64_t N, uint64_t D, unsigned seed, int rounds) {
    Context context(N, D);
    SecretKey seckey(context);
    srand(seed);
    for (int r = 0; r < rounds; ++r) {
        int na = 1 + rand() % 9, nb = 1 + rand() % 9;
        int xa = 0, xb = 0;
        Ciphertext A, B;
        for (int i = 0; i < na; ++i) {
            Plaintext p(rand() % 2);
            xa ^= p.getValue();
            Ciphertext e = seckey.encrypt(p);
            if (i == 0) A = e; else A += e;
        }
        for (int j = 0; j < nb; ++j) {
            Plaintext p(rand() % 2);
            xb ^= p.getValue();
            Ciphertext e = seckey.encrypt(p);
            if (j == 0) B = e; else B = B + e;
        }
        Plaintext pc(rand() % 2);
        Ciphertext C = seckey.encrypt(pc);
        Ciphertext prod = A * B;
        EXPECT(prod.getLen() == (uint64_t)na * nb * context.getDefaultN());
        Ciphertext circuit = prod + C;
        EXPECT(seckey.decrypt(A).getValue() == xa);
        EXPECT(seckey.decrypt(B).getValue() == xb);
        EXPECT(seckey.decrypt(prod).getValue() == (xa & xb));
        EXPECT(seckey.decrypt(circuit).getValue() == ((xa & xb) ^ pc.getValue()));
        A *= B;
        EXPECT(memcmp(A.getValues(), prod.getValues(), prod.getLen() * 8) == 0);
        // every word of the canonical bitlen pattern
        const uint64_t *bl = prod.getBitlen();
        const uint64_t L = context.getDefaultN(), rem = N % 64;
        for (uint64_t i = 0; i < prod.getLen(); ++i) EXPECT(bl[i] == (((i % L) + 1 == L && rem) ? rem : 64));
        // a permuted multi-block product still decrypts under the permuted key
        Permutation pi(context);
        SecretKey pk = seckey.applyPermutation(pi);
        Ciphertext pprod = prod.applyPermutation(pi);
        EXPECT(pprod.getLen() == prod.getLen());
        EXPECT(pk.decrypt(pprod).getValue() == (xa & xb));
    }
}

// Lazy products: operator* keeps the factors; decrypt, permutation and copies never multiply out.
static void lazy_products() {
    Context context(1247, 16);
    SecretKey seckey(context);
    srand(77);
    auto sum_of = [&](int n, int &parity) {
        Ciphertext acc;
        parity = 0;
        for (int i = 0; i < n; ++i) {
            Plaintext p(rand() % 2);
            parity ^= p.getValue();
            Ciphertext e = seckey.encrypt(p);
            if (i == 0) acc = e; else acc += e;
        }
        return acc;
    };
    int pa, pb, pd;
    Ciphertext A = sum_of(40, pa), B = sum_of(30, pb), Dd = sum_of(20, pd);
    Ciphertext eager = (A * B) * Dd;                         // 24,000 blocks, multiplied out
    Library::setLazyProducts(true);
    Ciphertext lazy = (A * B) * Dd;                          // three factors, nothing multiplied
    EXPECT(lazy.getLen() == eager.getLen() && lazy.getBlocks() == 24000);
    EXPECT(seckey.decrypt(lazy).getValue() == (pa & pb & pd));
    EXPECT(seckey.decrypt(eager).getValue() == (pa & pb & pd));
    Permutation pi(context);
    SecretKey pk = seckey.applyPermutation(pi);
    Ciphertext lazy_p = lazy.applyPermutation(pi);           // permutes 90 blocks, not 24,000
    EXPECT(pk.decrypt(lazy_p).getValue() == (pa & pb & pd));
    // a chain far beyond any memory: 10^3 * 10^3 * 10^3 * 10^3 = 10^12 blocks, decrypted from its factors
    int p1, p2, p3, p4;
    Ciphertext c1 = sum_of(1000, p1), c2 = sum_of(1000, p2), c3 = sum_of(1000, p3), c4 = sum_of(1000, p4);
    Ciphertext huge = c1 * c2;
    huge *= c3;
    huge = huge * c4;
    EXPECT(huge.getBlocks() == 1000000000000ull);
    EXPECT(seckey.decrypt(huge).getValue() == (p1 & p2 & p3 & p4));
    // words on demand: multiplying out gives exactly the eager product; copies are independent
    Ciphertext copy = lazy;
    EXPECT(memcmp(lazy.getValues(), eager.getValues(), eager.getLen() * 8) == 0);
    EXPECT(memcmp(lazy_p.getValues(), eager.applyPermutation(pi).getValues(), eager.getLen() * 8) == 0);
    copy += A;
    EXPECT(copy.getLen() == eager.getLen() + A.getLen() && lazy.getLen() == eager.getLen());
    EXPECT(seckey.decrypt(copy).getValue() == ((pa & pb & pd) ^ pa));
    Ciphertext mixed = lazy + (A * B);                       // sums multiply their operands out
    EXPECT(seckey.decrypt(mixed).getValue() == ((pa & pb & pd) ^ (pa & pb)));
    Library::setLazyProducts(false);
    // save / load: the words, the context and the decrypted bit survive the file
    const std::string path = scratch_file("demo.ct");
    eager.save(path);
    Ciphertext loaded = Ciphertext::load(path);
    EXPECT(loaded.getLen() == eager.getLen() && loaded.getContext().getN() == 1247 && loaded.getContext().getD() == 16);
    EXPECT(memcmp(loaded.getValues(), eager.getValues(), eager.getLen() * 8) == 0);
    EXPECT(seckey.decrypt(loaded).getValue() == (pa & pb & pd));
    remove(path.c_str());
    // batched GPU encryption: 100,000 fresh blocks in one call, decrypting to the XOR of the bits
    std::vector<unsigned char> many(100000);
    int xorbits = 0;
    for (size_t i = 0; i < many.size(); ++i) { many[i] = rand() & 1; xorbits ^= many[i]; }
    Ciphertext batch = seckey.encryptBatch(many.data(), many.size(), 2024);
    EXPECT(batch.getBlocks() == many.size() && seckey.decrypt(batch).getValue() == xorbits);
    Ciphertext batch_sq = batch * A;
    EXPECT(seckey.decrypt(batch_sq).getValue() == (xorbits & pa));
    // n decrypts with one synchronisation (the folds overlap on the library's lanes)
    {
        Ciphertext group[5] = {A, B, eager, batch, batch_sq};
        unsigned char bits[5];
        seckey.decryptBatch(group, 5, bits);
        for (int i = 0; i < 5; ++i) EXPECT(bits[i] == seckey.decrypt(group[i]).getValue());
    }
    // copy-on-write: a copy shares the buffer until one side grows
    Ciphertext x = A, y = x;
    y += B;
    EXPECT(x.getLen() == A.getLen() && y.getLen() == A.getLen() + B.getLen());
    EXPECT(memcmp(x.getValues(), A.getValues(), A.getLen() * 8) == 0);
    x += x;
    EXPECT(x.getLen() == 2 * A.getLen() && seckey.decrypt(x).getValue() == 0);
}

// Fused products (the default): operator* notes its operands; SecretKey::decrypt of a product that has not been written
// yet writes it AND folds it in one kernel.  Everything observable must equal the one-kernel-per-operator behaviour.
static void fused_products() {
    Context context(1247, 16);
    SecretKey seckey(context);
    srand(99);
    auto sum_of = [&](int n, int &parity) {
        Ciphertext acc;
        parity = 0;
        for (int i = 0; i < n; ++i) {
            Plaintext p(rand() % 2);
            parity ^= p.getValue();
            Ciphertext e = seckey.encrypt(p);
            if (i == 0) acc = e; else acc += e;
        }
        return acc;
    };
    int pa, pb, pd;
    Ciphertext A = sum_of(37, pa), B = sum_of(23, pb), Dd = sum_of(11, pd);
    Library::setFusedProducts(false);
    Ciphertext eager = A * B;                                  // csgn_mul, now
    Ciphertext eager3 = eager * Dd;
    Library::setFusedProducts(true);
    EXPECT(Library::getFusedProducts() && Library::getAutoLanes());
    // decrypt first: the fused kernel writes the product and folds it; the words are there afterwards
    Ciphertext f1 = A * B;
    EXPECT(f1.getLen() == eager.getLen() && f1.getBlocks() == 37 * 23);
    Plaintext p1 = seckey.decrypt(f1);                         // pending until read
    Plaintext p1copy = p1;
    EXPECT(memcmp(f1.getValues(), eager.getValues(), eager.getLen() * 8) == 0);
    EXPECT(p1.getValue() == (pa & pb) && p1copy.getValue() == (pa & pb));
    EXPECT(seckey.decrypt(f1).getValue() == (pa & pb));        // again, now a plain fold of the written product
    // words first: a plain multiply, then a plain fold
    Ciphertext f2 = A * B;
    EXPECT(memcmp(f2.getValues(), eager.getValues(), eager.getLen() * 8) == 0);
    EXPECT(seckey.decrypt(f2).getValue() == (pa & pb));
    // copies of a pending product: whichever is used first writes it, the other picks it up
    Ciphertext f3 = A * B, f3copy = f3;
    EXPECT(seckey.decrypt(f3copy).getValue() == (pa & pb));
    EXPECT(memcmp(f3.getValues(), eager.getValues(), eager.getLen() * 8) == 0);
    // chains: the inner product is written once, the outer one is fused with its decrypt
    Ciphertext inner = A * B;
    Ciphertext c1 = inner * Dd, c2 = inner * A;
    EXPECT(c1.getBlocks() == 37 * 23 * 11);
    EXPECT(seckey.decrypt(c1).getValue() == (pa & pb & pd));
    EXPECT(seckey.decrypt(c2).getValue() == (pa & pb & pa));
    EXPECT(memcmp(c1.getValues(), eager3.getValues(), eager3.getLen() * 8) == 0);
    Ciphertext acc = A;
    acc *= B;
    acc *= Dd;
    EXPECT(seckey.decrypt(acc).getValue() == (pa & pb & pd));
    EXPECT(memcmp(acc.getValues(), eager3.getValues(), eager3.getLen() * 8) == 0);
    // a pending product in a sum, permuted, saved
    Ciphertext s = (A * B) + Dd;
    EXPECT(s.getLen() == eager.getLen() + Dd.getLen() && seckey.decrypt(s).getValue() == ((pa & pb) ^ pd));
    Permutation pi(context);
    SecretKey pk = seckey.applyPermutation(pi);
    Ciphertext fp = (A * B).applyPermutation(pi);              // permutes the operands; still pending
    EXPECT(pk.decrypt(fp).getValue() == (pa & pb));
    EXPECT(memcmp(fp.getValues(), eager.applyPermutation(pi).getValues(), eager.getLen() * 8) == 0);
    // many decrypts in flight, read afterwards (one synchronisation at the first read)
    std::vector<Ciphertext> prods;
    std::vector<Plaintext> plains;
    for (int i = 0; i < 40; ++i) prods.push_back(i % 2 ? A * B : B * Dd);
    for (int i = 0; i < 40; ++i) plains.push_back(seckey.decrypt(prods[i]));
    for (int i = 0; i < 40; ++i) EXPECT(plains[i].getValue() == (i % 2 ? (pa & pb) : (pb & pd)));
    std::ostringstream os;
    os << plains[1];
    EXPECT(os.str() == std::string(1, (char)('0' | (pa & pb))) + "\n");
    Plaintext set = seckey.decrypt(prods[0]);
    set.setValue(1);                                            // overrides a pending value
    EXPECT(set.getValue() == 1);
}

// Zero-copy sums (the default): operator+ of large ciphertexts refers to the operands instead of copying them.
static void rope_sums() {
    Context context(1247, 16);
    SecretKey seckey(context);
    srand(123);
    std::vector<unsigned char> bx(9000), by(8000), bz(3);
    int px = 0, py = 0, pz = 0;
    for (size_t i = 0; i < bx.size(); ++i) { bx[i] = rand() & 1; px ^= bx[i]; }
    for (size_t i = 0; i < by.size(); ++i) { by[i] = rand() & 1; py ^= by[i]; }
    for (size_t i = 0; i < bz.size(); ++i) { bz[i] = rand() & 1; pz ^= bz[i]; }
    Ciphertext x = seckey.encryptBatch(bx.data(), bx.size(), 1), y = seckey.encryptBatch(by.data(), by.size(), 2);
    Ciphertext z = seckey.encryptBatch(bz.data(), bz.size(), 3);
    Library::setRopeSums(false);
    Ciphertext copied = x + y;                              // csgn_concat: both operands copied
    Library::setRopeSums(true);
    EXPECT(Library::getRopeSums());
    Ciphertext sum = x + y;                                 // refers to x and y
    EXPECT(sum.getLen() == copied.getLen() && sum.getBlocks() == 17000);
    EXPECT(seckey.decrypt(sum).getValue() == (px ^ py));
    Permutation pi(context);
    SecretKey pk = seckey.applyPermutation(pi);
    Ciphertext psum = sum.applyPermutation(pi);
    EXPECT(pk.decrypt(psum).getValue() == (px ^ py));
    EXPECT(memcmp(psum.getValues(), copied.applyPermutation(pi).getValues(), copied.getLen() * 8) == 0);
    Ciphertext left = sum * z, right = z * sum;             // sum on the left: per part; on the right: made dense once
    EXPECT(seckey.decrypt(left).getValue() == ((px ^ py) & pz));
    EXPECT(memcmp(left.getValues(), (copied * z).getValues(), left.getLen() * 8) == 0);
    EXPECT(memcmp(right.getValues(), (z * copied).getValues(), right.getLen() * 8) == 0);
    // growing an operand afterwards must not change the sum
    Ciphertext sum2 = x + y;
    x += z;
    EXPECT(x.getBlocks() == 9003 && sum2.getBlocks() == 17000);
    EXPECT(memcmp(sum2.getValues(), copied.getValues(), copied.getLen() * 8) == 0);
    EXPECT(seckey.decrypt(x).getValue() == (px ^ pz));
    // a sum of sums, grown in place afterwards
    Ciphertext big = (sum2 + copied) + sum2;
    EXPECT(big.getBlocks() == 51000 && seckey.decrypt(big).getValue() == (px ^ py));
    big += z;
    EXPECT(big.getBlocks() == 51003 && seckey.decrypt(big).getValue() == (px ^ py ^ pz));
}

// SecretKey / Permutation files, and a ciphertext as one file per rank (here: the single rank of this process).
static void files() {
    Context context(1247, 16);
    SecretKey seckey(context);
    srand(321);
    Permutation pi(context);
    std::vector<unsigned char> bits(5000);
    int parity = 0;
    for (size_t i = 0; i < bits.size(); ++i) { bits[i] = rand() & 1; parity ^= bits[i]; }
    Ciphertext c = seckey.encryptBatch(bits.data(), bits.size(), 9);
    const std::string sk = scratch_file("accept.sk"), pm = scratch_file("accept.pm"), ct = scratch_file("accept.ct");
    seckey.save(sk);
    pi.save(pm);
    srand(5);
    const int before = rand();
    srand(5);
    SecretKey k2 = SecretKey::load(sk);
    EXPECT(rand() == before);                                   // loading a key leaves the caller's rand() sequence alone
    Permutation p2 = Permutation::load(pm);
    EXPECT(k2.getLength() == seckey.getLength() && memcmp(k2.getKey(), seckey.getKey(), 16 * 8) == 0);
    EXPECT(p2.getLength() == 1247 && memcmp(p2.getPermutation(), pi.getPermutation(), 1247 * 8) == 0);
    EXPECT(k2.decrypt(c).getValue() == parity);
    EXPECT(k2.applyPermutation(p2).decrypt(*new Ciphertext(c.applyPermutation(p2))).getValue() == parity);
    c.saveSharded(ct);
    Ciphertext back = Ciphertext::loadSharded(ct);
    EXPECT(back.isSharded() && back.getBlocks() == 5000);
    EXPECT(memcmp(back.getValues(), c.getValues(), c.getLen() * 8) == 0);
    bool threw = false;
    try { Ciphertext::load(ct + ".shard0of1"); } catch (const Error &) { threw = true; }
    EXPECT(threw);
    remove(sk.c_str());
    remove(pm.c_str());
    remove((ct + ".shard0of1").c_str());
}

static void misuse_is_loud() {
    Context context(1247, 16);
    uint64_t words[20] = {0}, bitlen[20];
    for (int i = 0; i < 20; ++i) bitlen[i] = 64;  // last word should be 31
    bool threw = false;
    try { Ciphertext bad(words, bitlen, 20, context); } catch (const Error &) { threw = true; }
    EXPECT(threw);
    threw = false;
    try { Ciphertext bad(words, nullptr, 19, context); } catch (const Error &) { threw = true; }
    EXPECT(threw);
    // staged construction through the setters, in the order the reference allows
    bitlen[19] = 31;
    Ciphertext staged;
    staged.setValues(words, 20);
    staged.setBitlen(bitlen, 20);
    staged.setContext(context);
    EXPECT(staged.getLen() == 20);
    EXPECT(staged.getBitlen()[19] == 31 && staged.getValues()[0] == 0);
    Ciphertext empty;
    EXPECT(empty.getLen() == 0 && empty.getValues() == nullptr);
}

int main() {
    std::cout << "Initializing certFHE library................OK" << endl;
    Library::initializeLibrary();
    basic_operations();
    permutations();
    timings_and_sizes();
    random_circuits(1247, 16, 1, 6);
    random_circuits(16383, 64, 2, 2);
    random_circuits(191, 5, 3, 4);   // odd number of words per block
    random_circuits(128, 4, 4, 4);   // N % 64 == 0 (the reference overflows its arrays here)
    lazy_products();
    fused_products();
    rope_sums();
    files();
    Library::setLazyProducts(true);
    random_circuits(1247, 16, 5, 4);  // the same circuits with products kept lazy
    Library::setLazyProducts(false);
    Library::setFusedProducts(false);  // ... and with one kernel per operator on one stream (the first release)
    Library::setAutoLanes(false);
    random_circuits(1247, 16, 6, 4);
    random_circuits(191, 5, 7, 2);
    Library::setFusedProducts(true);
    Library::setAutoLanes(true);
    misuse_is_loud();
    if (!scratch.empty()) rmdir(scratch.c_str());
    if (failures) {
        std::cerr << failures << " expectation(s) failed" << endl;
        return 1;
    }
    std::cout << "accept_demos: all expectations hold" << endl;
    return 0;
}
