// certFHE.h -- the certFHE C++ API, re-implemented over the B200 engine.
//
// Source-level drop-in for the reference's umbrella header (reference src/certFHE.h:1-11
// and the nine class headers it pulls in): same namespace, class names, public member
// signatures and stream operators, so that programs written against the reference --
// its tests/*.cpp and the README example -- compile unchanged and link against this
// repository's libcertFHE.so.
//
// What is different underneath:
//   * a Ciphertext's blocks live in GPU memory behind a csgn_buf handle
//     (include/csgn.h); + += * *= decrypt applyPermutation are one C-ABI call each
//     into hand-written sm_100a kernels.  There is no CPU evaluation path.
//   * getValues()/getBitlen() hand out a lazily materialised host mirror (the
//     reference hands out its internal arrays: src/Ciphertext.h:92-102);
//   * the `bitlen` side array is never stored: it is always [64]*(L-1)+[N%64]
//     per block (src/SecretKey.cpp:171-173, propagated by src/Ciphertext.cpp:165-176);
//   * defects of the reference that are undefined behaviour there are defined here
//     (operator= keeps the context, N%64==0 works, 64-bit indices) -- DESIGN.md lists them.
// Key generation, encryption and Permutation generation stay on the host and consume
// glibc rand() in exactly the reference's call order, so seeded runs agree bit for bit.
#ifndef CSGN_CERTFHE_API_H_
#define CSGN_CERTFHE_API_H_

#include "utils.h"

#include <memory>
#include <stdexcept>
#include <utility>

struct csgn_buf;
struct csgn_key;
struct csgn_perm;
struct csgn_result;

namespace certFHE {

class CiphertextArray;
class EncryptedUInt;
class UIntCircuit;

// Raised where the reference would run into undefined behaviour or where the GPU
// engine reports a failure.  The reference has no error channel at all; an uncaught
// Error terminates with its message, which is the loud failure we want.
class Error : public std::runtime_error {
public:
    explicit Error(const std::string &what) : std::runtime_error(what) {}
};

// ---- Library / Helper (reference src/Helpers.h:14-43) -----------------------------
class Library {
    Library() {}

public:
    // Seeds rand() with the wall clock (src/Helpers.cpp:8-12) and brings up the GPU
    // engine (csgn_init).  Throws Error when no B200 is usable.
    static void initializeLibrary();

    // Extensions (not in the reference).
    // applyPermutation on a multi-block ciphertext: false (default) permutes every
    // block; true reproduces the reference exactly, whose result is block 0 permuted
    // and one block long (src/Ciphertext.cpp:33-40).  Also set by CSGN_STRICT_REF_PERMUTE=1.
    static void setStrictReferencePermutation(bool strict);
    static bool getStrictReferencePermutation();
    // Block until every enqueued GPU operation has finished (for timing).
    static void synchronize();
    // Lazy products (off by default; also CSGN_LAZY_PRODUCTS=1).  When on, operator* / *= do
    // not materialise the T1*T2 product: the result remembers its factors.  decrypt of such a
    // ciphertext folds the factors only (Dec(a*b) = Dec(a) & Dec(b), exact for this scheme),
    // applyPermutation permutes the factors, and anything that needs the words (getValues,
    // operator<<, +, +=) multiplies them out first.  Results are identical either way; a
    // 10^9-block chain that is only ever decrypted never touches 160 GB of HBM.
    static void setLazyProducts(bool lazy);
    static bool getLazyProducts();
    // Fused products (ON by default; CSGN_FUSED_PRODUCTS=0 or setFusedProducts(false) gives one kernel per operator,
    // as in the first release).  The reference's callers multiply and then decrypt (tests/basic_operations.cpp:35-40:
    // `c = a * b; sk.decrypt(c)`).  With fused products operator* / *= only note their operands; the product is
    // written by the first operation that needs its words -- and when that operation is SecretKey::decrypt, ONE
    // kernel writes the product and evaluates the decrypt predicate on the product words while they are in registers
    // (csgn_mul_decrypt_deferred): one pass over HBM instead of a write and a read.  The product is kept, so
    // anything that follows (getValues, +, applyPermutation, another decrypt) sees the same words as before.
    static void setFusedProducts(bool fused);
    static bool getFusedProducts();
    // Automatic lanes (ON by default in this API; CSGN_AUTO_LANES=0 or setAutoLanes(false) keeps one stream).  A loop
    // over operator* / decrypt of independent ciphertexts is spread over the engine's internal streams, so that the
    // tail of one kernel overlaps the ramp of the next (csgn_set_auto_lanes); operations that touch the same
    // ciphertext stay ordered.  Together with the deferred Plaintext below this gives plain reference-style code the
    // overlap that the batch entry points give.
    static void setAutoLanes(bool on);
    static bool getAutoLanes();
    // Zero-copy sums (ON by default; CSGN_ROPE_SUMS=0 or setRopeSums(false) copies both operands, as the first release
    // did).  operator+ of two large ciphertexts returns a ciphertext that REFERS to the operands' device storage
    // instead of copying 2 x their size (csgn_concat_lazy): decrypt, applyPermutation and a product with the sum on
    // the left walk the parts; anything that needs one array (getValues, a product with the sum on the right, save)
    // makes it dense once.  Small operands are copied -- a loop of `acc = acc + fresh` stays one array.
    static void setRopeSums(bool on);
    static bool getRopeSums();
    // Multi-GPU, one process per GPU (SURVEY.md 8e).  connectPeers joins the `world` processes of a job: every
    // rank publishes the handle of its mailbox under rendezvous_dir (csgn_comm_connect_dir; `job_tag` unique per
    // job) and maps the others' over NVLink.  initializeLibrary() does this by itself when the launcher exports
    // WORLD_SIZE, RANK, LOCAL_RANK and CSGN_RENDEZVOUS_DIR (optionally CSGN_JOB_TAG; default: MASTER_PORT).
    // Afterwards Ciphertext::shard() keeps this rank's block range of a replicated ciphertext, products with a
    // replicated right operand stay shard-local, and SecretKey::decrypt of a sharded ciphertext returns the
    // GLOBAL bit on every rank (the fold kernel exchanges the counts itself).  Every rank must run the same
    // sequence of sharded decrypts.
    static void connectPeers(int rank, int world, const std::string &rendezvous_dir, const std::string &job_tag);
    static int getRank();
    static int getWorldSize();
};

class Helper {
    Helper() {}

public:
    static bool exists(const uint64_t *v, const uint64_t len, const uint64_t value);
    static void deletePointer(void *pointer, bool isArray);
};

// ---- Context (reference src/Context.h:15-73) ----------------------------------------
class Context {
    uint64_t N, D, S, defaultLen;

public:
    Context() = delete;
    Context(const Context &context);
    Context(const uint64_t pN, const uint64_t pD);
    virtual ~Context();
    Context &operator=(const Context &context);
    friend ostream &operator<<(ostream &out, const Context &c);

    uint64_t getN() const;
    uint64_t getD() const;
    uint64_t getS() const;
    uint64_t getDefaultN() const;  // words per block
    void setN(uint64_t n);
    void setD(uint64_t d);
};

// ---- Plaintext (reference src/Plaintext.h:14-46) --------------------------------------
class Plaintext {
    mutable unsigned char value;
    // SecretKey::decrypt returns at once: the fold and the copy of its count are enqueued on the GPU and the value is
    // read when somebody asks for it (getValue, operator<<).  A loop of decrypts therefore costs one host
    // synchronisation at the first read instead of one per ciphertext.  Copies share the pending result.
    mutable std::shared_ptr<csgn_result> pending;
    void resolve() const;
    friend class SecretKey;

public:
    Plaintext();
    Plaintext(const int value);
    virtual ~Plaintext();
    unsigned char getValue() const;
    void setValue(unsigned char value);
    friend ostream &operator<<(ostream &out, const Plaintext &c);
};

// ---- Permutation (reference src/Permutation.h:15-90) ----------------------------------
class Permutation {
    uint64_t *permutation;
    uint64_t length;
    mutable csgn_perm *device_map;  // bit-source map on the GPU, built on first use

    void drop_device_map() const;

public:
    Permutation();
    Permutation(const uint64_t *perm, const uint64_t len);
    Permutation(const Context &context);  // random, N entries
    Permutation(const uint64_t len);      // random, rand() order of src/Permutation.cpp:139-157
    Permutation(const Permutation &perm);
    virtual ~Permutation();

    uint64_t getLength() const;
    void setLength(uint64_t len);
    void setPermutation(uint64_t *perm, uint64_t len);
    uint64_t *getPermutation() const;  // internal array: do not delete

    friend ostream &operator<<(ostream &out, const Permutation &c);
    Permutation &operator=(const Permutation &perm);
    Permutation getInverse();
    Permutation operator+(const Permutation &permB) const;  // (this o permB)[i] = this[permB[i]]
    Permutation &operator+=(const Permutation &permB);

    // Extension: binary file (64-byte header + the entries, checksummed; csgn_perm_entries_save / _load).
    void save(const std::string &path) const;
    static Permutation load(const std::string &path);

    // engine side
    csgn_perm *deviceMap(uint64_t N) const;
};

// ---- Ciphertext (reference src/Ciphertext.h:15-144) -----------------------------------
class Ciphertext {
    // Device-resident blocks.  Buffers are immutable once shared, so copies share them
    // (the reference deep-copies on every by-value return); += clones first if shared.
    mutable std::shared_ptr<csgn_buf> dev;
    // Non-empty: the value is the product of these buffers, not written yet (fused mode: exactly two, written by the
    // first operation that needs the words; lazy mode: any number, never written by decrypt / applyPermutation).
    mutable std::vector<std::shared_ptr<csgn_buf> > factors;
    // Shared by the copies of one pending product: whichever copy writes the product first leaves it here, the
    // others pick it up instead of multiplying again.
    mutable std::shared_ptr<std::shared_ptr<csgn_buf> > product_slot;
    Context *certFHEcontext;   // context of encryption (null for a default-constructed object)
    mutable uint64_t *host_v;  // host mirror of the words / host staging before upload
    mutable uint64_t *host_bitlen;
    mutable uint64_t host_len; // length of the mirrors, in words
    mutable bool host_v_valid;
    bool staged;               // words exist only in host_v (no context yet / not uploadable)
    bool sharded;              // holds only this rank's block range of a ciphertext spread over the job's GPUs

    void invalidate_mirror() const;
    void release();
    void upload_staged();
    void materialize() const;  // multiply pending factors out into `dev`
    // the same, with the decrypt fold of the product done by the kernel that writes it; returns the pending count
    csgn_result *materialize_and_fold(const csgn_key *key, int *status) const;
    void collect_factors(std::vector<std::shared_ptr<csgn_buf> > &into, bool flatten) const;
    bool adopt_written_product() const;  // a copy has already written the pending product: take it
    friend class SecretKey;
    friend class CiphertextArray;

public:
    Ciphertext();
    Ciphertext(const uint64_t *V, const uint64_t *Bitlen, const uint64_t len, const Context &context);
    Ciphertext(const Ciphertext &ctxt);
    Ciphertext(Ciphertext &&ctxt) noexcept;
    virtual ~Ciphertext();

    void setValues(const uint64_t *V, const uint64_t length);
    void setBitlen(const uint64_t *Bitlen, const uint64_t length);
    void setContext(const Context &context);
    uint64_t getLen() const;  // in 64-bit words, as the reference counts
    Context getContext() const;
    uint64_t *getValues() const;  // host mirror: do not delete; refreshed after every mutation
    uint64_t *getBitlen() const;  // host mirror of the synthesised pattern: do not delete

    friend ostream &operator<<(ostream &out, const Ciphertext &c);

    Ciphertext operator+(const Ciphertext &c) const;
    Ciphertext &operator+=(const Ciphertext &c);
    Ciphertext operator*(const Ciphertext &c) const;
    Ciphertext &operator*=(const Ciphertext &c);
    Ciphertext &operator=(const Ciphertext &c);
    Ciphertext &operator=(Ciphertext &&c) noexcept;

    void applyPermutation_inplace(const Permutation &permutation);
    Ciphertext applyPermutation(const Permutation &permutation);
    long size();

    // engine side (extensions)
    // Binary file: 64-byte header (N, D, L, blocks, checksum) + raw words, streamed GPU <-> file
    // through pinned staging (csgn_buf_save / csgn_buf_load).  The reference has no serialisation.
    void save(const std::string &path) const;
    static Ciphertext load(const std::string &path);
    // The blocks with at least D set bits, in order (csgn_seg_mul_sum_compact): no key of the context can satisfy
    // the others, so the satisfied-block count is the same under every key.  A pending product or lazy sum is made
    // dense first; an empty ciphertext stays empty.
    Ciphertext compact() const;
    // The first occurrence, in order, of every block value that occurs an odd number of times (csgn_seg_cancel): equal
    // blocks are satisfied by the same keys, so the decryption is unchanged under every key, while the satisfied-block
    // count changes by an even number (unlike compact()).  x*x cancels to x.  A pending product or lazy sum is made
    // dense first; an empty ciphertext stays empty.
    Ciphertext cancel() const;
    // A sharded ciphertext as one file per rank, `<prefix>.shard<rank>of<world>` (csgn_buf_save_shard): every rank
    // writes / reads its own blocks, no collective.  loadSharded returns a ciphertext marked sharded.
    void saveSharded(const std::string &prefix) const;
    static Ciphertext loadSharded(const std::string &prefix);
    // This rank's contiguous block range (csgn_shard_range) of a ciphertext that every rank holds in full.
    // The result is marked sharded: * with a replicated right operand, applyPermutation and + of two sharded
    // ciphertexts stay shard-local; getValues()/getLen()/operator<< see the local blocks only.
    Ciphertext shard() const;
    bool isSharded() const;
    uint64_t getBlocks() const;            // number of N-bit blocks
    const csgn_buf *deviceBuffer() const;  // uploads staged words first
};

// ---- SecretKey (reference src/SecretKey.h:18-147) ---------------------------------------
class SecretKey {
    uint64_t *s;  // secret positions in [0, N)
    long length;
    Context *certFHEContext;
    mutable csgn_key *device_key;  // position mask on the GPU, built on first decrypt

    void drop_device_key() const;
    uint64_t *encrypt(unsigned char bit, uint64_t n, uint64_t d, uint64_t *s);

public:
    SecretKey() = delete;
    SecretKey(const Context &context);
    SecretKey(const SecretKey &secKey);
    virtual ~SecretKey();

    Ciphertext encrypt(Plaintext &plaintext);
    Plaintext decrypt(Ciphertext &ciphertext);
    // Extension: n fresh encryptions built on the GPU in one call (csgn_encrypt_batch) -- the
    // ciphertext Enc(bits[0]) + ... + Enc(bits[n-1]), n blocks, decrypting to the XOR of the bits.
    // Same construction as encrypt(); randomness is Philox keyed by `seed` instead of rand().
    Ciphertext encryptBatch(const unsigned char *bits, uint64_t n, uint64_t seed);
    // Extension: decrypt n ciphertexts with ONE synchronisation (csgn_decrypt_batch: the folds are spread over
    // the library's lanes and overlap); bits[i] = decrypt(ciphertexts[i]).getValue().
    void decryptBatch(Ciphertext *ciphertexts, uint64_t n, unsigned char *bits);
    // Extension: n fresh one-block encryptions as a CiphertextArray of n elements (csgn_encrypt_batch), and the
    // decryption of every element of an array with one launch and one synchronisation (csgn_seg_decrypt).
    CiphertextArray encryptArray(const unsigned char *bits, uint64_t n, uint64_t seed);
    void decryptArray(const CiphertextArray &array, unsigned char *bits);
    // Extension: n integers of `width` bits (1..64) as an EncryptedUInt, one launch (csgn_encrypt_uint); throws Error
    // on a value that does not fit.  decryptUInt writes x.size() values with one launch and one synchronisation
    // (csgn_decrypt_uint).
    EncryptedUInt encryptUInt(const uint64_t *values, uint64_t n, uint32_t width, uint64_t seed);
    void decryptUInt(const EncryptedUInt &x, uint64_t *values);
    void applyPermutation_inplace(const Permutation &permutation);
    SecretKey applyPermutation(const Permutation &permutation);

    friend ostream &operator<<(ostream &out, const SecretKey &c);
    SecretKey &operator=(const SecretKey &secKey);

    uint64_t getLength() const;
    uint64_t *getKey() const;  // internal array: do not delete
    void setKey(uint64_t *s, uint64_t len);
    long size();

    // Extension: binary file (64-byte header with N, D + the secret positions, checksummed;
    // csgn_key_positions_save / _load).  The file holds the secret: protect it like the key.
    void save(const std::string &path) const;
    static SecretKey load(const std::string &path);
};

// ---- CiphertextArray (extension; include/csgn.h, "ciphertext arrays") ----------------------------------------------
// n independent ciphertexts -- the encrypted bits of a circuit over encrypted integers, say -- held as ONE device buffer
// plus block offsets: element k is blocks [offsets[k], offsets[k+1]).  operator*, operator+, gather and
// applyPermutation act element by element with one kernel launch for all small elements, where a loop over
// Ciphertext operators costs one launch and its host bookkeeping per element.  Arrays are always evaluated eagerly:
// the fused, lazy and rope modes of Ciphertext do not apply to them.
class CiphertextArray {
    std::shared_ptr<csgn_buf> storage;
    std::vector<uint64_t> offsets;   // n + 1 block offsets
    Context context;
    CiphertextArray(csgn_buf *storage, const std::vector<uint64_t> &offsets, const Context &context);
    static CiphertextArray gate(const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products,
                                const std::vector<CiphertextArray> &terms, bool compact);
    friend class SecretKey;
    friend class Circuit;
    friend class UIntCircuit;

public:
    // Packs the ciphertexts into one array with one launch (csgn_concat_n); pending products and lazy sums are
    // written first.  Sharded ciphertexts are refused.
    explicit CiphertextArray(const std::vector<Ciphertext> &elements);

    uint64_t size() const;                 // number of elements
    uint64_t getBlocks(uint64_t k) const;  // blocks of element k
    Ciphertext get(uint64_t k) const;      // element k as an ordinary Ciphertext (a device copy of its blocks)
    Context getContext() const;

    CiphertextArray operator*(const CiphertextArray &c) const;   // element k = this_k * c_k
    CiphertextArray operator+(const CiphertextArray &c) const;   // element k = this_k + c_k
    CiphertextArray gather(const std::vector<uint64_t> &idx) const;   // element j = this_{idx[j]}
    CiphertextArray applyPermutation(const Permutation &permutation) const;   // every element permuted
    // element k = A0_k*B0_k + A1_k*B1_k + ... + C0_k + ... (csgn_seg_mul_sum): one gate of a circuit -- carry,
    // majority, multiplexer -- in one call, every output word written once.  Throws Error on arrays of different sizes
    // or contexts, or when both lists are empty.
    static CiphertextArray sumOfProducts(const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products,
                                         const std::vector<CiphertextArray> &terms = {});
    // sumOfProducts keeping only the blocks with at least D set bits (csgn_seg_mul_sum_compact, min_bits = D of the
    // context): no key of the context can satisfy the others, so every element decrypts as before, with the same
    // satisfied-block count, under every key.  Throws as sumOfProducts does.  compact() drops them from this array.
    static CiphertextArray compactSumOfProducts(
        const std::vector<std::pair<CiphertextArray, CiphertextArray>> &products,
        const std::vector<CiphertextArray> &terms = {});
    CiphertextArray compact() const;
    // Every element reduced to the first occurrence, in order, of each block value that occurs an odd number of times
    // in it (csgn_seg_cancel): x*x -> x, a + a -> empty.  Every element decrypts as before under every key; its
    // satisfied-block count changes by an even number.  The usual gate is compactSumOfProducts(...).cancel().
    CiphertextArray cancel() const;

    const std::vector<uint64_t> &getOffsets() const;
    const csgn_buf *deviceBuffer() const;
};

// ---- Circuit (extension; include/csgn.h, "circuits") ----------------------------------------------------------------
// A netlist of gates over CiphertextArrays, evaluated over every lane in one call (csgn_seg_circuit) instead of one
// call per gate.  Wires 0 .. inputs - 1 are the inputs; gate() adds sum(u*v) + sum(terms) over earlier wires and
// returns its wire.  Throws Error on a gate with no operands or an operand that is not an earlier wire.
class Circuit {
    uint32_t inputs, gates = 0;
    std::vector<uint32_t> netlist;   // per gate: p, q, the p operand pairs, the q terms
    uint64_t fallback = 0;

public:
    explicit Circuit(uint32_t inputs);
    uint32_t gate(const std::vector<std::pair<uint32_t, uint32_t>> &products, const std::vector<uint32_t> &terms = {});
    // The arrays of wires `outputs` over the lanes of `inputs` (one array per input wire, all of the same size and
    // context): each gate compacted to minBits set bits (-1: D of the context; 0: no compaction) and, with cancel,
    // cancelled, as compactSumOfProducts(...).cancel() would give.  laneCapacity: blocks per lane on the device (0: the
    // library chooses).  Throws Error on mismatched sizes or contexts, or a bad output wire.
    std::vector<CiphertextArray> evaluate(const std::vector<CiphertextArray> &inputs,
                                          const std::vector<uint32_t> &outputs, int64_t minBits = -1,
                                          bool cancel = false, uint64_t laneCapacity = 0);
    uint64_t lastFallback() const { return fallback; }   // lanes of the last evaluate() evaluated gate by gate
    uint32_t wires() const { return inputs + gates; }
    uint32_t inputCount() const { return inputs; }
    const std::vector<uint32_t> &getNetlist() const { return netlist; }
};

// ---- encrypted integers (extension; include/csgn.h, "encrypted integers") ------------------------------------------
// A vector of n encrypted W-bit unsigned integers: W CiphertextArrays of n elements, its bit planes, LSB first.  The
// operators + - * (mod 2^W), < > (1-bit results) and & ^ | build a one-operation UIntCircuit and make one call, compacted
// and cancelled; operands may differ in width (the shorter is zero-extended).  Throws Error on arrays of different sizes or contexts.
class EncryptedUInt {
    std::vector<CiphertextArray> planes;

public:
    explicit EncryptedUInt(const std::vector<CiphertextArray> &planes);
    uint32_t width() const { return (uint32_t)planes.size(); }
    uint64_t size() const { return planes[0].size(); }
    const std::vector<CiphertextArray> &getPlanes() const { return planes; }
    Context getContext() const { return planes[0].getContext(); }

    EncryptedUInt operator+(const EncryptedUInt &b) const;
    EncryptedUInt operator-(const EncryptedUInt &b) const;
    EncryptedUInt operator*(const EncryptedUInt &b) const;
    EncryptedUInt operator<(const EncryptedUInt &b) const;
    EncryptedUInt operator>(const EncryptedUInt &b) const;
    EncryptedUInt operator&(const EncryptedUInt &b) const;
    EncryptedUInt operator^(const EncryptedUInt &b) const;
    EncryptedUInt operator|(const EncryptedUInt &b) const;
    // c ? x : y lane by lane (c of 1 bit)
    static EncryptedUInt select(const EncryptedUInt &c, const EncryptedUInt &x, const EncryptedUInt &y);
};

// Integer netlists, built on the host and evaluated as ONE Circuit call; the netlists of the Python UIntCircuit,
// wire for wire.  An integer is a vector of wires, LSB first.  Wires: operand i, bit j is input i*width + j; then the
// `one` input (one = true: the caller passes an encryption of 1 per lane to evaluate); then the zero input (n empty
// elements, supplied by evaluate).  Every operation is a sum of products plus terms; a gate that folds to one wire
// (x + 0, x*1, a single term) adds no gate.  eq, le, ge and invert need `one` and throw Error without it.  Cancelled
// results hold the blocks of their function's algebraic normal form: small for add, bitwise, select and shifts at any
// width, about threefold per bit for sub, neg, comparisons, min, max and mul (practical up to about 8-12 bits).
class UIntCircuit {
public:
    typedef std::vector<uint32_t> UInt;

    UIntCircuit(uint32_t width, uint32_t operands, bool one = false);
    const std::vector<UInt> &inputs() const { return in; }
    uint32_t width() const { return w; }
    const Circuit &circuit() const { return c; }
    uint64_t lastFallback() const { return c.lastFallback(); }

    UInt add(const UInt &a, const UInt &b);
    UInt sub(const UInt &a, const UInt &b);
    UInt neg(const UInt &a);
    UInt lt(const UInt &a, const UInt &b);
    UInt gt(const UInt &a, const UInt &b);
    UInt ne(const UInt &a, const UInt &b);
    UInt eq(const UInt &a, const UInt &b);
    UInt le(const UInt &a, const UInt &b);
    UInt ge(const UInt &a, const UInt &b);
    UInt invert(const UInt &a);
    UInt select(const UInt &s, const UInt &x, const UInt &y);
    UInt min(const UInt &a, const UInt &b);
    UInt max(const UInt &a, const UInt &b);
    UInt mul(const UInt &a, const UInt &b);
    UInt and_(const UInt &a, const UInt &b);
    UInt xor_(const UInt &a, const UInt &b);
    UInt or_(const UInt &a, const UInt &b);
    UInt shl(const UInt &a, uint32_t k);
    UInt shr(const UInt &a, uint32_t k);

    // One csgn_seg_circuit call for every result.  operands: one EncryptedUInt per operand, of at most width() bits;
    // one: the array that encrypts 1 in every lane, for a circuit built with one = true (null otherwise).
    std::vector<EncryptedUInt> evaluate(const std::vector<EncryptedUInt> &operands, const std::vector<UInt> &results,
                                        int64_t minBits = -1, bool cancel = false, uint64_t laneCapacity = 0,
                                        const CiphertextArray *one = nullptr);

private:
    uint32_t w, operands;
    bool has_one;
    uint32_t one_w, zero_w;
    std::vector<UInt> in;
    Circuit c;

    uint32_t gate(std::vector<std::pair<uint32_t, uint32_t>> products, std::vector<uint32_t> terms);
    uint32_t notw(uint32_t x);
    uint32_t borrow(uint32_t a, uint32_t b, uint32_t r, uint32_t t);
    void pair(UInt &a, UInt &b) const;
};

// ---- Timer (reference src/Timer.h:13-74) -------------------------------------------------
class Timer {
    string name;
    std::chrono::duration<double> chronometer;
    std::chrono::high_resolution_clock::time_point start_fingerprint;
    std::chrono::high_resolution_clock::time_point stop_fingerprint;

public:
    Timer(string name = "Default timer");
    virtual ~Timer();
    void start();
    double stop();          // milliseconds
    void reset();
    double stopAndPrint();
    void print();
    double getValue();
};

}  // namespace certFHE

#endif  // CSGN_CERTFHE_API_H_
