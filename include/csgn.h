/*
 * csgn.h -- C ABI of the B200-native CSGN / certFHE ciphertext evaluation engine.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.
 * It sits exactly on the raw-pointer seam the reference already has -- the private
 * member functions of Ciphertext / SecretKey that take `uint64_t*` + lengths
 * (reference src/Ciphertext.h:34,43,58 and src/SecretKey.h:47,60).  The certFHE C++
 * classes of this repository (csgn_b200/certfhe/) call nothing else; a maintainer
 * of the reference would bind the same entry points from src/Ciphertext.cpp and
 * src/SecretKey.cpp (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every function returns CSGN_OK (0) or a negative csgn_status; the message of
 *     the last failure on the calling thread is csgn_last_error();
 *   - there is no CPU fallback: without a usable sm_100 device every call fails;
 *   - a "block" is one N-bit ciphertext unit stored as L = ceil(N/64) uint64 words,
 *     bits MSB-first (position p -> word p>>6, bit 63-(p&63)); a ciphertext is a
 *     dense array of n_blocks*L words; the reference's `bitlen` side array is the
 *     fixed pattern [64]*(L-1)+[N%64] and is never materialised on the device;
 *   - `csgn_buf` handles own device memory, are created and freed only here, and
 *     belong to the process' bound device (one process per GPU);
 *   - work is enqueued on the current stream (csgn_set_stream); calls that return data to
 *     the host (download, decrypt) synchronise that stream, the others do not.  A caller may
 *     move between streams from call to call to overlap independent ciphertexts: operations
 *     on one buffer must then be ordered by the caller (same stream or events), as with any
 *     CUDA library; freeing a buffer is always safe -- the library orders the release after
 *     the stream that used it last.
 */
#ifndef CSGN_H_
#define CSGN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum csgn_status {
    CSGN_OK = 0,
    CSGN_ERR_NOT_INITIALIZED = -1,
    CSGN_ERR_INVALID_ARGUMENT = -2,
    CSGN_ERR_CUDA = -3,
    CSGN_ERR_NO_DEVICE = -4,
    CSGN_ERR_SHAPE_MISMATCH = -5,
    CSGN_ERR_OUT_OF_MEMORY = -6,
    CSGN_ERR_TIMEOUT = -7
} csgn_status;

typedef struct csgn_buf csgn_buf;   /* device-resident ciphertext words            */
typedef struct csgn_key csgn_key;   /* secret positions as a device position mask  */
typedef struct csgn_perm csgn_perm; /* permutation as a device bit-source map      */

/* ---- library ------------------------------------------------------------- */

/* One-time initialisation; the CUDA half of Library::initializeLibrary
 * (src/Helpers.cpp:8-12).  Binds the process to `device` (-1: LOCAL_RANK env or 0),
 * creates the work stream and the memory pool.  Idempotent for the same device. */
int csgn_init(int device);
int csgn_shutdown(void);
int csgn_is_initialized(void);
const char *csgn_last_error(void);
const char *csgn_version(void);
/* SM count, total/free HBM bytes, compute capability (major*10+minor). */
int csgn_device_info(int *sm_count, uint64_t *hbm_total, uint64_t *hbm_free, int *cc);
/* Use an external cudaStream_t (e.g. torch's current stream); NULL restores the
 * library's own stream. */
int csgn_set_stream(void *cuda_stream);
void *csgn_get_stream(void);
/* Automatic lanes (off by default; CSGN_AUTO_LANES=1 or Library::setAutoLanes in C++).  The reference's API has no
 * batch calls: a user writes a loop over Ciphertext::operator* (src/Ciphertext.cpp:231-247) and SecretKey::decrypt
 * (src/SecretKey.cpp:208-224).  With automatic lanes the library itself places consecutive INDEPENDENT operations
 * (csgn_mul, csgn_mul_into / csgn_permute_into with a library-owned output, csgn_concat, csgn_append, csgn_permute,
 * csgn_buf_clone / _slice, csgn_decrypt_deferred, csgn_mul_decrypt_deferred) on alternating internal streams, so
 * that the tail of one kernel overlaps the ramp of the next; operations that depend on each other through a buffer
 * are ordered by per-buffer last-writer / reader tracking and stay on one stream.  Calls that hand device memory to
 * the caller (csgn_buf_device_ptr, *_async with a caller-owned destination) run on, or are joined into, the current
 * stream, and csgn_sync waits for the lanes as well. */
int csgn_set_auto_lanes(int on);
int csgn_get_auto_lanes(void);
int csgn_sync(void);
/* Kernels launched by this library since csgn_init (for bench.py's gpu_launches). */
uint64_t csgn_launch_count(void);

/* Block geometry of Context(N,D): src/Context.cpp:20-29. */
uint32_t csgn_words_per_block(uint64_t N);

/* Pinned host staging memory for uploads/downloads that should overlap compute. */
int csgn_host_alloc(size_t bytes, void **out);
int csgn_host_free(void *p);

/* ---- ciphertext buffers (storage behind certFHE::Ciphertext, src/Ciphertext.h:17-21) */

/* Deep-copies n_blocks*L host words to the device: the Ciphertext(V,Bitlen,len,ctx)
 * constructor / setValues (src/Ciphertext.cpp:344-358, :392-403).  Asynchronous: `host_words` (ideally pinned) must
 * stay valid and unchanged until the copy has run (csgn_sync, or any blocking call on a consumer of the buffer). */
int csgn_buf_upload(const uint64_t *host_words, uint64_t n_blocks, uint32_t L, csgn_buf **out);
/* The same with the reference constructor's ownership contract and no synchronisation: the words are copied into
 * library-owned pinned staging by the host before the call returns (the caller may free or overwrite its array at
 * once), and travel to the device from there, asynchronously.  Uploads beyond 64 MB copy straight from the caller's
 * memory and wait. */
int csgn_buf_upload_copy(const uint64_t *host_words, uint64_t n_blocks, uint32_t L, csgn_buf **out);
/* n uploads in one call (the operands of a batch of products): one device allocation shared by the n buffers, the
 * copies issued back to back (operands adjacent in host memory travel as one copy), one ordering event per consuming
 * stream instead of one per operand.  host_words[i]
 * (ideally pinned) holds n_blocks[i]*L words and must stay valid until the copies have run, as for csgn_buf_upload.
 * out[0..n) are ordinary read-only operands (not growable by csgn_append); the shared storage is released when the
 * last of them is freed.  csgn_buf_free_batch frees n handles in one call. */
int csgn_buf_upload_batch(const uint64_t *const *host_words, const uint64_t *n_blocks, uint32_t n, uint32_t L,
                          csgn_buf **out);
int csgn_buf_free_batch(csgn_buf *const *bufs, uint32_t n);
/* Uninitialised device storage for n_blocks blocks. */
int csgn_buf_alloc(uint64_t n_blocks, uint32_t L, csgn_buf **out);
/* Non-owning view over caller-owned device memory (e.g. a torch tensor). */
int csgn_buf_wrap(void *device_words, uint64_t n_blocks, uint32_t L, csgn_buf **out);
/* Device-to-device deep copy: the copy constructor / operator= (src/Ciphertext.cpp:306-363). */
int csgn_buf_clone(const csgn_buf *src, csgn_buf **out);
/* getValues() (src/Ciphertext.cpp:422-425): all words, or a block range, to the host. */
int csgn_buf_download(const csgn_buf *buf, uint64_t *host_words);
int csgn_buf_download_range(const csgn_buf *buf, uint64_t first_block, uint64_t n_blocks,
                            uint64_t *host_words);
/* Device-to-device copy of the block range [first_block, first_block + n_blocks): the shard of a replicated
 * ciphertext that one rank keeps (with csgn_shard_range). */
int csgn_buf_slice(const csgn_buf *src, uint64_t first_block, uint64_t n_blocks, csgn_buf **out);
int csgn_buf_free(csgn_buf *buf);
uint64_t csgn_buf_blocks(const csgn_buf *buf);
uint32_t csgn_buf_words_per_block(const csgn_buf *buf);
void *csgn_buf_device_ptr(const csgn_buf *buf);

/* ---- the hot path -------------------------------------------------------- */

/* Ciphertext::multiply (src/Ciphertext.cpp:133-179, :124-131):
 *   out[(i*T2+j)*L+k] = a[i*L+k] & b[j*L+k],  T1*T2 blocks, i-major.
 * csgn_mul allocates the result; csgn_mul_into writes into a buffer of exactly
 * T1*T2 blocks (a view from csgn_buf_wrap included). */
int csgn_mul(const csgn_buf *a, const csgn_buf *b, csgn_buf **out);
int csgn_mul_into(const csgn_buf *a, const csgn_buf *b, csgn_buf *out);

/* Ciphertext::add / operator+ (src/Ciphertext.cpp:107-122, :204-229): out = a || b. */
int csgn_concat(const csgn_buf *a, const csgn_buf *b, csgn_buf **out);
/* operator+= (src/Ciphertext.cpp:249-281): a = a || b, growing a's storage
 * geometrically so that a chain of += copies each block O(1) times. */
int csgn_append(csgn_buf *a, const csgn_buf *b);
/* The same sum WITHOUT moving a word (SURVEY.md 8f-1, "add as a zero-copy rope"): the result refers to the storage of
 * a and b -- each kept alive by a reference, so the caller may free its own handles at once -- and is one logical
 * ciphertext of a.blocks + b.blocks blocks.  decrypt folds segment by segment and sums the counts, permute and a
 * product with the sum as LEFT operand ((A1||A2)*B = (A1*B)||(A2*B)) write each segment's share straight into the
 * dense result; everything else (download, right operand, save, csgn_buf_device_ptr ...) first makes it one dense
 * array, once, inside the library (csgn_buf_flatten does it by hand).  Operands below 1 MiB, and sums that would
 * exceed 32 segments, are copied as by csgn_concat.  A buffer that a lazy sum refers to (csgn_buf_retained) cannot be
 * grown or overwritten in place: csgn_append / *_into refuse it; clone it first. */
int csgn_concat_lazy(const csgn_buf *a, const csgn_buf *b, csgn_buf **out);
int csgn_buf_segments(const csgn_buf *buf);   /* 1 for a dense buffer */
int csgn_buf_retained(const csgn_buf *buf);   /* 1 while some lazy sum refers to it */
int csgn_buf_flatten(csgn_buf *buf);

/* Secret key as the per-word position mask M[s>>6] |= 1<<(63-(s&63)); the block
 * predicate of SecretKey::decrypt (src/SecretKey.cpp:131-137) is all_w((v&M)==M). */
int csgn_key_create(uint64_t N, const uint64_t *positions, uint32_t D, csgn_key **out);
int csgn_key_free(csgn_key *key);

/* SecretKey::decrypt (src/SecretKey.cpp:104-147, :208-224): XOR over blocks of the
 * AND of the D secret bits.  *bit receives 0/1.  An empty buffer decrypts to 0. */
int csgn_decrypt(const csgn_buf *c, const csgn_key *key, uint8_t *bit);
/* Number of blocks whose secret bits are all one (decrypt = count & 1).  This is
 * the per-shard partial a multi-GPU decrypt all-reduces (sum, then & 1). */
int csgn_decrypt_count(const csgn_buf *c, const csgn_key *key, uint64_t *count);
/* Same, asynchronous: the count is written to a device uint64 (caller-owned, e.g.
 * the tensor handed to the NCCL all-reduce); no host synchronisation. */
int csgn_decrypt_count_async(const csgn_buf *c, const csgn_key *key, uint64_t *device_count);
/* Decrypt of a product that is never materialised (SURVEY.md 8f, the caller side of the path:
 * operator* followed by decrypt).  For raw blocks the satisfied-block count is multiplicative,
 * count(f1*f2*...*fn) = count(f1)*...*count(fn), because block (i,j) of a product is a_i & b_j and
 * (a_i & b_j) & M == M  <=>  a_i & M == M and b_j & M == M; so Dec(f1*...*fn) is the AND of the factors'
 * decryptions.  Folds the n factors (n launches, one synchronisation); *bit receives the plaintext bit,
 * *count (optional) the product of the counts, saturated at UINT64_MAX. */
int csgn_decrypt_product(const csgn_buf *const *factors, uint32_t n_factors, const csgn_key *key, uint8_t *bit,
                         uint64_t *count);
/* A decrypt whose result the host reads later: the fold and the device-to-host copy of its count are enqueued and the
 * call returns at once; csgn_result_wait blocks until the count has landed (and may be called again), csgn_result_ready
 * polls, csgn_result_free releases the slot.  This is what lets a loop over SecretKey::decrypt run without one host
 * synchronisation per ciphertext -- certFHE::Plaintext resolves its value on first use (csgn_b200/certfhe). */
typedef struct csgn_result csgn_result;
int csgn_decrypt_deferred(const csgn_buf *c, const csgn_key *key, csgn_result **out);
int csgn_result_ready(const csgn_result *r);
int csgn_result_wait(csgn_result *r, uint64_t *count);
int csgn_result_free(csgn_result *r);

/* ---- fused multiply -> decrypt (SURVEY.md 8f-1; the caller pattern tests/basic_operations.cpp:35-40: operator*, then
 * SecretKey::decrypt of the product).  ONE kernel writes the product a*b (src/Ciphertext.cpp:153-163) and evaluates
 * the decrypt predicate (src/SecretKey.cpp:131-140) on the product words while they are still in registers: one pass
 * over HBM (the product is written, never read back) instead of two.
 * The `out` convention of every entry point below:  out == NULL  -> count only, nothing is stored (decrypt-only
 * consumers);  *out == NULL -> the product is allocated by the library and returned in *out;  otherwise the product
 * is written into *out, which must hold exactly T1*T2 blocks (a view from csgn_buf_wrap included).
 * The count of satisfied product blocks goes to a device uint64 (decrypt = count & 1); no host synchronisation. */
int csgn_mul_count_async(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **out, uint64_t *device_count);
/* Blocking convenience: *bit = Dec(a*b), *count (optional) the satisfied-block count. */
int csgn_mul_decrypt(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **out, uint8_t *bit,
                     uint64_t *count);
/* n independent pairs in one call, spread over the library's lanes (see "batches" below); out may be NULL (count only)
 * or an array of n handles following the convention above entry by entry. */
int csgn_mul_count_batch_async(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, const csgn_key *key,
                               csgn_buf **out, uint64_t *device_counts);
/* Deferred form (see csgn_decrypt_deferred); `prod` follows the `out` convention. */
int csgn_mul_decrypt_deferred(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **prod,
                              csgn_result **out);

/* ---- batches of independent items -------------------------------------------------------------
 * n independent products / folds in ONE call: what a caller of the reference writes as a loop over
 * Ciphertext::operator* (src/Ciphertext.cpp:231-247) or SecretKey::decrypt (src/SecretKey.cpp:208-224).  The library forks its internal lane streams (CSGN_LANES, default 2)
 * from the current stream, enqueues item i on lane i % lanes and joins them back, so the tail of one kernel
 * overlaps the launch ramp and first-load latency of the next item's: +12 % over n single calls at the
 * 160 MB products of Context(1247,16) 1000x1000 (profiles/README.md).  Ordering seen by the caller is that
 * of one call on the current stream: after everything enqueued before, before everything enqueued after. */
int csgn_mul_batch(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, csgn_buf **out);
int csgn_mul_into_batch(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, csgn_buf *const *out);
/* device_counts[i] = satisfied blocks of c[i]; no host synchronisation. */
int csgn_decrypt_count_batch_async(const csgn_buf *const *c, uint32_t n, const csgn_key *key, uint64_t *device_counts);
/* SecretKey::decrypt of n ciphertexts with one synchronisation: bits[i] (and/or counts[i]) on the host. */
int csgn_decrypt_batch(const csgn_buf *const *c, uint32_t n, const csgn_key *key, uint8_t *bits, uint64_t *counts);

/* One-shot convenience without a key handle. */
int csgn_decrypt_positions(const csgn_buf *c, uint64_t N, const uint64_t *positions, uint32_t D,
                           uint8_t *bit);

/* Batched fresh encryptions on the GPU (SURVEY.md 8f; the reference encrypts one bit per call on the
 * host from glibc rand(), src/SecretKey.cpp:35-80 -- that path, rand() order included, stays in
 * csgn_b200/certfhe for seeded parity).  Block i of *out encrypts bits[i] (host array, 0/1) under
 * `key`, with the reference's construction and Philox-4x32-10 keyed by `seed`, counter
 * (first_block + i, unit): the result does not depend on how a batch is split.  The n-block buffer
 * is the ciphertext Enc(bits[0]) + ... + Enc(bits[n-1]) and decrypts to the XOR of the bits. */
int csgn_encrypt_batch(const csgn_key *key, const uint8_t *bits, uint64_t n, uint64_t first_block, uint64_t seed,
                       csgn_buf **out);

/* ---- ciphertext arrays ---------------------------------------------------------------------------------------
 * A plaintext is one bit, so a circuit over encrypted integers holds thousands of small, independent ciphertexts.  A
 * ciphertext array of n elements is an ordinary dense csgn_buf (the elements' blocks one after another) plus a host
 * array off[n+1] of uint64 BLOCK offsets: element k is blocks [off[k], off[k+1]) (empty elements allowed).  Every
 * existing call works on the storage: csgn_permute permutes every element (offsets unchanged), csgn_buf_slice /
 * csgn_buf_download_range read one element, and the n-block result of csgn_encrypt_batch is an array of n one-block
 * encryptions with off = 0, 1, ..., n.
 * Offsets are checked on the host on every call (off[0] == 0, non-decreasing, off[n] == csgn_buf_blocks(buf);
 * CSGN_ERR_INVALID_ARGUMENT or CSGN_ERR_SHAPE_MISMATCH, nothing allocated) and copied to the device by the library
 * through its pinned staging, without a host synchronisation: the caller may free its arrays when the call returns.
 * Output arrays are allocated by the library; their offsets go to the caller's out_off[n+1] (m+1 for a gather).
 * All small elements are served by ONE kernel launch per call; elements whose product (multiply) or whose blocks
 * (decrypt) reach 8 MB run on the single-ciphertext kernels, one launch each, straight into the output.  Ordering,
 * streams and automatic lanes are those of the single-ciphertext entry points. */
/* element k = a_k * b_k (src/Ciphertext.cpp:153-163): T1_k*T2_k blocks, i-major; empty if either operand is empty. */
int csgn_seg_mul(const csgn_buf *a, const uint64_t *a_off, const csgn_buf *b, const uint64_t *b_off, uint64_t n,
                 uint64_t *out_off, csgn_buf **out);
/* element k = a_k || b_k (src/Ciphertext.cpp:107-122): the element-wise homomorphic XOR. */
int csgn_seg_concat(const csgn_buf *a, const uint64_t *a_off, const csgn_buf *b, const uint64_t *b_off, uint64_t n,
                    uint64_t *out_off, csgn_buf **out);
/* element k = a[0]_k*b[0]_k || ... || a[p-1]_k*b[p-1]_k || c[0]_k || ... || c[q-1]_k   (p = n_products, q = n_terms)
 * the element-wise homomorphic XOR of p ANDs and q plain terms, every output word written once: one gate of a circuit
 * (carry x*y + (x+y)*c, majority x*y + x*z + y*z, multiplexer s*a + s*b + b) in one call and one launch.  The words
 * of element k are those of (a[0]*b[0] + ... ) + c[0] + ... built with csgn_seg_mul and csgn_seg_concat, in that
 * block order; a product is empty when either operand element is empty.  p + q >= 1, every buffer has the same L, and
 * a buffer may appear any number of times (x*x, x*y + x). */
int csgn_seg_mul_sum(const csgn_buf *const *a, const uint64_t *const *a_off, const csgn_buf *const *b,
                     const uint64_t *const *b_off, uint32_t n_products, const csgn_buf *const *c,
                     const uint64_t *const *c_off, uint32_t n_terms, uint64_t n, uint64_t *out_off, csgn_buf **out);
/* csgn_seg_mul_sum with only the blocks that have at least min_bits set bits (min_bits = D of the context: no key can
 * satisfy the others, so every element's satisfied-block count is unchanged under every key).  Element k is the stable
 * subsequence of element k of csgn_seg_mul_sum's result.  n_products = 0 with one term compacts an existing array.
 * The sizes depend on the data: the call returns after the counting pass, like csgn_seg_decrypt.  The checks are
 * those of csgn_seg_mul_sum, plus 1 <= min_bits <= 64*L.  A block's pad bits count (the library leaves them zero);
 * an element with no surviving block is empty. */
int csgn_seg_mul_sum_compact(const csgn_buf *const *a, const uint64_t *const *a_off, const csgn_buf *const *b,
                             const uint64_t *const *b_off, uint32_t n_products, const csgn_buf *const *c,
                             const uint64_t *const *c_off, uint32_t n_terms, uint64_t n, uint32_t min_bits,
                             uint64_t *out_off, csgn_buf **out);
/* element k = the first occurrence, in order, of every block value that occurs an odd number of times in element k.
 * Equal blocks are satisfied by the same keys, so every decryption is unchanged under every key; satisfied-block
 * counts change by an even number.  Sizes depend on the data: the call returns after its counting pass.  Equality is
 * decided on all L words; the result depends on nothing else.  An element may hold at most 2^30 blocks. */
int csgn_seg_cancel(const csgn_buf *c, const uint64_t *c_off, uint64_t n, uint64_t *out_off, csgn_buf **out);
/* element j = src_{idx[j]}, j < m: any order, repeats allowed; idx[j] < n_src is checked. */
int csgn_seg_gather(const csgn_buf *src, const uint64_t *src_off, uint64_t n_src, const uint64_t *idx, uint64_t m,
                    uint64_t *out_off, csgn_buf **out);
/* parts[0] || ... || parts[n-1] in one launch: n separate ciphertexts packed into an array (its offsets are the
 * prefix sums of the parts' block counts). */
int csgn_concat_n(const csgn_buf *const *parts, uint64_t n, csgn_buf **out);
/* device_counts[k] = satisfied blocks of element k (0 for an empty one); no host synchronisation. */
int csgn_seg_decrypt_count_async(const csgn_buf *c, const uint64_t *c_off, uint64_t n, const csgn_key *key,
                                 uint64_t *device_counts);
/* SecretKey::decrypt of every element with one synchronisation: bits[k] = count_k & 1 and/or counts[k]. */
int csgn_seg_decrypt(const csgn_buf *c, const uint64_t *c_off, uint64_t n, const csgn_key *key, uint8_t *bits,
                     uint64_t *counts);

/* Permutation as a device source map: out_bit[i] = in_bit[perm[i]], i < N
 * (src/Ciphertext.cpp:33-34).  Fails unless perm is a bijection of [0,N). */
int csgn_perm_create(uint64_t N, const uint64_t *perm, csgn_perm **out);
int csgn_perm_free(csgn_perm *perm);
/* Ciphertext::applyPermutation (src/Ciphertext.cpp:7-89).  strict_ref_truncate = 0
 * permutes every block (Dec_{pi(k)}(pi(c)) = Dec_k(c) for multi-block c);
 * strict_ref_truncate = 1 reproduces the reference exactly: the result is block 0
 * permuted, one block long (src/Ciphertext.cpp:33-40). Pad bits of the last word
 * come out zero. */
int csgn_permute(const csgn_buf *c, const csgn_perm *perm, int strict_ref_truncate, csgn_buf **out);
int csgn_permute_into(const csgn_buf *c, const csgn_perm *perm, csgn_buf *out);

/* Three order-insensitive/-sensitive folds of all words of a buffer, computed on the
 * device (xor, wrapping sum, and sum of word*(2*index+1) mod 2^64) -- lets tests
 * compare products that are too large to download. */
int csgn_buf_checksum(const csgn_buf *buf, uint64_t *xor_out, uint64_t *sum_out, uint64_t *wsum_out);

/* ---- serialisation (SURVEY.md 8f: absent upstream, which only reports size()) -------------
 * File = 64-byte little-endian header {magic "CSGNCT01", N, D, L, n_blocks, xor-of-words,
 * reserved} followed by n_blocks*L raw uint64 words.  Blocks stream between the device and
 * the file through two pinned staging buffers, so a ciphertext far larger than host memory
 * can be written or read; the checksum is verified on load. */
int csgn_buf_save(const csgn_buf *buf, uint64_t N, uint64_t D, const char *path);
int csgn_buf_load(const char *path, uint64_t *N, uint64_t *D, csgn_buf **out);
/* A ciphertext sharded over the job's GPUs (8e) as one file per rank, `<prefix>.shard<rank>of<world>`: the ordinary
 * file of the rank's local blocks, with the shard's identity and first global block in the header.  No collective:
 * every rank writes / reads its own file; loading checks that the file was written as this rank of this world. */
int csgn_buf_save_shard(const csgn_buf *buf, uint64_t N, uint64_t D, const char *prefix, int rank, int world,
                        uint64_t first_block);
int csgn_buf_load_shard(const char *prefix, int rank, int world, uint64_t *N, uint64_t *D, uint64_t *first_block,
                        csgn_buf **out);
/* SecretKey and Permutation files (SURVEY.md 8f-3 names all three types; upstream has only SecretKey::size(),
 * src/SecretKey.cpp:269-276, and the Permutation state of src/Permutation.cpp:139-171 to persist).  Host only -- no
 * device is touched and csgn_init is not needed.  64-byte header {magic "CSGNSK01" / "CSGNPM01", N, D, count, xor of
 * the entries} + count uint64 entries; positions / entries are validated on save and load.  *_load with a null
 * destination only reports the count (and N, D). */
int csgn_key_positions_save(const char *path, uint64_t N, uint64_t D, const uint64_t *positions, uint64_t n);
int csgn_key_positions_load(const char *path, uint64_t *N, uint64_t *D, uint64_t *positions, uint64_t capacity, uint64_t *n);
int csgn_perm_entries_save(const char *path, const uint64_t *perm, uint64_t n);
int csgn_perm_entries_load(const char *path, uint64_t *perm, uint64_t capacity, uint64_t *n);

/* ---- sharding (one process per GPU) ------------------------------------------ */

/* Contiguous range of the LEFT operand's blocks owned by `rank` of `world`:
 * rank g multiplies a[first..first+count) by the replicated right operand and owns
 * output blocks [first*T2, (first+count)*T2) -- globally i-major like the reference. */
int csgn_shard_range(uint64_t n_blocks, int rank, int world, uint64_t *first, uint64_t *count);

/* Sharded decrypt: the fold and its cross-GPU exchange in ONE kernel.
 *
 * A ciphertext sharded by block range decrypts to the parity of the SUM of the per-shard
 * satisfied-block counts (src/SecretKey.cpp:139 folds blocks with (dec + _dec) % 2).  That
 * one word per rank is the only exchange step of the path.  A csgn_comm gives every rank a
 * small mailbox in device memory that all its peers map over NVLink / NVSwitch; the decrypt
 * kernel that closes a batch has its last CTA store the batch's counts straight into every
 * rank's mailbox ("publish": posted 8-byte peer stores) and then poll its own mailbox until
 * every rank's words have arrived, writing the sums ("collect").  There is no separate
 * all-reduce launch and no collective library on the data path.
 *
 * Set-up:  csgn_comm_create on every rank -> exchange the CSGN_IPC_HANDLE_BYTES handles by
 * any means (torch.distributed / MPI all-gather, a file) -> csgn_comm_connect with all
 * `world` handles in rank order.  csgn_comm_connect_ptrs takes mailbox pointers that are
 * already peer-mapped (symmetric-memory allocators); world == 1 needs neither.
 * Contract (as for any collective): every rank issues the same sequence of pushes and
 * collects, and a closing launch is stream-ordered after the pushes it publishes (same stream, or
 * joined by events when the pushes were spread over several streams);
 * at most CSGN_COMM_MAX_PENDING pushes may stay unpublished, and a collect window
 * (n + lag) spans at most as many.  A rank that never arrives makes the collect time out
 * (CSGN_PEER_TIMEOUT_MS, default 30000): the totals read UINT64_MAX, blocking calls return
 * CSGN_ERR_TIMEOUT, the GPU is never left spinning.  After a timeout the ranks no longer agree on
 * the push sequence: free the communicator and build a new one. */
typedef struct csgn_comm csgn_comm;
#define CSGN_IPC_HANDLE_BYTES 64
#define CSGN_COMM_MAX_PENDING 64
int csgn_comm_create(int rank, int world, csgn_comm **out, unsigned char *handle_out);
int csgn_comm_connect(csgn_comm *comm, const unsigned char *handles);
int csgn_comm_connect_ptrs(csgn_comm *comm, void *const *peer_mailboxes);
/* Handle exchange through a directory every rank can see (a launcher without a communication library:
 * N processes started by a shell loop).  Writes `handle` to <dir>/csgn_<tag>_<world>_<rank>.handle, waits up
 * to timeout_ms for the other ranks' files, connects.  `tag` must be unique per job; files older than two
 * minutes before this call are taken for leftovers of a dead job and ignored; csgn_comm_free removes
 * this rank's file. */
int csgn_comm_connect_dir(csgn_comm *comm, const unsigned char *handle, const char *dir, const char *tag,
                          int timeout_ms);
/* This rank's mailbox (device pointer) and its size in bytes. */
void *csgn_comm_mailbox(const csgn_comm *comm, size_t *bytes);
int csgn_comm_free(csgn_comm *comm);
/* Pushes issued but not yet published to the peers. */
uint32_t csgn_comm_pending(const csgn_comm *comm);
/* Enqueue: fold this rank's shard `c`; its count becomes push number seq (0, 1, 2, ...) of this
 * communicator and stays in a local ring.  collect_n > 0 makes this launch close the batch: the
 * same kernel's last CTA publishes every unpublished push to every rank's mailbox and then collects
 * the collect_n pushes that end collect_lag pushes before this one (lag 0: ending with this one),
 * writing their sums over all ranks to device_totals[0..collect_n), oldest first.  Collecting the
 * previous batch (lag = batch size) never waits for a slower rank.  device_local (optional)
 * receives this rank's own count.  No host synchronisation. */
int csgn_decrypt_sharded_async(const csgn_buf *c, const csgn_key *key, csgn_comm *comm, uint32_t collect_n,
                               uint32_t collect_lag, uint64_t *device_totals, uint64_t *device_local);
/* A batch of n sharded folds: n-1 pushes spread over the lanes, then the closing launch on the current stream
 * publishes all n and collects the n pushes that end collect_lag pushes earlier (0: this batch) into device_totals. */
int csgn_decrypt_sharded_batch_async(const csgn_buf *const *c, uint32_t n, const csgn_key *key, csgn_comm *comm,
                                     uint32_t collect_lag, uint64_t *device_totals);
/* Fused multiply -> sharded decrypt: multiply this rank's shard a (its block range of the left operand) by the
 * replicated b, fold the product AND do the cross-GPU exchange in ONE kernel -- compute, reduction and collective
 * tile by tile in a single launch.  Arguments as csgn_decrypt_sharded_async, `out` as in csgn_mul_count_async. */
int csgn_mul_decrypt_sharded_async(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **out,
                                   csgn_comm *comm, uint32_t collect_n, uint32_t collect_lag, uint64_t *device_totals,
                                   uint64_t *device_local);
int csgn_mul_decrypt_sharded_batch_async(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n,
                                         const csgn_key *key, csgn_buf **out, csgn_comm *comm, uint32_t collect_lag,
                                         uint64_t *device_totals);
/* Enqueue a publish + collect on its own (one small launch): the n pushes ending lag pushes before
 * the most recent one. */
int csgn_comm_collect_async(csgn_comm *comm, uint32_t n, uint32_t lag, uint64_t *device_totals);
/* Blocking convenience = SecretKey::decrypt of a sharded ciphertext: push + collect of one
 * decrypt; *bit = total & 1 on every rank; *total (optional) the global count. */
int csgn_decrypt_sharded(const csgn_buf *c, const csgn_key *key, csgn_comm *comm, uint8_t *bit, uint64_t *total);
/* Mailbox addressing of push number `seq` (host-side mirror of the kernel's arithmetic). */
void csgn_comm_slot_tag(uint64_t seq, uint32_t *slot, uint64_t *tag);

#ifdef __cplusplus
}
#endif
#endif /* CSGN_H_ */
