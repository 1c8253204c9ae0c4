"""Python host layer over the C ABI -- used by tests, bench.py and torch.distributed
launches.  It mirrors the names of the reference's interface for this path
(Context / Ciphertext + * / SecretKey.decrypt / applyPermutation), but holds no
arithmetic of its own: every operation is one call into libcsgn.so.

The product for C++ users is csgn_b200/certfhe (libcertFHE.so); this module is the
same boundary seen from Python.
"""
import ctypes

import numpy as np

from . import _native
from ._native import CsgnError, check  # noqa: F401

_vp = ctypes.c_void_p


_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        _LIB = _native.load()
    return _LIB


def init(device=-1):
    """csgn_init: bind this process to one GPU (LOCAL_RANK by default)."""
    check(_lib().csgn_init(int(device)))


def shutdown():
    check(_lib().csgn_shutdown())


def is_initialized():
    return bool(_lib().csgn_is_initialized())


def sync():
    check(_lib().csgn_sync())


def launch_count():
    return int(_lib().csgn_launch_count())


def set_stream(cuda_stream_ptr):
    """Enqueue on an external stream (e.g. torch.cuda.current_stream().cuda_stream); 0/None = own."""
    check(_lib().csgn_set_stream(_vp(cuda_stream_ptr or 0)))


def set_auto_lanes(on):
    """csgn_set_auto_lanes: the library spreads consecutive independent operations over its internal streams."""
    check(_lib().csgn_set_auto_lanes(1 if on else 0))


def version():
    return _lib().csgn_version().decode()


def has_variants():
    """True when libcsgn.so was built with -DCSGN_BUILD_VARIANTS (the losing kernel variants kept for A/B sweeps)."""
    return "+variants" in version()


def device_info():
    sm, cc = ctypes.c_int(), ctypes.c_int()
    tot, fr = ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib().csgn_device_info(ctypes.byref(sm), ctypes.byref(tot), ctypes.byref(fr), ctypes.byref(cc)))
    return {"sm_count": sm.value, "hbm_total": tot.value, "hbm_free": fr.value, "cc": cc.value}


def words_per_block(N):
    return int(_lib().csgn_words_per_block(int(N)))


def shard_range(n_blocks, rank, world):
    first, count = ctypes.c_uint64(), ctypes.c_uint64()
    check(_lib().csgn_shard_range(int(n_blocks), int(rank), int(world), ctypes.byref(first), ctypes.byref(count)))
    return first.value, count.value


class Context:
    """Context(N, D): reference src/Context.cpp:20-29."""

    def __init__(self, N, D):
        self.N, self.D = int(N), int(D)
        self.S = self.N // (2 * self.D)
        self.L = words_per_block(self.N)

    def getN(self):
        return self.N

    def getD(self):
        return self.D

    def getS(self):
        return self.S

    def getDefaultN(self):
        return self.L


def _host_words(a):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.uint64).reshape(-1))
    return a


class Ciphertext:
    """Device-resident ciphertext: n_blocks blocks of ctx.L words behind a csgn_buf."""

    def __init__(self, handle, ctx, keepalive=None):
        self._h = handle
        self.ctx = ctx
        self._keepalive = keepalive  # e.g. the torch tensor a view was built over

    # -- construction -----------------------------------------------------
    @classmethod
    def from_host(cls, words, ctx):
        """Ciphertext(V, Bitlen, len, ctx) with the canonical Bitlen (src/Ciphertext.cpp:344-358)."""
        w = _host_words(words)
        if w.size % ctx.L:
            raise ValueError("len must be a multiple of the %d words per block" % ctx.L)
        h = _vp()
        check(_lib().csgn_buf_upload(w.ctypes.data_as(_vp), w.size // ctx.L, ctx.L, ctypes.byref(h)))
        sync()  # `w` may be a temporary; the copy is asynchronous
        return cls(h, ctx)

    @classmethod
    def from_host_ptr(cls, host_ptr, n_blocks, ctx):
        """Asynchronous upload from caller-managed (ideally pinned) host memory."""
        h = _vp()
        rc = _LIB.csgn_buf_upload(host_ptr, n_blocks, ctx.L, ctypes.byref(h))
        if rc:
            check(rc)
        return cls(h, ctx)

    @classmethod
    def empty(cls, n_blocks, ctx):
        h = _vp()
        check(_lib().csgn_buf_alloc(int(n_blocks), ctx.L, ctypes.byref(h)))
        return cls(h, ctx)

    @classmethod
    def view(cls, device_ptr, n_blocks, ctx, keepalive=None):
        h = _vp()
        check(_lib().csgn_buf_wrap(_vp(device_ptr), int(n_blocks), ctx.L, ctypes.byref(h)))
        return cls(h, ctx, keepalive)

    @classmethod
    def from_tensor(cls, t, ctx):
        """View over a torch int64/uint64 CUDA tensor of n_blocks*L words (no copy)."""
        assert t.is_cuda and t.is_contiguous() and t.element_size() == 8
        return cls.view(t.data_ptr(), t.numel() // ctx.L, ctx, keepalive=t)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _LIB is not None:
            try:
                _LIB.csgn_buf_free(h)
            except Exception:
                pass

    # -- accessors ----------------------------------------------------------
    @property
    def n_blocks(self):
        return int(_lib().csgn_buf_blocks(self._h))

    def getLen(self):
        """Length in 64-bit words, as the reference reports it (src/Ciphertext.cpp:417-420)."""
        return self.n_blocks * self.ctx.L

    def device_ptr(self):
        return _lib().csgn_buf_device_ptr(self._h) or 0

    def getValues(self):
        out = np.empty(self.getLen(), dtype=np.uint64)
        check(_lib().csgn_buf_download(self._h, out.ctypes.data_as(_vp)))
        return out

    def download_range(self, first_block, n_blocks):
        out = np.empty(n_blocks * self.ctx.L, dtype=np.uint64)
        check(_lib().csgn_buf_download_range(self._h, int(first_block), int(n_blocks), out.ctypes.data_as(_vp)))
        return out

    def getBitlen(self):
        """The reference's side array, synthesised: [64]*(L-1)+[N%64 or 64] per block."""
        L, rem = self.ctx.L, self.ctx.N % 64
        one = np.full(L, 64, dtype=np.uint64)
        if rem:
            one[L - 1] = rem
        return np.tile(one, self.n_blocks)

    def size(self):
        """Bytes, by the reference's formula (src/Ciphertext.cpp:91-101)."""
        return 32 + 16 * self.getLen()

    def checksum(self):
        x, s, h = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        check(_lib().csgn_buf_checksum(self._h, ctypes.byref(x), ctypes.byref(s), ctypes.byref(h)))
        return x.value, s.value, h.value

    def save(self, path):
        """csgn_buf_save: header + raw words, streamed through pinned staging."""
        check(_lib().csgn_buf_save(self._h, self.ctx.N, self.ctx.D, str(path).encode()))

    @classmethod
    def load(cls, path):
        h, n, d = _vp(), ctypes.c_uint64(), ctypes.c_uint64()
        check(_lib().csgn_buf_load(str(path).encode(), ctypes.byref(n), ctypes.byref(d), ctypes.byref(h)))
        return cls(h, Context(n.value, d.value))

    def save_shard(self, prefix, rank, world, first_block=0):
        """csgn_buf_save_shard: this rank's local blocks as `<prefix>.shard<rank>of<world>`."""
        check(_lib().csgn_buf_save_shard(self._h, self.ctx.N, self.ctx.D, str(prefix).encode(), int(rank), int(world),
                                         int(first_block)))

    @classmethod
    def load_shard(cls, prefix, rank, world):
        """-> (ciphertext of the rank's local blocks, first global block as recorded at save time)"""
        h, n, d, first = _vp(), ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        check(_lib().csgn_buf_load_shard(str(prefix).encode(), int(rank), int(world), ctypes.byref(n), ctypes.byref(d),
                                         ctypes.byref(first), ctypes.byref(h)))
        return cls(h, Context(n.value, d.value)), first.value

    def clone(self):
        h = _vp()
        check(_lib().csgn_buf_clone(self._h, ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    # -- the hot path ---------------------------------------------------------
    def __mul__(self, other):
        h = _vp()
        rc = _LIB.csgn_mul(self._h, other._h, ctypes.byref(h))
        if rc:
            check(rc)
        return Ciphertext(h, self.ctx)

    def mul_into(self, other, out):
        rc = _LIB.csgn_mul_into(self._h, other._h, out._h)
        if rc:
            check(rc)
        return out

    def __imul__(self, other):
        h = _vp()
        check(_lib().csgn_mul(self._h, other._h, ctypes.byref(h)))
        old, self._h = self._h, h
        _lib().csgn_buf_free(old)
        return self

    def __add__(self, other):
        h = _vp()
        check(_lib().csgn_concat(self._h, other._h, ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    def __iadd__(self, other):
        check(_lib().csgn_append(self._h, other._h))
        return self

    def add_lazy(self, other):
        """csgn_concat_lazy: self || other without copying (a rope of the operands' storage)."""
        h = _vp()
        check(_lib().csgn_concat_lazy(self._h, other._h, ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    @property
    def segments(self):
        return int(_lib().csgn_buf_segments(self._h))

    def flatten(self):
        check(_lib().csgn_buf_flatten(self._h))
        return self

    def applyPermutation(self, perm, strict_ref_truncate=False):
        h = _vp()
        check(_lib().csgn_permute(self._h, perm._h, 1 if strict_ref_truncate else 0, ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    def compact(self):
        """A new ciphertext without the blocks that have fewer than D set bits (see CiphertextArray.compact): the same
        satisfied-block count under every key of the context."""
        return CiphertextArray(self, [0, self.n_blocks]).compact().storage

    def cancel(self):
        """A new ciphertext keeping the first occurrence of every block value that occurs an odd number of times (see
        CiphertextArray.cancel): the same decryption under every key, a satisfied-block count of the same parity."""
        return CiphertextArray(self, [0, self.n_blocks]).cancel().storage

    def permute_into(self, perm, out):
        check(_lib().csgn_permute_into(self._h, perm._h, out._h))
        return out


def handle_array(cts):
    """ctypes array of the csgn_buf handles of `cts` (build once and reuse for a fixed batch)."""
    return (_vp * len(cts))(*[c._h.value if isinstance(c._h, _vp) else c._h for c in cts])


class UploadBatch:
    """csgn_buf_upload_batch with its argument arrays built once: n operands go to the device in one call (one
    shared allocation, copies issued back to back).  upload() returns a ctypes array of n csgn_buf handles -- pass slices of it
    (handle_slice) to the batch entry points and release it with free_handles."""

    def __init__(self, host_ptrs, n_blocks, ctx):
        self.n, self.ctx = len(host_ptrs), ctx
        self._ptrs = (_vp * self.n)(*host_ptrs)
        self._nb = (ctypes.c_uint64 * self.n)(*n_blocks)

    def upload(self):
        out = (_vp * self.n)()
        rc = _LIB.csgn_buf_upload_batch(self._ptrs, self._nb, self.n, self.ctx.L, out)
        if rc:
            check(rc)
        return out


def handle_slice(arr, first, n):
    """entries [first, first+n) of a handle array, as an array the batch entry points accept (no copy)"""
    return (_vp * n).from_buffer(arr, first * ctypes.sizeof(_vp))


def free_handles(arr):
    """csgn_buf_free_batch: release every handle of a ctypes handle array"""
    _LIB.csgn_buf_free_batch(arr, len(arr))


def mul_batch_arrays(aa, ab, ao):
    """csgn_mul_batch on handle arrays: ao[i] (NULL on entry) receives the product aa[i] * ab[i]."""
    rc = _LIB.csgn_mul_batch(aa, ab, len(aa), ao)
    if rc:
        check(rc)


def mul_into_batch(a, b, out, arrays=None):
    """csgn_mul_into_batch: out[i] = a[i] * b[i]; the library overlaps the independent products on its lanes.
    `arrays` = (handle_array(a), handle_array(b), handle_array(out)) built beforehand skips the marshalling."""
    aa, ab, ao = arrays or (handle_array(a), handle_array(b), handle_array(out))
    rc = _LIB.csgn_mul_into_batch(aa, ab, len(aa), ao)
    if rc:
        check(rc)


def mul_batch(a, b):
    """csgn_mul_batch: the list of products a[i] * b[i] (allocated by the library)."""
    n = len(a)
    out = (_vp * n)()
    rc = _LIB.csgn_mul_batch(handle_array(a), handle_array(b), n, out)
    if rc:
        check(rc)
    return [Ciphertext(_vp(out[i]), a[i].ctx) for i in range(n)]


def mul_count_batch_async(key, a, b, device_counts_ptr, out=None, arrays=None):
    """csgn_mul_count_batch_async: the fused multiply -> decrypt of n independent pairs.  out = None: count only;
    out = list of Ciphertexts: the products are written into them; out = "alloc": the library allocates them and
    the list is returned.  `arrays` = (handle_array(a), handle_array(b), handle_array(out) or None) skips marshalling."""
    if arrays is not None:
        aa, ab, ao = arrays
    else:
        aa, ab = handle_array(a), handle_array(b)
        ao = None if out is None else ((_vp * len(aa))() if out == "alloc" else handle_array(out))
    rc = _LIB.csgn_mul_count_batch_async(aa, ab, len(aa), key._h, ao, device_counts_ptr)
    if rc:
        check(rc)
    if arrays is None and out == "alloc":
        return [Ciphertext(_vp(ao[i]), a[i].ctx) for i in range(len(aa))]
    return None


def _offsets(off):
    o = np.ascontiguousarray(np.asarray(off, dtype=np.uint64).reshape(-1))
    if o.size == 0:
        raise ValueError("offsets need n + 1 entries")
    return o


class CiphertextArray:
    """n independent ciphertexts as ONE device buffer (`storage`, a Ciphertext) plus numpy block offsets: element k is
    blocks [offsets[k], offsets[k+1]) (include/csgn.h, "ciphertext arrays").  Element-wise *, + and gather are one
    library call each, with one kernel launch for all small elements."""

    def __init__(self, storage, offsets):
        self.storage = storage
        self.offsets = _offsets(offsets)
        self.ctx = storage.ctx

    # -- construction -----------------------------------------------------
    @classmethod
    def from_host(cls, elements, ctx):
        """One upload of the host word arrays `elements` (each a multiple of ctx.L words)."""
        words = [_host_words(e) for e in elements]
        if any(w.size % ctx.L for w in words):
            raise ValueError("every element needs a multiple of the %d words per block" % ctx.L)
        off = np.zeros(len(words) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([w.size // ctx.L for w in words], dtype=np.uint64)
        flat = np.concatenate(words) if words else np.empty(0, dtype=np.uint64)
        return cls(Ciphertext.from_host(flat, ctx), off)

    @classmethod
    def pack(cls, cts):
        """csgn_concat_n: the ciphertexts `cts` packed into one array in one launch."""
        if not cts:
            raise ValueError("pack needs at least one ciphertext")
        h = _vp()
        check(_lib().csgn_concat_n(handle_array(cts), len(cts), ctypes.byref(h)))
        off = np.zeros(len(cts) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([c.n_blocks for c in cts], dtype=np.uint64)
        return cls(Ciphertext(h, cts[0].ctx), off)

    # -- access -------------------------------------------------------------
    def __len__(self):
        return self.offsets.size - 1

    def blocks(self, k):
        return int(self.offsets[k + 1] - self.offsets[k])

    def element(self, k):
        """Element k as an ordinary Ciphertext (a device copy of its blocks, csgn_buf_slice)."""
        if not 0 <= k < len(self):
            raise IndexError(k)
        h = _vp()
        check(_lib().csgn_buf_slice(self.storage._h, int(self.offsets[k]), self.blocks(k), ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    def to_host(self):
        """The words of every element, as a list of numpy arrays."""
        w = self.storage.getValues()
        L = self.ctx.L
        return [w[int(self.offsets[k]) * L:int(self.offsets[k + 1]) * L] for k in range(len(self))]

    # -- element-wise operations --------------------------------------------
    def _binary(self, fn, other):
        if len(other) != len(self):
            raise ValueError("arrays of %d and %d elements" % (len(self), len(other)))
        out_off = np.empty(len(self) + 1, dtype=np.uint64)
        h = _vp()
        check(fn(self.storage._h, self.offsets.ctypes.data_as(_vp), other.storage._h, other.offsets.ctypes.data_as(_vp),
                 len(self), out_off.ctypes.data_as(_vp), ctypes.byref(h)))
        return CiphertextArray(Ciphertext(h, self.ctx), out_off)

    def __mul__(self, other):
        """csgn_seg_mul: element k = self_k * other_k."""
        return self._binary(_lib().csgn_seg_mul, other)

    def __add__(self, other):
        """csgn_seg_concat: element k = self_k + other_k (block concatenation, the homomorphic XOR)."""
        return self._binary(_lib().csgn_seg_concat, other)

    @staticmethod
    def sum_of_products(products, terms=(), compact=False):
        """csgn_seg_mul_sum: element k = A0_k*B0_k + A1_k*B1_k + ... + C0_k + ... for `products` [(A0, B0), ...] and
        `terms` [C0, ...], every output word written once (one gate of a circuit in one call).  compact=True
        (csgn_seg_mul_sum_compact with min_bits = D): only the blocks with at least D set bits, which are the only
        blocks any key of the context can satisfy, so every decryption is unchanged."""
        products = [(x, y) for x, y in products]
        terms = list(terms)
        arrays = [x for pr in products for x in pr] + terms
        if not arrays:
            raise ValueError("sum_of_products needs at least one product or term")
        n, ctx = len(arrays[0]), arrays[0].ctx
        for x in arrays[1:]:
            if len(x) != n:
                raise ValueError("arrays of %d and %d elements" % (n, len(x)))
            if (x.ctx.N, x.ctx.D) != (ctx.N, ctx.D):
                raise ValueError("arrays of Context(%d,%d) and Context(%d,%d)" % (ctx.N, ctx.D, x.ctx.N, x.ctx.D))
        h = lambda xs: handle_array([x.storage for x in xs]) if xs else None                          # noqa: E731
        o = lambda xs: (_vp * len(xs))(*[x.offsets.ctypes.data for x in xs]) if xs else None          # noqa: E731
        left, right = [x for x, _ in products], [y for _, y in products]
        out_off = np.empty(n + 1, dtype=np.uint64)
        out = _vp()
        args = (h(left), o(left), h(right), o(right), len(products), h(terms), o(terms), len(terms), n)
        if compact:
            check(_lib().csgn_seg_mul_sum_compact(*args, ctx.D, out_off.ctypes.data_as(_vp), ctypes.byref(out)))
        else:
            check(_lib().csgn_seg_mul_sum(*args, out_off.ctypes.data_as(_vp), ctypes.byref(out)))
        return CiphertextArray(Ciphertext(out, ctx), out_off)

    def compact(self):
        """The array without the blocks that have fewer than D set bits (no key of the context satisfies them): every
        element keeps its other blocks in order and decrypts as before under every key."""
        return CiphertextArray.sum_of_products([], [self], compact=True)

    def cancel(self):
        """csgn_seg_cancel: every element keeps, in order, the first occurrence of each block value that occurs an odd
        number of times in it (x*x -> x, a + a -> empty).  Equal blocks are satisfied by the same keys, so every
        element decrypts as before under every key; unlike compact(), its satisfied-block count changes (by an even
        number).  The usual gate is sum_of_products(..., compact=True).cancel()."""
        out_off = np.empty(len(self) + 1, dtype=np.uint64)
        h = _vp()
        check(_lib().csgn_seg_cancel(self.storage._h, self.offsets.ctypes.data_as(_vp), len(self),
                                     out_off.ctypes.data_as(_vp), ctypes.byref(h)))
        return CiphertextArray(Ciphertext(h, self.ctx), out_off)

    def gather(self, idx):
        """csgn_seg_gather: element j = self_{idx[j]} (any order, repeats allowed)."""
        ix = np.ascontiguousarray(np.asarray(idx, dtype=np.uint64).reshape(-1))
        out_off = np.empty(ix.size + 1, dtype=np.uint64)
        h = _vp()
        check(_lib().csgn_seg_gather(self.storage._h, self.offsets.ctypes.data_as(_vp), len(self), ix.ctypes.data_as(_vp),
                                     ix.size, out_off.ctypes.data_as(_vp), ctypes.byref(h)))
        return CiphertextArray(Ciphertext(h, self.ctx), out_off)

    def applyPermutation(self, perm):
        """Every element permuted (csgn_permute on the storage; the offsets do not change)."""
        if self.storage.n_blocks == 0:
            return CiphertextArray(self.storage.clone(), self.offsets.copy())
        return CiphertextArray(self.storage.applyPermutation(perm), self.offsets.copy())


class Result:
    """A decrypt whose count the host reads later (csgn_result)."""

    def __init__(self, handle):
        self._h = handle

    def ready(self):
        return bool(_lib().csgn_result_ready(self._h))

    def count(self):
        c = ctypes.c_uint64()
        check(_lib().csgn_result_wait(self._h, ctypes.byref(c)))
        return int(c.value)

    def bit(self):
        return self.count() & 1

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _LIB is not None:
            try:
                _LIB.csgn_result_free(h)
            except Exception:
                pass


class SecretKey:
    """Secret positions held as a device position mask (csgn_key)."""

    def __init__(self, ctx, positions):
        self.ctx = ctx
        self.s = _host_words(positions)
        self._h = _vp()
        check(_lib().csgn_key_create(ctx.N, self.s.ctypes.data_as(_vp), self.s.size, ctypes.byref(self._h)))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib().csgn_key_free(h)
            except Exception:
                pass

    def decrypt(self, ct):
        bit = ctypes.c_uint8()
        check(_lib().csgn_decrypt(ct._h, self._h, ctypes.byref(bit)))
        return int(bit.value)

    def count_satisfied(self, ct):
        c = ctypes.c_uint64()
        check(_lib().csgn_decrypt_count(ct._h, self._h, ctypes.byref(c)))
        return int(c.value)

    def decrypt_deferred(self, ct):
        """csgn_decrypt_deferred: enqueue the fold and the copy of its count; read it later from the Result."""
        h = _vp()
        check(_lib().csgn_decrypt_deferred(ct._h, self._h, ctypes.byref(h)))
        return Result(h)

    def mul_decrypt(self, a, b, out=None):
        """csgn_mul_decrypt: Dec(a*b) by the fused kernel.  out = None: count only -> (bit, count);
        out = "alloc": -> (bit, count, product); out = Ciphertext: the product is written into it."""
        bit, cnt = ctypes.c_uint8(), ctypes.c_uint64()
        if out is None:
            check(_lib().csgn_mul_decrypt(a._h, b._h, self._h, None, ctypes.byref(bit), ctypes.byref(cnt)))
            return int(bit.value), int(cnt.value)
        h = _vp() if isinstance(out, str) else _vp(out._h.value if isinstance(out._h, _vp) else out._h)
        check(_lib().csgn_mul_decrypt(a._h, b._h, self._h, ctypes.byref(h), ctypes.byref(bit), ctypes.byref(cnt)))
        if isinstance(out, str):
            return int(bit.value), int(cnt.value), Ciphertext(h, a.ctx)
        return int(bit.value), int(cnt.value)

    def mul_count_async(self, a, b, device_count_ptr, out=None):
        """csgn_mul_count_async into a device word; out as in mul_decrypt (None / Ciphertext)."""
        if out is None:
            rc = _LIB.csgn_mul_count_async(a._h, b._h, self._h, None, device_count_ptr)
        else:
            h = _vp(out._h.value if isinstance(out._h, _vp) else out._h)
            rc = _LIB.csgn_mul_count_async(a._h, b._h, self._h, ctypes.byref(h), device_count_ptr)
        if rc:
            check(rc)

    def mul_decrypt_deferred(self, a, b, want_product=False):
        """csgn_mul_decrypt_deferred -> Result, or (Result, product)."""
        r = _vp()
        if not want_product:
            check(_lib().csgn_mul_decrypt_deferred(a._h, b._h, self._h, None, ctypes.byref(r)))
            return Result(r)
        h = _vp()
        check(_lib().csgn_mul_decrypt_deferred(a._h, b._h, self._h, ctypes.byref(h), ctypes.byref(r)))
        return Result(r), Ciphertext(h, a.ctx)

    def encrypt_batch(self, bits, seed, first_block=0):
        """n fresh blocks on the GPU, block i encrypting bits[i] (csgn_encrypt_batch, Philox keyed by seed)."""
        b = np.ascontiguousarray(np.asarray(bits, dtype=np.uint8))
        h = _vp()
        check(_lib().csgn_encrypt_batch(self._h, b.ctypes.data_as(_vp), b.size, int(first_block), int(seed), ctypes.byref(h)))
        return Ciphertext(h, self.ctx)

    def encrypt_array(self, bits, seed, first_block=0):
        """CiphertextArray of len(bits) one-block encryptions (csgn_encrypt_batch, offsets 0, 1, ..., n)."""
        n = np.asarray(bits).size
        return CiphertextArray(self.encrypt_batch(bits, seed, first_block), np.arange(n + 1, dtype=np.uint64))

    def decrypt_array_count_async(self, arr, device_counts_ptr):
        """csgn_seg_decrypt_count_async: device_counts[k] = satisfied blocks of element k, no synchronisation."""
        check(_lib().csgn_seg_decrypt_count_async(arr.storage._h, arr.offsets.ctypes.data_as(_vp), len(arr), self._h,
                                                  _vp(device_counts_ptr)))

    def decrypt_array(self, arr):
        """csgn_seg_decrypt: (bits, counts) of every element as numpy arrays, one synchronisation."""
        n = len(arr)
        bits, counts = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint64)
        check(_lib().csgn_seg_decrypt(arr.storage._h, arr.offsets.ctypes.data_as(_vp), n, self._h,
                                      bits.ctypes.data_as(_vp), counts.ctypes.data_as(_vp)))
        return bits, counts

    def decrypt_product(self, factors):
        """Dec(f1*f2*...*fn) without materialising the product (csgn_decrypt_product).
        Returns (bit, count) with count saturated at 2**64-1."""
        arr = (_vp * len(factors))(*[f._h for f in factors])
        bit, cnt = ctypes.c_uint8(), ctypes.c_uint64()
        check(_lib().csgn_decrypt_product(arr, len(factors), self._h, ctypes.byref(bit), ctypes.byref(cnt)))
        return int(bit.value), int(cnt.value)

    def count_satisfied_async(self, ct, device_count_ptr):
        rc = _LIB.csgn_decrypt_count_async(ct._h, self._h, device_count_ptr)
        if rc:
            check(rc)

    def count_satisfied_batch_async(self, cts, device_counts_ptr, array=None):
        """csgn_decrypt_count_batch_async: device_counts[i] = satisfied blocks of cts[i], no synchronisation."""
        arr = array or handle_array(cts)
        rc = _LIB.csgn_decrypt_count_batch_async(arr, len(arr), self._h, device_counts_ptr)
        if rc:
            check(rc)

    def decrypt_batch(self, cts):
        """csgn_decrypt_batch: (bits, counts) of n ciphertexts with one synchronisation."""
        n = len(cts)
        bits, counts = (ctypes.c_uint8 * n)(), (ctypes.c_uint64 * n)()
        check(_lib().csgn_decrypt_batch(handle_array(cts), n, self._h, bits, counts))
        return list(bits), list(counts)

    def size(self):
        return 16 + 8 * int(self.s.size)

    def save(self, path):
        """csgn_key_positions_save: header (N, D, count, checksum) + the secret positions."""
        check(_lib().csgn_key_positions_save(str(path).encode(), self.ctx.N, self.ctx.D, self.s.ctypes.data_as(_vp), self.s.size))

    @classmethod
    def load(cls, path):
        n, d, cnt = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        check(_lib().csgn_key_positions_load(str(path).encode(), ctypes.byref(n), ctypes.byref(d), None, 0, ctypes.byref(cnt)))
        pos = np.empty(cnt.value, dtype=np.uint64)
        check(_lib().csgn_key_positions_load(str(path).encode(), ctypes.byref(n), ctypes.byref(d), pos.ctypes.data_as(_vp),
                                             pos.size, ctypes.byref(cnt)))
        return cls(Context(n.value, d.value), pos)


IPC_HANDLE_BYTES = 64
COMM_MAX_PENDING = 64


def comm_slot_tag(seq):
    """(slot, tag) of push number `seq` in a mailbox -- csgn_comm_slot_tag."""
    slot, tag = ctypes.c_uint32(), ctypes.c_uint64()
    _lib().csgn_comm_slot_tag(int(seq), ctypes.byref(slot), ctypes.byref(tag))
    return slot.value, tag.value


class PeerComm:
    """csgn_comm: per-rank mailboxes mapped over NVLink, so that a sharded decrypt's fold
    kernel also does the cross-GPU exchange (csrc/peer.cuh).  `allgather_bytes(b)` must return
    the list of every rank's 64-byte handle in rank order (see sharding.connect_peers for the
    torch.distributed version); it is not needed for world == 1."""

    def __init__(self, rank, world, allgather_bytes=None):
        self.rank, self.world = int(rank), int(world)
        self._h = _vp()
        handle = (ctypes.c_ubyte * IPC_HANDLE_BYTES)()
        check(_lib().csgn_comm_create(self.rank, self.world, ctypes.byref(self._h), handle))
        if self.world > 1:
            if allgather_bytes is None:
                raise ValueError("world > 1 needs an allgather_bytes callable to exchange the mailbox handles")
            handles = allgather_bytes(bytes(handle))
            if len(handles) != self.world or any(len(h) != IPC_HANDLE_BYTES for h in handles):
                raise ValueError("allgather_bytes must return %d handles of %d bytes" % (self.world, IPC_HANDLE_BYTES))
            blob = (ctypes.c_ubyte * (IPC_HANDLE_BYTES * self.world)).from_buffer_copy(b"".join(handles))
            check(_lib().csgn_comm_connect(self._h, blob))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _LIB is not None:
            try:
                _LIB.csgn_comm_free(h)
            except Exception:
                pass

    @property
    def pending(self):
        return int(_lib().csgn_comm_pending(self._h))

    def push(self, key, ct, collect_n=0, device_totals_ptr=0, device_local_ptr=0, lag=0):
        """Enqueue the fold of this rank's shard (push number seq).  collect_n > 0 closes a batch in the
        same kernel: publish everything unpublished, collect the collect_n pushes ending `lag` pushes ago."""
        rc = _LIB.csgn_decrypt_sharded_async(ct._h, key._h, self._h, collect_n, lag, device_totals_ptr or None,
                                             device_local_ptr or None)
        if rc:
            check(rc)

    def push_batch(self, key, cts, device_totals_ptr, lag=0, array=None):
        """csgn_decrypt_sharded_batch_async: fold every shard of `cts` (spread over the library's lanes); the closing
        launch publishes all of them and collects the len(cts) pushes that end `lag` pushes earlier."""
        arr = array or handle_array(cts)
        rc = _LIB.csgn_decrypt_sharded_batch_async(arr, len(arr), key._h, self._h, lag, device_totals_ptr)
        if rc:
            check(rc)

    def mul_push(self, key, a, b, out=None, collect_n=0, device_totals_ptr=0, device_local_ptr=0, lag=0):
        """csgn_mul_decrypt_sharded_async: multiply this rank's shard by the replicated b, fold and exchange in one
        kernel.  out = None: count only; out = Ciphertext: the product shard is written into it."""
        if out is None:
            rc = _LIB.csgn_mul_decrypt_sharded_async(a._h, b._h, key._h, None, self._h, collect_n, lag,
                                                     device_totals_ptr or None, device_local_ptr or None)
        else:
            h = _vp(out._h.value if isinstance(out._h, _vp) else out._h)
            rc = _LIB.csgn_mul_decrypt_sharded_async(a._h, b._h, key._h, ctypes.byref(h), self._h, collect_n, lag,
                                                     device_totals_ptr or None, device_local_ptr or None)
        if rc:
            check(rc)

    def mul_push_batch(self, key, arrays, device_totals_ptr, lag=0):
        """csgn_mul_decrypt_sharded_batch_async; arrays = (handle_array(a), handle_array(b), handle_array(out) or None)."""
        aa, ab, ao = arrays
        rc = _LIB.csgn_mul_decrypt_sharded_batch_async(aa, ab, len(aa), key._h, ao, self._h, lag, device_totals_ptr)
        if rc:
            check(rc)

    def collect(self, n, device_totals_ptr, lag=0):
        check(_lib().csgn_comm_collect_async(self._h, int(n), int(lag), device_totals_ptr))

    def decrypt(self, key, ct):
        """Blocking sharded SecretKey::decrypt: (bit, global satisfied-block count), the same on every rank."""
        bit, tot = ctypes.c_uint8(), ctypes.c_uint64()
        check(_lib().csgn_decrypt_sharded(ct._h, key._h, self._h, ctypes.byref(bit), ctypes.byref(tot)))
        return int(bit.value), int(tot.value)


class Permutation:
    """Permutation of [0,N) held as a device bit-source map (csgn_perm)."""

    def __init__(self, ctx, perm):
        self.ctx = ctx
        self.p = _host_words(perm)
        self._h = _vp()
        check(_lib().csgn_perm_create(ctx.N, self.p.ctypes.data_as(_vp), ctypes.byref(self._h)))

    def save(self, path):
        """csgn_perm_entries_save: header (length, checksum) + the entries."""
        check(_lib().csgn_perm_entries_save(str(path).encode(), self.p.ctypes.data_as(_vp), self.p.size))

    @classmethod
    def load(cls, path, ctx):
        cnt = ctypes.c_uint64()
        check(_lib().csgn_perm_entries_load(str(path).encode(), None, 0, ctypes.byref(cnt)))
        perm = np.empty(cnt.value, dtype=np.uint64)
        check(_lib().csgn_perm_entries_load(str(path).encode(), perm.ctypes.data_as(_vp), perm.size, ctypes.byref(cnt)))
        if cnt.value != ctx.N:
            raise ValueError("permutation of %d entries, context has N = %d" % (cnt.value, ctx.N))
        return cls(ctx, perm)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib().csgn_perm_free(h)
            except Exception:
                pass


def decrypt_positions(ct, ctx, positions):
    s = _host_words(positions)
    bit = ctypes.c_uint8()
    check(_lib().csgn_decrypt_positions(ct._h, ctx.N, s.ctypes.data_as(_vp), s.size, ctypes.byref(bit)))
    return int(bit.value)
