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


class Circuit:
    """A netlist of gates over ciphertext arrays, evaluated over every lane in one call (csgn_seg_circuit).  Wires 0 ..
    n_inputs - 1 are the inputs; gate(products, terms) adds the gate sum(u*v for (u, v) in products) + sum(terms) over
    earlier wires and returns its wire."""

    def __init__(self, n_inputs):
        if n_inputs < 1:
            raise ValueError("a circuit needs at least one input")
        self.n_inputs = int(n_inputs)
        self.n_gates = 0
        self._gates = []
        self.last_fallback = None       # lanes of the last evaluate() that took the gate-by-gate path

    @property
    def n_wires(self):
        return self.n_inputs + self.n_gates

    def gate(self, products=(), terms=()):
        products = [(int(u), int(v)) for u, v in products]
        terms = [int(w) for w in terms]
        if not products and not terms:
            raise ValueError("a gate needs at least one product or term")
        for w in [x for pr in products for x in pr] + terms:
            if not 0 <= w < self.n_wires:
                raise ValueError("wire %d is not below the gate's own wire %d" % (w, self.n_wires))
        self._gates += [len(products), len(terms)] + [x for pr in products for x in pr] + terms
        self.n_gates += 1
        return self.n_wires - 1

    def evaluate(self, inputs, outputs, min_bits=None, cancel=False, lane_capacity=0):
        """The arrays of wires `outputs` over the lanes of `inputs` (one CiphertextArray per input wire, all of n
        elements): each gate as sum_of_products, compacted to min_bits set bits (None: D of the context; 0: no
        compaction) and, with cancel, cancelled.  lane_capacity: blocks per lane on the device (0: the library chooses);
        lanes that do not fit are evaluated gate by gate (last_fallback counts them)."""
        inputs = list(inputs)
        outputs = [int(w) for w in outputs]
        if len(inputs) != self.n_inputs:
            raise ValueError("the circuit has %d inputs, got %d arrays" % (self.n_inputs, len(inputs)))
        n, ctx = len(inputs[0]), inputs[0].ctx
        for x in inputs[1:]:
            if len(x) != n:
                raise ValueError("arrays of %d and %d elements" % (n, len(x)))
            if (x.ctx.N, x.ctx.D) != (ctx.N, ctx.D):
                raise ValueError("arrays of Context(%d,%d) and Context(%d,%d)" % (ctx.N, ctx.D, x.ctx.N, x.ctx.D))
        if not outputs:
            raise ValueError("evaluate needs at least one output wire")
        gates = np.asarray(self._gates, dtype=np.uint32)
        outs = np.asarray(outputs, dtype=np.uint32)
        out_offs = [np.empty(n + 1, dtype=np.uint64) for _ in outputs]
        out = (_vp * len(outputs))()
        fallback = ctypes.c_uint64(0)
        check(_lib().csgn_seg_circuit(
            handle_array([x.storage for x in inputs]), (_vp * len(inputs))(*[x.offsets.ctypes.data for x in inputs]),
            len(inputs), n, gates.ctypes.data_as(_vp), gates.size, self.n_gates, outs.ctypes.data_as(_vp), outs.size,
            ctx.D if min_bits is None else int(min_bits), 1 if cancel else 0, int(lane_capacity),
            (_vp * len(outputs))(*[o.ctypes.data for o in out_offs]), out, ctypes.byref(fallback)))
        self.last_fallback = fallback.value
        return [CiphertextArray(Ciphertext(_vp(out[j]), ctx), out_offs[j]) for j in range(len(outputs))]


class UIntCircuit:
    """Integer netlists over encrypted integers (EncryptedUInt), built on the host and evaluated as ONE Circuit call.

    An integer is a list of wire ids, LSB first.  Wires: operand i, bit j is input i*width + j; then the `one` input
    (one=True: the caller supplies an encryption of 1 per lane, which only the key holder can make); then the zero
    input, n empty elements, which the builder declares and evaluate() supplies (an empty ciphertext decrypts to 0).
    Every operation is a sum of products plus terms over GF(2) (XOR of ANDs); a gate that folds to one wire (x + 0,
    x*1, a single term) adds no gate.  Operands may differ in width: the shorter one is zero-extended, and the result
    has the larger width.  certFHE::UIntCircuit builds the same netlists, wire for wire.

    Size: with cancel=True a result holds, per lane, the blocks of its function's algebraic normal form over the input
    blocks (whatever the netlist) that compaction keeps.  That form stays small for add, and, xor, or, select and the
    shifts at any width, but grows about threefold per bit for sub, neg, the comparisons, min, max and mul (lt and ne
    of two W-bit operands have 3^W - 1 monomials), so those are practical up to about 8-12 bits, and compositions of
    them at fewer."""

    def __init__(self, width, n_operands, one=False):
        width, n_operands = int(width), int(n_operands)
        if not 1 <= width <= 64:
            raise ValueError("width %d outside 1..64" % width)
        if n_operands < 0:
            raise ValueError("negative operand count")
        self.width, self.n_operands = width, n_operands
        self.inputs = [[i * width + j for j in range(width)] for i in range(n_operands)]
        self.one = n_operands * width if one else None
        self.zero = n_operands * width + (1 if one else 0)
        self.circuit = Circuit(self.zero + 1)

    @property
    def last_fallback(self):
        return self.circuit.last_fallback

    def netlist(self):
        """(inputs, flat gates) as csgn_seg_circuit takes them: per gate p, q, p operand pairs, q terms."""
        return self.circuit.n_inputs, list(self.circuit._gates)

    # -- gates ----------------------------------------------------------------------------------------------------
    def _gate(self, products, terms):
        z, o = self.zero, self.one
        terms = [w for w in terms if w != z]
        prods = []
        for u, v in products:
            if u == z or v == z:
                continue
            if u == o:
                terms.append(v)
            elif v == o:
                terms.append(u)
            else:
                prods.append((u, v))
        if not prods and not terms:
            return z
        if not prods and len(terms) == 1:
            return terms[0]
        return self.circuit.gate(prods, terms)

    def _not(self, w):
        if self.one is None:
            raise ValueError("NOT needs the `one` input: build the circuit with UIntCircuit(..., one=True)")
        return self._gate([], [w, self.one])

    def _pair(self, a, b):
        a, b = list(a), list(b)
        w = max(len(a), len(b))
        return a + [self.zero] * (w - len(a)), b + [self.zero] * (w - len(b))

    # -- operations -----------------------------------------------------------------------------------------------
    def add(self, a, b):
        """a + b mod 2^W: s = t + c, c' = a*b + t*c with t = a + b (no carry out of the top bit)."""
        a, b = self._pair(a, b)
        out, c = [], self.zero
        for i in range(len(a)):
            t = self._gate([], [a[i], b[i]])
            out.append(self._gate([], [t, c]))
            if i + 1 < len(a):
                c = self._gate([(a[i], b[i]), (t, c)], [])
        return out

    def _borrow(self, a, b, r, t):
        """borrow of a - b - r: a*b + t*r + b + r, which is (not a and b) or (not (a xor b) and r)"""
        return self._gate([(a, b), (t, r)], [b, r])

    def sub(self, a, b):
        """a - b mod 2^W: d = t + r, borrow r' = a*b + t*r + b + r."""
        a, b = self._pair(a, b)
        out, r = [], self.zero
        for i in range(len(a)):
            t = self._gate([], [a[i], b[i]])
            out.append(self._gate([], [t, r]))
            if i + 1 < len(a):
                r = self._borrow(a[i], b[i], r, t)
        return out

    def neg(self, a):
        return self.sub([self.zero] * len(a), a)

    def lt(self, a, b):
        """[a < b] (unsigned, 1 bit): the borrow out of a - b."""
        a, b = self._pair(a, b)
        r = self.zero
        for i in range(len(a)):
            t = self._gate([], [a[i], b[i]]) if r != self.zero else self.zero
            r = self._borrow(a[i], b[i], r, t)
        return [r]

    def gt(self, a, b):
        return self.lt(b, a)

    def ne(self, a, b):
        """[a != b] (1 bit): OR over the bits of a + b, o' = o + t + o*t."""
        a, b = self._pair(a, b)
        o = self.zero
        for i in range(len(a)):
            t = self._gate([], [a[i], b[i]])
            o = t if o == self.zero else self._gate([(o, t)], [o, t])
        return [o]

    def eq(self, a, b):
        return [self._not(self.ne(a, b)[0])]

    def le(self, a, b):
        return [self._not(self.gt(a, b)[0])]

    def ge(self, a, b):
        return [self._not(self.lt(a, b)[0])]

    def invert(self, a):
        return [self._not(w) for w in a]

    def select(self, s, x, y):
        """s ? x : y per bit (s one bit): s*x + s*y + y."""
        if len(s) != 1:
            raise ValueError("select needs a 1-bit condition, got %d bits" % len(s))
        x, y = self._pair(x, y)
        return [self._gate([(s[0], x[i]), (s[0], y[i])], [y[i]]) for i in range(len(x))]

    def min(self, a, b):
        return self.select(self.lt(a, b), a, b)

    def max(self, a, b):
        return self.select(self.lt(a, b), b, a)

    def mul(self, a, b):
        """a * b mod 2^W: schoolbook rows a*b_j shifted by j, each added to the accumulator with ripple carries
        (a column of three addends carries their majority, of two their product)."""
        a, b = self._pair(a, b)
        W, z = len(a), self.zero
        acc = [z] * W
        for j in range(W):
            pp = [z] * j + [self._gate([(a[i], b[j])], []) for i in range(W - j)]
            c, out = z, []
            for k in range(W):
                ops = [x for x in (acc[k], pp[k], c) if x != z]
                out.append(self._gate([], ops))
                prods = [(ops[p], ops[q]) for p in range(len(ops)) for q in range(p + 1, len(ops))]
                c = self._gate(prods, []) if prods and k + 1 < W else z
            acc = out
        return acc

    def and_(self, a, b):
        a, b = self._pair(a, b)
        return [self._gate([(x, y)], []) for x, y in zip(a, b)]

    def xor(self, a, b):
        a, b = self._pair(a, b)
        return [self._gate([], [x, y]) for x, y in zip(a, b)]

    def or_(self, a, b):
        a, b = self._pair(a, b)
        return [self._gate([(x, y)], [x, y]) for x, y in zip(a, b)]

    def shl(self, a, k):
        """a << k, keeping a's width (no gates)."""
        a, k = list(a), int(k)
        if k < 0:
            raise ValueError("negative shift")
        return ([self.zero] * k + a)[:len(a)]

    def shr(self, a, k):
        """a >> k, keeping a's width (no gates)."""
        a, k = list(a), int(k)
        if k < 0:
            raise ValueError("negative shift")
        return (a + [self.zero] * k)[k:k + len(a)]

    # -- evaluation -----------------------------------------------------------------------------------------------
    def evaluate(self, operands, results, min_bits=None, cancel=False, lane_capacity=0, one=None):
        """One Circuit.evaluate call (csgn_seg_circuit) for every result (a list of wires each): one EncryptedUInt per
        result.  operands: one EncryptedUInt per operand, of at most `width` bits (missing high bits are zero);
        one: the CiphertextArray that encrypts 1 in every lane, for a circuit built with one=True."""
        operands = list(operands)
        if len(operands) != self.n_operands:
            raise ValueError("the circuit has %d operands, got %d" % (self.n_operands, len(operands)))
        if (one is None) != (self.one is None):
            raise ValueError("the circuit was built with one=%s" % (self.one is not None))
        arrays = [one] if one is not None else []
        for x in operands:
            arrays.append(x.planes[0])
        if not arrays:
            raise ValueError("evaluate needs at least one operand or the `one` input")
        n, ctx = len(arrays[0]), arrays[0].ctx
        zero = CiphertextArray(Ciphertext.empty(0, ctx), np.zeros(n + 1, dtype=np.uint64))
        inputs = []
        for x in operands:
            if x.width > self.width:
                raise ValueError("an operand of %d bits in a %d-bit circuit" % (x.width, self.width))
            inputs += list(x.planes) + [zero] * (self.width - x.width)
        if one is not None:
            inputs.append(one)
        inputs.append(zero)
        results = [[int(w) for w in r] for r in results]
        flat = [w for r in results for w in r]
        arrs = self.circuit.evaluate(inputs, flat, min_bits, cancel, lane_capacity)
        out, at = [], 0
        for r in results:
            out.append(EncryptedUInt(arrs[at:at + len(r)]))
            at += len(r)
        return out


class EncryptedUInt:
    """A vector of n encrypted W-bit unsigned integers: W CiphertextArrays of n elements, its bit planes, LSB first
    (planes[j] element k encrypts bit j of lane k).  Made by SecretKey.encrypt_uint or UIntCircuit.evaluate, read by
    SecretKey.decrypt_uint.  The operators + - * (mod 2^W), < > (1-bit results) and & ^ | each build a one-operation
    UIntCircuit and make one call, compacted and cancelled."""

    def __init__(self, planes):
        self.planes = list(planes)
        if not self.planes:
            raise ValueError("an encrypted integer needs at least one bit plane")
        n = len(self.planes[0])
        if any(len(p) != n for p in self.planes):
            raise ValueError("bit planes of different lengths")
        self.ctx = self.planes[0].ctx

    @property
    def width(self):
        return len(self.planes)

    def __len__(self):
        return len(self.planes[0])

    @staticmethod
    def _apply(op, *xs):
        c = UIntCircuit(max(x.width for x in xs), len(xs))
        return c.evaluate(xs, [getattr(c, op)(*c.inputs)], cancel=True)[0]

    def __add__(self, other):
        return self._apply("add", self, other)

    def __sub__(self, other):
        return self._apply("sub", self, other)

    def __mul__(self, other):
        return self._apply("mul", self, other)

    def __lt__(self, other):
        return self._apply("lt", self, other)

    def __gt__(self, other):
        return self._apply("gt", self, other)

    def __and__(self, other):
        return self._apply("and_", self, other)

    def __xor__(self, other):
        return self._apply("xor", self, other)

    def __or__(self, other):
        return self._apply("or_", self, other)

    @staticmethod
    def select(c, x, y):
        """c ? x : y lane by lane, c a 1-bit EncryptedUInt."""
        if c.width != 1:
            raise ValueError("select needs a 1-bit condition, got %d bits" % c.width)
        u = UIntCircuit(max(x.width, y.width), 3)
        return u.evaluate([c, x, y], [u.select(u.inputs[0][:1], u.inputs[1], u.inputs[2])], cancel=True)[0]


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

    def encrypt_uint(self, values, width, seed, first_block=0):
        """EncryptedUInt of len(values) lanes of `width` bits (csgn_encrypt_uint: one launch, no synchronisation).
        A value that does not fit in `width` bits is an error."""
        v = np.ascontiguousarray(np.asarray(values, dtype=np.uint64).reshape(-1))
        width = int(width)
        h = (_vp * max(1, width))()
        check(_lib().csgn_encrypt_uint(self._h, v.ctypes.data_as(_vp), v.size, width, int(first_block), int(seed), h))
        off = np.arange(v.size + 1, dtype=np.uint64)
        return EncryptedUInt([CiphertextArray(Ciphertext(_vp(h[j]), self.ctx), off) for j in range(width)])

    def _uint_args(self, x):
        planes = (_vp * x.width)(*[p.storage._h for p in x.planes])
        offs = (_vp * x.width)(*[p.offsets.ctypes.data for p in x.planes])
        return planes, offs

    def decrypt_uint(self, x):
        """csgn_decrypt_uint: the lanes of x as a numpy uint64 array (one launch, one synchronisation)."""
        values = np.zeros(len(x), dtype=np.uint64)
        planes, offs = self._uint_args(x)
        check(_lib().csgn_decrypt_uint(planes, offs, x.width, len(x), self._h, values.ctypes.data_as(_vp)))
        return values

    def decrypt_uint_async(self, x, device_values_ptr):
        """csgn_decrypt_uint_async: the lanes of x to len(x) device uint64 words, no synchronisation."""
        planes, offs = self._uint_args(x)
        check(_lib().csgn_decrypt_uint_async(planes, offs, x.width, len(x), self._h, _vp(device_values_ptr)))

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
