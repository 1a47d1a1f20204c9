"""Device context and the column-planar device block (the stand-in for ``cupy.ndarray`` on this path).

A ``DeviceBlock`` is the reference's ``(3 n^3, k)`` complex128 array (lobpcg.py:365) kept on the
GPU as k independent planar columns (DESIGN.md, "Data layout in HBM").  Column slicing
``blk[:, a:b]`` / ``blk[:, [j0, j1]]`` yields views (pointer lists, no copies) -- this is what
turns the reference's soft-locking compaction (lobpcg.py:431-436) into index bookkeeping.
The reference's row-major layout exists only at ``from_host`` / ``get``.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import _lib as L

_contexts = {}
_immortal = []
_default_device = None


def set_device(device):
    """Select the CUDA device used by contexts created afterwards (one process per GPU)."""
    global _default_device
    _default_device = int(device)


def default_device():
    if _default_device is not None:
        return _default_device
    return int(os.environ.get("PCB200_DEVICE", os.environ.get("LOCAL_RANK", "0")))


class Context:
    """One GPU + one grid size N (pcb_ctx)."""

    def __init__(self, N, device=None, slab=None):
        """slab = (z0, z1): a slab context of the large-grid mode owning the i2 planes [z0, z1) of every column."""
        self.N = int(N)
        self.nn = self.N ** 3
        self.slab = None if slab is None else (int(slab[0]), int(slab[1]))
        self.nloc = self.nn if slab is None else (self.slab[1] - self.slab[0]) * self.N ** 2
        self.R = 3 * self.nloc          # rows of a column on this context
        self.device = default_device() if device is None else int(device)
        h = C.c_void_p()
        if slab is None:
            L.check(L.lib().pcb_ctx_create(self.device, self.N, C.byref(h)), "pcb_ctx_create")
        else:
            L.check(L.lib().pcb_ctx_create_slab(self.device, self.N, self.slab[0], self.slab[1], C.byref(h)), "pcb_ctx_create_slab")
        self.h = h
        self._lib = L.lib()
        self._alloc_cached = 0
        _immortal.append(self)      # see drop_contexts(): destroyed at interpreter exit only
        self._fin = weakref.finalize(self, self._lib.pcb_ctx_destroy, h)

    # -- plumbing ---------------------------------------------------------------------
    def sync(self):
        L.check(self._lib.pcb_sync(self.h), "pcb_sync")

    def option(self, name, value):
        """Pass-structure switch of this context (pcb_ctx_option); applies to operators created or updated afterwards."""
        L.check(self._lib.pcb_ctx_option(self.h, name.encode(), int(value)), "pcb_ctx_option")

    def record(self, slot):
        """Mark the work enqueued on this context's stream so far (pcb_ctx_record)."""
        L.check(self._lib.pcb_ctx_record(self.h, int(slot)), "pcb_ctx_record")

    def wait_for(self, other, slot):
        """Later work of this context starts after `other`'s mark `slot` (stream/event ordering, no host sync)."""
        L.check(self._lib.pcb_ctx_wait(self.h, other.h, int(slot)), "pcb_ctx_wait")

    def launches(self):
        n = C.c_longlong()
        L.check(self._lib.pcb_launch_count(self.h, C.byref(n)), "pcb_launch_count")
        return n.value

    def mem_info(self):
        f, t = C.c_size_t(), C.c_size_t()
        L.check(self._lib.pcb_mem_info(self.h, C.byref(f), C.byref(t)), "pcb_mem_info")
        return f.value, t.value

    def timer_start(self):
        L.check(self._lib.pcb_timer_start(self.h), "pcb_timer_start")

    def timer_stop(self):
        ms = C.c_float()
        L.check(self._lib.pcb_timer_stop(self.h, C.byref(ms)), "pcb_timer_stop")
        return ms.value

    # Block allocations are recycled by exact size: cudaMalloc + cudaFree of a 1.3 GB block cost ~40 ms each on B200 (the free
    # synchronises the device and unmaps), and a band-structure run allocates and drops a few such blocks per k-point (the
    # solver's result copy, A(x) of the post-processing) -- 80 ms per k-point against 230 ms of solve before this cache.
    # Everything runs on the context's one stream, so handing a freed block to the next user is ordered.
    ALLOC_CACHE_BYTES = int(float(os.environ.get("PCB200_ALLOC_CACHE_GB", "8")) * 2 ** 30)

    def malloc(self, nbytes):
        cache = self.__dict__.setdefault("_alloc_cache", {})
        lst = cache.get(nbytes)
        if lst:
            self._alloc_cached -= nbytes
            return lst.pop()
        p = C.c_void_p()
        rc = self._lib.pcb_malloc(self.h, nbytes, C.byref(p))
        if rc != 0 and self.trim():
            rc = self._lib.pcb_malloc(self.h, nbytes, C.byref(p))      # out of memory: give the cached blocks back and retry
        L.check(rc, f"pcb_malloc({nbytes})")
        return p.value

    def free(self, ptr, nbytes=0):
        """Return an allocation: blocks of at least 1 MiB go to the size-keyed cache (up to ALLOC_CACHE_BYTES)."""
        held = self.__dict__.setdefault("_alloc_cached", 0)
        if nbytes >= (1 << 20) and held + nbytes <= self.ALLOC_CACHE_BYTES:
            self.__dict__.setdefault("_alloc_cache", {}).setdefault(nbytes, []).append(ptr)
            self._alloc_cached = held + nbytes
            return
        L.check(self._lib.pcb_free(self.h, ptr), "pcb_free")

    def trim(self):
        """cudaFree every cached block and the context's cached band-velocity columns (pcb_ctx_trim); returns the number of
        bytes released."""
        cache = self.__dict__.get("_alloc_cache", {})
        freed = int(self._lib.pcb_ctx_trim(self.h))
        for nbytes, lst in cache.items():
            while lst:
                self._lib.pcb_free(self.h, lst.pop())
                freed += nbytes
        self._alloc_cached = 0
        return freed

    # -- blocks -------------------------------------------------------------------------
    def empty(self, k):
        return DeviceBlock(self, int(k))

    def work_block(self, tag, k):
        """A cached k-column block (solver work space S / HS): cudaMalloc/cudaFree of several GB per k-point would cost
        as much as a few LOBPCG iterations.  The caller must not keep views beyond its own call."""
        pool = self.__dict__.setdefault("_work_blocks", {})
        blk = pool.get(tag)
        if blk is None or blk.k < k:
            pool[tag] = None          # release the smaller block first
            blk = pool[tag] = DeviceBlock(self, int(k))
            hook = getattr(self, "_on_work_block", None)      # large-grid mode: map the solver's work space into all ranks
            if hook is not None:
                hook(blk)
        return blk if blk.k == k else blk.cols(range(k))

    def from_host(self, x):
        return DeviceBlock.from_host(self, x)

    def random_block(self, k, seed):
        """x0 = rand + 1j*rand on the device (numerical_experiments.py:66)."""
        b = DeviceBlock(self, int(k))
        L.check(self._lib.pcb_fill_uniform(self.h, b.k, L.ptr_array(b.ptrs), int(seed)), "pcb_fill_uniform")
        return b


def get_context(N, device=None):
    """Cached context for (device, N)."""
    dev = default_device() if device is None else int(device)
    key = (L.lib_path(), dev, int(N))
    if key not in _contexts:
        _contexts[key] = Context(N, dev)
    return _contexts[key]


def drop_contexts():
    """Synchronise every cached context.  Contexts are deliberately never destroyed before interpreter exit:
    blocks, operators and dielectric handles point into them, and Python may finalise a garbage cycle in any
    order (at exit, weakref.finalize runs in reverse creation order, i.e. contexts last)."""
    for ctx in _contexts.values():
        ctx.sync()


class _Allocation:
    """Owner of one cudaMalloc; freed when the last view dies."""

    def __init__(self, ctx, nbytes):
        self.ctx = ctx
        self.ptr = ctx.malloc(nbytes)
        self._fin = weakref.finalize(self, _free, ctx, self.ptr, nbytes)


def _free(ctx, ptr, nbytes=0):
    try:
        ctx.free(ptr, nbytes)
    except Exception:
        pass


class DeviceBlock:
    """k planar columns of 3 N^3 complex128 on the GPU; behaves like an (R, k) array for the
    operations the hot path uses (shape, column slicing, get/set, copy)."""

    __array_priority__ = 1000

    def __init__(self, ctx, k=None, _owners=None, _ptrs=None, vec=False):
        self.ctx = ctx
        self.vec = vec          # True: presents itself as a 1-D vector of length R
        if _ptrs is None:
            a = _Allocation(ctx, 16 * ctx.R * max(k, 1))
            self._owners = (a,)
            self.ptrs = [a.ptr + 16 * ctx.R * j for j in range(k)]
        else:
            self._owners = _owners
            self.ptrs = list(_ptrs)

    # -- array-like surface ---------------------------------------------------------------
    @property
    def k(self):
        return len(self.ptrs)

    @property
    def shape(self):
        return (self.ctx.R,) if self.vec else (self.ctx.R, self.k)

    @property
    def ndim(self):
        return 1 if self.vec else 2

    dtype = np.dtype(np.complex128)

    def cols(self, idx):
        """View of the listed columns."""
        return DeviceBlock(self.ctx, _owners=self._owners, _ptrs=[self.ptrs[int(j)] for j in idx])

    def __getitem__(self, key):
        if isinstance(key, tuple) and len(key) == 2 and key[0] == slice(None):
            c = key[1]
            if isinstance(c, slice):
                return self.cols(range(*c.indices(self.k)))
            if isinstance(c, (int, np.integer)):
                v = self.cols([c])
                v.vec = True
                return v
            return self.cols(list(c))
        raise IndexError("DeviceBlock supports column selection only: blk[:, a:b], blk[:, j], blk[:, [..]]")

    def __setitem__(self, key, value):
        dst = self[key]
        if isinstance(value, DeviceBlock):
            dst.assign(value)
        else:
            dst.set(np.asarray(value))

    def assign(self, src):
        """Column-wise device copy src -> self."""
        if src.k != self.k:
            raise ValueError(f"column count mismatch {src.k} vs {self.k}")
        lib = L.lib()
        for d, s in zip(self.ptrs, src.ptrs):
            if d != s:
                L.check(lib.pcb_memcpy_d2d(self.ctx.h, d, s, 16 * self.ctx.R), "pcb_memcpy_d2d")

    def copy(self):
        out = DeviceBlock(self.ctx, self.k, vec=self.vec)
        out.assign(self)
        return out

    def set(self, host):
        host = np.ascontiguousarray(host, dtype=np.complex128)
        if host.ndim == 1:
            host = host.reshape(-1, 1)
        if host.shape != (self.ctx.R, self.k):
            raise ValueError(f"host block has shape {host.shape}, expected {(self.ctx.R, self.k)}")
        L.check(L.lib().pcb_block_upload(self.ctx.h, host.ctypes.data, host.shape[1], self.k, L.ptr_array(self.ptrs)),
                "pcb_block_upload")

    def get(self, out=None):
        """Row-major (R, k) NumPy copy (``cupy.ndarray.get``)."""
        if out is None:
            out = np.empty((self.ctx.R, self.k), dtype=np.complex128)
        L.check(L.lib().pcb_block_download(self.ctx.h, out.ctypes.data, out.shape[1], self.k, L.ptr_array(self.ptrs)),
                "pcb_block_download")
        return out.reshape(-1) if self.vec else out

    def __array__(self, dtype=None, copy=None):
        a = self.get()
        return a if dtype is None else a.astype(dtype)

    @staticmethod
    def from_host(ctx, x):
        x = np.asarray(x)
        vec = x.ndim == 1
        b = DeviceBlock(ctx, 1 if vec else x.shape[1], vec=vec)
        b.set(x)
        return b


_pinned = {}


def pinned_empty(shape, dtype=np.complex128):
    """NumPy array over page-locked host memory (pcb_host_alloc) for full-speed H2D/D2H.
    The buffer lives until pinned_free(arr) or process exit."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    L.check(L.lib().pcb_host_alloc(max(n, 1), C.byref(p)), "pcb_host_alloc")
    buf = (C.c_char * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    _pinned[arr.ctypes.data] = (p.value, buf)
    return arr


def pinned_free(arr):
    ent = _pinned.pop(arr.ctypes.data, None)
    if ent is not None:
        L.check(L.lib().pcb_host_free(ent[0]), "pcb_host_free")


def as_block(ctx, x):
    """Device view of x: DeviceBlock stays, NumPy arrays are uploaded.  Returns (block, was_host)."""
    if isinstance(x, DeviceBlock):
        if x.ctx is not ctx:
            raise ValueError("block belongs to another context (grid size / device)")
        return x, False
    return DeviceBlock.from_host(ctx, x), True
