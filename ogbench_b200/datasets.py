"""Host-side mirror of the reference sampler API (impls/utils/datasets.py) over the CUDA library.

Same names, arguments, key sets, shapes and dtypes as the reference:

    dataset = Dataset.create(**fields)                       # datasets.py:45-57
    sampler = GCDataset(dataset, config)                     # datasets.py:149-211   (HGCDataset: :467-643)
    batch = sampler.sample(batch_size, idxs=None, evaluation=False)

What differs is where things live: the fields are uploaded once and stay resident in HBM, the whole of
``sample()`` is one or two CUDA launches, and the returned dict holds device arrays (``DeviceArray``: DLPack +
``__cuda_array_interface__``; ``output='numpy'`` copies the batch to host like the reference returns it).
Keyword-only extras (``device``, ``seed``, ``stream_id``, ``rng``, ``output``, ``dedup``) have defaults that keep
reference call sites working unchanged.  There is no CPU implementation behind this module.
"""

from __future__ import annotations

import collections
import ctypes as C
import weakref
from typing import Any, Dict, Mapping

import numpy as np

from . import _native
from .device_array import BatchHandle, DeviceArray

TRL_AGENTS = ('trl', 'latent_trl', 'discrete_latent_trl')


SEP = '/'   # path separator of flattened pytree fields: {'observations': {'image': a, 'state': b}} -> 'observations/image', ...


def _leaves(tree, prefix=''):
    """(path, leaf) pairs of a nested dict, keys sorted like jax's dict flattening (datasets.py:13,80 map over pytrees)."""
    if isinstance(tree, Mapping):
        for k in sorted(tree):
            yield from _leaves(tree[k], f'{prefix}{SEP}{k}' if prefix else str(k))
    else:
        yield prefix, tree


def _flatten(fields) -> Dict[str, Any]:
    return dict(_leaves(fields))


def _nest(flat: Dict[str, Any]) -> Dict[str, Any]:
    """Inverse of _flatten for a batch: 'value_goals/image' -> batch['value_goals']['image']."""
    out: Dict[str, Any] = {}
    for path, v in flat.items():
        parts = path.split(SEP)
        node = out
        for p in parts[:-1]:
            node = node.setdefault(p, {})
        node[parts[-1]] = v
    return out


def get_size(data) -> int:
    """Return the size of the dataset: the longest leaf of the field pytree (datasets.py:11-14)."""
    return max(len(v) for _, v in _leaves(data))


def _is_device_array(x) -> bool:
    return not isinstance(x, np.ndarray) and (hasattr(x, '__cuda_array_interface__') or hasattr(x, 'data_ptr'))


def ring_plan(pointer: int, size: int, max_size: int, n: int):
    """(row0, skip, pointer, size) of n add_transition calls on a ring of max_size rows (datasets.py:134-142): rows
    (row0 + i) % max_size for i in [skip, n) are written (only the last max_size transitions survive), and pointer and size
    end where n single calls leave them -- size = max(pointer, size) after every call, so it never reaches max_size
    through a wrap (:141-142)."""
    if n == 0:
        return pointer, 0, pointer, size
    end = pointer + n
    if end < max_size:                       # no wrap: the largest pointer visited is the last one
        top = end
    elif pointer <= max_size - 2:            # the pointer passes max_size - 1 before it wraps to 0
        top = max_size - 1
    else:                                    # it starts at max_size - 1: 0, 1, ..., n - 1 after that
        top = min(n - 1, max_size - 1)
    return pointer, max(0, n - max_size), end % max_size, max(size, top)


_KDL_CUDA = 2
_DL_DTYPES = {(0, 8): np.int8, (0, 16): np.int16, (0, 32): np.int32, (0, 64): np.int64, (1, 8): np.uint8, (1, 16): np.uint16,
              (1, 32): np.uint32, (1, 64): np.uint64, (2, 16): np.float16, (2, 32): np.float32, (2, 64): np.float64,
              (6, 8): np.bool_}


def _is_device_leaf(x) -> bool:
    """A CUDA array (DLPack device kDLCUDA, or __cuda_array_interface__ without DLPack); CPU tensors are host leaves."""
    if isinstance(x, np.ndarray):
        return False
    if hasattr(x, '__dlpack_device__') and hasattr(x, '__dlpack__'):
        return x.__dlpack_device__()[0] == _KDL_CUDA
    return hasattr(type(x), '__cuda_array_interface__')   # (on the type: evaluating the property may synchronise)


def _c_contiguous(shape, strides, itemsize) -> bool:
    """strides in bytes; dimensions of length 1 may carry any stride."""
    step = itemsize
    for n, st in zip(reversed(shape), reversed(strides)):
        if n != 1 and st != step:
            return False
        step *= n
    return True


def _device_source(name, leaf, dtype, shape, device, stream):
    """(pointer, keepalive, producer stream or None) of a device leaf, which must already have the field's dtype, the row
    shape `shape` and be C-contiguous (no cast on the device).  DLPack leaves are exported with `stream` as the consumer,
    so the producer orders its writes before the sampler's stream reads them."""
    from .device_array import _DLManagedTensorHead, _PyCapsule_GetPointer

    if hasattr(leaf, '__dlpack__'):
        dev_type, dev_id = leaf.__dlpack_device__()
        if dev_id != device:
            raise ValueError(f'field {name!r}: the leaf lives on cuda:{dev_id}, the buffer on cuda:{device}')
        capsule = leaf.__dlpack__(stream=stream)
        head = _DLManagedTensorHead.from_address(_PyCapsule_GetPointer(capsule, b'dltensor'))
        got_dtype = _DL_DTYPES.get((head.code, head.bits)) if head.lanes == 1 else None
        got_shape = tuple(C.cast(head.shape, C.POINTER(C.c_int64))[d] for d in range(head.ndim))
        itemsize = head.bits // 8
        strides = (None if not head.strides else
                   tuple(C.cast(head.strides, C.POINTER(C.c_int64))[d] * itemsize for d in range(head.ndim)))
        ptr, keep, producer = (head.data or 0) + head.byte_offset, capsule, None
    else:
        cai = leaf.__cuda_array_interface__
        got_dtype, got_shape = np.dtype(cai['typestr']), tuple(cai['shape'])
        strides = None if cai.get('strides') is None else tuple(cai['strides'])
        ptr, keep, producer = cai['data'][0], leaf, cai.get('stream')
    if got_dtype is None or np.dtype(got_dtype) != dtype:
        raise ValueError(f'field {name!r}: device leaves must already have the dtype {dtype} (got {got_dtype}); '
                         'there is no cast on the device')
    if got_shape != tuple(shape):
        raise ValueError(f'field {name!r}: expected a device leaf of shape {tuple(shape)}, got {got_shape}')
    if strides is not None and not _c_contiguous(got_shape, strides, dtype.itemsize):
        raise ValueError(f'field {name!r}: device leaves must be C-contiguous')
    return ptr, keep, producer


class _ZeroField:
    """Placeholder for a field that is allocated zero-filled on the device (ReplayBuffer.create)."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)

    def __len__(self):
        return self.shape[0]


def _describe_field(name: str, arr, keepalive: list) -> _native.Field:
    f = _native.Field()
    f.name = name.encode()
    if isinstance(arr, _ZeroField):
        np_dtype, shape, ptr = arr.dtype, arr.shape, None
        f.on_device = 2
    elif _is_device_array(arr):
        if hasattr(arr, 'data_ptr'):  # torch tensor
            if not arr.is_cuda or not arr.is_contiguous():
                raise ValueError(f'field {name!r}: device tensors must be contiguous CUDA tensors')
            import torch

            np_dtype = np.dtype(str(arr.dtype).replace('torch.', '').replace('bool', 'bool_'))
            shape, ptr = tuple(arr.shape), arr.data_ptr()
            torch.cuda.current_stream(arr.device).synchronize()
        else:
            cai = arr.__cuda_array_interface__
            if cai.get('strides') is not None:
                raise ValueError(f'field {name!r}: device arrays must be C-contiguous')
            np_dtype, shape, ptr = np.dtype(cai['typestr']), tuple(cai['shape']), cai['data'][0]
        f.on_device = 1
    else:
        arr = np.ascontiguousarray(arr)
        np_dtype, shape, ptr = arr.dtype, arr.shape, arr.ctypes.data
        f.on_device = 0
    keepalive.append(arr)
    if np_dtype not in _native.DTYPE_TO_CODE:
        raise TypeError(f'field {name!r}: unsupported dtype {np_dtype}')
    if not 1 <= len(shape) <= _native.OGB_MAX_NDIM:
        raise ValueError(f'field {name!r}: unsupported rank {len(shape)}')
    f.data = ptr
    f.dtype = _native.DTYPE_TO_CODE[np_dtype]
    f.ndim = len(shape)
    for d, n in enumerate(shape):
        f.shape[d] = n
    return f


class _NativeDataset:
    """Owns the ogb_dataset handle (the HBM-resident copy)."""

    def __init__(self, fields: Mapping[str, Any], device: int):
        _native.require_device()
        keepalive: list = []
        descs = (_native.Field * len(fields))(*[_describe_field(k, v, keepalive) for k, v in fields.items()])
        out = C.c_void_p()
        _native.check(_native.lib().ogb_dataset_create(descs, len(fields), device, C.byref(out)))
        self.ptr = out
        self.device = device

    @classmethod
    def empty(cls, fields: Mapping[str, '_ZeroField'], device: int) -> '_NativeDataset':
        """ogb_dataset_create_empty: the layout of `fields` (shape[0] = capacity), rows written later, tables built at seal."""
        _native.require_device()
        keepalive: list = []
        descs = (_native.Field * len(fields))(*[_describe_field(k, v, keepalive) for k, v in fields.items()])
        out = C.c_void_p()
        _native.check(_native.lib().ogb_dataset_create_empty(descs, len(fields), device, C.byref(out)))
        return cls._adopt(out, device)

    def view(self, row0: int, n_rows: int) -> '_NativeDataset':
        """ogb_dataset_view: rows [row0, row0 + n_rows) of this (sealed) dataset as a dataset of their own."""
        out = C.c_void_p()
        _native.check(_native.lib().ogb_dataset_view(self.ptr, int(row0), int(n_rows), C.byref(out)))
        return self._adopt(out, self.device)

    @classmethod
    def _adopt(cls, ptr, device) -> '_NativeDataset':
        self = cls.__new__(cls)
        self.ptr, self.device = ptr, device
        return self

    def size(self) -> int:
        n = C.c_int64()
        _native.check(_native.lib().ogb_dataset_size(self.ptr, C.byref(n)))
        return n.value

    def resident_bytes(self) -> int:
        n = C.c_size_t()
        _native.check(_native.lib().ogb_dataset_resident_bytes(self.ptr, C.byref(n)))
        return n.value

    def __del__(self):
        ptr, self.ptr = getattr(self, 'ptr', None), None
        if ptr:
            try:
                _native.lib().ogb_dataset_destroy(ptr)
            except Exception:
                pass


class Dataset(Mapping):
    """Immutable field dict (the reference's FrozenDict-based Dataset, datasets.py:36-83).

    Supports compact datasets (no 'next_observations'; 'valids' masks each trajectory's last row) and regular ones.
    Field values may be numpy arrays (uploaded once) or CUDA arrays (torch tensors / __cuda_array_interface__).
    """

    @classmethod
    def create(cls, freeze=True, **fields):
        data = fields
        assert 'observations' in data
        if freeze:
            for _, arr in _leaves(data):
                if isinstance(arr, np.ndarray):
                    arr.setflags(write=False)
        return cls(data)

    def __init__(self, *args, **kwargs):
        if len(args) == 1 and isinstance(args[0], Dataset) and not kwargs:
            self._dict = dict(args[0]._dict)
        else:
            self._dict = dict(*args, **kwargs)
        # nested dicts (pytree fields, e.g. observations = {'image': ..., 'state': ...}) are flattened into one resident field
        # per leaf; every key derived from them comes back nested the same way
        self._nested = any(isinstance(v, Mapping) for v in self._dict.values())
        self.size = get_size(self._dict)
        if 'valids' in self._dict and isinstance(self._dict['valids'], np.ndarray):
            (self.valid_idxs,) = np.nonzero(self['valids'] > 0)
        self._native: Dict[int, _NativeDataset] = {}
        self._plain: Dict[int, '_Sampler'] = {}

    # ---- Mapping ----
    def __getitem__(self, key):
        return self._dict[key]

    def __iter__(self):
        return iter(self._dict)

    def __len__(self):
        return len(self._dict)

    def copy(self, add_or_replace=None):
        merged = dict(self._dict)
        merged.update(add_or_replace or {})
        return type(self)(merged)

    # ---- reference API ----
    def get_random_idxs(self, num_idxs):
        """Return `num_idxs` random indices from the global np.random stream (datasets.py:65-70)."""
        if hasattr(self, 'valid_idxs'):
            return self.valid_idxs[np.random.randint(len(self.valid_idxs), size=num_idxs)]
        return np.random.randint(self.size, size=num_idxs)

    def native(self, device: int = 0) -> _NativeDataset:
        if device not in self._native:
            self._native[device] = _NativeDataset(_flatten(self._dict) if self._nested else self._dict, device)
        return self._native[device]

    def _plain_sampler(self, device=0) -> '_Sampler':
        if device not in self._plain:
            self._plain[device] = _Sampler(self, None, _native.KIND_PLAIN, device=device, output=self.output)
        return self._plain[device]

    rng = 'philox'     # 'numpy': draw the indices on the host from np.random, exactly like the reference
    output = 'device'  # 'numpy': return host arrays like the reference

    def sample(self, batch_size, idxs=None):
        """Sample a batch of transitions (datasets.py:72-76)."""
        if idxs is None and self.rng == 'numpy':
            idxs = self.get_random_idxs(batch_size)
        return self._plain_sampler().sample(batch_size, idxs)

    def get_subset(self, idxs):
        """Return the rows `idxs` of every field plus next_observations (datasets.py:78-83)."""
        idxs = np.asarray(idxs, dtype=np.int64)
        return self._plain_sampler().sample(len(idxs), idxs)


class ResidentDataset(Dataset):
    """A Dataset whose fields live only in HBM (built by loader.ResidentShards): a whole directory of shards, or the view
    of one shard inside it.

    The host side keeps what it needs and no copy of the fields: `size`, one byte per row of `valids` (get_random_idxs
    under rng='numpy') and the field names.  Indexing a field raises, as for ReplayBuffer.  Samplers are created on the
    device the table lives on; any other device is refused.
    """

    def __init__(self, nds: _NativeDataset, keys, nested: bool, valids):
        self._dict = {}
        self._keys = list(keys)
        self._nested = nested
        self.device = nds.device
        self.size = nds.size()
        self._valids = valids               # uint8 [size] (valids > 0), or None when the dataset has no 'valids'
        self._valid_idxs = None
        self._native = {nds.device: nds}
        self._plain = {}

    @property
    def valid_idxs(self):
        if self._valids is None:
            raise AttributeError('valid_idxs')
        if self._valid_idxs is None:
            self._valid_idxs = np.flatnonzero(self._valids)
        return self._valid_idxs

    def __getitem__(self, key):
        raise NotImplementedError(f'field {key!r}: a resident dataset keeps no host copy of its fields')

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)

    def copy(self, add_or_replace=None):
        raise NotImplementedError('a resident dataset keeps no host copy of its fields to copy')

    def native(self, device: int = 0) -> _NativeDataset:
        if device not in self._native:
            raise ValueError(f'the dataset is resident on device {self.device}; a sampler on device {device} cannot read it')
        return self._native[device]

    def _plain_sampler(self, device=None) -> '_Sampler':
        return super()._plain_sampler(self.device if device is None else device)


class ReplayBuffer(Dataset):
    """Replay buffer class, device-resident (reference: datasets.py:86-146).

    The buffers live in HBM; `add_transition` writes one row per field, stream-ordered with `sample`.  Indexing the
    buffer (`rb['observations']`) is not supported: there is no host mirror.
    """

    @classmethod
    def create(cls, transition, size, **kwargs):
        """Create a replay buffer from the example transition (datasets.py:92-106)."""
        fields = {k: _ZeroField((size, *np.array(v).shape), np.array(v).dtype) for k, v in _leaves(transition)}   # pytrees: one buffer per leaf
        return cls(fields, **kwargs)

    @classmethod
    def create_from_initial_dataset(cls, init_dataset, size, **kwargs):
        """Create a replay buffer from the initial dataset (datasets.py:108-125)."""
        init = {k: np.asarray(v) for k, v in _leaves(dict(init_dataset))}
        n = get_size(init)

        def create_buffer(init_buffer):
            buffer = np.zeros((size, *init_buffer.shape[1:]), dtype=init_buffer.dtype)
            buffer[:len(init_buffer)] = init_buffer
            return buffer

        rb = cls({k: create_buffer(v) for k, v in init.items()}, **kwargs)
        rb.size = rb.pointer = n
        rb.native(rb._device)            # one bulk upload per field (not a write per row); active rows = n
        rb._dict = {k: _ZeroField(v.shape, v.dtype) for k, v in rb._dict.items()}   # the host copies are not kept
        return rb

    def __init__(self, fields, rng='philox', output='device', device=0):
        self._dict = dict(fields)
        self._nested = any(SEP in k for k in self._dict)      # leaves of pytree transitions, flattened by create()
        self.rng, self.output, self._device = rng, output, device
        self.max_size = get_size(self._dict)
        self.size = 0
        self.pointer = 0
        self._native = {}
        self._plain = {}
        self._names = list(self._dict)

    def __getitem__(self, key):
        raise NotImplementedError('the device ReplayBuffer keeps no host mirror of its buffers')

    def native(self, device: int = 0) -> _NativeDataset:
        fresh = device not in self._native
        nds = super().native(device)
        if fresh:  # a new buffer holds no rows yet (datasets.py:131)
            _native.check(_native.lib().ogb_dataset_set_active_rows(nds.ptr, int(self.size)))
        return nds

    def _sync_size(self):
        _native.check(_native.lib().ogb_dataset_set_active_rows(self.native(self._device).ptr, int(self.size)))

    def _write(self, row, transition):
        sampler = self._plain_sampler(self._device)
        ptrs = (C.c_void_p * len(self._names))()
        keep = []
        if self._nested:
            transition = _flatten(transition)
        for i, name in enumerate(self._names):
            zf = self._dict[name]
            arr = np.ascontiguousarray(np.asarray(transition[name]), dtype=zf.dtype).reshape(zf.shape[1:])
            keep.append(arr)
            ptrs[i] = arr.ctypes.data
        _native.check(_native.lib().ogb_sampler_write_row(sampler.ptr, int(row), ptrs, len(self._names)))

    def add_transition(self, transition):
        """Add a transition to the replay buffer (datasets.py:134-142).  Leaves on the buffer's GPU (torch, JAX, CuPy) are
        read in place, with the rules of add_transitions."""
        if any(_is_device_leaf(v) for _, v in _leaves(transition)):
            self._write_ring(transition, single=True)
            return
        self._write(self.pointer, transition)
        self.pointer = (self.pointer + 1) % self.max_size
        self.size = max(self.pointer, self.size)
        self._sync_size()

    def add_transitions(self, transitions):
        """Add n transitions at once: `transitions` is a dict (or pytree) like add_transition's whose leaves carry a
        leading axis of length n.  Same effect as `for i in range(n): add_transition({k: v[i] ...})` -- rows, `pointer` and
        `size` included -- in one stream-ordered launch.

        numpy leaves are cast to the field's dtype as add_transition casts them.  Leaves on the buffer's GPU (anything with
        `__dlpack__` or `__cuda_array_interface__`: torch, JAX, CuPy) are read in place, after the work their producer has
        issued so far; they must already have the field's dtype and row shape and be C-contiguous (ValueError otherwise:
        there is no cast on the device).  Host and device leaves may be mixed.  The call does not wait for the GPU: the
        library keeps device leaves referenced until the write has read them."""
        self._write_ring(transitions, single=False)

    def _write_ring(self, transitions, single):
        sampler = self._plain_sampler(self._device)
        if self._nested:
            transitions = _flatten(transitions)
        leaves = [transitions[name] for name in self._names]          # a missing key is a KeyError, as in tree_map
        lengths, hosts, devices = {}, {}, {}
        for name, leaf in zip(self._names, leaves):
            zf = self._dict[name]
            if _is_device_leaf(leaf):
                devices[name] = leaf
                continue
            arr = np.asarray(leaf)
            if single:
                arr = arr.reshape(1, *zf.shape[1:])
            elif arr.ndim == 0:
                raise ValueError(f'field {name!r}: add_transitions needs a leading axis of transitions')
            try:
                hosts[name] = np.ascontiguousarray(arr, dtype=zf.dtype).reshape(len(arr), *zf.shape[1:])
            except ValueError as exc:
                raise ValueError(f'field {name!r}: rows of shape {zf.shape[1:]} expected ({exc})') from None
            lengths[name] = len(arr)
        stream, keep, producers = None, [], set()
        ptrs = (C.c_void_p * len(self._names))()
        on_device = (C.c_int32 * len(self._names))()
        for i, name in enumerate(self._names):
            if name in hosts:
                ptrs[i] = hosts[name].ctypes.data
                continue
            leaf, zf = devices[name], self._dict[name]
            if single:
                rows = zf.shape[1:]
            else:
                shape = tuple(getattr(leaf, 'shape', ()))
                if not shape:
                    raise ValueError(f'field {name!r}: add_transitions needs a leading axis of transitions')
                rows = (shape[0], *zf.shape[1:])
            if stream is None:
                handle = C.c_void_p()
                _native.check(_native.lib().ogb_sampler_get_stream(sampler.ptr, C.byref(handle)))
                stream = handle.value or 1                             # (DLPack's name for the legacy default stream)
            ptrs[i], src, producer = _device_source(name, leaf, zf.dtype, rows, self._device, stream)
            on_device[i] = 1
            keep.append(src)
            if producer is not None:
                producers.add(producer)
            lengths[name] = 1 if single else rows[0]
        if len(set(lengths.values())) > 1:
            raise ValueError(f'the leaves hold different numbers of transitions: {lengths}')
        if len(producers) > 1:
            raise ValueError('device leaves produced on different streams (__cuda_array_interface__ "stream"): pass them in separate calls')
        n = next(iter(lengths.values())) if lengths else 0
        if n == 0:
            return
        row0, skip, pointer, size = ring_plan(self.pointer, self.size, self.max_size, n)
        ticket, retired = C.c_uint64(), C.c_uint64()
        _native.check(_native.lib().ogb_sampler_write_ring(
            sampler.ptr, row0, n, skip, ptrs, len(self._names), on_device, C.c_void_p(producers.pop() if producers else None),
            C.byref(ticket), C.byref(retired)))
        in_flight = sampler._in_flight
        if keep:
            in_flight.append((ticket.value, keep))
        while in_flight and in_flight[0][0] <= retired.value:
            in_flight.popleft()
        self.pointer, self.size = pointer, size
        self._sync_size()

    def clear(self):
        """Clear the replay buffer (datasets.py:144-146)."""
        self.size = self.pointer = 0
        self._sync_size()

    def get_random_idxs(self, num_idxs):
        return np.random.randint(self.size, size=num_idxs)  # no 'valids' in a replay buffer: datasets.py:70

    def sample(self, batch_size, idxs=None):
        if idxs is None and self.rng == 'numpy':
            idxs = self.get_random_idxs(batch_size)
        return self._plain_sampler(self._device).sample(batch_size, idxs)


class _PinnedPool:
    """Reusable page-locked host blocks for output='numpy'.

    Block sizes are rounded up to one of eight steps per power of two (at most 12.5 % slack; a 545 MB batch pins 576 MB,
    not 1 GiB), returned blocks are kept for the next call of the same size class, and the pool gives page-locked
    memory back to the system once more than `max_idle_bytes` of it sits unused.
    """

    max_idle_bytes = 4 << 30

    def __init__(self):
        self.free: Dict[int, list] = {}
        self.idle_bytes = 0

    @staticmethod
    def bucket_of(nbytes: int) -> int:
        bits = (max(nbytes, 1) - 1).bit_length()
        if bits <= 12:
            return 4096
        step = 1 << (bits - 4)
        return -(-nbytes // step) * step

    def take(self, nbytes: int) -> '_PinnedBlock':
        bucket = self.bucket_of(nbytes)
        stack = self.free.setdefault(bucket, [])
        if stack:
            self.idle_bytes -= bucket
            return _PinnedBlock(self, bucket, stack.pop())
        out = C.c_void_p()
        _native.check(_native.lib().ogb_host_alloc(bucket, C.byref(out)))
        return _PinnedBlock(self, bucket, out.value)

    def give_back(self, bucket: int, ptr: int):
        if self.idle_bytes + bucket > self.max_idle_bytes:
            _native.lib().ogb_host_free(C.c_void_p(ptr))
            return
        self.free.setdefault(bucket, []).append(ptr)
        self.idle_bytes += bucket


class _PinnedBlock:
    def __init__(self, pool, bucket, ptr):
        self.pool, self.bucket, self.ptr = pool, bucket, ptr

    def __del__(self):
        try:
            self.pool.give_back(self.bucket, self.ptr)
        except Exception:  # interpreter shutdown
            pass


_PINNED = _PinnedPool()


def _destroy_sampler(ptr, in_flight):
    _native.lib().ogb_sampler_destroy(ptr)      # (waits for the sampler's stream)
    in_flight.clear()


class _Sampler:
    """Thin owner of an ogb_sampler handle; builds the C config from the reference's config mapping."""

    def __init__(self, dataset: Dataset, config, kind: int, device: int = 0, seed: int = 0, stream_id: int = 0,
                 dedup: bool = True, output: str = 'device', crop_padding: int = 3, jax_compat: bool = False):
        assert output in ('device', 'numpy')
        self.dataset = dataset
        self.kind = kind
        self.device = device
        self.output = output
        self.nested = bool(getattr(dataset, '_nested', False))   # pytree fields: batches are re-nested on the way out
        self._keepalive = []
        cfg = _native.Config()
        cfg.dedup_keys = int(dedup)
        cfg.jax_compat = int(bool(jax_compat))
        cfg.crop_padding = crop_padding  # 3 in GCDataset.augment (datasets.py:331); ATC: config['augment_padding'] (:440)
        if kind == _native.KIND_ATC:
            p_aug = config['p_aug']
            cfg.has_p_aug = int(p_aug is not None)
            cfg.p_aug = float(p_aug) if p_aug is not None else 0.0
            fs = config['frame_stack']
            cfg.frame_stack = int(fs) if fs is not None else 0
        elif kind != _native.KIND_PLAIN:
            cfg.discount = float(config['discount'])
            for side in ('value', 'actor'):
                for part in ('cur', 'traj', 'random'):
                    setattr(cfg, f'{side}_p_{part}goal', float(config[f'{side}_p_{part}goal']))
                setattr(cfg, f'{side}_geom_sample', int(bool(config[f'{side}_geom_sample'])))
            cfg.gc_negative = int(bool(config['gc_negative']))
            p_aug = config['p_aug']
            cfg.has_p_aug = int(p_aug is not None)
            cfg.p_aug = float(p_aug) if p_aug is not None else 0.0
            fs = config['frame_stack']
            cfg.frame_stack = int(fs) if fs is not None else 0
            cfg.trl = int(kind == _native.KIND_GC and config.get('agent_name') in TRL_AGENTS)
        if kind == _native.KIND_HGC:
            # datasets.py:515-518, :543, :592-594 -- the optional overrides, resolved as the reference resolves them
            high = config.get('high_subgoal_steps', config['subgoal_steps'])
            value = high if config.get('value_subgoal_steps') is None else config['value_subgoal_steps']
            actor = high if config.get('actor_subgoal_steps') is None else config['actor_subgoal_steps']
            low = config.get('low_subgoal_steps', config['subgoal_steps'])
            cfg.value_subgoal_steps, cfg.actor_subgoal_steps, cfg.low_subgoal_steps = int(value), int(actor), int(low)
            low_discount = config.get('low_discount')
            cfg.has_low_discount = int(low_discount is not None)
            cfg.low_discount = float(low_discount) if low_discount is not None else 0.0
            # numpy's own `discount ** steps` (its SIMD pow is not libm's), evaluated exactly as datasets.py:537-541
            steps = np.arange(max(value, actor, low) + 1)
            discount = config['discount']
            neg = np.ascontiguousarray(-(1 - discount**steps) / (1 - discount), dtype=np.float64)
            pw = np.ascontiguousarray(discount**steps, dtype=np.float64)
            self._keepalive += [neg, pw]
            cfg.lut_len = len(steps)
            cfg.neg_reward_lut = neg.ctypes.data_as(C.POINTER(C.c_double))
            cfg.pow_lut = pw.ctypes.data_as(C.POINTER(C.c_double))
        self._cfg = cfg
        self._nds = dataset.native(device)
        out = C.c_void_p()
        _native.check(_native.lib().ogb_sampler_create(self._nds.ptr, C.byref(cfg), kind, seed, stream_id, C.byref(out)))
        self.ptr = out
        # (ticket, sources) of ogb_sampler_write_ring calls whose device sources the stream may still read: released once the
        # library reports the call retired, or after the sampler (and with it its stream) is gone
        self._in_flight = collections.deque()
        self._finalizer = weakref.finalize(self, _destroy_sampler, out, self._in_flight)
        if output == 'numpy':  # the batch is read on the host anyway: let the kernel range-check given idxs (IndexError at the copy)
            _native.check(_native.lib().ogb_sampler_set_deferred_index_check(out, 1))
        self._layouts: Dict[Any, Any] = {}
        # ogb_sampler_set_host_chunks(n > 1) would issue big host-bound launches in row chunks and copy each finished
        # chunk out under the next one's kernels.  Measured on B200 (C2, 67 MB per call): the 36 per-key, per-chunk copies
        # lose more PCIe efficiency (1.33 vs 1.21 ms) than the overlap gains (the kernels are 0.05 ms), so it stays off.

    # ---- bounds (terminal_locs / initial_locs, datasets.py:186-187) ----
    def bounds(self):
        n = C.c_int64()
        _native.check(_native.lib().ogb_sampler_num_terminals(self.ptr, C.byref(n)))
        term = np.empty(n.value, dtype=np.int64)
        init = np.empty(n.value, dtype=np.int64)
        _native.check(_native.lib().ogb_sampler_copy_bounds(self.ptr, term.ctypes.data_as(C.c_void_p),
                                                            init.ctypes.data_as(C.c_void_p)))
        return term, init

    def set_stream(self, cuda_stream: int):
        _native.check(_native.lib().ogb_sampler_set_stream(self.ptr, C.c_void_p(cuda_stream)))

    def set_debug(self, on=True):
        """bit 0 (True / 1): keep the index vectors readable; bit 1 (2): canary-fill every batch block first; bit 3 (8):
        statically strided tiles in the row gathers instead of ticket scheduling.  Any other bit raises ValueError."""
        _native.check(_native.lib().ogb_sampler_set_debug(self.ptr, int(on)))

    @property
    def counter(self) -> int:
        n = C.c_uint64()
        _native.check(_native.lib().ogb_sampler_get_counter(self.ptr, C.byref(n)))
        return n.value

    @counter.setter
    def counter(self, value: int):
        _native.check(_native.lib().ogb_sampler_set_counter(self.ptr, int(value)))

    # ---- the hot call ----
    def sample_native(self, batch_size, n_batches=1, idxs=None, evaluation=False, draws=None) -> BatchHandle:
        lib = _native.lib()
        keep = []
        idx_ptr = None
        if idxs is not None:
            idxs = np.ascontiguousarray(np.asarray(idxs), dtype=np.int64)
            if idxs.ndim != 1:
                raise ValueError('idxs must be one-dimensional')
            if len(idxs) % int(n_batches) != 0:
                raise ValueError('len(idxs) must be a multiple of n_batches')
            batch_size = len(idxs) // int(n_batches)  # datasets.py:74-76,298: len(idxs) rules
            idx_ptr = idxs.ctypes.data_as(C.c_void_p)
            keep.append(idxs)
        c_draws = None
        if draws is not None:
            c_draws = _pack_draws(draws, keep)
        out = C.c_void_p()
        _native.check(lib.ogb_sampler_sample(self.ptr, int(batch_size), int(n_batches), idx_ptr, int(bool(evaluation)),
                                             C.byref(c_draws) if c_draws is not None else None, C.byref(out)))
        return BatchHandle(out, self.device, None)

    def num_choices(self) -> int:
        n = C.c_int64()
        _native.check(_native.lib().ogb_sampler_num_choices(self.ptr, C.byref(n)))
        return n.value

    def gather(self, which: int, idxs):
        """get_observations (which=0) / get_goal_observations (which=1) for explicit rows; returns one array."""
        idxs = np.ascontiguousarray(np.asarray(idxs), dtype=np.int64).reshape(-1)
        out = C.c_void_p()
        _native.check(_native.lib().ogb_sampler_gather(self.ptr, which, idxs.ctypes.data_as(C.c_void_p), len(idxs), C.byref(out)))
        return next(iter(self.wrap(BatchHandle(out, self.device, None), ('gather', int(which), len(idxs))).values()))   # (a dict of leaves for pytree observations)

    def sample_atc(self, batch_size, k, evaluation=False, draws=None, n_batches=1, keep_axis=False):
        keep = []
        c_draws = _pack_draws(draws, keep) if draws is not None else None
        out = C.c_void_p()
        _native.check(_native.lib().ogb_sampler_sample_atc(self.ptr, int(batch_size), int(n_batches), int(k), int(bool(evaluation)),
                                                           C.byref(c_draws) if c_draws is not None else None, C.byref(out)))
        if keep_axis:
            _native.check(_native.lib().ogb_batch_keep_leading_axis(out, 1))
        return self.wrap(BatchHandle(out, self.device, None), ('atc', int(batch_size), int(n_batches), int(k), bool(evaluation), bool(keep_axis)))

    def atc_anchors(self, k) -> np.ndarray:
        n = C.c_int64()
        _native.check(_native.lib().ogb_sampler_num_atc_anchors(self.ptr, int(k), C.byref(n)))
        out = np.empty(n.value, dtype=np.int64)
        _native.check(_native.lib().ogb_sampler_copy_atc_anchors(self.ptr, int(k), out.ctypes.data_as(C.c_void_p)))
        return out

    def _read_layout(self, handle: BatchHandle):
        """(block bytes, [(name, dtype, shape, offset, nbytes) per key]) of a batch, asked from the library."""
        lib = _native.lib()
        n = C.c_int32()
        _native.check(lib.ogb_batch_num_keys(handle.ptr, C.byref(n)))
        keys = []
        for i in range(n.value):
            info = _native.KeyInfo()
            _native.check(lib.ogb_batch_key_info(handle.ptr, i, C.byref(info)))
            keys.append((info.name.decode(), _native.CODE_TO_DTYPE[info.dtype], tuple(int(info.shape[d]) for d in range(info.ndim)),
                         int(info.offset), int(info.nbytes)))
        nbytes = C.c_size_t()
        _native.check(lib.ogb_batch_nbytes(handle.ptr, C.byref(nbytes)))
        return (max(nbytes.value, 1), keys)

    def _layout(self, handle: BatchHandle, layout_key):
        layout = self._layouts.get(layout_key) if layout_key is not None else None
        if layout is None:
            layout = self._read_layout(handle)
            if layout_key is not None:
                self._layouts[layout_key] = layout
        return layout

    def wrap(self, handle: BatchHandle, layout_key=None, begun_block=None) -> Dict[str, Any]:
        """Batch handle -> dict of arrays.  The layout of a batch's block (name, dtype, shape, offset of every key) is a
        function of the call's shape only, so it is read once per (batch_size, n_batches, evaluation, ...) and reused:
        a steady-state call crosses the C boundary once or twice, not once per key."""
        lib = _native.lib()
        total, keys = self._layout(handle, layout_key)
        if self.output == 'device':
            base = C.c_void_p()
            _native.check(lib.ogb_batch_device_block(handle.ptr, C.byref(base)))
            base = base.value or 0
            out = {name: DeviceArray(handle, i, name, dtype, shape, base + off, nb) for i, (name, dtype, shape, off, nb) in enumerate(keys)}
            return _nest(out) if self.nested else out
        # output == 'numpy': one D2H copy of the whole block into pinned memory, keys are views into it
        # (launch() may have begun the copy already: copies begun one after the other run back to back on the copy stream)
        if begun_block is None:
            block = _PINNED.take(total)
            _native.check(lib.ogb_batch_copy_to_host(handle.ptr, C.c_void_p(block.ptr), block.bucket))
        else:
            block = begun_block
            _native.check(lib.ogb_batch_copy_to_host_end(handle.ptr))
        raw = (C.c_ubyte * total).from_address(block.ptr)
        raw._owner = block  # numpy views -> ctypes buffer -> pinned block: returned to the pool when all views die
        flat = np.frombuffer(raw, dtype=np.uint8)
        out = {name: flat[off:off + nb].view(dtype).reshape(shape) for name, dtype, shape, off, nb in keys}
        return _nest(out) if self.nested else out

    def launch(self, batch_size, idxs=None, evaluation=False, n_batches=1, keep_axis=False) -> PendingBatch:
        """sample() split in two: the launch now, the hand-over (and, for host output, the copy) in PendingBatch.result()."""
        handle = self.sample_native(batch_size, n_batches, idxs, evaluation, None)
        if keep_axis:
            _native.check(_native.lib().ogb_batch_keep_leading_axis(handle.ptr, 1))
        n_rows = len(idxs) // int(n_batches) if idxs is not None else int(batch_size)
        layout_key = ('sample', n_rows, int(n_batches), bool(evaluation), bool(keep_axis))
        block = None
        if self.output != 'device':
            # the device-to-host copy is queued behind the launch right away (on the copy stream); result() waits for it
            total, _ = self._layout(handle, layout_key)
            block = _PINNED.take(total)
            _native.check(_native.lib().ogb_batch_copy_to_host_begin(handle.ptr, C.c_void_p(block.ptr), block.bucket))
        return PendingBatch(self, handle, layout_key, block)

    def sample(self, batch_size, idxs=None, evaluation=False, draws=None, n_batches=1, keep_axis=False):
        handle = self.sample_native(batch_size, n_batches, idxs, evaluation, draws)
        if keep_axis:   # sample_many: arrays are [n_batches, batch, ...] for every n_batches, 1 included
            _native.check(_native.lib().ogb_batch_keep_leading_axis(handle.ptr, 1))
        n_rows = len(idxs) // int(n_batches) if idxs is not None else int(batch_size)
        return self.wrap(handle, ('sample', n_rows, int(n_batches), bool(evaluation), bool(keep_axis)))


def _pack_draws(draws, keep) -> _native.Draws:
    """`draws` is an oracle-style record: .idx_pos, .goals (list of records with rand_pos/offset/dist/u_traj/u_cur,
    in reference call order: value, [low-value], actor), .aug_coin, .crop."""
    d = _native.Draws()

    def ptr(arr, dtype):
        if arr is None:
            return None
        a = np.ascontiguousarray(arr, dtype=dtype)
        keep.append(a)
        return a.ctypes.data

    d.idx_pos = ptr(getattr(draws, 'idx_pos', None), np.int64)
    goals = list(draws.goals)
    slots = {1: [0], 2: [0, 2], 3: [0, 1, 2]}[len(goals)] if goals else []
    for slot, g in zip(slots, goals):
        d.goals[slot].rand_pos = ptr(g.rand_pos, np.int64)
        d.goals[slot].offset = ptr(g.offset, np.int64)
        d.goals[slot].dist = ptr(g.dist, np.float64)
        d.goals[slot].u_traj = ptr(g.u_traj, np.float64)
        d.goals[slot].u_cur = ptr(g.u_cur, np.float64)
    d.has_aug_coin = int(draws.aug_coin is not None)
    d.aug_coin = float(draws.aug_coin) if draws.aug_coin is not None else 0.0
    d.crop = ptr(getattr(draws, 'crop', None), np.int64)
    d.trl_midpoints = ptr(getattr(draws, 'trl_midpoints', None), np.int64)
    return d


class _HostDraws:
    """The reference's np.random call sequence for one sample() (SURVEY.md Appendix C), made on the host so the
    device sampler consumes exactly the draws the reference would have consumed (rng='numpy')."""

    class _Goal:
        __slots__ = ('rand_pos', 'offset', 'dist', 'u_traj', 'u_cur')

        def __init__(self):
            self.rand_pos = self.offset = self.dist = self.u_traj = self.u_cur = None

    def __init__(self):
        self.idx_pos = None
        self.goals = []
        self.aug_coin = None
        self.crop = None
        self.trl_midpoints = None

    def goal(self, n_choices, batch, geom, discount, p_cur):
        g = self._Goal()
        g.rand_pos = np.random.randint(n_choices, size=batch)          # datasets.py:303 -> :68/:70
        if geom:
            g.offset = np.random.geometric(p=1 - discount, size=batch)  # :309
        else:
            g.dist = np.random.rand(batch)                              # :313
        if p_cur != 1.0:
            g.u_traj = np.random.rand(batch)                            # :321
            g.u_cur = np.random.rand(batch)                             # :325
        self.goals.append(g)


def _crop_array(arr, crop_froms, padding, device, output):
    """batched_random_crop (datasets.py:17-33) of one [B, H, W, C] array on the device: the array becomes a temporary
    resident dataset whose rows are gathered with the crop fused in (the same kernels as sample())."""
    ds = Dataset.create(freeze=False, observations=arr)
    sampler = _Sampler(ds, None, _native.KIND_PLAIN, device=device, output=output)
    n = len(crop_froms)
    idxs = np.arange(n, dtype=np.int64)
    crop = np.ascontiguousarray(crop_froms, dtype=np.int64)
    out = C.c_void_p()
    _native.check(_native.lib().ogb_sampler_gather_cropped(sampler.ptr, idxs.ctypes.data_as(C.c_void_p), n,
                                                           crop.ctypes.data_as(C.c_void_p), int(padding), C.byref(out)))
    return next(iter(sampler.wrap(BatchHandle(out, device, None)).values()))


class PendingBatch:
    """A batch whose kernels have been launched; `result()` returns the dict `sample()` would have returned.

    With output='numpy' the device-to-host copy is queued behind the kernels at launch time, on a stream of its own
    (`ogb_batch_copy_to_host_begin`), and `result()` waits for it: launching the next batch before asking for this one's
    result puts that launch (index upload, kernels) under this copy, and its copy directly behind this one on the copy
    engine (what Prefetcher does)."""

    __slots__ = ('_sampler', '_handle', '_layout_key', '_result', '_block')

    def __init__(self, sampler, handle, layout_key, block=None):
        self._sampler, self._handle, self._layout_key, self._result = sampler, handle, layout_key, None
        self._block = block      # output='numpy': the pinned block a begun device-to-host copy is writing into

    def result(self):
        if self._result is None:
            handle, block = self._handle, self._block
            self._handle = self._block = None
            self._result = self._sampler.wrap(handle, self._layout_key, block)
        return self._result

    def __del__(self):
        # a copy that was begun and never asked for must finish before its pinned block goes back to the pool
        if getattr(self, '_block', None) is not None and self._handle is not None:
            try:
                _native.lib().ogb_batch_copy_to_host_end(self._handle.ptr)
            except Exception:
                pass


class _Lookahead:
    """K successive sample(batch) calls drawn in ONE launch and handed out one at a time (GCDataset(..., lookahead=K)).

    The Philox draws of a launch of K batches are those of K single launches (counter = batch index), so the sequence of
    batches is exactly the one direct sample() calls return (tests/test_gpu_lookahead.py)."""

    __slots__ = ('counter0', 'n', 'pos', 'batch', 'evaluation', 'handle', 'keys', 'host', 'nested')

    def __init__(self, counter0, n, batch, evaluation, many):
        self.counter0, self.n, self.pos, self.batch, self.evaluation = counter0, n, 0, batch, evaluation
        self.nested = any(isinstance(v, Mapping) for v in many.values())       # pytree fields: slices are re-nested
        if self.nested:
            many = _flatten(many)
        first = next(iter(many.values()))
        if isinstance(first, DeviceArray):
            self.handle, self.host = first._batch, None
            # (name, key index, dtype, shape of one batch, device address of batch 0, bytes per batch)
            self.keys = [(k, v._index, v.dtype, v.shape[1:], v.ptr, v.nbytes // n) for k, v in many.items()]
        else:
            self.handle, self.keys, self.host = None, None, many

    def take(self):
        i = self.pos
        self.pos = i + 1
        if self.host is not None:
            out = {k: v[i] for k, v in self.host.items()}        # views into the pinned block of the whole launch
        else:
            handle = self.handle
            out = {k: DeviceArray(handle, idx, k, dtype, shape, ptr + i * step, step, i) for k, idx, dtype, shape, ptr, step in self.keys}
        return _nest(out) if self.nested else out


class GCDataset:
    """Dataset class for goal-conditioned RL, device-resident (reference: datasets.py:149-366).

    Reads from `config`: discount, value_p_{cur,traj,random}goal, value_geom_sample, actor_p_*goal,
    actor_geom_sample, gc_negative, p_aug, frame_stack.  `preprocess_frame_stack` is accepted for compatibility;
    frames are always stacked inside the gather (same values, none of the 3x resident copy of datasets.py:209-211).

    rng='philox' (default): indices, offsets and crop shifts are drawn on the device from a counter RNG keyed by
    (seed, stream_id, batch counter).  rng='numpy': the global np.random stream is consumed with exactly the
    reference's calls and the device computes the batch from those draws -- bit-identical to the reference for the
    same np.random.seed.

    lookahead=K (rng='philox'): the unchanged training loop of impls/main.py:202 -- one `sample(batch_size)` per step --
    gets the amortised rate of K-batch launches: the first call draws K batches in one launch and every call pops the
    next one; the sequence of batches is the one K = 0 returns.  Calls with `idxs`, `draws`, `sample_many`,
    `sample_goals` and `load_state_dict` settle the look-ahead first (the batch counter is put back to the number of
    batches actually handed out), so mixing them in keeps the sequence too.

    jax_compat=True: masks / rewards come out as float32 and offsets / steps as int32 -- what `jit` makes of the
    reference's float64 / int64 arrays with JAX's default x64-off -- so `jax.dlpack.from_dlpack` needs no cast.
    """

    _KIND = _native.KIND_GC

    def __init__(self, dataset: Dataset, config: Any, preprocess_frame_stack: bool = True, *, device: int = 0,
                 seed: int = 0, stream_id: int = 0, rng: str = 'philox', output: str = 'device', dedup: bool = True,
                 lookahead: int = 0, jax_compat: bool = False):
        if not isinstance(dataset, Dataset):
            dataset = Dataset.create(freeze=False, **dataset)
        assert rng in ('philox', 'numpy')
        self.dataset = dataset
        self.config = config
        self.preprocess_frame_stack = preprocess_frame_stack
        self.rng = rng
        self.size = dataset.size
        self.lookahead = int(lookahead)
        self._ahead = None
        # datasets.py:191-196 (checked before touching the device, like the reference's __post_init__)
        assert np.isclose(config['value_p_curgoal'] + config['value_p_trajgoal'] + config['value_p_randomgoal'], 1.0)
        assert np.isclose(config['actor_p_curgoal'] + config['actor_p_trajgoal'] + config['actor_p_randomgoal'], 1.0)
        if getattr(dataset, '_nested', False) and config['p_aug']:
            # the reference's augment() reads batch[key].shape (datasets.py:337): a pytree observation has none
            raise NotImplementedError('image augmentation (p_aug > 0) is not defined for pytree observations (datasets.py:329-339)')
        self._trl = self._KIND == _native.KIND_GC and config.get('agent_name') in TRL_AGENTS
        if self._trl:
            # datasets.py:254-257 asserts idxs != value_goal_idxs on every call; with any current/random goal mass that
            # assert fires at random in the reference, so such configs are refused here instead of failing mid-training
            if config['value_p_curgoal'] != 0.0 or config['value_p_randomgoal'] != 0.0:
                raise NotImplementedError('TRL sampling needs value_p_curgoal == value_p_randomgoal == 0 (datasets.py:257)')
        self._sampler = _Sampler(dataset, config, self._KIND, device=device, seed=seed, stream_id=stream_id,
                                 dedup=dedup, output=output, jax_compat=jax_compat)
        self.terminal_locs, self.initial_locs = self._sampler.bounds()
        self._n_choices = self._sampler.num_choices()  # len(valid_idxs); every non-terminal row for TRL (:198-204)
        self._trl_rows = None

    # ---- the reference's draw order, host side (rng='numpy') ----
    def _goal_sets(self):
        cfg = self.config
        return [(cfg['value_geom_sample'], cfg['discount'], cfg['value_p_curgoal']),
                (cfg['actor_geom_sample'], cfg['discount'], cfg['actor_p_curgoal'])]

    def _trl_valid_rows(self):
        """valid_idxs of the TRL agents: every row that is not a terminal row (datasets.py:198-204)."""
        if self._trl_rows is None:
            keep = np.ones(self.size, dtype=bool)
            keep[self.terminal_locs] = False
            (self._trl_rows,) = np.nonzero(keep)
        return self._trl_rows

    def _host_draws(self, batch_size, idxs, evaluation):
        """The reference's np.random calls of one sample(), in its order; returns (draws, idxs)."""
        d = _HostDraws()
        if idxs is None:
            d.idx_pos = np.random.randint(self._n_choices, size=batch_size)      # datasets.py:226 -> :68/:70
        for geom, discount, p_cur in self._goal_sets():
            d.goal(self._n_choices, batch_size, geom, discount, p_cur)
        if self._trl:
            # :259 draws randint(idxs, value_goal_idxs): the goal rows come from the device (phase one: the value goals of
            # these very draws), the midpoint draw is made here, and the launch then replays everything (phase two)
            rows = np.ascontiguousarray(idxs, dtype=np.int64) if idxs is not None else self._trl_valid_rows()[d.idx_pos]
            cfg = self.config
            goals = self._goals_native(rows, cfg['value_p_curgoal'], cfg['value_p_trajgoal'], cfg['value_geom_sample'],
                                       cfg['discount'], d.goals[0])
            final = self.terminal_locs[np.searchsorted(self.terminal_locs, rows)]
            assert (rows != final).all()                                         # :256
            assert (rows != goals).all()                                         # :257
            d.trl_midpoints = np.random.randint(rows, goals)                     # :259
            d.idx_pos, idxs = None, rows
        if self.config['p_aug'] is not None and not evaluation:                  # :278-279 / :621-622
            d.aug_coin = np.random.rand()
            if d.aug_coin < self.config['p_aug']:
                d.crop = np.random.randint(0, 2 * 3 + 1, (batch_size, 2))        # :333
        return d, idxs

    def sample(self, batch_size, idxs=None, evaluation=False, *, draws=None):
        """Sample a batch of transitions with goals (datasets.py:213-294).

        Returns the reference's keys: every dataset field, next_observations, value_goals, actor_goals,
        masks, rewards.  `draws` (an oracle-style record) selects validation mode explicitly.
        """
        if idxs is not None:
            batch_size = len(idxs)
        elif draws is None and self.lookahead > 1 and self.rng == 'philox':
            return self._sample_ahead(int(batch_size), bool(evaluation))
        self._settle()
        if draws is None and self.rng == 'numpy':
            draws, idxs = self._host_draws(batch_size, idxs, evaluation)
        return self._sampler.sample(batch_size, idxs, evaluation, draws)

    # ---- look-ahead: K batches per launch behind the reference's one-call-per-step loop (impls/main.py:202) ----
    def _sample_ahead(self, batch_size, evaluation):
        la = self._ahead
        if la is None or la.pos == la.n or la.batch != batch_size or la.evaluation != evaluation:
            self._settle()
            counter0 = self._sampler.counter
            many = self._sampler.sample(batch_size, None, evaluation, None, n_batches=self.lookahead, keep_axis=True)
            la = self._ahead = _Lookahead(counter0, self.lookahead, batch_size, evaluation, many)
        return la.take()

    def _settle(self):
        """Drop the batches drawn ahead but not handed out: the batch counter goes back to the number of batches the caller
        has actually received, so whatever is drawn next continues the sequence direct calls would have produced."""
        la, self._ahead = self._ahead, None
        if la is not None and la.pos < la.n:
            self._sampler.counter = la.counter0 + la.pos

    def sample_many(self, num_batches, batch_size, evaluation=False, idxs=None):
        """`num_batches` successive sample(batch_size) calls in one launch; every key gains a leading axis of that length.
        `idxs` (optional, num_batches * batch_size rows) plays the role of sample()'s `idxs`."""
        self._settle()
        return self._sampler.sample(batch_size, idxs, evaluation, None, n_batches=num_batches, keep_axis=True)

    def sample_async(self, batch_size, idxs=None, evaluation=False, num_batches=None) -> PendingBatch:
        """Launch `sample(batch_size, idxs, evaluation)` (or, with `num_batches`, `sample_many`) and return at once;
        `.result()` of the returned object gives the batch.  rng='philox' only: the draws are made by the launch."""
        if self.rng != 'philox':
            raise ValueError("sample_async needs rng='philox' (rng='numpy' draws on the host, in the reference's call order)")
        self._settle()
        if idxs is not None and num_batches is None:
            batch_size = len(idxs)
        if num_batches is None:
            return self._sampler.launch(batch_size, idxs, evaluation)
        return self._sampler.launch(batch_size, idxs, evaluation, n_batches=num_batches, keep_axis=True)

    # ---- reference helpers that other scripts call (impls/pretrain_atc.py:195, pretrain_vae.py:162) ----
    def get_observations(self, idxs):
        """Return the observations for the given indices, frame-stacked as configured (datasets.py:341-346)."""
        return self._sampler.gather(0, idxs)

    def get_goal_observations(self, idxs):
        """Return goal observations: `oracle_reps` if the dataset has them, else observations (datasets.py:348-357)."""
        return self._sampler.gather(1, idxs)

    def get_stacked_observations(self, idxs):
        """Return the frame-stacked observations for the given indices (datasets.py:359-366)."""
        assert self.config['frame_stack'] is not None
        return self._sampler.gather(0, idxs)

    def sample_goals(self, idxs, p_curgoal, p_trajgoal, p_randomgoal, geom_sample, discount=None):
        """Sample goals for the given indices (datasets.py:296-327); returns int64 row indices on the host.

        rng='numpy' makes the reference's own np.random calls (randint, geometric or rand, rand, rand) and the device
        computes the goals from them; rng='philox' draws on the device."""
        self._settle()
        idxs = np.ascontiguousarray(np.asarray(idxs), dtype=np.int64).reshape(-1)
        if discount is None:
            discount = self.config['discount']
        goal_draws = None
        if self.rng == 'numpy':
            d = _HostDraws()
            d.goal(self._n_choices, len(idxs), geom_sample, discount, p_curgoal)
            goal_draws = d.goals[0]
        return self._goals_native(idxs, p_curgoal, p_trajgoal, geom_sample, discount, goal_draws)

    def _goals_native(self, idxs, p_curgoal, p_trajgoal, geom_sample, discount, goal_draws):
        """Goal rows for `idxs` from the given draws (None: drawn on the device), as int64 on the host."""
        n = len(idxs)
        c_draws, keep = None, []
        if goal_draws is not None:
            c_draws = _native.GoalDraws()
            for name, dtype in (('rand_pos', np.int64), ('offset', np.int64), ('dist', np.float64), ('u_traj', np.float64), ('u_cur', np.float64)):
                arr = getattr(goal_draws, name)
                if arr is not None:
                    arr = np.ascontiguousarray(arr, dtype=dtype)
                    keep.append(arr)
                    setattr(c_draws, name, arr.ctypes.data)
        out = np.empty(n, dtype=np.int64)
        if n == 0:      # (the np.random calls were still made, with size 0, like the reference's)
            return out
        _native.check(_native.lib().ogb_sampler_sample_goals(
            self._sampler.ptr, idxs.ctypes.data_as(C.c_void_p), n, float(p_curgoal), float(p_trajgoal), int(bool(geom_sample)),
            float(discount), C.byref(c_draws) if c_draws is not None else None, out.ctypes.data_as(C.c_void_p)))
        return out

    def augment(self, batch, keys):
        """Apply image augmentation to the given keys, in place (datasets.py:329-339): one (cy, cx) shift per sample from
        np.random.randint -- the reference's own call -- shared by all keys; arrays that are not 4-D pass through."""
        padding = 3
        batch_size = len(batch[keys[0]])
        crop_froms = np.random.randint(0, 2 * padding + 1, (batch_size, 2))
        for key in keys:
            if len(batch[key].shape) == 4:
                batch[key] = _crop_array(batch[key], crop_froms, padding, self._sampler.device, self._sampler.output)

    # ---- checkpointable sampler state: one integer ----
    def state_dict(self):
        """The number of batches handed out so far (batches drawn ahead and not yet handed out do not count)."""
        la = self._ahead
        return {'counter': la.counter0 + la.pos if la is not None else self._sampler.counter}

    def load_state_dict(self, state):
        self._ahead = None
        self._sampler.counter = state['counter']


class HGCDataset(GCDataset):
    """Dataset class for hierarchical goal-conditioned RL (reference: datasets.py:467-643).

    Additional config keys: subgoal_steps (optional: high_/low_/value_/actor_subgoal_steps), low_discount.
    """

    _KIND = _native.KIND_HGC

    def compute_high_next_idxs(self, idxs, final_state_idxs, high_goal_idxs, subgoal_steps):
        """Compute the next indices for high-level goals (datasets.py:478-491); returns (idxs + steps, steps)."""
        arrs = [np.ascontiguousarray(np.asarray(a), dtype=np.int64).reshape(-1) for a in (idxs, final_state_idxs, high_goal_idxs)]
        n = len(arrs[0])
        nxt, steps = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64)
        if n == 0:
            return nxt, steps
        _native.check(_native.lib().ogb_sampler_compute_high_next_idxs(
            self._sampler.ptr, *[a.ctypes.data_as(C.c_void_p) for a in arrs], n, int(subgoal_steps),
            nxt.ctypes.data_as(C.c_void_p), steps.ctypes.data_as(C.c_void_p)))
        return nxt, steps

    def get_high_actions(self, target_idxs, cur_idxs):
        return self.get_goal_observations(target_idxs)  # datasets.py:493-494

    def _goal_sets(self):
        cfg = self.config
        sets = [(cfg['value_geom_sample'], cfg['discount'], cfg['value_p_curgoal'])]
        if cfg.get('low_discount') is not None:                                  # datasets.py:563-571
            sets.append((True, cfg['low_discount'], cfg['value_p_curgoal']))
        sets.append((cfg['actor_geom_sample'], cfg['discount'], cfg['actor_p_curgoal']))
        return sets


class ATCDataset:
    """Dataset class for ATC pretraining, device-resident (reference: datasets.py:369-464).

    Samples anchor/positive observation pairs (o_t, o_{t+k}) from the same trajectory, with frame stacking and the
    random-shift augmentation fused into the gather.  Config keys: frame_stack, p_aug, augment_padding (default 4).
    """

    def __init__(self, dataset: Dataset, config: Any, preprocess_frame_stack: bool = True, *, device: int = 0,
                 seed: int = 0, stream_id: int = 0, rng: str = 'philox', output: str = 'device'):
        if not isinstance(dataset, Dataset):
            dataset = Dataset.create(freeze=False, **dataset)
        assert rng in ('philox', 'numpy')
        self.dataset = dataset
        self.config = config
        self.preprocess_frame_stack = preprocess_frame_stack
        self.rng = rng
        self.size = dataset.size
        self._padding = int(config.get('augment_padding', 4))                      # datasets.py:440
        self._sampler = _Sampler(dataset, config, _native.KIND_ATC, device=device, seed=seed, stream_id=stream_id,
                                 output=output, crop_padding=self._padding)
        self.terminal_locs, self.initial_locs = self._sampler.bounds()

    def get_valid_atc_idxs(self, k):
        """Return valid anchor indices for a given temporal offset k (datasets.py:417-436; cached per k natively)."""
        return self._sampler.atc_anchors(k)

    def get_observations(self, idxs):
        """Return the observations for the given indices, frame-stacked as configured (datasets.py:451-456)."""
        return self._sampler.gather(0, idxs)

    def get_stacked_observations(self, idxs):
        """Return the frame-stacked observations for the given indices (datasets.py:458-464)."""
        assert self.config['frame_stack'] is not None
        return self._sampler.gather(0, idxs)

    def augment(self, batch, keys):
        """Apply random-shift augmentation to image observations, in place (datasets.py:438-448)."""
        batch_size = len(batch[keys[0]])
        crop_froms = np.random.randint(0, 2 * self._padding + 1, (batch_size, 2))
        for key in keys:
            if len(batch[key].shape) == 4:
                batch[key] = _crop_array(batch[key], crop_froms, self._padding, self._sampler.device, self._sampler.output)

    def _host_draws(self, batch_size, k, evaluation) -> _HostDraws:
        d = _HostDraws()
        n = C.c_int64()
        _native.check(_native.lib().ogb_sampler_num_atc_anchors(self._sampler.ptr, int(k), C.byref(n)))
        d.idx_pos = np.random.randint(0, n.value, size=batch_size)               # np.random.choice(valid_idxs, size=B)  :404
        if self.config['p_aug'] is not None and not evaluation:                  # :411-412
            d.aug_coin = np.random.rand()
            if d.aug_coin < self.config['p_aug']:
                d.crop = np.random.randint(0, 2 * self._padding + 1, (batch_size, 2))  # :442
        return d

    def sample(self, batch_size, k, evaluation=False, *, draws=None):
        """Sample a batch of anchor/positive observations from the same trajectory (datasets.py:401-415)."""
        if draws is None and self.rng == 'numpy':
            draws = self._host_draws(batch_size, k, evaluation)
        return self._sampler.sample_atc(batch_size, k, evaluation, draws)

    def sample_many(self, num_batches, batch_size, k, evaluation=False):
        return self._sampler.sample_atc(batch_size, k, evaluation, None, n_batches=num_batches, keep_axis=True)
