"""Upstream feeder for the packed-CSR kernels (SURVEY §8f rank 4; reference: dataset.py:366-393).

The reference's Dataset returns ONE slide per sample: `np.load(<pathology_path>/<hospital>/<Biopsy|Resection>/
<patient>.npy)` -> [n, 768] float, optionally thinned by the augmentation of dataset.py:375-381 (keep a sorted random
90 % of a biopsy's rows, 80 % of a resection's), zero-padded to 15 592 rows when batch_size > 1 (dataset.py:383-390)
and converted with `.float()`.  The DataLoader then collates, and `.cuda()` ships fp32.

`PackedBagFeeder` produces what the B200 kernels want instead: per step, the slides of the batch are gathered by native
threads (`milb200_pack_bags_host`) straight into a pinned staging buffer — rows back to back, already bf16 (RNE), with
the int32 CSR offsets — and copied to the device on a copy stream while the previous step computes.  Nothing is padded
and half the bytes cross PCIe.  Two staging/device buffer pairs rotate; a worker thread packs batch k+1 while batch k
is in flight.  The numpy arrays may be memory-mapped (`np.load(..., mmap_mode="r")`), in which case the page-cache reads
happen inside the packing threads.

`ResidentBagFeeder` is the route for a slide set that fits in device memory: the slides are uploaded once, and every
batch, augmentation subsets included, is sampled and packed on the device by two kernels (csrc/resident.cu), so neither
PCIe nor Python's sampling sits in the training loop.  Its subsets come from a device Philox stream, not from Python's
Mersenne Twister: PackedBagFeeder stays the route for bit-for-bit use of the host RNG and for data sets that do not fit.
"""
from __future__ import annotations

import ctypes as C
import queue
import random
import threading

import numpy as np
import torch

from . import _lib as L
from . import functional as F

_HOST_CODES = {np.dtype(np.float32): L.HOST_F32, np.dtype(np.float64): L.HOST_F64, np.dtype(np.float16): L.HOST_F16}

# dataset.py:375-381: fraction of rows KEPT in train mode with augmentation, by slide type
AUGMENT_KEEP = {"Biopsy": 0.9, "Resection": 0.8}


def augmentation_count(n, slide_type):
    """Rows the augmentation keeps of an n-row slide, `int(n * keep)` (dataset.py:378,381); None for a slide type it
    leaves whole.  Both feeders size their bags with it."""
    keep = AUGMENT_KEEP.get(slide_type)
    return None if keep is None else int(n * keep)


def augmentation_rows(n, slide_type, rng):
    """The reference's row thinning: `sorted(random.sample(range(n), int(n * keep)))` (dataset.py:377-381)."""
    k = augmentation_count(n, slide_type)
    if k is None:
        return None
    return np.asarray(sorted(rng.sample(range(n), k)), dtype=np.int32)


def _load(source):
    """A slide's feature matrix: `.npy` paths are memory-mapped, anything else is returned as it is."""
    if isinstance(source, (str, bytes)) or hasattr(source, "__fspath__"):
        return np.load(source, mmap_mode="r")
    return source


def pack_bags_host(bags, dst, offsets, keep_rows=None, n_threads=0):
    """Gather `bags` (list of 2-D numpy arrays [n_b, L], C-contiguous rows; or bf16 torch CPU tensors) into `dst`
    (CPU torch tensor [capacity, L], fp32 or bf16, normally pinned) and fill `offsets` (CPU int32 [len(bags)+1]).
    Returns the number of packed rows.  keep_rows: optional list (None or sorted int32 row indices per bag)."""
    nb = len(bags)
    if nb == 0:
        raise ValueError("pack_bags_host: empty batch")
    if dst.device.type != "cpu" or offsets.device.type != "cpu" or offsets.dtype != torch.int32 \
            or offsets.numel() < nb + 1 or not dst.is_contiguous() or dst.dim() != 2:
        raise ValueError("pack_bags_host: dst must be a contiguous CPU [rows, L] tensor and offsets CPU int32 [B+1]")
    Lf = dst.shape[1]
    ptrs = (C.c_void_p * nb)()
    rows = (C.c_int64 * nb)()
    pitch = (C.c_int64 * nb)()
    code = None
    for b, a in enumerate(bags):
        if isinstance(a, torch.Tensor):
            if a.dtype != torch.bfloat16 or a.device.type != "cpu" or a.dim() != 2 or a.stride(1) != 1:
                raise ValueError("pack_bags_host: torch sources must be CPU bf16 [n, L] with contiguous rows")
            c, ptr, n, lf, pb = L.HOST_BF16, a.data_ptr(), a.shape[0], a.shape[1], a.stride(0) * 2
        else:
            if a.ndim != 2 or a.dtype not in _HOST_CODES or (a.size and a.strides[1] != a.itemsize):
                raise ValueError("pack_bags_host: numpy sources must be [n, L] float16/32/64 with contiguous rows")
            c, ptr, n, lf, pb = _HOST_CODES[a.dtype], a.ctypes.data, a.shape[0], a.shape[1], a.strides[0]
        if lf != Lf:
            raise ValueError(f"pack_bags_host: bag {b} has {lf} features, destination {Lf}")
        if code is None:
            code = c
        elif code != c:
            raise ValueError("pack_bags_host: all bags of a batch must share one source dtype")
        ptrs[b], rows[b], pitch[b] = ptr, n, pb
    kp = kc = None
    keep_alive = []
    if keep_rows is not None and any(k is not None for k in keep_rows):
        kp = (C.c_void_p * nb)()
        kc = (C.c_int64 * nb)()
        for b, k in enumerate(keep_rows):
            if k is None:
                kp[b], kc[b] = None, rows[b]
            else:
                k = np.ascontiguousarray(k, dtype=np.int32)
                keep_alive.append(k)
                kp[b], kc[b] = k.ctypes.data, k.shape[0]
    L.check(L.lib().milb200_pack_bags_host(ptrs, rows, pitch, kp, kc, nb, Lf, code, dst.data_ptr(),
                                           L.dtype_code(dst), dst.shape[0], offsets.data_ptr(), int(n_threads)),
            "pack_bags_host")
    return int(offsets[nb])


class _EpochSchedule:
    """The batch schedule both feeders share: DistributedSampler's per-epoch order over `n_slides` slides, cut into
    batches of B.  Subclasses set n_slides, B, shuffle, seed, rank, world, drop_last and epoch."""

    def set_epoch(self, epoch):          # DistributedSampler's contract (train_ddp.py:201-202)
        self.epoch = int(epoch)

    def order(self):
        """This rank's bag indices for the epoch: DistributedSampler's permutation, padding and stride
        (train_ddp.py:191, drop_last=False): the index list is extended with its own head to a multiple of `world`, so
        every rank draws ceil(n / world) bags (and therefore the same number of batches — each step ends in one
        all-reduce, a rank that ran out of batches would leave the others waiting in it)."""
        n = self.n_slides
        if self.shuffle:
            g = torch.Generator().manual_seed(self.seed + self.epoch)
            idx = torch.randperm(n, generator=g).tolist()
        else:
            idx = list(range(n))
        if self.world > 1 and n > 0:
            total = (n + self.world - 1) // self.world * self.world
            pad = total - n
            if pad:
                idx = idx + (idx * ((pad + n - 1) // n))[:pad]
        return idx[self.rank::self.world]

    def batches(self):
        idx = self.order()
        out = [idx[i:i + self.B] for i in range(0, len(idx), self.B)]
        if self.drop_last and out and len(out[-1]) < self.B:
            out.pop()
        return out

    def __len__(self):
        return len(self.batches())


class PackedBagFeeder(_EpochSchedule):
    """Iterates packed-CSR batches on the device.

    sources: sequence of per-slide feature matrices (numpy arrays, possibly memory-mapped, or paths to `.npy` files).
    slide_types: optional sequence of "Biopsy"/"Resection" (dataset.py:376-381) enabling the train-mode augmentation.
    Each item is (X [total_n, L] on `device`, offsets int32 [B+1] on `device`, indices of the bags in the batch);
    X and offsets are views of a rotating device buffer: consume them before asking for the batch after next
    (the iterator waits on the consumer's stream before reusing a buffer)."""

    def __init__(self, sources, batch_bags, L_feat, device="cuda", dtype=torch.bfloat16, slide_types=None, augment=False,
                 shuffle=False, seed=1234, rank=0, world=1, n_threads=0, capacity_rows=None, drop_last=False):
        self.sources, self.B, self.L = list(sources), int(batch_bags), int(L_feat)
        self.n_slides = len(self.sources)
        self.device, self.dtype = torch.device(device), dtype
        self.slide_types, self.augment = slide_types, bool(augment)
        self.shuffle, self.seed, self.rank, self.world = shuffle, seed, rank, world
        self.n_threads, self.drop_last = n_threads, drop_last
        self.epoch = 0
        self._rows = [self._open(i).shape[0] for i in range(len(self.sources))]
        if capacity_rows is None:      # worst batch: the B largest bags
            capacity_rows = sum(sorted(self._rows, reverse=True)[:self.B])
        self.capacity = int(capacity_rows)
        pin = self.device.type == "cuda"
        self._stage = [torch.empty((self.capacity, self.L), dtype=dtype, pin_memory=pin) for _ in range(2)]
        self._off_h = [torch.empty(self.B + 1, dtype=torch.int32, pin_memory=pin) for _ in range(2)]
        self._dev = [torch.empty((self.capacity, self.L), dtype=dtype, device=self.device) for _ in range(2)]
        self._off_d = [torch.empty(self.B + 1, dtype=torch.int32, device=self.device) for _ in range(2)]
        if pin:
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._copied = [torch.cuda.Event() for _ in range(2)]
            self._consumed = [torch.cuda.Event() for _ in range(2)]
            self._staged_free = [torch.cuda.Event() for _ in range(2)]

    def _open(self, i):
        return _load(self.sources[i])

    def _pack(self, slot, bag_ids, rng):
        arrays = [self._open(i) for i in bag_ids]
        keep = None
        if self.augment and self.slide_types is not None:
            keep = [augmentation_rows(a.shape[0], self.slide_types[i], rng) for a, i in zip(arrays, bag_ids)]
        n = pack_bags_host(arrays, self._stage[slot], self._off_h[slot], keep, self.n_threads)
        return n

    def __iter__(self):
        batches = self.batches()
        rng = random.Random(self.seed + 7919 * self.epoch + self.rank)
        cuda = self.device.type == "cuda"
        q: "queue.Queue" = queue.Queue(maxsize=1)
        free = [threading.Semaphore(1), threading.Semaphore(1)]      # staging slot may be overwritten

        stop = threading.Event()            # set when the consumer abandons the iteration: the worker must not block forever

        def put(item):
            while not stop.is_set():
                try:
                    q.put(item, timeout=0.2)
                    return True
                except queue.Full:
                    continue
            return False

        def worker():
            try:
                for k, ids in enumerate(batches):
                    slot = k & 1
                    while not free[slot].acquire(timeout=0.2):
                        if stop.is_set():
                            return
                    if cuda:
                        self._staged_free[slot].synchronize()      # the H2D copy that last read this staging slot is done
                    n = self._pack(slot, ids, rng)
                    if not put((slot, n, ids)):
                        return
                put(None)
            except BaseException as e:       # surface packing errors in the consumer
                put(e)

        th = threading.Thread(target=worker, daemon=True)
        th.start()
        if cuda:
            main = torch.cuda.current_stream(self.device)
            for ev in self._consumed:
                ev.record(main)
        try:
            yield from self._consume(q, free, cuda)
        finally:
            stop.set()
            th.join()

    def _consume(self, q, free, cuda):
        while True:
            item = q.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            slot, n, ids = item
            nb = len(ids)
            if cuda:
                main = torch.cuda.current_stream(self.device)
                with torch.cuda.stream(self._copy_stream):
                    self._copy_stream.wait_event(self._consumed[slot])     # kernels that read this device buffer are done
                    self._dev[slot][:n].copy_(self._stage[slot][:n], non_blocking=True)
                    self._off_d[slot][:nb + 1].copy_(self._off_h[slot][:nb + 1], non_blocking=True)
                    self._copied[slot].record(self._copy_stream)
                    self._staged_free[slot].record(self._copy_stream)
                free[slot].release()
                main.wait_event(self._copied[slot])
                yield self._dev[slot][:n], self._off_d[slot][:nb + 1], ids
                self._consumed[slot].record(torch.cuda.current_stream(self.device))
            else:
                self._dev[slot][:n].copy_(self._stage[slot][:n])
                self._off_d[slot][:nb + 1].copy_(self._off_h[slot][:nb + 1])
                free[slot].release()
                yield self._dev[slot][:n], self._off_d[slot][:nb + 1], ids


class ResidentBagFeeder(_EpochSchedule):
    """Iterates packed-CSR batches built on the device from a slide set held in device memory.

    The slides are uploaded once, at construction, into one store [total_rows, L_feat] of `dtype` (fp32 or bf16, rows
    of a multiple of 16 bytes) with int64 slide_start [S+1].  Each batch is then two kernels on the consumer's current
    stream: `select_rows` picks the store rows of every bag (all of them, or with `augment` and a Biopsy/Resection slide
    type the random `int(n * keep)`-row subset of dataset.py:375-381, drawn from a Philox stream keyed by
    (seed, epoch, rank, slide id): the same counts as PackedBagFeeder, not the same rows), and `gather_rows` copies them
    into one of two rotating output buffers.  The schedule (DistributedSampler's order, padding, stride, drop_last,
    set_epoch) is PackedBagFeeder's.

    sources: per-slide [n, L_feat] matrices: numpy arrays (float16/32/64), `.npy` paths (memory-mapped), CPU bf16 tensors
    or CUDA tensors of `dtype`.  Host sources are converted by the native packer and staged through two bounded pinned
    buffers; CUDA sources are copied device to device.
    labels: optional [S, C] per-slide targets; each item then carries y = labels[ids] as a contiguous fp32 [B, C] device
    tensor from a pair of rotating buffers (what AbmilTrainer.step_labels takes).

    Items are (X [offsets[B], L] on the device, offsets int32 [B+1] on the device, slide ids of the batch[, y]); X's
    shape is known on the host, nothing synchronises.  X, offsets and y are views of rotating buffers: consume a batch
    before asking for the batch after next.  Row counts change from batch to batch: feed AbmilTrainer.step /
    step_labels, not step_graphed (which captures one graph per shape).

    Device memory, on every rank (each rank draws different slides every epoch, so each holds them all):
    total_rows * L * itemsize for the store + 2 * capacity * (L * itemsize + 8) for the batch buffers and their row
    lists, capacity being the rows of the B largest bags, + 8 * (S + 1) + (labels: 4 * C * (S + 2 * B)).  The
    constructor compares the store and batch buffers with the free device memory before allocating anything."""

    STAGE_BYTES = 64 << 20      # per pinned staging buffer of the upload (two of them)

    def __init__(self, sources, batch_bags, L_feat, device="cuda", dtype=torch.bfloat16, slide_types=None, augment=False,
                 shuffle=False, seed=1234, rank=0, world=1, labels=None, n_threads=0, drop_last=False):
        self.B, self.L = int(batch_bags), int(L_feat)
        self.device, self.dtype = torch.device(device), dtype
        self.augment, self.shuffle, self.seed, self.rank, self.world = bool(augment), shuffle, int(seed), rank, world
        self.n_threads, self.drop_last = n_threads, drop_last
        self.epoch = 0
        if self.device.type != "cuda":
            raise L.MilB200Error("ResidentBagFeeder keeps the slide set in CUDA device memory")
        if dtype not in (torch.float32, torch.bfloat16):
            raise L.MilB200Error(f"ResidentBagFeeder stores fp32 or bf16 rows, not {dtype}")
        row_bytes = self.L * torch.empty((), dtype=dtype).element_size()
        if row_bytes % 16:
            raise L.MilB200Error(f"ResidentBagFeeder: a row of {self.L} {dtype} features is {row_bytes} bytes; the "
                                 "device gather copies rows of a multiple of 16 bytes")
        srcs = [_load(s) for s in sources]
        for i, a in enumerate(srcs):
            if len(a.shape) != 2 or int(a.shape[1]) != self.L:
                raise ValueError(f"ResidentBagFeeder: slide {i} has shape {tuple(a.shape)}, the store holds rows of "
                                 f"{self.L} features")
            if isinstance(a, torch.Tensor) and a.is_cuda and (a.dtype != dtype or a.device != self._cuda_device()):
                raise ValueError(f"ResidentBagFeeder: CUDA slide {i} must be {dtype} on {self._cuda_device()}")
        self.n_slides = len(srcs)
        rows = [int(a.shape[0]) for a in srcs]
        counts = []
        for i, n in enumerate(rows):
            k = augmentation_count(n, slide_types[i]) if self.augment and slide_types is not None else None
            k = n if k is None else k
            if k < 1:
                raise L.MilB200Error(f"ResidentBagFeeder: slide {i} has {n} rows and would keep {k}; every bag needs at "
                                     "least one instance")
            counts.append(k)
        self.counts = counts
        self.capacity = sum(sorted(counts, reverse=True)[:self.B])
        if self.capacity > 2 ** 31 - 1:
            raise L.MilB200Error("ResidentBagFeeder: a batch may hold more than 2^31-1 rows (int32 offsets)")
        start = np.zeros(self.n_slides + 1, dtype=np.int64)
        np.cumsum(rows, out=start[1:])
        total = int(start[-1])
        need = total * row_bytes + 2 * self.capacity * (row_bytes + 8)
        free = torch.cuda.mem_get_info(self.device)[0]
        if need > free:
            raise L.MilB200Error(f"ResidentBagFeeder: the slide store and its batch buffers need {need} bytes, the device "
                                 f"has {free} bytes free")
        self.store = torch.empty((total, self.L), dtype=dtype, device=self.device)
        self.slide_start = torch.from_numpy(start).to(self.device)
        self._start = start
        self._upload(srcs, start, row_bytes)
        self._out = [torch.empty((self.capacity, self.L), dtype=dtype, device=self.device) for _ in range(2)]
        self._src = [torch.empty(self.capacity, dtype=torch.int64, device=self.device) for _ in range(2)]
        self.labels = None
        if labels is not None:
            lab = torch.as_tensor(labels)
            if lab.dim() != 2 or lab.shape[0] != self.n_slides:
                raise ValueError(f"ResidentBagFeeder: labels must be [{self.n_slides}, C], got {tuple(lab.shape)}")
            self.labels = lab.to(device=self.device, dtype=torch.float32).contiguous()
            self._y = [torch.empty((self.B, lab.shape[1]), dtype=torch.float32, device=self.device) for _ in range(2)]
        self._consumed = [torch.cuda.Event() for _ in range(2)]

    def _cuda_device(self):
        return torch.device("cuda", self.device.index if self.device.index is not None else torch.cuda.current_device())

    def _upload(self, srcs, start, row_bytes):
        """Host slides -> native packer -> one of two pinned staging buffers -> one async copy per chunk; a staging buffer
        is packed again only after the copy that read it has completed.  CUDA slides are copied device to device."""
        chunk = max(1, self.STAGE_BYTES // row_bytes)
        stage = [torch.empty((chunk, self.L), dtype=self.dtype, pin_memory=True) for _ in range(2)]
        copied = [None, None]
        pending, kind, slot = [], None, 0            # pieces (matrix, first store row) of the chunk being filled
        filled = 0
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream()

            def flush():
                nonlocal pending, kind, slot, filled
                if not pending:
                    return
                if copied[slot] is not None:
                    copied[slot].synchronize()
                off = torch.empty(len(pending) + 1, dtype=torch.int32)
                n = pack_bags_host([p for p, _ in pending], stage[slot], off, n_threads=self.n_threads)
                r0 = pending[0][1]
                self.store[r0:r0 + n].copy_(stage[slot][:n], non_blocking=True)
                copied[slot] = torch.cuda.Event()
                copied[slot].record(stream)
                pending, kind, slot, filled = [], None, slot ^ 1, 0

            for i, a in enumerate(srcs):
                if isinstance(a, torch.Tensor) and a.is_cuda:
                    flush()
                    self.store[start[i]:start[i + 1]].copy_(a, non_blocking=True)
                    continue
                k = str(a.dtype)                             # 'torch.bfloat16', 'float32', ...
                n, r = int(a.shape[0]), 0
                while r < n:
                    if kind is not None and kind != k:      # the packer takes one source dtype per call
                        flush()
                    take = min(n - r, chunk - filled)
                    pending.append((a[r:r + take], int(start[i]) + r))
                    kind, filled, r = k, filled + take, r + take
                    if filled == chunk:
                        flush()
            flush()
            stream.synchronize()                           # the staging buffers are released on return

    def __iter__(self):
        batches = self.batches()
        if not batches:
            return
        # the epoch's whole batch table (slide ids, then int32 offsets per batch) goes to the device in one copy
        ids_h, offs_h = [], []
        for ids in batches:
            ids_h.append(np.asarray(ids, dtype=np.int32))
            o = np.zeros(len(ids) + 1, dtype=np.int64)
            np.cumsum([self.counts[i] for i in ids], out=o[1:])
            offs_h.append(o.astype(np.int32))
        n_ids = sum(len(x) for x in ids_h)
        table = torch.from_numpy(np.concatenate(ids_h + offs_h)).pin_memory().to(self.device, non_blocking=True)
        ids_long = table[:n_ids].long() if self.labels is not None else None
        main = torch.cuda.current_stream(self.device)
        for ev in self._consumed:
            ev.record(main)
        io, oo = 0, n_ids
        for k, ids in enumerate(batches):
            slot, nb = k & 1, len(ids)
            n = int(offs_h[k][-1])
            ids_d, off_d = table[io:io + nb], table[oo:oo + nb + 1]
            main = torch.cuda.current_stream(self.device)
            main.wait_event(self._consumed[slot])           # kernels that read this slot's buffers are done
            with torch.cuda.device(self.device):
                src = F.select_rows(self.slide_start, ids_d, off_d, n, self.seed, self.epoch, self.rank, out=self._src[slot])
                X = F.gather_rows(self.store, src, out=self._out[slot])
                if self.labels is None:
                    item = (X, off_d, ids)
                else:
                    y = self._y[slot][:nb]
                    torch.index_select(self.labels, 0, ids_long[io:io + nb], out=y)
                    item = (X, off_d, ids, y)
            yield item
            self._consumed[slot].record(torch.cuda.current_stream(self.device))
            io, oo = io + nb, oo + nb + 1
