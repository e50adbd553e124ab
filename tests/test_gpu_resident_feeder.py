"""The resident feeder (csrc/resident.cu, feeder.ResidentBagFeeder): batches built on the device from a slide set held in
device memory.  Without augmentation they are PackedBagFeeder's batches bit for bit; the row sampler is checked against
a host Philox reference, for its subset properties and for uniformity; the gather against the host packer and against
index_select past 2^31 elements; and a trainer fed by the feeder against the same trainer fed hand-built batches."""
import random

import numpy as np
import pytest
import scipy.stats
import torch

import mil_b200
from mil_b200 import feeder, functional as F

pytestmark = pytest.mark.gpu

EDGE_LENS = [1, 2, 127, 128, 129, 300, 17, 64, 1000]


def _bags(lens, L, seed, dtype=np.float32):
    rng = np.random.default_rng(seed)
    return [(rng.standard_normal((n, L)) * 3).astype(dtype) for n in lens]


def _host_keys(seed, slide, epoch, rank, n):
    """Host Philox4x32-10 of counter (row, slide, epoch, rank), key (seed low, seed high) -> 64-bit keys (x << 32 | y)."""
    M = np.uint64(0xFFFFFFFF)
    x = np.arange(n, dtype=np.uint64)
    y = np.full(n, slide, dtype=np.uint64)
    z = np.full(n, epoch, dtype=np.uint64)
    w = np.full(n, rank, dtype=np.uint64)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * x
        p1 = np.uint64(0xCD9E8D57) * z
        x, y, z, w = (p1 >> np.uint64(32)) ^ y ^ k0, p1 & M, (p0 >> np.uint64(32)) ^ w ^ k1, p0 & M
        k0 = (k0 + np.uint64(0x9E3779B9)) & M
        k1 = (k1 + np.uint64(0xBB67AE85)) & M
    return (x << np.uint64(32)) | y


def _host_subset(seed, slide, epoch, rank, n, k):
    """The documented subset: the k rows with the smallest (key, row), in increasing row order."""
    if k == n:
        return np.arange(n)
    keys = _host_keys(seed, slide, epoch, rank, n)
    order = np.lexsort((np.arange(n), keys))
    return np.sort(order[:k])


def _select(lens, ids, counts, seed, epoch=0, rank=0):
    """select_rows over slides of `lens`, bags ids with counts -> per-bag local row arrays (host)."""
    start = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=start[1:])
    off = np.zeros(len(ids) + 1, dtype=np.int32)
    np.cumsum(counts, out=off[1:])
    src = F.select_rows(torch.from_numpy(start).cuda(), torch.tensor(ids, dtype=torch.int32, device="cuda"),
                        torch.from_numpy(off).cuda(), int(off[-1]), seed, epoch, rank).cpu().numpy()
    return [src[off[b]:off[b + 1]] - start[i] for b, i in enumerate(ids)]


def _sources(bags, dtype, tmp_path):
    """The same slides as every source kind the store dtype takes, cycled so the upload switches between staging and
    device copies: numpy arrays, .npy paths, CUDA tensors of the store dtype and (bf16 stores) CPU bf16 tensors."""
    kinds = ["numpy", "path", "cuda", "numpy"] + (["cpu_bf16"] if dtype == torch.bfloat16 else [])
    out = []
    for i, b in enumerate(bags):
        k = kinds[i % len(kinds)]
        if k == "path":
            p = tmp_path / f"slide{i}.npy"
            np.save(p, b)
            out.append(str(p))
        elif k == "cpu_bf16":
            out.append(torch.from_numpy(b).to(torch.bfloat16))
        elif k == "cuda":
            out.append(torch.from_numpy(b).to(dtype).cuda())
        else:
            out.append(b)
    return out


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


# ---- 1. without augmentation: PackedBagFeeder's batches, bit for bit -----------------------------------------------------

@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("Lf", [96, 768, 1024])
def test_batches_equal_packed_feeder(dtype, Lf, tmp_path, monkeypatch):
    bags = _bags(EDGE_LENS, Lf, seed=Lf)
    srcs = _sources(bags, dtype, tmp_path)
    monkeypatch.setattr(feeder.ResidentBagFeeder, "STAGE_BYTES", 100 * Lf * 4)   # slides straddle staging chunks
    for (rank, world) in ((0, 1), (1, 2), (2, 3)):
        for shuffle, drop_last in ((False, False), (True, False), (True, True)):
            kw = dict(batch_bags=4, L_feat=Lf, device="cuda", dtype=dtype, shuffle=shuffle, seed=11, rank=rank,
                      world=world, drop_last=drop_last)
            res = feeder.ResidentBagFeeder(srcs, **kw)
            ref = feeder.PackedBagFeeder(bags, **kw)
            for epoch in (0, 1):
                res.set_epoch(epoch)
                ref.set_epoch(epoch)
                assert res.batches() == ref.batches() and len(res) == len(ref)
                got = [(X.clone(), off.clone(), ids) for X, off, ids in res]
                want = [(X.clone(), off.clone(), ids) for X, off, ids in ref]
                assert len(got) == len(want) == len(ref)
                for (X, off, ids), (Xr, offr, idsr) in zip(got, want):
                    assert ids == idsr
                    assert off.dtype == torch.int32 and torch.equal(off, offr)
                    assert X.shape == Xr.shape and torch.equal(_bits(X), _bits(Xr))


# ---- 2. the gather -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gather_equals_host_pack_on_the_host_subsets(dtype):
    lens = [50, 200, 11, 129, 1]
    types = ["Biopsy", "Resection", "Biopsy", "Resection", "Other"]
    bags = _bags(lens, 64, seed=9)
    f = feeder.ResidentBagFeeder(bags, batch_bags=5, L_feat=64, dtype=dtype)
    rng = random.Random(5)
    keep = [feeder.augmentation_rows(n, t, rng) for n, t in zip(lens, types)]
    src = np.concatenate([f._start[i] + (np.arange(n) if k is None else k) for i, (n, k) in enumerate(zip(lens, keep))])
    X = F.gather_rows(f.store, torch.from_numpy(src).cuda())
    out = torch.empty((len(src), 64), dtype=dtype)
    off = torch.zeros(len(lens) + 1, dtype=torch.int32)
    n = feeder.pack_bags_host(bags, out, off, keep_rows=keep)
    assert n == len(src) == X.shape[0]
    assert torch.equal(_bits(X.cpu()), _bits(out))


def test_gather_past_2_31_elements():
    Lf, rows = 1024, 2_200_000                       # 2.25e9 fp32 elements, 9 GB
    store = torch.empty((rows, Lf), dtype=torch.int32, device="cuda")
    col = torch.arange(Lf, dtype=torch.int64, device="cuda")
    for r0 in range(0, rows, 200_000):               # element (r, c) holds r * L + c mod 2^32: every row differs
        r = torch.arange(r0, min(rows, r0 + 200_000), dtype=torch.int64, device="cuda")
        store[r0:r0 + r.numel()] = (r[:, None] * Lf + col).to(torch.int32)
    g = torch.Generator().manual_seed(3)
    src = torch.cat([torch.randint(0, rows, (3000,), generator=g), torch.tensor([0, rows - 1, 2 ** 31 // Lf,
                                                                                  2 ** 31 // Lf - 1, rows - 2])])
    src = src.cuda()
    out = F.gather_rows(store.view(torch.float32), src)
    assert torch.equal(out.view(torch.int32), torch.index_select(store, 0, src))
    assert int((src * Lf).max()) >= 2 ** 31


# ---- 3. sampler properties ---------------------------------------------------------------------------------------------

def test_sampler_subsets_match_the_documented_rule_and_do_not_depend_on_the_batch():
    ns = [2, 3, 10, 127, 128, 129, 1000, 20_000, 70_000]
    lens = ns + ns
    keeps = [0.8] * len(ns) + [0.9] * len(ns)
    counts = [int(n * k) for n, k in zip(lens, keeps)]
    ids = list(range(len(lens)))
    seed = 0x1234_5678_9ABC
    got = _select(lens, ids, counts, seed, epoch=3, rank=1)
    for i, (n, k, rows) in enumerate(zip(lens, counts, got)):
        assert len(rows) == k and k >= 1
        assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < n
        assert np.array_equal(rows, _host_subset(seed, i, 3, 1, n, k)), (n, k)
    # the whole slide when k == n: the identity
    full = _select(lens, ids, lens, seed, epoch=3, rank=1)
    assert all(np.array_equal(r, np.arange(n)) for r, n in zip(full, lens))
    # another batch composition: other batch sizes, positions and repeated slides give every slide the same subset
    perm = [17, 5, 5, 0, 12, 8, 3]
    again = _select(lens, perm, [counts[i] for i in perm], seed, epoch=3, rank=1)
    for i, rows in zip(perm, again):
        assert np.array_equal(rows, got[i])
    # ... and epochs and ranks draw other subsets
    for epoch, rank in ((4, 1), (3, 0)):
        other = _select(lens, ids, counts, seed, epoch=epoch, rank=rank)
        assert all(not np.array_equal(a, b) for a, b, n in zip(got, other, lens) if n >= 127)


# ---- 4. sampler uniformity ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,k", [(5, 4), (6, 4), (10, 8)])
def test_sampler_draws_every_subset_equally_often(n, k):
    import math
    S = 60_000
    rows = _select([n] * S, list(range(S)), [k] * S, seed=20261022, epoch=0, rank=0)
    codes = np.stack(rows).astype(np.int64) @ (np.int64(n) ** np.arange(k, dtype=np.int64))
    _, freq = np.unique(codes, return_counts=True)
    assert len(freq) == math.comb(n, k)
    p = scipy.stats.chisquare(freq).pvalue
    assert p > 1e-4, (n, k, p, freq.min(), freq.max())


def test_sampler_includes_every_row_of_a_large_slide_at_rate_k_over_n():
    n, S = 20_000, 200
    k = int(n * 0.8)
    rows = np.stack(_select([n] * S, list(range(S)), [k] * S, seed=77, epoch=2, rank=5))
    hits = np.zeros(n)
    np.add.at(hits, rows.reshape(-1), 1)
    rate = hits / S
    for part in (rate[:1000], rate[n // 2 - 500:n // 2 + 500], rate[-1000:]):
        assert abs(part.mean() - k / n) < 0.006                          # 200 000 draws each: sd 0.0009
    assert abs(rate.mean() - k / n) < 1e-12


# ---- 5. training equivalence -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("with_labels", [False, True])
def test_trainer_fed_by_the_resident_feeder_equals_hand_built_batches(with_labels):
    from mil_b200.dp import AbmilTrainer
    lens = [700, 45, 1200, 333, 90, 2048, 5, 129]
    types = ["Biopsy", "Resection"] * 4
    bags = _bags(lens, 1024, seed=8)
    C = 2 if with_labels else 0
    onehot = torch.nn.functional.one_hot(torch.arange(len(lens)) % 2, 2).float() if with_labels else None
    torch.manual_seed(1)
    module = mil_b200.ABMIL(None, L=1024).cuda()
    tr = [AbmilTrainer(1024, 192, torch.bfloat16, device="cuda", head_classes=C) for _ in range(2)]
    for t in tr:
        t.load_from(module)
        if C:
            w = t._views(t.params)["head_w"]
            w.copy_(torch.randn(w.shape, generator=torch.Generator().manual_seed(4)) * 0.05)
    f = feeder.ResidentBagFeeder(bags, batch_bags=3, L_feat=1024, slide_types=types, augment=True, shuffle=True, seed=9,
                                 labels=onehot)
    n_batches = 0
    for epoch in (0, 1):
        f.set_epoch(epoch)
        for item in f:
            X, off, ids = item[:3]
            keep = [_host_subset(9, i, epoch, 0, lens[i], feeder.augmentation_count(lens[i], types[i])) for i in ids]
            want = torch.cat([torch.from_numpy(bags[i][k]) for i, k in zip(ids, keep)]).to(torch.bfloat16).cuda()
            want_off = torch.tensor([0] + np.cumsum([len(k) for k in keep]).tolist(), dtype=torch.int32, device="cuda")
            assert torch.equal(off, want_off) and torch.equal(_bits(X), _bits(want))
            if with_labels:
                y = item[3]
                assert y.is_contiguous() and y.dtype == torch.float32 and torch.equal(y.cpu(), onehot[ids])
                tr[0].step_labels(X, off, y)
                tr[1].step_labels(want, want_off, onehot[ids].cuda())
            else:
                tr[0].step(X, off)
                tr[1].step(want, want_off)
            n_batches += 1
    assert n_batches == 6
    assert torch.equal(tr[0].params, tr[1].params)


# ---- 6. rotation safety ------------------------------------------------------------------------------------------------

def test_batches_stay_intact_until_the_batch_after_next():
    lens = [300, 17, 1, 950, 64, 129, 511, 2, 77, 400, 33]
    bags = _bags(lens, 256, seed=4)
    f = feeder.ResidentBagFeeder(bags, batch_bags=3, L_feat=256, dtype=torch.bfloat16)
    torch.manual_seed(0)
    m = mil_b200.ABMIL(None, L=256).cuda().eval()
    held = []
    for X, off, ids in f:
        want = torch.cat([torch.from_numpy(bags[i]) for i in ids]).to(torch.bfloat16).cuda()
        want_off = torch.tensor([0] + np.cumsum([lens[i] for i in ids]).tolist(), dtype=torch.int32, device="cuda")
        assert torch.equal(off, want_off) and torch.equal(_bits(X), _bits(want))
        assert torch.equal(m.forward_csr(X, off), m.forward_csr(want, want_off))
        held.append((X, off, want, want_off))
        if len(held) >= 2:                                                # the previous batch is still intact
            Xp, offp, wp, wop = held[-2]
            assert Xp.data_ptr() != X.data_ptr()
            assert torch.equal(_bits(Xp), _bits(wp)) and torch.equal(offp, wop)
    assert len(held) == 4


# ---- 7. errors ---------------------------------------------------------------------------------------------------------

def test_errors():
    bags = _bags([4, 1, 6], 64, seed=1)
    with pytest.raises(mil_b200.MilB200Error, match="would keep 0"):     # int(1 * 0.8) = 0 rows under augmentation
        feeder.ResidentBagFeeder(bags, batch_bags=2, L_feat=64, slide_types=["Biopsy", "Resection", "Biopsy"],
                                 augment=True)
    feeder.ResidentBagFeeder(bags, batch_bags=2, L_feat=64, slide_types=["Biopsy", "Resection", "Biopsy"])   # no augment
    with pytest.raises(ValueError, match="features"):                     # feature width mismatch
        feeder.ResidentBagFeeder(bags + _bags([3], 32, seed=2), batch_bags=2, L_feat=64)
    odd = _bags([4, 5], 100, seed=3)                                      # 100 bf16 = 200 bytes a row
    with pytest.raises(mil_b200.MilB200Error, match="multiple of 16"):
        feeder.ResidentBagFeeder(odd, batch_bags=2, L_feat=100)
    store = torch.zeros((9, 100), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(mil_b200.MilB200Error, match=r"code -5\).*multiple of 16"):
        F.gather_rows(store, torch.arange(3, device="cuda"))
    # larger than free device memory: 4 slides of 2^27 broadcast rows are 256 GB in bf16 and nothing is allocated
    row = np.ones((1, 1024), dtype=np.float32)
    huge = [np.broadcast_to(row, (1 << 27, 1024)) for _ in range(4)]
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    with pytest.raises(mil_b200.MilB200Error) as e:
        feeder.ResidentBagFeeder(huge, batch_bags=2, L_feat=1024)
    need = 4 * (1 << 27) * 2048 + 2 * 2 * (1 << 27) * (2048 + 8)
    assert f"need {need} bytes" in str(e.value) and "bytes free" in str(e.value)
    assert torch.cuda.memory_allocated() == before
