"""Host-fed peer steps without a GPU: the owned plan the device derives from a staged batch (peer_plan_kernel in csrc/peer.cu,
restated in numpy) equals the host plan of the resident stream (peer_batch_plan); the validation every rank makes before it
enqueues anything (check_host_batch) rejects bad batches with the reference's exceptions; the shares partition every batch;
and the new C entry points reject NULL arguments before they touch a device."""
import ctypes
import os
import re

import numpy as np
import pytest

from lstep_b200 import _lib
from lstep_b200.peer import check_host_batch, peer_batch_plan, share_of

INVALID_ARG = 1


def device_plan(ids: np.ndarray, world: int, rank: int, threads: int):
    """peer_plan_kernel step by step: blocks of `threads` ids; per warp a ballot of the owned ids, a thread's rank in the warp
    = popcount of the ballot's lower lanes; an exclusive scan of the warp counts; a running base across blocks."""
    ids_mine, pos_mine = np.full(len(ids), -1, np.int64), np.full(len(ids), -1, np.int64)
    base = 0
    for i0 in range(0, len(ids), threads):
        blk = np.full(threads, -1, np.int64)
        part = ids[i0:i0 + threads]
        blk[:len(part)] = part
        mine = (blk >= 0) & (blk % world == rank)
        warps = mine.reshape(-1, 32)
        counts = warps.sum(axis=1)
        woff = np.concatenate([[0], np.cumsum(counts)[:-1]])
        for w in range(warps.shape[0]):
            ballot = sum(1 << l for l in range(32) if warps[w, l])
            for lane in range(32):
                if warps[w, lane]:
                    p = base + woff[w] + bin(ballot & ((1 << lane) - 1)).count("1")
                    ids_mine[p] = blk[w * 32 + lane]
                    pos_mine[p] = i0 + w * 32 + lane
        base += int(counts.sum())
    return ids_mine[:base], pos_mine[:base]


def _threads(n_ids: int) -> int:  # the launch of peer_plan_mine
    return min(1024, (n_ids + 31) // 32 * 32)


def _batches():
    rng = np.random.default_rng(11)
    out = []
    for n in (1, 7, 200, 777, 2000):  # random, ragged
        out.append(("random", rng.integers(1, 10_000, n), rng.integers(1, 10_000, n)))
    hub = rng.integers(1, 50_000, 1500)
    out.append(("hub", np.where(rng.random(1500) < 0.7, 3, hub), rng.integers(1, 50_000, 1500)))
    out.append(("one_owner", 8 * rng.integers(1, 500, 300), 8 * rng.integers(1, 500, 300)))  # ranks != 0 own nothing at world 2, 8
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_device_plan_equals_host_plan(world):
    for kind, src, dst in _batches():
        src, dst = src.astype(np.int64), dst.astype(np.int64)
        ids = np.unique(np.concatenate([src, dst]))
        owned = 0
        for rank in range(world):
            want = peer_batch_plan(src, dst, len(src), world, rank)
            got_ids, got_pos = device_plan(ids, world, rank, _threads(len(ids)))
            assert np.array_equal(got_ids, want["mine"]), (kind, world, rank)
            assert np.array_equal(got_pos, want["pos"]), (kind, world, rank)
            assert np.array_equal(ids[got_pos], got_ids)
            owned += len(got_ids)
        assert owned == len(ids), kind  # the owners' lists partition the batch's ids


@pytest.mark.parametrize("world", [1, 2, 3, 8, 16])
def test_shares_partition_every_batch(world):
    for n in (1, 2, 3, 7, 8, 15, 200, 2000, 1999):
        cover = []
        for rank in range(world):
            q_off, q_rows = share_of(n, world, rank)
            assert q_rows >= 0
            cover.extend(range(q_off, q_off + q_rows))
            assert (q_off, q_rows) == peer_batch_plan(np.arange(n), np.arange(n), n, world, rank)["share"][0]
        assert cover == list(range(n)), (world, n)


def test_validation_rejects_bad_batches_and_changes_nothing():
    V1, B = 100, 16
    rng = np.random.default_rng(2)
    src, dst = rng.integers(1, V1, B), rng.integers(1, V1, B)
    t = np.sort(rng.random(B) * 100.0)
    qs = [src, dst, rng.integers(1, V1, B)]
    ing = (V1, 0.0, 1)  # (sampler rows, last time ingested, first edge id)
    keep = [a.copy() for a in (src, dst, t, *qs)]

    def rejects(exc, *args, **kw):
        with pytest.raises(exc):
            check_host_batch(*args, **kw)
        for a, b in zip((src, dst, t, *qs), keep):  # nothing the caller passed has changed
            assert np.array_equal(a, b)

    check_host_batch(src, dst, t, qs, V1, B, ingest=ing)  # the good batch passes
    rejects(ValueError, src, dst[:-1], t, qs, V1, B)  # wrong lengths
    rejects(ValueError, src, dst, t, [q[:-1] for q in qs], V1, B)
    rejects(ValueError, src[:0], dst[:0], t[:0], [q[:0] for q in qs], V1, B)  # empty
    for bad in (V1, -1):  # out-of-range ids: endpoints and queries
        s2 = src.copy()
        s2[3] = bad
        rejects(IndexError, s2, dst, t, qs, V1, B)
        q2 = [q.copy() for q in qs]
        q2[2][5] = bad
        rejects(IndexError, src, dst, t, q2, V1, B)
    rejects(IndexError, src, dst, t, qs, V1, B, ingest=(int(src.max()), 0.0, 1))  # outside the sampler's rows
    t2 = t.copy()
    t2[5] = t2[4] - 1.0
    rejects(ValueError, src, dst, t2, qs, V1, B, ingest=ing)  # unsorted times
    rejects(ValueError, src, dst, t, qs, V1, B, ingest=(V1, float(t[0]) + 1.0, 1))  # before the last time ingested
    for bad in (np.nan, np.inf):
        t3 = t.copy()
        t3[-1] = bad
        rejects(ValueError, src, dst, t3, qs, V1, B, ingest=ing)  # non-finite times
    rejects(ValueError, src, dst, t, qs, V1, B - 1)  # longer than batch_size
    rejects(ValueError, src, dst, t, qs, V1, B, ingest=(V1, 0.0, 2 ** 31 - B + 1))  # edge ids past int32
    check_host_batch(src, dst, t, qs, V1, B, ingest=(V1, 0.0, 2 ** 31 - B))  # (the last one that fits)
    rejects(ValueError, src, dst, t, qs * 3, V1, B)  # more than 8 query sets
    ids = np.unique(np.concatenate([src, dst]))
    check_host_batch(src, dst, t, qs, V1, B, ids=ids)
    rejects(ValueError, src, dst, t, qs, V1, B, ids=ids[::-1].copy())  # ids not sorted


def test_peer_host_entry_points_reject_null_arguments():
    lib = _lib.load(require_device=False)
    desc, cl, csr, grp = _lib.PEStreamDesc(), _lib.ChangeLog(), _lib.CSR(), _lib.PeerGroup()
    src = (ctypes.c_int64 * 4)(1, 2, 3, 4)
    t = (ctypes.c_double * 4)(1.0, 2.0, 3.0, 4.0)
    G = (ctypes.c_float * 4)()
    not_null = ctypes.c_void_p(8)  # (a non-NULL stepper is never dereferenced once another argument is NULL)

    def step(h, s, c, g):
        ticket = ctypes.c_int64(-1)
        return lib.lstep_pe_step_peer_host(h, s, c, csr, g, 4, src, src, t, None, 0, 0, 0, G, None, 0, None, 20, _lib.PEMLP(), _lib.PEMLP(),
                                           None, 0, None, 0, 1000, 7, None, ctypes.byref(ticket))

    def steps(h, s, c, g):
        head, ln, done, epoch = ctypes.c_int(0), ctypes.c_int(100), ctypes.c_int64(-1), ctypes.c_uint32(0)
        res = (ctypes.c_float * 4)()
        rc = lib.lstep_pe_steps_peer_host(h, s, c, csr, g, 4, 4, src, src, t, None, 0, ctypes.byref(head), ctypes.byref(ln), G, 20,
                                          _lib.PEMLP(), _lib.PEMLP(), None, 0, None, ctypes.byref(epoch), 1000, None, res, ctypes.byref(done))
        assert done.value == 0 and head.value == 0 and epoch.value == 0
        return rc

    for fn in (step, steps):
        assert fn(None, desc, cl, grp) == INVALID_ARG
        assert fn(not_null, None, cl, grp) == INVALID_ARG
        assert fn(not_null, desc, None, grp) == INVALID_ARG
        assert fn(not_null, desc, cl, None) == INVALID_ARG


def test_no_source_names_the_batched_copy_api():
    """The batched async copies (the Memcpy...BatchAsync family of the runtime and driver APIs) are not used anywhere in the
    project's sources and scripts: copies go through cudaMemcpyAsync or copy kernels."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pat = re.compile("cu(da)?" + "Memcpy" + "(3D)?" + "Batch" + "Async")
    hits = []
    for d, dirs, files in os.walk(root):
        dirs[:] = [x for x in dirs if not x.startswith(".") and x not in ("__pycache__", "_ref")]
        for f in files:
            if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp", ".c", ".py", ".sh")) or f in ("Makefile", "CMakeLists.txt"):
                p = os.path.join(d, f)
                with open(p, errors="replace") as fh:
                    if pat.search(fh.read()):
                        hits.append(os.path.relpath(p, root))
    assert not hits, hits
