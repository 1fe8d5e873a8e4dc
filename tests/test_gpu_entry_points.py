"""The batch entry points against each other: the plain approximate entry points give what their _ex forms give with every
hit and no distances, a single-copy host batch reports exactly the PCIe bytes of the arrays it moved, and every count-only
device form gives the offsets of its full device form."""
import ctypes as C

import numpy as np
import pytest

from collection_truth import random_starts

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def on_device(q, off):
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(q if q.size else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    torch.cuda.synchronize()
    return d_q, d_off


def device_array(view, dtype):
    """A DeviceResult array view (or None) as a host numpy array of `dtype` (None stays None)."""
    import torch
    if view is None:
        return None
    if view.__cuda_array_interface__["shape"][0] == 0:
        return np.zeros(0, dtype)
    torch.cuda.synchronize()
    return torch.as_tensor(view, device=torch.device("cuda", 0)).cpu().numpy().view(dtype)


def device_arrays(r, Q):
    """Every array of a device result, on the host."""
    return {"offsets": device_array(r.offsets(), np.uint64),
            "status": device_array(r.status(), np.uint8) if Q else np.zeros(0, np.uint8),
            "positions": device_array(r.positions(), np.uint32) if r.positions_ptr else None,
            "distances": device_array(r.distances(), np.uint8),
            "best_distances": device_array(r.best_distances(), np.uint8),
            "seed_offsets": device_array(r.seed_offsets(), np.uint32),
            "kmer_counts": device_array(r.kmer_counts(), np.uint32)}


def host_arrays(r):
    return {"offsets": r.offsets, "status": r.status, "positions": r.positions, "distances": r.distances,
            "best_distances": r.best_distance, "seed_offsets": r.seed_offsets, "kmer_counts": r.kmer_counts}


def assert_same(a, b, label):
    assert a.keys() == b.keys(), label
    for name in a:
        if a[name] is None or b[name] is None:
            assert a[name] is None and b[name] is None, f"{label}: {name}"
        else:
            assert a[name].dtype == b[name].dtype and np.array_equal(a[name], b[name]), f"{label}: {name}"


def text_and_batch(kb, collection, seed):
    from kmer_index_b200 import synth
    text = synth.random_text(40_000, 4, seed)
    text[2000:2300] = 1                                  # a repeat: long candidate lists
    q, off = synth.stress_queries(text, 300, 4, 60, 4, seed + 1)
    starts = random_starts(text.size, 40, np.random.default_rng(seed + 2), short=6) if collection else None
    return text, starts, q, off


def make_index(kb, text, starts, ks):
    ix = kb.KmerIndex(text, 4, ks, mode=kb.MODE_CORRECT if starts is not None else kb.MODE_REFERENCE_EXACT)
    if starts is not None:
        ix.attach_records(starts)
    return ix


@pytest.mark.parametrize("collection", [False, True], ids=["plain", "collection"])
def test_plain_approx_equals_ex_with_every_hit(kb, collection):
    """kmer_b200_search_approx_batch, _search_approx_batch_device and _count_approx_batch_device against their _ex forms
    with {e, HITS_ALL, 0, 0}, called through the C ABI: every array identical, no distances and no best distances."""
    from kmer_index_b200 import _capi
    L = _capi.lib()
    text, starts, q, off = text_and_batch(kb, collection, 11)
    Q = off.size - 1
    max_len = int(np.diff(off.astype(np.int64)).max())
    d_q, d_off = on_device(q, off)
    with make_index(kb, text, starts, [7, 11]) as ix:
        for e in (0, 2):
            opt = _capi.ApproxOptions(e, _capi.HITS_ALL, 0, 0)
            label = f"{'collection' if collection else 'plain'} e={e}"
            r_plain, r_ex = C.c_void_p(), C.c_void_p()
            _capi.check(L.kmer_b200_search_approx_batch(ix.handle, q.ctypes.data, off.ctypes.data, Q, e, C.byref(r_plain)))
            _capi.check(L.kmer_b200_search_approx_batch_ex(ix.handle, q.ctypes.data, off.ctypes.data, Q, C.byref(opt),
                                                           C.byref(r_ex)))
            plain, ex = ix._host_result(r_plain, Q, True), ix._host_result(r_ex, Q, True)
            assert plain.distances is None and plain.best_distance is None and plain.positions.size > 0, label
            assert_same(host_arrays(plain), host_arrays(ex), f"{label} host")
            for fn_plain, fn_ex, form in ((L.kmer_b200_search_approx_batch_device, L.kmer_b200_search_approx_batch_device_ex, "device"),
                                          (L.kmer_b200_count_approx_batch_device, L.kmer_b200_count_approx_batch_device_ex, "count")):
                a = ix._device_call(fn_plain, d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e)
                b = ix._device_call(fn_ex, d_q.data_ptr(), d_off.data_ptr(), Q, max_len, C.byref(opt))
                got_a, got_b = device_arrays(a, Q), device_arrays(b, Q)
                a.free()
                b.free()
                assert got_a["distances"] is None and got_a["best_distances"] is None, f"{label} {form}"
                assert (got_a["positions"] is None) == (form == "count"), f"{label} {form}"
                assert_same(got_a, got_b, f"{label} {form}")
                assert np.array_equal(got_a["offsets"], plain.offsets), f"{label} {form}"


def test_single_copy_transfer_accounting(kb):
    """A small host batch takes the single-copy path and reports the bytes of the arrays it moved: the ranks and offsets
    in; offsets, status, positions and whatever else the result holds out."""
    from kmer_index_b200 import synth
    text = synth.random_text(40_000, 4, 21)
    q, off = synth.stress_queries(text, 300, 8, 60, 4, 22)
    Q = off.size - 1
    n_sym = int(off[-1] - off[0])
    h2d = n_sym + 8 * (Q + 1)
    with kb.KmerIndex(text, 4, [7, 11]) as ix:
        r = ix.search_batch(q, off, kb.MODE_CORRECT)
        assert r.positions.size > 0
        assert ix.last_search_host_path()["pipeline"] == "single copy"
        assert ix.last_search_transfer() == (h2d, 8 * (Q + 1) + Q + 4 * r.positions.size)

        r = ix.search_approx(q, off, 2, hits="strata", strata=1, distances=True)
        assert r.positions.size > 0 and r.distances.size == r.positions.size and r.best_distance.size == Q
        assert ix.last_search_host_path()["pipeline"] == "single copy"
        assert ix.last_search_transfer() == (h2d, 8 * (Q + 1) + Q + 4 * r.positions.size + r.distances.size + r.best_distance.size)

        # random 60-symbol queries: no window of the text within one mismatch
        zq = synth.random_text(60 * 20, 4, 23)
        zoff = np.arange(0, 60 * 21, 60, dtype=np.uint64)
        r = ix.search_approx(zq, zoff, 1, hits="strata", strata=1, distances=True)
        assert r.positions.size == 0 and r.distances is not None and r.distances.size == 0 and r.best_distance.size == 20
        assert ix.last_search_transfer() == (zq.size + 8 * 21, 8 * 21 + 20 + 20)

        r = ix.seeds(q, off, k=11)
        assert r.positions.size > 0 and r.kmer_counts.size > 0
        assert ix.last_search_host_path()["pipeline"] == "single copy"
        assert ix.last_search_transfer() == (h2d, 8 * (Q + 1) + Q + 8 * r.positions.size + 4 * r.kmer_counts.size)


@pytest.mark.parametrize("collection", [False, True], ids=["plain", "collection"])
def test_count_only_offsets_equal_full(kb, collection):
    """The offsets of every count-only device form equal those of the matching full device call: exact, approximate
    under each hit strategy, and seeding."""
    text, starts, q, off = text_and_batch(kb, collection, 31)
    Q = off.size - 1
    max_len = int(np.diff(off.astype(np.int64)).max())
    d_q, d_off = on_device(q, off)
    args = (d_q.data_ptr(), d_off.data_ptr(), Q, max_len)
    mode = kb.MODE_CORRECT if collection else kb.MODE_DEFAULT
    pairs = [("exact", lambda: ix.search_batch_device(*args, mode), lambda: ix.count_batch_device(*args, mode)),
             ("seeds", lambda: ix.seeds_batch_device(*args, k=11), lambda: ix.count_seeds_batch_device(*args, k=11))]
    for hits in ("all", "all_best", "single_best", "strata"):
        pairs.append((f"approx {hits}",
                      lambda h=hits: ix.search_approx_batch_device(*args, 2, hits=h, strata=1, distances=True),
                      lambda h=hits: ix.count_approx_batch_device(*args, 2, hits=h, strata=1, distances=True)))
    with make_index(kb, text, starts, [7, 11]) as ix:
        for label, full_fn, count_fn in pairs:
            full, count = full_fn(), count_fn()
            got_full, got_count = device_arrays(full, Q), device_arrays(count, Q)
            full.free()
            count.free()
            assert got_full["positions"] is not None and got_count["positions"] is None, label
            assert got_full["offsets"][-1] > 0, label
            assert np.array_equal(got_full["offsets"], got_count["offsets"]), label
            assert np.array_equal(got_full["status"], got_count["status"]), label
