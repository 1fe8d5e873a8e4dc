"""bench.py --dump-outputs: two runs with the same arguments write the same files, within 64 MB, and the files hold the
oracle's answer for the benchmark's own inputs (config 1: 10^4 queries, all of them in the sample, on the GPU); the
seeded sample of a larger batch and its cut to the byte budget on the CPU, with a result held in host tensors."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_results_equal


class _HostResult:
    """A search result of Q queries in host tensors, shaped like kmer_index_b200.DeviceResult for bench.dump_result."""

    def __init__(self, counts, seed=0):
        import torch
        rng = np.random.default_rng(seed)
        self.off = np.zeros(counts.size + 1, dtype=np.int64)
        np.cumsum(counts, out=self.off[1:])
        self.pos = rng.integers(0, 1 << 32, int(self.off[-1]), dtype=np.uint64).astype(np.uint32)
        self.st = rng.integers(0, 3, counts.size).astype(np.uint8)
        self.offsets = lambda: torch.from_numpy(self.off)
        self.positions = lambda: torch.from_numpy(self.pos.view(np.int32))
        self.status = lambda: torch.from_numpy(self.st)


def _dump(tmp_path, name, counts, count_only=False):
    import bench
    res = _HostResult(counts)
    bench.dump_result(str(tmp_path / name), res, counts.size, "cpu", count_only)
    files = {n[:-4]: np.load(tmp_path / name / n) for n in os.listdir(tmp_path / name)}
    size = sum(os.path.getsize(tmp_path / name / n) for n in os.listdir(tmp_path / name))
    assert all(v.dtype in (np.float32, np.float64) for v in files.values())
    ids = files["query_ids"].astype(np.int64)
    assert np.all(np.diff(ids) > 0) and np.array_equal(np.diff(files["offsets"]).astype(np.int64), counts[ids])
    assert np.array_equal(files["status"], res.st[ids])
    if count_only:
        assert "positions" not in files
    else:
        want = [res.pos[res.off[i]:res.off[i + 1]] for i in ids]
        assert np.array_equal(files["positions"], np.concatenate(want or [[]]).astype(np.float64))
    return ids, size


def test_dump_result_sample_budget_and_modes(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_QUERIES", 5000)
    rng = np.random.default_rng(3)
    counts = rng.integers(0, 4, 50_000)
    ids, size = _dump(tmp_path, "a", counts)                 # a seeded sample: it depends on Q alone
    again, _ = _dump(tmp_path, "b", rng.integers(0, 4, 50_000))
    assert ids.size == 5000 and np.array_equal(ids, again) and size <= bench.DUMP_BYTES
    monkeypatch.setattr(bench, "DUMP_BYTES", 5000 * 20 + 4096 + 8 * 3000)
    ids, size = _dump(tmp_path, "c", counts)                 # hit lists past the budget: the longest prefix that fits
    assert 0 < ids.size < 5000 and size <= bench.DUMP_BYTES
    assert counts[ids].sum() <= 3000 < counts[ids].sum() + counts[np.setdiff1d(again, ids)[0]]
    ids, _ = _dump(tmp_path, "d", counts, count_only=True)  # count-only: no positions file and no cut
    assert ids.size == 5000
    ids, _ = _dump(tmp_path, "e", np.zeros(700, dtype=np.int64))   # no hits at all: an empty positions file
    assert ids.size == 700 and np.load(tmp_path / "e" / "positions.npy").size == 0


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "2", "--warmup", "1",
           "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    files = {n[:-4]: np.load(os.path.join(out_dir, n)) for n in os.listdir(out_dir)}
    return line, files, sum(os.path.getsize(os.path.join(out_dir, n)) for n in os.listdir(out_dir))


@pytest.mark.gpu
def test_dump_outputs_reproducible_and_equal_to_the_oracle(tmp_path, oracle_mod):
    import torch

    import bench
    from kmer_index_b200 import _capi, synth
    line, got, size = _bench(tmp_path / "a")
    _, again, _ = _bench(tmp_path / "b")
    assert sorted(got) == ["offsets", "positions", "query_ids", "status"]
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert all(np.array_equal(got[k], again[k]) for k in got)
    assert size <= 64 << 20
    wl = bench.WORKLOADS["c1"]
    sigma, ks, n, Q, (m_lo, m_hi) = wl["sigma"], wl["ks"], wl["n"], wl["Q"], wl["m"]
    assert line["steps"] == 2 and line["config"]["queries"] == Q
    assert np.array_equal(got["query_ids"], np.arange(Q))
    # the benchmark's inputs, made the way bench.py makes them
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(bench.QUERY_SEED)
    lens = torch.randint(m_lo, m_hi + 1, (Q,), generator=g, device=dev, dtype=torch.int64).cpu().numpy()
    off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    q = torch.empty(int(off[-1]), dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(q.data_ptr(), q.numel(), 0, sigma, bench.QUERY_SEED ^ 0xC0FFEE,
                                                         torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    with oracle_mod.Oracle(synth.random_text(n, sigma, bench.TEXT_SEED), sigma, ks) as o:
        want = o.search(q.cpu().numpy(), off)
        ub = o.last_ub
    assert want[1].size > 0
    assert_results_equal((got["offsets"].astype(np.uint64), got["positions"].astype(np.uint32), got["status"].astype(np.uint8)),
                         want, skip=ub, label="bench.py --dump-outputs, config 1")
