"""Config 5 through the host C ABI (kmer_b200_search_batch, kmer_b200_create) under each share of raw chunks
(KMER_B200_HOST_RAW_PCT), pinned and pageable, and a sigma-27 batch of as many queries: which share is the fastest on
this box. Prints one line per setting.
usage: python profiles/tools/host_path_sweep.py [text_symbols] [queries]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import torch

import kmer_index_b200 as kb
from kmer_index_b200 import _capi

n = int(sys.argv[1]) if len(sys.argv) > 1 else 3_000_000_000
Q = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000_000
dev = torch.device("cuda", 0)
L = _capi.lib()
text = torch.empty(n, dtype=torch.uint8, device=dev)
_capi.check(L.kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, 205, None))
g = torch.Generator(device=dev)
g.manual_seed(1239)
lens = torch.randint(16, 65, (Q,), generator=g, device=dev, dtype=torch.int64)
off = torch.zeros(Q + 1, dtype=torch.int64, device=dev)
torch.cumsum(lens, 0, out=off[1:])
n_sym = int(off[-1].item())
q = torch.empty(n_sym, dtype=torch.uint8, device=dev)
_capi.check(L.kmer_b200_synth_ranks_device(q.data_ptr(), n_sym, 0, 4, 1239 ^ 0xC0FFEE, None))
torch.cuda.synchronize()
h_q, h_off, h_text = q.cpu().pin_memory(), off.cpu().pin_memory(), text.cpu().pin_memory()
p_q, p_off = h_q.numpy().copy(), h_off.numpy().copy()      # the same batch in pageable memory
del q, off, lens
ix = kb.KmerIndex(None, 4, [16], text_device_ptr=text.data_ptr(), n=n)
torch.cuda.synchronize()


def run(label, env, qa, oa, reps=3):
    os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
    os.environ.update(env)
    best, fp = 1e30, None
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        r = ix.search_batch(qa, oa.view(np.uint64), copy=False)
        dt = time.perf_counter() - t0
        fp = (int(r.offsets[-1]), int(r.status.sum()))
        r.free()
        best = min(best, dt)
    print(f"search  {label:44s} {best * 1e3:8.1f} ms  {Q / best / 1e9:6.2f} Gq/s  h2d {ix.last_search_transfer()[0] / 1e9:5.2f} GB  "
          f"{ix.last_search_host_path()}  hits/status {fp}", flush=True)


run("pinned, default", {}, h_q.numpy(), h_off.numpy())
run("pinned, raw chunks only (round-2 start)", {"KMER_B200_HOST_RAW_PCT": "100"}, h_q.numpy(), h_off.numpy())
run("pinned, streaming pack only", {"KMER_B200_HOST_RAW_PCT": "0"}, h_q.numpy(), h_off.numpy())
for pct in (20, 30, 40, 50, 60):
    run(f"pinned, streaming pack + {pct} % raw", {"KMER_B200_HOST_RAW_PCT": str(pct)}, h_q.numpy(), h_off.numpy())
run("pageable, default (streaming pack)", {}, p_q, p_off)
run("pageable, raw chunks (driver-staged copies)", {"KMER_B200_HOST_RAW_PCT": "100"}, p_q, p_off, reps=1)
os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
ix.close()
del text

# sigma 27 (8-bit words: packing saves no link bytes): the same query lengths over a 200 Mbp text, k = 5
n27 = min(n, 200_000_000)
text = torch.empty(n27, dtype=torch.uint8, device=dev)
_capi.check(L.kmer_b200_synth_ranks_device(text.data_ptr(), n27, 0, 27, 206, None))
q = torch.from_numpy(p_q).to(dev)
_capi.check(L.kmer_b200_synth_ranks_device(q.data_ptr(), n_sym, 0, 27, 1240, None))
torch.cuda.synchronize()
h_q.copy_(q.cpu())
p_q = h_q.numpy().copy()
del q
ix = kb.KmerIndex(None, 27, [5], text_device_ptr=text.data_ptr(), n=n27)
torch.cuda.synchronize()
run("sigma 27 pinned, default (raw chunks)", {}, h_q.numpy(), h_off.numpy())
run("sigma 27 pinned, streaming pack only", {"KMER_B200_HOST_RAW_PCT": "0"}, h_q.numpy(), h_off.numpy())
run("sigma 27 pageable, default (streaming pack)", {}, p_q, p_off)
run("sigma 27 pageable, raw chunks (driver-staged copies)", {"KMER_B200_HOST_RAW_PCT": "100"}, p_q, p_off, reps=1)
os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
ix.close()
del text
if os.environ.get("SWEEP_NO_BUILD"):
    sys.exit(0)


def build(label, env, src, reps=2):
    os.environ.pop("KMER_B200_NO_TEXT_PIPELINE", None)
    os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
    os.environ.update(env)
    best = 1e30
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        b = kb.KmerIndex(src, 4, [16])
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
        b.close()
    print(f"build   {label:44s} {best * 1e3:8.1f} ms  {n / best / 1e9:6.2f} Gbases/s", flush=True)


build("pinned text, default", {}, h_text.numpy())
build("pinned text, plain upload", {"KMER_B200_NO_TEXT_PIPELINE": "1"}, h_text.numpy())
for pct in (0, 30, 50, 70):
    build(f"pinned text, streaming pack + {pct} % raw", {"KMER_B200_HOST_RAW_PCT": str(pct)}, h_text.numpy())
p_text = h_text.numpy().copy()
build("pageable text, default (streaming pack)", {}, p_text, reps=1)
build("pageable text, plain upload", {"KMER_B200_NO_TEXT_PIPELINE": "1"}, p_text, reps=1)
