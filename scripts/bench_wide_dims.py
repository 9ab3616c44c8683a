"""Tensor-core vs exact IVF search across embedding widths on one GPU.

    python scripts/bench_wide_dims.py [--dims 384,512,768,1024,1536,2048] [--steps 20] [--warmup 5] [--out FILE]

Per width D: 1M synthetic rows (fvdb_synth_rows_device), nlist 1024 trained on 64 rows per list, nprobe 32,
1024-query batches, k = 10.  The same handle is timed in tensor-core mode and in exact mode (median of the
per-step device-event times of `--steps` warm synchronous batches, four rotating query sets), every query of one
batch is compared bit for bit between the two modes, and recall@10 is taken against an exact flat scan of all
rows.  The scan line is the posting-list scan kernel's device time (fvdb_stats.last_scan_ms) and the batch's
algorithmic bytes (each probed list's rows, norms and ids read once), over the 6544 GB/s HBM copy peak measured
on the B200 the repository's figures use.  The D = 512 line is the baseline the wider ones compare with: kernel R
runs 64-query items up to D = 512, 32-query items up to 1024 and 16-query items above.  Prints one JSON object
(also written to --out) with the card's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_ROWS, NLIST, NPROBE, NQ, K = 1_000_000, 1024, 32, 1024, 10
SIGMA, SEED, SEED_Q, TRAIN_ITERS, N_QSETS = 1.0, 1234, 5678, 10, 4
HBM_PEAK_GBS = 6544.3   # measured HBM copy bandwidth of one B200 (SURVEY.md)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=10).stdout.strip()
        name, power, clk = [p.strip() for p in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # the measurement stands without it, but says so
        return {"error": repr(e)}


def build(torch, lib, eng, d):
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    n_comp = 4 * NLIST
    n_train = 64 * NLIST
    stride = N_ROWS // n_train
    train = torch.empty((n_train, d), dtype=torch.float32, device=dev)
    assert lib.fvdb_synth_rows_strided_device(train.data_ptr(), 0, n_train, d, n_comp, SIGMA, SEED, 64, stride,
                                              stream) == 0
    blk = torch.arange(NLIST, device=dev)
    init = train[blk * 64 + (blk // (NLIST // 16)) % 64].contiguous()   # one seed per mixture component
    eng.train_device(train.data_ptr(), n_train, NLIST, TRAIN_ITERS, init.data_ptr(), SEED)
    torch.cuda.synchronize()
    del train, init
    ch = 1 << 17
    buf = torch.empty((ch, d), dtype=torch.float32, device=dev)
    for r0 in range(0, N_ROWS, ch):
        n = min(ch, N_ROWS - r0)
        assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, d, n_comp, SIGMA, SEED, stream) == 0
        ids = torch.arange(r0, r0 + n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        eng.ivf_add_device(buf.data_ptr(), ids.data_ptr(), n, 1, 0)
    torch.cuda.synchronize()
    return buf


def queries(torch, lib, d, s):
    from fabstir_vectordb_b200 import synth
    q = torch.empty((NQ, d), dtype=torch.float32, device="cuda")
    assert lib.fvdb_synth_queries_device(q.data_ptr(), s * NQ, NQ, d, N_ROWS, 4 * NLIST, SIGMA, SEED,
                                         synth.default_qnoise(d, SIGMA), SEED_Q,
                                         torch.cuda.current_stream().cuda_stream) == 0
    return q


def truth(torch, lib, d, q, buf):
    """Exact top-k over all rows: the exact flat-tier scan of a second handle."""
    from fabstir_vectordb_b200 import Engine, _lib as L
    g = Engine(d, k_max=16)
    g.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    stream = torch.cuda.current_stream().cuda_stream
    ch = buf.shape[0]
    for r0 in range(0, N_ROWS, ch):
        n = min(ch, N_ROWS - r0)
        assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, d, 4 * NLIST, SIGMA, SEED, stream) == 0
        ids = torch.arange(r0, r0 + n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        g.flat_add_device(buf.data_ptr(), ids.data_ptr(), n)
    out = [torch.empty((NQ, K), dtype=torch.int32, device="cuda"),
           torch.empty((NQ, K), dtype=torch.float32, device="cuda"),
           torch.empty((NQ,), dtype=torch.int32, device="cuda")]
    g.search_device(q.data_ptr(), NQ, K, 0, L.TIER_RECENT, 0, 0, *(t.data_ptr() for t in out))
    torch.cuda.synchronize()
    res = out[0].cpu().numpy().view(np.uint32).copy(), out[2].cpu().numpy().view(np.uint32).copy()
    g.close()
    return res


def recall(ids, cnt, t_ids, t_cnt):
    acc = 0.0
    for i in range(ids.shape[0]):
        t = set(t_ids[i, :t_cnt[i]].tolist())
        acc += len(t & set(ids[i, :cnt[i]].tolist())) / max(1, len(t))
    return acc / ids.shape[0]


def time_mode(torch, eng, qs, out, steps, warmup):
    """Median per-step device time of synchronous batches; the stats of the last step; the last batch's result
    on query set 0."""
    from fabstir_vectordb_b200 import _lib as L

    def step(i):
        eng.search_device(qs[i % N_QSETS].data_ptr(), NQ, K, NPROBE, L.TIER_HISTORICAL, 0, 0,
                          *(t.data_ptr() for t in out))

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    ms, scan_ms, fb = [], [], 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(steps):
        ev0.record()
        step(i)
        ev1.record()
        torch.cuda.synchronize()
        ms.append(ev0.elapsed_time(ev1))
        st = eng.stats()
        scan_ms.append(st.last_scan_ms)
        fb = max(fb, st.last_fallback_queries)
    st = eng.stats()
    step(0)
    torch.cuda.synchronize()
    res = tuple(t.cpu().numpy().copy() for t in out)
    return float(np.median(ms)), float(np.median(scan_ms)), st, fb, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dims", default="384,512,768,1024,1536,2048")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from fabstir_vectordb_b200 import Engine, _lib as L
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_dims.py needs a CUDA device")
    lib = L.load()
    result = {"card": card(), "workload": f"IVF search {N_ROWS} rows x D, nlist={NLIST} nprobe={NPROBE} "
              f"nq={NQ}/batch k={K}, synthetic (sigma {SIGMA}), {TRAIN_ITERS} training iterations",
              "timing": f"median of {args.steps} synchronous batches after {args.warmup} warm-up, CUDA events; "
              "index >> 126 MB L2, 4 rotating query sets", "hbm_peak_gbs": HBM_PEAK_GBS, "dims": []}
    for d in [int(v) for v in args.dims.split(",")]:
        eng = Engine(d, k_max=16)
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
        eng.set_option(L.OPT_KMEANS_TC, 1)
        buf = build(torch, lib, eng, d)
        qs = [queries(torch, lib, d, s) for s in range(N_QSETS)]
        out = [torch.empty((NQ, K), dtype=torch.int32, device="cuda"),
               torch.empty((NQ, K), dtype=torch.float32, device="cuda"),
               torch.empty((NQ,), dtype=torch.int32, device="cuda")]
        line = {"dim": d}
        for mode in ("tc", "exact"):
            eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC if mode == "tc" else L.SCAN_EXACT)
            ms, scan_ms, st, fb, res = time_mode(torch, eng, qs, out, args.steps, args.warmup)
            line[mode] = {"qps": NQ / (ms * 1e-3), "ms_per_batch": ms, "scan_ms": scan_ms,
                          "fallback_queries_max": fb, "launches": st.last_launches}
            if mode == "tc":
                alg = int(st.last_scanned_rows) * (d * 4 + 4)   # rows + |x|^2, each probed row once (as bench.py)
                line["tc"].update({"scanned_rows": int(st.last_scanned_rows), "algorithmic_bytes": alg,
                                   "scan_gbs": alg / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else None,
                                   "scan_share_of_hbm_peak": alg / (scan_ms * 1e-3) / 1e9 / HBM_PEAK_GBS
                                   if scan_ms > 0 else None})
            line[mode]["_res"] = res
        a, b = line["tc"].pop("_res"), line["exact"].pop("_res")
        same = (a[0] == b[0]).all(axis=1) & (a[1].view(np.uint32) == b[1].view(np.uint32)).all(axis=1) & (a[2] == b[2])
        line["identical_queries"] = int(same.sum())
        t_ids, t_cnt = truth(torch, lib, d, qs[0], buf)
        line["recall_at_10"] = recall(a[0].view(np.uint32), a[2].view(np.uint32), t_ids, t_cnt)
        line["tc_over_exact"] = line["tc"]["qps"] / line["exact"]["qps"]
        print(json.dumps(line), file=sys.stderr, flush=True)
        result["dims"].append(line)
        eng.close()
        del buf, qs, out
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
