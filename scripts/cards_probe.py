"""Cost of whole-card requests on one GPU; prints one JSON object.

Snapshot: cfg3-style 1 M-row batches scored on a table of full cards (100, 183359) at D = 8 and
D = 64, as pipelined device launches (EGPU_F_INPUTS_READY) on one stream.  A ring of 32 batches
(256 MB of requests, twice the L2) so every launch reads its inputs from HBM.  Per D: the existing
egpu_bestfit_batch_dev on the single-card rows, then egpu_bestfit_cards_dev without and with card
masks with 0 %, 1 % and 10 % of the rows turned into whole-card requests of 2..4 cards.
us_per_step = CUDA-event time of a CUDA graph of `steps` launches / steps, median of 5 replays.

Replay: cfg5 churn (100 000 events, D = 8) through egpu_replay, and with 5 % of its ALLOCs turned
into whole-card requests (mem 0) through egpu_replay_cards; next to the C oracle of each.

    python scripts/cards_probe.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import elastic_gpu_agent_b200 as e  # noqa: E402
from oracle import cards_c, oracle_c  # noqa: E402

R, NB, STEPS, WARM, WINDOWS = 1_000_000, 32, 256, 64, 5


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def whole_rows(c, share, rng):
    c = c.copy()
    pick = rng.random(c.size) < share
    c[pick] = 100 * rng.integers(2, 5, int(pick.sum()))
    return c


def time_launches(launch):
    """the `steps` launches captured once in a CUDA graph (no host launch cost in the window), replayed"""
    st = torch.cuda.current_stream()
    for k in range(WARM):
        launch(k)
    st.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        for k in range(STEPS):
            launch(k)
    g.replay()
    torch.cuda.synchronize()
    res = []
    for _ in range(WINDOWS):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(st)
        g.replay()
        t1.record(st)
        t1.synchronize()
        res.append(t0.elapsed_time(t1) * 1000.0 / STEPS)
    return float(np.median(res)), [round(x, 4) for x in res]


def snapshot_part(a, D):
    dev = torch.device("cuda", 0)
    fc, fm = np.full(D, 100, np.int32), np.full(D, 183_359, np.int32)
    a.set_table(fc, fm)
    st = torch.cuda.current_stream()
    sh = st.cuda_stream
    rng = np.random.default_rng(D)
    base = [e.synth.requests(3, 6, R, b * R) for b in range(NB)]
    outs = [(torch.empty(R, dtype=torch.int32, device=dev), torch.empty(R, dtype=torch.int64, device=dev),
             torch.zeros(2 * D, dtype=torch.int64, device=dev), torch.zeros(3 * D, dtype=torch.int32, device=dev)) for _ in range(NB)]
    res = {}

    def ring(share):
        return [(torch.from_numpy(whole_rows(c, share, rng)).to(dev), torch.from_numpy(m).to(dev)) for c, m in base]

    inp = ring(0.0)

    def batch(k):
        (c, m), (i, _, dl, to) = inp[k % NB], outs[k % NB]
        a.bestfit_dev(c.data_ptr(), m.data_ptr(), R, i.data_ptr(), dl.data_ptr(), to.data_ptr(), stream=sh, inputs_ready=True)
    res["bestfit_batch_dev"] = time_launches(batch)
    for share in (0.0, 0.01, 0.10):
        inp = ring(share)
        for masks in (False, True):
            def cards(k, masks=masks):
                (c, m), (i, cm, dl, to) = inp[k % NB], outs[k % NB]
                a.bestfit_cards_dev(c.data_ptr(), m.data_ptr(), R, i.data_ptr(), cm.data_ptr() if masks else 0, dl.data_ptr(),
                                    to.data_ptr(), stream=sh, inputs_ready=True)
            res[f"bestfit_cards_dev{'_masks' if masks else ''}_{int(share * 100)}pct"] = time_launches(cards)
        # one output checked against the oracle, so the timed path is known to compute the right thing
        c, m = inp[0]
        o = outs[0]
        a.bestfit_cards_dev(c.data_ptr(), m.data_ptr(), R, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), stream=sh)
        torch.cuda.synchronize()
        ei, ec_, edc, edm, _ = cards_c.bestfit_cards_snapshot(fc, fm, c.cpu().numpy(), m.cpu().numpy())
        assert np.array_equal(o[0].cpu().numpy(), ei) and np.array_equal(o[1].cpu().numpy().view(np.uint64), ec_)
        assert np.array_equal(o[2].cpu().numpy(), np.concatenate([edc, edm]))
    return {k: {"us_per_step": round(v[0], 4), "windows": v[1]} for k, v in res.items()}


def replay_part(a):
    w = e.synth.workload("cfg5")
    kind, ea, eb = e.synth.churn_events(w["seed"], w["R"])
    rng = np.random.default_rng(5)
    whole = (kind == 0) & (rng.random(kind.size) < 0.05)
    ca, cb = ea.copy(), eb.copy()
    ca[whole] = 100 * rng.integers(2, 5, int(whole.sum()))
    cb[whole] = 0
    out = {"events": int(kind.size), "whole_card_allocs": int(whole.sum())}

    def gpu(fn, ka, kb):
        best = None
        for _ in range(3):
            a.set_table(w["free_core"], w["free_mem"])
            t = time.perf_counter()
            r = fn(kind, ka, kb)
            dt = time.perf_counter() - t
            best = dt if best is None else min(best, dt)
        return r, best * 1e9 / kind.size

    def cpu(fn, ka, kb):
        t = time.perf_counter()
        r = fn(w["free_core"], w["free_mem"], kind, ka, kb)
        return r, (time.perf_counter() - t) * 1e9 / kind.size

    r, ns = gpu(a.replay, ea, eb)
    o, ons = cpu(oracle_c.replay, ea, eb)
    assert np.array_equal(r, o[0])
    out["egpu_replay_ns_per_event"] = round(ns, 2)
    out["oracle_replay_ns_per_event"] = round(ons, 2)
    (r, cards), ns = gpu(a.replay_cards, ca, cb)
    o, ons = cpu(cards_c.replay_cards, ca, cb)
    assert np.array_equal(r, o[0]) and np.array_equal(cards, o[1])
    out["egpu_replay_cards_ns_per_event"] = round(ns, 2)
    out["oracle_replay_cards_ns_per_event"] = round(ons, 2)
    out["note"] = "host wall time of one synchronous call (copies in and out included), best of 3"
    return out


def main():
    a = e.BestFitAllocator(0)
    torch.cuda.set_stream(torch.cuda.Stream())  # graphs are captured on a stream of their own
    result = {"gpu": gpu_info(), "rows_per_batch": R, "ring_batches": NB, "steps_per_window": STEPS,
              "snapshot": {f"D{D}": snapshot_part(a, D) for D in (8, 64)}, "replay_cfg5": replay_part(a)}
    result["gpu_after"] = gpu_info()
    a.close()
    s = json.dumps(result, indent=1)
    print(s)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        open(sys.argv[1], "w").write(s + "\n")


if __name__ == "__main__":
    main()
