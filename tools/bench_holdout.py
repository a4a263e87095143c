"""Cost of choosing K by held-out likelihood on one GPU; prints ONE JSON line.

    python tools/bench_holdout.py [--steps 20] [--warmup 5] [--repeats 5]

  masked_ms_per_step     the masked step (bigclam_set_holdout: every node on the general path) on the training graph
                         of a 20 % split (seed 0) of com-amazon, K = 200, synthetic F0 as in BASELINE.md (density 0.05,
                         seed 1234): step-kernel time per step of the device loop (bigclam_run, CUDA events around every
                         step kernel, BIGCLAM_F_TIME_KERNELS), median over the repeats
  unmasked_ms_per_step   the same, shipped default routing (tiles, split hubs, bounds), same training graph and F0
  holdout_llh_ms         bigclam_holdout_loglikelihood (per-node kernel + fixed-order sum + the 8-byte copy back), CUDA
                         events, median over 20 calls after 3 warm-up calls
  select_K_s             wall time of BigClam.select_K(Ks=[20, 50, 100], repeats=2) on Email-Enron (simple graph)

Every repeat starts both contexts from F0 and runs the warm-up steps untimed; the masked and unmasked runs alternate.
Nothing is written to the tree."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:                       # (the number is still reported; say why the card is unknown)
        return {"name": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--no-select", action="store_true", help="skip the select_K wall time")
    args = ap.parse_args()
    import numpy as np
    import torch
    from bigclam_apachespark_b200 import BigClam, graphs as G
    from bigclam_apachespark_b200.holdout import split_pairs

    if not torch.cuda.is_available():
        raise SystemExit("bench_holdout.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    rp0, col0, _ = G.load_npz_graph("com-amazon")
    n, K = len(rp0) - 1, 200
    s = split_pairs(rp0, col0, 0.2, 0)
    F0 = G.synthetic_F0(n, K, seed=1234, density=0.05)
    stream = torch.cuda.current_stream()
    ctx = {}
    for name in ("masked", "unmasked"):
        b = BigClam(device=0, time_kernels=True, sparse_rows=True)
        b.set_graph(s.rowptr, s.col).set_K(K)
        b.set_stream(stream.cuda_stream)
        if name == "masked":
            b.set_holdout(s.ho_rowptr, s.ho_col, s.ho_is_edge)
        ctx[name] = b
    ms = {"masked": [], "unmasked": []}
    llh_end = {}
    for _ in range(args.repeats):
        for name, b in ctx.items():
            b.set_F(F0)                                  # (the held-out lists stay with the context)
            b._run(4, 0.0, args.warmup)
            if name == "unmasked":                       # let the tile cut settle, as bench.py does
                for _ in range(3):
                    b.retile()
                    b._run(4, 0.0, 2)
            torch.cuda.synchronize()
            b._run(4, 0.0, args.steps)
            kern_ms, nk, _ = b.kernel_time()
            assert b.last_calls == args.steps and nk == args.steps
            ms[name].append(kern_ms / nk)
            llh_end[name] = float(b.last_trace[-1])
    bm = ctx["masked"]
    for _ in range(3):
        bm.holdout_loglikelihood()
    ho_ms = []
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        L_ho = bm.holdout_loglikelihood()
        e1.record(stream)
        torch.cuda.synchronize()
        ho_ms.append(e0.elapsed_time(e1))
    n_pairs = bm.last_holdout_pairs
    for b in ctx.values():
        b.close()

    sel = None
    if not args.no_select:
        rpe, cole, _ = G.load_npz_graph("email-enron")
        b = BigClam(device=0)
        b.set_graph(rpe, cole)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        K_best, rows = b.select_K(Ks=[20, 50, 100], repeats=2, seed=0)
        torch.cuda.synchronize()
        sel = {"s": time.perf_counter() - t0, "K_best": K_best,
               "rows": [{"K": r[0], "mean": r[1], "values": r[2], "calls": r[3]} for r in rows]}
        b.close()

    med = {k: float(np.median(v)) for k, v in ms.items()}
    print(json.dumps({
        "workload": "com-amazon K=200, synthetic F0 (density 0.05, seed 1234), 20 % held out (seed 0)",
        "n": n, "train_nnz_directed": int(len(s.col)), "holdout_pairs": int(n_pairs),
        "steps": args.steps, "warmup": args.warmup, "repeats": args.repeats,
        "masked_ms_per_step": med["masked"], "unmasked_ms_per_step": med["unmasked"],
        "masked_over_unmasked": med["masked"] / med["unmasked"],
        "masked_ms_all": ms["masked"], "unmasked_ms_all": ms["unmasked"],
        "llh_end": llh_end, "holdout_llh": L_ho,
        "holdout_llh_ms": float(np.median(ho_ms)), "holdout_llh_ms_min": float(np.min(ho_ms)),
        "select_K_enron": sel, "select_K_s": None if sel is None else sel["s"],
        "gpu": gpu_info(),
    }))


if __name__ == "__main__":
    main()
