"""Aggregate NLL + gradient evaluations per second of the batched evaluation (pigp_nll_grad_batch) against a loop of
single-theta calls (pigp_nll_grad), and multi-start Adam steps per second (pigp_adam_batch_host) against sequential
pigp_adam_host runs.  Sizes: C2 (N = 498), C3 (N = 1180) and C4 (N = 2640) with the reference generator's points
(tests/golden/ref_c*.npz, as tools/optimizer_rate.py), and stokes2d_scaling at N = 5018 and 10570.  Every call of a timed
loop is enqueued back to back on one stream; the window ends with a device synchronise and lasts at least 0.5 s.  A
separate pass records the per-class kernel time (pigp_profile_*) of one single call and of one 8-slot call.  The first
line names the card and its power limit, then one JSON object per size.

    python tools/batch_rate.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from stopro_b200 import _lib, synthetic

BATCHES = (1, 8, 32, 64)
STARTS = (8, 32)
ADAM_STEPS = 100
WINDOW_S = 0.5
WORKSPACE_CAP = 120e9  # bytes of batch workspace a measurement may ask for (the card has 180 GB)


def _cases():
    for name in ("ref_c2_poiseuille_additive", "ref_c3_sinusoidal", "ref_c4_drag3d"):
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        yield name[4:], synthetic.from_golden(path)
    for n in (5018, 10570):
        yield f"stokes2d_N{n}", dict(synthetic.stokes2d_scaling(n, n_test=8), eps=1e-6)


def _timed(call, sync):
    """Calls per second of `call` enqueued back to back (warmed up; window >= WINDOW_S, closed by a synchronise)."""
    for _ in range(3):
        call()
    sync()
    reps = 3
    while True:
        t0 = time.perf_counter()
        for _ in range(reps):
            call()
        sync()
        dt = time.perf_counter() - t0
        if dt >= WINDOW_S:
            return reps / dt
        reps = max(reps * 2, int(reps * 1.2 * WINDOW_S / max(dt, 1e-6)))


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit": q[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    a = ap.parse_args()
    lines = [_card()]
    print(json.dumps(lines[0]), flush=True)
    dev = torch.device("cuda:0")
    sync = torch.cuda.synchronize
    for name, cfg in _cases():
        gp = synthetic.make_model(cfg)
        gp.set_constants(cfg["r_train"], cfg["delta_y"], cfg["eps"], only_training=True)
        solver = gp._solver_for(cfg["r_train"])
        N, P = len(cfg["delta_y"]), solver.plan.theta_len
        npad = -(-N // 128) * 128
        per_slot = 8 * ((npad + 128) * npad + npad * 128 + 2 * npad * npad)
        rng = np.random.default_rng(0)
        bmax = max(BATCHES)
        th = torch.as_tensor(np.asarray(cfg["theta0"]) + 0.05 * rng.standard_normal((bmax, P)), device=dev)
        y = torch.as_tensor(np.asarray(cfg["delta_y"], dtype=np.float64), device=dev)
        out = torch.empty(bmax * (1 + P), dtype=torch.float64, device=dev)
        nll_p, grad_p = out.data_ptr(), out.data_ptr() + 8 * bmax
        stream = torch.cuda.current_stream().cuda_stream
        rec = {"workload": name, "N": N, "T": npad // 128}
        single = _timed(lambda: solver.nll_grad(th.data_ptr(), y.data_ptr(), cfg["eps"], nll_p, grad_p, None, stream), sync)
        rec["single_evals_per_s"] = single
        for nb in BATCHES:
            if nb * per_slot > WORKSPACE_CAP:
                rec[f"B{nb}_evals_per_s"] = None  # workspace over the cap: not measured
                continue
            rate = nb * _timed(lambda: solver.nll_grad_batch(nb, th.data_ptr(), y.data_ptr(), cfg["eps"], nll_p, grad_p, None,
                                                               stream), sync)
            rec[f"B{nb}_evals_per_s"] = rate
            rec[f"B{nb}_vs_single"] = rate / single
        # per-class kernel time of one single call and of one 8-slot call (separate pass: one event pair per launch)
        for label, call in (("single", lambda: solver.nll_grad(th.data_ptr(), y.data_ptr(), cfg["eps"], nll_p, grad_p, None, stream)),
                            ("B8", lambda: solver.nll_grad_batch(8, th.data_ptr(), y.data_ptr(), cfg["eps"], nll_p, grad_p, None,
                                                                 stream))):
            call()
            sync()
            _lib.profile_start()
            call()
            prof = _lib.profile_stop()
            rec[f"{label}_class_ms"] = {k: round(v["ms"], 4) for k, v in prof.items()}
        if npad <= 2688:
            kw = dict(max_iter=ADAM_STEPS, lr=1e-2, stop_eps=0.0, ntraining=float(N), check_every=16)
            for ns in STARTS:
                starts = [t for t in th[:ns].cpu().numpy()]
                solver.adam_batch_host(starts[:2], cfg["delta_y"], cfg["eps"], **dict(kw, max_iter=4))  # warm-up
                t0 = time.perf_counter()
                many = solver.adam_batch_host(starts, cfg["delta_y"], cfg["eps"], **kw)
                t_many = time.perf_counter() - t0
                t0 = time.perf_counter()
                seq = [solver.adam_host(s, cfg["delta_y"], cfg["eps"], **kw) for s in starts]
                t_seq = time.perf_counter() - t0
                steps_many, steps_seq = sum(len(m[2]) for m in many), sum(len(m[2]) for m in seq)
                rec[f"adam_{ns}_starts_steps_per_s"] = steps_many / t_many
                rec[f"adam_{ns}_sequential_steps_per_s"] = steps_seq / t_seq
                rec[f"adam_{ns}_speedup"] = (steps_many / t_many) / (steps_seq / t_seq)
        gp.close()
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for r in lines:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
