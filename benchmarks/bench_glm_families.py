"""Throughput of the tensor-core GLM kernel per family, with and without fitted family parameters.

    python benchmarks/bench_glm_families.py                      # 8 shards x 10M rows x 256 features, bf16, 1 GPU

The headline shape of ``bench.py`` (one GPU) for logistic / normal / student_t / negative_binomial at K = 1 and
K = 16 chains per launch.  Each case is first checked against the fp64 oracle (``GlmShards.reference_partial``),
then timed with device events around back-to-back ``launch()`` calls with theta parked in device memory, exactly
like ``bench.py``'s device-timed region; the window is at least ``--min-seconds`` long.  One JSON line per case,
with the GPU's name and power limit read in the same run.  Needs a CUDA device: without one it fails.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# data-generating and evaluation parameters (sigma / (sigma, nu) / alpha); intercept 0.3 as in the logistic headline
PHI = {"logistic": (), "normal": (0.7,), "student_t": (1.3, 4.0), "negative_binomial": (2.0,)}


def gpu_info(index: int) -> dict:
    import torch

    info = {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        limit, smax = [v.strip() for v in out.strip().splitlines()[0].split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(limit), float(smax)
    except Exception as ex:  # noqa: BLE001 - reported, not fatal
        info["power_limit_w"] = f"unavailable ({ex})"
    return info


def draw_inputs(family: str, K: int, P: int, rng):
    ic = 0.3 + rng.normal(size=(K, 1)) * 0.05
    beta = (rng.normal(size=(K, P)) * 0.03).astype(np.float32)
    inputs = [ic, beta]
    if PHI[family]:
        inputs.append((np.asarray(PHI[family])[None, :] * np.exp(rng.normal(size=(K, len(PHI[family]))) * 0.1)).astype(np.float32))
    if K == 1:
        inputs = [v[0] for v in inputs]
    return inputs


def max_rel_err(got: np.ndarray, want: np.ndarray, K: int) -> float:
    g, w = got.reshape(K, -1), want.reshape(K, -1)
    e_lp = np.abs(g[:, 0] - w[:, 0]) / np.maximum(np.abs(w[:, 0]), 1e-30)
    # gradient entries relative to the largest of the chain (entries near zero carry no signal)
    e_gr = np.abs(g[:, 1:] - w[:, 1:]).max(axis=1) / np.maximum(np.abs(w[:, 1:]).max(axis=1), 1e-30)
    return float(max(e_lp.max(), e_gr.max()))


def main():
    import torch

    from pytensor_federated_b200.models import GlmShards, synth_glm_shard
    from pytensor_federated_b200.parallel import FederatedEngine

    ap = argparse.ArgumentParser()
    ap.add_argument("--shards", type=int, default=8)
    ap.add_argument("--rows", type=int, default=10_000_000, help="rows per shard")
    ap.add_argument("--features", type=int, default=256)
    ap.add_argument("--families", nargs="+", default=list(PHI))
    ap.add_argument("--chains", type=int, nargs="+", default=[1, 16])
    ap.add_argument("--min-seconds", type=float, default=0.5)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_glm_families.py measures the GPU kernel and needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    P = args.features
    for family in args.families:
        Xs, ys = [], []
        for s in range(args.shards):
            X, y, _ = synth_glm_shard(args.rows, P, family=family, phi=PHI[family], seed=1000 + s, device=dev)
            Xs.append(X)
            ys.append(y)
        for K in args.chains:
            model = GlmShards(Xs, ys, family=family, n_chains=K, kernel="tc")
            rng = np.random.default_rng(K)
            with FederatedEngine(model) as eng:
                assert model.selected_kernel == "tc"
                # ---- correctness first: the fused result vs the fp64 oracle -------------------------------------
                verify = draw_inputs(family, K, P, rng)
                got = np.array(eng.evaluate_raw(verify))
                err = max_rel_err(got, model.reference_partial(verify, dtype=torch.float64), K)
                torch.cuda.empty_cache()
                # ---- device-timed region: back-to-back launches, theta in device memory -------------------------
                stream = eng.torch_stream()
                eng.set_device_theta(draw_inputs(family, K, P, rng), enable=True)
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record(stream)
                last = 0
                for _ in range(args.warmup):
                    last = eng.launch()
                end.record(stream)
                eng.wait(last)
                end.synchronize()
                n = max(args.warmup, math.ceil(args.min_seconds * 1e3 / max(start.elapsed_time(end) / args.warmup, 1e-3)))
                launches0 = eng.kernel_launches
                start.record(stream)
                for _ in range(n):
                    last = eng.launch()
                end.record(stream)
                eng.wait(last)
                end.synchronize()
                ms = start.elapsed_time(end)
                launches = eng.kernel_launches - launches0
                eng.set_device_theta(draw_inputs(family, K, P, rng), enable=False)
            per_eval = ms / n
            rows = args.shards * args.rows
            print(json.dumps({
                "bench": "glm_families", "family": family, "chains": K, "n_family_params": len(PHI[family]),
                "shards": args.shards, "rows_per_shard": args.rows, "features": P, "dtype": "bf16", "n_gpus": 1,
                "verified": bool(err <= 2e-4), "max_rel_err": err, "evals": n, "launches": launches,
                "timed_s": ms / 1e3, "eval_ms": per_eval, "rows_per_s": rows / (per_eval / 1e3),
                "chain_evals_per_s": K / (per_eval / 1e3), "hbm_gb_s": model.bytes_per_eval() / (per_eval / 1e3) / 1e9,
                **info,
            }), flush=True)
        del Xs, ys, model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
