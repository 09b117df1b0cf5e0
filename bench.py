"""Headline benchmark: logp+grad evals/sec of the 8-shard federated logistic GLM.

Config (BASELINE.json): 8 shards x 10M rows x 256 features, bf16 design matrix, one theta per
evaluation; shards are spread over the N GPUs (8/N per GPU => strong scaling).  Synthetic data,
random parameters.  Rank 0 prints one JSON line; ``--dump-outputs DIR`` also writes what the last timed step
returned, one ``DIR/<name>.npy`` (float64) per array, so that two builds can be compared output for output.

    python bench.py                       # N=1, default steps
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 bench.py --gpus 8 --steps 50 --warmup 5
    python bench.py --impl reference ...  # the reference arm (see baseline/)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "logp+grad evals/sec for 8-shard federated GLM"   # the headline; the other configs: CONFIGS


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100,
                   help="timed evaluations; the default keeps the N = 1 headline region near 0.5 s, long enough to run "
                        "at the clocks the power cap sustains")
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference", "nccl"])
    p.add_argument("--rows", type=int, default=10_000_000, help="rows per shard")
    p.add_argument("--features", type=int, default=256)
    p.add_argument("--shards", type=int, default=8)
    p.add_argument("--kernel", default=os.environ.get("B200FED_GLM_KERNEL", "auto"), choices=["auto", "simt", "tc", "fp8"])
    p.add_argument("--chains", type=int, default=1)
    p.add_argument("--config", default="glm", choices=["glm", "fp8", "ode", "linreg"],
                   help="BASELINE.json configuration (glm = the headline; --kernel fp8 is an alias of --config fp8)")
    p.add_argument("--series", type=int, default=20_000, help="ode: time series per shard")
    p.add_argument("--timepoints", type=int, default=32, help="ode: observations per series")
    p.add_argument("--speculative-us", type=float, default=1000.0,
                   help="e2e region: FederatedEngine.set_speculative(wait_us) — the next evaluation's kernel is enqueued "
                        "before theta exists (0 = one launch per evaluation only)")
    p.add_argument("--nuts-draws", type=int, default=200, help="linreg: draws (= tune) of the NUTS run")
    p.add_argument("--out", default=None, help="also append the JSON line to this file")
    p.add_argument("--dump-outputs", default=None, metavar="DIR",
                   help="write the arrays the last timed step returned (logp, then one gradient per input) as DIR/<name>.npy")
    return p.parse_args()


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.

    NVML is polled from a thread every 5 ms (timed regions can be as short as tens of milliseconds
    at N = 8); falls back to an ``nvidia-smi -lms`` subprocess when pynvml is unavailable.
    """

    QUERY = (
        "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
        "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    )
    REASON_BITS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, gpu_index: int = 0):
        self.gpu_index = gpu_index
        self.lines = []
        self.proc = None
        self.samples = []       # (sm_mhz, max_mhz, power_w, reason_mask)
        self._stop = threading.Event()
        self._nvml = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.gpu_index]) if visible and visible.split(",")[0].isdigit() else self.gpu_index
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self._nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _poll(self):
        nv = self._nvml
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self._handle, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self._handle) / 1000.0
                self.samples.append((float(sm), float(mx), pw, int(get_reasons(self._handle))))
            except Exception:
                pass
            time.sleep(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self._nvml is not None:
            self._stop.set()
            self.thread.join(1.0)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no NVML samples"]}
            reasons = set()
            for _, _, _, mask in self.samples:
                for bit, name in self.REASON_BITS.items():
                    if mask & bit:
                        reasons.add(name)
            return {
                "sm_mhz": statistics.median(s[0] for s in self.samples),
                "sm_max_mhz": max(s[1] for s in self.samples),
                "power_w_max": max(s[2] for s in self.samples),
                "samples": len(self.samples),
                "reasons": sorted(reasons),
                "source": "nvml",
            }
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
            "source": "nvidia-smi",
        }


CONFIGS = {
    # name: (metric, model description)
    "glm": ("logp+grad evals/sec for 8-shard federated GLM", "federated logistic GLM (logp + gradient)"),
    "fp8": ("logp+grad evals/sec for hierarchical GLM, fp8 block-scaled design matrix",
            "hierarchical logistic GLM, one group intercept per shard (logp + gradient)"),
    "ode": ("logp+grad evals/sec for federated ODE parameter estimation",
            "Lotka-Volterra ODE, RK4 x8 with forward sensitivities, Gaussian likelihood (logp + gradient)"),
    "linreg": ("logp+grad evals/sec for federated Bayesian linear regression",
               "the reference's demo model (demo_node.py): Gaussian linear regression, 10 rows per shard"),
}


def build_workload(args, world, rank, dev):
    """This rank's shard model of the chosen BASELINE.json configuration, a theta sampler and descriptive keys."""
    import numpy as np
    import torch

    from pytensor_federated_b200.models import (
        Fp8GlmShards, GlmShards, LinregShards, OdeShards, make_demo_data, synth_logistic_shard,
        synth_logistic_shard_fp8, synth_lv_shard,
    )

    rng = np.random.default_rng(7)
    K = args.chains
    my_shards = [s for s in range(args.shards) if s % world == rank]
    if args.config in ("glm", "fp8"):
        P = args.features
        Xs, ys, scs = [], [], []
        for s in my_shards:
            if args.config == "fp8":
                X, sc, y = synth_logistic_shard_fp8(args.rows, P, seed=1000 + s, device=dev)
                scs.append(sc)
            else:
                X, y, _ = synth_logistic_shard(args.rows, P, seed=1000 + s, device=dev)
            Xs.append(X)
            ys.append(y)
        torch.cuda.synchronize()
        if args.config == "fp8":  # hierarchical config: one partial-pooling group (intercept) per shard
            n_groups = args.shards
            model = Fp8GlmShards(Xs, scs, ys, groups=my_shards, n_groups=n_groups, n_chains=K)
        else:
            n_groups = 1
            model = GlmShards(Xs, ys, n_groups=1, family="logistic", n_chains=K, kernel=args.kernel)

        def draw_theta():
            ic = rng.normal(size=(K, n_groups) if K > 1 else (n_groups,)).astype(np.float32) * 0.1
            beta = rng.normal(size=(K, P) if K > 1 else (P,)).astype(np.float32) * 0.02
            return ic, beta

        keys = {"rows_per_shard": args.rows, "features": P, "global_batch": args.shards * args.rows, "seq_len": P,
                "l2_policy": "inputs (>= 2.5 GB per GPU) are larger than the 126 MB L2; no flush needed"}
    elif args.config == "ode":
        shards = [synth_lv_shard(args.series, args.timepoints, seed=s, device=dev) for s in my_shards]
        model = OdeShards([s[0] for s in shards], [s[1] for s in shards], [s[2] for s in shards], [s[3] for s in shards])

        def draw_theta():
            return (np.array([1.0, 0.4, 0.8, 0.2]) + 0.01 * rng.normal(size=4),)

        keys = {"series_per_shard": args.series, "timepoints": args.timepoints, "global_batch": args.shards * args.series,
                "seq_len": args.timepoints,
                "l2_policy": "compute-bound (RK4 + sensitivities in registers); inputs fit in L2 and are re-read every "
                             "evaluation by design, theta changes every step"}
    else:  # linreg
        xs, ys_, sg = [], [], []
        for s in my_shards:
            x, y, sigma = make_demo_data(seed=123 + s)
            xs.append(x)
            ys_.append(y)
            sg.append(sigma)
        model = LinregShards(xs, ys_, sg, local_ids=my_shards, n_shards_total=args.shards, device=dev)

        def draw_theta():
            return rng.normal(size=args.shards), np.asarray(rng.normal())

        keys = {"rows_per_shard": 10, "global_batch": args.shards * 10, "seq_len": 1,
                "l2_policy": "latency-bound: 10 rows per shard; theta changes every step"}
    return model, draw_theta, keys


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from pytensor_federated_b200.parallel import FederatedEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    own_pg = world > 1 and not dist.is_initialized()   # benchmarks/run_configs.py runs several configs in one group
    if own_pg:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    if args.kernel == "fp8":
        args.config = "fp8"
    model, draw_theta, cfg_keys = build_workload(args, world, rank, dev)
    backend = "fused" if args.impl == "b200" else "collective"
    eng = FederatedEngine(model, backend=backend, timeout=120.0)
    W, S, K = args.warmup, args.steps, args.chains
    n_verify = 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def share(n: int) -> int:
        """The root decides how many evaluations a phase has; the peers serve exactly that many."""
        if world == 1:
            return n
        t = torch.tensor([n], device=dev, dtype=torch.int64)
        dist.broadcast(t, src=0)
        return int(t.item())

    def oracle_sum(inputs):
        """fp64 oracle of the same evaluation: every rank evaluates ITS shards with stock PyTorch, NCCL sums."""
        import inspect

        kw = {"dtype": torch.float64} if "dtype" in inspect.signature(model.reference_partial).parameters else {}
        part = torch.from_numpy(np.asarray(model.reference_partial(inputs, **kw), dtype=np.float64)).to(dev)
        if world > 1:
            dist.all_reduce(part, op=dist.ReduceOp.SUM)
        return part.cpu().numpy()

    # ---- every rank draws the same thetas (same seed) so the peers can evaluate the oracle too -------------
    verify_thetas = [draw_theta() for _ in range(n_verify)]
    result = {}
    if rank == 0:
        # ---- correctness first: fused result vs the fp64 oracle on the same shards, at this N -------------
        got = [np.array(eng.evaluate_raw(th)) for th in verify_thetas]
        barrier()
        max_rel = 0.0
        for th, g in zip(verify_thetas, got):
            want = oracle_sum(th)
            v = np.asarray(want).reshape(K, -1) if args.config in ("glm", "fp8") else np.asarray(want).reshape(1, -1)
            gg = g.reshape(v.shape)
            # logp: relative; gradient block: relative to its largest entry (entries near zero carry no signal)
            if args.config == "linreg":
                scale = np.maximum(np.abs(v), 1e-9)
                err = float(np.max(np.abs(gg - v) / np.maximum(scale, np.abs(v).max() * 1e-6)))
            else:
                e_lp = np.abs(gg[:, 0] - v[:, 0]) / np.maximum(np.abs(v[:, 0]), 1e-30)
                e_gr = np.abs(gg[:, 1:] - v[:, 1:]).max(axis=1) / np.maximum(np.abs(v[:, 1:]).max(axis=1), 1e-30)
                err = float(max(e_lp.max(), e_gr.max()))
            max_rel = max(max_rel, err)
        tol = {"glm": 2e-4, "fp8": 3e-3, "ode": 2e-3, "linreg": 1e-9}[args.config]
        if backend == "collective" and args.config in ("glm", "fp8"):
            tol = 5e-3   # the NCCL baseline's eager compute rounds theta and the residuals to bf16 for its two GEMMs
        verified = bool(max_rel <= tol)
        if not verified:
            print(json.dumps({"error": "verification failed", "max_rel_err": max_rel, "tolerance": tol, "n_gpus": world}),
                  flush=True)
        thetas = [draw_theta() for _ in range(W + S)]
        # ---- warm-up through the public API -------------------------------------------------------------------
        share(W)
        for i in range(W):
            eng.evaluate(*thetas[i])
        barrier()
        share(S)
        sampler = ClockSampler(local_rank).start()
        # ---- device-timed region: S back-to-back fused evaluations ---------------------------------------------
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if backend == "fused":
            stream = eng.torch_stream()
            eng.set_device_theta(thetas[W], enable=True)
            launches0 = eng.kernel_launches
            start.record(stream)
            last = 0
            for _ in range(S):
                last = eng.launch()
            end.record(stream)
            last_vals, last_theta = np.array(eng.wait(last), dtype=np.float64), thetas[W]
            end.synchronize()
            launches = eng.kernel_launches - launches0
            eng.set_device_theta(thetas[W], enable=False)
        else:
            start.record()
            for i in range(S):
                last_vals, last_theta = eng.evaluate_raw(thetas[W + i]), thetas[W + i]
            end.record()
            end.synchronize()
            launches = 0
        timed_ms = start.elapsed_time(end)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, model.unpack_result(last_vals, model.call_context(last_theta)))
        barrier()
        # ---- end-to-end region: public API, pinned H2D of theta + D2H of the result each step -----------------
        e2e_steps = share(S)

        evaluated = [0]   # evaluations of the current phase (the peers serve exactly as many as the root announced)

        def e2e_region():
            t0 = time.perf_counter()
            acc = 0.0
            for i in range(e2e_steps):
                out = eng.evaluate(*thetas[W + i % S])
                evaluated[0] += 1
                if i < S:
                    acc += float(np.sum(out[0]))
            return time.perf_counter() - t0, acc   # evaluate() returned: the result has been read back

        e2e_plain_s, checksum = e2e_region()
        e2e_s = e2e_plain_s
        torch.cuda.synchronize()
        barrier()
        try:
            spec_on = bool(backend == "fused" and args.speculative_us > 0 and eng.set_speculative(args.speculative_us))
        except Exception as ex:
            print(f"[bench] speculative launches unavailable ({ex})", file=sys.stderr, flush=True)
            spec_on = False
        share(3 + e2e_steps if spec_on else 0)
        if spec_on:
            # same loop, same public call; the engine keeps the next evaluation's kernel enqueued ahead of theta
            evaluated[0] = 0
            e2e_spec_s = None
            try:
                for i in range(3):
                    eng.evaluate(*thetas[W + i % S])
                    evaluated[0] += 1
                e2e_spec_s, spec_sum = e2e_region()
                eng.set_speculative(0.0)
            except Exception as ex:   # the optional mode must never cost the run its line: finish the phase plainly
                print(f"[bench] speculative end-to-end region failed ({type(ex).__name__}: {ex}); "
                      "keeping the one-launch-per-evaluation number", file=sys.stderr, flush=True)
                e2e_spec_s = None
                eng.set_speculative(0.0)
                while evaluated[0] < 3 + e2e_steps:
                    eng.evaluate(*thetas[W])
                    evaluated[0] += 1
            if e2e_spec_s is not None and spec_sum != checksum:
                raise SystemExit(f"speculative launches changed the result: {spec_sum!r} vs {checksum!r}")
            torch.cuda.synchronize()
            barrier()
            # both settings go through the same public call; the headline is the engine's better mode, and the
            # JSON line names it and carries the other number too
            if e2e_spec_s is not None and e2e_spec_s < e2e_plain_s:
                e2e_s = e2e_spec_s
            else:
                spec_on = False
        clocks = sampler.stop()
        result = dict(timed_ms=timed_ms, e2e_s=e2e_s, e2e_steps=e2e_steps, launches=launches, checksum=checksum,
                      clocks=clocks, verified=verified, max_rel_err=max_rel, e2e_plain_s=e2e_plain_s,
                      e2e_speculative=spec_on, e2e_spec_s=locals().get("e2e_spec_s"))
    else:
        # peers: each phase serves exactly as many epochs as the root evaluates; their kernels wait on the
        # device for the root's theta, the host only keeps the queue filled
        eng.serve(max_epochs=n_verify)
        barrier()
        for th in verify_thetas:
            oracle_sum(th)
        eng.serve(max_epochs=share(0))
        barrier()
        eng.serve(max_epochs=share(0))
        barrier()
        eng.serve(max_epochs=share(0))
        barrier()
        n_spec = share(0)          # the root repeats the end-to-end region with speculative launches
        if n_spec:
            eng.serve(max_epochs=n_spec)
            barrier()
        if args.config == "linreg" and backend == "fused":
            eng.serve()   # the NUTS run of the root: as many evaluations as the sampler asks for, until it shuts down

    # max over ranks of the device-timed region (the root's kernels cannot finish before every peer delivered
    # its partial, so the root time already dominates; reduce anyway)
    comm_mode = eng.comm_mode
    bytes_per_eval = model.bytes_per_eval()
    flops_per_eval = model.flops_per_eval()
    n_theta_words, n_vals = model.n_theta_words, model.n_vals
    extra = {}
    if rank == 0 and args.config == "linreg" and backend == "fused":
        extra = linreg_nuts(eng, args)   # NUTS driving FederatedLogpGradOp over the live federation
    eng.shutdown()
    if world > 1:
        dist.barrier()
        if own_pg:
            dist.destroy_process_group()
    if rank != 0:
        return

    ms_per_step = result["timed_ms"] / S
    value = 1000.0 / ms_per_step * K
    e2e_value = result["e2e_steps"] / result["e2e_s"] * K
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    metric, model_name = CONFIGS[args.config]
    config = {
        "model": model_name,
        "shards": args.shards,
        "chains_per_eval": K,
        **cfg_keys,
        "parallelism": f"shard-parallel x{world} ({args.shards // world} shards/GPU)",
        "kernel": args.kernel if args.config == "glm" else args.config,
        "backend": backend,
        "comm": comm_mode,
        "timed_seconds": result["timed_ms"] / 1e3,
        "hbm_bytes_per_eval_per_gpu": bytes_per_eval,
    }
    if bytes_per_eval:
        config["hbm_roofline_frac_of_measured"] = (bytes_per_eval / (ms_per_step * 1e-3)) / (hbm * 1e9)
    if args.config in ("glm", "fp8"):
        # three-term roofline of the fused broadcast->compute->reduce kernel (seconds per eval per GPU):
        # HBM stream of the shard, tensor-core time of the two skinny GEMMs (N padded to 16 columns each),
        # NVLink bytes (theta in, partial out) at the measured 770 GB/s peer bandwidth
        config["roofline_s"] = {
            "hbm": bytes_per_eval / (hbm * 1e9),
            "tensor": flops_per_eval * (32.0 / max(1, 4 * K)) / (peaks.get("bf16_tflops", 1590.0) * 1e12),
            "nvlink": (n_theta_words * 4 + n_vals * 8) / 770e9,
            "bound": "hbm",
        }
    line = {
        "metric": metric,
        "value": value,
        "unit": "evals/s",
        "n_gpus": world,
        "steps": S,
        "warmup": W,
        "ms_per_step": ms_per_step,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": {"glm": "bf16", "fp8": "fp8-e4m3 block-scaled (32x32 UE8M0)", "ode": "fp32", "linreg": "fp64"}[args.config],
        "data": "synthetic",
        "impl": args.impl,
        "config": config,
        "verified": result["verified"],
        "max_rel_err": result["max_rel_err"],
        "clocks": result["clocks"],
        "e2e": {
            "value": e2e_value,
            "unit": "evals/s",
            "steps": result["e2e_steps"],
            # speculative launches read theta as tagged 8-byte words
            "h2d_bytes_per_step": n_theta_words * (8 if result.get("e2e_speculative") else 4),
            "d2h_bytes_per_step": n_vals * 8 + 8,
            "speculative_us": args.speculative_us if result.get("e2e_speculative") else 0.0,
            "value_one_launch_per_eval": result["e2e_steps"] / result["e2e_plain_s"] * K if result.get("e2e_plain_s") else None,
            "value_speculative": result["e2e_steps"] / result["e2e_spec_s"] * K if result.get("e2e_spec_s") else None,
        },
        "gpu_launches": int(result["launches"]) * world if backend == "fused" else 0,
        "checksum": result["checksum"],
        **extra,
    }
    out = json.dumps(line)
    print(out, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write(out + "\n")
    if not result["verified"]:
        raise SystemExit(3)
    return line


def dump_outputs(out_dir, arrays):
    """``logp.npy``, ``grad_0.npy``, ... (float64): what a caller of the evaluation receives."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    names = ["logp"] + [f"grad_{i}" for i in range(len(arrays) - 1)]
    for name, a in zip(names, arrays):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def linreg_nuts(eng, args):
    """BASELINE.json config 2: the sampler drives one federated Op per node; all of them are answered by ONE
    fused launch per model evaluation (the peers serve without bound until the root shuts down)."""
    import numpy as np

    from pytensor_federated_b200.federation import NodeFederation
    from pytensor_federated_b200.sampling import Model, nuts_sample

    fed = NodeFederation(eng)
    ops = fed.node_ops()
    m = Model()
    mu = m.Normal("intercept_mu", 0.0, 1.0)
    icpt = m.Normal("intercept", mu, 0.1, size=args.shards)
    slope = m.Normal("slope", 0.0, 1.0)
    for i, off in enumerate(np.linspace(-4, 4, args.shards)):
        logp, *_ = ops[i](icpt[i] + off, slope)
        m.Potential(f"p{i}", logp)
    m.compile()
    spec = False
    try:
        spec = bool(args.speculative_us > 0 and eng.set_speculative(args.speculative_us))
    except Exception as ex:
        print(f"[bench] speculative launches unavailable ({ex})", file=sys.stderr, flush=True)
    t0 = time.perf_counter()
    res = nuts_sample(m.logp_dlogp, np.zeros(m.dim), draws=args.nuts_draws, tune=args.nuts_draws, seed=1)
    dt = time.perf_counter() - t0
    # the same posterior with the WHOLE federation behind one Op (`NodeFederation.all_nodes_op`): the graph no longer
    # grows with the number of nodes
    from pytensor_federated_b200.graph import core as at

    m1 = Model()
    mu1 = m1.Normal("intercept_mu", 0.0, 1.0)
    icpt1 = m1.Normal("intercept", mu1, 0.1, size=args.shards)
    slope1 = m1.Normal("slope", 0.0, 1.0)
    logp1, *_ = fed.all_nodes_op()(icpt1 + at.as_tensor(np.linspace(-4, 4, args.shards)), slope1)
    m1.Potential("all", logp1)
    m1.compile()
    launches0 = fed.n_launches
    t1 = time.perf_counter()
    res1 = nuts_sample(m1.logp_dlogp, np.zeros(m1.dim), draws=args.nuts_draws, tune=args.nuts_draws, seed=1)
    dt1 = time.perf_counter() - t1
    one_op = {"seconds": dt1, "n_logp_evals": res1.n_logp_evals, "model_evals_per_s": res1.n_logp_evals / dt1,
              "node_evals_per_s": args.shards * res1.n_logp_evals / dt1, "fused_launches": fed.n_launches - launches0,
              "divergences": int(res1.divergences),
              # (the two graphs add the node terms in different orders, so the chains part ways after a few
              # hundred steps; what has to agree is the posterior)
              "posterior_mean_max_abs_diff_vs_per_node_ops": float(np.max(np.abs(res1.samples.mean(0) - res.samples.mean(0)))),
              "posterior_sd_max": float(np.max(res.samples.std(0)))}
    if spec:
        eng.set_speculative(0.0)
    return {"nuts": {"draws": args.nuts_draws, "tune": args.nuts_draws, "seconds": dt, "n_logp_evals": res.n_logp_evals,
                     "speculative_us": args.speculative_us if spec else 0.0, "one_op_for_the_federation": one_op,
                     "model_evals_per_s": res.n_logp_evals / dt, "node_evals_per_s": args.shards * res.n_logp_evals / dt,
                     "fused_launches": launches0, "divergences": int(res.divergences)}}


def run_reference(args):
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import reference_arm
    except Exception as ex:  # noqa: BLE001
        print(json.dumps({"impl": "reference", "unavailable": f"reference arm not importable: {ex}"}))
        return
    reference_arm.main(args)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
