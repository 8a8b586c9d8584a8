#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its config: 1024px images/sec, BitDance-14B-64x (random-init, synthetic prompt).

One "step" = one pass of the hot path over one batch: prefill -> 64 AR steps (each = 51 diffusion-head evaluations +
sign + projector + one Qwen3-14B block pass) -> tokenizer decode, for ``--bs`` images. See DESIGN.md §Measurement.

  python bench.py --gpus N --steps K --warmup W            # this repo (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU cores (oracle port)

Prints ONE JSON line (rank 0). ``--dump-outputs DIR`` also writes what the last timed step returned (rank 0) as
``DIR/<name>.npy``; the weights, prompt and sampler noise are seeded, so the same arguments give the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "BitDance-14B-64x"
METRIC = "1024px images/sec (14B-64x)"
P_LLM, P_HEAD, P_COND, P_PROJ = 13.2125e9, 1.7585e9, 26.2e6, 26.4e6   # SURVEY.md §8d
KV_BYTES_PER_TOKEN = 163840
DUMP_BYTES = 64 << 20        # --dump-outputs: at most this many bytes in all (arrays, indices, headers, outputs.json)
DEFAULT_LLM_STREAM = True    # one persistent launch per Qwen3 AR block (on par with the chained kernels: profiles/r02_bench_*)


def algorithmic_bytes_per_ar_step(R: int, S: int, avg_ctx: float) -> float:
    """SURVEY.md §8(d): weights streamed once per AR step (cond+uncond batched, cond_embed hoisted) + KV reads."""
    return 2 * P_LLM + (S + 1) * 2 * (P_HEAD - P_COND) + 2 * (P_COND + P_PROJ) + R * avg_ctx * KV_BYTES_PER_TOKEN


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as ``out_dir/<name>.npy`` in float32 and their shapes to ``out_dir/outputs.json``. When they would
    exceed DUMP_BYTES, each is replaced by the same fixed, seeded sample of its C-order flattened elements (a share of the
    budget proportional to its size), and the flat indices kept go to ``out_dir/<name>.index.npy`` (float64, exact
    integers): 12 bytes per kept element."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    n = sum(a.size for a in arrays.values())
    room = DUMP_BYTES - (1 << 16)                 # .npy headers and outputs.json
    sampled = 4 * n > room
    os.makedirs(out_dir, exist_ok=True)
    manifest = {}
    for name, a in arrays.items():
        manifest[name] = {"shape": list(a.shape), "sampled": sampled}
        if sampled:
            keep = int(a.size * (room // 12) // n)
            idx = np.sort(np.random.default_rng(0).choice(a.size, size=keep, replace=False))
            np.save(os.path.join(out_dir, name + ".index.npy"), idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))
    with open(os.path.join(out_dir, "outputs.json"), "w") as f:
        json.dump(manifest, f)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# Reference arms: the UNMODIFIED reference (oracle/_ref, shipped by oracle/make_ref.py) on the host cores / on the GPU
# ---------------------------------------------------------------------------------------------------------------------
AR_STEPS_PER_IMAGE = {"BitDance-14B-64x": 64, "BitDance-14B-16x": 256}


def reference_sample(model: str, device: str, n_warm: int, n_timed: int, S: int, guidance: float, height: int, bs: int,
                     threads: int | None = None, with_decode: bool = True):
    """Times the reference's own ``BitDanceT2IPipeline.gen_image`` (oracle/ref_runner.py: its classes, its loop, random-init
    weights of the named architecture, bf16 autocast as in ``generate()``) on a BOUNDED sample: the causal prefill of the
    cond + uncond prompts, then ``n_warm + n_timed`` AR steps of the unmodified loop (each = 51-evaluation DiffHead.sample
    + sign + MLPconnector + two Qwen3-14B passes over the growing KV cache), then the tokenizer decode of one grid. The
    image time is extrapolated: prefill + (AR steps per image) x median timed step + decode. The sampled steps are the
    FIRST ones of an image (KV cache of ~130-600 tokens against ~2 100 on average): the attention share is underestimated,
    i.e. the extrapolation favours the reference."""
    import statistics
    import torch
    from oracle import ref_runner as rr
    if device == "cpu" and threads:
        torch.set_num_threads(threads)
    pipe, info = rr.build_pipeline(model, device, with_ae=with_decode)
    note = ""
    run = rr.run_bounded(pipe, info, n_ar=n_warm + n_timed, image_px=height, guidance=guidance, S=S, num_images=bs)
    timed = run["ar_s"][n_warm:]
    ar = statistics.median(timed)
    dec = rr.time_decode(pipe, image_px=height, num_images=bs) if with_decode else 0.0
    steps = AR_STEPS_PER_IMAGE.get(model, 64)
    sec_per_batch = run["prefill_s"] + steps * ar + dec
    desc = (f"unmodified reference gen_image on {device} ({'all ' + str(threads) + ' host threads, ' if device == 'cpu' else ''}"
            f"bf16 autocast, random-init {model}): prefill {run['prefill_s']:.2f} s + {n_warm} warm-up + {n_timed} timed AR steps "
            f"(median {ar:.3f} s, all {[round(x, 3) for x in run['ar_s']]}) + decode {dec:.2f} s; image = prefill + {steps} x "
            f"median + decode (extrapolated){note}")
    out = dict(n_warm=n_warm, n_timed=n_timed, images_per_s=bs / sec_per_batch, ar_step_s=ar, prefill_s=run["prefill_s"], decode_s=dec, build_s=info["build_s"],
               sample=desc, measured_s=run["total_s"] + dec)
    del pipe, info
    return out


class CpuReferenceWorker:
    """The unmodified ``gen_image`` on the HOST cores in a subprocess (``python -m oracle.ref_runner``) that logs every event
    as it happens and is killed at its deadline. ``hold=True``: the worker imports and builds the 33 GB model with 4 threads
    right away (overlapping whatever the caller does meanwhile) and waits for ``release()`` before it computes."""

    def __init__(self, model: str, n_warm: int, n_timed: int, S: int, guidance: float, height: int, bs: int,
                 with_decode: bool = False, hold: bool = False):
        import subprocess
        import tempfile
        from bitdance_b200.hostinfo import usable_cpus
        self.args = dict(model=model, n_warm=n_warm, S=S, bs=bs)
        self.threads = usable_cpus()
        prog = tempfile.NamedTemporaryFile(prefix="bd_ref_progress_", suffix=".jsonl", delete=False)
        prog.close()
        self.progress = prog.name
        self.go_file = prog.name + ".go" if hold else ""
        cmd = [sys.executable, "-m", "oracle.ref_runner", "--model", model, "--device", "cpu", "--n-ar", str(n_warm + n_timed),
               "--S", str(S), "--guidance", str(guidance), "--px", str(height), "--bs", str(bs), "--threads", str(self.threads),
               "--decode", "1" if with_decode else "0", "--progress", self.progress] + (["--go-file", self.go_file] if hold else [])
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")   # host-only: flash_attn etc. see the CPU-only process they are tested in
        self.t0 = time.perf_counter()
        self.proc = subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)

    def release(self):
        if self.go_file:
            open(self.go_file, "w").close()

    def result(self, deadline_s: float):
        """Wait at most ``deadline_s`` (from now), kill, derive the number from the event log."""
        import subprocess
        killed = False
        try:
            err = self.proc.communicate(timeout=deadline_s)[1]
        except subprocess.TimeoutExpired:
            self.proc.kill()                              # exactly the process we started
            err = self.proc.communicate()[1]
            killed = True
        wall = time.perf_counter() - self.t0
        ev = []
        with open(self.progress) as f:
            for ln in f:
                try:
                    ev.append(json.loads(ln))
                except ValueError:
                    pass
        for path in (self.progress, self.go_file):
            if path and os.path.exists(path):
                os.unlink(path)
        if not killed and self.proc.returncode != 0:
            raise RuntimeError(f"reference worker failed: {(err or b'').decode(errors='replace')[-300:]}")
        return derive_reference_sample(ev, killed=killed, wall=wall, threads=self.threads, deadline_s=deadline_s, **self.args)

    def abort(self):
        if self.proc.poll() is None:
            self.proc.kill()
            self.proc.communicate()
        for path in (self.progress, self.go_file):
            if path and os.path.exists(path):
                os.unlink(path)


def cpu_reference_sample(model: str, n_warm: int, n_timed: int, S: int, guidance: float, height: int, bs: int,
                         deadline_s: float, with_decode: bool = False):
    """One AR step of the 14B reference costs seconds on some hosts and many minutes on others, so the number is derived
    from whatever finished before the deadline — in this order of preference:
      (a) complete AR steps (median of those after the warm-up ones);
      (b) fewer complete steps than asked: the median of the complete ones (the first excluded when there are several);
      (c) no complete step: per-call stopwatches around the reference's own ``TransEncoder.forward`` and ``Qwen3Model.forward``
          INSIDE the running loop -> AR step = (S + 1) x median evaluation + 2 x median block pass (labelled).
    Raises RuntimeError when not even (c) is possible. Returns the same dict as reference_sample."""
    return CpuReferenceWorker(model, n_warm, n_timed, S, guidance, height, bs, with_decode).result(deadline_s)


def derive_reference_sample(ev, *, killed: bool, wall: float, threads: int, model: str, n_warm: int, S: int, bs: int,
                            deadline_s: float):
    """The number from the worker's event log (see cpu_reference_sample). Pure: tests/test_bench_reference_arm_cpu.py."""
    import statistics
    built = next((e["s"] for e in ev if e["ev"] == "built"), None)
    if built is None:
        raise RuntimeError(f"the reference model was not built within {deadline_s:.0f} s on {threads} host threads")
    steps_t = [e["t"] for e in ev if e["ev"] == "step"]
    gen0 = next((e["t"] for e in ev if e["ev"] == "gen_start"), None)
    done = next((e for e in ev if e["ev"] == "gen_done"), None)
    evals = [e for e in ev if e["ev"] == "eval"]
    llm = [e for e in ev if e["ev"] == "llm"]
    pn = next((e.get("pn") for e in ev if e["ev"] == "built"), None) or 64
    if done is not None:
        ar_all = done["ar_s"]
    else:
        ar_all = [steps_t[i + 1] - steps_t[i] for i in range(len(steps_t) - 1)]   # complete steps only
    # prefill = everything gen_image does before the first head evaluation (4 Qwen3 passes + embeddings)
    first_eval_t0 = (evals[0]["t"] - evals[0]["s"]) if evals else None
    prefill = (first_eval_t0 - gen0) if (first_eval_t0 is not None and gen0 is not None) else None
    if len(ar_all) > n_warm:
        ar, how = statistics.median(ar_all[n_warm:]), f"{n_warm} warm-up + {len(ar_all) - n_warm} timed AR steps"
    elif ar_all:
        use = ar_all[1:] if len(ar_all) > 1 else ar_all
        ar, how = statistics.median(use), f"{len(ar_all)} complete AR step(s) before the deadline (median of {len(use)})"
    else:
        # a block pass = a Qwen3Model call over parallel_num rows per sequence (the two first-block passes of the prefill
        # have the same shape as the two passes of an AR step, over a shorter cache)
        blk = [e["s"] for e in llm if e["rows"] == pn * bs]
        ev_use = [e["s"] for e in (evals[1:] if len(evals) > 2 else evals)]
        if not ev_use or not blk:
            raise RuntimeError(f"not one head evaluation + one block pass of the reference finished within {deadline_s:.0f} s on "
                               f"{threads} host threads (build {built:.0f} s, {len(llm)} Qwen3 passes, {len(evals)} evaluations)")
        ar = (S + 1) * statistics.median(ev_use) + 2 * statistics.median(blk)
        how = (f"NO complete AR step before the deadline: AR step = {S + 1} x median DiffHead evaluation "
               f"({statistics.median(ev_use):.2f} s, {len(ev_use)} samples) + 2 x median Qwen3 block pass ({statistics.median(blk):.2f} s, "
               f"{len(blk)} samples), stopwatches around the reference's own modules inside its running loop")
    dec = next((e["s"] for e in ev if e["ev"] == "decode"), 0.0)
    steps = AR_STEPS_PER_IMAGE.get(model, 64)
    sec = prefill + steps * ar + dec
    desc = (f"unmodified reference gen_image on cpu ({threads} host threads of {os.cpu_count()}, bf16 autocast, random-init {model}), "
            f"subprocess {'killed at its ' + format(deadline_s, '.0f') + ' s deadline' if killed else 'finished in ' + format(wall, '.0f') + ' s'}: "
            f"build {built:.0f} s, prefill {prefill:.2f} s, {how}; AR step {ar:.3f} s; decode "
            f"{'%.2f s' % dec if dec else 'not timed'}; image = prefill + {steps} x AR step + decode (extrapolated)")
    return dict(n_warm=min(n_warm, max(0, len(ar_all) - 1)), n_timed=max(0, len(ar_all) - n_warm), images_per_s=bs / sec, ar_step_s=ar,
                prefill_s=prefill, decode_s=dec, build_s=built, sample=desc, measured_s=wall, threads=threads)


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, S = args.bs, args.sampling_steps
    try:
        r = cpu_reference_sample(args.model, args.warmup, args.steps, S, args.guidance, args.height, B,
                                 deadline_s=float(os.environ.get("BD_REF_DEADLINE_S", "270")), with_decode=True)
    except Exception as e:  # the shipped copy is missing (oracle/make_ref.py not run) or the host cannot hold / run the model
        print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"[:400]}))
        return
    threads = r["threads"]
    value = r["images_per_s"]
    steps = AR_STEPS_PER_IMAGE.get(args.model, 64)
    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * B / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{args.model} random-init, {args.height}x{args.width}, {steps} AR steps, bs={B}, "
                                   f"CFG {args.guidance}, S={S} (+1), synthetic 64-token prompt",
                       "extrapolated": True, "step": "one AR step of the unmodified loop",
                       "ar_steps_run": {"warmup": r["n_warm"], "timed": r["n_timed"]}, "ms_per_ar_step": 1e3 * r["ar_step_s"],
                       "prefill_ms": 1e3 * r["prefill_s"], "decode_ms": 1e3 * r["decode_s"]},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "reference", "sample": r["sample"]},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="bitdance_b200", choices=["bitdance_b200", "reference"])
    ap.add_argument("--model", default=MODEL)
    ap.add_argument("--bs", type=int, default=1)
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--sampling-steps", type=int, default=50)
    ap.add_argument("--guidance", type=float, default=7.5)
    ap.add_argument("--ar-steps", type=int, default=None, help="debug only: truncate the AR loop (invalidates the metric)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the GPU-eager reference leg")
    ap.add_argument("--no-roofline", action="store_true", help="profiling runs: skip the live dominant-kernel timing")
    ap.add_argument("--graph", type=int, default=1, help="replay the AR step as a CUDA graph (1) or launch it eagerly (0)")
    ap.add_argument("--llm-stream", type=int, default=-1,
                    help="Qwen3 AR block as one persistent launch (1) or as chained kernels (0); -1: BD_LLM_STREAM or the default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the tokens and image of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        return run_reference_arm(args)

    cpu_worker = None
    have_ref = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "reference")) or os.path.isdir("/root/reference/modeling")
    if have_ref and not args.no_cpu_baseline and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        # cpu_baseline (rank 0, N = 1): the host-core worker imports and builds its 33 GB model NOW, with 4 threads, while
        # the GPU arm runs; it computes only after release(), when every GPU measurement is done
        import atexit
        try:
            cpu_worker = CpuReferenceWorker(args.model, 1, 1, args.sampling_steps, args.guidance, args.height, args.bs, hold=True)
            atexit.register(cpu_worker.abort)
        except Exception:
            cpu_worker = None

    import torch
    import torch.distributed as dist

    try:   # host-side torch ops of this process: never a wider OpenMP team than the cgroup grants (16 of 128 on this pool)
        from bitdance_b200.hostinfo import usable_cpus
        torch.set_num_threads(max(1, min(torch.get_num_threads(), usable_cpus())))
    except Exception:
        pass
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from bitdance_b200 import _lib
    from bitdance_b200.synthetic import MODELS, build_synthetic_engine

    lib = _lib.load()
    lib.bd_launch_count.restype = __import__("ctypes").c_ulonglong
    _lib.check(lib.bd_device_check(), "bd_device_check")
    llm_stream = None if args.llm_stream < 0 else bool(args.llm_stream)
    if llm_stream is None and "BD_LLM_STREAM" not in os.environ:
        llm_stream = DEFAULT_LLM_STREAM
    eng, embed = build_synthetic_engine(args.model, dev, seed=rank, llm_stream=llm_stream)
    eng.use_graph = bool(args.graph)
    collectives = {}
    if world > 1:
        # the two collectives of the sharded path (SURVEY.md section 8e), on NCCL over NVLink: a start-up broadcast of rank 0's
        # prepacked weight set (what replaces N checkpoint reads), and — inside the e2e region below — one all-gather of the
        # packed token grids per batch. Neither is on the per-step data path: replicas stay independent.
        from bitdance_b200 import parallel
        try:
            ts = eng.weight_tensors() + [embed]
            nbytes = sum(t.numel() * t.element_size() for t in ts)
            dist.barrier()
            torch.cuda.synchronize()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            parallel.broadcast_tensors(ts, src=0)
            b1.record()
            torch.cuda.synchronize()
            tb = torch.tensor([b0.elapsed_time(b1)], device=dev)
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
            collectives["weight_broadcast"] = {"gb": nbytes / 1e9, "tensors": len(ts), "ms": tb.item(),
                                               "gbs_per_receiver": nbytes / 1e9 / (tb.item() / 1e3)}
        except Exception as e:
            collectives["weight_broadcast"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    m = MODELS[args.model]
    pn, vps = m["parallel_num"], eng.vae_patch_size
    h, w = args.height // vps, args.width // vps
    B, S = args.bs, args.sampling_steps
    R = 2 * B if args.guidance > 1.0 else B
    # synthetic prompt (SURVEY.md §8d): 64 cond ids, 3 uncond ids, fixed special ids
    g = torch.Generator().manual_seed(1 + rank)
    cond_ids = torch.randint(0, 151000, (64,), generator=g)
    uncond_ids = torch.randint(0, 151000, (3,), generator=g)
    start_ids = torch.tensor([151700, 151701 + h % 100, 151701 + w % 100] + [151810 + i for i in range(1, pn)])
    ids_host = torch.cat([cond_ids, uncond_ids, start_ids]).pin_memory()
    img_host = torch.empty((B, args.height, args.width, 3), dtype=torch.uint8).pin_memory()

    def gen_resident(ids_dev):
        ce, ue, se = embed[ids_dev[:64]], embed[ids_dev[64:67]], embed[ids_dev[67:]]
        tokens, packed = eng.gen_tokens(ce, ue, se, h=h, w=w, num_images=B, guidance_scale=args.guidance,
                                        num_sampling_steps=S, num_steps=args.ar_steps)
        if args.ar_steps is not None:
            return tokens, None
        return tokens, eng.decode(tokens, h, w)

    # ---- the PUBLIC call: BitDanceT2IPipeline.generate(prompt, ...) -> list[PIL.Image] (t2i_pipeline.py:110-155) over the
    # same engine: host tokenizer, embedding lookup, token ids H2D, the whole path, uint8 pixels D2H, PIL conversion
    from bitdance_b200.modeling.t2i_pipeline import BitDanceT2IPipeline
    from bitdance_b200.synthetic import synthetic_tokenizer
    tokenizer, prompt = synthetic_tokenizer(m["llm"]["vocab_size"], pn, n_words=59)
    pipe = BitDanceT2IPipeline.from_engine(eng, tokenizer=tokenizer, embed_weight=embed, device=dev)
    n_prompt = len(tokenizer.encode(f"<|im_start|>user\n{prompt}<|im_end|>\n<|im_start|>assistant\n"))
    n_uncond = len(tokenizer.encode("<|im_start|>assistant\n"))
    e2e_h2d = 8 * (n_prompt + n_uncond + 2 + pn)

    def gen_e2e():
        if args.ar_steps is not None:
            return gen_resident(ids_host.to(dev, non_blocking=True))
        imgs = pipe.generate(prompt, height=args.height, width=args.width, num_sampling_steps=S,
                             guidance_scale=args.guidance, num_images=B, seed=1234 + rank)
        assert len(imgs) == B and imgs[0].size == (args.width, args.height)
        if world > 1:   # the finished (packed, 16 KB / image) token grids of every rank, one all-gather per batch
            from bitdance_b200 import parallel
            try:
                allg = parallel.gather_token_grids(pipe.last_packed_tokens)
                collectives["token_grid_all_gather"] = {"bytes_per_rank": int(pipe.last_packed_tokens.numel() * 4),
                                                        "gathered_shape": list(allg.shape)}
            except Exception as e:   # never lose the bench line to the optional exchange step
                collectives["token_grid_all_gather"] = {"error": f"{type(e).__name__}: {e}"[:200]}

    ids_dev = ids_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    torch.manual_seed(1234 + rank)    # the sampler noise: the same for every run with the same arguments
    for _ in range(args.warmup):
        gen_resident(ids_dev)
    barrier()
    launches0 = lib.bd_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        for i in range(args.steps):
            if i < args.steps - 1:
                gen_resident(ids_dev)
            else:                             # only the final step's outputs are kept (for --dump-outputs)
                last = gen_resident(ids_dev)
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        tokens, image = last
        dump_outputs(args.dump_outputs, {"tokens": tokens} if image is None else {"tokens": tokens, "image": image})
    del last
    launches = lib.bd_launch_count() - launches0
    # per-phase split of the last configuration (one extra, untimed-for-the-metric pass)
    eng.gen_tokens(embed[ids_dev[:64]], embed[ids_dev[64:67]], embed[ids_dev[67:]], h=h, w=w, num_images=B,
                   guidance_scale=args.guidance, num_sampling_steps=S, num_steps=args.ar_steps, timers=True)
    phases = dict(eng.timings)
    # e2e through host buffers
    gen_e2e()
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        gen_e2e()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    n_img = world * B * args.steps
    value = n_img / (ms / 1e3)
    e2e_value = n_img / (ms_e2e / 1e3)
    ar_steps = phases.get("ar_steps", 0)
    ms_ar = 1e3 * phases.get("ar_s", 0.0) / max(ar_steps, 1)
    avg_ctx = 64 / 2 + 2 + pn + (h * w) / 2
    step_bytes = algorithmic_bytes_per_ar_step(R, S, avg_ctx)
    roof = {} if args.no_roofline else dominant_kernel_roofline(eng, hbm_peak, peak_src, S, args.guidance, B)
    roof["ar_step"] = {"algorithmic_gb": step_bytes / 1e9, "ms": ms_ar, "achieved_gbs": step_bytes / 1e9 / (ms_ar / 1e3) if ms_ar else None,
                       "frac": (step_bytes / 1e9 / (ms_ar / 1e3)) / hbm_peak if ms_ar else None}
    if R * pn > 128 and ms_ar:
        step_flops = 2.0 * P_LLM * R * pn + (S + 1) * 2.0 * P_HEAD * R * pn
        tpk = peaks.get("bf16_tflops_sustained", 1400.0)
        roof["ar_step"].update({"bound": "tensor", "algorithmic_tflop": step_flops / 1e12,
                                "achieved_tflops": step_flops / 1e12 / (ms_ar / 1e3),
                                "frac_tensor": step_flops / 1e12 / (ms_ar / 1e3) / tpk})
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"{args.model} random-init, {args.height}x{args.width}, {(h * w) // pn} AR steps, bs={B}/GPU, "
                               f"CFG {args.guidance}, S={S} (+1), synthetic 64-token prompt",
                   "parallelism": f"replicas x{world} (independent images per GPU, no data-path collective)",
                   "l2": "inputs >> L2: 33 GB of bf16 weights streamed per AR step",
                   "cuda_graph": bool(args.graph), "llm_ar_block": "one persistent launch" if eng.llm.w.layer_tab else "chained kernels",
                   "ms_per_ar_step": ms_ar, "prefill_ms": 1e3 * phases.get("prefill_s", 0.0),
                   "truncated_ar_steps": args.ar_steps},
        "clocks": clk.summary(),
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": int(e2e_h2d),
                "d2h_bytes_per_step": int(img_host.numel()),
                "call": f"BitDanceT2IPipeline.generate(prompt[{n_prompt} tokens], {args.height}, {args.width}, {S}, "
                        f"{args.guidance}, num_images={B}) -> list[PIL.Image]: host tokenizer + embedding lookup + ids H2D + "
                        f"prefill + AR loop + decode + uint8 D2H + PIL"},
        "gpu_launches": int(launches),
        "roofline": roof,
    }
    if collectives:
        line["collectives"] = collectives
    if not args.no_gpu_reference and world == 1:
        # SURVEY.md section 8d's "number to beat": the unmodified reference, eager PyTorch on this same B200 under CUDA
        # autocast (bounded: prefill + 1 warm-up + 3 timed AR steps, extrapolated like the CPU arm)
        try:
            del pipe
            torch.cuda.empty_cache()
            g = reference_sample(args.model, f"cuda:{local}", 1, 3, S, args.guidance, args.height, B)
            line["gpu_eager_reference"] = {"value": g["images_per_s"], "unit": "images/s", "ms_per_ar_step": 1e3 * g["ar_step_s"],
                                           "prefill_ms": 1e3 * g["prefill_s"], "decode_ms": 1e3 * g["decode_s"],
                                           "speedup_e2e": e2e_value / g["images_per_s"], "sample": g["sample"]}
            torch.cuda.empty_cache()
        except Exception as e:
            line["gpu_eager_reference"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    if not args.no_cpu_baseline and world == 1:
        try:
            if cpu_worker is None:
                raise RuntimeError("the reference is not shipped (oracle/make_ref.py) or the worker could not start")
            cpu_worker.release()
            r = cpu_worker.result(float(os.environ.get("BD_CPU_BASELINE_DEADLINE_S", "150")))
            line["cpu_baseline"] = {"value": r["images_per_s"], "unit": "images/s", "cores": r["threads"], "kind": "reference",
                                    "sample": r["sample"] + " [decode not timed in this leg]"}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": os.cpu_count() or 1, "kind": "reference",
                                    "sample": f"unavailable: {type(e).__name__}: {e}"[:300]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dominant_kernel_roofline(eng, hbm_peak, peak_src, S, guidance, B):
    """The dominant kernel is bd_stream_kernel: ONE launch = one DiffHead.sample() = S+1 evaluations of the 1.76 B-parameter
    head + the SDE updates (87 % of an AR step's bytes). Timed live with CUDA events on the launching (current) stream.
    Algorithmic bytes per launch (SURVEY.md section 8d): (S+1) * 2 * (P_head - P_cond) + 2 * P_cond — every weight streamed
    once per evaluation, cond_embed once per launch. `traffic` is dram__bytes_read + dram__bytes_write of the same launch
    from the committed ncu --set full capture (profiles/r01_stream_kernel_ncu.json), or null when that file is absent.
    `gemm_chain`: the same kernel on a bare chain of 157 MB GEMM ops (M=128, N=15360, K=5120, 4 different weight buffers
    = 629 MB >> L2) — the steady-state streaming rate without the head's row / attention ops."""
    import torch
    from bitdance_b200 import ops
    head = eng.head
    D, Dz = head.cfg["D"], head.cfg["Dz"]
    dev = eng.device
    pn = eng.pn
    R = (2 if guidance > 1.0 else 1) * B
    z = torch.randn(R, pn, Dz, device=dev)
    stream_path = head.w_stream is not None and R * pn <= 128

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms = timed(lambda: head.sample(z, guidance, S), 3)
    if not stream_path:
        # batch > one 128-row tile (bs >= 2 with CFG): M = R * pn rows per Linear is past the ridge (~280 rows at 2.25 PFLOP/s
        # over 8 TB/s), the sampler is TENSOR-bound: algorithmic flops = (S + 1) evaluations x 2 x P_head x M rows
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        tpeak = peaks.get("bf16_tflops_sustained", 1400.0)
        flops = (S + 1) * 2.0 * P_HEAD * R * pn
        ach = flops / 1e12 / (ms / 1e3)
        return {"bound": "tensor", "kernel": "bd_head_sample multi-kernel path (bd_gemm_kernel, M = %d rows)" % (R * pn),
                "achieved": ach, "peak": tpeak, "peak_source": "measured (sustained)" if peaks else "fallback", "unit": "TFLOP/s",
                "frac": ach / tpeak, "traffic": None, "ms_per_launch": ms, "us_per_evaluation": ms * 1e3 / (S + 1),
                "algorithmic_flops_per_launch": flops}
    bytes_alg = (S + 1) * 2 * (P_HEAD - P_COND) + 2 * P_COND
    ach = bytes_alg / 1e9 / (ms / 1e3)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r01_stream_kernel_ncu.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    out = {"bound": "hbm",
           "kernel": ("bd_stream_kernel (persistent: one launch = DiffHead.sample, %d evaluations)" % (S + 1)) if stream_path
           else "bd_head_sample multi-kernel path (batch > one 128-row tile)",
           "achieved": ach, "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / hbm_peak,
           "traffic": traffic, "traffic_source": "profiles/r01_stream_kernel_ncu.json (ncu --set full of one launch of this "
                                                 "kernel, committed; a citation, not a measurement of this run)",
           "ms_per_launch": ms, "us_per_evaluation": ms * 1e3 / (S + 1), "algorithmic_bytes_per_launch": bytes_alg}
    if stream_path:
        N, K, nbuf = 3 * D, D, 4
        w = (torch.randn(N, K, device=dev) * 0.02).to(torch.bfloat16)
        p0 = ops.stream_pack_weight(w, None)
        n = p0.data.numel()
        big = p0.data.repeat(nbuf)
        views = [ops.StreamWeight(big[i * n:(i + 1) * n], p0.bias, N, K, 1, p0.n_ctas, 0) for i in range(nbuf)]
        a = ops.to_blocked(torch.randn(128, K, device=dev).to(torch.bfloat16))
        reps = 8
        msg = timed(lambda: ops.stream_gemm(a, views, epi="bias", repeat=reps, a_is_blocked=True, M=128), 2)
        per_op_us = msg * 1e3 / (reps * nbuf)
        out["gemm_chain"] = {"shape": "M=128 N=%d K=%d, %d ops per launch" % (N, K, reps * nbuf), "us_per_op": per_op_us,
                             "achieved_gbs": N * K * 2 / 1e9 / (per_op_us / 1e6),
                             "frac": N * K * 2 / 1e9 / (per_op_us / 1e6) / hbm_peak}
        del big, views, p0, w
    return out


if __name__ == "__main__":
    main()
