"""bench.py — decode tokens/sec of the soft-attention LSTM decode path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl sat|reference] [--workload 2|3|4|5]
                    [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" is one pass of the hot path over one batch of synthetic contexts: project the
contexts + initialize + T decode steps for B images (BASELINE config 2: B=64, L=196, D=512,
H=1024, V=10000, T=20), i.e. B*T tokens.  Inputs rotate over a pool of distinct context
batches larger than L2.  Weights: random U(-0.08, 0.08) of the reference architecture.

  value     tokens/s with the contexts resident in HBM when the timed region starts
  e2e       the same metric through the C ABI host-buffer call (pinned host contexts in,
            tokens out, host<->device copies inside the timed region)
  roofline  the fused attention kernel timed alone with CUDA events (L2 flushed between
            launches) against the measured HBM copy peak
  cpu_baseline  the numpy oracle (oracle/ref_step.py, "port": TensorFlow cannot be installed
            here) on the host cores, bounded sample
--impl reference times that CPU restatement as its own arm (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1] and configs[2]
    2: dict(name="config2: B=64 L=196 D=512 H=1024 E=512 A=512 Dd=1024 V=10000 T=20 (2-layer attend/decode/init)",
            B=64, L=196, D=512, H=1024, V=10000, T=20),
    3: dict(name="config3: B=256 L=196 D=2048 H=1536 E=512 A=512 Dd=1024 V=10000 T=20",
            B=256, L=196, D=2048, H=1536, V=10000, T=20),
    # BASELINE.json configs[3]: training step, 64 images per GPU (512 on 8 GPUs), forward + backward + gradient
    # all-reduce + clip + Adam; tokens = teacher-forced words per step
    4: dict(name="config4: training step B=64/GPU L=196 D=512 H=1024 V=10000 T=20, fwd+bwd+all-reduce+Adam (large "
                 "products on the tcgen05 dense kernel as split bf16x3, the rest fp32 CUDA-core kernels; dropout on)", B=64, L=196, D=512, H=1024, V=10000, T=20, train=True),
    # BASELINE.json configs[4]: beam search, 128 images x beam 3, T=30 (tokens = images x T)
    5: dict(name="config5: beam search beam=3, 128 images, L=196 D=512 H=1024 V=10000 T=30 (device-side TopN)",
            B=128, L=196, D=512, H=1024, V=10000, T=30, beam=3),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx or None, reasons=sorted(reasons),
                    samples=len(sm))


def loop_kernel_times(model, ctx, T, work, pk):
    """Per-kernel durations of the greedy loop measured on the device (option "trace" = 3: every launch stamps
    min CTA start / min dependency-release / max accumulator-ready / max end with %globaltimer).  Returns the list
    for roofline.kernels[].  `work`: name -> (algorithmic bytes, flops incl. the 3 passes of the bf16x3 split)."""
    import numpy as np
    import torch
    import cuda.bindings.runtime as cr
    model.set_option("graphs", 0)
    for _ in range(2):
        model.loop_device(ctx, T)
    torch.cuda.synchronize()
    model.set_option("trace", 3)
    model.loop_device(ctx, T)
    torch.cuda.synchronize()
    n = model.info("tl_count")
    host = np.zeros(1024 * 16, np.uint64)
    cr.cudaMemcpy(host.ctypes.data, model.info("trace_ptr"), host.nbytes, cr.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    names = []
    for i in range(n):
        model.info("tl_tag_%d" % i)
        names.append(model.lib.sat_last_error().decode().strip())
    model.set_option("trace", 0)
    model.set_option("graphs", 1)
    cell = lambda i, k: float(int(host[4 * i + k])) if 0 < int(host[4 * i + k]) < 2 ** 62 else float("nan")
    groups = {}
    for i, nm in enumerate(names):
        start, end, go, acc = cell(i, 0), cell(i, 1), cell(i, 2), cell(i, 3)
        groups.setdefault(nm, []).append(((end - go) / 1e3, (end - start) / 1e3, (acc - go) / 1e3))
    med = lambda v: float(np.nanmedian(np.array(v))) if len(v) else float("nan")
    out = []
    label = {"lstm": "LSTM cell", "dec1": "decode fc_1 || attend fc_1b", "dec2": "vocabulary layer + arg-max", "attention": "attention"}
    for nm, rows in groups.items():
        if len(rows) < T // 2:
            continue                                   # prologue launches (projection, initialize)
        fam, grid = nm.split("/")[0], nm.split("/")[-1]
        # (phases of the chained launch stamp: phase opened -> last CTA arrived)
        us = med([r[1] for r in rows]) if fam.startswith("phase") else med([r[0] for r in rows])
        ent = dict(kernel=nm, launches=len(rows), us_in_loop=us, us_first_cta_start_to_end=med([r[1] for r in rows]),
                   timing="device %globaltimer inside one eager loop: first CTA through its dependency wait -> last CTA done (median)")
        key = {"phase0": "lstm", "phase1": "dec1", "phase2": "dec2"}.get(fam, fam)
        if key in work:
            by, fl = work[key]
            ent.update(what=label[key], algorithmic_bytes=by, achieved_gbs=by / (us * 1e3), frac_hbm=by / (us * 1e3) / pk["hbm"])
            if fl:
                ent.update(flops_bf16x3=fl, tflops=fl / (us * 1e6), frac_tensor=fl / (us * 1e6) / pk["tf_sust"])
        elif fam == "chain":
            by = sum(work[k][0] for k in ("lstm", "dec1", "dec2"))
            fl = sum(work[k][1] for k in ("lstm", "dec1", "dec2"))
            ent.update(what="chained dense launch: LSTM -> fc_1 || q -> vocabulary layer (sat_chain.cu)", algorithmic_bytes=by,
                       achieved_gbs=by / (us * 1e3), frac_hbm=by / (us * 1e3) / pk["hbm"], flops_bf16x3=fl,
                       tflops=fl / (us * 1e6), frac_tensor=fl / (us * 1e6) / pk["tf_sust"])
        out.append(ent)
    tops = [e for e in out if not e["kernel"].startswith("phase")]
    if tops:
        top = max(tops, key=lambda e: e["us_in_loop"])
        for e in out:
            e["dominant"] = e is top
    return out


def dump_outputs(directory, arrays):
    """Write what the timed path returned in its last step as <directory>/<name>.npy: float64 stays float64, every
    other type becomes float32 (token ids < 2**24 are exact).  Inputs and weights are seeded, so two builds run with
    the same arguments can be compared output for output: two runs of one build give bit-identical greedy and beam
    outputs, and training losses that agree to fp32 round-off.  Every workload's outputs are far below 64 MB."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def oracle_setup(wl, seed=1234):
    from oracle import ref_step as R
    ocfg = R.OracleConfig(batch_size=wl["B"], num_ctx=wl["L"], dim_ctx=wl["D"], num_lstm_units=wl["H"],
                          vocabulary_size=wl["V"], max_caption_length=wl["T"])
    return R, ocfg, R.init_weights(ocfg, seed)


def time_cpu_oracle(wl, steps, warmup, budget_s=25.0):
    """The reference's CPU path (restated oracle: fc_1a projection recomputed every step, exactly as
    model.py:259-262 does), all host cores through numpy's BLAS.  Bounded sample."""
    import numpy as np
    R, ocfg, w = oracle_setup(wl)
    ctx = R.synth_contexts(ocfg, wl["B"])
    c, h = R.initialize(ocfg, w, ctx)
    word = np.zeros(wl["B"], np.int32)
    R.decode_step(ocfg, w, ctx, word, c, h)               # warm-up (BLAS thread pool, page faults)
    # give the CPU its best case: pick the BLAS thread count that runs one step fastest
    ncpu = os.cpu_count() or 1
    best_t, per_step, limiter = ncpu, None, None
    try:
        from threadpoolctl import threadpool_limits
        cands = sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu})
        for t in cands:
            with threadpool_limits(limits=t):
                R.decode_step(ocfg, w, ctx, word, c, h)
                t0 = time.perf_counter()
                R.decode_step(ocfg, w, ctx, word, c, h)
                dt = time.perf_counter() - t0
            if per_step is None or dt < per_step:
                best_t, per_step = t, dt
        limiter = threadpool_limits(limits=best_t)
    except Exception:
        t0 = time.perf_counter()
        R.decode_step(ocfg, w, ctx, word, c, h)
        per_step = time.perf_counter() - t0
    T_s = max(1, min(wl["T"], int(budget_s / max(per_step, 1e-3) / max(steps + warmup, 1))))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        c, h = R.initialize(ocfg, w, ctx)
        word = np.zeros(wl["B"], np.int32)
        for t in range(T_s):
            r = R.decode_step(ocfg, w, ctx, word, c, h)
            c, h = r["memory"], r["output"]
            word = r["logits"].argmax(1).astype(np.int32)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    toks = wl["B"] * T_s * len(times)
    if limiter is not None:
        limiter.restore_original_limits()
    return dict(value=toks / total, unit="tokens/s", cores=best_t, kind="port",
                sample="%d x (initialize + %d of %d decode steps) at B=%d, numpy/BLAS fp32 oracle restating "
                       "model.py (not TensorFlow: not installable here); %d BLAS threads (fastest of the counts "
                       "tried on %d host cores)" % (len(times), T_s, wl["T"], wl["B"], best_t, ncpu),
                ms_per_step=1e3 * total / len(times),              # of the MEASURED sample (T_s decode steps per bench step)
                ms_per_full_step=1e3 * total / len(times) * (wl["T"] / T_s), steps_sampled=T_s, host_cores=ncpu)


def bench_config(wl, world, pool=None, pool_mb=None):
    """The `config` object of a bench line: the same keys for the sat arm and the reference arm."""
    B, T = wl["B"], wl["T"]
    beam = wl.get("beam", 1)
    if wl.get("train"):
        step = "one optimisation step: forward + backward + gradient all-reduce + clip + Adam on %d images per GPU" % B
    elif beam > 1:
        step = "beam search: %d images x beam %d, %d steps, device-side TopN; tokens = images x steps" % (B, beam, T)
    else:
        step = ("project contexts + initialize + %d decode steps (greedy) for %d images; consecutive batches overlap: "
                "the prologue of batch i+1 runs under the decode steps of batch i" % (T, B))
    return {"workload": wl["name"], "per_gpu_batch": B, "global_batch": B * world,
            "parallelism": "dp%d (batch sharded, replicated weights, no data-path collective in decoding)" % world,
            "precision": "fp32 in/out; GEMMs as split bf16x3 on tcgen05 with fp32 TMEM accumulation",
            "l2": ("inputs rotate over %d context batches (%.0f MB + 137 MB weights/activations) > 126 MB L2" % (pool, pool_mb))
                  if pool else "inputs larger than L2 (context batches rotate)",
            "step": step}


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    cb = time_cpu_oracle(wl, args.steps, max(args.warmup, 1))
    line = {"impl": "reference", "metric": "decode tokens/sec", "value": cb["value"], "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(bench_config(wl, args.gpus),
                           note="reference arm: CPU restatement of the reference path (TensorFlow 1.x cannot be installed "
                                "offline), rank 0 only; each timed step is a bounded sample of the workload: initialize + "
                                "%d of its %d decode steps for the full batch (ms_per_step is that sample's own time; "
                                "tokens/s counts the tokens it produced)" % (cb["steps_sampled"], wl["T"])),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def measure_training(wl, model, rank, local_rank, world, dev, steps, warmup, e2e=True, sample_clocks=True, dump=None):
    """config 4: one optimisation step per bench step (forward + backward + gradient all-reduce + clip + Adam); weak
    scaling, 64 images per GPU.  dump: directory for the losses and squared gradient norm of the last timed step.
    Returns the record (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from sat_b200 import parallel
    B, L, D, T, V = wl["B"], wl["L"], wl["D"], wl["T"], wl["V"]
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    model.train_setup(B, T)
    pool = 3
    ctx_host = [torch.relu(torch.randn(B, L, D, generator=g)).pin_memory() for _ in range(pool)]
    ctx_dev = [c.to(dev) for c in ctx_host]
    sent = torch.randint(1, V, (B, T), generator=g, dtype=torch.int32).to(dev)
    lens = torch.randint(8, T + 1, (B,), generator=g)
    masks = (torch.arange(T)[None, :] < lens[:, None]).float().to(dev)
    st = model.stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(warmup, 3 * pool)):   # eager pass + graph capture + first replay per context buffer
        out = model.train_step(ctx_dev[i % pool], sent, masks, seed=1 + i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0 and sample_clocks:
        sampler.start()
        time.sleep(0.3)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(st):
        ev0.record(st)
        for i in range(steps):
            last = model.train_step(ctx_dev[i % pool], sent, masks, seed=100 + i, sync=False)   # losses stay on the device
        ev1.record(st)
    barrier()
    if dump and rank == 0:
        dump_outputs(dump, dict(losses=last[0], gradient_norm_squared=last[1]))
    ms = parallel.max_over_ranks(ev0.elapsed_time(ev1), dev)
    clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
    value = world * B * T * steps / (ms / 1e3)
    # the collective alone: the flat gradient buffer (+ the packed scalars) all-reduced back to back, CUDA events, max over ranks
    ar_ms = None
    if world > 1:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            model.allreduce_gradients()
        barrier()
        with torch.cuda.stream(st):
            e0.record(st)
            for _ in range(5):
                model.allreduce_gradients()
            e1.record(st)
        barrier()
        ar_ms = parallel.max_over_ranks(e0.elapsed_time(e1) / 5, dev)
    rec_e2e = None
    if e2e:
        # end to end: contexts come from pinned host memory every step (into two device staging buffers, as an input
        # pipeline would: the captured step graph is keyed by the buffer addresses), the losses go back to the host
        stage = [torch.empty_like(ctx_dev[0]) for _ in range(2)]
        for i in range(4):
            stage[i % 2].copy_(ctx_host[i % pool], non_blocking=True)
            model.train_step(stage[i % 2], sent, masks, seed=7)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            stage[i % 2].copy_(ctx_host[i % pool], non_blocking=True)
            out = model.train_step(stage[i % 2], sent, masks, seed=200 + i)
        torch.cuda.synchronize()
        e2e_s = parallel.max_over_ranks(time.perf_counter() - t0, dev)
        rec_e2e = {"value": world * B * T * steps / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": B * L * D * 4,
                   "d2h_bytes_per_step": 24, "ms_per_step": 1e3 * e2e_s / steps}
    if rank != 0:
        return None
    nparams = int(model.params.numel())
    return {"metric": "training tokens/sec (teacher-forced words per second, fwd+bwd+all-reduce+Adam)",
            "value": value, "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": max(warmup, 3 * pool),
            "ms_per_step": ms / steps, "allreduce_ms": ar_ms,
            "collective": ("ONE NCCL all-reduce per step over the flat fp32 gradient buffer (%d floats = %.1f MB) with the "
                           "whole-batch mask sum and the loss scalars packed into its tail" % (nparams, nparams * 4 / 1e6))
                          if world > 1 else None,
            "per_gpu_batch": B, "global_batch": B * world, "e2e": rec_e2e, "clocks": clocks, "last_losses": out}


def run_training(args, wl, model, cfg, rank, local_rank, world, dev):
    import torch.distributed as dist
    rec = measure_training(wl, model, rank, local_rank, world, dev, args.steps, args.warmup, dump=args.dump_outputs)
    if rank == 0:
        line = {"metric": rec["metric"], "value": rec["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
                "warmup": rec["warmup"], "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(bench_config(wl, world), l2="activations of a step (>1.5 GB stashed) exceed L2",
                               parallelism="dp%d: batch sharded, replicated weights; %s" % (world, rec["collective"] or "single GPU")),
                "e2e": rec["e2e"], "gpu_launches": None, "clocks": rec["clocks"], "roofline": None, "cpu_baseline": None,
                "detail": {"last_losses": rec["last_losses"], "allreduce_ms": rec["allreduce_ms"]}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="sat", choices=["sat", "reference"])
    ap.add_argument("--workload", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-train", action="store_true", help="skip the training sub-record of the default line")
    ap.add_argument("--pool", type=int, default=6, help="distinct context batches rotated through")
    ap.add_argument("--profile-run", action="store_true",
                    help="for runs under ncu: only the device-resident timed loop (no clock pre/post roll, no e2e, no roofline legs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "sat":
        ap.error("--dump-outputs applies to --impl sat")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return run_reference(args, wl, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist
    import sat_b200
    from sat_b200 import parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: no CUDA device visible (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        parallel.init_process_group("nccl")
    dev = torch.device("cuda", local_rank)
    B, L, D, H, V, T = (wl[k] for k in "BLDHVT")

    beam = wl.get("beam", 1)
    cfg = sat_b200.Config(batch_size=B, beam_size=beam, num_ctx=L, dim_ctx=D, num_lstm_units=H, vocabulary_size=V,
                          max_caption_length=T)
    model = sat_b200.CaptionGenerator(cfg)
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    shapes = sat_b200.weight_shapes(cfg)
    wg = torch.Generator(device="cpu").manual_seed(1234)           # identical replicas on every rank
    weights = {n: (torch.rand(*s, generator=wg) * 0.16 - 0.08) for n, s in shapes.items()}
    assert model.set_weights(weights) == 0
    del weights

    if wl.get("train"):
        return run_training(args, wl, model, cfg, rank, local_rank, world, dev)

    pool = max(1, args.pool)
    ctx_host = [torch.relu(torch.randn(B, L, D, generator=g)).pin_memory() for _ in range(pool)]
    ctx_dev = [c.to(dev) for c in ctx_host]
    tok_host = torch.empty(B, T, dtype=torch.int32).pin_memory()
    pool_mb = pool * B * L * D * 4 / 1e6
    st = model.stream
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident loop
    # the context batches are complete in HBM before anything is timed, which is what "xbatch" asks of the caller:
    # the projection / initialize prologue of batch i+1 then runs on its own stream under the decode steps of batch i
    if beam == 1:
        model.set_option("xbatch", 1)

    def loop(i):
        if beam > 1:
            return model.beam_device(ctx_dev[i % pool], beam, T, 2)
        return model.loop_device(ctx_dev[i % pool], T)[:1]

    for i in range(max(args.warmup, 3) + 2 * pool):       # warm-up also builds one CUDA graph per pool entry
        loop(i)
    barrier()
    # The timed region (K loops, a few tens of ms) is shorter than nvidia-smi's sampling period, so it is embedded
    # in a continuous run of the SAME loop: identical untimed loops keep the GPU in the same state while the
    # sampler collects clocks / throttle reasons before, during and after the K timed ones.
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    def roll(seconds, need_rows):
        t_end = time.time() + seconds
        i = 0
        while time.time() < t_end or (rank == 0 and len(sampler.rows) < need_rows and time.time() < t_end + 3.0):
            loop(i); i += 1
            if i % 16 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
    if not args.profile_run:
        roll(0.4, 2)
    model.set_option("reset_counters", 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(st):
        ev0.record(st)
        for i in range(args.steps):
            last = loop(i)
        ev1.record(st)
    barrier()
    if args.dump_outputs and rank == 0:      # (persistent buffers: dumped before any later loop overwrites them)
        names = ("sentences", "lengths", "scores", "num_results", "complete") if beam > 1 else ("tokens",)
        dump_outputs(args.dump_outputs, dict(zip(names, last)))
    ms = ev0.elapsed_time(ev1)
    launches = model.info("launches")
    if not args.profile_run:
        roll(0.3, len(sampler.rows) + 2 if rank == 0 else 0)
    clocks = sampler.stop() if rank == 0 else None
    if args.profile_run:
        if rank == 0:
            print(json.dumps({"profile_run": True, "value": value if False else world * B * T * args.steps / (ms / 1e3),
                              "ms_per_step": ms / args.steps, "note": "numbers printed under a profiler are not bench values"}))
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    if clocks is not None:
        clocks["note"] = ("nvidia-smi sampled every 50 ms while the same decode loop ran back to back for ~0.4 s before, "
                          "during and ~0.3 s after the timed steps")
    ms = parallel.max_over_ranks(ms, dev)
    value = world * B * T * args.steps / (ms / 1e3)

    # ---------------------------------------------------------------- end to end (host buffers)
    import ctypes as C
    hp = lambda t: C.c_void_p(t.data_ptr())

    if beam > 1:
        b_sent = torch.empty(B, beam, T, dtype=torch.int32).pin_memory()
        b_len = torch.empty(B, beam, dtype=torch.int32).pin_memory()
        b_sc = torch.empty(B, beam, dtype=torch.float64).pin_memory()
        b_n = torch.empty(B, dtype=torch.int32).pin_memory()
        b_c = torch.empty(B, dtype=torch.int32).pin_memory()

    def e2e_step(i):
        if beam > 1:
            rc = model.lib.sat_beam_search_host(model._h, hp(ctx_host[i % pool]), B, beam, T, 2, hp(b_sent), hp(b_len),
                                                hp(b_sc), hp(b_n), hp(b_c), model._st())
        else:
            rc = model.lib.sat_decode_loop_host(model._h, hp(ctx_host[i % pool]), B, T, None, hp(tok_host), model._st())
        assert rc == 0, model.lib.sat_last_error()

    tok_pipe = [torch.empty(B, T, dtype=torch.int32).pin_memory() for _ in range(2)]

    def e2e_run(n):
        """n batches through the public host-buffer API; every batch's contexts are uploaded from pinned host
        memory and its tokens read back inside the region."""
        if beam > 1:
            for i in range(n):
                e2e_step(i)                              # synchronous: returns with the captions in host memory
            return
        # greedy loop: the pipelined form (submit batch i+1, then wait for batch i) overlaps uploads with decoding
        checksum = 0
        for i in range(n):
            model.loop_host_submit(ctx_host[i % pool], T, tok_pipe[i & 1], i & 1)
            if i >= 1:
                checksum += int(model.loop_host_wait((i - 1) & 1)[0, 0])      # tokens of batch i-1 are on the host
        checksum += int(model.loop_host_wait((n - 1) & 1)[0, 0])
        return checksum

    e2e_run(4)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    torch.cuda.synchronize()
    e2e_s = parallel.max_over_ranks(time.perf_counter() - t0, dev)
    # the plain synchronous call (upload, decode, download, one after the other), for reference
    t1 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t1
    e2e = dict(value=world * B * T * args.steps / e2e_s, unit="tokens/s", h2d_bytes_per_step=B * L * D * 4,
               d2h_bytes_per_step=B * T * 4, ms_per_step=1e3 * e2e_s / args.steps,
               api=("sat_decode_loop_host_submit/_wait (two staging slots: upload of batch i+1 overlaps decode of batch i)"
                    if beam == 1 else "sat_beam_search_host (synchronous)"),
               synchronous_call_tokens_per_s=B * T * args.steps / e2e_sync_s)

    # ---------------------------------------------------------------- attention kernel roofline
    roof = None
    extra = {}
    if rank == 0 and beam == 1:
        pk = peaks()
        A = cfg.dim_attend_layer
        flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
        hstate = torch.rand(B, H, device=dev) - 0.5
        alpha = torch.empty(B, L, device=dev)
        z = torch.empty(B, D, device=dev)
        model.prepare(ctx_dev[0], want_state=False)
        torch.cuda.synchronize()
        def time_attention(sms, reps=20):
            """Duration of one attention launch with a cold L2, from CUDA events on the launch stream.  Events around
            a single ~12 us kernel mostly measure launch latency (~6 us here), so the interval covers `reps`
            back-to-back (256 MB L2 flush, attention kernel) pairs and the same number of flushes alone is
            subtracted: (T[reps x (flush + kernel)] - T[reps x flush]) / reps."""
            model.set_option("att_sms", sms)
            rc = model.lib.sat_attention_fwd(model._h, hp(ctx_dev[0]), hp(hstate), hp(alpha), hp(z), B, 1, model._st())
            assert rc == 0, model.lib.sat_last_error()
            model.set_option("att_reuse_q", 1)        # q of the call above: the following calls launch the kernel alone
            def series(with_kernel):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(st):
                    flush.zero_()
                    e0.record(st)
                    for i in range(reps):
                        flush.zero_()
                        if with_kernel:
                            rc = model.lib.sat_attention_fwd(model._h, hp(ctx_dev[0]), hp(hstate), hp(alpha), hp(z), B, 1,
                                                             model._st())
                            assert rc == 0, model.lib.sat_last_error()
                    e1.record(st)
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) * 1e6
            series(True); series(False)
            both = min(series(True) for _ in range(3))
            base = min(series(False) for _ in range(3))
            model.set_option("att_reuse_q", 0)
            model.set_option("att_sms", 0)
            return (both - base) / reps
        loop_grid = model.info("att_loop_grid")       # CTAs of the attention launches inside the timed decode loop
        att_ns_full = time_attention(0)                # whole GPU
        att_ns = time_attention(loop_grid) if 0 < loop_grid < 148 else att_ns_full
        # per-family times of one eager step (cold L2), for the breakdown
        model.set_option("profile", 1)
        lw = torch.zeros(B, dtype=torch.int32, device=dev)
        c_in = torch.rand(B, H, device=dev) - 0.5
        with torch.cuda.stream(st):
            for i in range(5):
                flush.zero_()
                model.step_device(ctx_dev[0], lw, c_in, hstate, want=())
        torch.cuda.synchronize()
        fam = {t: model.info("prof_ns_" + t) / max(1, model.info("prof_n_" + t)) / 1e3
               for t in ("att_state", "att", "lstm", "dec1", "dec2")}
        model.set_option("profile", 0)
        att_bytes = 4 * (B * L * (D + A) + B * A + A + B * L + B * D)       # SURVEY.md §8(d)
        achieved = att_bytes / att_ns                                       # bytes/ns == GB/s
        # DRAM traffic is NOT measured by this run (it needs ncu): the figure below is read from the committed ncu capture
        # and labelled as such
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "att_traffic.json")   # dram__bytes_read+write of one ncu --set full capture
        if os.path.exists(tp) and args.workload == 2:
            tj = json.load(open(tp))
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_src = "not measured in this run: " + tj["source"]
        roof = dict(bound="hbm", achieved=achieved, peak=pk["hbm"], unit="GB/s", frac=achieved / pk["hbm"],
                    traffic=traffic, traffic_source=traffic_src,
                    kernel=("att_wpc_kernel<1>" if (D == 512 and A == 512) else "att_fused_kernel<1>"),
                    grid=loop_grid, us_per_launch=att_ns / 1e3, us_per_launch_whole_gpu=att_ns_full / 1e3,
                    achieved_whole_gpu=att_bytes / att_ns_full,
                    algorithmic_bytes=att_bytes, peak_source=pk["src"] + " HBM copy, burst",
                    timing=("CUDA events on the launch stream around 20 x (256 MB L2 flush, kernel) minus 20 x flush, / 20; "
                            "grid = the one the decode loop launches (there it shares the GPU with the vocabulary layer), "
                            "timed alone"))
        E = cfg.dim_embedding
        Dd = cfg.dim_decode_layer
        lstm_bytes = 4 * ((D + E + H) * 4 * H + 4 * H)
        dec2_bytes = 4 * (Dd * V + V)
        dec1_bytes = 4 * ((H + D + E) * Dd + Dd + H * A + A)
        # ---- the other kernels of a step, timed INSIDE the loop on the device clock (%globaltimer stamps of every launch
        # of one eager loop: first CTA through its dependency -> last CTA done; CUDA events cannot bracket one kernel of
        # a programmatic-dependent-launch chain).  Weight-stream fraction against the HBM peak and tensor fraction
        # (2*M*N*K x 3 passes of the bf16x3 split) against the sustained bf16 peak, per kernel; `dominant` = longest.
        kernels = loop_kernel_times(model, ctx_dev[0], T, dict(
            lstm=(lstm_bytes, 3 * 2 * B * (D + E + H) * 4 * H), dec1=(dec1_bytes, 3 * 2 * B * ((H + D + E) * Dd + H * A)),
            dec2=(dec2_bytes, 3 * 2 * B * Dd * V), attention=(att_bytes, 0)), pk)
        roof["kernels"] = kernels
        step_bytes = att_bytes + lstm_bytes + dec1_bytes + dec2_bytes
        roof["step"] = dict(algorithmic_bytes=step_bytes, us=1e3 * ms / args.steps / T,
                            achieved=step_bytes / (1e6 * ms / args.steps / T), frac=step_bytes / (1e6 * ms / args.steps / T) / pk["hbm"],
                            note="whole decode step (all kernels): algorithmic bytes / (timed loop / T)")
        extra = dict(kernel_us_cold=fam,
                     lstm_weight_stream_gbs=lstm_bytes / (fam["lstm"] * 1e3) if fam["lstm"] else None,
                     vocab_weight_stream_gbs=dec2_bytes / (fam["dec2"] * 1e3) if fam["dec2"] else None,
                     lstm_tflops=2 * B * (D + E + H) * 4 * H / (fam["lstm"] * 1e-6) / 1e12 if fam["lstm"] else None,
                     step_floor_us=1e-3 * (att_bytes + lstm_bytes + dec2_bytes + 4 * ((H + D + E) * Dd + H * A))
                     / pk["hbm"])

    cpu = None
    if rank == 0 and not args.no_cpu and beam == 1:
        cpu = time_cpu_oracle(wl, 3, 1)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # ---------------------------------------------------------------- strong scaling (SURVEY §8e: next to the weak number)
    # the SAME 64-image batch cut into contiguous shards of B / N images per GPU (no collective): what one caption batch
    # gains from N GPUs.  Weight-bound layers lose efficiency as the per-GPU batch shrinks; reported, not optimised for.
    strong = None
    if beam == 1 and world > 1 and B % world == 0:
        Bs = B // world
        shard = [c[rank * Bs:(rank + 1) * Bs].contiguous() for c in ctx_dev]
        for i in range(3 + 2 * pool):
            model.loop_device(shard[i % pool], T)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            s0.record(st)
            for i in range(args.steps):
                model.loop_device(shard[i % pool], T)
            s1.record(st)
        barrier()
        sms = parallel.max_over_ranks(s0.elapsed_time(s1), dev)
        strong = {"value": B * T * args.steps / (sms / 1e3), "unit": "tokens/s", "scaling": "strong", "global_batch": B,
                  "per_gpu_batch": Bs, "ms_per_step": sms / args.steps,
                  "speedup_vs_one_gpu_line": None, "note": "same metric with the 64-image batch sharded over the GPUs"}

    # ---------------------------------------------------------------- training sub-record (BASELINE config 4)
    # The default run also takes a short measurement of the data-parallel training step at the same per-GPU shapes
    # (64 images per GPU, weak scaling), so that the driver's 1/2/4/8-GPU scaling runs record the step that contains
    # the design's only collective.  Its own line: `python bench.py --workload 4`.
    train_rec = None
    if beam == 1 and args.workload == 2 and not args.no_train:
        try:
            train_rec = measure_training(WORKLOADS[4], model, rank, local_rank, world, dev, max(4, args.steps // 2), 3,
                                         e2e=False, sample_clocks=False)
        except Exception as exc:                      # never lose the decode line over the sub-record
            train_rec = {"error": repr(exc)} if rank == 0 else None

    if rank == 0:
        line = {"metric": "decode tokens/sec", "value": value, "unit": "tokens/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": bench_config(wl, world, pool, pool_mb),
                "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "train": train_rec, "strong_scaling": strong, "detail": extra}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
