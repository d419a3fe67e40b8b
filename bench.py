#!/usr/bin/env python
"""bench.py — SVC inference throughput (audio samples/s) on N B200s of one node.

Workload (BASELINE.json configs[3], the configuration the 1->8 GPU metric is quoted on): full
SynthesizerInfer — NSF source + prior encoder + reverse flow + NSF-BigVGAN generator — on a batch
of 32 synthetic 10 s utterances (T=1000 frames -> 320,000 samples each) PER GPU (weak scaling:
utterances shard across ranks, no data-path collective).  A step = one pass of that hot path
over one batch.  Seeded synthetic weights in the reference checkpoint format (no pretrained
weights exist offline), synthetic inputs per SURVEY.md §8d.

  value : whole-job samples/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e   : same metric through the public SynthesizerInfer API with HOST pinned inputs
          (H2D of ppg/vec/pit/spk/lengths and D2H of the waveform inside the timed region)
  roofline / cpu_baseline : see DESIGN.md §Measurement

The same JSON line carries three sub-records under "configs" (N=1 only) so that every BASELINE
configuration is visible to a driver that only runs `python bench.py --gpus N`:
  configs.generator : BASELINE configs[1]  NSF-BigVGAN generator forward, 80-ch x 864 latent, batch 8, 24 kHz label
  configs.whisper   : BASELINE configs[2]  truncated Whisper large-v2 encoder, 16 x 30 s log-mel
  configs.hubert    : SURVEY 8f-2 (no BASELINE config)  HuBERT-Soft units, 16 x 20 s of 16 kHz audio
each with its own value / e2e / roofline / cpu_baseline.

`--impl reference` times the reference's own CPU algorithm on the host cores: the unmodified
reference modules when an install exists under baseline/_ref (kind "reference"), else the oracle
restatement (kind "port"; checked bit-exact against the imported reference — the Python reference
itself cannot travel to the GPU box).  Each step is a bounded sample of the headline workload: one
10 s utterance (T=1000) of the 32.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "audio samples/sec (SVC infer: F0+PPG+vec+spk -> waveform)"
UNIT = "samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="utterances per GPU per step")
    ap.add_argument("--frames", type=int, default=1000, help="frames per utterance (100 fps)")
    ap.add_argument("--precision", type=int, default=3, help="3 bf16x3 tensor-core (parity grade, default), 1 bf16, 0 fp32 CUDA cores")
    ap.add_argument("--workload", default="svc", choices=["svc", "whisper", "hubert"],
                    help="svc = BASELINE configs[3] (headline); whisper = configs[2] PPG extraction, 16 x 30 s log-mel")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subconfigs", action="store_true", help="skip the configs[1] / configs[2] sub-records")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy "
                         "(float32; rank 0's shard when several GPUs run), so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has nothing to dump")
    return args


DUMP_BYTES = 63_000_000   # all dumped arrays together, kept under 64 MB with the .npy headers


def dump_outputs(dirname, arrays):
    """Write each tensor of `arrays` as <dirname>/<name>.npy in float32.  When together they exceed DUMP_BYTES,
    each is replaced by tests.util.seeded_sample of its share of that budget: the same positions on every run."""
    from tests.util import seeded_sample
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if total > DUMP_BYTES:
            a = seeded_sample(a, a.numel() * DUMP_BYTES // total)
        np.save(os.path.join(dirname, name + ".npy"), a.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]),
                    tf_sust=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_threads() -> int:
    """Threads for the CPU arm.  torch's intra-op pool over-subscribes badly on the many tiny
    depthwise convolutions of this path: on the 128-core GPU-box host 128 threads ran 60x slower
    than 8 (gpurun_out of round 1), so the arm uses the count that is fastest in practice, capped
    by what the box has; SVCB_CPU_THREADS overrides."""
    env = os.environ.get("SVCB_CPU_THREADS")
    if env:
        return max(1, int(env))
    return max(1, min(os.cpu_count() or 1, 16))


def synth_inputs(hp, B, T, seed):
    from tests.util import make_inputs
    return make_inputs(seed, B, T, hp)


# ------------------------------------------------------------------------------ reference arm
HEADLINE_WORKLOAD = ("BASELINE configs[3]: full SynthesizerInfer (F0->NSF source, prior, flow, generator), "
                     "{B} x {S:.0f} s utterances per GPU per step, 32 kHz/hop 320")


def headline_config(B, T, L, world):
    """Identical for both arms (the driver compares the two lines' `config`)."""
    return {"workload": HEADLINE_WORKLOAD.format(B=B, S=T / 100), "batch_per_gpu": B, "frames": T,
            "samples_per_item": L, "parallelism": f"utterance-shard x{world}"}


def installed_reference(hp, sd):
    """The unmodified reference from a driver-side install under baseline/_ref, if one exists (the
    reference has no setup.py / pyproject, so `pip install --target baseline/_ref /root/reference`
    has nothing to build: DESIGN.md §9).  Returns a callable running pitch2source + inference, or None."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref_root, "vits", "models.py")):
        return None
    try:
        sys.path.insert(0, ref_root)
        from vits.models import SynthesizerInfer  # noqa
        from oracle.ref_import import to_attr
        m = SynthesizerInfer(hp.data.filter_length // 2 + 1, hp.data.segment_size // hp.data.hop_length, to_attr(hp)).eval()
        m.load_state_dict(sd)

        def run(d):
            with torch.no_grad():
                src = m.pitch2source(d["pit"])
                return m.inference(d["ppg"], d["vec"], d["pit"], d["spk"], d["ppg_l"], src)
        return run
    except Exception as e:  # a broken install must not take the arm down: fall back to the port
        print(f"baseline/_ref present but unusable ({e}); using the oracle port", file=sys.stderr)
        return None


def cpu_reference_run(hp, sd, T, repeats, ref_fn=None):
    """The reference's CPU algorithm on one utterance of T frames; returns best seconds."""
    from oracle import svc_oracle as O
    d = synth_inputs(hp, 1, T, 4242)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        if ref_fn is not None:
            ref_fn(d)
        else:
            with torch.no_grad():
                src = O.pitch2source(sd, hp, d["pit"], d["rand_ini"], d["noise"])
                O.synthesizer_infer(sd, hp, d["ppg"], d["vec"], d["pit"], d["spk"], d["ppg_l"], src, d["eps"])
        best = min(best, time.perf_counter() - t0)
    return best


def run_reference(args, hp, sd):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    ref_fn = installed_reference(hp, sd)
    kind = "reference" if ref_fn is not None else "port"
    T = args.frames  # one utterance of the headline workload per step (same item size as our arm)
    hop = int(np.prod(list(hp.gen.upsample_rates)))
    for _ in range(max(min(args.warmup, 2), 1)):
        cpu_reference_run(hp, sd, T, 1, ref_fn)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_run(hp, sd, T, 1, ref_fn)
    dt = time.perf_counter() - t0
    val = args.steps * T * hop / dt
    sample = (f"{args.steps} steps x ONE {T / 100:.0f} s utterance of the {args.batch} per step (bounded sample; CPU throughput "
              f"per sample is batch-independent, BASELINE.md §4), torch CPU fp32, {cores} threads, "
              + ("unmodified reference modules from baseline/_ref" if ref_fn else "oracle port of the reference CPU path"))
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded weights + inputs)",
        "config": headline_config(args.batch, T, T * hop, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------ roofline bookkeeping
FP32_PEAK_TF = 148 * 128 * 2 * 1.965e9 / 1e12   # 148 SMs x 128 FMA lanes x 2 FLOP x max SM clock (nominal; no measured figure)


def kernel_families(rep: str, steps: int):
    """svcb_timing_report() -> rows per kernel family (launch shapes of one kernel merged)."""
    import re
    fam = {}
    for line in rep.strip().splitlines():
        f = line.split()
        nm, n, tms, fl, by = f[:5]
        aux = float(f[5]) if len(f) > 5 else 0.0
        # launches of one kernel with different shapes are tagged _c<ch>k<taps> / _<cin>to<cout>_...: one family
        key = re.sub(r"(_c\d+(k\d+)?(r\d+)?|_\d+to\d+_k\d+_o\d+)$", "", nm)
        a = fam.setdefault(key, dict(name=key, launches=0, ms=0.0, flops=0.0, bytes=0.0, aux=0.0))
        a["launches"] += int(n); a["ms"] += float(tms); a["flops"] += float(fl); a["bytes"] += float(by); a["aux"] += aux
    rows = sorted(fam.values(), key=lambda r: -r["ms"])
    tot = sum(r["ms"] for r in rows) or 1.0
    table = [dict(name=r["name"], launches=r["launches"], share=round(r["ms"] / tot, 4),
                  ms_per_step=round(r["ms"] / steps, 3),
                  tflops=round(r["flops"] / (r["ms"] * 1e-3) / 1e12, 2) if r["ms"] else 0.0,
                  gbs=round(r["bytes"] / (r["ms"] * 1e-3) / 1e9, 1) if r["ms"] else 0.0) for r in rows]
    return rows, table, tot


def roofline_of(top, tot_ms, steps, peaks):
    """Roofline record of the dominant kernel family.  `flops` booked by the kernels are SURVEY.md §8(d)
    algorithmic FLOPs (2*Cin*Cout*k*L per conv; attention / GEMM products) — activation work (Snake,
    softmax) is booked separately as `aux` and never enters `achieved`.  Tensor-core kernels are held
    against the measured sustained bf16 peak; CUDA-core kernels above the fp32 ridge against the fp32
    FMA peak (nominal, stated) with the tensor fraction beside it; the rest against copy bandwidth."""
    dur = top["ms"] * 1e-3
    intensity = top["flops"] / max(top["bytes"], 1.0)
    tensor = any(t in top["name"] for t in ("tc", "gemm", "attn", "s2d"))
    ach_tf = top["flops"] / dur / 1e12
    if tensor and intensity > 0.1 * peaks["tf_sust"] * 1e12 / (peaks["hbm"] * 1e9):
        roof = {"kernel": top["name"], "bound": "tensor", "achieved": ach_tf, "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                "frac": ach_tf / peaks["tf_sust"]}
    elif not tensor and intensity > FP32_PEAK_TF * 1e12 / (peaks["hbm"] * 1e9):
        roof = {"kernel": top["name"], "bound": "fp32", "achieved": ach_tf, "peak": FP32_PEAK_TF, "unit": "TFLOP/s",
                "frac": ach_tf / FP32_PEAK_TF, "frac_of_tensor_peak": ach_tf / peaks["tf_sust"],
                "note": "CUDA-core (FFMA) kernel: peak = 148 SMs x 128 lanes x 2 x 1.965 GHz, nominal"}
    else:
        ach = top["bytes"] / dur / 1e9
        roof = {"kernel": top["name"], "bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                "frac": ach / peaks["hbm"]}
    roof["traffic"] = None
    try:  # measured DRAM traffic of this family (ncu --set full capture committed under profiles/)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as tf:
            tr = json.load(tf).get(top["name"])
        if tr:
            roof["traffic"] = tr["bytes_per_launch"]
            roof["traffic_unit"] = "bytes per launch (dram read+write, " + tr["source"] + ")"
    except (OSError, ValueError, KeyError):
        pass
    roof["algorithmic_bytes_per_launch"] = round(top["bytes"] / max(top["launches"], 1))
    roof["flops_survey_per_launch"] = round(top["flops"] / max(top["launches"], 1))
    if top.get("aux"):
        roof["flops_incl_activation_per_launch"] = round((top["flops"] + top["aux"]) / max(top["launches"], 1))
    roof["intensity_flop_per_byte"] = round(intensity, 1)
    roof["peak_source"] = f"of {peaks['src']} (MEASURED_PEAKS.json sustained bf16 / copy bandwidth)"
    roof["how"] = (f"CUDA events around every launch of this kernel over {steps} steps identical to the timed region "
                   "(svcb_timing_enable); achieved = summed SURVEY §8(d) FLOPs (or bytes) / summed duration")
    roof["launches_per_step"] = top["launches"] // steps
    roof["share_of_step"] = round(top["ms"] / tot_ms, 4)
    return roof


def timed_region(fn, steps, warmup, dev):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return float(e0.elapsed_time(e1))


class E2EPipeline:
    """End-to-end loop through the public API with HOST buffers: every step copies its inputs from pinned
    host memory and its result back, but the copies run on their own streams with two buffer sets, so
    step i+1's H2D and step i-1's D2H overlap step i's kernels (what a serving loop does).  All K H2D
    and K D2H copies complete inside the timed region."""

    def __init__(self, dev, host_inputs: dict, out_shape, compute):
        self.dev, self.host, self.compute = dev, host_inputs, compute
        self.cs, self.os = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.dbuf = [{k: torch.empty_like(v, device=dev) for k, v in host_inputs.items()} for _ in range(2)]
        self.out_host = [torch.empty(out_shape, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.h2d = sum(v.numel() * v.element_size() for v in host_inputs.values())
        self.d2h = self.out_host[0].numel() * 4

    def _prefetch(self, i, free):
        j = i & 1
        with torch.cuda.stream(self.cs):
            if free[j] is not None:
                self.cs.wait_event(free[j])
            for k, v in self.host.items():
                self.dbuf[j][k].copy_(v, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.cs)
        return ev

    def run(self, steps):
        cur = torch.cuda.current_stream(self.dev)
        free = [None, None]
        out_free = [None, None]
        ready = self._prefetch(0, free)
        for i in range(steps):
            j = i & 1
            cur.wait_event(ready)
            if i + 1 < steps:
                ready = self._prefetch(i + 1, free)
            w = self.compute(self.dbuf[j])
            done = torch.cuda.Event()
            done.record(cur)
            free[j] = done
            with torch.cuda.stream(self.os):
                self.os.wait_event(done)
                self.out_host[j].copy_(w, non_blocking=True)
            w.record_stream(self.os)
        cur.wait_stream(self.os)


# ------------------------------------------------------------------------------ our arm
def run_ours(args, hp, sd):
    from whisper_vits_svc_b200 import _lib, models, shard

    rank, local, world = shard.init()
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs CUDA devices; there is no CPU path"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    B, T = args.batch, args.frames
    hop = int(np.prod(list(hp.gen.upsample_rates)))
    L = T * hop

    m = models.SynthesizerInfer(hp.data.filter_length // 2 + 1, hp.data.segment_size // hp.data.hop_length, hp,
                                precision=args.precision)
    if world == 1:
        m.load_state_dict(sd)
        m.to(dev)
        m._ensure()
    else:  # rank 0 packs, one NCCL broadcast of the packed blob (SURVEY.md §8e)
        blob = table = None
        if rank == 0:
            m.load_state_dict(sd)
            m.to(dev)
            blob, table = m.packed_blob()
        else:
            m.to(dev)
        blob, table = shard.broadcast_blob(blob, table, dev)
        if rank != 0:
            m.install_blob(blob, table)

    d = synth_inputs(hp, B, T, 1000 + rank)
    dv = {k: v.to(dev) for k, v in d.items()}
    host = {k: d[k].pin_memory() for k in ("ppg", "vec", "pit", "spk", "ppg_l")}
    launches = [0]

    def step_device():
        src = m.pitch2source(dv["pit"], rand_ini=dv["rand_ini"], noise=dv["noise"])
        launches[0] += _lib.last_launch_count()
        w = m.inference(dv["ppg"], dv["vec"], dv["pit"], dv["spk"], dv["ppg_l"], src, eps=dv["eps"])
        launches[0] += _lib.last_launch_count()
        return w

    def compute_e2e(x):
        src = m.pitch2source(x["pit"])  # device-side RNG draws, as the reference does on its device
        return m.inference(x["ppg"], x["vec"], x["pit"], x["spk"], x["ppg_l"], src)

    pipe = E2EPipeline(dev, host, (B, 1, L), compute_e2e)

    def timed(loop, steps, warmup, sampler=None):
        loop(warmup)
        torch.cuda.synchronize(dev)
        shard.barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches[0] = 0
        e0.record()
        loop(steps)
        e1.record()
        torch.cuda.synchronize(dev)
        shard.barrier()
        clocks = sampler.stop() if sampler else None
        ms = shard.max_over_ranks(float(e0.elapsed_time(e1)), dev)
        return ms, clocks

    last = {}

    def device_loop(n):
        for _ in range(n):
            last["wave"] = step_device()

    sampler = ClockSampler(local) if rank == 0 else None
    ms, clocks = timed(device_loop, args.steps, args.warmup, sampler)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    del last
    n_launch = launches[0]
    total_samples = float(world * B * L * args.steps)
    value = total_samples / (ms * 1e-3)
    ms_e2e, _ = timed(pipe.run, args.steps, max(1, min(args.warmup, 2)))
    e2e_value = total_samples / (ms_e2e * 1e-3)

    roof, kernels = None, None
    peaks = load_peaks()
    if rank == 0 and not args.no_roofline:
        lib.svcb_timing_enable(1)
        for _ in range(args.steps):
            step_device()
        torch.cuda.synchronize(dev)
        rep = lib.svcb_timing_report().decode()
        lib.svcb_timing_enable(0)
        if os.environ.get("SVCB_DUMP_KERNELS"):
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", "kernels_raw.txt"), "w") as f:
                f.write(rep)
        rows, kernels, tot = kernel_families(rep, args.steps)
        roof = roofline_of(rows[0], tot, args.steps, peaks)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        torch.set_num_threads(cores)
        Tc = 250
        cpu_reference_run(hp, sd, 50, 1)  # warm-up of the oneDNN primitives
        sec = cpu_reference_run(hp, sd, Tc, 2)
        cpu = {"value": Tc * hop / sec, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"best of 2 x one {Tc / 100:.1f} s utterance (same per-item workload), oracle port of the "
                         f"reference CPU path, torch fp32, {cores} threads, {sec:.2f} s"}

    sub = None
    if rank == 0 and world == 1 and not args.no_subconfigs:
        del dv, pipe
        torch.cuda.empty_cache()
        sub = {}
        for name, fn in (("generator", lambda: bench_generator(args, hp, dev, lib, peaks)),
                         ("whisper", lambda: bench_whisper(args, dev, lib, peaks)),
                         ("hubert", lambda: bench_hubert(args, dev, lib, peaks))):
            try:
                sub[name] = fn()
            except Exception as e:  # a sub-record must never take the headline down
                sub[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    if rank == 0:
        step_s = ms * 1e-3 / args.steps
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {0: "f32", 1: "bf16", 3: "bf16x3 (bf16 operands split 3-way, fp32 accumulate) + f32"}[args.precision],
            "data": "synthetic (seeded weights in the reference checkpoint format + seeded inputs)",
            "config": headline_config(B, T, L, world),
            "timing": {"cache": "inputs (ppg+vec+noise+eps ~ %.0f MB per step) exceed the 126 MB L2" % (
                           (d["ppg"].numel() + d["vec"].numel() + d["noise"].numel() + d["eps"].numel()) * 4 / 1e6),
                       "rtf_32k": step_s / (world * B * L / 32000.0), "rtf_24k_label": step_s / (world * B * L / 24000.0)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": pipe_h2d(host), "d2h_bytes_per_step": B * L * 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "how": "pinned host inputs -> H2D -> pitch2source + inference -> D2H of the waveform, every step; copies on "
                           "side streams with two buffer sets overlap the neighbouring steps' kernels"},
            "gpu_launches": n_launch,
            "clocks": clocks,
        }
        if roof:
            out["roofline"] = roof
            out["kernels"] = kernels
        if cpu:
            out["cpu_baseline"] = cpu
        if sub:
            out["configs"] = sub
        print(json.dumps(out), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def pipe_h2d(host):
    return sum(v.numel() * v.element_size() for v in host.values())


def bench_generator(args, hp, dev, lib, peaks):
    """BASELINE configs[1]: NSF-BigVGAN generator forward only — random 80-ch x 864 latent -> wave, batch 8
    (`Generator.inference(spk, x, har_source)`, vits_decoder/generator.py:175-200) with the 80-channel /
    24 kHz-label override of SURVEY.md §8d config 2."""
    from tests.util import make_inputs
    from whisper_vits_svc_b200 import hparams, models, synth
    hp24 = hparams.override(hp, gen__upsample_input=80, data__sampling_rate=24000)
    sd24 = synth.svc_state_dict(hp24, 1234)
    m = models.SynthesizerInfer(hp24.data.filter_length // 2 + 1, hp24.data.segment_size // hp24.data.hop_length, hp24,
                                precision=args.precision)
    m.load_state_dict(sd24)
    m.to(dev)
    m._ensure()
    B, T = 8, 864
    hop = int(np.prod(list(hp24.gen.upsample_rates)))
    L = T * hop
    d = make_inputs(0, B, T, hp24, gen_only=True)
    dv = {k: v.to(dev) for k, v in d.items()}
    src = m.pitch2source(dv["pit"], rand_ini=dv["rand_ini"], noise=dv["noise"])
    steps, warm = args.steps, max(args.warmup, 3)
    flush = torch.empty(160 * 1024 * 1024 // 4, device=dev)   # > L2: inputs (3.5 MB) would otherwise stay cached

    def step():
        flush.zero_()
        return m.generator(dv["spk"], dv["z"], src)

    def flush_only():
        flush.zero_()

    ms_all = timed_region(step, steps, warm, dev) / steps
    ms_flush = timed_region(flush_only, steps, 1, dev) / steps
    ms = ms_all - ms_flush
    host = {"spk": d["spk"].pin_memory(), "z": d["z"].pin_memory(), "source": src.cpu().pin_memory()}
    pipe = E2EPipeline(dev, host, (B, 1, L), lambda x: m.generator(x["spk"], x["z"], x["source"]))
    pipe.run(2)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); pipe.run(steps); e1.record(); torch.cuda.synchronize(dev)
    ms_e2e = e0.elapsed_time(e1) / steps
    lib.svcb_timing_enable(1)
    for _ in range(steps):
        m.generator(dv["spk"], dv["z"], src)
    torch.cuda.synchronize(dev)
    rep = lib.svcb_timing_report().decode(); lib.svcb_timing_enable(0)
    rows, table, tot = kernel_families(rep, steps)
    out = {"metric": "audio samples/sec (NSF-BigVGAN generator forward)", "value": B * L / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms, "config": {"workload": "BASELINE configs[1]: Generator.inference, latent [8, 80, 864] + source -> wave "
                                         "[8, 1, 276480], 24 kHz label (80-channel override)", "batch": B, "frames": T,
                                         "cache": "L2 flushed (160 MB memset) between steps; its time is subtracted"},
           "gflop_per_step_survey": 944.0, "tflops_model": 944e9 / (ms * 1e-3) / 1e12,
           "e2e": {"value": B * L / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": pipe.h2d,
                   "d2h_bytes_per_step": pipe.d2h},
           "roofline": roofline_of(rows[0], tot, steps, peaks), "kernels": table[:8]}
    if not args.no_cpu_baseline:
        from oracle import svc_oracle as O
        cores = cpu_threads()
        torch.set_num_threads(cores)
        Tc = 216
        dc = make_inputs(1, 1, Tc, hp24, gen_only=True)
        src_c = O.pitch2source(sd24, hp24, dc["pit"], dc["rand_ini"], dc["noise"])
        best = float("inf")
        for _ in range(2):
            t0 = time.perf_counter()
            with torch.no_grad():
                O.generator(sd24, hp24, dc["spk"], dc["z"], src_c)
            best = min(best, time.perf_counter() - t0)
        out["cpu_baseline"] = {"value": Tc * hop / best, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": f"best of 2 x one [1, 80, {Tc}] latent (a quarter-length item), oracle port of "
                                         f"Generator.inference, torch fp32, {cores} threads, {best:.2f} s"}
    return out


def bench_whisper(args, dev, lib, peaks, dump=None):
    """BASELINE configs[2]: truncated Whisper large-v2 encoder (24 blocks), 16 x 30 s log-mel per step.
    `dump`, when given, receives the PPG of the last timed step under "ppg"."""
    from whisper_vits_svc_b200 import synth, whisper_infer
    ck = synth.whisper_checkpoint(seed=1234)
    enc = whisper_infer.WhisperB200(ck, dev).encoder
    B, n = 16, 3000
    steps = args.steps
    g = torch.Generator().manual_seed(0)
    mel = torch.randn(B, 80, n, generator=g).clamp(-1, 1.5)
    mel_d = mel.to(dev)
    last = {} if dump is None else dump
    ms = timed_region(lambda: last.update(ppg=enc(mel_d)), steps, max(args.warmup, 3), dev) / steps
    del last
    pipe = E2EPipeline(dev, {"mel": mel.pin_memory()}, (B, 1500, 1280), lambda x: enc(x["mel"]))
    pipe.run(1)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); pipe.run(steps); e1.record(); torch.cuda.synchronize(dev)
    ms_e2e = e0.elapsed_time(e1) / steps
    # front end on the device (SURVEY.md §8f-1): 16 x 30 s of 16 kHz audio -> log-mel (+ the extractor's
    # noise term) -> encoder; `from_audio` = pinned host audio in, PPG back on the host
    audio = (torch.randn(B, n * 160, generator=g) * 0.1)
    noise_d = torch.randn(B, 80, n, generator=g).to(dev)
    audio_d = audio.to(dev)
    ms_fe = timed_region(lambda: enc.log_mel(audio_d, noise_d, 0.1), steps, 2, dev) / steps
    pipe_a = E2EPipeline(dev, {"audio": audio.pin_memory()}, (B, 1500, 1280), lambda x: enc(enc.log_mel(x["audio"], noise_d, 0.1)))
    pipe_a.run(1)
    torch.cuda.synchronize(dev)
    e0.record(); pipe_a.run(steps); e1.record(); torch.cuda.synchronize(dev)
    ms_audio = e0.elapsed_time(e1) / steps
    lib.svcb_timing_enable(1)
    for _ in range(steps):
        enc(enc.log_mel(audio_d, noise_d, 0.1))
    torch.cuda.synchronize(dev)
    rep = lib.svcb_timing_report().decode(); lib.svcb_timing_enable(0)
    rows, table, tot = kernel_families(rep, steps)
    flops = 1708.6e9 * B
    audio_s = 30.0 * B
    out = {"metric": "audio seconds/sec (Whisper-large-v2 truncated encoder, PPG extraction)", "value": audio_s / (ms * 1e-3),
           "unit": "audio s/s", "ms_per_step": ms, "dtype": "bf16",
           "config": {"workload": "BASELINE configs[2]: 16 x 30 s log-mel [16,80,3000] -> PPG [16,1500,1280], 24 blocks",
                      "tflops_model": flops / (ms * 1e-3) / 1e12,
                      "cache": "weights (955 MB bf16) + activations exceed the 126 MB L2"},
           "e2e": {"value": audio_s / (ms_e2e * 1e-3), "unit": "audio s/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": pipe.h2d, "d2h_bytes_per_step": pipe.d2h},
           "frontend": {"what": "svcb_whisper_log_mel: [16, 480000] audio -> [16, 80, 3000] log-mel + noise, on the device",
                        "ms_per_step": ms_fe, "audio_s_per_s": audio_s / (ms_fe * 1e-3)},
           "from_audio": {"what": "pinned host audio -> log-mel -> encoder -> PPG on the host", "ms_per_step": ms_audio,
                          "value": audio_s / (ms_audio * 1e-3), "unit": "audio s/s",
                          "h2d_bytes_per_step": pipe_a.h2d, "d2h_bytes_per_step": pipe_a.d2h},
           "roofline": roofline_of(rows[0], tot, steps, peaks), "kernels": table[:8],
           "gpu_launches": int(sum(r["launches"] for r in rows))}
    del enc, pipe, pipe_a
    if not args.no_cpu_baseline:
        from oracle import whisper_oracle as WO
        cores = cpu_threads()
        torch.set_num_threads(cores)
        WO.audio_encoder(ck, mel[:1, :, :200])   # warm-up
        t0 = time.perf_counter()
        WO.audio_encoder(ck, mel[:1])
        sec = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 30.0 / sec, "unit": "audio s/s", "cores": cores, "kind": "port",
                               "sample": f"one 30 s item (1 of the 16), oracle port of AudioEncoder.forward, torch fp32, "
                                         f"{cores} threads, {sec:.1f} s"}
    return out


def bench_hubert(args, dev, lib, peaks, dump=None):
    """SURVEY.md §8f-2 (not a BASELINE config): HuBERT-Soft units, 16 x 20 s chunks of 16 kHz audio per step
    (hubert/inference.py:30-33 chunk size) -> [16, 1000, 256].  `dump`, when given, receives the units of the
    last timed step under "units"."""
    from whisper_vits_svc_b200 import hubert_infer, synth
    sd = synth.hubert_checkpoint(1234)
    model = hubert_infer.HubertSoftB200(sd, dev)
    B, n = 16, 20 * 16000
    steps = args.steps
    g = torch.Generator().manual_seed(0)
    wav = torch.randn(B, n, generator=g) * 0.1
    wav_d = wav.to(dev)
    T = model.frames(n)
    last = {} if dump is None else dump
    ms = timed_region(lambda: last.update(units=model.units(wav_d)), steps, max(args.warmup, 3), dev) / steps
    del last
    pipe = E2EPipeline(dev, {"wav": wav.pin_memory()}, (B, T, 256), lambda x: model.units(x["wav"]))
    pipe.run(1)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); pipe.run(steps); e1.record(); torch.cuda.synchronize(dev)
    ms_e2e = e0.elapsed_time(e1) / steps
    lib.svcb_timing_enable(1)
    for _ in range(steps):
        model.units(wav_d)
    torch.cuda.synchronize(dev)
    rep = lib.svcb_timing_report().decode(); lib.svcb_timing_enable(0)
    rows, table, tot = kernel_families(rep, steps)
    audio_s = 20.0 * B
    # conv stem 2 * 512 * 512 * (3 * (32007 + 16003 + 8001 + 4000) + 2 * (2000 + 1000)) + conv0, pos conv, 12 layers, proj
    flops_item = (2 * 512 * 512 * (3 * 60011 + 2 * 3000) + 2 * 512 * 10 * 64015 + 2 * T * 768 * 48 * 128
                  + 2 * T * 512 * 768 + 12 * (2 * T * 768 * (2304 + 768 + 2 * 3072) + 4 * T * T * 768) + 2 * T * 768 * 256)
    out = {"metric": "audio seconds/sec (HuBERT-Soft units)", "value": audio_s / (ms * 1e-3), "unit": "audio s/s",
           "ms_per_step": ms, "dtype": "bf16 (tcgen05 GEMMs / attention, fp32 accumulate, fp32 residual stream); conv0 + GroupNorm f32",
           "config": {"workload": f"SURVEY 8f-2: 16 x 20 s of 16 kHz audio [16, 320000] -> units [16, {T}, 256], 12 layers",
                      "tflops_model": flops_item * B / (ms * 1e-3) / 1e12},
           "e2e": {"value": audio_s / (ms_e2e * 1e-3), "unit": "audio s/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": pipe.h2d, "d2h_bytes_per_step": pipe.d2h},
           "roofline": roofline_of(rows[0], tot, steps, peaks), "kernels": table[:8],
           "gpu_launches": int(sum(r["launches"] for r in rows))}
    del model, pipe
    if not args.no_cpu_baseline:
        from oracle import hubert_oracle as HO
        cores = cpu_threads()
        torch.set_num_threads(cores)
        HO.units(sd, wav[:1, None, :16000])   # warm-up
        t0 = time.perf_counter()
        HO.units(sd, wav[:1, None, :])
        sec = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 20.0 / sec, "unit": "audio s/s", "cores": cores, "kind": "port",
                               "sample": f"one 20 s chunk (1 of the 16), oracle port of HubertSoft.units, torch fp32, "
                                         f"{cores} threads, {sec:.1f} s"}
    return out


def run_whisper(args):
    from whisper_vits_svc_b200 import _lib
    assert torch.cuda.is_available()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dump = {}
    out = (bench_hubert if args.workload == "hubert" else bench_whisper)(args, dev, _lib.load(), load_peaks(), dump)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dump)
    out.update({"n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "data": "synthetic"})
    print(json.dumps(out), flush=True)


def main():
    args = parse()
    if args.workload in ("whisper", "hubert"):
        return run_whisper(args)
    from whisper_vits_svc_b200 import hparams, synth
    hp = hparams.load_hparams(os.path.join(ROOT, "configs", "base.yaml"))
    sd = synth.svc_state_dict(hp, 1234)
    if args.impl == "reference":
        run_reference(args, hp, sd)
    else:
        run_ours(args, hp, sd)


if __name__ == "__main__":
    main()
