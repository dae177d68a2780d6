#!/usr/bin/env python
"""bench.py — throughput of the VITS acoustic+vocoder hot path (SummerTTS SynthesizerTrn::infer NN half).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU implementation

Metric (BASELINE.json): audio samples/s (and RTF) on single_speaker_fast.  One "step" = one pass of
the whole hot path over one batch of synthetic utterances (default: 64 utterances x 128 phoneme ids
per GPU, 5 frames per id forced => 163 840 samples per utterance; weak scaling).
  value : samples/s with the ids already resident in HBM when the timed region starts (PCM left in HBM)
  e2e   : the same batch through the C ABI call stts_infer_batch_into with pinned HOST buffers —
          H2D of ids and D2H of the PCM inside the timed region
Timing: CUDA events on the engine's stream, barrier + synchronize on both sides, max over ranks.
L2 is flushed (256 MiB write) before every timed step.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes what the last timed `value` step computed, for comparing two builds output for output:
DIR/pcm.npy (the batch's int16 PCM as float32) and DIR/sample_offsets.npy (float64, utterance b is
pcm[so[b]:so[b+1]]); under torchrun each rank adds a _rank<r> suffix.  The inputs are seeded, so the
same arguments give the same inputs on every run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 16000


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def model_path(name):
    for d in (os.environ.get("STTS_MODEL_DIR", ""), os.path.join(ROOT, "oracle", "_ref", "models"),
              "/root/reference/models"):
        if not d:
            continue
        for fn in (name + ".nn.bin", name + ".bin"):
            p = os.path.join(d, fn)
            if os.path.exists(p):
                return p
    return None


def get_model(name):
    """Shipped weights if they travelled, else random-init weights of the same architecture."""
    from summertts_b200 import binfmt

    p = model_path(name)
    if p:
        return np.fromfile(p, dtype=np.float32), "shipped", p
    blob = binfmt.synthetic_model(seed=11, **binfmt.ARCH[name])
    p = os.path.join(tempfile.gettempdir(), "stts_%s_random_init_%d.bin" % (name, os.getuid()))   # per user: /tmp may be shared
    blob.tofile(p)
    return blob, "random-init", p


def make_utts(first, count, n_ids, vocab):
    """BASELINE config-5 style synthetic phoneme sequences, seeded per GLOBAL utterance index."""
    from parity_util import synth_ids

    return [synth_ids(np.random.default_rng(1234 + first + i), n_ids, vocab) for i in range(count)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = str(gpu_index)
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8 and f[0] == self.idx:
                self.rows.append(f)

    def stop(self):
        if self.p:
            self.p.terminate()
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = []
        for k, name in ((4, "hw_slowdown"), (5, "hw_thermal_slowdown"), (6, "sw_thermal_slowdown"), (7, "sw_power_cap")):
            if any(r[k].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def host_cores():
    """Cores this process may really use: sched affinity ∩ the cgroup CPU quota (cpu.max / cfs_quota).
    os.cpu_count() reports the box's cores even inside a cgroup-limited lease (round 1: 128 'cores' that
    were a small slice -> 5x box-to-box swing of the reference arm)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:  # noqa: BLE001
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:  # noqa: BLE001
            pass
    if quota:
        n = min(n, max(1, int(quota + 0.5)))
    return max(1, n)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:  # noqa: BLE001
        pass
    return "unknown"


def run_cpu_best(model_file, n_ids, vocab, forced_per_id, cores, reps, warm_reps):
    """Sweep the worker count over {cores/2, cores} (SMT siblings / memory bandwidth can make half the
    logical cores faster) and keep the best whole-box throughput.  Returns (samples/s, workers, seconds, table)."""
    best = None
    table = {}
    for w in sorted({max(1, cores // 2), cores}):
        samples, sec = run_cpu(model_file, 1, n_ids, vocab, forced_per_id, w, reps, warm_reps)
        table[str(w)] = samples / sec
        if best is None or samples / sec > best[0]:
            best = (samples / sec, w, sec)
    return best[0], best[1], best[2], table


DUMP_LIMIT = 64 << 20     # bytes of .npy data per --dump-outputs directory, all ranks together


def dump_outputs(d, pcm, sample_offsets, suffix, budget):
    """Write one step's outputs as DIR/<name><suffix>.npy.  A PCM over `budget` bytes is cut to a fixed,
    seeded sample of its positions, written as pcm_index (float64) beside the sampled pcm."""
    os.makedirs(d, exist_ok=True)
    out = {"sample_offsets": sample_offsets.astype(np.float64), "pcm": pcm.astype(np.float32)}
    room = budget - out["sample_offsets"].nbytes - 3 * 128      # 128: .npy header
    if out["pcm"].nbytes > room:
        idx = np.sort(np.random.default_rng(0).choice(pcm.size, room // 12, replace=False))
        out["pcm_index"], out["pcm"] = idx.astype(np.float64), out["pcm"][idx]
    for name, a in out.items():
        np.save(os.path.join(d, name + suffix + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1435.1), d.get("hbm_gbs", 6574.1), "measured"
    return 1400.0, 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation (oracle/_ref) on host cores
# ------------------------------------------------------------------------------------------------
def run_cpu(model_file, utts_per_worker, n_ids, vocab, forced_per_id, workers, reps, warm_reps):
    """`workers` single-threaded processes (the reference's Eigen path parallelises only its GEMMs, so
    independent single-thread processes are its best use of the host cores), each synthesising
    `utts_per_worker` utterances per rep.  Returns (samples, seconds) over the timed reps."""
    start_at = time.time() + 8.0 + 0.05 * workers
    procs = []
    for w in range(workers):
        utts = make_utts(100000 + w * utts_per_worker, utts_per_worker, n_ids, vocab)
        spec = {"model": model_file, "utts": utts, "threads": 1, "reps": reps + warm_reps, "start_at": start_at,
                "forced": None if forced_per_id is None else [[float(forced_per_id)] * n_ids for _ in utts]}
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "cpu_worker_steps.py"), json.dumps(spec)],
                                      stdout=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        o, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("cpu worker failed")
        outs.append(json.loads(o.strip().splitlines()[-1]))
    t0 = min(o["t0"][warm_reps] for o in outs)
    t1 = max(o["t1"][-1] for o in outs)
    samples = sum(sum(o["samples"][warm_reps:]) for o in outs)
    return samples, t1 - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="single_speaker_fast")
    ap.add_argument("--batch", type=int, default=64, help="utterances per GPU per step")
    ap.add_argument("--ids", type=int, default=128, help="phoneme ids per utterance")
    ap.add_argument("--durations", default="forced5", choices=["forced5", "model"])
    ap.add_argument("--tensor", type=int, default=-1, help="-1 library default (1), 0 fp32 FFMA tiles only, 1 tcgen05 split-fp16 "
                    "(fp32-accurate), 2 tcgen05 throughput mode (one fp16 MMA per K-step)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch utterances per GPU; strong: --batch utterances in total, split over the ranks (BASELINE config 5)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the PCM and sample offsets of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncpu = host_cores()

    if args.scaling == "strong":
        if args.batch % world:
            raise SystemExit("--scaling strong needs --batch divisible by the number of ranks")
        args.batch //= world
    blob, wkind, mfile = get_model(args.model)
    from summertts_b200 import binfmt

    M = binfmt.parse_model(blob)
    vocab = M["enc"]["vocab"]
    forced_per_id = 5 if (args.durations == "forced5" or wkind != "shipped") else None
    workload = "%s (%s weights), %d utterances x %d synthetic phoneme ids per GPU, %s" % (
        args.model, wkind, args.batch, args.ids,
        "forced 5 frames/id (163840 samples/utt)" if forced_per_id else "model-predicted durations")
    tmode = 1 if args.tensor < 0 else args.tensor
    dtype = {0: "f32", 1: "f32", 2: "f16"}[tmode]
    config = {"workload": workload, "batch_per_gpu": args.batch, "ids_per_utt": args.ids,
              "arithmetic": {0: "fp32 FFMA tiles", 1: "split-fp16 tcgen05 MMAs (3 per K-step), fp32 accumulate + fp32 promotion: fp32-accurate",
                             2: "throughput mode: one fp16 tcgen05 MMA per K-step, fp32 accumulate"}[tmode],
              "durations": "forced5" if forced_per_id else "model", "l2": "flushed (256 MiB write) before every timed step",
              "parallelism": "replicas x%d, no collective" % world}

    # ---------------------------------------------------------------- reference arm (CPU) ----------
    if args.impl == "reference":
        if rank != 0:
            return 0
        v, workers, sec, table = run_cpu_best(mfile, args.ids, vocab, forced_per_id, ncpu, args.steps, args.warmup)
        line = {"impl": "reference", "metric": "audio_samples_per_sec", "value": v, "unit": "samples/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic ids; %s weights" % wkind, "config": config, "rtf": SR / v,
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": workers, "kind": "reference",
                                 "cores_allowed": ncpu, "cores_logical": os.cpu_count(), "cpu_model": cpu_model(),
                                 "sweep_samples_per_s": table,
                                 "sample": "each step = %d single-thread processes x 1 utterance of the workload "
                                           "(compiled unmodified reference objects, oracle/_ref); worker count swept "
                                           "over {allowed/2, allowed}, best kept" % workers},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- our arm (GPU) ----------------
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from summertts_b200 import build, engine

    build.build_native()
    E = engine.SynthesizerTrn(blob, device=local)
    if args.tensor >= 0:
        E.set_tensor_path(args.tensor)
    utts = make_utts(rank * args.batch, args.batch, args.ids, vocab)
    ids, offs = E._pack(utts)
    Tt = int(offs[-1])
    if forced_per_id:
        E.set_forced_durations(np.full(Tt, float(forced_per_id), np.float32))
    stream = torch.cuda.ExternalStream(E.stream(), device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """sum of per-step CUDA-event durations on the engine's stream; L2 flushed before each step"""
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            tot += a.elapsed_time(b)
        return tot

    # ---- value: inputs resident in HBM ---------------------------------------------------------
    E.stage(utts)
    S = 0
    for _ in range(args.warmup):
        S = E.run()
    sampler = ClockSampler(torch.cuda.current_device() if os.environ.get("CUDA_VISIBLE_DEVICES") is None else local)
    barrier()
    sampler.start()
    l0 = E.kernel_launches()
    ms = timed(E.run, args.steps)
    launches = E.kernel_launches() - l0
    barrier()
    stage_ms = E.last_timing()
    if args.dump_outputs:
        pcm, so = E.fetch(S, args.batch)
        dump_outputs(args.dump_outputs, pcm, so, "_rank%d" % rank if world > 1 else "", DUMP_LIMIT // world)

    # ---- e2e: host buffers through the C ABI ------------------------------------------------------
    h_ids = torch.from_numpy(ids).pin_memory().numpy()
    h_offs = torch.from_numpy(offs).pin_memory().numpy()
    h_pcm = torch.empty(S + 1024, dtype=torch.int16).pin_memory().numpy()
    h_soff = np.zeros(args.batch + 1, dtype=np.int64)

    def e2e_step():
        E.infer_batch_into(h_ids, h_offs, None, None, h_pcm, h_soff)

    for _ in range(2):
        e2e_step()
    barrier()
    ms_e2e = timed(e2e_step, args.steps)
    barrier()
    clocks = sampler.stop()

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    s = torch.tensor([float(S)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
    ms, ms_e2e = t.tolist()
    S_all = s.item()

    # ---- roofline of the dominant conv class (live, CUDA events around each launch) ---------------
    roof = None
    prof = {}
    if rank == 0:
        E.profile_enable(True)
        for _ in range(2):
            E.run()
        prof = E.profile_fetch()
        E.profile_enable(False)
        peak_tf, peak_gbs, how = peaks()
        dom = max(prof, key=lambda k: prof[k]["ms"])
        d = prof[dom]
        ach = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and args.model == "single_speaker_fast" and args.batch == 64 and args.ids == 128:
            tj = json.load(open(tp))        # ncu DRAM bytes per launch of the class, captured on the default workload
            traffic = tj.get("%s@t%d" % (dom, tmode), tj.get(dom) if tmode == 1 else None)
        roof = {"bound": "tensor", "kernel_class": dom, "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": ach / peak_tf, "traffic": traffic, "peak_source": how + " bf16 sustained",
                "avg_launch_ms": d["ms"] / max(d["launches"], 1),
                "algorithmic_flops_per_launch": d["flops"] / max(d["launches"], 1),
                "share_of_conv_time": d["ms"] / max(sum(v["ms"] for v in prof.values()), 1e-9)}
        if traffic:   # measured DRAM bytes per launch (ncu) over the live launch time: the class's HBM utilisation
            gbs = traffic / (roof["avg_launch_ms"] * 1e-3) / 1e9
            roof["hbm_view"] = {"achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
                                "note": "ncu dram bytes per launch / live launch time"}

    # ---- single-utterance latency (BASELINE config 2 shape), informational ------------------------
    single = None
    if rank == 0:
        from parity_util import TEST_TXT_IDS

        E.set_forced_durations(None)
        one = TEST_TXT_IDS if vocab >= 219 else make_utts(0, 1, 76, vocab)[0]
        E.stage([one])
        for _ in range(3):
            s1 = E.run()
        ms1 = timed(E.run, 10) / 10
        single = {"ids": len(one), "samples": s1, "ms": ms1, "rtf": (ms1 / 1e3) / (s1 / SR)}

    # ---- cpu_baseline beside it (rank 0, N=1 only; bounded sample) ---------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v_cpu, workers, sec, table = run_cpu_best(mfile, args.ids, vocab, forced_per_id, ncpu, 1, 0)
            cpu = {"value": v_cpu, "unit": "samples/s", "cores": workers, "kind": "reference",
                   "cores_allowed": ncpu, "cores_logical": os.cpu_count(), "cpu_model": cpu_model(),
                   "sweep_samples_per_s": table,
                   "sample": "%d utterances of the workload (one per worker, single-thread processes of the compiled "
                             "unmodified reference objects), %.1f s; worker count swept over {allowed/2, allowed}" % (workers, sec)}
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "error": str(ex)}

    if rank == 0:
        v = S_all * args.steps / (ms * 1e-3)
        ve = S_all * args.steps / (ms_e2e * 1e-3)
        line = {"metric": "audio_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": dtype, "data": "synthetic ids; %s weights" % wkind, "config": config,
                "clocks": clocks,
                "e2e": {"value": ve, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": int(ids.nbytes + offs.nbytes + 8 * args.batch + 8),
                        "d2h_bytes_per_step": int(2 * S + 4 * args.batch)},
                "gpu_launches": int(launches), "tensor_fallbacks": E.tensor_fallbacks(), "rtf": SR / v, "x_realtime_per_gpu": v / world / SR,
                "samples_per_step": S_all, "stage_ms_last_step": stage_ms, "roofline": roof,
                "conv_classes": {k: {"ms": round(x["ms"] / 2, 4), "tflops": (x["flops"] / (x["ms"] * 1e-3) / 1e12) if x["ms"] > 0 else 0,
                                     "launches": x["launches"] // 2} for k, x in prof.items() if x["launches"]},
                "single_utterance": single, "cpu_baseline": cpu, "library": engine.load_library().stts_version().decode()}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    E.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
