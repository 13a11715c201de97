#!/usr/bin/env python
"""bench.py -- throughput of the batched voice path on B200, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload svf|biquad|delay|mfcc] [--impl reference] [--dump-outputs DIR]

A "step" is one block (1024 frames) of one bank: BASELINE.json configs[1] by default -- 1 Mi voices of
maxiOsc::saw -> maxiSVF (low-pass mix), per-voice fp64 output materialised time-major in HBM. With N > 1
(launched by torch.distributed.run, one rank per GPU) every rank owns its own 1 Mi voices (weak scaling);
voices are independent, so the headline block has no collective at any N.

  value      voice-samples/s of the whole job, inputs and state resident in HBM, CUDA-event timed, max over ranks
  workloads  (N = 1, default run) the other BASELINE.json configurations measured the same way in the same run, each with
             its own value / roofline / e2e / cpu_baseline:  biquad_bank = configs[4]'s shard in bank mode (saw ->
             maxiBiquad, output materialised), delay = configs[2] (256 Ki voices saw -> ADSR -> 4096-tap delay line),
             mfcc = configs[3] (64 Ki channels FFT-1024 / hop 512 + 40 MFCCs, frames/s); modulated = configs[1]'s and configs[2]'s
             banks with a per-sample frequency array (FM; SURVEY.md 8(f) rank 1: +8 B read per voice-sample)
  mixdown    BASELINE.json configs[4] in "mix mode" (SURVEY.md 8(d) config 5), timed separately in the same run:
             1 Mi voices/GPU saw -> maxiBiquad -> maxiMix::stereo -> sum over voices, only the stereo bus is
             written; for N > 1 the bus is summed over the GPUs -- the path's only exchange step (--collective
             p2p: peer-memory exchange fused into the mix-reduce kernel; nccl: all_reduce). fp64-pipe bound,
             reported as such; `check` compares the exchanged bus with an NCCL all-reduce of the local buses.
             `--mix 1` instead adds the bus to the headline block (output AND bus).
  e2e        the same block through the C ABI with HOST control data, pipelined: per step one fp64 frequency array
             (8 MiB, pinned) goes up with mxb_bank_set_param_async (double-buffered, copy stream) and the stereo mix
             (16 KiB) comes back with mxb_bank_process(MXB_MEM_SPLIT | MXB_MEM_ASYNC); the voice signals stay on the device
  roofline   algorithmic bytes per launch / CUDA-event launch time against MEASURED_PEAKS.json
  cpu_baseline  the reference's own scalar code (oracle/_ref) on all host cores (pinned threads, >= 3 s timed), the
             -O2 parity build and an -O3 -march=x86-64-v3 build side by side; a reported baseline, not the target

`--impl reference` times only that CPU leg with the same metric/config (rank 0; other ranks exit 0).
`--dump-outputs DIR` writes what the headline's last timed step computed as DIR/<name>.npy (rank 0; a fixed, seeded sample of
DUMP_COLUMNS voices or channels of each array, fewer for the spectral arrays). Inputs are seeded, so two builds run with the same
arguments compare output for output. Every --workload dumps its outputs; `--impl reference` times the CPU reference only and refuses
the flag.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if "MXB_PATCH_CACHE" not in os.environ:     # patch kernels compiled at run time are cached in a directory removed at exit
    _patch_cache = tempfile.TemporaryDirectory(prefix="mxb_patch_cache_")
    os.environ["MXB_PATCH_CACHE"] = _patch_cache.name

BLOCK = 1024
SR = 48000

WORKLOADS = {
    # name: (voices/GPU, osc, filt, env, delay_taps, algorithmic bytes per voice-sample, description)
    "svf": dict(voices=1 << 20, osc="saw", filt="svf", env=False, delay=0, bytes_per=8.0 + (88 + 32) / BLOCK,
                desc="configs[1]: 1Mi voices maxiOsc::saw -> maxiSVF lp, 1024-frame block, fp64 out[1024][V] materialised"),
    "biquad": dict(voices=1 << 20, osc="saw", filt="biquad", env=False, delay=0, bytes_per=8.0 + (80 + 24) / BLOCK,
                   desc="configs[4] shard: 1Mi voices/GPU maxiOsc::saw -> maxiBiquad lowpass, fp64 out materialised + stereo mix"),
    "delay": dict(voices=1 << 18, osc="saw", filt="none", env=True, delay=4096, bytes_per=24.0 + (108 + 60) / BLOCK,
                  desc="configs[2]: 256Ki voices saw -> maxiEnv::adsr -> maxiDelayline::dl(4096), fp64 out materialised"),
}
CPU_BLOCKS_PER_STEP = 8       # the reference arm: one step = this many consecutive blocks of the CPU sample (32 for the delay chain)
DUMP_COLUMNS = 4096           # --dump-outputs: voices (channels) kept per array; 4096 x 1024 frames of fp64 = 32 MiB


def dump_output(E, args, name, t, dim=1, columns=DUMP_COLUMNS):
    """--dump-outputs: device tensor `t`, the result of the last timed step, as DIR/<name>.npy; along `dim` (voices or channels) a
    fixed, seeded sample of `columns` entries, in ascending order, when it has more."""
    if not args.dump_outputs or E.rank != 0:
        return
    n = t.shape[dim]
    if n > columns:
        idx = np.sort(np.random.default_rng(0).choice(n, columns, replace=False))
        t = t.index_select(dim, E.torch.from_numpy(idx).to(t.device))
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel of workload `key`,
    from the committed `ncu --set full` capture of this same bench command (profiles/traffic.json names the summary
    file each figure was read from). None when no capture of that configuration is committed."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[key]
        return {"traffic": float(d["dram_bytes_per_launch"]), "traffic_unit": "bytes/launch", "traffic_source": d["source"]}
    except Exception:
        return {"traffic": None}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for (t, r) in self.rows if t0 <= t <= t1] or [r for (_, r) in self.rows]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for i, n in enumerate(names):
                if len(r) > 5 + i and r[5 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(rows[0][2]) if rows[0][2].replace(".", "").isdigit() else None,
                "reasons": sorted(reasons), "samples": len(rows)}


# ------------------------------------------------------------------------------------------- CPU reference leg

class CpuFarm:
    """The reference on all host cores. `threads` persistent workers, each pinned to one core of this process's
    affinity mask (sched_setaffinity), each building its OWN slice of the work inside the worker (first touch = local NUMA
    node). A run releases all workers through a barrier and times until the last one is back at the next barrier: thread
    start-up, object construction and page faults of fresh buffers are outside the clock."""

    def __init__(self, threads, make_part):
        cores = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
        self.threads = max(1, threads)
        self.cores = cores
        self.parts = [None] * self.threads
        self.job = None
        self.err = []
        self._go = threading.Barrier(self.threads + 1)
        self._done = threading.Barrier(self.threads + 1)
        self._ts = [threading.Thread(target=self._worker, args=(i, make_part), daemon=True) for i in range(self.threads)]
        [t.start() for t in self._ts]
        self._done.wait()                      # every worker has built its part

    def _worker(self, i, make_part):
        try:
            if hasattr(os, "sched_setaffinity"):
                os.sched_setaffinity(threading.get_native_id(), {self.cores[i % len(self.cores)]})
        except Exception:
            pass
        try:
            self.parts[i] = make_part(i)
        except Exception as e:                 # noqa: BLE001 -- reported by run()
            self.err.append(repr(e))
        self._done.wait()
        while True:
            self._go.wait()
            if self.job is None:
                return
            try:
                self.job(i, self.parts[i])
            except Exception as e:             # noqa: BLE001
                self.err.append(repr(e))
            self._done.wait()

    def run(self, job):
        """Seconds for job(i, part) on every worker, barrier to barrier."""
        assert not self.err, self.err
        self.job = job
        self._go.wait()
        t0 = time.perf_counter()
        self._done.wait()
        dt = time.perf_counter() - t0
        assert not self.err, self.err
        return dt

    def close(self):
        self.job = None
        try:
            self._go.wait(timeout=5)
        except Exception:
            pass


def cpu_kinds():
    """[parity build, best-effort build] of the compiled reference, or the C port when the reference is absent."""
    from oracle import oracle_py as O
    kinds = [k for k in ("reference", "reference_o3") if O.available(k)]
    if not kinds:
        O.build("port")
        kinds = ["port"]
    return kinds


CPU_FLAGS = {"reference": "-O2 -ffp-contract=off (the parity build the oracle tests use)",
             "reference_o3": "-O3 -march=x86-64-v3 (AVX2 + FMA, contraction allowed; best-effort CPU, timed only)",
             "port": "-O2 -ffp-contract=off (plain-C restatement)"}


def cpu_sample_voices(wl):
    # each reference maxiDelayline is a 5.6 MB object (src/maximilian.h:273): keep the sample in RAM (16 voices per core,
    # 512 .. 2048 voices = 2.9 .. 11.5 GB)
    if wl["delay"]:
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        return int(min(2048, max(512, 16 * cores)))
    return 65536


def cpu_blocks_per_step(wl):
    return 32 if wl["delay"] else CPU_BLOCKS_PER_STEP


def bank_farm(wl, voices, kind):
    from maximilian_b200 import workloads as W
    from oracle import oracle_py as O
    O.load(kind)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = max(1, min(cores, voices))
    bounds = np.linspace(0, voices, threads + 1).astype(int)
    p = W.voice_params(voices, seed=W.SEED, delay_size=wl["delay"] or 4096)

    def make(i):
        lo, hi = int(bounds[i]), int(bounds[i + 1])
        b = O.Bank(hi - lo, osc=wl["osc"], filt=wl["filt"], env=wl["env"], delay=wl["delay"] > 0, sample_rate=SR,
                   delay_capacity=max(wl["delay"], 1), kind=kind)
        W.configure_bank(b, wl["filt"], {k: v[lo:hi] for k, v in p.items()}, wl["env"], wl["delay"] > 0)
        out = np.zeros((BLOCK, hi - lo), dtype=np.float64)
        out[:] = 1.0                                        # touch every page here, on the worker's own core
        return b, out, lo, hi
    return CpuFarm(threads, make), threads


def bank_job(wl, voices, nblocks, block_index0=0):
    from maximilian_b200 import workloads as W
    from oracle import oracle_py as O
    gates = [(W.gate(voices, BLOCK, block_index0 + k) if wl["env"] else (None, None)) for k in range(nblocks)]

    def job(i, part):
        b, out, lo, hi = part
        for on, off in gates:
            on_i = np.ascontiguousarray(on[lo:hi]) if on is not None else None
            off_i = np.ascontiguousarray(off[lo:hi]) if off is not None else None
            rc = b.lib.mxo_bank_process(b.h, BLOCK, O._ip(on_i), O._ip(off_i), O._dp(out), None, 0, hi - lo)
            assert rc == 0, rc
    return job


def cpu_bank_rate(wl, kind, budget_s, steps=None, warm=1):
    """voice-samples/s of the reference on all cores; >= budget_s seconds timed (or exactly `steps` steps of
    CPU_BLOCKS_PER_STEP blocks for the reference arm)."""
    voices = cpu_sample_voices(wl)
    farm, threads = bank_farm(wl, voices, kind)
    farm.run(bank_job(wl, voices, warm, 0))
    n, total = 0, 0.0
    if steps is not None:
        total = farm.run(bank_job(wl, voices, steps * cpu_blocks_per_step(wl), warm))
        n = steps * cpu_blocks_per_step(wl)
    else:
        per = CPU_BLOCKS_PER_STEP
        while total < budget_s and n < 4096:
            dt = farm.run(bank_job(wl, voices, per, warm + n))
            total += dt; n += per
            if dt < budget_s / 4:
                per *= 2                                    # few, long timed regions
    farm.close()
    return voices * BLOCK * n / total, voices, threads, n, total


def cpu_baseline(wl, budget_s=3.0):
    kinds = cpu_kinds()
    res = {}
    for k in kinds:
        v, voices, threads, n, total = cpu_bank_rate(wl, k, budget_s)
        res[k] = dict(value=v, flags=CPU_FLAGS[k], blocks=n, seconds=total)
    main = kinds[0]
    out = {"value": res[main]["value"], "unit": "samples/s", "cores": threads, "kind": "reference" if main.startswith("reference") else "port",
           "flags": res[main]["flags"], "timed_seconds": res[main]["seconds"],
           "sample": f"{voices} voices x {BLOCK} frames x {res[main]['blocks']} blocks of the same chain; {threads} pinned host threads, each with its own "
                     "slice of the voices as reference objects (frame-outer / voice-inner like a reference play())"}
    if len(kinds) > 1:
        out["best_effort"] = {"value": res[kinds[1]]["value"], "flags": res[kinds[1]]["flags"], "timed_seconds": res[kinds[1]]["seconds"]}
    return out


def reference_arm(args, wl_name, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kinds = cpu_kinds()
    kind = kinds[-1]                           # the fastest build of the unmodified reference that exists here
    v, voices, threads, n, dt = cpu_bank_rate(wl, kind, None, steps=args.steps, warm=max(1, args.warmup))
    extra = {}
    if len(kinds) > 1:
        v2, _, _, n2, dt2 = cpu_bank_rate(wl, kinds[0], 2.0)
        extra = {"parity_build": {"value": v2, "flags": CPU_FLAGS[kinds[0]], "timed_seconds": dt2}}
    line = {"impl": "reference", "metric": "voice_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["desc"], "cpu_sample_voices": voices, "block": BLOCK, "sample_rate": SR,
                       "blocks_per_step": cpu_blocks_per_step(wl)},
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": threads, "kind": "reference" if kind.startswith("reference") else "port",
                             "flags": CPU_FLAGS[kind], "timed_seconds": dt,
                             "sample": f"each step = {voices} voices x {BLOCK} frames x {cpu_blocks_per_step(wl)} blocks of the same chain on {threads} pinned host threads",
                             **extra},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU leg

def onbox_peaks(torch, out):
    """SURVEY.md 8(d): the streaming-WRITE and copy bandwidth of THIS box, measured with library kernels on the output
    buffer the bank just wrote (torch fill_ / copy_, best of 5, CUDA events), reported beside the driver-measured copy
    peak: the bank kernel is write-only traffic, which the copy figure does not isolate."""
    try:
        flat = out.view(-1)
        half = flat.numel() // 2
        a, b = flat[:half], flat[half:2 * half]
        best_fill = best_copy = best_r1w2 = 0.0
        # one read : two writes, the traffic mix of the delay-line kernel (ring in, ring out, voice out): complex(x, x) reads 8 B
        # and writes 16 B per element
        third = (flat.numel() // 3) & ~1          # even: view_as_complex wants an even storage offset
        x, z = flat[:third], torch.view_as_complex(flat[third:3 * third].view(third, 2)) if flat.dtype == torch.float64 else None
        for _ in range(5):
            e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
            e0.record(); flat.fill_(0.0); e1.record(); b.copy_(a); e2.record()
            if z is not None:
                torch.complex(x, x, out=z)
            e3.record()
            torch.cuda.synchronize()
            best_fill = max(best_fill, flat.numel() * flat.element_size() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
            best_copy = max(best_copy, 2 * half * flat.element_size() / (e1.elapsed_time(e2) * 1e-3) / 1e9)
            if z is not None:
                best_r1w2 = max(best_r1w2, 3 * third * flat.element_size() / (e2.elapsed_time(e3) * 1e-3) / 1e9)
        return {"fill_gbs": best_fill, "copy_gbs": best_copy, "read1_write2_gbs": best_r1w2 or None,
                "how": "torch fill_ over the %.1f GB output buffer (write-only), copy_ of one half onto the other (read+write bytes), "
                       "complex(x, x) of one third into the other two (1 read : 2 writes), best of 5" % (flat.numel() * flat.element_size() / 1e9)}
    except Exception as e:      # a missing number must not take the bench line down
        return {"error": str(e)[:200]}


def pcie_rates(torch, dev, mb=256):
    """Pinned-memory copy rates of this box (GB/s), the ceiling of every e2e number that moves bulk data."""
    try:
        h = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
        d = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
        best = [0.0, 0.0]
        for _ in range(4):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record(); d.copy_(h, non_blocking=True); e1.record(); h.copy_(d, non_blocking=True); e2.record()
            torch.cuda.synchronize()
            best[0] = max(best[0], (mb << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9)
            best[1] = max(best[1], (mb << 20) / (e1.elapsed_time(e2) * 1e-3) / 1e9)
        return {"h2d_gbs": best[0], "d2h_gbs": best[1]}
    except Exception as e:
        return {"error": str(e)[:200]}


class Env:
    """Process-wide pieces shared by the legs."""
    pass


def setup_env(args):
    import torch
    import torch.distributed as dist
    from maximilian_b200 import capi
    from maximilian_b200 import workloads as W
    E = Env()
    E.torch, E.dist, E.capi, E.W = torch, dist, capi, W
    E.rank = int(os.environ.get("RANK", "0")); E.world = int(os.environ.get("WORLD_SIZE", "1"))
    E.local = int(os.environ.get("LOCAL_RANK", "0"))
    assert E.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE {E.world}"
    torch.cuda.set_device(E.local)
    E.dev = torch.device("cuda", E.local)
    if E.world > 1:
        dist.init_process_group("nccl", device_id=E.dev)
    E.ctx = capi.Context(E.local, SR)
    E.stream = torch.cuda.current_stream()
    E.sampler = ClockSampler(E.local)
    if E.rank == 0:
        E.sampler.start()
        time.sleep(0.12)
    return E


def barrier(E):
    if E.world > 1:
        E.dist.barrier()
    E.torch.cuda.synchronize()


def max_over_ranks(E, x):
    t = E.torch.tensor([x], dtype=E.torch.float64, device=E.dev)
    if E.world > 1:
        E.dist.all_reduce(t, op=E.dist.ReduceOp.MAX)
    return float(t.item())


def bank_leg(E, args, wl_name, steps, warmup, want_mix=False, with_onbox=False, full_readback=False, dump=False):
    """One bank workload: resident-throughput, roofline and the pipelined e2e number. dump: --dump-outputs of the timed block."""
    torch, capi, W = E.torch, E.capi, E.W
    wl = WORKLOADS[wl_name]
    V = int(os.environ.get("MXB_BENCH_VOICES", wl["voices"]))      # experiment hook (wave-quantisation probes); the JSON states voices_per_gpu
    rank, world, dev, stream = E.rank, E.world, E.dev, E.stream
    p = W.voice_params(V, seed=W.SEED + rank, delay_size=wl["delay"] or 4096)
    bank = capi.Bank(V, osc=wl["osc"], filt=wl["filt"], env=wl["env"], delay=wl["delay"] > 0,
                     delay_capacity=max(wl["delay"], 1), max_frames=BLOCK, ctx=E.ctx, sample_rate=SR)
    W.configure_bank(bank, wl["filt"], p, wl["env"], wl["delay"] > 0)
    p2p = world > 1 and want_mix and args.collective == "p2p"
    if p2p:
        exch = capi.Exchange(E.ctx, rank, world, max_doubles=2 * BLOCK)
        exch.connect_with_torch_distributed()      # the IPC handles travel over the process group; the data never does
        exch.attach(bank)
    out_dtype = torch.float32 if args.f32_out else torch.float64
    out = torch.empty((BLOCK, V), dtype=out_dtype, device=dev)             # 8 GiB (fp64, 1 Mi voices) >> 126 MB L2
    mix = torch.zeros((BLOCK, 2), dtype=torch.float64, device=dev)
    gates = []
    if wl["env"]:   # gate arrays for 4 consecutive blocks, resident on the device (control data of the resident leg)
        for k in range(4):
            on, off = W.gate(V, BLOCK, k, seed=W.SEED + rank)
            gates.append((torch.from_numpy(on).to(dev), torch.from_numpy(off).to(dev)))

    def step(k):
        on_p = off_p = None
        if gates:
            on_p, off_p = gates[k % 4][0].data_ptr(), gates[k % 4][1].data_ptr()
        bank.process_device(BLOCK, out_ptr=out.data_ptr(), mix_ptr=mix.data_ptr() if want_mix else None,
                            trig_on_ptr=on_p, trig_off_ptr=off_p, f32=args.f32_out, stream=stream.cuda_stream)
        if world > 1 and want_mix and not p2p:
            E.dist.all_reduce(mix)

    for k in range(warmup):
        step(k)
    barrier(E)
    launches0 = bank.launches
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    t_wall0 = time.perf_counter()
    evs[0].record(stream)
    for k in range(steps):
        step(warmup + k)
        evs[k + 1].record(stream)
    torch.cuda.synchronize()
    t_wall1 = time.perf_counter()
    barrier(E)
    if dump:
        dump_output(E, args, "out", out)
        if want_mix:
            dump_output(E, args, "mix", mix)
    launches = bank.launches - launches0
    ms_total = evs[0].elapsed_time(evs[-1])
    per_launch_ms = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
    ms_max = max_over_ranks(E, ms_total)
    samples_per_step = V * BLOCK
    value = world * samples_per_step * steps / (ms_max * 1e-3)

    # ---- end to end through the C ABI with host control data, pipelined over three streams ---------------------------
    # per step: this block's frequency array goes up from pinned memory on the bank's copy stream (double-buffered on the
    # device), the block runs on the process stream, its stereo bus comes down into one of two pinned host buffers; the
    # host never blocks inside the loop -- one synchronisation at the end, inside the timed region.
    freq_host = [torch.from_numpy(p["freq"].copy()).pin_memory() for _ in range(2)]
    mix_host = [torch.zeros((BLOCK, 2), dtype=torch.float64).pin_memory() for _ in range(2)]
    on_h = off_h = None
    if wl["env"]:
        on, off = W.gate(V, BLOCK, 0, seed=W.SEED + rank)
        on_t, off_t = torch.from_numpy(on).pin_memory(), torch.from_numpy(off).pin_memory()
        on_h, off_h = on_t.numpy(), off_t.numpy()
    e2e_steps = max(3, min(steps, 50))

    def e2e_step(k):
        fh, mh = freq_host[k & 1].numpy(), mix_host[k & 1].numpy()
        bank.set_host_array("freq", fh, stream=stream.cuda_stream)        # H2D: this block's control data (copy stream)
        bank.process_split(BLOCK, out.data_ptr(), mh, on_h, off_h, f32=args.f32_out, stream=stream.cuda_stream, wait=False)   # D2H: mix bus
        if world > 1 and want_mix and not p2p:     # with the peer-memory exchange attached the bus that comes back is already the global one
            torch.cuda.current_stream().synchronize()
            m = mix_host[k & 1].to(dev, non_blocking=True)
            E.dist.all_reduce(m)

    for k in range(3):
        e2e_step(k)
    barrier(E)
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        e2e_step(k)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    e2e_value = world * samples_per_step * e2e_steps / max_over_ranks(E, dt)
    h2d = freq_host[0].numpy().nbytes + (on_h.nbytes + off_h.nbytes if on_h is not None else 0)
    d2h = mix_host[0].numpy().nbytes

    res = {"value": value, "unit": "samples/s", "ms_per_step": ms_max / steps, "steps": steps, "warmup": warmup, "gpu_launches": launches}
    if rank == 0:
        peak, peak_src = load_peaks()
        med_ms = per_launch_ms[len(per_launch_ms) // 2]
        avg_ms = ms_total / steps
        bytes_per = (4.0 if args.f32_out else 8.0) + (wl["bytes_per"] - 8.0)
        achieved = bytes_per * samples_per_step / (avg_ms * 1e-3) / 1e9
        res["config"] = {"workload": wl["desc"] + (" + stereo mix bus" if want_mix else ""), "voices_per_gpu": V, "block": BLOCK,
                         "sample_rate": SR, "out_storage": "f32" if args.f32_out else "f64", "parallelism": f"voices sharded x{world}",
                         "collective": ("none" if not (world > 1 and want_mix) else
                                        "peer-memory exchange of mix[1024][2] fp64 fused into the mix-reduce kernel (CUDA IPC over NVLink, rank-ordered sum)" if p2p
                                        else "NCCL sum all-reduce of mix[1024][2] fp64 per block"),
                         "l2": "no flush needed: each step writes %.1f GB, inputs+outputs >> 126 MB L2" % (samples_per_step * (4 if args.f32_out else 8) / 1e9)}
        res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                           **load_traffic(wl_name + ("_mix" if want_mix else "") + ("_f32" if args.f32_out else "")),
                           "algorithmic_bytes_per_launch": bytes_per * samples_per_step,
                           "peak_source": peak_src, "kernel": "bank_kernel" if not wl["delay"] else "delay_bank_kernel",
                           "algorithmic_bytes_per_voice_sample": bytes_per, "launch_ms_avg": avg_ms, "launch_ms_median": med_ms}
        res["e2e"] = {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "steps": e2e_steps, "frac_of_resident": e2e_value / value,
                      "what": "per step mxb_bank_set_param_async(freq, pinned host; copy stream, double-buffered) + "
                              "mxb_bank_process(MXB_MEM_SPLIT|MXB_MEM_ASYNC): host gates in, host mix out, voice signals "
                              "materialised on the device; one synchronisation at the end of the timed region"}
        res["clocks"] = E.sampler.summary(t_wall0, t_wall1)
        if with_onbox:
            onbox = onbox_peaks(torch, out)
            # the same store pattern with next to no arithmetic: a bank of bare phasors (3 fp64 operations per voice-sample) writing the same
            # time-major out[1024][V] -- what this box's memory system takes from V / 64 warps that each append 512 B to their own column
            # block of one row after the other (a library fill_ is ONE linear stream)
            try:
                pb = capi.Bank(V, osc="phasor", filt="none", env=False, delay=False, delay_capacity=1, max_frames=BLOCK, ctx=E.ctx, sample_rate=SR)
                pb.set("freq", p["freq"]); pb.set("phase", p["phase"])
                for _ in range(3):
                    pb.process_device(BLOCK, out_ptr=out.data_ptr(), mix_ptr=None, f32=args.f32_out, stream=stream.cuda_stream)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(10):
                    pb.process_device(BLOCK, out_ptr=out.data_ptr(), mix_ptr=None, f32=args.f32_out, stream=stream.cuda_stream)
                e1.record(stream)
                torch.cuda.synchronize()
                onbox["pattern_write_gbs"] = (4.0 if args.f32_out else 8.0) * samples_per_step * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9
                res["roofline"]["frac_of_onbox_pattern_write"] = achieved / onbox["pattern_write_gbs"]
                del pb
            except Exception as e:      # a missing number must not take the bench line down
                onbox["pattern_write_error"] = str(e)[:200]
            res["roofline"]["onbox_peaks"] = onbox
            if "fill_gbs" in onbox:
                res["roofline"]["frac_of_onbox_fill"] = achieved / onbox["fill_gbs"]
    if full_readback and world == 1:
        # the whole per-voice result back in host memory (MXB_MEM_HOST): PCIe-bound by construction, 8 B per voice-sample
        try:
            hout = torch.empty((BLOCK, V), dtype=out_dtype).pin_memory()
            ho = hout.numpy()
            bank.process(BLOCK, out=ho, out_dtype=ho.dtype)
            t0 = time.perf_counter()
            for _ in range(2):
                bank.process(BLOCK, out=ho, out_dtype=ho.dtype)
            dt = (time.perf_counter() - t0) / 2
            res["e2e_full_readback"] = {"value": samples_per_step / dt, "unit": "samples/s", "d2h_bytes_per_step": int(ho.nbytes), "steps": 2,
                                        "what": "mxb_bank_process(MXB_MEM_HOST): the whole out[1024][V] returns to pinned host memory every block (PCIe-bound)"}
            del hout, ho
        except Exception as e:
            res["e2e_full_readback"] = {"error": str(e)[:200]}
    del bank, out
    torch.cuda.empty_cache()
    return res


def measure_mixdown(E, args, sm_mhz):
    """BASELINE.json configs[4] in SURVEY.md 8(d)'s "mix mode", one shard per GPU: 1 Mi voices maxiOsc::saw ->
    maxiBiquad -> maxiMix::stereo -> sum over voices; no per-voice output is written, the stereo bus [1024][2] is the
    result. With N > 1 the bus is summed over the GPUs (the path's only exchange step). The kernel moves 0.1 B per
    voice-sample, so it is reported against the fp64 pipe (SURVEY.md 8(d) config 5), not against HBM; it is never
    mixed into the headline."""
    torch, dist, capi, W = E.torch, E.dist, E.capi, E.W
    rank, world, dev, stream = E.rank, E.world, E.dev, E.stream
    wl = WORKLOADS["biquad"]
    V = wl["voices"]
    p = W.voice_params(V, seed=W.SEED + 100 + rank)
    bank = capi.Bank(V, osc=wl["osc"], filt=wl["filt"], env=False, delay=False, delay_capacity=1, max_frames=BLOCK,
                     ctx=E.ctx, sample_rate=SR)
    W.configure_bank(bank, wl["filt"], p, False, False)
    mix = torch.zeros((BLOCK, 2), dtype=torch.float64, device=dev)
    p2p = world > 1 and args.collective == "p2p"
    check = None
    if p2p:
        exch = capi.Exchange(E.ctx, rank, world, max_doubles=2 * BLOCK)
        exch.connect_with_torch_distributed()      # the IPC handles travel over the process group; the data never does
        # correctness of the fused exchange, before anything is timed: a clone of the bank (same state, no exchange) gives
        # this rank's LOCAL bus; an NCCL sum all-reduce of the local buses must equal the exchanged bus to fp64
        # reassociation, and the exchanged bus must be the same bits on every rank
        twin = bank.clone()
        exch.attach(bank)
        local = torch.zeros_like(mix)
        ok, worst = True, 0.0
        for _ in range(3):
            bank.process_device(BLOCK, out_ptr=None, mix_ptr=mix.data_ptr(), stream=stream.cuda_stream)
            twin.process_device(BLOCK, out_ptr=None, mix_ptr=local.data_ptr(), stream=stream.cuda_stream)
            ref = local.clone()
            dist.all_reduce(ref)
            err = float(((mix - ref).abs() / (ref.abs() + 1e-9)).max().item())
            worst = max(worst, err)
            gathered = [torch.empty_like(mix) for _ in range(world)]
            dist.all_gather(gathered, mix)
            same = all(bool(torch.equal(g, gathered[0])) for g in gathered)
            ok = ok and err <= 1e-12 and same
        ok = ok and exch.status() == 0
        flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        check = {"result": "ok" if flag.item() == 1.0 else "FAILED", "max_rel_err_vs_nccl_allreduce": worst,
                 "what": "3 blocks: peer-exchanged bus == NCCL sum all-reduce of the ranks' local buses (<= 1e-12 relative), "
                         "bit-equal on every rank, no exchange time-out"}
        del twin
    steps = max(3, min(args.steps, 50))

    def step():
        bank.process_device(BLOCK, out_ptr=None, mix_ptr=mix.data_ptr(), stream=stream.cuda_stream)
        if world > 1 and not p2p:
            dist.all_reduce(mix)

    for _ in range(3):
        step()
    barrier(E)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    barrier(E)
    ms = max_over_ranks(E, e0.elapsed_time(e1)) / steps
    # e2e of mix mode: the WHOLE result of the block (the stereo bus) lands in host memory every step, the block's
    # frequency array goes up every step; pipelined like the headline's e2e
    freq_host = [torch.from_numpy(p["freq"].copy()).pin_memory() for _ in range(2)]
    mix_host = [torch.zeros((BLOCK, 2), dtype=torch.float64).pin_memory() for _ in range(2)]

    def e2e_step(k):
        bank.set_host_array("freq", freq_host[k & 1].numpy(), stream=stream.cuda_stream)
        bank.process_split(BLOCK, None, mix_host[k & 1].numpy(), stream=stream.cuda_stream, wait=False)
        if world > 1 and not p2p:
            torch.cuda.current_stream().synchronize()
            m = mix_host[k & 1].to(dev, non_blocking=True)
            dist.all_reduce(m)
    for k in range(3):
        e2e_step(k)
    barrier(E)
    t0 = time.perf_counter()
    for k in range(steps):
        e2e_step(k)
    torch.cuda.synchronize()
    e2e_dt = max_over_ranks(E, time.perf_counter() - t0)
    # fp64-pipe instructions per voice-sample in the SASS of this instantiation: saw 3 (DSETP, 2 DADD), biquad 9
    # (5 DMUL, 4 DADD: -fmad=false keeps the reference's roundings), mix 2 (DMUL/DFMA per channel) + 1 (row sums)
    instr = 15.0
    rate = instr * V * BLOCK / (ms * 1e-3)                    # fp64 lane-instructions per second per GPU
    pipe_peak = 148 * 64 * (sm_mhz or 1920.0) * 1e6           # 64 fp64 lanes per SM (16 per sub-partition), one instr per lane-clock
    res = {"workload": "configs[4] shard, mix mode: 1Mi voices/GPU maxiOsc::saw -> maxiBiquad lowpass -> maxiMix::stereo -> sum over voices, "
                       "stereo bus [1024][2] fp64 per block, no per-voice output",
           "value": world * V * BLOCK / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": steps,
           "bound": "fp64 pipe", "fp64_instr_per_voice_sample": instr, "fp64_pipe_frac_per_gpu": rate / pipe_peak,
           "fp64_pipe_peak": "148 SMs x 64 lanes x %.0f MHz (sampled SM clock)" % (sm_mhz or 1920.0),
           "e2e": {"value": world * V * BLOCK * steps / e2e_dt, "unit": "samples/s", "h2d_bytes_per_step": int(freq_host[0].numpy().nbytes),
                   "d2h_bytes_per_step": int(mix_host[0].numpy().nbytes), "steps": steps,
                   "what": "frequency array up, the block's whole result (the stereo bus) down into pinned host memory, every step"},
           "collective": ("none (one GPU)" if world == 1 else
                          "peer-memory exchange of mix[1024][2] fp64 fused into the mix-reduce kernel (CUDA IPC over NVLink, rank-ordered sum)"
                          if p2p else "NCCL sum all-reduce of mix[1024][2] fp64 per block")}
    if check is not None:
        res["check"] = check
    del bank
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------- configs[3]: FFT + MFCC frames/s

MFCC_WL = dict(channels=65536, fft=1024, hop=512, filters=42, coeffs=40, hops_per_step=8,
               # minimum traffic per (channel, hop) frame: 512 new fp32 samples in, 40 fp64 coefficients out (SURVEY.md 8d)
               bytes_per=512 * 4 + 40 * 8,
               desc="configs[3]: 64Ki channels maxiFFT(1024, hop 512) + maxiMFCC(42 filters, 40 coeffs), streaming, "
                    "8 hops (524288 frames) per step, fused: spectra stay on chip, fp64 MFCCs written")


def mfcc_farm(channels, kind):
    from maximilian_b200 import workloads as W
    from oracle import oracle_py as O
    O.load(kind)
    wl = MFCC_WL
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = max(1, min(cores, channels // 8))      # at least 8 channels per host thread
    bounds = np.linspace(0, channels, threads + 1).astype(int)
    per_call = 16       # hops per library call: the time goes to the reference's C++ loops, not to Python call overhead
    x = W.channel_streams(channels, per_call * wl["hop"], seed=5)

    def make(i):
        c = int(bounds[i + 1] - bounds[i])
        return (O.Stft(c, wl["fft"], wl["hop"], kind=kind), O.Mfcc(wl["fft"] // 2, wl["filters"], wl["coeffs"], 20.0, 20000.0, SR, kind=kind),
                np.ascontiguousarray(x[bounds[i]:bounds[i + 1]]))
    return CpuFarm(threads, make), threads, per_call


def cpu_mfcc_rate(kind, budget_s, channels=4096, calls=None):
    """frames/s of maxiFFT + maxiMFCC per channel on all cores."""
    farm, threads, per_call = mfcc_farm(channels, kind)

    def job_n(n):
        def job(i, part):
            st, mf, xi = part
            for _ in range(n):
                r = st.process(xi, want=("mags",))
                mf.process(r["mags"])
        return job
    farm.run(job_n(1))
    n, total = 0, 0.0
    if calls is not None:
        total = farm.run(job_n(calls)); n = calls
    else:
        per = 1
        while total < budget_s and n < 1024:
            dt = farm.run(job_n(per))
            total += dt; n += per
            if dt < budget_s / 4:
                per *= 2
    farm.close()
    return channels * per_call * n / total, channels, threads, n * per_call, total


def cpu_baseline_mfcc(budget_s=3.0):
    kinds = cpu_kinds()
    res = {}
    for k in kinds:
        v, ch, threads, hops, total = cpu_mfcc_rate(k, budget_s)
        res[k] = dict(value=v, flags=CPU_FLAGS[k], hops=hops, seconds=total)
    main = kinds[0]
    out = {"value": res[main]["value"], "unit": "frames/s", "cores": threads, "kind": "reference" if main.startswith("reference") else "port",
           "flags": res[main]["flags"], "timed_seconds": res[main]["seconds"],
           "sample": f"{ch} channels x {res[main]['hops']} hops, maxiFFT+maxiMFCC per channel, channels partitioned over {threads} pinned host threads"}
    if len(kinds) > 1:
        out["best_effort"] = {"value": res[kinds[1]]["value"], "flags": res[kinds[1]]["flags"], "timed_seconds": res[kinds[1]]["seconds"]}
    return out


def mfcc_leg(E, args, steps, warmup, dump=False):
    torch, capi, W = E.torch, E.capi, E.W
    rank, world, dev, stream = E.rank, E.world, E.dev, E.stream
    wl = MFCC_WL
    C, n, hop, H = wl["channels"], wl["fft"], wl["hop"], wl["hops_per_step"]
    st = capi.Stft(C, n, hop, ctx=E.ctx); mf = capi.Mfcc(n // 2, wl["filters"], wl["coeffs"], 20.0, 20000.0, ctx=E.ctx)
    base = W.channel_streams(1024, H * hop, seed=5 + rank)
    x_host = torch.from_numpy(np.tile(base, (C // 1024, 1))).pin_memory()           # [C][H*hop] planar fp32, 1 GiB
    x = x_host.to(dev)
    coeffs = torch.empty((C, H, wl["coeffs"]), dtype=torch.float64, device=dev)
    co_host = torch.empty((C, H, wl["coeffs"]), dtype=torch.float64).pin_memory()

    def step():
        f = st.process_device(x.data_ptr(), H * hop, 1, H * hop, H, mfcc=mf, coeffs=coeffs.data_ptr(), stream=stream.cuda_stream)
        assert f == H

    for _ in range(warmup):
        step()
    barrier(E)
    l0 = st.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    tw1 = time.perf_counter()
    barrier(E)
    if dump:
        dump_output(E, args, "mfcc", coeffs, dim=0)
    ms = e0.elapsed_time(e1)
    ms_max = max_over_ranks(E, ms)
    frames_per_step = C * H
    value = world * frames_per_step * steps / (ms_max * 1e-3)
    launches = st.launches - l0
    # e2e: host samples in (pinned), host MFCCs out, through the C ABI (MXB_MEM_HOST): the library slices the channels and
    # pipelines upload / transform / download over three streams
    import ctypes as C_
    xh, ch_ = x_host.numpy(), co_host.numpy()
    nf = C_.c_int32(0)

    def e2e_step():
        capi.check(capi.lib().mxb_stft_process(st.h, xh.ctypes.data, H * hop, 1, H * hop, H, None, None, None, None, mf.h, ch_.ctypes.data,
                                               C_.byref(nf), capi.MEM_HOST, C_.c_void_p(stream.cuda_stream)), "mxb_stft_process")
    e2e_steps = max(3, min(steps, 10))
    for _ in range(2):
        e2e_step()
    barrier(E)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_dt = max_over_ranks(E, time.perf_counter() - t0)
    e2e_value = world * frames_per_step * e2e_steps / e2e_dt
    res = {"metric": "fft_mfcc_frames_per_sec", "value": value, "unit": "frames/s", "ms_per_step": ms_max / steps, "steps": steps, "warmup": warmup,
           "gpu_launches": launches}
    if rank == 0:
        peak, peak_src = load_peaks()
        avg_ms = ms / steps
        achieved = wl["bytes_per"] * frames_per_step / (avg_ms * 1e-3) / 1e9
        pcie = pcie_rates(torch, dev)
        res["config"] = {"workload": wl["desc"], "channels_per_gpu": C, "hops_per_step": H, "parallelism": f"channels sharded x{world}", "collective": "none",
                         "l2": "per step 1.07 GB of samples in + 168 MB of MFCCs out: larger than the 126 MB L2"}
        res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, **load_traffic("mfcc"),
                           "algorithmic_bytes_per_launch": wl["bytes_per"] * frames_per_step,
                           "peak_source": peak_src, "kernel": "stft_stream_kernel", "algorithmic_bytes_per_frame": wl["bytes_per"],
                           "launch_ms_avg": avg_ms, "note": "fp32 issue bound by design of the reference transform (bit-exact radix-2 replay + fp64 mel/DCT); "
                                                          "HBM fraction is reported as north_star asks, not expected to be high"}
        e2e_bytes = int(xh.nbytes) + int(ch_.nbytes)
        res["e2e"] = {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(xh.nbytes), "d2h_bytes_per_step": int(ch_.nbytes),
                      "steps": e2e_steps, "pcie": pcie,
                      "what": "mxb_stft_process(MXB_MEM_HOST): pinned host samples in, fused STFT+MFCC, host MFCCs out; channel slices pipelined "
                              "over copy-in / compute / copy-out streams"}
        if "h2d_gbs" in pcie:
            # the link moves both directions at once: the floor is the slower of the two transfers
            floor_s = max(xh.nbytes / (pcie["h2d_gbs"] * 1e9), ch_.nbytes / (pcie["d2h_gbs"] * 1e9))
            res["e2e"]["frac_of_pcie_floor"] = (floor_s * e2e_steps) / e2e_dt
            res["e2e"]["bytes_per_step"] = e2e_bytes
        res["clocks"] = E.sampler.summary(tw0, tw1)
    del st, mf, x, coeffs
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ voice patch (SURVEY.md 8(f))

PATCH_WL = dict(voices=1 << 18, bytes_per=8.0 + 1.0 / 8 + (12 * 16 + 8 * 8) / BLOCK,
                desc="15.polysynth voice patch x 256Ki voices: 2 pulse VCOs (one detuned by a sinebuf LFO) -> lores VCF with per-sample cutoff "
                     "(coefficients designed every sample: cos, pow, sqrt) -> x ADSR (per-sample trigger, one bit per voice-sample), fp64 out[1024][V] materialised + stereo bus")


def _tables():
    g = np.load(os.path.join(ROOT, "tests", "golden", "tables.npz"))      # the reference's sineBuffer / transition DATA (extracted by make_golden.py)
    return g["sine"], g["transition"], float(g["sine_before"])


def cpu_patch_rate(kind, budget_s, voices=4096, blocks=None):
    """the reference's own objects run the same stage list per sample (oracle/ref_shim.cpp), voices partitioned over pinned threads;
    >= budget_s seconds timed (or exactly `blocks` blocks for the reference arm)"""
    from maximilian_b200 import workloads as W
    from oracle import oracle_py as O
    O.load(kind)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = max(1, min(cores, voices // 8))
    bounds = np.linspace(0, voices, threads + 1).astype(int)
    prm = W.polysynth_params(voices)
    pat = W.note_pattern(voices)
    d = W.polysynth_patch()

    def make(i):
        lo, hi = int(bounds[i]), int(bounds[i + 1])
        q = O.Patch(d, hi - lo, sample_rate=SR, kind=kind)
        for k, v in prm.items():
            q.set(k, v[lo:hi])
        trig = [W.note_triggers(pat, BLOCK, b, lo, hi, dtype=np.float64) for b in range(2)]
        return q, trig

    farm = CpuFarm(threads, make)

    def job_n(n, b0):
        def job(i, part):
            q, trig = part
            for b in range(n):
                q.process(BLOCK, {"trigger": trig[(b0 + b) & 1]}, want_out=True, want_mix=False)
        return job
    farm.run(job_n(1, 0))
    n, total, per = 0, 0.0, 2
    if blocks is not None:
        total, n = farm.run(job_n(blocks, 0)), blocks
    while blocks is None and total < budget_s and n < 1024:
        dt = farm.run(job_n(per, n))
        total += dt; n += per
        if dt < budget_s / 4:
            per *= 2
    farm.close()
    return voices * BLOCK * n / total, voices, threads, n, total


def cpu_baseline_patch(budget_s=3.0):
    kinds = cpu_kinds()
    res = {}
    for k in kinds:
        v, voices, threads, n, total = cpu_patch_rate(k, budget_s)
        res[k] = dict(value=v, flags=CPU_FLAGS[k], blocks=n, seconds=total)
    main = kinds[0]
    out = {"value": res[main]["value"], "unit": "samples/s", "cores": threads, "kind": "reference" if main.startswith("reference") else "port",
           "flags": res[main]["flags"], "timed_seconds": res[main]["seconds"],
           "sample": f"{voices} voices x {BLOCK} frames x {res[main]['blocks']} blocks of the same patch run by the reference's own objects, per sample, "
                     f"voices partitioned over {threads} pinned host threads"}
    if len(kinds) > 1:
        out["best_effort"] = {"value": res[kinds[1]]["value"], "flags": res[kinds[1]]["flags"], "timed_seconds": res[kinds[1]]["seconds"]}
    return out


def patch_leg(E, args, steps, warmup, dump=False):
    """The reference's polysynth example as a voice patch: the kernel generated + NVRTC-compiled for its stage list (K8f), the
    interpreting kernel (K8) beside it, and the e2e loop with the trigger bytes coming from the host every block."""
    torch, capi, W = E.torch, E.capi, E.W
    rank, world, dev, stream = E.rank, E.world, E.dev, E.stream
    wl = PATCH_WL
    V = int(os.environ.get("MXB_BENCH_PATCH_VOICES", wl["voices"]))
    capi.set_tables(*_tables(), ctx=E.ctx)
    assert V % 32 == 0
    d = W.polysynth_patch("bits")
    prm = W.polysynth_params(V, seed=W.SEED + rank)
    pat = tuple(torch.from_numpy(a).to(dev) for a in W.note_pattern(V, seed=W.SEED + rank))
    weights = (torch.ones(32, dtype=torch.int64, device=dev) << torch.arange(32, dtype=torch.int64, device=dev))

    def triggers(block_index):          # the same formula as workloads.note_triggers, evaluated on the device for 256 Ki voices, then
        t = (torch.arange(BLOCK, dtype=torch.int64, device=dev) + BLOCK * block_index)[:, None]      # packed: voice v = bit v % 32 of word v / 32
        on = (((t + pat[1][None, :]) % pat[0][None, :]) < pat[2][None, :]).to(torch.int64)
        return (on.view(BLOCK, V // 32, 32) * weights).sum(-1).to(torch.int32).contiguous()
    trig = [triggers(b) for b in range(2)]
    out = torch.empty((BLOCK, V), dtype=torch.float64, device=dev)
    mix = [torch.zeros((BLOCK, 2), dtype=torch.float64, device=dev) for _ in range(2)]
    res_modes = {}
    t_wall = [0.0, 0.0]
    patches = {}
    for mode in ("fused", "interpret"):
        t_c0 = time.perf_counter()
        pt = capi.Patch(d, V, max_frames=BLOCK, ctx=E.ctx, sample_rate=SR, mode=mode)
        compile_s = time.perf_counter() - t_c0
        for k, v in prm.items():
            pt.set(k, v)
        patches[mode] = pt
        n = steps if mode == "fused" else max(3, min(steps, 5))

        def step(k):
            pt.process_device(BLOCK, [trig[k & 1].data_ptr()], out.data_ptr(), mix[k & 1].data_ptr(), stream=stream.cuda_stream)
        for k in range(warmup):
            step(k)
        barrier(E)
        l0 = pt.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.perf_counter()
        e0.record(stream)
        for k in range(n):
            step(warmup + k)
        e1.record(stream)
        torch.cuda.synchronize()
        tw1 = time.perf_counter()
        barrier(E)
        ms = e0.elapsed_time(e1)
        ms_max = max_over_ranks(E, ms)
        res_modes[mode] = dict(value=world * V * BLOCK * n / (ms_max * 1e-3), ms_per_step=ms_max / n, steps=n, launches=pt.launches - l0, ms_local=ms / n,
                               create_seconds=compile_s)
        if mode == "fused":
            t_wall = [tw0, tw1]
            if dump:
                dump_output(E, args, "out", out)
                dump_output(E, args, "mix", mix[(warmup + n - 1) & 1])
    # ---- e2e: per step this block's trigger bytes go up from pinned memory on a copy stream (double-buffered on the device), the
    # fused patch runs, the stereo bus comes back into one of two pinned buffers; one synchronisation at the end
    pt = patches["fused"]
    trig_host = [t.cpu().pin_memory() for t in trig]
    trig_dev = [torch.empty_like(trig[0]) for _ in range(2)]
    mix_host = [torch.zeros((BLOCK, 2), dtype=torch.float64).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ev_up = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]

    def e2e_step(k):
        b = k & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_done[b])
            trig_dev[b].copy_(trig_host[b], non_blocking=True)
            ev_up[b].record(copy_stream)
        stream.wait_event(ev_up[b])
        pt.process_device(BLOCK, [trig_dev[b].data_ptr()], out.data_ptr(), mix[b].data_ptr(), stream=stream.cuda_stream)
        ev_done[b].record(stream)
        mix_host[b].copy_(mix[b], non_blocking=True)
    e2e_steps = max(3, min(steps, 30))
    for k in range(3):
        e2e_step(k)
    barrier(E)
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        e2e_step(k)
    torch.cuda.synchronize()
    dt = max_over_ranks(E, time.perf_counter() - t0)
    f = res_modes["fused"]
    res = {"metric": "voice_samples_per_sec", "value": f["value"], "unit": "samples/s", "ms_per_step": f["ms_per_step"], "steps": f["steps"], "warmup": warmup,
           "gpu_launches": f["launches"]}
    if rank == 0:
        peak, peak_src = load_peaks()
        achieved = wl["bytes_per"] * V * BLOCK / (f["ms_local"] * 1e-3) / 1e9
        res["config"] = {"workload": wl["desc"], "voices_per_gpu": V, "block": BLOCK, "sample_rate": SR, "parallelism": f"voices sharded x{world}", "collective": "none",
                         "l2": "no flush needed: each step writes %.1f GB (and reads %.0f MB of packed trigger bits)" % (V * BLOCK * 8 / 1e9, V * BLOCK / 8e6)}
        res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, **load_traffic("patch"),
                           "algorithmic_bytes_per_launch": wl["bytes_per"] * V * BLOCK, "algorithmic_bytes_per_voice_sample": wl["bytes_per"],
                           "peak_source": peak_src, "kernel": "mxb_fused_patch (generated per patch, NVRTC)", "launch_ms_avg": f["ms_local"],
                           "note": "fp64-arithmetic bound, not HBM bound: the per-sample lores design (cos + pow + sqrt + 3 divisions) and two oscillator "
                                   "increments (2 divisions each) are ~1000 instructions per voice-sample; the HBM fraction is reported as north_star asks"}
        res["interpreter"] = {"value": res_modes["interpret"]["value"], "unit": "samples/s", "ms_per_step": res_modes["interpret"]["ms_per_step"],
                              "steps": res_modes["interpret"]["steps"], "fused_speedup": f["value"] / res_modes["interpret"]["value"],
                              "what": "the same patch on the interpreting kernel (MXB_PATCH_INTERPRET): identical results bit for bit"}
        res["compile_seconds"] = f["create_seconds"]
        res["e2e"] = {"value": world * V * BLOCK * e2e_steps / dt, "unit": "samples/s", "h2d_bytes_per_step": int(trig_host[0].numel() * trig_host[0].element_size()),
                      "d2h_bytes_per_step": int(mix_host[0].numel() * 8), "steps": e2e_steps, "frac_of_resident": world * V * BLOCK * e2e_steps / dt / f["value"],
                      "what": "per step: packed trigger bits [1024][V/32] words from pinned host memory (copy stream, double-buffered), mxb_patch_process(MXB_MEM_DEVICE) "
                              "of the fused patch, stereo bus back to pinned host memory; voice signals materialised on the device"}
        res["clocks"] = E.sampler.summary(t_wall[0], t_wall[1])
    del patches, pt, out, trig, trig_dev
    torch.cuda.empty_cache()
    return res



# ------------------------------------------------------------------------------------------------ spectral round trip + analysers (SURVEY.md 8(f))

SPEC_WL = dict(channels=1 << 14, fft=1024, hop=512, hops_per_step=8,
               desc="16Ki channels, 8 hops per step: maxiFFT 1024/512 (magnitudes + phases written) -> maxiIFFT SPECTRUM resynthesis; and the same "
                    "analysis with maxiFFTOctaveAnalyzer (averages + peaks) and maxiBark (specific / relative / total loudness) fused in")


def modulated_leg(E, args, steps, warmup, dump=False):
    """SURVEY.md 8(f) rank 1, timed: the banks with a per-sample oscillator frequency (FM: `osc.saw(f + lfo)`, the reference takes the
    frequency by argument on every call) -- one more 8-byte stream READ per voice-sample, resident on the device like the output.
    fm_svf: configs[1]'s bank (K1, MOD instantiation); fm_delay: configs[2]'s bank (K2, the modulated instantiation of its windows)."""
    torch, capi, W = E.torch, E.capi, E.W
    dev, stream, rank = E.dev, E.stream, E.rank
    res = {}
    for key, wl_name in (("fm_svf", "svf"), ("fm_delay", "delay")):
        wl = WORKLOADS[wl_name]
        V = wl["voices"]
        p = W.voice_params(V, seed=W.SEED + rank, delay_size=wl["delay"] or 4096)
        bank = capi.Bank(V, osc=wl["osc"], filt=wl["filt"], env=wl["env"], delay=wl["delay"] > 0,
                         delay_capacity=max(wl["delay"], 1), max_frames=BLOCK, ctx=E.ctx, sample_rate=SR)
        W.configure_bank(bank, wl["filt"], p, wl["env"], wl["delay"] > 0)
        out = torch.empty((BLOCK, V), dtype=torch.float64, device=dev)
        # freq_tv[t][v] = f_v * (1 + 0.02 sin(2 pi 5 t / sr + v)): a 5 Hz vibrato, built in place on the device (synthetic control data)
        ft = torch.arange(BLOCK, dtype=torch.float64, device=dev).mul_(2.0 * math.pi * 5.0 / SR)[:, None].expand(BLOCK, V).contiguous()
        ft.add_(torch.arange(V, dtype=torch.float64, device=dev)[None, :]).sin_().mul_(0.02).add_(1.0)
        ft.mul_(torch.from_numpy(p["freq"]).to(dev)[None, :])
        gates = None
        if wl["env"]:
            on, off = W.gate(V, BLOCK, 0, seed=W.SEED + rank)
            gates = (torch.from_numpy(on).to(dev), torch.from_numpy(off).to(dev))
        torch.cuda.synchronize()

        def step():
            bank.process_mod_device(BLOCK, out_ptr=out.data_ptr(), freq_tv_ptr=ft.data_ptr(),
                                    trig_on_ptr=gates[0].data_ptr() if gates else None, trig_off_ptr=gates[1].data_ptr() if gates else None,
                                    stream=stream.cuda_stream)
        for _ in range(warmup):
            step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        l0 = bank.launches
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        torch.cuda.synchronize()
        if dump:
            dump_output(E, args, key + "_out", out, columns=DUMP_COLUMNS // 2)
        ms = e0.elapsed_time(e1) / steps
        peak, peak_src = load_peaks()
        bytes_per = wl["bytes_per"] + 8.0
        achieved = bytes_per * V * BLOCK / (ms * 1e-3) / 1e9
        res[key] = {"value": V * BLOCK / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
                    "gpu_launches": bank.launches - l0,
                    "config": {"workload": wl["desc"] + " + per-sample frequency freq_tv[1024][V] fp64 (device-resident)", "voices_per_gpu": V,
                               "block": BLOCK, "l2": "no flush needed: each step streams far more than the 126 MB L2"},
                    "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                                 "note": "the reference recomputes the increment 1./(sampleRate/frequency) on every call: an IEEE fp64 division and a reciprocal "
                                         "per voice-sample, kept for bit parity (straight-line sequences, csrc/bank_kernels.cuh osc_increment_unchecked)",
                                 "algorithmic_bytes_per_voice_sample": bytes_per, "peak_source": peak_src,
                                 "kernel": "delay_bank_kernel<..., MODK>" if wl["delay"] else "bank_kernel<..., MOD = 1>"}}
        del bank, out, ft
        torch.cuda.empty_cache()
    return res


def spectral_extra_leg(E, args, steps, warmup, dump=False):
    """The rows of SURVEY.md 8(f) around the transform that the MFCC leg does not touch: the full-spectrum analysis (cartToPol incl.
    atan2), the octave-analyser / Bark epilogues, and maxiIFFT. Each sub-leg: CUDA events over `steps` steps, algorithmic bytes.
    dump: --dump-outputs of each sub-leg's last step, DUMP_COLUMNS / 8 channels (8 MiB per spectrum array)."""
    import ctypes as C_
    torch, capi, W = E.torch, E.capi, E.W
    dev, stream, world = E.dev, E.stream, E.world
    wl = SPEC_WL
    C, n, hop, H = wl["channels"], wl["fft"], wl["hop"], wl["hops_per_step"]
    bins = n // 2
    base = W.channel_streams(1024, H * hop, seed=11 + E.rank)
    x = torch.from_numpy(np.tile(base, (C // 1024, 1))).to(dev)                  # [C][H*hop] planar fp32
    mags = torch.empty((C, H, bins), dtype=torch.float32, device=dev); phases = torch.empty_like(mags)
    y = torch.empty((C, H * hop), dtype=torch.float32, device=dev)
    L = capi.lib()
    sp = C_.c_void_p(stream.cuda_stream)
    nf = C_.c_int32(0)
    peak, peak_src = load_peaks()
    out = {}

    def timed(fn, n_steps):
        for _ in range(warmup):
            fn()
        barrier(E)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n_steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        barrier(E)
        return max_over_ranks(E, e0.elapsed_time(e1)) / n_steps

    def entry(ms, bytes_per_frame, kernel, what, traffic_key=None):
        frames = C * H
        ach = bytes_per_frame * frames / (ms * 1e-3) / 1e9
        return {"value": world * frames / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "steps": steps,
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, **load_traffic(traffic_key), "peak_source": peak_src,
                             "kernel": kernel, "algorithmic_bytes_per_frame": bytes_per_frame, "algorithmic_bytes_per_launch": bytes_per_frame * frames}, "what": what}

    # (1) analysis with the whole spectrum leaving the chip: magnitudes + phases (atan2f per bin)
    st = capi.Stft(C, n, hop, ctx=E.ctx)
    ms = timed(lambda: st.process_device(x.data_ptr(), H * hop, 1, H * hop, H, mags=mags.data_ptr(), phases=phases.data_ptr(), stream=stream.cuda_stream), steps)
    if dump:
        dump_output(E, args, "analysis_mags", mags, dim=0, columns=DUMP_COLUMNS // 8)
        dump_output(E, args, "analysis_phases", phases, dim=0, columns=DUMP_COLUMNS // 8)
    out["analysis_mags_phases"] = entry(ms, hop * 4 + 2 * bins * 4, "stft_stream_kernel<FULL>", "maxiFFT::process + cartToPol, magnitudes and phases written")
    # (2) resynthesis: maxiIFFT SPECTRUM from those magnitudes / phases
    ist = capi.Istft(C, n, hop, ctx=E.ctx)

    def resyn():
        capi.check(L.mxb_istft_process(ist.h, C_.c_void_p(mags.data_ptr()), C_.c_void_p(phases.data_ptr()), H, C_.c_void_p(y.data_ptr()), capi.MEM_DEVICE, sp), "mxb_istft_process")
    ms = timed(resyn, steps)
    if dump:
        dump_output(E, args, "resynthesis", y, dim=0, columns=DUMP_COLUMNS // 8)
    out["resynthesis"] = entry(ms, 2 * bins * 4 + hop * 4, "istft1024_kernel", "maxiIFFT::process(SPECTRUM): polToCart, inverse transform, window, overlap-add", "istft")
    del ist, y, phases
    # (3) analysis with the octave analyser and Bark loudness fused in (magnitudes written too)
    oc = capi.Octave(C, float(SR), bins, 3, ctx=E.ctx)
    nA = oc.n_averages
    av = torch.empty((C, H, nA), dtype=torch.float32, device=dev); pk = torch.empty_like(av)
    bs = torch.empty((C, H, 24), dtype=torch.float64, device=dev); br = torch.empty_like(bs); bt = torch.empty((C, H), dtype=torch.float64, device=dev)
    o = capi.StftOutputs(mags.data_ptr(), None, None, None, None, None, None, None)
    post = capi.StftPost(oc.h, av.data_ptr(), pk.data_ptr(), 1, bs.data_ptr(), br.data_ptr(), bt.data_ptr())

    def analyse():
        capi.check(L.mxb_stft_process3(st.h, C_.c_void_p(x.data_ptr()), H * hop, 1, H * hop, H, C_.byref(o), C_.byref(post), None, C_.byref(nf), capi.MEM_DEVICE, sp), "mxb_stft_process3")
    ms = timed(analyse, steps)
    if dump:
        for name, t in (("octave_bark_mags", mags), ("octave_averages", av), ("octave_peaks", pk), ("bark_specific", bs), ("bark_relative", br),
                        ("bark_total", bt)):
            dump_output(E, args, name, t, dim=0, columns=DUMP_COLUMNS // 8)
    out["analysis_octave_bark"] = entry(ms, hop * 4 + bins * 4 + 2 * nA * 4 + (48 + 1) * 8, "stft_stream_kernel<FULL> + octave / Bark epilogues",
                                        f"maxiFFT::process + maxiFFTOctaveAnalyzer::calculate ({nA} averages, peaks) + maxiBark, magnitudes written")
    out["config"] = {"workload": wl["desc"], "channels_per_gpu": C, "hops_per_step": H}
    del st, oc, x, mags, av, pk, bs, br, bt
    torch.cuda.empty_cache()
    return out



def finish(E):
    if E.rank == 0:
        time.sleep(0.06)
        E.sampler.stop()
    if E.world > 1:
        E.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS) + ["mfcc", "patch", "spectral", "modulated"],
                    help="headline workload (default svf = BASELINE.json configs[1]; without this flag and with one GPU the other "
                         "configurations are measured too and reported under 'workloads')")
    ap.add_argument("--mix", type=int, default=-1,
                    help="1: the timed block also produces the stereo mix bus (+ the cross-GPU mix-down when gpus > 1). Default: the "
                         "headline block is the configured chain alone (same work at every N) and the mix-down configuration "
                         "(configs[4]) is timed separately and reported under 'mixdown'")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only")
    ap.add_argument("--f32-out", action="store_true", help="store the materialised output as fp32 (declared in the JSON)")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1 mix-down: p2p = peer-memory exchange fused into the mix-reduce kernel (default); nccl = torch.distributed all_reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step computed as DIR/<name>.npy (a fixed, seeded sample of voices or channels)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference only times the CPU reference")
    extras_wanted = args.workload is None and not args.no_extras
    wl_name = args.workload or "svf"
    if args.impl == "reference":
        if wl_name == "mfcc":
            return reference_arm_mfcc(args)
        if wl_name == "patch":
            return reference_arm_patch(args)
        return reference_arm(args, wl_name, WORKLOADS[wl_name])
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    E = setup_env(args)

    if wl_name == "spectral":
        r = spectral_extra_leg(E, args, args.steps, args.warmup, dump=True)
        if E.rank == 0:
            print(json.dumps({"metric": "fft_frames_per_sec", "unit": "frames/s", "n_gpus": E.world, "higher_is_better": True, "data": "synthetic", **r}), flush=True)
        return finish(E)

    if wl_name == "modulated":
        r = modulated_leg(E, args, args.steps, args.warmup, dump=True)
        if E.rank == 0:
            print(json.dumps({"metric": "voice_samples_per_sec", "unit": "samples/s", "n_gpus": E.world, "higher_is_better": True, "data": "synthetic", **r}), flush=True)
        return finish(E)

    if wl_name == "patch":
        head = patch_leg(E, args, args.steps, args.warmup, dump=True)
        if E.rank == 0:
            line = {"metric": "voice_samples_per_sec", "value": head["value"], "unit": "samples/s", "n_gpus": E.world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f64", "data": "synthetic", **{k: head[k] for k in ("config", "roofline", "e2e", "gpu_launches", "clocks", "interpreter", "compile_seconds")}}
            if not args.no_cpu and E.world == 1:
                line["cpu_baseline"] = cpu_baseline_patch()
            print(json.dumps(line), flush=True)
        return finish(E)

    if wl_name == "mfcc":
        head = mfcc_leg(E, args, args.steps, args.warmup, dump=True)
        if E.rank == 0:
            line = {"metric": "fft_mfcc_frames_per_sec", "value": head["value"], "unit": "frames/s", "n_gpus": E.world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": head["config"], "roofline": head["roofline"], "e2e": head["e2e"],
                    "gpu_launches": head["gpu_launches"], "clocks": head["clocks"]}
            if not args.no_cpu and E.world == 1:
                line["cpu_baseline"] = cpu_baseline_mfcc()
            print(json.dumps(line), flush=True)
        return finish(E)

    want_mix = args.mix == 1
    head = bank_leg(E, args, wl_name, args.steps, args.warmup, want_mix=want_mix, with_onbox=True, full_readback=extras_wanted, dump=True)
    mixdown = None
    if args.mix < 0 and not WORKLOADS[wl_name]["delay"]:
        mhz = E.torch.tensor([float((head.get("clocks") or {}).get("sm_mhz") or 0.0)], dtype=E.torch.float64, device=E.dev)
        if E.world > 1:
            E.dist.broadcast(mhz, 0)
        mixdown = measure_mixdown(E, args, float(mhz.item()) or None)
    extras = None
    if extras_wanted and E.world == 1:
        xs = max(3, min(args.steps, 40)); xw = max(3, min(args.warmup, 5))
        extras = {}

        def extra(key, run, cpu=None):
            # a leg that fails is reported as such under its key; it never takes the headline line with it
            try:
                r = run()
                if cpu is not None and not args.no_cpu:
                    r["cpu_baseline"] = cpu()
            except Exception as e:       # noqa: BLE001
                r = {"error": f"{type(e).__name__}: {e}"}
                try:
                    E.torch.cuda.synchronize(); E.torch.cuda.empty_cache()
                except Exception:    # noqa: BLE001
                    pass
            extras[key] = r
        for key, name in (("biquad_bank", "biquad"), ("delay", "delay")):
            extra(key, lambda name=name: bank_leg(E, args, name, xs, xw), lambda name=name: cpu_baseline(WORKLOADS[name], budget_s=3.0))
        extra("mfcc", lambda: mfcc_leg(E, args, max(3, min(args.steps, 20)), xw), lambda: cpu_baseline_mfcc(3.0))
        extra("patch", lambda: patch_leg(E, args, max(3, min(args.steps, 20)), xw), lambda: cpu_baseline_patch(3.0))
        extra("spectral_extras", lambda: spectral_extra_leg(E, args, 5, 3))
        extra("modulated", lambda: modulated_leg(E, args, max(3, min(args.steps, 20)), xw))
    if E.rank == 0:
        line = {"metric": "voice_samples_per_sec", "value": head["value"], "unit": "samples/s", "n_gpus": E.world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": head["config"], "roofline": head["roofline"],
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"]}
        if "e2e_full_readback" in head:
            line["e2e_full_readback"] = head["e2e_full_readback"]
        if mixdown is not None:
            line["mixdown"] = mixdown
        if extras is not None:
            line["workloads"] = extras
        if not args.no_cpu and E.world == 1:
            line["cpu_baseline"] = cpu_baseline(WORKLOADS[wl_name], budget_s=4.0)
        print(json.dumps(line), flush=True)
    finish(E)


def reference_arm_mfcc(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    wl = MFCC_WL
    kind = cpu_kinds()[-1]
    v, ch, threads, hops, dt = cpu_mfcc_rate(kind, None, calls=4 * max(1, args.steps))
    print(json.dumps({"impl": "reference", "metric": "fft_mfcc_frames_per_sec", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": 1, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": wl["desc"], "cpu_sample_channels": ch, "hops_per_step": 64},
                      "cpu_baseline": {"value": v, "unit": "frames/s", "cores": threads, "kind": "reference" if kind.startswith("reference") else "port",
                                       "flags": CPU_FLAGS[kind], "timed_seconds": dt,
                                       "sample": f"each step = 64 hops of {ch} channels on {threads} pinned host threads"},
                      "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


def reference_arm_patch(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    kind = cpu_kinds()[-1]
    v, voices, threads, n, dt = cpu_patch_rate(kind, None, blocks=args.steps)
    print(json.dumps({"impl": "reference", "metric": "voice_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": 1, "ms_per_step": 1e3 * dt / max(1, n), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                      "data": "synthetic", "config": {"workload": PATCH_WL["desc"], "cpu_sample_voices": voices, "block": BLOCK, "sample_rate": SR},
                      "cpu_baseline": {"value": v, "unit": "samples/s", "cores": threads, "kind": "reference" if kind.startswith("reference") else "port",
                                       "flags": CPU_FLAGS[kind], "timed_seconds": dt, "sample": f"{voices} voices x {BLOCK} frames x {n} blocks on {threads} pinned host threads"},
                      "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


if __name__ == "__main__":
    main()
