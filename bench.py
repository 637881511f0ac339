#!/usr/bin/env python
"""bench.py — headline measurement of the hot path (SURVEY.md §8d, BASELINE.json configs[1]).

Workload: 4096 SUBSYNTH32 voices (32-node subtractive-synth graph, per-voice f0 = 55*(1 + v mod 40) Hz) per GPU,
512-sample blocks @ 48 kHz.  One "step" = one block of all voices through the fused render kernel K1 (+ K2, the
mix-bus reduction, + K4, the cross-GPU sum of the [1][512] mix bus when N > 1).  Weak scaling: every rank
owns its own 4096 voices; the only data-path collective is the mix-bus sum (SURVEY.md §8e).

  value  : Msamples/s, device-resident (state, delay rings and parameters in HBM; no host I/O in the step),
           CUDA events per step on the launching stream, L2 flushed (256 MiB memset) between steps outside the events;
           at N > 1 a device-side cross-GPU barrier sits between the flush and the first event, so the skew of the
           per-rank flushes is not charged to the step.
  e2e    : same metric through the public API call a user makes (elem_b200_process: host output buffers,
           D2H of the mix bus and the synchronisation inside the timed region; the graph has no audio inputs,
           so h2d_bytes_per_step is 0).
  roofline: K1 only — algorithmic bytes per launch (DESIGN.md §4) / mean launch duration measured with CUDA events
           around every K1 launch on its own stream (a second pass of the same steps: the event pairs sit between the
           kernels of a step and would cost `value` a few microseconds of launch gap), against MEASURED_PEAKS.json hbm_gbs; beside it the issue-slot
           roofline (K1's real bound): warp instructions per launch (ncu capture of the SAME K1 sources, else null)
           / duration against SMs x 4 schedulers x the SM clock sampled during the run.
  parity : after the timed loops the SAME runtime renders one more block with per-voice outputs; every voice and the
           mix bus are compared with the reference engine advanced by exactly as many blocks (parity_checked,
           worst_err_over_tol).  A bench line whose kernel computed something else says so.
  cpu_baseline / --impl reference: the UNMODIFIED reference engine (oracle/_ref/libelem_ref.so, built from
           the reference sources in place) on the box's host cores: T = all threads (value) and T = 1, pinned threads created
           and warmed up outside the timed region, >= 2 s timed (oracle/ref_driver.cpp:elem_ref_bench_stable).
  --dump-outputs DIR: after the timed steps, the mix bus [1][512] (float32) that the last step of the `value` loop left in the
           engine — what enqueue_block hands its caller — as DIR/mix.npy, and that of the 131072-voice row as DIR/t1_mix.npy.
           Every input is fixed by the arguments (per-voice f0 from the voice index, no random state), so two builds of the
           project run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, BS = 48000.0, 512
VOICES_PER_GPU = 4096
T1_VOICES_PER_GPU = 131072                      # 8 x 131072 = the 1 M-voice target of BASELINE.json's north_star
ALGO_BYTES_PER_VOICE_BLOCK_MIX_ONLY = 4236      # SURVEY.md §8d / DESIGN.md §4: 88 state + 52 params + 4096 delay ring
METRIC = "Msamples/s (voices x 512-sample blocks / s), 4096-voice SUBSYNTH32 per GPU @ 48 kHz"
K1_SOURCES = ("render_kernel.cu", "render_ops.inc", "program.h")


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def k1_source_sha16():
    h = hashlib.sha256()
    for f in K1_SOURCES:
        h.update(open(os.path.join(ROOT, "elementary_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def build_runtime(voices, device, rank, stream_handle=None, **opts):
    import numpy as np
    from elementary_b200 import Runtime, graphs
    rt = Runtime(SR, BS, voices, device=device, **opts)
    if stream_handle is not None:
        rt.set_stream(stream_handle)
    assert rt.apply_instructions(graphs.subsynth32()) == 0, rt.last_error()
    ida, idb = graphs.subsynth32_param_ids()
    f0 = np.array([graphs.subsynth32_f0(rank * voices + v) for v in range(voices)], dtype=np.float64)
    assert rt.set_property_per_voice(ida, "value", f0) == 0
    assert rt.set_property_per_voice(idb, "value", f0 * 1.007) == 0
    return rt


# ---- the reference engine on the host cores ---------------------------------------------------------------------------------
def cpu_reference_run(voices, threads, warmup_blocks, blocks, min_seconds, voice_offset=0):
    """Time the unmodified reference (or, if oracle/_ref did not travel, nothing) on `threads` pinned host threads."""
    from elementary_b200 import graphs
    from oracle import oracle as orc
    if not orc.ref_available():
        return None
    vb = [graphs.subsynth32_voice_props(voice_offset + v) for v in range(voices)]
    secs, chk, nb = orc.ref_bench(SR, BS, graphs.subsynth32(), vb, voices, threads, 0, 1, warmup_blocks, blocks, min_seconds=min_seconds)
    if secs <= 0:
        return None
    return {"seconds": secs, "blocks": nb, "msamples_per_s": voices * BS * nb / secs / 1e6,
            "voice_blocks_per_s": voices * nb / secs, "checksum": chk}


def host_description():
    from oracle import oracle as orc
    try:
        model = orc.ref_cpu_model()
    except Exception:
        model = "unknown"
    try:
        usable = len(os.sched_getaffinity(0))
    except Exception:
        usable = os.cpu_count() or 1
    quota = None                       # a container CPU quota (cgroup v2 cpu.max / v1 cfs_quota) bounds the cores the threads really get
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    try:
        load1 = float(open("/proc/loadavg").read().split()[0])
    except Exception:
        load1 = None
    # threads the reference arm uses: one per CPU the container may really use (a CFS quota of 16 on a 128-CPU host means 16 —
    # 128 pinned threads there are throttled 8:1 and measure the throttling, not the engine)
    import math
    threads = usable if quota is None else max(1, min(usable, int(math.ceil(quota))))
    return {"nproc": os.cpu_count() or 1, "usable_cpus": usable, "cgroup_cpu_quota": quota, "threads_used": threads,
            "loadavg_1m_before": load1, "cpu_model": model}


def bench_config(voices_per_gpu, world):
    """The workload description — the SAME dict in both arms (`--impl b200` and `--impl reference`), so that the driver's
    same-config check compares like with like; everything engine specific lives in the line's "engine" key."""
    return {"workload": f"{voices_per_gpu} SUBSYNTH32 voices per GPU (BASELINE.json configs[1]: 32-node subtractive synth), 512-sample blocks, 48 kHz",
            "voices_per_gpu": voices_per_gpu, "voices_total": world * voices_per_gpu, "block": BS, "sample_rate": SR,
            "l2": "GPU arm: L2 flushed between steps (256 MiB memset outside the timed events); CPU arm: the voices' state exceeds the host caches"}


def run_reference(args, rank, world, emit=print):
    if rank != 0:
        return
    host = host_description()
    cores = host["threads_used"]
    voices = VOICES_PER_GPU * world
    rall = cpu_reference_run(voices, cores, max(1, args.warmup), args.steps, 2.5)
    if rall is None:
        emit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libelem_ref.so missing (built only where /root/reference exists)"}))
        return
    r1 = cpu_reference_run(32, 1, 5, 20, 2.0)
    ms = rall["seconds"] / rall["blocks"] * 1e3
    sample = (f"all {voices} voices, {rall['blocks']:.1f} blocks of 512 each in {rall['seconds']:.2f} s (time-bounded, >= {args.steps} blocks), "
              f"{cores} pinned threads created and warmed up outside the timed region (whole workload, not a subset)")
    line = {
        "impl": "reference", "metric": METRIC, "value": rall["msamples_per_s"], "unit": "Msamples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(VOICES_PER_GPU, world),
        "engine": {"name": "elem::Runtime<float> (unmodified reference, oracle/_ref), one instance per voice, round-robin per thread"},
        "voice_blocks_per_s": rall["voice_blocks_per_s"],
        "cpu_baseline": {"value": rall["msamples_per_s"], "unit": "Msamples/s", "cores": cores, "kind": "reference", "sample": sample,
                         "t1": None if r1 is None else {"value": r1["msamples_per_s"], "unit": "Msamples/s", "cores": 1,
                                                        "sample": f"32 voices x {r1['blocks']:.0f} blocks on one pinned thread, {r1['seconds']:.2f} s"},
                         "host": host},
        "e2e": {"value": rall["msamples_per_s"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))


# ---- the CUDA path ----------------------------------------------------------------------------------------------------------
def class_references(n_blocks):
    """SUBSYNTH32 has 40 distinct voices (f0 = 55 * (1 + v mod 40)).  Advance one reference engine per class by n_blocks blocks and
    return the LAST block of each: [40, BS] float32.  Compiled reference if it travelled, else the bit-exact CPU restatement."""
    import numpy as np
    from elementary_b200 import graphs
    from oracle import oracle as orc
    cls = orc.RefRuntime if orc.ref_available() else orc.PortRuntime
    out = np.zeros((40, BS), dtype=np.float32)
    for c in range(40):
        o = cls(SR, BS)
        assert o.apply(graphs.subsynth32()) == 0 and o.apply(graphs.subsynth32_voice_props(c)) == 0
        last = None
        for _ in range(n_blocks):
            last = o.process(None, 1, BS)
        out[c] = last[0]
    return out, cls.__name__


def measure(args, voices, steps, warmup, rank, local_rank, world, stream, flush, with_clocks, check_parity, keep_mix=False):
    import numpy as np
    import torch
    import torch.distributed as dist
    from elementary_b200.runtime import FLAG_MIX, FLAG_ALLREDUCE, FLAG_VOICE_OUT
    from elementary_b200.distributed import attach_peer_mix

    extra = {"tile_width": args.tile_width} if args.tile_width else {}
    extra["specialize"] = args.specialize
    for kv in args.opt:
        k, v = kv.split("=")
        extra[k] = float(v)
    rt = build_runtime(voices, local_rank, rank, stream.cuda_stream, time_kernels=1, **extra)
    mix = torch.as_tensor(rt.mix_device(1), device=f"cuda:{local_rank}")
    host_mix = torch.empty((1, BS), dtype=torch.float32).pin_memory()

    # The single collective of the path: the sum of the [1][512] mix bus over the ranks.  Default: the engine's own
    # kernel over NVLink/NVSwitch peer memory (K4, launched by enqueue_block in the same stream); --collective nccl
    # (or a box without peer access) uses torch.distributed.all_reduce instead.
    fused, fused_note = False, None
    if world > 1 and args.collective == "fused":
        try:
            attach_peer_mix(rt)
            fused = True
        except Exception as e:      # reported in the JSON line, never silent
            fused_note = f"peer attach failed ({e}); NCCL all_reduce used"
        ok = torch.tensor([1 if fused else 0], device=f"cuda:{local_rank}")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        fused = bool(int(ok[0]))
    step_flags = FLAG_MIX | (FLAG_ALLREDUCE if fused else 0)
    blocks_done = 0

    def step_device(flags=step_flags):
        nonlocal blocks_done
        rt.enqueue_block(0, 1, BS, flags)
        blocks_done += 1
        if world > 1 and not fused:
            dist.all_reduce(mix)

    def line_up():
        """all ranks' streams meet here (device side), so a timed region starts on every GPU together"""
        if world > 1:
            if fused:
                rt.peer_barrier()
            else:
                dist.barrier()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also carries every voice past the 20 ms root fade) ----
    for _ in range(max(3, warmup)):
        step_device()
    barrier()
    rt.take_kernel_time_ms()

    # ---- value: device-resident, per-step CUDA events, L2 flushed between steps ----
    # The engine's own per-kernel event pairs are OFF in this loop: they sit between the kernels of a step and cost a few microseconds
    # of launch gap per step (at N > 1 they made `value` slower than `e2e`).  The per-kernel durations the roofline needs come from a
    # second pass of the same steps right below, with the pairs on.
    rt.set_option("time_kernels", 0)
    sampler = ClockSampler(local_rank) if with_clocks and rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = rt.kernel_launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for a, b in evs:
        flush.zero_()
        line_up()
        a.record(stream)
        step_device()
        b.record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    last_mix = mix.cpu().numpy().copy() if keep_mix else None      # the last timed step's output, before the passes below overwrite it
    launches = rt.kernel_launches - launches0      # K1 + K2 (+ K4) per step; the line-up barriers are not counted by the engine

    # ---- per-kernel durations (roofline, kernel_ms): the same steps once more, event pairs around every launch ----
    rt.set_option("time_kernels", 1)
    barrier()
    for _ in range(min(steps, 100)):
        flush.zero_()
        line_up()
        step_device()
    barrier()
    k1_ms, k1_n = rt.take_kernel_time_ms()
    kinds = rt.last_kernel_times()

    # ---- e2e: the public call with host buffers (D2H + sync inside) ----
    # (per-kernel event pairs are a measurement device of the loop above, not part of what a caller of process() pays: off here)
    rt.set_option("time_kernels", 0)
    barrier()
    e2e_s = 0.0
    for _ in range(steps):
        flush.zero_()
        line_up()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if world == 1 or fused:
            rt.process(None, 1, BS)      # with peers attached process() returns the mix of ALL ranks on every rank (K4 inside)
            blocks_done += 1
        else:
            step_device()
            if rank == 0:
                host_mix.copy_(mix[:1], non_blocking=True)
            stream.synchronize()
        e2e_s += time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if sampler else None      # nvidia-smi samples cover both timed regions (value and e2e)

    # ---- parity of what was just timed: one more block, every voice + the (all-reduced) mix against the reference ----
    parity = {"parity_checked": False}
    if check_parity:
        step_device(step_flags | FLAG_VOICE_OUT)
        barrier()
        got = torch.as_tensor(rt.voice_out_device(1), device=f"cuda:{local_rank}")[:, 0].cpu().numpy()
        got_mix = mix[0].cpu().numpy().astype(np.float64)
        refs, oracle_name = class_references(blocks_done)
        tol40 = 1e-5 * np.abs(refs.astype(np.float64)).max(axis=1, keepdims=True) + 1e-7
        worst, exact = 0.0, 0
        for v0 in range(0, voices, 8192):                    # chunked: 131072 voices x 512 samples in float64 would be 0.5 GB per temporary
            cls_of = (rank * voices + np.arange(v0, min(voices, v0 + 8192))) % 40
            g = got[v0:v0 + 8192]
            worst = max(worst, float((np.abs(g.astype(np.float64) - refs[cls_of]) / tol40[cls_of]).max()))
            exact += int((g == refs[cls_of]).sum())
        counts = np.bincount((np.arange(world * voices)) % 40, minlength=40).astype(np.float64)    # the mix bus is the sum over ALL ranks
        want_mix = (refs.astype(np.float64) * counts[:, None]).sum(axis=0)
        mix_tol = 1e-5 * np.abs(want_mix).max() + 1e-7
        worst_mix = float((np.abs(got_mix - want_mix) / mix_tol).max())
        w = torch.tensor([worst, worst_mix], dtype=torch.float64, device=f"cuda:{local_rank}")
        if world > 1:
            dist.all_reduce(w, op=dist.ReduceOp.MAX)
        parity = {"parity_checked": True, "worst_err_over_tol": float(w[0]), "mix_worst_err_over_tol": float(w[1]),
                  "parity_ok": bool(float(w[0]) <= 1.0 and float(w[1]) <= 1.0),
                  "parity_detail": f"block {blocks_done} of the timed runtime: all {voices} voices per rank vs {oracle_name} (40 f0 classes), "
                                   f"mix bus vs the float64 sum of the references over all {world * voices} voices; tolerance 1e-5 x block peak",
                  "bit_exact_rate": exact / float(voices * BS)}

    peer_fail = rt.peer_status() if fused else 0
    t = torch.tensor([dev_ms, e2e_s * 1e3, kinds["K1"][0], kinds["K2"][0], kinds["K4"][0]], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    desc = rt.describe()["groups"][0]
    res = {"voices": voices, "steps": steps, "dev_ms": float(t[0]), "e2e_ms": float(t[1]), "k1_ms": float(t[2]), "k1_n": k1_n,
           "k2_ms": float(t[3]), "k2_n": kinds["K2"][1], "k4_ms": float(t[4]), "k4_n": kinds["K4"][1],
           "launches": int(launches), "t_wall": t_wall, "clocks": clocks, "desc": desc, "fused": fused, "fused_note": fused_note,
           "peer_fail": peer_fail, "parity": parity, "last_mix": last_mix}
    rt.close()
    return res


def run_b200(args, rank, local_rank, world, emit=print):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    # NCCL prints its version banner to stdout when NCCL_DEBUG=VERSION (it honours NCCL_DEBUG_FILE only above that level)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    voices = args.voices
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")
        keep = bool(args.dump_outputs)
        m = measure(args, voices, args.steps, args.warmup, rank, local_rank, world, stream, flush, True, not args.no_parity, keep)
        t1 = None
        if not args.no_t1 and voices != T1_VOICES_PER_GPU:      # row T1: the 1 M-voice target = 131072 voices on each of 8 GPUs
            t1 = measure(args, T1_VOICES_PER_GPU, min(args.steps, 30), 5, rank, local_rank, world, stream, flush, False, not args.no_parity, keep)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    if rank != 0:
        return
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "mix.npy"), m["last_mix"].astype(np.float32))
        if t1 is not None:
            np.save(os.path.join(args.dump_outputs, "t1_mix.npy"), t1["last_mix"].astype(np.float32))

    steps = args.steps
    dev_ms, e2e_ms = m["dev_ms"], m["e2e_ms"]
    total_samples = world * voices * BS * steps
    value = total_samples / (dev_ms * 1e-3) / 1e6
    e2e_value = total_samples / (e2e_ms * 1e-3) / 1e6
    peak, peak_kind = measured_hbm_peak()
    k1_avg_ms = m["k1_ms"] / max(1, m["k1_n"])
    algo_bytes = ALGO_BYTES_PER_VOICE_BLOCK_MIX_ONLY * voices
    achieved = algo_bytes / (k1_avg_ms * 1e-3) / 1e9 if k1_avg_ms > 0 else 0.0
    desc, clocks = m["desc"], m["clocks"]
    specialised = desc.get("spec_state") == 2

    # ncu numbers (DRAM traffic, instruction count) are only quoted when the capture was made from the K1 sources of THIS build
    traffic, ncu, issue = None, None, None
    sha = k1_source_sha16()
    try:
        tj_all = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = "render_block_kernel_spec" if specialised else "render_block_kernel"
        tj = tj_all.get(key, {}).get(str(voices))
        if tj and tj_all.get("k1_source_sha16") == sha:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            ncu = {k: tj[k] for k in ("warp_instructions", "issue_active_pct", "registers_per_thread", "fp64_pipe_pct",
                                      "active_threads_per_warp_inst", "report", "local_load_sectors", "local_store_sectors") if k in tj}
            if "warp_instructions" in tj:
                ncu["warp_instructions_per_voice_sample"] = tj["warp_instructions"] / (voices * BS)
                clk_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
                slots = 148 * 4 * clk_hz
                rate = tj["warp_instructions"] / (k1_avg_ms * 1e-3) if k1_avg_ms > 0 else 0.0
                issue = {"bound": "issue", "achieved": rate / 1e9, "peak": slots / 1e9, "unit": "G warp-instr/s", "frac": rate / slots,
                         "note": "warp instructions per launch (ncu) / K1 duration (CUDA events) against 148 SMs x 4 schedulers x the SM clock sampled during the run"}
        elif tj:
            ncu = {"stale": True, "note": f"profiles/ncu_traffic.json was captured from other K1 sources ({tj_all.get('k1_source_sha16')} != {sha}): not quoted"}
    except Exception:
        pass

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        host = host_description()
        cores = host["threads_used"]
        rall = cpu_reference_run(16 * cores, cores, 10, 50, 10.0)
        r1 = cpu_reference_run(16, 1, 5, 20, 3.0)
        if rall is not None:
            cpu = {"value": rall["msamples_per_s"], "unit": "Msamples/s", "cores": cores, "kind": "reference",
                   "sample": f"{16 * cores} voices (16 per thread) x {rall['blocks']:.0f} blocks of 512, {rall['seconds']:.1f} s timed on {cores} pinned threads, unmodified reference via oracle/_ref",
                   "t1": None if r1 is None else {"value": r1["msamples_per_s"], "unit": "Msamples/s", "cores": 1,
                                                  "sample": f"16 voices x {r1['blocks']:.0f} blocks on one pinned thread, {r1['seconds']:.1f} s"},
                   "host": host}

    fused, fused_note, peer_fail = m["fused"], m["fused_note"], m["peer_fail"]
    line = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(voices, world),
        "engine": {"name": "elementary_b200 (libelem_b200.so through the C ABI)",
                   "tile_width": desc["tile_width"], "slots": desc["slots"], "state_rows": desc["state_rows"],
                   "k1": ("specialised per program (NVRTC, option specialize=%d)" % args.specialize) if specialised else "interpreter",
                   "spec": {k: desc[k] for k in ("spec_state", "spec_regs", "spec_local_bytes", "spec_cubin_bytes", "spec_log") if k in desc},
                   "collective": "none (1 GPU)" if world == 1 else
                                 ("K4 mix_exchange_kernel: all-reduce(sum,f32) of the [1][512] mix bus per block over NVLink peer memory, one launch in the render stream"
                                  + ("" if not peer_fail else " — PEER TIMEOUT REPORTED") if fused else
                                  "NCCL all_reduce(sum,f32) of the [1][512] mix bus per block" + (f" ({fused_note})" if fused_note else ""))},
        "voice_blocks_per_s": world * voices * steps / (dev_ms * 1e-3),
        "realtime_factor": value * 1e6 / (world * voices * SR),
        "wall_ms_per_step_incl_flush": m["t_wall"] / steps * 1e3,
        "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4 * BS,
                "ms_per_step": e2e_ms / steps, "api": "elem_b200_process (host out buffers; the kernel that finishes the mix bus stores it into mapped host memory)" if world == 1 else
                       ("elem_b200_process on every rank (render + K4 cross-GPU mix, delivered to host memory by K4)" if fused else "elem_b200_enqueue_block + NCCL all_reduce + D2H of the mix bus")},
        "gpu_launches": m["launches"],
        "kernel_ms": {"K1_render": k1_avg_ms, "K2_mix_reduce": m["k2_ms"] / max(1, m["k2_n"]),
                      "K4_mix_exchange": (m["k4_ms"] / m["k4_n"]) if m["k4_n"] else None,
                      "note": "mean device time per launch, CUDA events around each launch on the render stream, max over ranks; measured in a second pass of the same steps (the timed loop of `value` runs without these event pairs)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_kind": f"of {peak_kind}", "kernel": "render_block_kernel<NITER,LOGL> (K1)" + (" specialised" if specialised else ""),
                     "kernel_ms": k1_avg_ms, "kernel_launches_timed": m["k1_n"], "ncu": ncu, "k1_source_sha16": sha,
                     "algorithmic_bytes_per_launch": algo_bytes, "issue_slots": issue,
                     "note": "K1 is instruction-issue bound, not HBM bound (intermediates never leave the SM); see DESIGN.md section 4"},
        "clocks": clocks,
        "cpu_baseline": cpu,
    }
    line.update(m["parity"])
    if t1 is not None:
        ms = t1["dev_ms"] / t1["steps"]
        line["t1_million_voices"] = {
            "voices_per_gpu": T1_VOICES_PER_GPU, "voices_total": world * T1_VOICES_PER_GPU, "ms_per_block": ms,
            "block_budget_ms": BS / SR * 1e3, "realtime_factor": (BS / SR * 1e3) / ms,
            "value": world * T1_VOICES_PER_GPU * BS / (ms * 1e-3) / 1e6, "unit": "Msamples/s",
            "k1_ms": t1["k1_ms"] / max(1, t1["k1_n"]), "tile_width": t1["desc"]["tile_width"],
            "k1": "specialised" if t1["desc"].get("spec_state") == 2 else "interpreter",
            "hbm_frac": (ALGO_BYTES_PER_VOICE_BLOCK_MIX_ONLY * T1_VOICES_PER_GPU / (t1["k1_ms"] / max(1, t1["k1_n"]) * 1e-3) / 1e9) / peak,
            "steps": t1["steps"], **t1["parity"]}
    if world == 1 and not args.no_configs:
        line["other_configs"] = other_configs()
    emit(json.dumps(line))


def other_configs():
    """BASELINE.json configs 3, 4 and 5 at their per-GPU share (bench_configs.py), so that they are driver-run numbers too: ms per block
    (device resident), Msamples/s, the kernel's algorithmic-bytes roofline fraction (K3 for config 4), a bounded CPU reference sample
    and — config 5 — the parity check of a sample of the graphs.  Short runs: the whole leg takes well under a minute."""
    import bench_configs
    out = {}
    for key, fn, quick in (("3_additive64_8192_voices", bench_configs.config3, True), ("4_convolve_16384_taps_1024_channels", bench_configs.config4, True),
                           ("5_random_graphs_1250", bench_configs.config5, False)):
        try:
            r = fn(quick)
            r.pop("program", None)
            out[key] = r
        except Exception as e:      # reported, never silent
            out[key] = {"failed": repr(e)[:300]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--voices", type=int, default=VOICES_PER_GPU, help="voices per GPU (default: the BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity check of the timed runtime (exploration only)")
    ap.add_argument("--no-t1", action="store_true", help="skip the extra 131072-voices-per-GPU measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 3/4/5 leg (N = 1 only)")
    ap.add_argument("--specialize", type=int, default=2, help="K1 per-program specialisation: 0 interpreter, 2 NVRTC at COMMIT (default)")
    ap.add_argument("--collective", default="fused", choices=["fused", "nccl"], help="N > 1: K4 peer-memory kernel (default) or NCCL all_reduce")
    ap.add_argument("--tile-width", type=int, default=0, help="override the voices-per-warp heuristic (exploration only)")
    ap.add_argument("--opt", action="append", default=[], help="extra runtime option key=value (exploration only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the mix bus of the last timed step as DIR/mix.npy (and DIR/t1_mix.npy), see the module docstring")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm reports a checksum, not the rendered samples")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly ONE JSON line: anything a native library writes to fd 1 meanwhile (NCCL's banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    lines = []
    emit = lambda text: lines.append(text)
    try:
        if args.impl == "reference":
            run_reference(args, rank, world, emit)
        else:
            run_b200(args, rank, local_rank, world, emit)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for text in lines:
        print(text, flush=True)


if __name__ == "__main__":
    main()
