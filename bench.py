#!/usr/bin/env python
"""bench.py -- PBS/s for PARAM_MESSAGE_2_CARRY_2_KS_PBS, batch 4096 per GPU.

  python bench.py --gpus N --steps K --warmup W              (our arm)
  python bench.py --impl reference --gpus N --steps K --warmup W
      (the reference's CPU algorithm -- the oracle port -- on the host cores)

A "step" is one programmable bootstrap of the whole batch (4096 small-key LWE
ciphertexts per GPU, one shared identity LUT, trivial indexes) through
cuda_programmable_bootstrap_64_async.  `value` is timed on the device with
inputs resident in HBM; `e2e` is the same step through the reference-facing
ffi call (scratch -> run -> cleanup) with HOST buffers, H2D/D2H inside the
timed region.  One process per GPU; keys are replicated by one NCCL
broadcast; no collective in the timed region; max over ranks.

The GPU arm never touches oracle/: its keys and inputs are synthetic
(numpy, seeded).  Only the `cpu_baseline` leg and the post-run parity check
(rank 0, N = 1) load the oracle -- as the timed CPU baseline / the checker.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# PARAM_MESSAGE_2_CARRY_2_KS_PBS_TUNIFORM_2M128
# (tfhe/src/shortint/parameters/v1_4/classic/tuniform/p_fail_2_minus_128/ks_pbs.rs:29-47)
P22 = dict(n=918, k=1, N=2048, pbs_base_log=23, pbs_level=1, ks_base_log=4, ks_level=4)
BSK_BYTES_PER_PBS = 918 * 4 * 1 * 1024 * 16  # 60,162,048 (SURVEY.md 8d)
METRIC = "PBS/s (PARAM_MESSAGE_2_CARRY_2, batch 4096)"
# what tfhe-rs itself publishes for this PBS on CPU (BASELINE.md section 1): the calibration point of the port
PUBLISHED_CPU = {"ms_per_pbs_per_core": 5.64, "hardware": "1 thread of AWS hpc8a.96xlarge (EPYC 9R45), tfhe-fft AVX-512",
                 "source": "tfhe/docs/.gitbook/assets/cpu-pbs-benchmark-tuniform-2m128.svg:13"}
# fp64-pipe work of the PBS kernel: DADD+DFMA+DMUL warp instructions per CMUX per LWE (ncu instruction mix,
# profiles/); the pipe issues one DP warp instruction per 2 cycles per SM sub-partition on B200
DP_WARP_INSTR_PER_CMUX = 4960


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []  # (host time, line)
        self.t0 = self.t1 = None

    def start(self):
        """Start polling (before the warm-up: nvidia-smi needs a moment to come up)."""
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def samples_in_region(self) -> int:
        return sum(1 for t, _ in self.lines if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e300))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.lines:
            if self.t0 is not None and not (self.t0 <= t <= (self.t1 or 1e300)):
                continue
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
                power.append(float(parts[6]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def identity_lut(p: int = 16, N: int = 2048, delta: int = 1 << 59) -> np.ndarray:
    """generate_programmable_bootstrap_glwe_lut with f = id
    (core_crypto/algorithms/lwe_programmable_bootstrapping/mod.rs:26-83), k = 1."""
    from tfhe_rs_b200 import algorithms

    return algorithms.generate_programmable_bootstrap_glwe_lut(N, 2, p, delta, lambda x: x)


DUMP_ROWS = 1024  # x 2049 words in float64 = 16.8 MB per dump; the whole 4096-row batch would be 67 MB


def dump_outputs(directory: str, cts: np.ndarray) -> None:
    """Write the output LWE ciphertexts of the last timed step to
    `directory`/pbs_output.npy: a fixed sample of DUMP_ROWS rows (seed 0, kept
    in ascending order), every word as a signed torus value int64(word) / 2^64
    in float64, so that two builds can be compared output for output."""
    rows = np.sort(np.random.default_rng(0).choice(len(cts), size=min(DUMP_ROWS, len(cts)), replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "pbs_output.npy"), cts[rows].view(np.int64).astype(np.float64) / 2.0 ** 64)


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (oracle port; the Rust
    crate cannot be built here) on all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    P = O.PARAM_MESSAGE_2_CARRY_2_KS_PBS
    cores = O.max_threads()
    keys = O.keygen(P, 0xB2000001, with_ksk=False)
    keys.fourier_bsk()
    rng = O.Rng(2)
    lut = O.make_lut(P, list(range(16)))
    # calibrate on 4 PBS per thread; a step is the WHOLE 4096 batch (same config
    # as our arm) when K + W such steps fit ~150 s, else a bounded sample of it
    calib = max(cores * 4, 8)
    c_cts = O.lwe_encrypt_batch(rng, keys.lwe_sk, (np.arange(calib) % 16).astype(np.uint64) * np.uint64(P.delta),
                                P.lwe_noise_log2)
    O.pbs_batch(keys, lut, c_cts[: max(cores, 1)], threads=cores)
    t0 = time.perf_counter()
    O.pbs_batch(keys, lut, c_cts, threads=cores)
    rate = calib / (time.perf_counter() - t0)
    if args.batch * (args.steps + 1) / rate <= 150.0:
        sample = args.batch
    else:
        sample = int(min(args.batch, max(calib, round(rate * 150.0 / (args.steps + 1) / cores) * cores)))
    msgs = np.arange(sample) % 16
    cts = O.lwe_encrypt_batch(rng, keys.lwe_sk, msgs.astype(np.uint64) * np.uint64(P.delta), P.lwe_noise_log2)
    for _ in range(max(args.warmup, 1)):
        O.pbs_batch(keys, lut, cts[: max(cores, 1)], threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = O.pbs_batch(keys, lut, cts, threads=cores)
    dt = time.perf_counter() - t0
    ok = bool(np.array_equal(O.decode(O.lwe_decrypt_batch(keys.glwe_sk, out), P.delta, 16), msgs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    value = sample * args.steps / dt
    desc = (f"{sample} PBS per step (of the {args.batch}-batch workload), FFT-mode oracle port (restatement of "
            f"tfhe-rs fft64 PBS, not tfhe-rs itself), {cores} threads (affinity / cgroup count, OMP_NUM_THREADS ignored)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "PBS/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "shortint PBS batch=4096, PARAM_MESSAGE_2_CARRY_2_KS_PBS (N=2048)", **P22,
                   "sample_per_step": sample},
        "cpu_baseline": {"value": value, "unit": "PBS/s", "cores": cores, "kind": "port", "sample": desc,
                         "ms_per_pbs_per_core": 1e3 * cores / value, "decrypt_ok": ok,
                         "published_calibration": PUBLISHED_CPU},
        "e2e": {"value": value, "unit": "PBS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import tfhe_rs_b200
    from tfhe_rs_b200 import gpu, multi_gpu

    L = tfhe_rs_b200.lib()
    streams = gpu.CudaStreams.new_single_gpu(local_rank)
    stream = streams.streams[0]
    n, k, N, base_log, level = P22["n"], P22["k"], P22["N"], P22["pbs_base_log"], P22["pbs_level"]
    # weak scaling (default, what the driver's 1..8 sweep runs): `--batch` LWEs per GPU.
    # --scaling strong / --batch-global B: B LWEs in total, split over the ranks with the
    # reference's rule (helper_multi_gpu.cu:64-101).
    if args.scaling == "strong" or args.batch_global:
        global_batch = args.batch_global or args.batch
        batch = multi_gpu.get_num_inputs_on_gpu(global_batch, rank, world)
    else:
        global_batch = args.batch * world
        batch = args.batch
    bsk_words = n * (k + 1) * (k + 1) * level * N

    # ---- keys: rank 0 converts a synthetic standard-domain BSK, then ONE
    # NCCL broadcast replicates the Fourier key (60 MB) to every GPU --------
    if rank == 0:
        h_bsk = np.random.default_rng(0xB2000001).integers(0, 1 << 64, size=bsk_words, dtype=np.uint64)
        bsk = gpu.CudaLweBootstrapKey.from_lwe_bootstrap_key(
            h_bsk, n, k, N, base_log, level, gpu.CudaModulusSwitchNoiseReductionConfiguration.CENTERED, streams)
        del h_bsk
    else:
        bsk = gpu.CudaLweBootstrapKey(gpu.CudaVec.new(bsk_words, streams, np_dtype=np.float64), n, k, N, base_log,
                                      level, gpu.CudaModulusSwitchNoiseReductionConfiguration.CENTERED)
    key_bcast_ms = 0.0
    if world > 1:
        streams.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        multi_gpu.broadcast_vec(bsk.d_vec, bsk_words, np.float64, streams, src=0)
        key_bcast_ms = (time.perf_counter() - t0) * 1e3

    # ---- this rank's shard of the ciphertext list (weak scaling: `batch`
    # LWEs per GPU), uniform masks, messages s mod 16 ----------------------
    rng = np.random.default_rng(1000 + rank)
    h_in = rng.integers(0, 1 << 64, size=(batch, n + 1), dtype=np.uint64)
    h_lut = identity_lut()
    d_in = gpu.CudaLweCiphertextList.from_lwe_ciphertext_list(h_in, streams)
    d_lut = gpu.CudaGlweCiphertextList.from_glwe_ciphertext_list(h_lut, k, N, streams)
    d_out = gpu.CudaLweCiphertextList.new(k * N, batch, streams)
    d_idx = gpu.trivial_indexes(batch, streams)
    d_lut_idx = gpu.CudaVec.new(batch, streams)
    scratch = gpu.PbsScratch(streams, n, k, N, level, batch, centered=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=streams.device(0))  # > 126 MB L2
    gi, sp = local_rank, streams.ptr(0)

    def step_device():
        L.cuda_programmable_bootstrap_64_async(
            sp, gi, d_out.d_vec.as_c_ptr(), d_idx.as_c_ptr(), d_lut.d_vec.as_c_ptr(), d_lut_idx.as_c_ptr(),
            d_in.d_vec.as_c_ptr(), d_idx.as_c_ptr(), bsk.d_vec.as_c_ptr(), scratch.buf, n, k, N, base_log, level,
            batch, 1, 0)

    def sync_all():
        streams.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            flush.zero_()
            step_device()
    sync_all()

    # ---- timed region: exactly K steps, device events on the launch stream
    launches0 = L.b200_kernel_launch_count()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    sync_all()
    sampler.mark_begin()
    wall0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for i in range(args.steps):
            flush.zero_()  # L2 flush between timed iterations (256 MiB write)
            starts[i].record(stream)
            step_device()
            ends[i].record(stream)
    sync_all()
    wall_ms = (time.perf_counter() - wall0) * 1e3
    gpu_launches = L.b200_kernel_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        # read back before anything else reuses d_out (the KS+PBS extra below writes into it)
        dump_outputs(args.dump_outputs, d_out.to_lwe_ciphertext_list(streams))
    clock_note = "sampled during the timed steps"
    if sampler.samples_in_region() < 2:
        # a K-step region shorter than nvidia-smi's period: keep the same load
        # running (untimed) until the clocks have been read under it
        clock_note = "timed region shorter than the nvidia-smi period: sampled during extra untimed steps of the same load right after it"
        deadline = time.perf_counter() + 5.0
        while sampler.samples_in_region() < 2 and time.perf_counter() < deadline:
            with torch.cuda.stream(stream):
                step_device()
            streams.synchronize()
    sampler.mark_end()
    clocks = sampler.stop()
    clocks["note"] = clock_note
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = float(sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=streams.device(0))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = global_batch * args.steps / (total_ms / 1e3)

    # ---- e2e: the same step through the C ABI with HOST buffers: every step
    # copies its 4096 input LWEs from pinned host memory (cuda_memcpy_async_to_gpu),
    # bootstraps (cuda_programmable_bootstrap_64_async, scratch kept alive as the
    # reference's integer layer does) and copies the 4096 output LWEs back
    # (cuda_memcpy_async_to_cpu).  Two C-ABI streams / buffer sets alternate so
    # that step i+1's upload and step i-1's download overlap step i's kernel;
    # all K steps are inside the timed region, one host sync at the end. -------
    import ctypes as C

    e2e_steps = args.steps
    in_bytes, out_bytes = batch * (n + 1) * 8, batch * (k * N + 1) * 8
    sets = []
    for _ in range(2):
        st = L.cuda_create_stream_ffi(gi)
        buf = C.POINTER(C.c_int8)()
        L.scratch_cuda_programmable_bootstrap_64_async(st, gi, C.byref(buf), n, k, N, level, batch, True, 1)
        sets.append(dict(
            stream=st, scratch=buf,
            pin_in=torch.from_numpy(h_in.view(np.int64).copy()).pin_memory(),
            pin_out=torch.empty(batch * (k * N + 1), dtype=torch.int64).pin_memory(),
            d_in=torch.empty(batch * (n + 1), dtype=torch.int64, device=streams.device(0)),
            d_out=torch.empty(batch * (k * N + 1), dtype=torch.int64, device=streams.device(0))))

    def step_e2e(s):
        L.cuda_memcpy_async_to_gpu(s["d_in"].data_ptr(), s["pin_in"].data_ptr(), in_bytes, s["stream"], gi)
        L.cuda_programmable_bootstrap_64_async(
            s["stream"], gi, s["d_out"].data_ptr(), d_idx.as_c_ptr(), d_lut.d_vec.as_c_ptr(), d_lut_idx.as_c_ptr(),
            s["d_in"].data_ptr(), d_idx.as_c_ptr(), bsk.d_vec.as_c_ptr(), s["scratch"], n, k, N, base_log, level,
            batch, 1, 0)
        L.cuda_memcpy_async_to_cpu(s["pin_out"].data_ptr(), s["d_out"].data_ptr(), out_bytes, s["stream"], gi)

    def sync_sets():
        for s in sets:
            L.cuda_synchronize_stream(s["stream"], gi)

    sync_all()
    for s in sets:  # warm-up, one per set
        step_e2e(s)
    sync_sets()
    sync_all()
    ext = [torch.cuda.ExternalStream(int(s["stream"]), device=streams.device(0)) for s in sets]
    ev_start = torch.cuda.Event(enable_timing=True)
    ev_ends = [torch.cuda.Event(enable_timing=True) for _ in sets]
    ev_start.record(ext[0])
    for i in range(e2e_steps):
        step_e2e(sets[i % 2])
    for e, x in zip(ev_ends, ext):
        e.record(x)
    sync_sets()
    e2e_ms = max(ev_start.elapsed_time(e) for e in ev_ends)  # device clock, last stream to finish
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device=streams.device(0))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = global_batch * e2e_steps / (e2e_ms / 1e3)
    for s in sets:
        L.cleanup_cuda_programmable_bootstrap_64(s["stream"], gi, C.byref(s["scratch"]))
        L.cuda_destroy_stream(s["stream"], gi)
    scratch.close()

    # ---- extra (not the headline): the KS_PBS atomic pattern, keyswitch
    # kN -> n then PBS, on the same batch; synthetic KSK --------------------
    ks_ms = ks_pbs_ms = None
    if not args.no_extras:
        kl, kb = P22["ks_level"], P22["ks_base_log"]
        h_ksk = np.random.default_rng(7).integers(0, 1 << 64, size=k * N * kl * (n + 1), dtype=np.uint64)
        ksk = gpu.CudaLweKeyswitchKey.from_lwe_keyswitch_key(h_ksk, k * N, n, kb, kl, streams)
        del h_ksk
        h_big = rng.integers(0, 1 << 64, size=(batch, k * N + 1), dtype=np.uint64)
        d_big = gpu.CudaLweCiphertextList.from_lwe_ciphertext_list(h_big, streams)
        scratch2 = gpu.PbsScratch(streams, n, k, N, level, batch, centered=True)

        def step_ks():
            L.cuda_keyswitch_gemm_64_64_async(sp, gi, d_in.d_vec.as_c_ptr(), d_idx.as_c_ptr(),
                                              d_big.d_vec.as_c_ptr(), d_idx.as_c_ptr(), ksk.d_vec.as_c_ptr(),
                                              k * N, n, kb, kl, batch, True)

        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(stream):
            step_ks()
            flush.zero_()
            evs[0].record(stream)
            step_ks()
            evs[1].record(stream)
            flush.zero_()
            evs[2].record(stream)
            step_ks()
            L.cuda_programmable_bootstrap_64_async(
                sp, gi, d_out.d_vec.as_c_ptr(), d_idx.as_c_ptr(), d_lut.d_vec.as_c_ptr(), d_lut_idx.as_c_ptr(),
                d_in.d_vec.as_c_ptr(), d_idx.as_c_ptr(), bsk.d_vec.as_c_ptr(), scratch2.buf, n, k, N, base_log,
                level, batch, 1, 0)
            evs[3].record(stream)
        sync_all()
        ks_ms = evs[0].elapsed_time(evs[1])
        ks_pbs_ms = evs[2].elapsed_time(evs[3])
        scratch2.close()

    # ---- extras, rank 0 at N = 1: the other BASELINE configs that fit one GPU, as
    # driver-visible numbers -- configs[2] multi-bit g=3 batch 4096 and configs[3]
    # FheUint64 x FheUint64 (32 blocks, full KS+PBS cascade) ----------------
    other_configs = None
    if not args.no_extras and world == 1:
        other_configs = other_config_measurements(L, gpu, streams, torch, flush)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- the kernel to beat on the SAME box: the reference's own CUDA backend
    # (oracle/_ref, built unmodified for sm_100) through the same C-ABI harness,
    # in its own process (tools/ab_bench.py --lib ref) -------------------------
    reference_gpu = None
    if world == 1 and not args.no_reference_gpu:
        reference_gpu = reference_gpu_measurements(args)

    peak, peak_src = measured_hbm_peak()
    kernel_ms = float(np.mean(step_ms))
    achieved = BSK_BYTES_PER_PBS * batch / (kernel_ms / 1e3) / 1e9
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": args.traffic_bytes, "kernel": "pbs_n2048_k1_l1_v6_kernel<2, true, 2, 1> (tensor-memory exchange 2 + TMA key ring, see DESIGN.md section 4)",
        "algorithmic_bytes_per_launch": BSK_BYTES_PER_PBS * batch,
        "note": f"peak = {peak_src}; algorithmic bytes = Fourier BSK streamed once per PBS; the BSK (57 MiB) is "
                "L2 resident and shared by the batch, so DRAM traffic is far below the algorithmic figure; the "
                "kernel is fp64-pipe bound (see `secondary` and DESIGN.md)",
    }
    # the ceiling that actually binds (SURVEY 8d "secondary ceiling"): fp64 pipe.  DP warp instructions per
    # launch (counted by ncu: DADD+DFMA+DMUL, profiles/) / launch time, against 1 DP warp instruction per
    # 2 cycles per sub-partition x 4 x SMs at the SM clock sampled during the timed region.
    sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    sms = L.cuda_get_number_of_sms()
    dp_instr = DP_WARP_INSTR_PER_CMUX * n * batch
    dp_peak = sms * 4 * 0.5 * sm_mhz * 1e6
    roofline["secondary"] = {
        "bound": "fp64", "achieved": dp_instr / (kernel_ms / 1e3) / 1e9, "peak": dp_peak / 1e9,
        "unit": "G DP warp-instr/s", "frac": dp_instr / (kernel_ms / 1e3) / dp_peak,
        "source": f"{DP_WARP_INSTR_PER_CMUX} DP warp instructions per CMUX per LWE (ncu instruction mix of the shipped "
                  f"kernel, profiles/) x n x batch; peak = {sms} SMs x 4 sub-partitions x 0.5 instr/cycle x "
                  f"{sm_mhz:.0f} MHz (sampled); ncu's sm__pipe_fp64_cycles_active of the committed capture is in "
                  "profiles/traffic.json",
        "ncu": traffic_json(),
    }

    cpu_baseline, parity = None, None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, parity = cpu_baseline_and_parity(streams, args)

    line = {
        "metric": METRIC, "value": value, "unit": "PBS/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if (args.scaling == "strong" or args.batch_global) else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "shortint PBS batch=4096 per GPU, PARAM_MESSAGE_2_CARRY_2_KS_PBS (N=2048), "
                               "centered-mean modulus switch, one shared identity LUT",
                   **P22, "batch_per_gpu": batch, "global_batch": batch * world,
                   "parallelism": f"batch-sharded x{world}, keys replicated by 1 NCCL broadcast",
                   "l2": "device-timed steps: L2 flushed between steps (256 MiB write), BSK 57 MiB re-read from L2 "
                         "inside a step; e2e steps: not flushed, each step moves 97 MB of host I/O + the 60 MB key "
                         "(> 126 MB L2)",
                   "key_broadcast_ms": key_bcast_ms},
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "e2e": {"value": e2e_value, "unit": "PBS/s", "h2d_bytes_per_step": int(batch * (n + 1) * 8),
                "d2h_bytes_per_step": int(batch * (k * N + 1) * 8), "steps": e2e_steps,
                "api": "C ABI: cuda_memcpy_async_to_gpu -> cuda_programmable_bootstrap_64_async -> cuda_memcpy_async_to_cpu on "
                       "two alternating streams (cuda_create_stream_ffi), pinned host buffers; timed with CUDA events "
                       "recorded on those streams: first upload enqueued -> last download complete, all K steps "
                       "inside, max over the two streams and over ranks"},
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
        "wall_ms_timed_region": wall_ms,
        "step_ms": [round(float(x), 3) for x in step_ms],  # this rank's K timed steps, one by one
        "parity_check": parity,
        "extras": {"keyswitch_ms_per_batch": ks_ms, "ks_pbs_ms_per_batch": ks_pbs_ms,
                   "ks_pbs_per_s_this_rank": (batch / (ks_pbs_ms / 1e3)) if ks_pbs_ms else None,
                   "other_configs": other_configs},
        "reference_gpu": reference_gpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def traffic_json():
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def other_config_measurements(L, gpu, streams, torch, flush):
    """BASELINE configs[2] (multi-bit g=3, batch 4096) and configs[3] (FheUint64 x
    FheUint64) on this GPU, synthetic keys, CUDA events / host clock.  Side
    numbers: not the headline metric."""
    out = {}
    stream = streams.streams[0]
    rng = np.random.default_rng(3)
    try:
        n, k, N, bl, lv, g, batch = 918, 1, 2048, 15, 2, 3, 4096
        num_ggsw = (n // g) << g
        h = rng.integers(0, 1 << 64, size=num_ggsw * lv * 4 * N, dtype=np.uint64)
        mb = gpu.CudaLweMultiBitBootstrapKey.from_lwe_multi_bit_bootstrap_key(h, n, k, N, bl, lv, g, streams)
        del h
        d_in = gpu.CudaLweCiphertextList.from_lwe_ciphertext_list(
            rng.integers(0, 1 << 64, size=(batch, n + 1), dtype=np.uint64), streams)
        d_out = gpu.CudaLweCiphertextList.new(k * N, batch, streams)
        d_lut = gpu.CudaGlweCiphertextList.from_glwe_ciphertext_list(identity_lut(), k, N, streams)
        idx, lidx = gpu.trivial_indexes(batch, streams), gpu.CudaVec.new(batch, streams)
        sc = gpu.PbsScratch(streams, n, k, N, lv, batch, centered=False, multi_bit=True)

        def run():
            L.cuda_multi_bit_programmable_bootstrap_64_async(
                streams.ptr(0), streams.gpu_indexes[0],
                d_out.d_vec.as_c_ptr(), idx.as_c_ptr(), d_lut.d_vec.as_c_ptr(), lidx.as_c_ptr(),
                d_in.d_vec.as_c_ptr(), idx.as_c_ptr(), mb.d_vec.as_c_ptr(), sc.buf, n, k, N, g, bl, lv, batch, 1, 0)

        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(3)]
        with torch.cuda.stream(stream):
            run()
            for s_, e_ in evs:
                flush.zero_()
                s_.record(stream)
                run()
                e_.record(stream)
        streams.synchronize()
        ms = float(np.median([s_.elapsed_time(e_) for s_, e_ in evs]))
        sc.close()
        del mb
        out["multi_bit_g3_batch4096"] = {
            "config": "multi-bit PBS batch=4096, PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3 (n=918,N=2048,l=2,logB=15)",
            "ms_per_step": ms, "pbs_per_s": batch / ms * 1e3}
    except Exception as e:  # side measurement: never take the headline down
        out["multi_bit_g3_batch4096"] = {"error": repr(e)}
    # two more classic parameter sets, each on its own register kernel:
    # PARAM_MESSAGE_1_CARRY_1_KS_PBS (n=879, k=4, N=512, l=1; csrc/pbs_n512.cuh) at batch 4096 and
    # PARAM_MESSAGE_3_CARRY_3_KS_PBS (n=1077, k=1, N=8192, l=2; csrc/pbs_n8192.cuh) at batch 592
    for key, (n, k, N, bl, lv, batch), what in (
            ("param_message_1_carry_1_batch4096", (879, 4, 512, 23, 1, 4096),
             "PARAM_MESSAGE_1_CARRY_1_KS_PBS (n=879,k=4,N=512,l=1,logB=23), register kernel pbs_n512_kernel "
             "(not a BASELINE config; reference CUDA backend on a B200: 16.5 k PBS/s, profiles/round2.md)"),
            ("param_message_3_carry_3_batch592", (1077, 1, 8192, 15, 2, 592),
             "PARAM_MESSAGE_3_CARRY_3_KS_PBS (n=1077,k=1,N=8192,l=2,logB=15), tensor-memory register kernel "
             "pbs_n8192_k1_l2_v2_kernel (not a BASELINE config; reference CUDA backend on a B200: 0.68 k PBS/s, "
             "profiles/round2.md)")):
        try:
            h = rng.integers(0, 1 << 64, size=n * (k + 1) * (k + 1) * lv * N, dtype=np.uint64)
            sb = gpu.CudaLweBootstrapKey.from_lwe_bootstrap_key(h, n, k, N, bl, lv, "Centered", streams)
            del h
            d_in = gpu.CudaLweCiphertextList.from_lwe_ciphertext_list(
                rng.integers(0, 1 << 64, size=(batch, n + 1), dtype=np.uint64), streams)
            d_out = gpu.CudaLweCiphertextList.new(k * N, batch, streams)
            lut_x = np.zeros((k + 1) * N, dtype=np.uint64)
            lut_x[k * N:] = np.repeat(np.arange(4, dtype=np.uint64) << np.uint64(61), N // 4)
            d_lut = gpu.CudaGlweCiphertextList.from_glwe_ciphertext_list(lut_x, k, N, streams)
            idx, lidx = gpu.trivial_indexes(batch, streams), gpu.CudaVec.new(batch, streams)
            sc = gpu.PbsScratch(streams, n, k, N, lv, batch, centered=True)

            def run_x():
                L.cuda_programmable_bootstrap_64_async(
                    streams.ptr(0), streams.gpu_indexes[0], d_out.d_vec.as_c_ptr(), idx.as_c_ptr(),
                    d_lut.d_vec.as_c_ptr(), lidx.as_c_ptr(), d_in.d_vec.as_c_ptr(), idx.as_c_ptr(),
                    sb.d_vec.as_c_ptr(), sc.buf, n, k, N, bl, lv, batch, 1, 0)

            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(3)]
            with torch.cuda.stream(stream):
                run_x()
                for s_, e_ in evs:
                    flush.zero_()
                    s_.record(stream)
                    run_x()
                    e_.record(stream)
            streams.synchronize()
            ms = float(np.median([s_.elapsed_time(e_) for s_, e_ in evs]))
            sc.close()
            del sb, d_in, d_out
            out[key] = {"config": "classic PBS batch=%d, %s" % (batch, what),
                        "ms_per_step": ms, "pbs_per_s": batch / ms * 1e3}
        except Exception as e:
            out[key] = {"error": repr(e)}
    try:
        from tfhe_rs_b200 import integer, server_key

        n, k, N = 918, 1, 2048
        h_bsk = rng.integers(0, 1 << 64, size=n * 4 * N, dtype=np.uint64)
        h_ksk = rng.integers(0, 1 << 64, size=k * N * 4 * (n + 1), dtype=np.uint64)
        skey = server_key.upload_server_key(h_bsk, h_ksk, n=n, k=k, N=N, pbs_base_log=23, pbs_level=1,
                                            ks_base_log=4, ks_level=4, centered_ms=True, streams=streams)
        luts = rng.integers(0, 1 << 64, size=(len(integer.lut_functions()), 2 * N), dtype=np.uint64)
        rsk = integer.CudaRadixServerKey(skey, luts, k, N)
        mk = lambda: integer.CudaUnsignedRadixCiphertext(
            rsk.engine.from_numpy(rng.integers(0, 1 << 64, size=(32, k * N + 1), dtype=np.uint64)))
        a, b = mk(), mk()
        rsk.unchecked_mul(a, b)
        streams.synchronize()
        rsk.engine.pbs_count = 0
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            rsk.unchecked_mul(a, b)
        streams.synchronize()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        out["fheuint64_mul"] = {"config": "FheUint64 x FheUint64 (32-block radix, full KS+PBS cascade), 1 GPU",
                                "latency_ms": dt * 1e3, "pbs_per_mul": rsk.engine.pbs_count // reps,
                                "timing": "host clock around 3 back-to-back multiplications, synchronised"}
        del skey, rsk
    except Exception as e:
        out["fheuint64_mul"] = {"error": repr(e)}
    try:
        # same cascade on the reference's GPU default multi-bit set (what its published 31.9 ms / 8xH100 uses)
        from tfhe_rs_b200 import integer, server_key

        n, k, N, g = 920, 1, 2048, 4
        h_bsk = rng.integers(0, 1 << 64, size=((n // g) << g) * 4 * N, dtype=np.uint64)
        h_ksk = rng.integers(0, 1 << 64, size=k * N * 5 * (n + 1), dtype=np.uint64)
        skey = server_key.upload_server_key(h_bsk, h_ksk, n=n, k=k, N=N, pbs_base_log=22, pbs_level=1,
                                            ks_base_log=3, ks_level=5, grouping_factor=g, centered_ms=False,
                                            streams=streams)
        del h_bsk
        luts = rng.integers(0, 1 << 64, size=(len(integer.lut_functions()), 2 * N), dtype=np.uint64)
        rsk = integer.CudaRadixServerKey(skey, luts, k, N)
        mk = lambda: integer.CudaUnsignedRadixCiphertext(
            rsk.engine.from_numpy(rng.integers(0, 1 << 64, size=(32, k * N + 1), dtype=np.uint64)))
        a, b = mk(), mk()
        rsk.unchecked_mul(a, b)
        streams.synchronize()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            rsk.unchecked_mul(a, b)
        streams.synchronize()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        out["fheuint64_mul_multi_bit_g4"] = {
            "config": "FheUint64 x FheUint64, PARAM_GPU_MULTI_BIT_GROUP_4_MESSAGE_2_CARRY_2 (n=920,l=1,logB=22), 1 GPU",
            "latency_ms": dt * 1e3, "timing": "host clock around 3 back-to-back multiplications, synchronised"}
    except Exception as e:
        out["fheuint64_mul_multi_bit_g4"] = {"error": repr(e)}
    return out


def reference_gpu_measurements(args):
    """The reference's CUDA backend on this GPU, same harness (tools/ab_bench.py)."""
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libtfhe_cuda_backend_ref.so")
    if not os.path.exists(ref_so):
        return {"unavailable": "oracle/_ref/libtfhe_cuda_backend_ref.so not built (oracle/build_ref_cuda.sh)"}
    env = dict(os.environ)
    for key in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "B200_LIB_PATH"):
        env.pop(key, None)
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ab_bench.py"), "--lib", "ref", "--what",
                            "classic,ks,multibit3,multibit4", "--batches", "1,4096", "--steps", "3"],
                           capture_output=True, text=True, env=env, timeout=600)
    except Exception as e:
        return {"error": repr(e)}
    rows = []
    for ln in r.stdout.splitlines():
        try:
            rows.append(json.loads(ln))
        except Exception:
            pass
    if r.returncode != 0 and not rows:
        return {"error": (r.stderr or r.stdout)[-600:]}
    head = next((x for x in rows if x.get("what", "").startswith("classic") and x.get("batch") == 4096), None)
    return {"library": "oracle/_ref/libtfhe_cuda_backend_ref.so (reference sources unmodified, nvcc sm_100, "
                       "--use_fast_math as in its CMakeLists)",
            "kernel": "device_programmable_bootstrap_specialized_2_2_params_throughput (library's own dispatch)",
            "pbs_per_s": head["pbs_per_s"] if head else None, "ms_per_step": head["ms"] if head else None,
            "batch": 4096, "timing": "CUDA events on the launch stream, L2 flushed, same synthetic key and inputs "
                                     "as tools/ab_bench.py --lib ours",
            "measurements": rows, "returncode": r.returncode}


def cpu_baseline_and_parity(streams, args):
    """Rank 0, N = 1 only.  (a) the oracle's FFT-mode PBS on all host cores on
    a bounded sample of the same workload; (b) the oracle as the checker: real
    keys, GPU KS->PBS on 64 samples must decrypt like the oracle's."""
    from oracle import oracle as O
    from tfhe_rs_b200 import gpu, server_key

    P = O.PARAM_MESSAGE_2_CARRY_2_KS_PBS
    cores = O.max_threads()
    keys = O.keygen(P, 0xB2000001)
    keys.fourier_bsk()
    rng = O.Rng(2)
    lut = O.make_lut(P, list(range(16)))
    # calibrate on 4 PBS per thread, then time ~12 s of wall time (capped at the full 4096 batch)
    calib = max(cores * 4, 8)
    c_big = O.lwe_encrypt_batch(rng, keys.glwe_sk, (np.arange(calib) % 16).astype(np.uint64) * np.uint64(P.delta),
                                P.lwe_noise_log2)
    c_small = O.keyswitch_batch(keys, c_big)
    O.pbs_batch(keys, lut, c_small[:cores], threads=cores)  # warm-up
    t0 = time.perf_counter()
    O.pbs_batch(keys, lut, c_small, threads=cores)
    rate = calib / (time.perf_counter() - t0)
    sample = int(min(4096, max(64, round(rate * 12.0 / cores) * cores)))
    msgs = np.arange(sample) % 16
    big = O.lwe_encrypt_batch(rng, keys.glwe_sk, msgs.astype(np.uint64) * np.uint64(P.delta), P.lwe_noise_log2)
    small = O.keyswitch_batch(keys, big)
    t0 = time.perf_counter()
    ref = O.pbs_batch(keys, lut, small, threads=cores)
    dt = time.perf_counter() - t0
    base = {"value": sample / dt, "unit": "PBS/s", "cores": cores, "kind": "port",
            "sample": f"{sample} PBS of the 4096-batch workload, oracle FFT mode (restatement of tfhe-rs "
                      f"fft64 PBS, not tfhe-rs itself), {cores} threads, {dt:.2f} s",
            "ms_per_pbs_per_core": dt * 1e3 * cores / sample, "published_calibration": PUBLISHED_CPU}
    skey = server_key.upload_server_key(keys.bsk, keys.ksk, n=P.n, k=P.k, N=P.N, pbs_base_log=P.pbs_base_log,
                                        pbs_level=P.pbs_level, ks_base_log=P.ks_base_log, ks_level=P.ks_level,
                                        centered_ms=True, streams=streams)
    d_big = gpu.CudaLweCiphertextList.from_lwe_ciphertext_list(big[:64], streams)
    d_lut = gpu.CudaGlweCiphertextList.from_glwe_ciphertext_list(lut, 1, 2048, streams)
    d_small = skey.keyswitch(d_big)
    got = skey.bootstrap(d_small, d_lut).to_lwe_ciphertext_list(streams)
    ks_exact = bool(np.array_equal(d_small.to_lwe_ciphertext_list(streams), small[:64]))
    dec = O.decode(O.lwe_decrypt_batch(keys.glwe_sk, got), P.delta, 16)
    dec_ref = O.decode(O.lwe_decrypt_batch(keys.glwe_sk, ref[:64]), P.delta, 16)
    parity = {"samples": 64, "keyswitch_bit_exact": ks_exact,
              "pbs_decrypt_equal": bool(np.array_equal(dec, dec_ref) and np.array_equal(dec, msgs[:64]))}
    return base, parity


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--batch", type=int, default=4096, help="LWE ciphertexts per GPU (BASELINE: 4096)")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: --batch LWEs per GPU (default); strong: --batch LWEs in total, split over the GPUs")
    ap.add_argument("--batch-global", type=int, default=0,
                    help="total LWEs over all GPUs (BASELINE configs[4]: 65536 over 8); implies strong scaling")
    ap.add_argument("--no-reference-gpu", action="store_true",
                    help="skip timing the reference's CUDA backend (oracle/_ref) on this GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the keyswitch / KS+PBS side measurement")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch of the PBS kernel from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the PBS outputs of the last timed step (rank 0) to DIR/pbs_output.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.traffic_bytes is None:
            p = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(p):
                try:
                    args.traffic_bytes = json.load(open(p)).get("pbs_n2048_k1_l1_kernel_dram_bytes_per_launch")
                except Exception:
                    pass
        run_b200(args)


if __name__ == "__main__":
    main()
