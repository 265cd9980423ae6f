#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on B200: generated audio samples per second
(22.05 kHz) of batched MoL WaveRNN.generate(), BASELINE.json configs[1]:
a 10-second 80-bin mel (T=800 frames) folded with target=11000 / overlap=550 into 19 folds x
12,100 steps, rnn_dims=512, random-init weights, synthetic mel.

    python bench.py --gpus 1 --steps 5 --warmup 3            # this framework (CUDA engine)
    python bench.py --impl reference --steps 2 --warmup 1    # the reference algorithm on host cores
    torchrun ... bench.py --gpus N ...                       # N ranks, folds sharded, weak scaling

One "step" = one full pass of the hot path over the workload (all folds x all steps).
`value`  : fold-samples generated per second, inputs (upsampled conditioning, RNG draws)
           resident in HBM, timed with CUDA events on the launching stream, max over ranks.
`e2e`    : the same metric through the public call WaveRNN.generate(host mel, ...) including
           H2D of the mel and of the reference-compatible RNG draws, the conditioning network,
           the kernel, D2H of the samples and the host epilogue (xfade/unfold), wall clock.
N > 1    : weak scaling -- the mel is lengthened so every rank owns 19 folds; one NCCL
           all-gather of the sample blocks is inside the timed region.
--dump-outputs DIR : after the timing, what the timed path returned in its last step, as DIR/<name>.npy (see
           dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FLOP_PER_SAMPLE_MOL = 7_650_304          # SURVEY.md 8(d): 3,825,152 MAC per fold-sample
BYTES_PER_SAMPLE = 836                   # 208 fp32 conditioning values in + 1 fp32 sample out
TARGET, OVERLAP, HOP = 11_000, 550, 275
FOLDS_PER_GPU = 19
CTOR = dict(rnn_dims=512, fc_dims=512, bits=9, pad=2, upsample_factors=(5, 5, 11), feat_dims=80,
            compute_dims=128, res_out_dims=128, res_blocks=10, hop_length=HOP, sample_rate=22050, mode='MOL')


def frames_for(n_gpus: int) -> int:
    """Mel frames giving exactly 19 folds per GPU with no padding (N=1 -> 800)."""
    L = FOLDS_PER_GPU * n_gpus * (TARGET + OVERLAP) + OVERLAP
    assert L % HOP == 0
    return L // HOP


def workload_config(world: int, workload: str = "cfg2", folds5: int = 4096) -> dict:
    """The `config` object BOTH arms print (identical for the same --gpus / --workload, so the driver's same_config
    check compares like with like)."""
    if workload == "cfg5":
        T5 = 42 * folds5 + 2                  # exactly `folds5` folds, no padding: L = folds5 * 11550 + 550 = T5 * 275
        return {"workload": f"cfg5: mel T={T5} frames ({T5 * HOP / 22050 / 60:.1f} min) -> {folds5} folds x 12100 steps, target=11000 overlap=550, "
                            "MoL head, rnn_dims=512, random-init weights (seed 0), torch.rand mel (seed 0)", "folds": folds5, "steps_per_fold": 12100}
    T = frames_for(world)
    head = {"cfg2": "MoL head", "cfg3": "RAW head (bits=9, mu-law)"}[workload]
    return {"workload": f"{workload} x{world}: mel T={T} frames ({T * HOP / 22050:.1f} s) -> {FOLDS_PER_GPU * world} folds x 12100 steps "
                        f"({FOLDS_PER_GPU} folds per GPU), target={TARGET} overlap={OVERLAP}, {head}, rnn_dims=512, random-init weights "
                        f"(seed 0), torch.rand mel (seed 0), sampler seed 1234",
            "folds": FOLDS_PER_GPU * world, "steps_per_fold": 12100}


def build_model(device, mode="MOL"):
    from wavernn_b200 import WaveRNN
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = WaveRNN(**dict(CTOR, mode=mode))
    m.gen_verbose = False
    return m.to(device)


def measured_traffic(args, model):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel on this workload, taken from
    the committed ncu --set full capture (profiles/r02_tc_traffic.json, else round 1's); None when no capture matches."""
    if args.workload != "cfg2" or args.seg_steps:
        return None
    for name in ("r02_tc_traffic.json", "r01_tc_traffic.json"):
        p = ROOT / "profiles" / name
        if p.is_file():
            d = json.loads(p.read_text())
            if str(d.get("engine", "")).startswith("tcgen05"):
                return d.get("dram_bytes_per_launch")
    return None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.is_file():
        d = json.loads(p.read_text())
        return dict(tflops=float(d["bf16_tflops"]), tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    hbm_gbs=float(d["hbm_gbs"]), src="measured")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, src="fallback")


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict):
    """Writes every array as out_dir/<name>.npy (float32 stays float32, everything else becomes float64).  When they
    come to more than 64 MB together, each is replaced by the same share of its entries (flattened, sorted indices
    drawn from a fixed seed), so two runs with the same arguments store the same entries."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            k = a.size * DUMP_LIMIT_BYTES // total
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, size=k, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port on torch CPU operators) on the host cores
# ------------------------------------------------------------------------------------------
def cpu_conditioning(model_cpu, mel):
    with torch.no_grad():
        model_cpu.eval()
        mp = torch.nn.functional.pad(mel, (2, 2))
        m_up, aux = model_cpu.upsample(mp)
        mels_f = model_cpu.fold_with_overlap(m_up, TARGET, OVERLAP)
        aux_f = model_cpu.fold_with_overlap(aux, TARGET, OVERLAP)
    return mels_f, aux_f


def time_cpu_port(sample_steps: int):
    """cpu_baseline leg of the GPU arm: the port of the reference loop on a bounded sample (first `sample_steps` steps of
    all 19 folds), best thread count of a sweep."""
    from oracle import torch_port
    threads, sweep, (sd, mels_f, aux_f) = best_cpu_threads(FOLDS_PER_GPU)
    torch.set_num_threads(threads)
    torch.manual_seed(1234)
    _, dt = torch_port.generate_segments_torch(sd, mels_f, aux_f, steps=sample_steps)
    return dict(B=mels_f.shape[0], steps=sample_steps, seconds=[dt], cores=threads, threads=threads,
                host_cores=os.cpu_count() or 1, sweep=sweep)


def best_cpu_threads(folds: int):
    """The loop is small-batch GEMVs: torch's default (all cores) oversubscribes badly on a many-core host (128 threads:
    ~40x slower than 8).  Both the port and the unmodified reference get the best thread count of a short sweep."""
    from oracle import torch_port
    cores = os.cpu_count() or 1
    model = build_model("cpu")
    torch.manual_seed(0)
    mel = torch.rand(1, 80, frames_for(max(1, folds // FOLDS_PER_GPU)))
    mels_f, aux_f = cpu_conditioning(model, mel)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    trials = {}
    for n in sorted({min(cores, c) for c in (4, 8, 16, 32, 64, cores)}):
        torch.set_num_threads(n)
        torch.manual_seed(1234)
        _, dt = torch_port.generate_segments_torch(sd, mels_f, aux_f, steps=40)
        trials[n] = dt
    best = min(trials, key=trials.get)
    return best, {str(k): round(40 * mels_f.shape[0] / v, 1) for k, v in trials.items()}, (sd, mels_f, aux_f)


def run_reference_arm(args):
    """bench.py --impl reference: the reference's own CPU implementation of the path on this box's host cores.
    With oracle/_ref (oracle/make_ref.py: the unmodified reference files) it is the reference's `WaveRNN.generate()`
    itself, end to end, all 12,100 steps of all folds (`kind: "reference"`); otherwise the torch-operator port of its loop
    (`kind: "port"`, bit-identical samples, tests/test_oracle_vs_reference.py).  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    cfg = workload_config(world, "cfg2")
    folds, S = cfg["folds"], cfg["steps_per_fold"]
    threads, sweep, (sd, mels_f, aux_f) = best_cpu_threads(folds)
    torch.set_num_threads(threads)
    sys.path.insert(0, str(ROOT / "oracle"))
    import make_ref
    use_ref = make_ref.verify()
    # one bench step = one pass over the workload; at N > 1 the CPU pass is bounded to 12100 // N steps of every fold
    # (the same number of fold-steps as at N = 1) so that a --steps K run still ends within minutes
    sample_steps = S if world == 1 else max(1210, S // world)
    times = []
    on_cuda = args.ref_device == "cuda"
    if on_cuda and not (use_ref and world == 1 and torch.cuda.is_available()):
        raise SystemExit("--ref-device cuda needs oracle/_ref, --gpus 1 and a CUDA device")
    if use_ref and world == 1:
        os.environ["WAVERNN_REFERENCE"] = str(ROOT / "oracle" / "_ref")
        from oracle import ref_shim
        ref_shim.REF_ROOT = str(ROOT / "oracle" / "_ref")
        model = ref_shim.build_reference_model(seed=0, mode="MOL")
        if on_cuda:                 # extra datapoint (not the driver's arm): the unmodified reference's eager CUDA path on this GPU
            model = model.to("cuda")
        torch.manual_seed(0)
        mel = torch.rand(1, 80, frames_for(world))
        for i in range(args.warmup + args.steps):
            torch.manual_seed(1234)
            t0 = time.perf_counter()
            wav = model.generate(mel, "/dev/null.wav", True, TARGET, OVERLAP, False)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
        assert len(wav) == (frames_for(world) - 1) * HOP
        outputs = {"wav": np.asarray(wav)}
        kind = "reference"
        how = ("UNMODIFIED reference WaveRNN.generate() (oracle/_ref, " + ("eager torch CUDA operators on this GPU" if on_cuda else "CPU") +
               ", fp32), whole call: upsample network + fold + 12100-step loop + xfade")
    else:
        from oracle import torch_port
        for i in range(args.warmup + args.steps):
            torch.manual_seed(1234)
            samples, dt = torch_port.generate_segments_torch(sd, mels_f, aux_f, steps=sample_steps)
            if i >= args.warmup:
                times.append(dt)
        outputs = {"samples": np.asarray(samples)}
        kind = "port"
        how = "torch-operator port of the reference loop (oracle/torch_port.py; bit-identical samples), loop only"
    per_step = float(np.mean(times))
    value = folds * sample_steps / per_step
    sample = (f"{folds} folds x {sample_steps} of {S} steps per bench step; {how}; {threads} torch threads (best of sweep, samples/s by "
              f"threads: {sweep}) on {os.cpu_count()} host cores")
    line = {"impl": "reference", "metric": "audio samples/sec (22.05 kHz) batched MoL generate", "value": value,
            "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg, "reference_device": args.ref_device,
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "x_realtime": value / 22050.0}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    emit(line)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from wavernn_b200.sharding import fold_geometry, gather_segments, shard_folds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    if args.workload == "cfg4":
        return run_cfg4(args, device, rank, world, local)
    cfg3 = args.workload == "cfg3"                     # BASELINE configs[2]: cfg2's mel with the 9-bit RAW head (mu-law)
    model = build_model(device, "RAW" if cfg3 else "MOL")
    model.gen_precision, model.gen_engine = args.precision, args.engine
    cfg5 = args.workload == "cfg5"
    if cfg3:
        model.gen_rng = "philox"                       # (parity mode would stream 471 MB of Exp(1) draws per call)
    if cfg5:
        # BASELINE configs[4] (SURVEY 8d choice A): T=172,034 frames = 35.8 min -> exactly 4096 folds with the
        # reference's own target/overlap; the 4096 folds are sharded over the ranks (strong scaling); in-kernel RNG
        model.gen_rng = "philox"
    T = (42 * args.cfg5_folds + 2) if cfg5 else frames_for(world)
    torch.manual_seed(0)
    mel_host = torch.rand(1, 80, T).pin_memory()
    geo = fold_geometry(T * HOP, TARGET, OVERLAP)
    shard = shard_folds(geo, rank, world, HOP)
    B_total, S = geo.n_seg, geo.seg_len

    # ---- resident inputs for the device-timed region: exactly what WaveRNN.generate() hands to the library by default
    # (frame-rate conditioning: padded mel, MelResNet frames, 5-tap table; the library forms the x275 rows itself) ------
    model.eval()
    with torch.no_grad():
        mp = torch.nn.functional.pad(mel_host.to(device), (2, 2))
        mel_fr = mp[0].transpose(0, 1).contiguous().float()
        aux_fr = model.upsample.resnet(mp)[0].transpose(0, 1).contiguous().float()
        taps = model.upsample_taps(device)
    f0, n = shard.seg_first, shard.n_seg
    if cfg5 or cfg3:
        u_all, uni_ptr, h2d_rng = None, 0, 0
    else:
        torch.manual_seed(1234)
        u_all, _ = model._reference_draws(geo, S)
        uni = torch.cat([u_all[:, 10 * f0:10 * (f0 + n)], u_all[:, 10 * B_total + f0:10 * B_total + f0 + n]], 1).contiguous().to(device)
        uni_ptr, h2d_rng = uni.data_ptr(), u_all.numel() * 4
    out = torch.empty((n, S), dtype=torch.float32, device=device)
    engine = model._get_engine(device)
    stream = torch.cuda.current_stream(device)

    def device_step():
        engine.generate(mels_up=0, aux=0, L=T * HOP, n_seg=n, seg_len=S, seg_stride=geo.seg_stride, out=out.data_ptr(),
                        seg_first=f0, uniforms=uni_ptr, steps=args.seg_steps, mel_frames=mel_fr.data_ptr(),
                        aux_frames=aux_fr.data_ptr(), up_taps=taps.data_ptr(), hop=HOP, cond_mode=0, stream=stream.cuda_stream)
        if world > 1:
            return gather_segments(out, shard, geo)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(args.warmup):
        device_step()
    barrier(); engine.check()
    launches0 = engine.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    with ClockSampler(local) as clk:
        barrier()
        ev[0].record(stream)
        for _ in range(args.steps):
            samples = device_step()
        ev[1].record(stream)
        barrier()
    engine.check()
    outputs = {"samples": samples.cpu().numpy()} if args.dump_outputs else {}
    t_dev = ev[0].elapsed_time(ev[1]) / 1e3
    gpu_launches = engine.launch_count - launches0
    clocks = clk.summary()

    # ---- end to end through the public API, host buffers --------------------------------
    def e2e_step():
        torch.manual_seed(1234)
        return model.generate(mel_host, None, True, TARGET, OVERLAP, cfg3)

    if args.skip_e2e:
        t_e2e = float("nan")
    else:
        for _ in range(min(args.warmup, 2)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            wav = e2e_step()
        barrier()
        t_e2e = time.perf_counter() - t0
        assert np.isfinite(wav).all()
        if args.dump_outputs:
            outputs["wav"] = wav

    times = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = times.tolist()

    if rank == 0:
        S_eff = args.seg_steps or S
        units = B_total * S_eff * args.steps
        value, e2e_value = units / t_dev, units / t_e2e
        peaks = measured_peaks()
        long_run = (t_dev / args.steps) > 1.0
        peak_tf = peaks["tflops_sustained"] if long_run else peaks["tflops"]
        ach_tf = value / world * (8_143_872 if cfg3 else FLOP_PER_SAMPLE_MOL) / 1e12          # per GPU (SURVEY 8d)
        step_us = t_dev / args.steps / S_eff * 1e6
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not cfg3:
            r = time_cpu_port(args.cpu_sample_steps)
            v = r["B"] * r["steps"] / r["seconds"][0]
            cpu = {"value": v, "unit": "samples/s", "cores": r["cores"], "kind": "port",
                   "sample": f"{r['B']} folds x first {r['steps']} of 12100 steps, torch CPU operators, best of thread sweep = {r['threads']} threads on {r['host_cores']} host cores; samples/s by threads: {r['sweep']}"}
        line = {
            "metric": "audio samples/sec (22.05 kHz) batched " + ("RAW 9-bit" if cfg3 else "MoL") + " generate", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong" if cfg5 else "weak", "vs_baseline": None,
            "dtype": {"fp16": "f16", "bf16": "bf16", "fp32": "f32"}[args.precision], "data": "synthetic",
            "config": workload_config(world, args.workload, args.cfg5_folds),
            "impl_details": {"engine": engine.name, "grid_ctas": engine.grid_ctas,
                             "parallelism": f"folds sharded x{world}, one NCCL all-gather of the sample blocks" if world > 1 else "single GPU",
                             "conditioning": "frame-rate tensors resident in HBM; the library forms the x275 rows (pre-pass per tile / staging warps)",
                             "l2_policy": "no flush: every step streams fresh conditioning rows and draws; the weights are SUPPOSED to stay on chip",
                             "rng": "in-kernel Philox4x32-10" if (cfg5 or cfg3) else "reference-compatible torch CPU draws, resident in HBM for `value`"},
            "clocks": clocks, "gpu_launches": int(gpu_launches),
            # whole job, counted from the tensors copied: every rank uploads the mel and its columns of the draw matrix, and
            # every rank reads the whole float64 waveform back (generate() returns it on every rank)
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(world * mel_host.numel() * 4 + h2d_rng),
                    "d2h_bytes_per_step": int(world * (T - 1) * HOP * 8), "ms_per_step": t_e2e / args.steps * 1e3},
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": ach_tf / peak_tf, "traffic": measured_traffic(args, model), "peak_source": peaks["src"],
                         "note": ("stream engine: one pass over the fp16 weights per step through each SM's shared memory; bounded by the MMA "
                                  "front end (~40 cycles per M=128 MMA with A from shared memory) and the ring depth, DESIGN.md 3.2") if cfg5 else
                                 ("latency/sync-bound at 19 folds per GPU (four L2 exchanges per step, DESIGN.md 3.1): fraction of the "
                                  "dense-fp16 tensor roofline is reported for completeness"),
                         "hbm_achieved_gbs": value / world * BYTES_PER_SAMPLE / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"]},
            "x_realtime": value / 22050.0, "x_realtime_per_fold": 1.0 / (step_us * 1e-6) / 22050.0,
            "us_per_sequential_step": step_us,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if args.seg_steps or args.skip_e2e:
            line["partial"] = "profiling run (--seg-steps/--skip-e2e): NOT a bench value"
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_cfg4(args, device, rank, world, local):
    """BASELINE configs[3] (gen_tacotron.py wavernn, 16 sentences): the reference Tacotron's mels of 16 sentences
    (committed fixture) vocoded with the reference's shipped LJSpeech checkpoint as ONE job through
    WaveRNN.generate_many (all folds of all sentences in one launch, sharded over the ranks, one all-gather).  Tacotron
    itself is out of scope (torch, run once in the build container to make the fixture).  The whole call is host-facing,
    so `value` and `e2e` are the same end-to-end measurement (host mels in, float64 waveforms out), stated in `config`."""
    import io as _io
    import zipfile
    import torch.distributed as dist
    model = build_model(device)
    with zipfile.ZipFile(ROOT / "tests" / "golden" / "pretrained" / "ljspeech.wavernn.mol.800k.zip") as z:
        model.load_state_dict(torch.load(_io.BytesIO(z.read("latest_weights.pyt")), map_location=device), strict=False)
    model.gen_precision, model.gen_engine, model.gen_rng = args.precision, args.engine, "philox"
    # the 16 mel spectrograms the reference's own Tacotron (shipped checkpoint, CPU) produced for 16 sentences -- the 6 of
    # sentences.txt plus 10 more -- prepared exactly as gen_tacotron.py:139-143 hands them to voc_model.generate
    # (fixture tests/golden/tacotron_mels.npz, generator tests/golden/make_tacotron_mels.py; uint16-quantised [0, 1])
    g = np.load(ROOT / "tests" / "golden" / "tacotron_mels.npz", allow_pickle=False)
    mels_np = [g[f"mel_{i:02d}"].astype(np.float32) / np.float32(65535.0) for i in range(16)]
    frames = [int(m.shape[1]) for m in mels_np]
    mels = [torch.from_numpy(m).unsqueeze(0).pin_memory() for m in mels_np]
    from wavernn_b200.sharding import fold_geometry
    S = TARGET + 2 * OVERLAP
    folds = [fold_geometry(T * HOP, TARGET, OVERLAP).n_seg for T in frames]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def step():
        return model.generate_many(mels, [None] * len(mels), TARGET, OVERLAP, False)

    for _ in range(args.warmup):
        step()
    engine = model._get_engine(device)
    launches0 = engine.launch_count
    with ClockSampler(local) as clk:
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            wavs = step()
        barrier()
        t = time.perf_counter() - t0
    assert all(np.isfinite(w).all() for w in wavs)
    tt = torch.tensor([t], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t = float(tt.item())
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {f"wav_{i:02d}": w for i, w in enumerate(wavs)})
        units = sum(folds) * S * args.steps
        value = units / t
        peaks = measured_peaks()
        ach_tf = value / world * FLOP_PER_SAMPLE_MOL / 1e12
        emit({"metric": "audio samples/sec (22.05 kHz) batched MoL generate", "value": value, "unit": "samples/s",
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
              "config": {"workload": f"cfg4: the reference Tacotron's mels of 16 sentences ({min(frames)}-{max(frames)} frames each, {sum(frames)} frames, "
                                     f"{sum(frames) * HOP / 22050:.1f} s of audio; fixture tests/golden/tacotron_mels.npz) -> {sum(folds)} folds x {S} steps in ONE "
                                     f"generate_many job, sharded over {world} GPU(s), WaveRNN weights = the reference's shipped LJSpeech checkpoint; Tacotron itself is not timed (torch, out of scope)",
                         "engine": model.gen_stats.get("engine"), "rng": "in-kernel Philox4x32-10",
                         "note": "value == e2e: the job is timed end to end through the public call (host mels in, float64 waveforms out)"},
              "clocks": clk.summary(), "gpu_launches": int(engine.launch_count - launches0),
              "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": int(sum(frames) * 80 * 4),
                      "d2h_bytes_per_step": int(sum((T - 1) * HOP for T in frames) * 8), "ms_per_step": t / args.steps * 1e3},
              "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peaks["tflops"], "unit": "TFLOP/s",
                           "frac": ach_tf / peaks["tflops"], "traffic": None, "peak_source": peaks["src"]},
              "x_realtime": value / 22050.0, "delivered_audio_x_realtime": sum((T - 1) * HOP for T in frames) * args.steps / t / 22050.0})
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def guard_stdout():
    """The contract is ONE JSON line on stdout.  Libraries below us write there too (NCCL prints its version banner
    to fd 1 whenever NCCL_DEBUG is VERSION/WARN/INFO in the environment): keep a private handle on the real stdout
    for the JSON line and point fd 1 at stderr for everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tcgen05", "stream"])
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference only: 'cuda' times the unmodified reference's eager CUDA path instead (extra datapoint)")
    ap.add_argument("--cpu-sample-steps", type=int, default=3000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 (default, the headline config: 19 folds per GPU) or cfg5 (4096 folds of a 35.8-min mel, "
                         "sharded over the ranks, in-kernel Philox draws)")
    ap.add_argument("--cfg5-folds", type=int, default=4096, help="cfg5 only: number of folds of the synthetic corpus (default: BASELINE's 4096)")
    ap.add_argument("--seg-steps", type=int, default=0,
                    help="PROFILING ONLY: generate just the first N steps of every fold in the device-timed region "
                         "(keeps ncu captures short); the printed line is then marked partial and is not a bench value")
    ap.add_argument("--skip-e2e", action="store_true", help="PROFILING ONLY: skip the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timing, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(at most 64 MB in all: a fixed, seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                             "(use --impl reference for the CPU arm)")
        run_ours(args)


if __name__ == "__main__":
    main()
