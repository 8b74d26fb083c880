#!/usr/bin/env python
"""Benchmark of the N-HANS inference hot path on B200 (contract: see the task statement / DESIGN.md §6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg1..cfg5] [--utts U]
                  [--dump-outputs DIR]

Metric (BASELINE.json): audio-seconds denoised / separated per wall-second.  A step = one pass of the hot path
(STFT -> embedding towers -> conditioned residual network -> iSTFT/overlap-add) over one batch of synthetic 16 kHz
utterances.  Workloads are BASELINE.json's `configs`:

  cfg1  nhans_denoiser, 1 x 4 s + --neg                      (the reference's own CPU-runnable case; GPU latency)
  cfg2  nhans_denoiser, 256 x 4 s + --neg                    (default at N = 1: the config the metric is quoted on)
  cfg3  selective noise, 256 x 8 s, --pos and --neg
  cfg4  nhans_separator, 256 x 10 s, target / interference speakers
  cfg5  utterance-sharded denoising, 8192 x 10 s over 8 GPUs = 1024 clips per GPU; a step processes a 256-clip
        slice of the GPU's shard (default at N > 1: weak scaling, no collective on the data path)

`value` is measured with the inputs resident in HBM (CUDA events on the engine's stream); `e2e` goes through
nhans_enhance_batch with pinned host buffers, H2D and D2H inside the timed region.  `--impl reference` times the
reference's own structure (oracle faithful mode: both towers per window, mb = 100) on the host cores.

`--dump-outputs DIR` writes what the last timed step returned to its caller (rank 0's batch), so that two builds
can be compared output for output on identical inputs: out_i16.npy (the int16 PCM, as float32), out_f32.npy (the
float32 samples of the same batch) and out_offsets.npy (utterance boundaries, float64).  Above DUMP_BYTES a fixed,
seeded sample of sample positions is written instead, listed in sample_index.npy (float64).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 16000
GFLOP_PER_WINDOW = 10.327145856       # 2 * 5 163 572 928 MAC (SURVEY.md App. B)
GFLOP_PER_TOWER_ROW = 15.11485632     # 2 * 7 557 428 160 MAC
CLOCK_QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
               "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

# name -> (variant, utterances per step and GPU, seconds, contexts, description)
CONFIGS = {
    "cfg1": (0, 1, 4.0, "neg", "nhans_denoiser on one 4 s utterance + --neg clip (BASELINE config 1: single-utterance latency)"),
    "cfg2": (0, 256, 4.0, "neg", "nhans_denoiser, 256 x 4 s utterances + --neg clip (BASELINE config 2)"),
    "cfg3": (0, 256, 8.0, "posneg", "selective noise suppression, 256 x 8 s utterances with --pos and --neg clips (BASELINE config 3)"),
    "cfg4": (1, 256, 10.0, "posneg", "nhans_separator, 256 x 10 s mixtures with target / interference speaker clips (BASELINE config 4; "
                                     "batch of 256 chosen here)"),
    "cfg5": (0, 256, 10.0, "neg", "nhans_denoiser, utterance-sharded 8192 x 10 s sweep: 1024 clips per GPU, one step = a 256-clip slice of "
                                  "the GPU's shard + --neg clips (BASELINE config 5)"),
}
DUMP_BYTES = 64 * 10 ** 6


class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + CLOCK_QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = []
        reasons = set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                out["sm_max_mhz"] = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            busy = [v for v in sm if v > 0.5 * max(sm)] or sm
            out["sm_mhz"] = float(np.median(busy))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 6650.0, "fallback"


def traffic_of(kernel):
    """DRAM bytes per launch of `kernel` from this round's `ncu --set full` capture (profiles/r02_traffic.json,
    written by scripts/profile_summarise.py from the raw ncu export; a profiled run is never a bench value)."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        d = json.load(open(path))
        k = d["kernels"][kernel]
        return k["dram_bytes_per_launch"], "profiles/r02_traffic.json: " + d.get("command", "ncu --set full")
    except Exception:
        return None, None


def contexts(variant, kind, u):
    """(ctx_a, ctx_b) int16 clips of utterance u in the engine's order (SN: pos, neg; SS: interference, target)."""
    from nhans_b200 import synth
    if variant == 0:
        return (synth.noise_clip(u, "pos") if kind == "posneg" else None), synth.noise_clip(u, "neg")
    return synth.speaker_clip(u, "interference"), synth.speaker_clip(u, "target")


def dump_outputs(out_dir, eng, out_i16, out_offs):
    """Write the outputs of the batch the engine processed last (see the module docstring) under out_dir."""
    out_f32 = np.zeros(out_i16.shape, np.float32)
    eng.download(out_f32=out_f32)
    eng.sync()
    arrays = {"out_i16": out_i16.astype(np.float32), "out_f32": out_f32}
    n = len(out_f32)
    header = 128                                        # bytes of an .npy header
    fixed = 3 * header + 8 * len(out_offs)
    if fixed + 8 * n > DUMP_BYTES:
        k = (DUMP_BYTES - fixed - header) // 16         # two float32 values and one float64 index per sampled position
        idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
        arrays = {name: a[idx] for name, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    arrays["out_offsets"] = np.asarray(out_offs, np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_baseline(weights, variant, kind, seconds, steps=1, warmup=0, dedup=True):
    """The reference's own structure on the host cores: oracle faithful mode (mb = 100, both towers per
    window, materialised windows), torch-CPU fp32, all threads; plus the algorithmically de-duplicated mode
    (towers once per clip) for an apples-to-apples figure."""
    import torch
    from nhans_b200 import synth
    from oracle import nhans_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    net = O.Net(weights, variant)
    mix = synth.mixture(seconds, 0)
    a, b = contexts(variant, kind, 0)
    if a is None:
        a = synth.silence()
    times = []
    for i in range(warmup + steps):
        t = time.perf_counter()
        O.apply_arrays(net, mix, a, b, faithful=True)
        if i >= warmup:
            times.append(time.perf_counter() - t)
    dt = float(np.mean(times))
    out = dict(value=seconds / dt, unit="audio-s/s", cores=os.cpu_count() or 1, kind="port",
               sample="oracle faithful mode (torch-CPU fp32, mb=100, both towers per window: SN/apply.py:339-450 restated) on one "
                      "%.1f s utterance of the workload + its context clip(s), %d step(s), %.1f s per step" % (seconds, steps, dt))
    if dedup:
        t = time.perf_counter()
        O.apply_arrays(net, mix, a, b, faithful=False)
        out["dedup_value"] = seconds / (time.perf_counter() - t)
        out["dedup_note"] = "same sample with the towers evaluated once per clip (the algorithm the GPU path runs), 1 step"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS))
    ap.add_argument("--utts", type=int, default=0, help="utterances per step and GPU (default: the config's)")
    ap.add_argument("--seconds", type=float, default=0.0)
    ap.add_argument("--win-capacity", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as .npy files under DIR (--impl ours, rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg_name = a.config or ("cfg2" if a.gpus == 1 else "cfg5")
    variant, utts, seconds, kind, descr = CONFIGS[cfg_name]
    if a.utts:
        utts = a.utts
    if a.seconds:
        seconds = a.seconds
    from nhans_b200 import synth, weights as W
    weights, wsrc = W.load_or_init(variant, os.environ.get("NHANS_MODEL_DIR"), 0, allow_random=True)
    workload = descr + (" [overridden: %d x %.0f s]" % (utts, seconds) if (a.utts or a.seconds) else "") + ", per GPU"
    base = {"metric": "audio-sec/sec", "unit": "audio-s/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
            "config": {"workload": workload, "name": cfg_name, "variant": "selective_noise" if variant == 0 else "source_separation",
                       "contexts": kind, "utterances_per_gpu": utts, "seconds": seconds, "weights": wsrc,
                       "l2": "working set per step (GBs of fp16 activations, >= 160 MB of spectra at 256 utterances) exceeds the 126 MB L2",
                       "parallelism": "utterance-sharded x%d, no collective" % a.gpus}}

    if a.impl == "reference":
        # The reference (TensorFlow graph code) cannot run on this image; its CPU path is the oracle's faithful mode.
        # Rank 0 alone runs it.  A step = ONE utterance of the workload (a bounded sample; cfg1 in full when it is 4 s):
        # the rate does not depend on the batch size (utterances are independent) and varies < 3 % with the length.
        if rank != 0:
            return 0
        n = a.steps + a.warmup
        secs = min(seconds, 4.0 if n <= 12 else (2.0 if n <= 30 else 1.0))
        cb = cpu_baseline(weights, variant, kind, secs, steps=a.steps, warmup=a.warmup)
        line = dict(base)
        line["config"] = dict(base["config"], reference_sample="one %.1f s utterance of the workload per step" % secs)
        line.update({"impl": "reference", "value": cb["value"], "ms_per_step": 1e3 * secs / cb["value"], "dtype": "f32",
                     "cpu_baseline": cb, "gpu_launches": 0,
                     "e2e": {"value": cb["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(line), flush=True)
        return 0

    from nhans_b200.engine import Engine, PinnedArray, pack, KIND_GEMM, KIND_STFT, KIND_ISTFT
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # NCCL prints its version banner on stdout when NCCL_DEBUG is set; stdout carries exactly one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()                    # creates the communicator (the only NCCL use: barrier + max over ranks)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    eng = Engine(local_rank, variant, win_capacity=a.win_capacity)
    eng.load_weights(weights, wsrc)

    # ---- synthetic batch (distinct utterances per rank), staged in pinned host memory ----
    n_distinct = min(utts, 16)
    mixes_d = [synth.mixture(seconds, rank * 1000 + u) for u in range(n_distinct)]
    ctx_d = [contexts(variant, kind, rank * 1000 + u) for u in range(n_distinct)]
    mix, mo = pack([mixes_d[u % n_distinct] for u in range(utts)])
    cb_, bo = pack([ctx_d[u % n_distinct][1] for u in range(utts)])
    has_a = ctx_d[0][0] is not None
    ca_, ao = pack([ctx_d[u % n_distinct][0] for u in range(utts)]) if has_a else (None, None)
    oo = eng.output_offsets(mo)
    p_mix, p_b = PinnedArray(mix.shape, np.int16), PinnedArray(cb_.shape, np.int16)
    p_out = PinnedArray((int(oo[-1]),), np.int16)
    p_mix.array[:] = mix
    p_b.array[:] = cb_
    p_a = None
    if has_a:
        p_a = PinnedArray(ca_.shape, np.int16)
        p_a.array[:] = ca_
    a_arr = p_a.array if has_a else None
    audio_s = float(mo[-1]) / FS
    h2d = int(mix.nbytes + cb_.nbytes + (ca_.nbytes if has_a else 0))

    def barrier():
        eng.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def over_ranks(x):
        """-> (max over ranks, list of every rank's value)"""
        if dist is None:
            return x, [x]
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        allv = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        vals = [float(v.item()) for v in allv]
        return max(vals), vals

    # ---- device-resident: inputs already in HBM when the timed region starts ----
    eng.upload(p_mix.array, mo, a_arr, ao, p_b.array, bo)
    for _ in range(a.warmup):
        eng.run()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    eng.profile_reset()
    eng.profile(True)
    eng.event_record(0)
    for _ in range(a.steps):
        eng.run()
    eng.event_record(1)
    barrier()
    ms_res, ms_res_all = over_ranks(eng.event_elapsed_ms(0, 1))
    st = {k: eng.profile_get(k) for k in range(6)}
    layers = eng.profile_layers(0)
    plan_gemm = eng.plan(0)["gemm"]
    eng.profile(False)
    clocks = sampler.stop() if rank == 0 else None
    value = world * a.steps * audio_s / (ms_res / 1e3)

    # ---- end to end: host buffers in, int16 PCM out, copies inside the timed region ----
    for _ in range(max(1, a.warmup - 1)):
        eng.enhance_packed(p_mix.array, mo, a_arr, ao, p_b.array, bo, out_i16=p_out.array)
    barrier()
    eng.event_record(2)
    t_host = time.perf_counter()
    for _ in range(a.steps):
        eng.enhance_packed(p_mix.array, mo, a_arr, ao, p_b.array, bo, out_i16=p_out.array, sync=False)
    eng.event_record(3)
    barrier()
    wall_e2e = time.perf_counter() - t_host
    ms_e2e, ms_e2e_all = over_ranks(eng.event_elapsed_ms(2, 3))
    e2e = world * a.steps * audio_s / (ms_e2e / 1e3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, eng, p_out.array, oo)

    if rank == 0:
        tf_peak, hbm_peak, which = peaks()
        g = st[KIND_GEMM]
        achieved = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
        walk = [l for l, pg in zip(layers, plan_gemm) if pg.get("walk")]
        rest = [l for l, pg in zip(layers, plan_gemm) if not pg.get("walk")]

        def agg(ls):
            ms = sum(l["ms"] for l in ls)
            fl = sum(l["tflops"] * l["ms"] for l in ls) * 1e9          # tflops * ms * 1e9 = FLOP
            n = sum(l["launches"] for l in ls)
            return {"launches": n, "ms_per_step": ms / a.steps, "TFLOPs": fl / ms / 1e9 if ms > 0 else 0.0,
                    "frac_tensor": (fl / ms / 1e9 / tf_peak) if ms > 0 else 0.0, "share_of_step": ms / ms_res if ms_res > 0 else 0.0}
        traffic, tsrc = traffic_of("gemm_shift_kernel")

        def hbm(kind_):
            s_ = st[kind_]
            gbps = s_["bytes"] / max(s_["ms"], 1e-9) / 1e6
            return {"launches": s_["launches"], "ms": s_["ms"], "GBps": gbps, "frac_hbm": gbps / hbm_peak,
                    "algorithmic_bytes_per_launch": s_["bytes"] / max(1, s_["launches"])}
        flop_per_audio_s = g["flops"] / a.steps / audio_s if audio_s > 0 else 0.0
        line = dict(base)
        line.update({
            "value": value, "ms_per_step": ms_res / a.steps, "dtype": "f16 operands, f32 accumulate",
            "per_rank_ms_per_step": [m / a.steps for m in ms_res_all],
            # whole-job figures: every rank copies its own shard and launches its own kernels
            "e2e": {"value": e2e, "unit": "audio-s/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": int(p_out.array.nbytes) * world, "ms_per_step": ms_e2e / a.steps,
                    "per_rank_ms_per_step": [m / a.steps for m in ms_e2e_all], "host_wall_ms_per_step": 1e3 * wall_e2e / a.steps},
            "gpu_launches": int(st[5]["launches"]) * world,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "tensor-core layers: gemm_shift_kernel (tcgen05 implicit-GEMM conv / dense layers) + "
                                                      "conv64_walk_kernel (tcgen05 row-walk 64-channel layers)",
                         "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                         "peak_source": which + " bf16_tflops_sustained", "traffic": traffic, "traffic_source": tsrc,
                         "launches": g["launches"], "avg_launch_ms": g["ms"] / max(1, g["launches"]),
                         "share_of_step": g["ms"] / ms_res,
                         "algorithmic_flop_per_launch": g["flops"] / max(1, g["launches"]),
                         "by_kernel": {"gemm_shift_kernel": agg(rest), "conv64_walk_kernel": agg(walk)}},
            "kernels": {
                "stft": hbm(KIND_STFT), "istft": hbm(KIND_ISTFT),
                "direct_conv": {"launches": st[3]["launches"], "ms": st[3]["ms"]},
                "other": {"launches": st[4]["launches"], "ms": st[4]["ms"]}},
            "layers": [{"name": l["name"], "ms_per_step": l["ms"] / a.steps, "TFLOPs": round(l["tflops"], 1)} for l in layers],
            "tensor_ceiling_audio_s_per_s": (tf_peak * 1e12 / flop_per_audio_s * world) if flop_per_audio_s > 0 else None,
        })
        if cfg_name == "cfg1":
            line["latency_ms"] = {"device_resident": ms_res / a.steps, "e2e": ms_e2e / a.steps}
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(weights, variant, kind, min(seconds, 4.0))   # one utterance (cfg1 in full for 4 s workloads)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
