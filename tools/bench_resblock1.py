"""Throughput of the ResBlock1 generator of the reference ``ModelConfig`` defaults on one B200.

Voices: ``synth_voice.default_config`` (ResBlock1, 512 channels, 8*8*2*2), single-speaker and 109 speakers.
Inputs: batch 64 x 80 ids from PCG64(1234) (``bench.make_inputs``), the voices' default scales.
Prints one JSON object: per call device-event and wall-clock ms, samples/s, the engine's stage timing, per MRF
stage the algorithmic FLOP (total checked against ``bench.algorithmic_flops_per_frame``) and fp32 activation bytes,
kernel time from ``torch.profiler``, its fractions of the dense fp16 tensor peak and of the HBM bandwidth and which of
the two bounds the stage, kernel launches and the kernels that ran; and the
same call through the fp32 CUDA-core path (``M3B200_FORCE_SIMT=1``) at a small batch, next to the tensor-core path at
that batch.  Without a GPU it exits with status 2.

    python tools/bench_resblock1.py [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from collections import Counter
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (algorithmic_flops_per_frame, make_inputs)

TENSOR_PEAK_FLOPS = 2.25e15  # dense FP16/BF16, one HGX B200 GPU (NVIDIA data sheet, 1000 W)
HBM_PEAK_BYTES = 7.7e12      # HBM3e, one HGX B200 GPU (same data sheet)
BATCH, IDS = 64, 80
SIMT_BATCH = 4


def mrf_stage_flops_per_frame(cfg) -> list:
    """2 * C^2 * k per output row for each of the two convs of every dilation step, rows at the stage rate."""
    out, rows = [], 1
    for i, u in enumerate(cfg.upsample_rates):
        rows *= u
        C = cfg.upsample_initial_channel >> (i + 1)
        out.append(sum(2 * 2 * C * C * k * len(d) * rows
                       for k, d in zip(cfg.resblock_kernel_sizes, cfg.resblock_dilation_sizes)))
    return out


def mrf_stage_bytes_per_frame(cfg) -> list:
    """fp32 activation bytes each MRF stage must move through HBM, per mel frame (halo re-reads not counted): per
    dilation step conv1 reads x and writes t, conv2 reads t and the residual and writes x'; the last step of every
    resblock after the first also reads the stage sum it adds to."""
    out, rows = [], 1
    for i, u in enumerate(cfg.upsample_rates):
        rows *= u
        C = cfg.upsample_initial_channel >> (i + 1)
        nk = len(cfg.resblock_kernel_sizes)
        steps = sum(len(d) for d in cfg.resblock_dilation_sizes)
        out.append((steps * 5 * 4 * C + (nk - 1) * 4 * C) * rows)
    return out


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # the numbers still stand; say what is missing
        return {"error": f"nvidia-smi: {e}"}


def timed(sess, ids, lens, scales, sid, steps, warmup):
    for _ in range(warmup):
        sess.infer(ids, lens, scales, sid)
    dev, wall = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        r = sess.infer(ids, lens, scales, sid)  # returns after the call's stream synchronise
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(r.device_ms)
    samples = int(r.sample_offsets[-1])
    return {"device_ms": float(np.median(dev)), "wall_ms": float(np.median(wall)),
            "device_ms_min_max": [float(min(dev)), float(max(dev))], "samples": samples,
            "samples_per_s_device": samples / (np.median(dev) / 1e3),
            "samples_per_s_wall": samples / (np.median(wall) / 1e3), "launches": r.launches}, r


def mrf_kernel_ms(sess, ids, lens, scales, sid, n_stages, per_stage):
    """Kernel time of each MRF stage: the residual-epilogue conv_tc_kernel launches and the conv that precedes each."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sess.infer(ids, lens, scales, sid)
    ev = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and not e.name.startswith("Memcpy")
                 and not e.name.startswith("Memset")), key=lambda e: e.time_range.start)
    names = Counter(e.name.replace("(anonymous namespace)::", "").split("(")[0].replace("void ", "") for e in ev)
    res_idx = [i for i, e in enumerate(ev) if "conv_tc_kernel<" in e.name and ", true, " in e.name]
    if len(res_idx) != n_stages * per_stage:
        return None, dict(names)
    ms = []
    for s in range(n_stages):
        idx = res_idx[s * per_stage:(s + 1) * per_stage]
        ms.append(sum(ev[i].time_range.elapsed_us() + ev[i - 1].time_range.elapsed_us() for i in idx) / 1e3)
    return ms, dict(names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        print("bench_resblock1: no CUDA device; this benchmark only runs on the GPU", file=sys.stderr)
        sys.exit(2)
    from mimic3_b200 import synth_voice as sv
    from mimic3_b200.engine import B200Session

    result = {"gpu": gpu_info(), "batch": BATCH, "ids_per_utt": IDS, "tensor_peak_tflops": TENSOR_PEAK_FLOPS / 1e12,
              "voices": {}}
    tmp = Path(tempfile.mkdtemp(prefix="m3_rb1_"))
    for name, nspk, seed in (("default_1spk", 1, 61), ("default_109spk", 109, 62)):
        cfg = sv.default_config(n_speakers=nspk)
        vd = tmp / name
        sv.write_voice(vd, cfg, seed=seed)
        inf = json.loads((vd / "config.json").read_text())["inference"]
        scales = (inf["noise_scale"], inf["length_scale"], inf["noise_w"])
        ids, lens, sid = bench.make_inputs(BATCH, IDS, cfg.num_symbols, nspk)
        sid = sid if nspk > 1 else None

        per_frame = mrf_stage_flops_per_frame(cfg)
        bytes_frame = mrf_stage_bytes_per_frame(cfg)
        ref = bench.algorithmic_flops_per_frame(cfg)
        assert sum(per_frame) == ref["mrf"] and per_frame == ref["mrf_stage"], (per_frame, ref["mrf_stage"])
        os.environ.pop("M3B200_FORCE_SIMT", None)
        sess = B200Session(str(vd))
        tc, r = timed(sess, ids, lens, scales, sid, args.steps, args.warmup)
        frames = int(r.frames.sum())
        st = sess.infer(ids, lens, scales, sid, stage_timing=True)
        tc["stage_ms"] = {k[3:]: float(v.reshape(-1)[0]) for k, v in st.tensors.items() if k.startswith("ms:")}
        nk = len(cfg.resblock_kernel_sizes) * len(cfg.resblock_dilation_sizes[0])
        kms, kernels = mrf_kernel_ms(sess, ids, lens, scales, sid, len(cfg.upsample_rates), nk)
        tc["kernels_per_call"] = kernels
        stages = []
        for i, f in enumerate(per_frame):
            C = cfg.upsample_initial_channel >> (i + 1)
            d = {"C": C, "gflop": f * frames / 1e9, "hbm_gb": bytes_frame[i] * frames / 1e9}
            if kms:
                s = kms[i] / 1e3
                d["kernel_ms"] = kms[i]
                d["tflops"] = f * frames / s / 1e12
                d["fraction_of_tensor_peak"] = f * frames / s / TENSOR_PEAK_FLOPS
                d["hbm_tb_per_s"] = bytes_frame[i] * frames / s / 1e12
                d["fraction_of_hbm_peak"] = bytes_frame[i] * frames / s / HBM_PEAK_BYTES
                # the least time the hardware could take is the larger of the two bounds; kernel_ms over it
                d["bound"] = "tensor" if d["fraction_of_tensor_peak"] >= d["fraction_of_hbm_peak"] else "hbm"
                d["fraction_of_bound"] = max(d["fraction_of_tensor_peak"], d["fraction_of_hbm_peak"])
            stages.append(d)
        tc["frames"] = frames
        tc["mrf_stages"] = stages
        tc["mrf_gflop_total"] = ref["mrf"] * frames / 1e9
        small = (ids[:SIMT_BATCH], lens[:SIMT_BATCH], scales, None if sid is None else sid[:SIMT_BATCH])
        tc_small, _ = timed(sess, *small, steps=3, warmup=1)
        sess.close()
        os.environ["M3B200_FORCE_SIMT"] = "1"
        simt_sess = B200Session(str(vd))
        os.environ.pop("M3B200_FORCE_SIMT")
        simt, _ = timed(simt_sess, *small, steps=2, warmup=1)
        simt_sess.close()
        result["voices"][name] = {"tensor_cores": tc, "small_batch": SIMT_BATCH,
                                  "tensor_cores_small_batch": tc_small, "fp32_simt_small_batch": simt}
        print(f"{name}: {tc['samples_per_s_device']:.3e} samples/s (device), fp32 path at batch {SIMT_BATCH} "
              f"{simt['samples_per_s_device']:.3e} vs tensor cores {tc_small['samples_per_s_device']:.3e}",
              file=sys.stderr)
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
