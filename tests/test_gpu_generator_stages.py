"""Every generator stage of the engine, row by row, against float64 references of the same stage
(``oracle.stage_check``: R64 plain float64; R16 float64 with the 16-bit operands of the engine's tensor-core convs).

Each stage is fed the engine's own input -- ``z`` for stage 0 (conv_pre, + speaker cond, upsampler 0, MRF 0),
``mrf{i-1}`` for stage i -- so errors do not compound across stages; the last stage is compared through conv_post
as float audio, 64 samples per row.  Which convs R16 rounds is written out per voice below, from the generator
dispatch in ``engine.cu`` (``pack_voice`` and the decoder section of the call); the profiler's kernel list checks
those expectations on every run.

The synthetic voices place ResBlock1 stages on both sides of the gate ``mrf1_tc_supported`` (DESIGN §3):
NC = 96 packings, many-chunk residual convs (NC = 32, 5-10 chunks), convs at the shared-memory limit (C = 320 and
352, one dilation step inside and one outside), nk = 4 / nd = 1 stages, voices mixing tensor-core and fp32 stages,
and one-tile upsamplers at K = 384.  The shipped ResBlock2 shape runs its fused kernels under every A/B switch.

Criteria (``oracle.stage_check``; every row of every utterance):
* tensor-core stages: rms(E - R64) <= 3 * rms(R16 - R64) + floor;
* ResBlock1 stages also: rms(E - R16) <= 0.5 * rms(R16 - R64) + floor -- R16 restates their per-conv staging
  exactly (why 0.5 and not 0.25: ``oracle.stage_check``).  Not applied to the fused ResBlock2 kernels, which keep
  some intermediates in 16-bit (DESIGN §3);
* stages without any tensor-core conv: max|E - R64| <= 1e-5 * stage RMS.
"""
import shutil
import time

import numpy as np
import pytest
import torch

from oracle import stage_check as sc

pytestmark = pytest.mark.gpu

SCALES = (0.0, 1.0, 0.0)
ENV_KEYS = ("M3B200_FORCE_SIMT", "M3B200_TC_FORMAT", "M3B200_MRF_V1", "M3B200_DEC_V1", "M3B200_DEC_V2",
            "M3B200_UNFUSED_DEC")

# Generator of each synthetic voice, and the path the engine takes per stage:
#   ups: "tc2" conv_tc/ups_tc kernel with two 128-row M tiles per CTA, "tc1" conv_tc_kernel<., ., 1> (only one tile
#        fits shared memory), "fp32" conv_gemm_kernel (C_in > 512);
#   mrf: "tc" ResBlock1 on conv_tc_kernel (C % 32 == 0 and every conv fits, mrf1_tc_supported), "fp32" otherwise,
#        "fused" the ResBlock2 kernels.
# conv_pre (K = inter_channels = 192) always runs on the tensor cores; conv_post on the tensor cores only inside the
# fused last-stage kernels of ResBlock2 voices.
R8842 = dict(upsample_rates=(8, 8, 2, 2), upsample_kernel_sizes=(16, 16, 4, 4))
R884 = dict(upsample_rates=(8, 8, 4), upsample_kernel_sizes=(16, 16, 8))
K3711 = dict(resblock_kernel_sizes=(3, 7, 11), resblock_dilation_sizes=((1, 3, 5),) * 3)
VOICES = {
    # ups0 K = 384 fits only one M tile (NC = 64); MRF C = 192 packs NC = 96 in 2 chunks, C = 96 NC = 96 in one;
    # C = 48 and 24 are not multiples of 32
    "A": dict(gen=dict(upsample_initial_channel=384, **R8842, **K3711),
              ups=("tc1", "tc2", "tc2", "tc2"), mrf=("tc", "tc", "fp32", "fp32")),
    # C = 288: NC = 32 in 9 chunks at every k <= 11, d <= 5 (k = 11, d = 5 is 256 + 50 staged rows)
    "B": dict(gen=dict(upsample_initial_channel=576, **R884, **K3711),
              ups=("fp32", "tc2", "tc2"), mrf=("tc", "fp32", "fp32")),
    # C = 320 fits while (k-1)*dil <= 39: 38 (k 3, d 19) runs on the tensor cores, 40 (k 3, d 20) does not;
    # C = 160: NC = 32 in 5 chunks in both
    "C+": dict(gen=dict(upsample_initial_channel=640, **R884, resblock_kernel_sizes=(3, 5),
                        resblock_dilation_sizes=((1, 19), (1, 9))),
               ups=("fp32", "tc2", "tc2"), mrf=("tc", "tc", "fp32")),
    "C-": dict(gen=dict(upsample_initial_channel=640, **R884, resblock_kernel_sizes=(3, 5),
                        resblock_dilation_sizes=((1, 20), (1, 9))),
               ups=("fp32", "tc2", "tc2"), mrf=("fp32", "tc", "fp32")),
    # C = 352 fits while (k-1)*dil <= 7: 6 yes, 8 no
    "D+": dict(gen=dict(upsample_initial_channel=704, **R884, resblock_kernel_sizes=(3,),
                        resblock_dilation_sizes=((1, 3),)),
               ups=("fp32", "tc2", "tc2"), mrf=("tc", "fp32", "fp32")),
    "D-": dict(gen=dict(upsample_initial_channel=704, **R884, resblock_kernel_sizes=(3,),
                        resblock_dilation_sizes=((1, 4),)),
               ups=("fp32", "tc2", "tc2"), mrf=("fp32", "fp32", "fp32")),
    # C = 384 never fits; nk = 4 with nd = 1: every second conv is the last of its resblock; speaker cond in stage 0
    "E": dict(gen=dict(upsample_initial_channel=768, **R8842, resblock_kernel_sizes=(1, 3, 5, 7),
                       resblock_dilation_sizes=((1,), (2,), (3,), (5,))),
              ups=("fp32", "tc1", "tc2", "tc2"), mrf=("fp32", "tc", "tc", "fp32"), speakers=16),
    # the shipped *_low shape: C = 128 mrf_ws128_kernel, C = 64 mrf_ws_kernel, last stage dec_planes_kernel
    # (with noise_w = 0 its ids all last 4 frames, so the durations carry the voice's default noise)
    "low_ms": dict(gen=None, ups=("tc2", "tc2", "fused"), mrf=("fused", "fused", "fused"), speakers=109,
                   scales=(0.667, 1.0, 0.8)),
}

# (voice, environment, what must run) -- kernel names that must appear in the call
CASES = {
    "A": ("A", {}, ()),
    "A-bf16": ("A", {"M3B200_TC_FORMAT": "bf16"}, ()),
    "A-simt": ("A", {"M3B200_FORCE_SIMT": "1"}, ()),
    "B": ("B", {}, ()),
    "C+": ("C+", {}, ()),
    "C-": ("C-", {}, ()),
    "D+": ("D+", {}, ()),
    "D-": ("D-", {}, ()),
    "E": ("E", {}, ()),
    "low_ms": ("low_ms", {}, ("mrf_ws128_kernel", "mrf_ws_kernel", "dec_planes_kernel")),
    "low_ms-MRF_V1": ("low_ms", {"M3B200_MRF_V1": "1"}, ("mrf_tc_kernel", "dec_planes_kernel")),
    "low_ms-DEC_V1": ("low_ms", {"M3B200_DEC_V1": "1"}, ("mrf_ws128_kernel", "dec_last_kernel")),
    "low_ms-DEC_V2": ("low_ms", {"M3B200_DEC_V2": "1"}, ("mrf_ws128_kernel", "dec_fused_kernel")),
    "low_ms-UNFUSED_DEC": ("low_ms", {"M3B200_UNFUSED_DEC": "1"}, ("mrf_ws128_kernel", "conv_post_kernel")),
}


def _config(name):
    from mimic3_b200 import synth_voice as sv
    v = VOICES[name]
    if v["gen"] is None:
        return sv.low_config(n_speakers=v["speakers"])
    ns = v.get("speakers", 1)
    # small text side (2 layers); the generator is what is under test
    return sv.SynthModelConfig(n_speakers=ns, n_layers=2, resblock="1", gin_channels=64 if ns > 1 else 0, **v["gen"])


@pytest.fixture(scope="module")
def stage_voices(tmp_path_factory):
    from mimic3_b200 import synth_voice as sv
    root = tmp_path_factory.mktemp("stage_voices")
    made = {}

    def get(name):
        if name not in made:
            sv.write_voice(root / name, _config(name), seed=80 + list(VOICES).index(name))
            made[name] = root / name
        return made[name]
    return get


def _plan(name, env):
    """Which conv groups the engine runs on 16-bit operands (the R16 rounding), per the table above."""
    v = VOICES[name]
    if env.get("M3B200_FORCE_SIMT"):
        return {}
    fmt = env.get("M3B200_TC_FORMAT", "fp16")
    rnd = {"pre": fmt}
    for i, (u, m) in enumerate(zip(v["ups"], v["mrf"])):
        if u != "fp32":
            rnd[f"ups{i}"] = fmt
        if m != "fp32":
            rnd[f"mrf{i}"] = fmt
    if v["mrf"][-1] == "fused" and not env.get("M3B200_UNFUSED_DEC"):
        rnd["post"] = fmt
    return rnd


def _pick_batch(orc, nsym, sids, scales):
    """Ids for one batch: utterances of 1, 2 and 3 ids, and three whose frame counts F have F mod 32 = 0, 1, 31,
    so that stage 0's 8F rows end exactly at, just past and just before a 256-row CTA edge (each spans several
    CTAs).  Frame counts from the oracle's duration predictor."""
    rng = np.random.default_rng(7)
    ids = [rng.integers(4, nsym, size=L) for L in (1, 2, 3)]
    for b, r in enumerate((0, 1, 31)):
        for _ in range(3000):
            x = rng.integers(4, nsym, size=int(rng.integers(12, 45)))
            F = max(1, int(orc.durations(x, scales, sid=sids[3 + b], row=3 + b).sum()))
            if F % 32 == r and 60 <= F <= 130:
                ids.append(x)
                break
        else:
            raise AssertionError(f"no utterance with F mod 32 = {r} found")
    return ids


def _t(a):  # engine rows (rows, C) -> oracle layout (1, C, rows), float64
    return torch.from_numpy(np.ascontiguousarray(a.T, dtype=np.float64))[None]


@pytest.mark.parametrize("case", list(CASES))
def test_generator_stages_row_by_row(stage_voices, built_library, monkeypatch, tmp_path, case):
    from torch.profiler import ProfilerActivity, profile

    from mimic3_b200.engine import B200Session
    from oracle.vits_oracle import VitsOracle

    t_start = time.time()
    name, env, must_run = CASES[case]
    v = VOICES[name]
    path = stage_voices(name)
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    orc = VitsOracle(str(path))
    sess = B200Session(str(path))
    n_st = len(v["ups"])
    ms = v.get("speakers", 1) > 1
    sids = [0, 5, v.get("speakers", 1) - 1, 1, 3, 2] if ms else [None] * 6
    scales = v.get("scales", SCALES)
    ids_l = _pick_batch(orc, sess.info.num_symbols, sids, scales)
    lens = np.array([len(x) for x in ids_l], dtype=np.int64)
    ids = np.zeros((len(ids_l), lens.max()), dtype=np.int64)
    for b, x in enumerate(ids_l):
        ids[b, :lens[b]] = x
    sid = np.array(sids, dtype=np.int64) if ms else None
    names = ("z",) + tuple(f"mrf{i}" for i in range(n_st - 1))
    r = sess.infer(ids, lens, scales, sid, keep_float=True, debug_tensors=names)
    frames = r.frames.astype(np.int64)
    assert {int(f) % 32 for f in frames[3:]} == {0, 1, 31}, frames
    off = np.concatenate([[0], np.cumsum(frames)])

    # ---- gate decisions, from the profiler's kernel list
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        plain = sess.infer(ids, lens, scales, sid, keep_float=True)
    np.testing.assert_array_equal(plain.audio, r.audio)
    kernels = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    nk, nd = len(orc.m["resblock_kernel_sizes"]), len(orc.m["resblock_dilation_sizes"][0])
    simt = bool(env.get("M3B200_FORCE_SIMT"))
    ups = ["fp32" if simt else u for u in v["ups"]]
    mrf = ["fp32" if simt else m for m in v["mrf"]]
    n_res = sum("conv_tc_kernel<" in k and ", true, " in k for k in kernels)
    n_one = sum("conv_tc_kernel<" in k and k.split("(")[0].endswith(", 1>") for k in kernels)
    n_gemm = sum("conv_gemm_kernel" in k for k in kernels)
    # every fp32 generator conv is one conv_gemm_kernel launch; so is the speaker-cond GEMM of a multi-speaker
    # voice.  Under M3B200_FORCE_SIMT every conv of the call is, so only the absence of tensor-core convs is checked.
    want_gemm = ups.count("fp32") + sum(2 * nk * nd for m in mrf if m == "fp32") + int(ms)
    n_tc = sum("_tc_kernel" in k or "mrf_ws" in k or "dec_" in k for k in kernels)
    if simt:
        want_gemm = n_gemm
    if v["gen"] is None:  # fused ResBlock2 voice: no ResBlock1 launches, no fp32 generator conv
        want_res = want_one = 0
    else:
        want_res = sum(nk * nd for m in mrf if m == "tc")
        want_one = ups.count("tc1")
    print(f"\n{case}: frames {frames.tolist()}; residual-epilogue launches {n_res} (expect {want_res}), one-tile "
          f"{n_one} (expect {want_one}), conv_gemm_kernel {n_gemm} (expect {want_gemm}); generator kernels "
          f"{sorted({k.split('(')[0].split('<')[0].split()[-1] for k in kernels if 'conv' in k or 'mrf' in k or 'dec_' in k})}")
    gate_msgs = []
    if (n_res, n_one, n_gemm) != (want_res, want_one, want_gemm):
        gate_msgs.append(f"kernel counts (res, one-tile, gemm) {(n_res, n_one, n_gemm)} != {(want_res, want_one, want_gemm)}")
    if simt and n_tc:
        gate_msgs.append(f"{n_tc} tensor-core kernels ran under M3B200_FORCE_SIMT")
    for k in must_run:
        if not any(k in e for e in kernels):
            gate_msgs.append(f"{k} did not run")

    # ---- every stage, every utterance, every row
    rnd = _plan(name, env)
    fused = v["mrf"][-1] == "fused"
    fails = list(gate_msgs)
    worst = {}
    scale = 1
    for i in range(n_st):
        scale_out = scale * orc.m["upsample_rates"][i]
        last = i == n_st - 1
        grp = [g for g in ("pre",) * (i == 0) + (f"ups{i}", f"mrf{i}") + ("post",) * last if g in rnd]
        if not grp:
            crit = ("fp32",)
        elif fused:
            crit = ("budget",)
        else:
            crit = ("budget", "r16")
        src = r.tensors["z"] if i == 0 else r.tensors[f"mrf{i - 1}"]
        w = worst.setdefault(i, {})
        for b in range(len(frames)):
            F = int(frames[b])
            x_in = _t(src[off[b] * scale:(off[b] + F) * scale])
            g = orc.speaker(int(sid[b])).double() if ms else None
            refs = []
            with torch.no_grad():
                for rr in (None, rnd) if grp else (None,):
                    x = orc.decoder_pre(x_in, g, rr) if i == 0 else x_in
                    x = orc.decoder_stage(i, x, rr)
                    if last:
                        refs.append(sc.audio_rows(orc.decoder_post(x, rr)[0, 0].numpy()))
                    else:
                        refs.append(x[0].t().numpy())
            r64 = refs[0]
            r16 = refs[-1]
            if last:
                e = sc.audio_rows(r.utterance_audio(b))
            else:
                e = r.tensors[f"mrf{i}"][off[b] * scale_out:(off[b] + F) * scale_out]
            ww, ff = sc.check_rows(e, r16, r64, crit, f"{case} stage {i} utt {b} ({F} frames)",
                                   row_scale=64 if last else 1)
            fails += ff
            for c, val in ww.items():
                w[c] = max(w.get(c, 0.0), val)
        path_s = (f"{'pre ' if i == 0 else ''}ups {ups[i]}, mrf {mrf[i]}{', post ' if last else ''}"
                  f"{('tc' if 'post' in rnd else 'fp32') if last else ''}")
        print(f"{case} stage {i} [{path_s}]: " + "  ".join(f"{c} {w[c]:.3f}" for c in crit if c in w))
        scale = scale_out

    # ---- weight-cache round trip: bit-identical PCM
    if case in ("A", "E"):
        vd = tmp_path / "v"
        shutil.copytree(path, vd)
        first = B200Session(str(vd), cache_dir=tmp_path / "cache")
        blob = B200Session(str(vd), cache_dir=tmp_path / "cache")
        assert first.load_stats["cache_written"] and blob.load_stats["from_cache"]
        for s in (first, blob):
            np.testing.assert_array_equal(s.infer(ids, lens, scales, sid).pcm, plain.pcm)
            s.close()
    sess.close()
    print(f"{case}: {time.time() - t_start:.1f} s")
    assert not fails, "\n".join(fails[:40])
