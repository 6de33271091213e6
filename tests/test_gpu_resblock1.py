"""The ResBlock1 generator of the reference ``ModelConfig`` defaults (``synth_voice.default_config``) on the
tensor cores: every MRF conv runs as ``conv_tc_kernel`` (16-bit operands, fp32 accumulators and residual
stream), the second conv of each dilation step with the residual epilogue.  Compared with the fp32 oracle,
with the fp32 CUDA-core path of the same library (``M3B200_FORCE_SIMT=1``) and with itself (batch-1 rows,
weight-cache blobs)."""
import shutil

import numpy as np
import pytest

from conftest import rand_ids

pytestmark = pytest.mark.gpu

RMS_TOL = 1e-3  # waveform RMS vs the fp32 oracle, as for the other generators
SCALES = (0.0, 1.0, 0.0)


@pytest.fixture(scope="module")
def rb1_voices(tmp_path_factory):
    from mimic3_b200 import synth_voice as sv
    root = tmp_path_factory.mktemp("rb1_voices")
    out = {}
    for name, n_speakers, seed in (("default", 1, 51), ("default_ms", 109, 52)):
        sv.write_voice(root / name, sv.default_config(n_speakers=n_speakers), seed=seed)
        out[name] = root / name
    return out


def _batch(rng, nsym, lengths):
    ids = np.zeros((len(lengths), max(lengths)), dtype=np.int64)
    for b, L in enumerate(lengths):
        ids[b, :L] = rand_ids(rng, nsym, L)
    return ids, np.array(lengths, dtype=np.int64)


def _session(path, monkeypatch, **env):
    from mimic3_b200.engine import B200Session
    for k in ("M3B200_FORCE_SIMT", "M3B200_TC_FORMAT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    s = B200Session(str(path))
    for k in env:
        monkeypatch.delenv(k)
    return s


@pytest.mark.parametrize("voice,lengths,sid", [
    ("default", [2, 47, 403, 1], None),
    ("default_ms", [3, 61, 402, 18], [108, 0, 57, 1]),
])
def test_default_generator_matches_oracle_fp16(rb1_voices, built_library, monkeypatch, voice, lengths, sid):
    """Durations identical and waveform RMS <= 1e-3 per utterance; the 1-3-id rows are shorter than one conv
    window, so a conv that reads a nonzero row past either end of the utterance (of x or of the intermediate t)
    shows up there."""
    from oracle.vits_oracle import VitsOracle
    sess = _session(rb1_voices[voice], monkeypatch)
    orc = VitsOracle(str(rb1_voices[voice]))
    ids, lens = _batch(np.random.default_rng(len(lengths)), sess.info.num_symbols, lengths)
    sid = None if sid is None else np.array(sid, dtype=np.int64)
    r = sess.infer(ids, lens, SCALES, sid, keep_float=True, debug_tensors=("durations",))
    tok = 0
    for b, L in enumerate(lengths):
        audio, inter = orc.infer(ids[b, :L], SCALES, sid=None if sid is None else int(sid[b]), row=b,
                                 return_intermediates=True)
        dur = r.tensors["durations"][tok:tok + L, 0].astype(np.int64)
        np.testing.assert_array_equal(dur, inter["durations"], err_msg=f"durations differ (utt {b})")
        got = r.utterance_audio(b)
        assert got.shape == audio.shape
        rms = float(np.sqrt(np.mean((got - audio) ** 2)))
        print(f"{voice} utt {b} ({L} ids, {got.shape[0]} samples): waveform RMS vs oracle {rms:.3e}")
        assert rms <= RMS_TOL, (b, L, rms)
        tok += L
    sess.close()


def test_tensor_core_path_vs_fp32_path(rb1_voices, built_library, monkeypatch):
    """Same inputs through the tensor-core MRF (fp16 and bf16 operands) and the fp32 CUDA-core convs; the
    profiler shows which kernels ran."""
    from torch.profiler import ProfilerActivity, profile
    path = rb1_voices["default_ms"]
    ids, lens = _batch(np.random.default_rng(3), 50, [40, 2, 75, 13])
    sid = np.array([5, 100, 42, 0], dtype=np.int64)
    names = ("mrf0", "mrf1", "mrf2", "mrf3")
    simt = _session(path, monkeypatch, M3B200_FORCE_SIMT="1")
    ref = simt.infer(ids, lens, SCALES, sid, keep_float=True, debug_tensors=names)
    simt_plain = simt.infer(ids, lens, SCALES, sid, keep_float=True)
    for fmt, tol_rel in (("fp16", 8e-3), ("bf16", 5e-2)):
        sess = _session(path, monkeypatch, M3B200_TC_FORMAT=fmt)
        r = sess.infer(ids, lens, SCALES, sid, keep_float=True, debug_tensors=names)
        np.testing.assert_array_equal(r.frames, ref.frames)
        for name in names:
            a, b = r.tensors[name], ref.tensors[name]
            rel = float(np.sqrt(np.mean((a - b) ** 2)) / np.sqrt(np.mean(b ** 2)))
            print(f"{fmt} {name}: relative RMS vs fp32 path {rel:.3e}")
            assert 0.0 < rel < tol_rel, (fmt, name, rel)
        rms = float(np.sqrt(np.mean((r.audio - ref.audio) ** 2)))
        print(f"{fmt}: waveform RMS vs fp32 path {rms:.3e}")
        assert rms <= (RMS_TOL if fmt == "fp16" else 5 * RMS_TOL), (fmt, rms)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            plain = sess.infer(ids, lens, SCALES, sid, keep_float=True)
        kernels = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
        n_res = sum("conv_tc_kernel<" in k and ", true, " in k for k in kernels)
        print(f"{fmt}: {plain.launches} launches (fp32 path {simt_plain.launches}); residual-epilogue kernels {n_res}")
        assert n_res == 4 * 3 * 3  # four stages x three resblocks x three dilations
        assert plain.launches < simt_plain.launches
        sess.close()
    simt.close()


def test_ragged_batch_rows_equal_batch1_calls(rb1_voices, built_library, monkeypatch):
    sess = _session(rb1_voices["default_ms"], monkeypatch)
    lengths = [9, 31, 2, 17, 1]
    ids, lens = _batch(np.random.default_rng(5), 50, lengths)
    sid = np.array([2, 0, 108, 1, 64], dtype=np.int64)
    r = sess.infer(ids, lens, SCALES, sid, keep_float=True)
    for b, L in enumerate(lengths):
        one = sess.infer(ids[b:b + 1, :L], lens[b:b + 1], SCALES, sid[b:b + 1], keep_float=True)
        np.testing.assert_array_equal(one.audio, r.utterance_audio(b))
        np.testing.assert_array_equal(one.pcm, r.utterance_pcm(b))
    sess.close()


def test_voice_from_weight_cache_blob_is_bit_identical(rb1_voices, built_library, tmp_path):
    from mimic3_b200.engine import B200Session
    vd = tmp_path / "v"
    shutil.copytree(rb1_voices["default"], vd)
    cache = tmp_path / "cache"
    ids, lens = _batch(np.random.default_rng(8), 50, [23, 3, 40])
    plain = B200Session(str(vd))
    first = B200Session(str(vd), cache_dir=cache)
    assert first.load_stats["cache_written"]
    blob = B200Session(str(vd), cache_dir=cache)
    assert blob.load_stats["from_cache"]
    want = plain.infer(ids, lens, SCALES).pcm
    for s in (first, blob):
        np.testing.assert_array_equal(s.infer(ids, lens, SCALES).pcm, want)
    for s in (plain, first, blob):
        s.close()


def test_every_generator_conv_runs_on_tensor_cores(rb1_voices, built_library, monkeypatch):
    """Single-speaker default voice: no fp32 conv kernel is left in a call.  The first upsampler (512 input channels,
    2 polyphase taps) only fits conv_tc_kernel with one 128-row M tile per CTA."""
    from torch.profiler import ProfilerActivity, profile
    sess = _session(rb1_voices["default"], monkeypatch)
    ids, lens = _batch(np.random.default_rng(9), 50, [35, 3, 60])
    sess.infer(ids, lens, SCALES)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sess.infer(ids, lens, SCALES)
    kernels = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    print(sorted(set(k.split("(")[0] for k in kernels)))
    assert not any("conv_gemm_kernel" in k for k in kernels)
    assert sum("conv_tc_kernel<" in k and ", 1>" in k for k in kernels) == 1  # the first upsampler
    assert sum("conv_tc_kernel<" in k and "true, 2>" in k for k in kernels) == 36
    sess.close()
