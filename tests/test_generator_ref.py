"""The float64 generator-stage references (``VitsOracle.decoder_pre`` / ``decoder_stage`` / ``decoder_post``) and the
row-by-row checker (``oracle.stage_check``) that ``test_gpu_generator_stages.py`` judges the engine with.  CPU only:
the stages chain to the oracle's decoder bit for bit, the 16-bit rounding touches exactly the convs it is asked
to, and the checker fails on small synthetic defects of the kind a kernel could have."""
import numpy as np
import pytest
import torch

from oracle import stage_check as sc
from oracle.vits_oracle import VitsOracle


@pytest.fixture(scope="module")
def gen_voices(tmp_path_factory):
    from mimic3_b200 import synth_voice as sv
    root = tmp_path_factory.mktemp("gen_ref")
    out = {}
    cfgs = {
        "rb1_ms": sv.tiny_config(n_speakers=3, resblock="1"),
        "rb2": sv.tiny_config(resblock="2"),
        # one stage of C = 64, ResBlock1 k 3/5 d 1/3: 4 rows per input frame, dilated halos of up to 6 rows
        "stage64": sv.SynthModelConfig(num_symbols=20, inter_channels=32, hidden_channels=32, filter_channels=64,
                                       n_layers=1, resblock="1", resblock_kernel_sizes=(3, 5),
                                       resblock_dilation_sizes=((1, 3), (1, 3)), upsample_rates=(4,),
                                       upsample_initial_channel=128, upsample_kernel_sizes=(8,)),
    }
    for i, (name, cfg) in enumerate(cfgs.items()):
        sv.write_voice(root / name, cfg, seed=70 + i)
        out[name] = root / name
    return out


def _z(orc, frames, seed):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((1, orc.I, frames)).astype(np.float32))


@pytest.mark.parametrize("voice,sid", [("rb1_ms", 2), ("rb2", None)])
def test_stages_chain_to_decoder_bit_for_bit(gen_voices, voice, sid):
    orc = VitsOracle(str(gen_voices[voice]))
    z, g = _z(orc, 37, 1), orc.speaker(sid)
    taps = {}
    with torch.no_grad():
        want = orc.decoder(z, g, taps)
        x = orc.decoder_pre(z, g)
        for i in range(len(orc.m["upsample_rates"])):
            x = orc.decoder_stage(i, x)
            np.testing.assert_array_equal(x[0].t().numpy(), taps[f"mrf{i}"])
        got = orc.decoder_post(x)
    assert got.dtype == torch.float32
    np.testing.assert_array_equal(got.numpy(), want.numpy())


def test_durations_match_infer(gen_voices):
    orc = VitsOracle(str(gen_voices["rb1_ms"]))
    ids = np.random.default_rng(4).integers(4, 20, size=11)
    for scales in ((0.0, 1.0, 0.0), (0.667, 1.1, 0.8)):
        audio, inter = orc.infer(ids, scales, sid=1, seed=3, row=2, return_intermediates=True)
        dur = orc.durations(ids, scales, sid=1, seed=3, row=2)
        np.testing.assert_array_equal(dur, inter["durations"])
        assert audio.shape[0] == max(1, int(dur.sum())) * int(np.prod(orc.m["upsample_rates"]))


class _Spy(VitsOracle):
    """Records the operands of every generator conv."""
    seen = None

    def _conv1d(self, x, w, b, name, transpose, **kw):
        self.seen.append((name, x, w))
        return super()._conv1d(x, w, b, name, transpose, **kw)


def _is16(t, dt):
    return bool(torch.equal(t.to(dt).to(t.dtype), t))


@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_rounding_reaches_exactly_the_chosen_convs(gen_voices, fmt):
    """R16 rounds the operands of every conv in its groups and of no other conv; with the rounding switched off
    it is R64 bit for bit."""
    orc = _Spy(str(gen_voices["rb1_ms"]))
    dt = VitsOracle._RND[fmt]
    z, g = _z(orc, 23, 2).double(), orc.speaker(1)
    rounding = {"pre": fmt, "mrf0": fmt, "ups1": fmt, "post": fmt}
    with torch.no_grad():
        def run(rnd):
            orc.seen = []
            x = orc.decoder_pre(z, g, rnd)
            for i in range(2):
                x = orc.decoder_stage(i, x, rnd)
            return orc.decoder_post(x, rnd)
        r64 = run(None)
        off = run({k: None for k in rounding})
        assert torch.equal(off, r64)
        r16 = run(rounding)
    assert r16.dtype == torch.float64 and not torch.equal(r16, r64)
    groups = {"dec.conv_pre": "pre", "dec.cond": None, "dec.ups.0": "ups0", "dec.ups.1": "ups1",
              "dec.conv_post": "post"}
    nk = len(orc.m["resblock_kernel_sizes"])
    for name, x, w in orc.seen:
        assert x.dtype == w.dtype == torch.float64, name
        grp = groups.get(name)
        if name.startswith("dec.resblocks."):
            grp = f"mrf{int(name.split('.')[2]) // nk}"
        if grp in rounding:
            assert _is16(x, dt) and _is16(w, dt), name
        else:  # random fp32-derived values are not 16-bit numbers
            assert not _is16(w, dt), name


class _Defect(VitsOracle):
    """Injects one synthetic kernel defect into one conv."""
    defect = None
    target = "dec.resblocks.1.convs1.1"  # k = 5, dilation 3: output row t reads t-6, t-3, t, t+3, t+6

    def _conv1d(self, x, w, b, name, transpose, **kw):
        out = super()._conv1d(x, w, b, name, transpose, **kw)
        if name != self.target or self.defect is None:
            return out
        if self.defect == "halo":  # the CTA at row 256 does not stage its left halo row 255
            x2 = x.clone()
            x2[..., 255] = 0
            out2 = super()._conv1d(x2, w, b, name, transpose, **kw)
            out = torch.cat([out[..., :256], out2[..., 256:]], -1)
        elif self.defect == "tap":  # tap 0 reads one row too late
            w0 = torch.zeros_like(w)
            w0[..., 0] = w[..., 0]
            xs = torch.nn.functional.pad(x[..., 1:], (0, 1))
            out = out - super()._conv1d(x, w0, None, name, transpose, **kw) + super()._conv1d(xs, w0, None, name, transpose, **kw)
        elif self.defect == "bias":  # the bias of the last 32-column chunk is not added
            b2 = b.clone()
            b2[32:] = 0
            out = super()._conv1d(x, w, b2, name, transpose, **kw)
        return out


def test_checker_catches_small_defects(gen_voices):
    orc = _Defect(str(gen_voices["stage64"]))
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((1, 128, 80))).double()  # 320 stage rows
    rnd = {"ups0": "fp16", "mrf0": "fp16"}
    with torch.no_grad():
        r64 = orc.decoder_stage(0, x)[0].t().numpy()
        r16 = orc.decoder_stage(0, x, rnd)[0].t().numpy()
        worst, fails = sc.check_rows(r16, r16, r64, ("budget", "r16"), "untouched")
        assert not fails and worst["budget"] <= 1.0 / sc.BUDGET_X
        for defect in ("halo", "tap", "bias"):
            orc.defect = defect
            bad = orc.decoder_stage(0, x, rnd)[0].t().numpy()
            orc.defect = None
            changed = np.flatnonzero(np.any(bad != r16, axis=1))
            worst, fails = sc.check_rows(bad, r16, r64, ("budget", "r16"), defect)
            print(f"{defect}: {changed.size} rows changed, worst ratios {worst}")
            assert changed.size, defect
            assert any(f.startswith(f"{defect}: r16") for f in fails), (defect, worst)
            if defect == "halo":
                # rows 258 and 261 read row 255 through a tap; the second conv (k = 5) spreads them by 2 rows
                assert set(changed) <= set(range(256, 264)), changed
                assert "row % 256 = " in fails[-1] and int(fails[-1].split("at row ")[1].split()[0]) in changed


def test_checker_rows_and_criteria():
    rng = np.random.default_rng(0)
    r64 = rng.standard_normal((300, 8))
    r16 = r64 + 1e-3 * rng.standard_normal(r64.shape)
    e = r16.copy()
    e[299, 3] += 0.05  # one element of the last row
    worst, fails = sc.check_rows(e, r16, r64, ("budget", "r16", "fp32"), "u0")
    assert len(fails) == 3 and all("at row 299 (last row)" in f for f in fails), fails
    assert "row % 256 = 43" in fails[0] and "1 of 300 rows fail" in fails[0]
    worst, fails = sc.check_rows(r64, r16, r64, ("budget", "fp32"), "exact")
    assert not fails and worst == {"budget": 0.0, "fp32": 0.0}
    a = sc.audio_rows(np.arange(130.0))
    assert a.shape == (3, 64) and a[2, 1] == 129 and a[2, 2] == 0
