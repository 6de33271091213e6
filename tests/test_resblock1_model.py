"""The oracle at the generator of the reference ``ModelConfig`` defaults (``synth_voice.default_config``:
ResBlock1, 512 initial channels, upsampling 8*8*2*2, kernels (3, 7, 11), dilations (1, 3, 5)) against
Hugging Face transformers' ``VitsModel``, whose only generator is this one.  The GPU tests of that generator
(tests/test_gpu_resblock1.py) compare the engine with the oracle, so this pins what they compare with."""
import numpy as np
import pytest

from mimic3_b200 import synth_voice as sv


def test_default_config_is_the_reference_generator():
    cfg = sv.default_config()
    assert (cfg.resblock, cfg.upsample_initial_channel) == ("1", 512)
    assert cfg.upsample_rates == (8, 8, 2, 2) and cfg.upsample_kernel_sizes == (16, 16, 4, 4)
    assert cfg.resblock_kernel_sizes == (3, 7, 11) and cfg.resblock_dilation_sizes == ((1, 3, 5),) * 3
    assert cfg.gin_channels == 0 and sv.default_config(n_speakers=109).gin_channels == 512
    assert sv.low_config().resblock == "2"  # the other presets keep their generator


@pytest.mark.parametrize("n_speakers", [1, 109])
def test_oracle_matches_transformers_vits_at_default_generator_shapes(tmp_path, n_speakers):
    torch = pytest.importorskip("torch")
    pytest.importorskip("transformers")
    from oracle.vits_oracle import VitsOracle
    from test_oracle_vs_hf_vits import _hf_model

    cfg = sv.default_config(n_speakers=n_speakers)
    params = sv.write_voice(tmp_path / "v", cfg, seed=41)
    assert any(".convs2.2.weight" in k for k in params)
    orc = VitsOracle(str(tmp_path / "v"))
    hf = _hf_model(cfg, params)
    multi = n_speakers > 1
    for T, sid in ((29, n_speakers - 1), (2, 0)):
        ids = np.random.default_rng(T).integers(4, cfg.num_symbols, size=T).astype(np.int64)
        audio = orc.infer(ids, (0.0, 1.0, 0.0), sid=sid if multi else None)
        hf.noise_scale, hf.noise_scale_duration, hf.speaking_rate = 0.0, 0.0, 1.0
        with torch.no_grad():
            out = hf(input_ids=torch.from_numpy(ids)[None], attention_mask=torch.ones(1, T, dtype=torch.long),
                     speaker_id=sid if multi else None)
        want = out.waveform[0].numpy()
        assert want.shape == audio.shape and audio.shape[0] % 256 == 0
        rms = float(np.sqrt(np.mean((audio - want) ** 2)))
        print(f"default generator, {n_speakers} speaker(s), {T} ids: {audio.shape[0]} samples, "
              f"oracle vs transformers RMS {rms:.2e}")
        assert rms <= 2e-5
