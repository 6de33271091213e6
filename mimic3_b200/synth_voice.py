"""Synthetic Mimic 3 voice directories (random weights, config-correct shapes).

No real voice (``generator.onnx`` from MycroftAI/mimic3-voices) is reachable from
this sandbox, so every test and benchmark runs on voices written by this module:
the same directory layout ``Mimic3Voice.load_from_directory`` reads
(reference ``mimic3_tts/voice.py:246-321``: ``config.json``, ``phonemes.txt``,
``generator.onnx``, optional ``speaker_map.csv``/``speakers.txt``) with the
hyper-parameters of the shipped ``*_low`` voices (SURVEY.md §0.5, §2.3) and
initializers named like the PyTorch module tree (SURVEY.md Appendix B).

Three initializer styles mirror what a TorchScript ONNX export can produce for
the weight-normalised WN convolutions of the flow:

* ``named``      -- plain ``...in_layers.0.weight`` initializers;
* ``weightnorm`` -- ``weight_g`` / ``weight_v`` pairs (fused ``g*v/||v||`` at load);
* ``folded``     -- constant-folded anonymous ``onnx::Conv_NNN`` weights that are
  only reachable through the Conv node that also consumes the named bias.

Also supports "tiny" shapes so CPU tests stay fast.
"""
from __future__ import annotations

import json
from dataclasses import dataclass, field, asdict
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import onnx_writer as ow


@dataclass
class SynthModelConfig:
    """Mirror of reference ``ModelConfig`` (``mimic3_tts/config.py:113-139``)."""

    num_symbols: int = 50
    n_speakers: int = 1
    inter_channels: int = 192
    hidden_channels: int = 192
    filter_channels: int = 768
    n_heads: int = 2
    n_layers: int = 6
    kernel_size: int = 3
    p_dropout: float = 0.1
    resblock: str = "2"
    resblock_kernel_sizes: Tuple[int, ...] = (3, 5, 7)
    resblock_dilation_sizes: Tuple[Tuple[int, ...], ...] = ((1, 2), (2, 6), (3, 12))
    upsample_rates: Tuple[int, ...] = (8, 8, 4)
    upsample_initial_channel: int = 256
    upsample_kernel_sizes: Tuple[int, ...] = (16, 16, 8)
    n_layers_q: int = 3
    use_spectral_norm: bool = False
    gin_channels: int = 0
    use_sdp: bool = True


def low_config(n_speakers: int = 1, num_symbols: int = 50) -> SynthModelConfig:
    """Shapes of the shipped ``*_low`` voices ([SIZE]-inferred, SURVEY.md §2.3)."""
    return SynthModelConfig(
        num_symbols=num_symbols,
        n_speakers=n_speakers,
        gin_channels=512 if n_speakers > 1 else 0,
    )


def default_config(n_speakers: int = 1, num_symbols: int = 50) -> SynthModelConfig:
    """Generator of the reference ``ModelConfig`` defaults (``mimic3_tts/config.py:126-135``):
    ResBlock1, 512 initial channels, upsampling 8*8*2*2 -- what a voice gets when its
    training config leaves the generator section alone."""
    return SynthModelConfig(
        num_symbols=num_symbols,
        n_speakers=n_speakers,
        resblock="1",
        resblock_kernel_sizes=(3, 7, 11),
        resblock_dilation_sizes=((1, 3, 5), (1, 3, 5), (1, 3, 5)),
        upsample_rates=(8, 8, 2, 2),
        upsample_initial_channel=512,
        upsample_kernel_sizes=(16, 16, 4, 4),
        gin_channels=512 if n_speakers > 1 else 0,
    )


def tiny_config(n_speakers: int = 1, num_symbols: int = 20, resblock: str = "2",
                use_sdp: bool = True) -> SynthModelConfig:
    """Small shapes for fast CPU/GPU tests; same graph, same code paths."""
    return SynthModelConfig(
        num_symbols=num_symbols,
        n_speakers=n_speakers,
        inter_channels=32,
        hidden_channels=32,
        filter_channels=64,
        n_heads=2,
        n_layers=2,
        resblock=resblock,
        resblock_kernel_sizes=(3, 5),
        resblock_dilation_sizes=((1, 2), (2, 3)) if resblock == "2" else ((1, 3), (1, 2)),
        upsample_rates=(4, 2),
        upsample_initial_channel=32,
        upsample_kernel_sizes=(8, 4),
        gin_channels=16 if n_speakers > 1 else 0,
        use_sdp=use_sdp,
    )


ATTN_WINDOW = 4          # VITS TextEncoder window_size [EXT]
FLOW_KERNEL = 5          # ResidualCouplingBlock WN kernel [EXT]
FLOW_WN_LAYERS = 4
FLOW_N_FLOWS = 4
SDP_KERNEL = 3
SDP_DDS_LAYERS = 3
SDP_N_FLOWS = 4
SDP_BINS = 10
DP_FILTER = 256          # plain DurationPredictor filter channels [EXT]


def _conv_w(rng, cout, cin, k, gain=1.0):
    std = gain / np.sqrt(cin * k)
    return (rng.standard_normal((cout, cin, k)) * std).astype(np.float32)


def _bias(rng, n, scale=0.05):
    return (rng.standard_normal(n) * scale).astype(np.float32)


def make_params(cfg: SynthModelConfig, seed: int = 0) -> Dict[str, np.ndarray]:
    """Random parameters keyed by PyTorch module path (SURVEY.md Appendix B)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    P: Dict[str, np.ndarray] = {}
    H, I, Ff = cfg.hidden_channels, cfg.inter_channels, cfg.filter_channels
    G = cfg.gin_channels if cfg.n_speakers > 1 else 0
    dk = H // cfg.n_heads

    P["enc_p.emb.weight"] = (rng.standard_normal((cfg.num_symbols, H)) * H ** -0.5).astype(np.float32)
    for l in range(cfg.n_layers):
        a = f"enc_p.encoder.attn_layers.{l}"
        for n in ("conv_q", "conv_k", "conv_v", "conv_o"):
            P[f"{a}.{n}.weight"] = _conv_w(rng, H, H, 1)
            P[f"{a}.{n}.bias"] = _bias(rng, H)
        P[f"{a}.emb_rel_k"] = (rng.standard_normal((1, 2 * ATTN_WINDOW + 1, dk)) * dk ** -0.5).astype(np.float32)
        P[f"{a}.emb_rel_v"] = (rng.standard_normal((1, 2 * ATTN_WINDOW + 1, dk)) * dk ** -0.5).astype(np.float32)
        for nm in ("norm_layers_1", "norm_layers_2"):
            P[f"enc_p.encoder.{nm}.{l}.gamma"] = (1.0 + 0.1 * rng.standard_normal(H)).astype(np.float32)
            P[f"enc_p.encoder.{nm}.{l}.beta"] = _bias(rng, H)
        f = f"enc_p.encoder.ffn_layers.{l}"
        P[f"{f}.conv_1.weight"] = _conv_w(rng, Ff, H, cfg.kernel_size, 1.4)
        P[f"{f}.conv_1.bias"] = _bias(rng, Ff)
        P[f"{f}.conv_2.weight"] = _conv_w(rng, H, Ff, cfg.kernel_size, 1.4)
        P[f"{f}.conv_2.bias"] = _bias(rng, H)
    P["enc_p.proj.weight"] = _conv_w(rng, 2 * I, H, 1, 0.5)
    P["enc_p.proj.bias"] = _bias(rng, 2 * I)

    def dds(prefix, ch):
        for i in range(SDP_DDS_LAYERS):
            P[f"{prefix}.convs_sep.{i}.weight"] = (rng.standard_normal((ch, 1, SDP_KERNEL)) * 0.6).astype(np.float32)
            P[f"{prefix}.convs_sep.{i}.bias"] = _bias(rng, ch)
            P[f"{prefix}.convs_1x1.{i}.weight"] = _conv_w(rng, ch, ch, 1, 1.2)
            P[f"{prefix}.convs_1x1.{i}.bias"] = _bias(rng, ch)
            for nm in ("norms_1", "norms_2"):
                P[f"{prefix}.{nm}.{i}.gamma"] = (1.0 + 0.1 * rng.standard_normal(ch)).astype(np.float32)
                P[f"{prefix}.{nm}.{i}.beta"] = _bias(rng, ch)

    if cfg.use_sdp:
        Fd = H  # SDP overrides filter_channels = in_channels [EXT]
        P["dp.pre.weight"] = _conv_w(rng, Fd, H, 1)
        P["dp.pre.bias"] = _bias(rng, Fd)
        P["dp.proj.weight"] = _conv_w(rng, Fd, Fd, 1)
        P["dp.proj.bias"] = _bias(rng, Fd)
        if G:
            P["dp.cond.weight"] = _conv_w(rng, Fd, G, 1)
            P["dp.cond.bias"] = _bias(rng, Fd)
        dds("dp.convs", Fd)
        # logw = (z0 - m0) * exp(-logs0): centre durations around ~3 frames / id
        # (constants chosen empirically for these random weights; see DESIGN.md)
        if H >= 128:
            P["dp.flows.0.m"] = np.array([[-6.0], [0.2]], dtype=np.float32)
            P["dp.flows.0.logs"] = np.array([[1.5], [-0.1]], dtype=np.float32)
        else:
            P["dp.flows.0.m"] = np.array([[-1.6], [0.2]], dtype=np.float32)
            P["dp.flows.0.logs"] = np.array([[0.0], [-0.1]], dtype=np.float32)
        for n in (3, 5, 7):  # flows.1 is the dropped "useless vflow"
            p = f"dp.flows.{n}"
            P[f"{p}.pre.weight"] = (rng.standard_normal((Fd, 1, 1)) * 0.7).astype(np.float32)
            P[f"{p}.pre.bias"] = _bias(rng, Fd)
            dds(f"{p}.convs", Fd)
            P[f"{p}.proj.weight"] = _conv_w(rng, 3 * SDP_BINS - 1, Fd, 1, 1.0)
            P[f"{p}.proj.bias"] = _bias(rng, 3 * SDP_BINS - 1, 0.3)
    else:
        P["dp.conv_1.weight"] = _conv_w(rng, DP_FILTER, H, 3, 1.4)
        P["dp.conv_1.bias"] = _bias(rng, DP_FILTER)
        P["dp.norm_1.gamma"] = (1.0 + 0.1 * rng.standard_normal(DP_FILTER)).astype(np.float32)
        P["dp.norm_1.beta"] = _bias(rng, DP_FILTER)
        P["dp.conv_2.weight"] = _conv_w(rng, DP_FILTER, DP_FILTER, 3, 1.4)
        P["dp.conv_2.bias"] = _bias(rng, DP_FILTER)
        P["dp.norm_2.gamma"] = (1.0 + 0.1 * rng.standard_normal(DP_FILTER)).astype(np.float32)
        P["dp.norm_2.beta"] = _bias(rng, DP_FILTER)
        P["dp.proj.weight"] = _conv_w(rng, 1, DP_FILTER, 1, 0.6)
        P["dp.proj.bias"] = np.array([1.1], dtype=np.float32)
        if G:
            P["dp.cond.weight"] = _conv_w(rng, H, G, 1)
            P["dp.cond.bias"] = _bias(rng, H)

    half = I // 2
    Hf = H
    for n in range(0, 2 * FLOW_N_FLOWS, 2):
        p = f"flow.flows.{n}"
        P[f"{p}.pre.weight"] = _conv_w(rng, Hf, half, 1)
        P[f"{p}.pre.bias"] = _bias(rng, Hf)
        for i in range(FLOW_WN_LAYERS):
            P[f"{p}.enc.in_layers.{i}.weight"] = _conv_w(rng, 2 * Hf, Hf, FLOW_KERNEL, 1.3)
            P[f"{p}.enc.in_layers.{i}.bias"] = _bias(rng, 2 * Hf)
            rs = 2 * Hf if i < FLOW_WN_LAYERS - 1 else Hf
            P[f"{p}.enc.res_skip_layers.{i}.weight"] = _conv_w(rng, rs, Hf, 1, 1.0)
            P[f"{p}.enc.res_skip_layers.{i}.bias"] = _bias(rng, rs)
        if G:
            P[f"{p}.enc.cond_layer.weight"] = _conv_w(rng, 2 * Hf * FLOW_WN_LAYERS, G, 1, 0.7)
            P[f"{p}.enc.cond_layer.bias"] = _bias(rng, 2 * Hf * FLOW_WN_LAYERS)
        P[f"{p}.post.weight"] = _conv_w(rng, half, Hf, 1, 0.5)
        P[f"{p}.post.bias"] = _bias(rng, half)

    C = cfg.upsample_initial_channel
    P["dec.conv_pre.weight"] = _conv_w(rng, C, I, 7, 1.0)
    P["dec.conv_pre.bias"] = _bias(rng, C)
    if G:
        P["dec.cond.weight"] = _conv_w(rng, C, G, 1, 0.5)
        P["dec.cond.bias"] = _bias(rng, C)
    nk = len(cfg.resblock_kernel_sizes)
    for i, (u, k) in enumerate(zip(cfg.upsample_rates, cfg.upsample_kernel_sizes)):
        cin, cout = C >> i, C >> (i + 1)
        # ConvTranspose1d weight layout (C_in, C_out, k); ~k/u taps overlap per output
        std = 1.3 / np.sqrt(cin * k / u)
        P[f"dec.ups.{i}.weight"] = (rng.standard_normal((cin, cout, k)) * std).astype(np.float32)
        P[f"dec.ups.{i}.bias"] = _bias(rng, cout)
        for j, (rk, dil) in enumerate(zip(cfg.resblock_kernel_sizes, cfg.resblock_dilation_sizes)):
            rb = f"dec.resblocks.{i * nk + j}"
            for d in range(len(dil)):
                if cfg.resblock == "2":
                    P[f"{rb}.convs.{d}.weight"] = _conv_w(rng, cout, cout, rk, 0.7)
                    P[f"{rb}.convs.{d}.bias"] = _bias(rng, cout)
                else:
                    P[f"{rb}.convs1.{d}.weight"] = _conv_w(rng, cout, cout, rk, 1.0)
                    P[f"{rb}.convs1.{d}.bias"] = _bias(rng, cout)
                    P[f"{rb}.convs2.{d}.weight"] = _conv_w(rng, cout, cout, rk, 0.6)
                    P[f"{rb}.convs2.{d}.bias"] = _bias(rng, cout)
    clast = C >> len(cfg.upsample_rates)
    P["dec.conv_post.weight"] = _conv_w(rng, 1, clast, 7, 0.8)
    if G:
        P["emb_g.weight"] = rng.standard_normal((cfg.n_speakers, G)).astype(np.float32)
    return P


def _is_wn_weight(name: str) -> bool:
    return name.startswith("flow.flows.") and ".enc." in name and name.endswith(".weight")


def write_generator_onnx(path: Path, cfg: SynthModelConfig, params: Dict[str, np.ndarray],
                         style: str = "named", alt_encoding: bool = False) -> None:
    """Serialise ``params`` as an ONNX ModelProto (see module docstring for styles).

    The node list is a *skeleton*: one Conv/ConvTranspose node per convolution with
    its (X, W, B) inputs, which is what a binder needs to recover constant-folded
    weights; it is not an executable graph (nothing here could run it anyway)."""
    assert style in ("named", "weightnorm", "folded")
    inits: List[bytes] = []
    nodes: List[bytes] = []
    anon = 1000
    for idx, (name, arr) in enumerate(params.items()):
        enc = dict(packed_dims=alt_encoding and idx % 2 == 0,
                   use_float_data=alt_encoding and idx % 3 == 0)
        wname = name
        if _is_wn_weight(name) and style == "weightnorm":
            # v = arr * s_c (any per-channel scale), g = ||arr||_c  =>  g * v / ||v|| == arr
            s = (1.0 + 0.5 * np.sin(np.arange(arr.shape[0], dtype=np.float32)))[:, None, None]
            v = (arr * s).astype(np.float32)
            g = np.sqrt((arr.astype(np.float64) ** 2).sum(axis=(1, 2), keepdims=True)).astype(np.float32)
            base = name[: -len(".weight")]
            inits.append(ow.tensor_proto(base + ".weight_g", g, **enc))
            inits.append(ow.tensor_proto(base + ".weight_v", v, **enc))
            continue
        if _is_wn_weight(name) and style == "folded":
            wname = f"onnx::Conv_{anon}"
            anon += 7
        inits.append(ow.tensor_proto(wname, arr, **enc))
        if name.endswith(".weight") and arr.ndim == 3 and not name.startswith("enc_p.emb"):
            base = name[: -len(".weight")]
            op = "ConvTranspose" if base.startswith("dec.ups.") else "Conv"
            ins = [f"/{base}/in", wname]
            if base + ".bias" in params:
                ins.append(base + ".bias")
            nodes.append(ow.node_proto(op, ins, [f"/{base}/out"], name=f"/{base}/{op}",
                                       attrs=[ow.attr_ints("kernel_shape", [arr.shape[2]])]))
    inputs = [
        ow.value_info("input", ow.INT64, ["batch_size", "phonemes"]),
        ow.value_info("input_lengths", ow.INT64, ["batch_size"]),
        ow.value_info("scales", ow.FLOAT, [3]),
    ]
    if cfg.n_speakers > 1:
        inputs.append(ow.value_info("sid", ow.INT64, ["batch_size"]))
    outputs = [ow.value_info("output", ow.FLOAT, ["batch_size", 1, "time"])]
    Path(path).write_bytes(ow.model_proto(nodes, inits, inputs, outputs))


def weightnorm_effective(params_g: np.ndarray, params_v: np.ndarray) -> np.ndarray:
    """w = g * v / ||v||, norm over (C_in, k) per output channel (PyTorch dim=0)."""
    v = params_v.astype(np.float32)
    norm = np.sqrt((v.astype(np.float64) ** 2).sum(axis=(1, 2), keepdims=True)).astype(np.float32)
    return (params_g * (v / norm)).astype(np.float32)


def write_voice(voice_dir: Path, cfg: Optional[SynthModelConfig] = None, seed: int = 0,
                style: str = "named", alt_encoding: bool = False,
                sample_rate: int = 22050,
                inference: Optional[Dict[str, float]] = None,
                speakers: Optional[Sequence[str]] = None) -> Dict[str, np.ndarray]:
    """Write a complete voice directory; returns the parameter dict used."""
    cfg = cfg or low_config()
    voice_dir = Path(voice_dir)
    voice_dir.mkdir(parents=True, exist_ok=True)
    params = make_params(cfg, seed)
    write_generator_onnx(voice_dir / "generator.onnx", cfg, params, style, alt_encoding)

    hop = int(np.prod(cfg.upsample_rates))
    model = asdict(cfg)
    model["resblock_kernel_sizes"] = list(cfg.resblock_kernel_sizes)
    model["resblock_dilation_sizes"] = [list(d) for d in cfg.resblock_dilation_sizes]
    model["upsample_rates"] = list(cfg.upsample_rates)
    model["upsample_kernel_sizes"] = list(cfg.upsample_kernel_sizes)
    config = {
        "seed": 1234,
        "audio": {"filter_length": 1024, "hop_length": hop, "win_length": 1024,
                  "mel_channels": 80, "sample_rate": sample_rate, "sample_bytes": 2, "channels": 1},
        "model": model,
        "phonemes": {"phoneme_separator": " ", "word_separator": "#", "pad": "_", "bos": "^",
                     "eos": "$", "blank": "#", "blank_word": None, "blank_between": "words",
                     "blank_at_start": True, "blank_at_end": True, "simple_punctuation": True},
        "text_language": "en-us",
        "phonemizer": "symbols",
        "datasets": [{"name": "synthetic", "metadata_format": "text", "multispeaker": cfg.n_speakers > 1}],
        "inference": inference or {"length_scale": 1.0, "noise_scale": 0.667, "noise_w": 0.8},
        "version": 1,
    }
    (voice_dir / "config.json").write_text(json.dumps(config, indent=4))
    syms = ["_", "^", "$", "#"] + [chr(ord("a") + (i % 26)) + (str(i // 26) if i >= 26 else "")
                                     for i in range(max(0, cfg.num_symbols - 4))]
    (voice_dir / "phonemes.txt").write_text(
        "".join(f"{i} {s}\n" for i, s in enumerate(syms[: cfg.num_symbols])), encoding="utf-8")
    if cfg.n_speakers > 1:
        names = list(speakers) if speakers else [f"p{200 + i}" for i in range(cfg.n_speakers)]
        (voice_dir / "speakers.txt").write_text("".join(n + "\n" for n in names))
        (voice_dir / "speaker_map.csv").write_text(
            "".join(f"{i}|synthetic|{n}|spk{i}\n" for i, n in enumerate(names)))
    (voice_dir / "VERSION").write_text("0.0.1\n")
    return params
