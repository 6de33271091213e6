"""TEST INFRASTRUCTURE -- CPU fp32 restatement of the Mimic 3 ids->waveform path.

**Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module.  It is the checker, never the
product: the product path (``mimic3_b200``) fails loudly without its CUDA library.**

PARITY UNPINNED AT THE REFERENCE BOUNDARY (anchored on an independent implementation instead: on
identical weights this module matches Hugging Face transformers' ``VitsModel`` -- a separately written
port of the same published algorithm -- to 1-3e-7 waveform RMS with identical output lengths,
``tests/test_oracle_vs_hf_vits.py``).  In the reference this path is one opaque call,
``onnxruntime.InferenceSession.run`` on the voice's ``generator.onnx``
(``/root/reference/mimic3_tts/voice.py:230``), followed by
``audio_float_to_int16`` (``mimic3_tts/utils.py:237-244``).  Neither onnxruntime
(``requirements.txt:6``, ``onnxruntime>=1.6,<2.0``, un-vendored wheel) nor any
``generator.onnx`` (MycroftAI/mimic3-voices, pinned only by sha256 in
``mimic3_tts/voices.json``) exists in this sandbox, and the reference's golden
WAVs (``tests/apope_sample_*.wav``) are text->WAV and need both plus espeak-ng.
This file therefore restates the *published* VITS inference algorithm
(jaywalnut310/vits ``models.py``/``modules.py``/``attentions.py``/
``transforms.py`` as exported by MycroftAI/vits-train; SURVEY.md Appendix A) and
is anchored on the reference's own call site contract:

* inputs ``input`` int64 (1,T), ``input_lengths`` (1,), ``scales`` f32 (3,) =
  [noise_scale, length_scale, noise_w], optional ``sid`` (1,)  (voice.py:180-218);
* output float32 (1,1,S), squeezed (voice.py:230);
* per-utterance peak normalisation to int16 (utils.py:237-244);
* hyper-parameters from ``config.json`` ``model.*`` (config.py:113-139).

It always runs **batch 1** (voice.py:180-181 -- the reference never batches), so it
defines the per-utterance edge semantics the batched engine must reproduce.
"""
from __future__ import annotations

import json
import math
from pathlib import Path
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import onnx_min, philox

LRELU_SLOPE = 0.1
ATTN_WINDOW = 4
SDP_BINS = 10
SDP_TAIL = 5.0
MIN_BIN = 1e-3
MIN_DERIV = 1e-3


def audio_float_to_int16(audio: np.ndarray, max_wav_value: float = 32767.0) -> np.ndarray:
    """Restates ``mimic3_tts/utils.py:237-244`` under NumPy-2 (fp32) promotion."""
    audio = np.asarray(audio, dtype=np.float32)
    peak = np.float32(max(np.float32(0.01), np.max(np.abs(audio)))) if audio.size else np.float32(0.01)
    scale = np.float32(max_wav_value) / peak
    y = audio * scale
    y = np.clip(y, -max_wav_value, max_wav_value)
    return y.astype("int16")  # C truncation toward zero


class VitsOracle:
    def __init__(self, voice_dir: str):
        voice_dir = Path(voice_dir)
        self.config = json.loads((voice_dir / "config.json").read_text())
        self.m = self.config["model"]
        P = onnx_min.named_parameters(str(voice_dir / "generator.onnx"))
        self.P = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in P.items()
                  if v is not None and v.dtype == np.float32}
        self.H = int(self.m["hidden_channels"])
        self.I = int(self.m["inter_channels"])
        self.n_heads = int(self.m["n_heads"])
        self.n_layers = int(self.m["n_layers"])
        self.n_speakers = int(self.m.get("n_speakers", 1))
        self.multispeaker = self.n_speakers > 1
        self.use_sdp = bool(self.m.get("use_sdp", True))
        inf = self.config.get("inference", {})
        self.defaults = (float(inf.get("noise_scale", 0.667)), float(inf.get("length_scale", 1.0)),
                         float(inf.get("noise_w", 0.8)))
        self.sample_rate = int(self.config.get("audio", {}).get("sample_rate", 22050))

    # ---- helpers -------------------------------------------------------------
    def conv(self, x, name, dilation=1, padding=0, groups=1):
        return F.conv1d(x, self.P[name + ".weight"], self.P.get(name + ".bias"),
                        dilation=dilation, padding=padding, groups=groups)

    def ln(self, x, name):  # modules.LayerNorm: over channels, eps 1e-5
        return F.layer_norm(x.transpose(1, 2), (x.shape[1],), self.P[name + ".gamma"],
                            self.P[name + ".beta"], 1e-5).transpose(1, 2)

    # ---- A.1 text encoder ------------------------------------------------------
    def attention(self, x, l):
        a = f"enc_p.encoder.attn_layers.{l}"
        T = x.shape[2]
        nh, dk, W = self.n_heads, self.H // self.n_heads, ATTN_WINDOW
        q = self.conv(x, a + ".conv_q").view(1, nh, dk, T).transpose(2, 3)  # (1,nh,T,dk)
        k = self.conv(x, a + ".conv_k").view(1, nh, dk, T).transpose(2, 3)
        v = self.conv(x, a + ".conv_v").view(1, nh, dk, T).transpose(2, 3)
        q = q / math.sqrt(dk)
        scores = q @ k.transpose(-2, -1)  # (1,nh,T,T)
        Ek = self.P[a + ".emb_rel_k"][0]  # (2W+1, dk), shared by heads
        Ev = self.P[a + ".emb_rel_v"][0]
        idx = torch.arange(T)
        rel = idx[None, :] - idx[:, None]  # j - i
        band = rel.abs() <= W
        rel_logits = q @ Ek.t()  # (1,nh,T,2W+1)
        gather = (rel.clamp(-W, W) + W)[None, None].expand(1, nh, T, T)
        scores = scores + torch.where(band, rel_logits.gather(-1, gather), torch.zeros(()))
        p = F.softmax(scores, dim=-1)  # B=1: attn_mask is all ones
        out = p @ v
        pw = torch.where(band, p, torch.zeros(()))  # (1,nh,T,T)
        relw = torch.zeros(1, nh, T, 2 * W + 1)
        relw.scatter_add_(-1, gather, pw)
        out = out + relw @ Ev
        out = out.transpose(2, 3).contiguous().view(1, self.H, T)
        return self.conv(out, a + ".conv_o")

    def text_encoder(self, ids: torch.Tensor):
        x = self.P["enc_p.emb.weight"][ids] * math.sqrt(self.H)  # (T,H)
        x = x.t().unsqueeze(0)
        k = int(self.m.get("kernel_size", 3))
        pl, pr = (k - 1) // 2, k // 2
        for l in range(self.n_layers):
            y = self.attention(x, l)
            x = self.ln(x + y, f"enc_p.encoder.norm_layers_1.{l}")
            f = f"enc_p.encoder.ffn_layers.{l}"
            y = torch.relu(self.conv(F.pad(x, (pl, pr)), f + ".conv_1"))
            y = self.conv(F.pad(y, (pl, pr)), f + ".conv_2")
            x = self.ln(x + y, f"enc_p.encoder.norm_layers_2.{l}")
        stats = self.conv(x, "enc_p.proj")
        return x, stats[:, : self.I], stats[:, self.I:]

    # ---- A.2 duration predictors -----------------------------------------------
    def dds(self, x, prefix, g=None):
        if g is not None:
            x = x + g
        ch = x.shape[1]
        for i in range(3):
            d = 3 ** i
            y = self.conv(x, f"{prefix}.convs_sep.{i}", dilation=d, padding=d, groups=ch)
            y = F.gelu(self.ln(y, f"{prefix}.norms_1.{i}"))
            y = self.conv(y, f"{prefix}.convs_1x1.{i}")
            y = F.gelu(self.ln(y, f"{prefix}.norms_2.{i}"))
            x = x + y
        return x

    @staticmethod
    def rqs_inverse(y, uw, uh, ud):
        """Inverse rational-quadratic spline with linear tails (transforms.py [EXT]).
        y: (T,), uw/uh: (T,10), ud: (T,9)."""
        out = y.clone()
        inside = (y >= -SDP_TAIL) & (y <= SDP_TAIL)
        if not inside.any():
            return out
        const = math.log(math.exp(1 - MIN_DERIV) - 1)
        ud = F.pad(ud, (1, 1))
        ud[..., 0] = const
        ud[..., -1] = const
        yi, uw, uh, ud = y[inside], uw[inside], uh[inside], ud[inside]
        nb = uw.shape[-1]

        def knots(u):
            w = F.softmax(u, dim=-1)
            w = MIN_BIN + (1 - MIN_BIN * nb) * w
            cw = F.pad(torch.cumsum(w, dim=-1), (1, 0), value=0.0)
            cw = 2 * SDP_TAIL * cw - SDP_TAIL
            cw[..., 0] = -SDP_TAIL
            cw[..., -1] = SDP_TAIL
            return cw, cw[..., 1:] - cw[..., :-1]

        cumw, widths = knots(uw)
        cumh, heights = knots(uh)
        deriv = MIN_DERIV + F.softplus(ud)
        loc = cumh.clone()
        loc[..., -1] += 1e-6
        b = (torch.sum(yi[..., None] >= loc, dim=-1) - 1)[..., None]
        in_cumw = cumw.gather(-1, b)[..., 0]
        in_w = widths.gather(-1, b)[..., 0]
        in_cumh = cumh.gather(-1, b)[..., 0]
        delta = heights / widths
        in_delta = delta.gather(-1, b)[..., 0]
        d0 = deriv.gather(-1, b)[..., 0]
        d1 = deriv[..., 1:].gather(-1, b)[..., 0]
        in_h = heights.gather(-1, b)[..., 0]
        s = d0 + d1 - 2 * in_delta
        a = (yi - in_cumh) * s + in_h * (in_delta - d0)
        bb = in_h * d0 - (yi - in_cumh) * s
        c = -in_delta * (yi - in_cumh)
        disc = bb.pow(2) - 4 * a * c
        root = (2 * c) / (-bb - torch.sqrt(disc))
        out[inside] = root * in_w + in_cumw
        return out

    def sdp(self, x, g, noise_w, z_noise):
        h = self.conv(x, "dp.pre")
        if g is not None:
            h = h + self.conv(g, "dp.cond")
        h = self.dds(h, "dp.convs")
        h = self.conv(h, "dp.proj")
        z = z_noise * noise_w  # (1,2,T)
        Fd = h.shape[1]
        for n in (7, 5, 3):
            z = torch.flip(z, [1])
            p = f"dp.flows.{n}"
            z0, z1 = z[:, :1], z[:, 1:]
            u = self.conv(z0, p + ".pre")
            u = self.dds(u, p + ".convs", g=h)
            u = self.conv(u, p + ".proj")  # (1,29,T)
            u = u[0].t()
            uw = u[:, :SDP_BINS] / math.sqrt(Fd)
            uh = u[:, SDP_BINS:2 * SDP_BINS] / math.sqrt(Fd)
            ud = u[:, 2 * SDP_BINS:]
            z1 = self.rqs_inverse(z1[0, 0], uw, uh, ud)[None, None]
            z = torch.cat([z0, z1], 1)
        z = torch.flip(z, [1])
        z = (z - self.P["dp.flows.0.m"][None]) * torch.exp(-self.P["dp.flows.0.logs"][None])
        return z[:, :1]

    def dp_plain(self, x, g):
        if g is not None:
            x = x + self.conv(g, "dp.cond")
        x = torch.relu(self.conv(x, "dp.conv_1", padding=1))
        x = self.ln(x, "dp.norm_1")
        x = torch.relu(self.conv(x, "dp.conv_2", padding=1))
        x = self.ln(x, "dp.norm_2")
        return self.conv(x, "dp.proj")

    # ---- A.3 flow ----------------------------------------------------------------
    def wn(self, x, prefix, g):
        Hf = x.shape[1]
        out = torch.zeros_like(x)
        nl = 4
        gc = self.conv(g, prefix + ".cond_layer") if g is not None else None
        k = self.P[prefix + ".in_layers.0.weight"].shape[2]
        for i in range(nl):
            a = self.conv(x, f"{prefix}.in_layers.{i}", padding=(k - 1) // 2)
            if gc is not None:
                a = a + gc[:, i * 2 * Hf:(i + 1) * 2 * Hf]
            act = torch.tanh(a[:, :Hf]) * torch.sigmoid(a[:, Hf:])
            rs = self.conv(act, f"{prefix}.res_skip_layers.{i}")
            if i < nl - 1:
                x = x + rs[:, :Hf]
                out = out + rs[:, Hf:]
            else:
                out = out + rs
        return out

    def flow(self, z, g):
        half = self.I // 2
        for n in (6, 4, 2, 0):
            z = torch.flip(z, [1])
            p = f"flow.flows.{n}"
            x0, x1 = z[:, :half], z[:, half:]
            h = self.conv(x0, p + ".pre")
            h = self.wn(h, p + ".enc", g)
            m = self.conv(h, p + ".post")
            z = torch.cat([x0, x1 - m], 1)
        return z

    # ---- A.4 HiFi-GAN --------------------------------------------------------------
    # The generator is split into a pre-stage (conv_pre + speaker cond), one stage per upsampler (ConvTranspose1d
    # + MRF) and a post-stage (conv_post + tanh), so that a test can feed each stage the engine's own input.
    #
    # Each piece runs in the dtype of its input: float32 is the oracle itself, float64 a high-precision reference.
    # ``rounding`` maps a conv group -- "pre", f"ups{i}", f"mrf{i}", "post" -- to "fp16" or "bf16": the input of
    # every conv in that group (after its leaky-relu) and its float32 weights are rounded to that format before
    # the product, which is what the engine's tensor-core kernels stage.  Biases, residual adds and the
    # accumulation stay in the input dtype.  Groups not in ``rounding`` are not rounded.
    _RND = {"fp16": torch.float16, "bf16": torch.bfloat16}

    def _gconv(self, x, name, fmt, transpose=False, bias=True, **kw):
        """One generator conv in x's dtype; ``fmt`` rounds its operands (see above)."""
        w = self.P[name + ".weight"]
        b = self.P.get(name + ".bias") if bias else None
        if fmt is not None:
            x = x.to(self._RND[fmt]).to(x.dtype)
            w = w.to(self._RND[fmt])
        w = w.to(x.dtype)
        if b is not None:
            b = b.to(x.dtype)
        return self._conv1d(x, w, b, name, transpose, **kw)

    def _conv1d(self, x, w, b, name, transpose, **kw):
        """The single place every generator conv goes through (tests override it to inject defects)."""
        return (F.conv_transpose1d if transpose else F.conv1d)(x, w, b, **kw)

    def decoder_pre(self, z, g, rounding=None):
        x = self._gconv(z, "dec.conv_pre", (rounding or {}).get("pre"), padding=3)
        if g is not None:
            x = x + self._gconv(g.to(z.dtype), "dec.cond", None)
        return x

    def decoder_stage(self, i, x, rounding=None):
        """Upsampler i, then its multi-receptive-field fusion (the mean of nk resblocks)."""
        m = self.m
        rounding = rounding or {}
        u, k = m["upsample_rates"][i], m["upsample_kernel_sizes"][i]
        fu, fm = rounding.get(f"ups{i}"), rounding.get(f"mrf{i}")
        nk = len(m["resblock_kernel_sizes"])
        x = F.leaky_relu(x, LRELU_SLOPE)
        x = self._gconv(x, f"dec.ups.{i}", fu, transpose=True, stride=u, padding=(k - u) // 2)
        xs = None
        for j, (rk, dils) in enumerate(zip(m["resblock_kernel_sizes"], m["resblock_dilation_sizes"])):
            rb = f"dec.resblocks.{i * nk + j}"
            y = x
            for d_i, d in enumerate(dils):
                if str(m["resblock"]) == "2":
                    t = self._gconv(F.leaky_relu(y, LRELU_SLOPE), f"{rb}.convs.{d_i}", fm,
                                    dilation=d, padding=d * (rk - 1) // 2)
                else:
                    t = self._gconv(F.leaky_relu(y, LRELU_SLOPE), f"{rb}.convs1.{d_i}", fm,
                                    dilation=d, padding=d * (rk - 1) // 2)
                    t = self._gconv(F.leaky_relu(t, LRELU_SLOPE), f"{rb}.convs2.{d_i}", fm,
                                    dilation=1, padding=(rk - 1) // 2)
                y = y + t
            xs = y if xs is None else xs + y
        return xs / nk

    def decoder_post(self, x, rounding=None):
        x = F.leaky_relu(x)  # slope 0.01
        x = self._gconv(x, "dec.conv_post", (rounding or {}).get("post"), bias=False, padding=3)
        return torch.tanh(x)

    def decoder(self, z, g, taps=None):
        x = self.decoder_pre(z, g)
        for i in range(len(self.m["upsample_rates"])):
            x = self.decoder_stage(i, x)
            if taps is not None:
                taps[f"mrf{i}"] = x[0].t().numpy().copy()
        return self.decoder_post(x)

    # ---- A.0 top level ---------------------------------------------------------------
    def _front(self, ids, noise_w, length_scale, sid, seed, row):
        """Text encoder, speaker embedding and duration predictor: everything before the length regulator."""
        T = int(ids.shape[0])
        x, m_p, logs_p = self.text_encoder(ids)
        g = self.speaker(sid)
        if self.use_sdp:
            zn = torch.zeros(1, 2, T)
            if noise_w != 0:
                zn = torch.from_numpy(philox.normal(seed, 0, row, np.arange(T)[None, :], np.arange(2)[:, None]))[None]
            logw = self.sdp(x, g, float(noise_w), zn)
        else:
            logw = self.dp_plain(x, g)
        w = torch.exp(logw) * float(length_scale)
        dur = torch.ceil(w)[0, 0].to(torch.int64)
        return x, m_p, logs_p, g, logw, dur

    @torch.no_grad()
    def durations(self, ids, scales=None, sid: Optional[int] = None, seed: int = 0, row: int = 0) -> np.ndarray:
        """Integer frames per id, as ``infer`` computes them, without the flow and the decoder; the utterance has
        ``max(1, durations.sum())`` frames."""
        _, length_scale, noise_w = scales if scales is not None else self.defaults
        ids = torch.as_tensor(np.asarray(ids, dtype=np.int64))
        return self._front(ids, noise_w, length_scale, sid, seed, row)[5].numpy()

    def speaker(self, sid: Optional[int]):
        """The speaker embedding g (1, G, 1) the decoder's cond conv reads; None for single-speaker voices."""
        return self.P["emb_g.weight"][int(sid or 0)][None, :, None] if self.multispeaker else None

    @torch.no_grad()
    def infer(self, ids, scales=None, sid: Optional[int] = None, seed: int = 0, row: int = 0,
              return_intermediates: bool = False):
        """One utterance (batch 1).  ``scales`` = [noise_scale, length_scale, noise_w]
        (order fixed by voice.py:182-189).  ``row`` = the utterance's row in the engine
        batch (only selects the noise stream)."""
        torch.set_grad_enabled(False)
        noise_scale, length_scale, noise_w = scales if scales is not None else self.defaults
        ids = torch.as_tensor(np.asarray(ids, dtype=np.int64))
        T = int(ids.shape[0])
        inter: Dict[str, np.ndarray] = {}
        x, m_p, logs_p, g, logw, dur = self._front(ids, noise_w, length_scale, sid, seed, row)
        Fr = max(1, int(dur.sum()))
        cum = torch.cumsum(dur, 0)
        tok = torch.searchsorted(cum, torch.arange(Fr), right=True)  # frame -> token (cum[t-1] <= y < cum[t])
        valid = tok < T
        tokc = tok.clamp(max=T - 1)
        m_e = torch.where(valid[None, None], m_p[:, :, tokc], torch.zeros(()))
        logs_e = torch.where(valid[None, None], logs_p[:, :, tokc], torch.zeros(()))
        z_p = m_e
        if noise_scale != 0:
            eps = torch.from_numpy(philox.normal(seed, 1, row, np.arange(Fr)[None, :], np.arange(self.I)[:, None]))[None]
            z_p = m_e + eps * torch.exp(logs_e) * float(noise_scale)
        z = self.flow(z_p, g)
        o = self.decoder(z, g, inter if return_intermediates else None)
        audio = o[0, 0].numpy()
        if return_intermediates:
            inter.update(x=x[0].t().numpy(), m_p=m_p[0].t().numpy(), logs_p=logs_p[0].t().numpy(),
                         logw=logw[0, 0].numpy(), durations=dur.numpy(), z_p=z_p[0].t().numpy(),
                         z=z[0].t().numpy())
            return audio, inter
        return audio

    def infer_pcm(self, ids, scales=None, sid=None, seed: int = 0, row: int = 0) -> np.ndarray:
        return audio_float_to_int16(self.infer(ids, scales, sid, seed, row))
