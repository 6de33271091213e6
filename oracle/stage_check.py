"""TEST INFRASTRUCTURE -- row-by-row comparison of one generator stage of the engine (E) with two float64
references of the same stage fed the same input (``VitsOracle.decoder_stage`` and friends):

* R64 -- plain float64;
* R16 -- float64 accumulation, with every conv the engine runs on the tensor cores fed operands rounded to the
  engine's 16-bit format (input after leaky-relu, and weights).

``rms_c(R16 - R64)`` of a row is the rounding error the 16-bit operands are expected to cause there, so it is the
row's budget.  Errors are judged row by row (one time step, all channels; for audio, one block of samples), so a
defect that touches a few rows -- a halo row at a CTA edge, the last row of an utterance, one N chunk -- is not
averaged away over a waveform.

Criteria (each a ratio that must stay <= 1 on every row):

* ``budget``: rms_c(E - R64) <= 3 * rms_c(R16 - R64) + floor -- every tensor-core stage;
* ``r16``:    rms_c(E - R16) <= 0.5 * rms_c(R16 - R64) + floor -- stages whose 16-bit staging R16 restates exactly
  (ResBlock1 generators: per-conv launches, fp32 accumulators and residual stream): E must sit at least twice as
  close to R16 as R16 sits to R64.  What separates E from R16 is fp32 accumulation and flips, where an
  intermediate the engine holds in fp32 and R16 in float64 rounds to different 16-bit neighbours.  The first
  expectation, 0.25, assumed flips are rare; they are not.  Once E and R16 differ slightly, every later 16-bit
  rounding along a resblock's chain of convs flips a share of elements proportional to that difference, by a
  whole unit in the last place each, so the gap settles at a fixed fraction of the rounding noise, in fp16 and bf16
  alike, on every row rather than at particular rows.  0.5 keeps this check six times tighter than ``budget``;
  the synthetic defects of ``tests/test_generator_ref.py`` (a dropped halo row, a shifted tap, a missing chunk
  bias) exceed it more than sixty-fold;
* ``fp32``:   max_c |E - R64| <= 1e-5 * rms(R64) -- stages that run no tensor-core conv at all.

floor = 1e-6 * rms(R64) over the utterance's stage, so that rows whose budget is exactly zero (no rounding error
at all, e.g. rows of a constant bias) do not divide by zero.
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np

BUDGET_X = 3.0
R16_X = 0.5
FLOOR = 1e-6
FP32_MAX = 1e-5
CTA_ROWS = (256, 128)


def audio_rows(a: np.ndarray, block: int = 64) -> np.ndarray:
    """A waveform as rows of ``block`` samples (the last row zero-padded)."""
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    n = -(-a.size // block) * block
    return np.pad(a, (0, n - a.size)).reshape(-1, block)


def _rms_rows(d: np.ndarray) -> np.ndarray:
    return np.sqrt(np.mean(np.square(d), axis=1))


def row_ratios(E: np.ndarray, R16: np.ndarray, R64: np.ndarray) -> Dict[str, np.ndarray]:
    """Per-row ratios of every criterion; E, R16, R64 are (rows, channels)."""
    E, R16, R64 = (np.asarray(a, dtype=np.float64) for a in (E, R16, R64))
    assert E.shape == R16.shape == R64.shape, (E.shape, R16.shape, R64.shape)
    scale = float(np.sqrt(np.mean(np.square(R64)))) if R64.size else 0.0
    floor = FLOOR * scale
    budget = _rms_rows(R16 - R64)
    return {
        "budget": _rms_rows(E - R64) / (BUDGET_X * budget + floor),
        "r16": _rms_rows(E - R16) / (R16_X * budget + floor),
        "fp32": np.max(np.abs(E - R64), axis=1) / (FP32_MAX * scale),
    }


def check_rows(E, R16, R64, criteria: Sequence[str], where: str = "", row_scale: int = 1
               ) -> Tuple[Dict[str, float], List[str]]:
    """Worst ratio per criterion and one message per failing criterion: the worst row, its offset from the
    start of a 256- and a 128-row CTA, and how many rows fail.  ``row_scale`` converts a row index to the
    stage's row index (64 for audio blocks) for that report."""
    ratios = row_ratios(E, R16, R64)
    worst: Dict[str, float] = {}
    fails: List[str] = []
    n = ratios["budget"].shape[0]
    for c in criteria:
        r = ratios[c]
        if not r.size:
            continue
        i = int(np.argmax(r))
        worst[c] = float(r[i])
        if not np.all(r <= 1.0):  # NaN fails too
            bad = int(np.sum(~(r <= 1.0)))
            row = i * row_scale
            edge = ", ".join(f"row % {m} = {row % m}" for m in CTA_ROWS)
            last = " (last row)" if i == n - 1 else ""
            fails.append(f"{where}: {c} ratio {r[i]:.3g} at row {row}{last} [{edge}]; {bad} of {n} rows fail")
    return worst, fails
