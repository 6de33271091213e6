"""One small invocation of the whole hot path on the `_low`-shaped voice (so every fused tensor-core kernel launches),
meant to run under compute-sanitizer:
    compute-sanitizer --tool memcheck|racecheck|synccheck python tools/sanitize_run.py [--default]
No oracle, no timing; three short ragged utterances, voice-default noise scales.  --default: the ResBlock1 generator
of the reference ModelConfig defaults (synth_voice.default_config) instead."""
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from mimic3_b200 import synth_voice as sv  # noqa: E402
from mimic3_b200.engine import B200Session  # noqa: E402


def main():
    with tempfile.TemporaryDirectory() as d:
        vd = Path(d) / "voice"
        cfg = sv.default_config(n_speakers=3) if "--default" in sys.argv[1:] else sv.low_config(n_speakers=3)
        sv.write_voice(vd, cfg, seed=5)
        sess = B200Session(str(vd), device=0)
        rng = np.random.default_rng(1)
        lengths = np.array([23, 9, 14], dtype=np.int64)
        ids = np.zeros((3, 23), dtype=np.int64)
        for b, L in enumerate(lengths):
            ids[b, :L] = rng.integers(4, 40, size=L)
        r = sess.infer(ids, lengths, (0.667, 1.0, 0.8), np.array([0, 2, 1], dtype=np.int64), seed=3, keep_float=True)
        a = np.concatenate([r.utterance_audio(b) for b in range(3)])
        assert np.isfinite(a).all()
        print(f"sanitize_run ok: {r.total_samples} samples, {r.launches} launches")
        sess.close()


if __name__ == "__main__":
    main()
