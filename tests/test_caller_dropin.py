"""Caller-level drop-in test (SURVEY.md s8b; VERDICT r1 next#9): the reference CLI's synthesis loop
(inference_am_vocoder_joint.py:70-74, :104-134, restated once in oracle/caller_loop.py and parametrised by the JETSGenerator
CLASS) is run on the reference's own 12 lines of data/inference/text with only the class swapped:

* fixtures (tests/golden/caller_*) come from the UNMODIFIED reference class (oracle/make_golden_caller.py);
* on the CPU the oracle port, wrapped in the same class interface, must reproduce the reference's int16 files exactly (both
  computed with pinned CPU arithmetic, oracle/caller_loop.PINNED_CPU_ENV, in a process of their own);
* on the GPU ``emotivoice_b200.modules.JETSGenerator`` must produce the same number of samples for every line (identical
  durations) and int16 samples within 1 LSB of the reference's (fp32 rounding differences of ~1e-6 can flip a truncation)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from emotivoice_b200 import synth
from emotivoice_b200.config import default_config
from oracle import caller_loop, jets_oracle as O


def _fixture():
    with open(os.path.join(GOLDEN, "caller_lines.json"), encoding="utf-8") as f:
        meta = json.load(f)
    pcm = np.load(os.path.join(GOLDEN, "caller_ref_pcm.npz"))
    with open(os.path.join(GOLDEN, "caller_ref_digests.json")) as f:
        dig = json.load(f)["sha1_of_reference_int16"]
    return meta, pcm, dig


class OracleJETS:
    """oracle/jets_oracle.py behind the reference class's interface (constructor, .to, .load_state_dict, .eval, __call__)."""

    def __init__(self, conf):
        self.conf, self.sd = conf, None

    def to(self, device):
        return self

    def load_state_dict(self, sd):
        self.sd = sd

    def eval(self):
        return self

    def __call__(self, **kw):
        kw.pop("alpha", None)
        return O.jets_forward(self.sd, self.conf, **kw)


def oracle_on_the_stored_lines():
    """[(line number, int16 audio)] of the oracle behind the caller loop, for the lines whose full waveform the fixture keeps."""
    meta, pcm, _ = _fixture()
    conf = default_config(meta["n_vocab"], meta["n_speaker"])
    sd = synth.make_state_dict(conf)
    short = [n for n in pcm["line_no"].tolist() if "pcm_%d" % n in pcm.files]
    lines = [meta["lines"][n - 1] for n in short]
    res = caller_loop.run_caller_loop(OracleJETS, conf, sd, lines, meta["token2id"], meta["speaker2id"], torch.device("cpu"))
    assert len(res) == len(short)
    return [(n, audio) for (_, audio), n in zip(res, short)]


_ORACLE_CHILD = r"""
import os, sys
import numpy as np
sys.path[:0] = [sys.argv[1], os.path.join(sys.argv[1], "tests")]
from oracle import caller_loop
caller_loop.pin_cpu_math()
import test_caller_dropin
np.savez(sys.argv[2], **{"pcm_%d" % n: a for n, a in test_caller_dropin.oracle_on_the_stored_lines()})
"""


def test_oracle_behind_the_caller_loop_reproduces_the_reference_files_exactly(tmp_path):
    meta, pcm, dig = _fixture()
    out = str(tmp_path / "oracle_pcm.npz")
    subprocess.run([sys.executable, "-c", _ORACLE_CHILD, ROOT, out], env=dict(os.environ, **caller_loop.PINNED_CPU_ENV), check=True, timeout=900)
    res = np.load(out)
    short = [n for n in pcm["line_no"].tolist() if "pcm_%d" % n in pcm.files]
    assert sorted(res.files) == sorted("pcm_%d" % n for n in short)
    for n in short:
        audio = res["pcm_%d" % n]
        assert audio.dtype == np.int16 and np.array_equal(audio, pcm["pcm_%d" % n])
        assert hashlib.sha1(audio.tobytes()).hexdigest() == dig[str(n)]


@pytest.mark.gpu
def test_reference_caller_loop_with_only_the_class_swapped(dev, lib, tmp_path):
    from scipy.io import wavfile
    from emotivoice_b200.modules import JETSGenerator
    meta, pcm, dig = _fixture()
    conf = default_config(meta["n_vocab"], meta["n_speaker"])
    sd = synth.make_state_dict(conf)
    res = caller_loop.run_caller_loop(JETSGenerator, conf, sd, meta["lines"], meta["token2id"], meta["speaker2id"], dev, wav_dir=str(tmp_path))
    assert [n for n, _ in res] == pcm["line_no"].tolist()
    assert [len(a) for _, a in res] == pcm["n_samples"].tolist()            # identical durations on every line
    exact = 0
    for n, audio in res:
        assert audio.dtype == np.int16
        sr, filed = wavfile.read(os.path.join(str(tmp_path), "%d.wav" % n))       # the file the caller wrote
        assert sr == 16000 and np.array_equal(filed, audio)
        exact += int(hashlib.sha1(audio.tobytes()).hexdigest() == dig[str(n)])
        if "pcm_%d" % n in pcm.files:
            ref = pcm["pcm_%d" % n].astype(np.int32)
            d = np.abs(audio.astype(np.int32) - ref)
            print("line %d: %d samples, %d differ by 1 LSB, max |diff| %d" % (n, len(ref), int((d > 0).sum()), int(d.max())))
            assert d.max() <= 1 and (d > 0).mean() < 0.02
    print("lines bit-identical to the reference's int16 files: %d of %d" % (exact, len(res)))
