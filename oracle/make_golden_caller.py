"""TEST INFRASTRUCTURE ONLY -- fixtures for the caller-level drop-in test (tests/test_caller_dropin_gpu.py).

    python oracle/make_golden_caller.py          (build container: needs /root/reference)

Runs oracle/caller_loop.run_caller_loop with the UNMODIFIED reference ``JETSGenerator`` class on the reference's own
data/inference/text (12 lines), token / speaker tables and config.yaml, with the seeded synthetic checkpoint, on the CPU with
pinned arithmetic (caller_loop.PINNED_CPU_ENV: the script re-executes itself with it), so the files are reproducible on any host.
Writes tests/golden/caller_lines.json (the 12 lines + the two symbol tables restricted to the symbols they use -- data, so the
test needs no reference tree) and tests/golden/caller_ref_pcm.npz (the reference's int16 output for every line, as sample
counts + sha1, and the full waveform of the three shortest lines)."""
import hashlib
import json
import os
import sys
import zipfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from emotivoice_b200 import synth                           # noqa: E402
from oracle import caller_loop, refshim                      # noqa: E402


def save_npz_lzma(path, **arrays):
    """np.savez_compressed with LZMA members and fixed member dates: about half the size for int16 audio, the same bytes on every
    run; np.load reads it like any .npz."""
    with zipfile.ZipFile(path, "w") as zf:
        for k, a in arrays.items():
            info = zipfile.ZipInfo(k + ".npy")
            info.compress_type = zipfile.ZIP_LZMA
            with zf.open(info, "w") as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def main():
    if any(os.environ.get(k) != v for k, v in caller_loop.PINNED_CPU_ENV.items()):
        os.execve(sys.executable, [sys.executable] + sys.argv, dict(os.environ, **caller_loop.PINNED_CPU_ENV))
    caller_loop.pin_cpu_math()
    ref_root = refshim.REF_ROOT
    lines = [l.rstrip("\n") for l in open(os.path.join(ref_root, "data", "inference", "text"), encoding="utf-8") if l.strip()]
    token2id = {t.strip(): i for i, t in enumerate(open(os.path.join(ref_root, "data", "youdao", "text", "tokenlist"), encoding="utf-8"))}
    speaker2id = {t.strip(): i for i, t in enumerate(open(os.path.join(ref_root, "data", "youdao", "text", "speaker2"), encoding="utf-8"))}
    used_tok = sorted({ph for l in lines for ph in l.split("|")[2].split()})
    used_spk = sorted({l.split("|")[0] for l in lines})
    conf = refshim.load_reference_config(len(token2id), len(speaker2id))
    from emotivoice_b200.config import default_config
    sd = synth.make_state_dict(default_config(len(token2id), len(speaker2id)))
    JETS = refshim.import_reference_jets()
    res = caller_loop.run_caller_loop(JETS, conf, sd, lines, token2id, speaker2id, torch.device("cpu"))
    gold = os.path.join(ROOT, "tests", "golden")
    with open(os.path.join(gold, "caller_lines.json"), "w", encoding="utf-8") as f:
        json.dump({"source": "data/inference/text, data/youdao/text/tokenlist, data/youdao/text/speaker2 of the reference",
                   "n_vocab": len(token2id), "n_speaker": len(speaker2id), "lines": lines,
                   "token2id": {t: token2id[t] for t in used_tok}, "speaker2id": {s: speaker2id[s] for s in used_spk}}, f, ensure_ascii=False, indent=0)
    order = sorted(res, key=lambda r: len(r[1]))
    keep = {n for n, _ in order[:3]}
    arrays = {"n_samples": np.array([len(a) for _, a in res], dtype=np.int64), "line_no": np.array([n for n, _ in res], dtype=np.int64)}
    digests = {}
    for n, a in res:
        digests[str(n)] = hashlib.sha1(a.tobytes()).hexdigest()
        if n in keep:
            arrays["pcm_%d" % n] = a
    save_npz_lzma(os.path.join(gold, "caller_ref_pcm.npz"), **arrays)
    with open(os.path.join(gold, "caller_ref_digests.json"), "w") as f:
        json.dump({"sha1_of_reference_int16": digests, "torch": torch.__version__}, f, indent=1)
    print("lines", len(res), "samples", arrays["n_samples"].tolist(), "kept", sorted(keep))


if __name__ == "__main__":
    main()
