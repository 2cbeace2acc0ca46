"""TEST INFRASTRUCTURE ONLY -- stores the reference's symbol tables, inference text and model config as fixtures.

    python oracle/make_golden_tables.py          (needs the reference tree, see oracle/refshim.py)

Writes under tests/golden/:
* reference_text/{tokenlist,speaker2,inference_text}: byte copies of the reference's data/youdao/text/tokenlist,
  data/youdao/text/speaker2 and data/inference/text (tests/test_frontdoor.py parses them with the front door);
* reference_config.json: the ``model`` section, ``n_mels`` and ``segment_size`` of the reference's config/joint/config.yaml
  (tests/test_host_logic.py holds default_config() to them)."""
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refshim                                   # noqa: E402

TEXT_FILES = {"tokenlist": "data/youdao/text/tokenlist", "speaker2": "data/youdao/text/speaker2",
              "inference_text": "data/inference/text"}


def main():
    gold = os.path.join(ROOT, "tests", "golden")
    os.makedirs(os.path.join(gold, "reference_text"), exist_ok=True)
    for name, rel in TEXT_FILES.items():
        shutil.copyfile(os.path.join(refshim.REF_ROOT, rel), os.path.join(gold, "reference_text", name))
    conf = refshim.load_reference_config()
    with open(os.path.join(gold, "reference_config.json"), "w") as f:
        json.dump({"source": "config/joint/config.yaml of the reference", "model": conf.model,
                   "n_mels": conf.n_mels, "segment_size": conf.segment_size}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", sorted(TEXT_FILES), "and reference_config.json to", gold)


if __name__ == "__main__":
    main()
