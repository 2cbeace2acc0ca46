"""Host plumbing either side of the hot path (SURVEY.md s8f rank 3): the 4-field input contract and the
micro-batching queue.  CPU only (a fake model stands in for the engine)."""
import os
import threading

import numpy as np
import pytest
import torch

from emotivoice_b200 import frontdoor as fd

# byte copies of the reference's data/youdao/text/{tokenlist,speaker2} and data/inference/text (oracle/make_golden_tables.py)
REF_TEXT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_text")


def test_parse_and_encode_follow_the_reference_contract(tmp_path):
    tok = tmp_path / "tokenlist"
    tok.write_text("_\n<sos/eos>\n[AA0]\nengsp1\nuo3\n")
    spk = tmp_path / "speaker2"
    spk.write_text("8051\n11614\n")
    t2i, s2i = fd.load_symbol_table(str(tok)), fd.load_symbol_table(str(spk))
    assert t2i == {"_": 0, "<sos/eos>": 1, "[AA0]": 2, "engsp1": 3, "uo3": 4} and s2i == {"8051": 0, "11614": 1}
    r = fd.parse_line("11614|Happy|<sos/eos>  [AA0] engsp1 uo3 <sos/eos>|hello | world\n")
    assert r.speaker == "11614" and r.prompt == "Happy" and r.phonemes == ["<sos/eos>", "[AA0]", "engsp1", "uo3", "<sos/eos>"]
    assert r.content == "hello "            # the reference takes field 3 only
    ids, s = fd.encode(r, t2i, s2i)
    assert ids.tolist() == [1, 2, 3, 4, 1] and ids.dtype == np.int64 and s == 1
    assert fd.encode(r._replace(speaker="nobody"), t2i, s2i) is None       # unknown speaker: skipped (:109-110)
    with pytest.raises(KeyError):
        fd.encode(r._replace(phonemes=["zz9"]), t2i, s2i)                  # unknown phoneme: KeyError like the reference
    with pytest.raises(ValueError):
        fd.parse_line("only|three|fields")


def test_reference_inference_fixture_parses_with_the_reference_tables():
    t2i = fd.load_symbol_table(os.path.join(REF_TEXT, "tokenlist"))
    s2i = fd.load_symbol_table(os.path.join(REF_TEXT, "speaker2"))
    assert len(t2i) == 502 and t2i["_"] == 0 and t2i["<sos/eos>"] == 1
    lens = []
    with open(os.path.join(REF_TEXT, "inference_text"), encoding="utf-8") as f:
        for line in f:
            enc = fd.encode(fd.parse_line(line), t2i, s2i)
            assert enc is not None and enc[0][0] == 1 and enc[0].max() <= 416
            lens.append(len(enc[0]))
    assert lens == [58, 27, 9, 92, 110, 111, 156, 137, 95, 223, 173, 177]       # SURVEY.md s4


def test_collate_pads_with_zero_and_keeps_dtypes():
    items = [(np.array([1, 5, 1]), 3, np.ones(768, np.float32), np.zeros(768, np.float32)),
             (np.array([1, 7, 8, 9, 1]), 4, np.zeros(768, np.float32), np.ones(768, np.float32))]
    b = fd.collate(items)
    assert b["inputs_ling"].tolist() == [[1, 5, 1, 0, 0], [1, 7, 8, 9, 1]] and b["inputs_ling"].dtype == torch.int64
    assert b["input_lengths"].tolist() == [3, 5] and b["inputs_speaker"].tolist() == [3, 4]
    assert b["inputs_style_embedding"].shape == (2, 768) and b["inputs_style_embedding"].dtype == torch.float32


def _fake_model(calls):
    def forward(inputs_ling, input_lengths, inputs_speaker, inputs_style_embedding, inputs_content_embedding):
        calls.append(int(inputs_ling.shape[0]))
        B, T = inputs_ling.shape
        mel = (input_lengths * 2).to(torch.int32)                       # 2 frames per phoneme
        wav = torch.zeros(B, 1, int(mel.max()) * 256)
        for b in range(B):
            wav[b, 0, :int(mel[b]) * 256] = float(inputs_speaker[b]) + inputs_ling[b, :int(input_lengths[b])].sum().item() * 1e-3
        return {"wav_predictions": wav, "mel_lengths": mel}
    return forward


def test_microbatcher_groups_requests_and_returns_per_item_results():
    calls = []
    with fd.MicroBatcher(_fake_model(calls), max_batch=4, max_wait_s=0.2) as mb:
        futs, want = [], []
        barrier = threading.Barrier(6)

        def worker(i):
            ids = np.arange(1, 3 + i)
            barrier.wait()
            futs.append((i, mb.submit(ids, i, np.zeros(768, np.float32), np.zeros(768, np.float32))))

        ths = [threading.Thread(target=worker, args=(i,)) for i in range(6)]
        [t.start() for t in ths]
        [t.join() for t in ths]
        for i, f in futs:
            w = f.result(timeout=10)
            n = 2 + i
            assert w.shape == (n * 2 * 256,)                               # trimmed to the item's own length
            assert torch.allclose(w, torch.full_like(w, i + sum(range(1, 3 + i)) * 1e-3))
    assert sum(calls) == 6 and max(calls) <= 4 and len(calls) <= 3         # grouped, never above max_batch


def test_microbatcher_delivers_errors_and_keeps_serving():
    state = {"fail": True}

    def forward(**kw):
        if state["fail"]:
            state["fail"] = False
            raise RuntimeError("boom")
        return _fake_model([])(**kw)

    with fd.MicroBatcher(forward, max_batch=2, max_wait_s=0.01) as mb:
        f1 = mb.submit(np.array([1, 2]), 0, np.zeros(768, np.float32), np.zeros(768, np.float32))
        with pytest.raises(RuntimeError, match="boom"):
            f1.result(timeout=10)
        f2 = mb.submit(np.array([1, 2, 3]), 1, np.zeros(768, np.float32), np.zeros(768, np.float32))
        assert f2.result(timeout=10).shape == (3 * 2 * 256,)
    with pytest.raises(RuntimeError):
        mb.submit(np.array([1]), 0, np.zeros(768, np.float32), np.zeros(768, np.float32))


def test_wav_container_is_the_canonical_pcm16_file():
    """SURVEY.md s8f rank 2: 16 kHz mono PCM16 RIFF, readable by the stdlib and byte-identical to scipy's writer."""
    import io
    import wave
    from scipy.io import wavfile
    rng = np.random.default_rng(0)
    for n in (0, 1, 12345):
        pcm = rng.integers(-32768, 32768, size=n).astype(np.int16)
        img = fd.pcm16_to_wav_bytes(pcm, 16000)
        assert len(img) == 44 + 2 * n
        with wave.open(io.BytesIO(img)) as w:
            assert (w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()) == (1, 2, 16000, n)
            assert np.array_equal(np.frombuffer(w.readframes(n), "<i2"), pcm)
        ref = io.BytesIO()
        wavfile.write(ref, 16000, pcm)
        assert ref.getvalue() == img
    with pytest.raises(ValueError):
        fd.pcm16_to_wav_bytes(np.zeros(4, np.float32))
    with pytest.raises(ValueError):
        fd.pcm16_to_wav_bytes(np.zeros((2, 4), np.int16))


def test_prompt_embedding_cache_batches_dedups_and_evicts():
    calls = []

    def tokenizer(texts, return_tensors="pt", padding=True):
        n = max(len(t) for t in texts)
        ids = torch.zeros((len(texts), n), dtype=torch.long)
        mask = torch.zeros_like(ids)
        for i, t in enumerate(texts):
            ids[i, :len(t)] = torch.tensor([ord(c) for c in t])
            mask[i, :len(t)] = 1
        return {"input_ids": ids, "token_type_ids": torch.zeros_like(ids), "attention_mask": mask}

    def encoder(input_ids, token_type_ids, attention_mask):
        calls.append(int(input_ids.shape[0]))
        s = (input_ids * attention_mask).sum(1, keepdim=True).float()
        return {"pooled_output": s.repeat(1, 4) / 1000.0}

    cache = fd.PromptEmbeddingCache(tokenizer, encoder, max_entries=3)
    e = cache.embed(["Happy", "Sad", "Happy", "hello world"])
    assert e.shape == (4, 4) and torch.equal(e[0], e[2]) and not torch.equal(e[0], e[1])
    assert calls == [3] and cache.forwards == 1 and (cache.hits, cache.misses) == (0, 4)      # one forward for the 3 distinct texts
    e2 = cache.embed(["Sad", "Happy"])
    assert calls == [3] and torch.equal(e2[0], e[1]) and cache.hits == 2                       # served from the cache
    cache.embed(["a", "b"])                                                                    # 5 distinct texts > 3 entries: LRU eviction
    assert calls == [3, 2] and len(cache._cache) == 3 and "hello world" not in cache._cache
    assert torch.equal(cache.embed(["hello world"])[0], e[3]) and calls == [3, 2, 1]


def test_collate_accepts_tensor_rows_and_cache_rows_survive_eviction():
    """ADVICE r1: PromptEmbeddingCache.embed returns tensors (on the encoder's device); collate must take them, and embed must
    not lose its own rows when the cache is smaller than the request."""
    import numpy as np
    import torch
    from emotivoice_b200 import frontdoor
    items = [(np.arange(5), 1, torch.ones(8), np.zeros(8, np.float32)), (np.arange(3), 2, torch.zeros(8), torch.ones(8))]
    b = frontdoor.collate(items)
    assert b["inputs_style_embedding"].shape == (2, 8) and b["inputs_content_embedding"].dtype == torch.float32
    assert b["inputs_ling"].shape == (2, 5) and b["input_lengths"].tolist() == [5, 3]

    class Tok:
        def __call__(self, texts, return_tensors="pt", padding=True):
            ids = torch.tensor([[len(t)] for t in texts])
            return {"input_ids": ids, "token_type_ids": torch.zeros_like(ids), "attention_mask": torch.ones_like(ids)}

    def enc(input_ids, token_type_ids, attention_mask):
        return {"pooled_output": input_ids.float().repeat(1, 4)}

    cache = frontdoor.PromptEmbeddingCache(Tok(), enc, max_entries=2)
    out = cache.embed(["a", "bb", "ccc", "a", "dddd"])          # more distinct texts than the cache holds
    assert out[:, 0].tolist() == [1.0, 2.0, 3.0, 1.0, 4.0]
    assert len(cache._cache) == 2 and cache.forwards == 1
    assert cache.embed(["dddd", "a"])[:, 0].tolist() == [4.0, 1.0]
