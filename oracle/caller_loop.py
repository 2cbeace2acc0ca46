"""TEST INFRASTRUCTURE ONLY -- the reference CLI's synthesis loop, restated once and parametrised by the JETSGenerator CLASS.

inference_am_vocoder_joint.py:70-74 builds the model (``JETSGenerator(conf).to(device)``, ``load_state_dict(ckpt['generator'])``,
``.eval()``) and :104-134 turns each ``<speaker>|<prompt>|<phoneme>|<content>`` line into a 16 kHz int16 waveform.  The drop-in
claim of emotivoice_b200 is that ONLY the import of that class changes (INTEGRATION.md); this module is that loop with the class
passed in, so the same code runs with the unmodified reference class (oracle/make_golden_caller.py, build container) and with
``emotivoice_b200.modules.JETSGenerator`` (tests/test_caller_dropin_gpu.py, GPU box).

What cannot run offline is replaced exactly as SURVEY.md s8c prescribes: yacs -> the yaml attr-dict shim, the checkpoint -> the
seeded synthetic state dict, ``get_style_embedding`` (simbert BERT, :25-38) -> seeded 768-d vectors in the pooler's tanh range,
soundfile -> ``scipy.io.wavfile`` / the returned arrays.  Nothing in the product path imports this file.
"""
import numpy as np
import torch

MAX_WAV_VALUE = 32768.0      # models/hifigan/get_vocoder.py (imported by inference_am_vocoder_joint.py:20)

# The int16 files truncate fp32 samples, so one ulp anywhere in the forward can move a sample by one LSB, and the fp32 bits of a
# CPU forward depend on the thread count and on the vector ISA torch's kernels pick for the host.  Files that are compared bit for
# bit are therefore computed with pinned CPU arithmetic: one thread, ATen's baseline kernels, MKL's conditional numerical
# reproducibility mode and no oneDNN, which gives the same bits on any x86-64 host.  ATen and MKL read these variables when
# they load, so they go into the environment of a fresh process, which then calls pin_cpu_math() first.
PINNED_CPU_ENV = {"ATEN_CPU_CAPABILITY": "default", "MKL_CBWR": "COMPATIBLE", "OMP_NUM_THREADS": "1", "MKL_NUM_THREADS": "1"}


def pin_cpu_math():
    import os
    if any(os.environ.get(k) != v for k, v in PINNED_CPU_ENV.items()) or torch.backends.cpu.get_cpu_capability() != "DEFAULT":
        raise RuntimeError("pinned CPU arithmetic needs a process started with %s in its environment" % PINNED_CPU_ENV)
    torch.set_num_threads(1)
    torch.backends.mkldnn.enabled = False


def synthetic_style_embedding(text, seed=1234, dim=768):
    """Stand-in for get_style_embedding(prompt, tokenizer, style_encoder) (:25-38): a vector that depends only on the text,
    in tanh range like BertPooler's output; float32 numpy like ``output["pooled_output"].cpu().squeeze().numpy()``."""
    import zlib
    rng = np.random.default_rng([int(seed), zlib.crc32(text.encode("utf-8"))])
    return np.tanh(rng.normal(size=dim)).astype(np.float32)


def run_caller_loop(JETSGenerator, conf, generator_state_dict, lines, token2id, speaker2id, device, wav_dir=None):
    """lines: iterable of ``speaker|prompt|phonemes|content`` strings.  Returns [(line number, int16 numpy array)]."""
    generator = JETSGenerator(conf).to(device)                        # :70
    generator.load_state_dict(generator_state_dict)                   # :73  model_CKPT['generator']
    generator.eval()                                                  # :74
    speakers, prompts, texts, contents = [], [], [], []
    for line in lines:                                                # :96-102
        line = line.strip().split("|")
        speakers.append(line[0])
        prompts.append(line[1])
        texts.append(line[2].split())
        contents.append(line[3])
    out = []
    for i, (speaker, prompt, text, content) in enumerate(zip(speakers, prompts, texts, contents)):   # :104
        style_embedding = synthetic_style_embedding(prompt)           # :106
        content_embedding = synthetic_style_embedding(content)        # :107
        if speaker not in speaker2id:                                 # :109-110
            continue
        speaker = speaker2id[speaker]
        text_int = [token2id[ph] for ph in text]                      # :113
        sequence = torch.from_numpy(np.array(text_int)).to(device).long().unsqueeze(0)          # :115
        sequence_len = torch.from_numpy(np.array([len(text_int)])).to(device)                  # :116
        style_embedding = torch.from_numpy(style_embedding).to(device).unsqueeze(0)            # :117
        content_embedding = torch.from_numpy(content_embedding).to(device).unsqueeze(0)        # :118
        speaker = torch.from_numpy(np.array([speaker])).to(device)                             # :119
        with torch.no_grad():
            infer_output = generator(                                                          # :122-129
                inputs_ling=sequence,
                inputs_style_embedding=style_embedding,
                input_lengths=sequence_len,
                inputs_content_embedding=content_embedding,
                inputs_speaker=speaker,
                alpha=1.0)
            audio = infer_output["wav_predictions"].squeeze() * MAX_WAV_VALUE                  # :130
            audio = audio.cpu().numpy().astype('int16')                                        # :131
        if wav_dir is not None:                                                                # :132-134 (soundfile -> scipy)
            import os
            from scipy.io import wavfile
            os.makedirs(wav_dir, exist_ok=True)
            wavfile.write(os.path.join(wav_dir, "%d.wav" % (i + 1)), 16000, audio)
        out.append((i + 1, audio))
    return out
