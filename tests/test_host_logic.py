"""CPU-only checks of the host side: weight packing (the load-time re-layouts the kernels
rely on), state-dict compatibility with the reference's names, the C-ABI library's exported
symbols, and the fail-loudly behaviour without a GPU."""
import json
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

from emotivoice_b200 import synth, packing, _abi
from emotivoice_b200.config import default_config
from oracle import jets_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_of_the_header(lib):
    hdr = open(os.path.join(ROOT, "include", "emotivoice_b200.h")).read()
    declared = set(re.findall(r"EV_API\s+[\w\s\*]+?\b(ev_\w+)\s*\(", hdr))
    assert len(declared) >= 19
    assert declared == set(_abi.SIGNATURES), declared ^ set(_abi.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.ev_abi_version() == 1
    assert lib.ev_launch_count() == 0 or lib.ev_launch_count() > 0


def test_ctypes_structs_match_header_sizes():
    import ctypes
    assert ctypes.sizeof(packing.WeightEntry) == 56 + 8 + 8
    assert ctypes.sizeof(_abi.EvConfig) == 4 * (16 + 8 + 8 + 1 + 4 + 1 + 16)


def test_null_and_bad_arguments_give_error_codes_without_gpu(lib):
    assert lib.ev_create(None, 0, None) == -1
    assert b"null" in lib.ev_last_error()
    assert lib.ev_phase1_workspace_bytes(None, 1, 10) == 0


def test_forward_without_cuda_fails_loudly(conf):
    from emotivoice_b200.modules import JETSGenerator
    m = JETSGenerator(conf)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(**synth.make_batch([5]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.reserve(1, 128, 1024)          # the serving set-up call builds the engine too: same failure, no silent no-op


def test_workspace_buckets_are_monotonic_and_coarse():
    """Arena sizes are rounded up to a geometric series so that requests of similar size share a buffer."""
    from emotivoice_b200.modules import _bucket
    prev = 0
    seen = set()
    for n in range(1, 400 << 20, 3 << 20):
        b = _bucket(n)
        assert b >= n and b >= prev and b % (2 << 20) == 0
        prev = b
        seen.add(b)
    assert len(seen) < 60 and _bucket(100 << 20) / (100 << 20) <= 1.2


def test_training_mode_arguments_are_rejected(conf):
    from emotivoice_b200.modules import JETSGenerator
    m = JETSGenerator(conf)
    b = synth.make_batch([5])
    with pytest.raises(NotImplementedError):
        m(**b, mel_targets=torch.zeros(1, 10, 80))


def test_module_state_dict_is_reference_compatible(conf, sd):
    """Same 422 keys/shapes as the reference's JETSGenerator (SURVEY.md s8b), strict load,
    legacy weight_g/weight_v checkpoints accepted."""
    from emotivoice_b200.modules import JETSGenerator
    m = JETSGenerator(conf)
    own = m.state_dict()
    assert list(own.keys()) == list(sd.keys())
    assert all(own[k].shape == sd[k].shape for k in sd)
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.state_dict()["am.to_mel.weight"], sd["am.to_mel.weight"])
    legacy = synth.make_state_dict(conf, legacy_weight_norm=True)
    assert any(k.endswith("weight_g") for k in legacy)
    m.load_state_dict(legacy, strict=True)
    k = "generator.ups.1.parametrizations.weight.original1"
    assert torch.equal(m.state_dict()[k], sd[k])
    assert m.upsample_factor == 256 and m.segment_size == 32
    assert hasattr(m, "am") and hasattr(m, "generator")
    assert {n for n, _ in runner_specs(conf)} == set(sd.keys())


def runner_specs(conf):
    from emotivoice_b200 import runner
    return runner.param_specs(conf)


def test_pe_table_matches_reference_formula():
    assert torch.equal(packing.build_pe_table(700, 384), O.positional_table(700, 384))


def test_weight_norm_fold_both_key_conventions(conf, sd):
    legacy = synth.make_state_dict(conf, legacy_weight_norm=True)
    for p in ("generator.conv_pre", "generator.ups.0", "generator.resblocks.7.convs2.1", "generator.conv_post"):
        w = packing.fold_weight_norm(sd, p)
        assert torch.equal(w, packing.fold_weight_norm(legacy, p))
        assert torch.equal(w, O.fold_weight_norm(sd, p))
        v = sd[p + ".parametrizations.weight.original1"].double()
        g = sd[p + ".parametrizations.weight.original0"].double()
        ref = g * v / v.pow(2).sum((1, 2), keepdim=True).sqrt()
        assert (w.double() - ref).abs().max() <= 1e-6 * ref.abs().max()


@pytest.mark.parametrize("cin,cout,k,u", [(16, 8, 16, 8), (8, 4, 4, 2), (4, 4, 7, 3), (4, 2, 12, 4), (6, 2, 8, 4)])
def test_polyphase_packing_equals_conv_transpose(cin, cout, k, u):
    g = torch.Generator().manual_seed(k * u)
    w, b, x = torch.randn(cin, cout, k, generator=g), torch.randn(cout, generator=g), torch.randn(2, cin, 13, generator=g)
    p = (k - u) // 2
    ref = F.conv_transpose1d(x, w, b, stride=u, padding=p)
    wp, bp = packing.polyphase_pack(w, b, u, p)
    K = wp.shape[0]
    assert K % 2 == 1
    y = F.conv1d(x, wp.permute(2, 1, 0).contiguous(), bp, padding=(K - 1) // 2)      # (B, u*cout, L)
    y = y.transpose(1, 2).reshape(2, 13 * u, cout).transpose(1, 2)
    n = min(ref.shape[-1], y.shape[-1])
    assert (ref[..., :n] - y[..., :n]).abs().max() <= 1e-5


def test_packed_layouts(conf, sd):
    pk = packing.pack_state_dict(sd, conf)
    H = 384
    assert pk["enc.0.wqkv"].shape == (H, 3 * H)
    assert torch.equal(pk["enc.0.wqkv"][:, H:2 * H], sd["am.encoder.encoders.0.self_attn.linear_k.weight"].t())
    assert pk["dec.3.w1"].shape == (3, H, 4 * H) and pk["dec.3.w2"].shape == (3, 4 * H, H)
    assert torch.equal(pk["dec.3.w1"][2, 5, 7], sd["am.decoder.encoders.3.feed_forward.w_1.weight"][7, 5, 2])
    W = sd["am.embed_projection1.weight"]
    assert torch.equal(pk["cond.wx"], W[:, :H].t()) and torch.equal(pk["cond.wc"], W[:, H:].t())
    assert pk["voc.up.0.w"].shape == (3, 512, 8 * 256) and pk["voc.up.3.b"].shape == (2 * 32,)
    assert pk["voc.rb.4.c1.2.w"].shape == (7, 128, 128)
    assert pk["voc.post.w"].shape == (7, 32)
    blob, index = packing.make_blob(pk)
    assert all(e.offset % 64 == 0 for e in index) and blob.numel() >= sum(v.numel() for v in pk.values())
    e = next(e for e in index if e.name == b"to_mel.b")
    assert torch.equal(blob[e.offset:e.offset + e.numel], sd["am.to_mel.bias"])
    assert all(len(k) < 56 for k in pk)


def test_default_config_mirrors_reference_yaml_keys(conf):
    c = _abi.make_config(conf)
    assert (c.hidden, c.n_heads, c.enc_layers, c.dec_layers, c.ffn_kernel, c.bert_dim) == (384, 8, 4, 4, 3, 768)
    assert [c.up_rates[i] for i in range(4)] == [8, 8, 2, 2] and [c.res_kernels[i] for i in range(3)] == [3, 7, 11]
    assert [c.res_dils[2][i] for i in range(3)] == [1, 3, 5]
    # the values of the reference's config/joint/config.yaml (oracle/make_golden_tables.py)
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_config.json")) as f:
        y = json.load(f)
    for k, v in conf.model.items():
        assert y["model"][k] == v, k
    assert y["n_mels"] == conf.n_mels and y["segment_size"] == conf.segment_size


def test_synthetic_inputs_follow_the_input_contract():
    b = synth.make_batch([7, 3, 5], seed=1)
    assert b["inputs_ling"].shape == (3, 7) and b["inputs_ling"].dtype == torch.int64
    assert b["inputs_ling"][1, 3:].eq(0).all() and b["inputs_ling"][1, 0] == 1 and b["inputs_ling"][1, 2] == 1
    assert b["inputs_ling"].max() <= 416 and b["inputs_style_embedding"].abs().max() < 1
    s = synth.slice_batch(b, 1)
    assert s["inputs_ling"].shape == (1, 3)


def test_oracle_int16_truncates_toward_zero():
    w = torch.tensor([[0.99999, -0.99999, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768, -1.5 / 32768]])
    assert O.to_int16(w).tolist() == [32767, -32767, 0, 0, 1, -1]


# ---- tensor-core convolution: launch plan invariants (host arithmetic, no GPU needed) -----------------------
_SHAPES = [  # (Cin, Cout, K, dil): every GEMM-shaped layer of the model
    (384, 1152, 1, 1), (384, 384, 1, 1), (384, 1536, 3, 1), (1536, 384, 3, 1), (384, 80, 1, 1), (384, 384, 3, 1),
    (80, 512, 7, 1), (512, 2048, 3, 1), (256, 1024, 3, 1), (128, 128, 3, 1), (64, 64, 3, 1),
] + [(c, c, k, d) for c in (256, 128, 64, 32) for k in (3, 7, 11) for d in (1, 3, 5)]


def _plan(lib, B, L, Cin, Cout, K, dil, split3, ksplit=0):
    import ctypes
    out = (ctypes.c_int * 11)()
    _abi.check(lib.ev_debug_tc_plan(B, L, Cin, Cout, K, dil, split3, ksplit, out))
    keys = ("BN", "MT", "KBG", "a_stages", "b_stages", "ngroups", "ksplit", "tmem_cols", "smem", "tiles", "rows_pad")
    return dict(zip(keys, list(out)))


@pytest.mark.parametrize("split3", [0, 1, 2])
def test_tc_plan_respects_hardware_limits_and_barrier_protocol(lib, split3):
    for Cin, Cout, K, dil in _SHAPES:
        if split3 == 2 and Cin % 16:
            continue
        for B, L in ((1, 100), (1, 537), (1, 4296), (1, 137472), (3, 300), (32, 1600), (128, 65536)):
            p = _plan(lib, B, L, Cin, Cout, K, dil, split3, ksplit=2)
            assert p["smem"] <= 227 * 1024 and p["tmem_cols"] <= 512 and 2 * p["MT"] * p["BN"] <= p["tmem_cols"]
            assert p["BN"] % 16 == 0 and p["BN"] <= 128 and p["MT"] in (1, 2, 4) and p["KBG"] in (4, 8)
            assert 2 <= p["a_stages"] <= 8 and 2 <= p["b_stages"] <= 8
            # a producer group may never run two uses of a ring slot ahead of the consumer: the parity wait on
            # a_empty cannot tell them apart (this was a real deadlock) -> groups <= ring depth
            assert p["ngroups"] in (1, 2, 3, 6) and p["ngroups"] <= p["a_stages"]
            assert p["rows_pad"] % 8 == 8 // p["KBG"]            # conflict-free 16-byte producer stores
            assert p["rows_pad"] >= 128 * p["MT"] + (K - 1) * dil


@pytest.mark.parametrize("split3", [0, 1, 2])
def test_tc_plan_summation_order_is_a_function_of_the_layer_only(lib, split3):
    """KBG (how the (channel block, tap) reduction is ordered) and the K-split factor must not depend on batch or
    length: that is what makes a batched run bitwise equal to the B=1 runs."""
    for Cin, Cout, K, dil in _SHAPES:
        if split3 == 2 and Cin % 16:
            continue
        seen = {(_plan(lib, B, L, Cin, Cout, K, dil, split3, ksplit=4)["KBG"], _plan(lib, B, L, Cin, Cout, K, dil, split3, ksplit=4)["ksplit"])
                for B, L in ((1, 64), (1, 537), (1, 34368), (2, 900), (32, 1600), (64, 40000))}
        assert len(seen) == 1, (Cin, Cout, K, dil, seen)


def test_tc_plan_rejects_unsupported_shapes(lib):
    import ctypes
    out = (ctypes.c_int * 11)()
    assert lib.ev_debug_tc_plan(1, 100, 30, 32, 3, 1, 0, 0, out) == -1       # Cin % 8
    assert lib.ev_debug_tc_plan(1, 100, 32, 200, 3, 1, 0, 0, out) == -1      # Cout > 128 and not a multiple of 128
    assert lib.ev_debug_tc_plan(1, 100, 32, 32, 4, 1, 0, 0, out) == -1       # even kernel size


def test_3xtf32_split_is_fp32_accurate_in_emulation():
    """The arithmetic behind the default "fp32" mode, emulated on the CPU: x = hi + lo with hi = tf32(x),
    lo = tf32(x - hi); a.b ~= sum(a_lo*b_hi + a_hi*b_lo + a_hi*b_hi) accumulated in fp32.  Its error against an
    fp64 dot product must be at the fp32 level (the dropped lo*lo term is 2^-22 relative), far below one tf32
    product (2^-11)."""
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(256, 1152, generator=g), torch.randn(1152, 64, generator=g)

    def split(x):
        hi = packing.round_tf32(x)
        return hi, packing.round_tf32(x - hi)

    a_hi, a_lo = split(a)
    b_hi, b_lo = split(b)
    exact = a.double() @ b.double()
    one = (a_hi.double() @ b_hi.double())
    three = (a_lo.double() @ b_hi.double() + a_hi.double() @ b_lo.double() + a_hi.double() @ b_hi.double()).float().double()
    fp32 = (a @ b).double()
    scale = exact.abs().max()
    e1, e3, ef = ((one - exact).abs().max() / scale).item(), ((three - exact).abs().max() / scale).item(), ((fp32 - exact).abs().max() / scale).item()
    assert e1 > 1e-5           # one tf32 product is visibly worse than fp32
    assert e3 < 3e-7           # the split is at the fp32 level ...
    assert e3 < 5 * max(ef, 1e-8) + 1e-7    # ... comparable to a plain fp32 matmul
    # hi + lo reconstructs x to ~2^-22
    assert ((a_hi + a_lo) - a).abs().max() <= a.abs().max() * 2.0 ** -21
