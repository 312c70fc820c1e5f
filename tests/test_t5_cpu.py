"""umT5 text encoder (SURVEY.md section 8f row 4): the oracle against the committed reference fixtures, and the host-side pieces of
wan2gp_b200/wan/t5.py that need no GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import t5_oracle
from tests.test_host_dryrun_cpu import stub_abi  # noqa: F401  (fixture)
from wan2gp_b200 import synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _case(name="t5_small"):
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    cfg = synth.T5_CONFIGS[name]
    sd = synth.make_t5_state_dict(cfg, int(g["seed"]))
    ids, mask = synth.make_t5_inputs(cfg, int(g["length"]), int(g["n_valid"]), int(g["seed"]))
    return cfg, sd, ids, mask, torch.from_numpy(g["out"])


def test_oracle_matches_reference_fixture():
    """tests/golden/t5_small.npz was produced by the UNMODIFIED reference T5Encoder (oracle/gen_golden.py t5_small)."""
    cfg, sd, ids, mask, ref = _case()
    out = t5_oracle.t5_encode(sd, cfg, ids, mask)
    assert float((out - ref).norm() / ref.norm()) < 1e-6


def test_oracle_matches_reference_module_live():
    """The reference T5Encoder on the fixture input and, unmasked, on its first 17 ids (tests/golden/t5_cases.npz)."""
    cfg, sd, ids, mask, ref = _case()
    out = t5_oracle.t5_encode(sd, cfg, ids, mask)
    assert float((out - ref).norm() / ref.norm()) < 1e-6
    ref2 = torch.from_numpy(np.load(os.path.join(GOLDEN, "t5_cases.npz"))["t5_small_prefix17"])
    assert float((t5_oracle.t5_encode(sd, cfg, ids[:17]) - ref2).norm() / ref2.norm()) < 1e-6


def test_relative_bias_table_is_the_expanded_bias():
    from wan2gp_b200.wan.t5 import relative_bias_table
    emb = synth._normal((32, 6), 0.5, 0, "pos", "cpu")
    for L in (1, 7, 40, 200):
        tab = relative_bias_table(emb, L, 32)                       # [heads, 2L-1]
        full = t5_oracle.position_bias(emb, L, L, 32)               # [heads, L, L]
        i, j = torch.meshgrid(torch.arange(L), torch.arange(L), indexing="ij")
        assert torch.equal(tab[:, j - i + L - 1], full)


def test_hf_names_map_to_reference_names():
    from wan2gp_b200.wan.t5 import hf_to_wan_names
    cfg = synth.T5_CONFIGS["t5_small"]
    sd = synth.make_t5_state_dict(cfg, 0)
    hf = {"shared.weight": sd["token_embedding.weight"], "encoder.final_layer_norm.weight": sd["norm.weight"]}
    for i in range(cfg["num_layers"]):
        b, h = f"blocks.{i}.", f"encoder.block.{i}.layer."
        hf[h + "0.layer_norm.weight"] = sd[b + "norm1.weight"]
        hf[h + "1.layer_norm.weight"] = sd[b + "norm2.weight"]
        for n in "qkvo":
            hf[h + f"0.SelfAttention.{n}.weight"] = sd[b + f"attn.{n}.weight"]
        hf[h + "0.SelfAttention.relative_attention_bias.weight"] = sd[b + "pos_embedding.embedding.weight"]
        hf[h + "1.DenseReluDense.wi_0.weight"] = sd[b + "ffn.gate.0.weight"]
        hf[h + "1.DenseReluDense.wi_1.weight"] = sd[b + "ffn.fc1.weight"]
        hf[h + "1.DenseReluDense.wo.weight"] = sd[b + "ffn.fc2.weight"]
    back = hf_to_wan_names(hf)
    assert set(back) == set(sd) and all(back[k] is sd[k] for k in sd)
    assert hf_to_wan_names(sd) is sd


def test_clean_prompt_is_the_reference_whitespace_clean():
    from wan2gp_b200.wan.t5 import clean_prompt
    assert clean_prompt("  a &amp;amp; b \n\t c  ") == "a & b c"
    assert clean_prompt("plain prompt") == "plain prompt"


# ---------------------------------------------------------------------------------------------- byT5 (classic T5 layout, shared position bias)
def test_oracle_matches_byt5_fixture_reference_and_transformers():
    """tests/golden/byt5_tiny.npz (oracle/gen_golden.py byt5_tiny): the reference T5Encoder(shared_pos=True) AND transformers' T5Stack built
    and called the way the reference builds / calls its byT5 glyph encoder (text_encoder/byT5/__init__.py:184-188, pipeline_hunyuan_video.py
    :1037) on the same weights.  The oracle reproduces both (they agree with each other on the rows the mask keeps)."""
    g = np.load(os.path.join(GOLDEN, "byt5_tiny.npz"))
    cfg = synth.T5_CONFIGS["byt5_tiny"]
    assert cfg["shared_pos"]
    sd = synth.make_t5_state_dict(cfg, int(g["seed"]))
    assert "pos_embedding.embedding.weight" in sd and not any(k.startswith("blocks.") and "pos_embedding" in k for k in sd)
    ids, mask = synth.make_t5_inputs(cfg, int(g["length"]), int(g["n_valid"]), int(g["seed"]))
    out = t5_oracle.t5_encode(sd, cfg, ids, mask)
    nv = int(g["n_valid"])
    for key in ("out", "out_hf"):
        ref = torch.from_numpy(g[key])
        assert float((out[:nv] - ref[:nv]).norm() / ref[:nv].norm()) < 1e-6, key


def test_byt5_oracle_matches_reference_module_live():
    """The reference T5Encoder(shared_pos=True) on another seed, length and padding (tests/golden/t5_cases.npz)."""
    cfg = synth.T5_CONFIGS["byt5_tiny"]
    sd = synth.make_t5_state_dict(cfg, 3)
    ids, mask = synth.make_t5_inputs(cfg, 33, 20, 3)
    ref = torch.from_numpy(np.load(os.path.join(GOLDEN, "t5_cases.npz"))["byt5_tiny_seed3"])
    out = t5_oracle.t5_encode(sd, cfg, ids, mask)
    assert float((out - ref).norm() / ref.norm()) < 1e-6


def test_t5stack_names_map_to_the_shared_position_layout():
    """A bare transformers T5Stack state dict (no `encoder.` prefix, relative_attention_bias in block 0 only -- what
    `T5ForConditionalGeneration.get_encoder().state_dict()` holds) maps onto T5Encoder(shared_pos=True) names; ByT5Encoder.from_state_dict reads
    widths, depth and vocabulary off it."""
    from wan2gp_b200.wan.t5 import hf_to_wan_names
    cfg = synth.T5_CONFIGS["byt5_tiny"]
    sd = synth.make_t5_state_dict(cfg, 0)
    hf = synth.t5_to_hf_t5stack_names(sd, cfg["num_layers"])
    assert not any(k.startswith("encoder.") for k in hf)
    back = hf_to_wan_names(hf)
    assert set(back) == set(sd) and all(back[k] is sd[k] for k in sd)
    back2 = hf_to_wan_names({"encoder." + k: v for k, v in hf.items()})          # T5EncoderModel naming
    assert set(back2) == set(sd)
    # umT5 naming (a bias in every block) still maps to per-block embeddings
    cfg_u = synth.T5_CONFIGS["t5_small"]
    sdu = synth.make_t5_state_dict(cfg_u, 0)
    assert any("blocks.1.pos_embedding" in k for k in sdu)


def test_byt5_encoder_host_path(stub_abi, monkeypatch):  # noqa: F811
    """ByT5Encoder (Hugging Face call surface over T5Encoder(shared_pos=True)): dry run with the stubbed C ABI -- shapes, the one shared bias
    table, the `(hidden,)` return."""
    import wan2gp_b200.wan.t5 as t5mod
    from wan2gp_b200.hyvideo.byt5 import ByT5Encoder
    monkeypatch.setattr(t5mod, "_s", lambda: 0)
    cfg = synth.T5_CONFIGS["byt5_tiny"]
    sd = synth.make_t5_state_dict(cfg, 0)
    m = ByT5Encoder.from_state_dict(synth.t5_to_hf_t5stack_names(sd, cfg["num_layers"]), device="cpu")
    e = m.encoder
    assert (e.vocab_size, e.dim, e.dim_attn, e.dim_ffn, e.num_heads, e.num_layers, e.num_buckets, e.shared_pos) == (400, 192, 128, 320, 2, 3, 32, True)
    ids, mask = synth.make_t5_inputs(cfg, 24, 9, 0)
    out = m(ids[None], attention_mask=mask[None].float())
    assert isinstance(out, tuple) and tuple(out[0].shape) == (1, 24, 192)
    assert len(e._bias_cache) == 1 and stub_abi.count("b200_t5_attention") == 3


def test_byt5_oracle_matches_transformers_t5stack_live():
    """Live pin against transformers' T5Stack, built and called as the reference builds / calls its byT5 glyph encoder
    (text_encoder/byT5/__init__.py:184-188, pipeline_hunyuan_video.py:1037); skips where transformers is not installed."""
    transformers = pytest.importorskip("transformers")
    cfg = synth.T5_CONFIGS["byt5_tiny"]
    sd = synth.make_t5_state_dict(cfg, 7)
    hf_cfg = transformers.T5Config(vocab_size=cfg["vocab_size"], d_model=cfg["dim"], d_kv=64, d_ff=cfg["dim_ffn"], num_layers=cfg["num_layers"],
                                   num_decoder_layers=1, num_heads=cfg["num_heads"], relative_attention_num_buckets=cfg["num_buckets"],
                                   relative_attention_max_distance=128, dropout_rate=0.0, layer_norm_epsilon=1e-6, feed_forward_proj="gated-gelu",
                                   tie_word_embeddings=False)
    hf = transformers.T5ForConditionalGeneration(hf_cfg).get_encoder().eval().float()
    hf.load_state_dict(synth.t5_to_hf_t5stack_names(sd, cfg["num_layers"]), strict=True)
    ids, mask = synth.make_t5_inputs(cfg, 41, 23, 7)
    with torch.no_grad():
        ref = hf(ids[None], attention_mask=mask[None].float())[0][0]
    out = t5_oracle.t5_encode(sd, cfg, ids, mask)
    assert float((out[:23] - ref[:23]).norm() / ref[:23].norm()) < 1e-6
