"""CPU (no GPU needed): the drop-in boundary.

  * libub200.so loads without a CUDA driver and exports every symbol include/ub200.h declares;
  * ctypes struct mirrors have the size the C compiler gives the header's structs;
  * UniterConfig / UniterModel keep the reference's constructor, parameter schema, from_pretrained
    renames and error conventions (SURVEY.md §8b-B1);
  * the reference's own task heads accept our UniterModel where the reference sources are staged,
    and the library's heads keep their state-dict schema and weight tying
    (tests/golden/reference_schema.json; construction + state-dict level, compute needs the GPU);
  * the product never silently falls back: forward on CPU / fp32 raises.
"""
import ctypes as C
import json
import os
import re
import subprocess
import tempfile

import pytest
import torch

from oracle import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ub200.h")
SCHEMA = os.path.join(ROOT, "tests", "golden", "reference_schema.json")


@pytest.fixture(scope="module")
def lib():
    from uniter_b200 import build, _lib
    build.build()
    return _lib.load()


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ub200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    names = _declared_functions()
    assert len(names) >= 20, names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, "declared in include/ub200.h but not exported: %s" % missing
    assert lib.ub200_version() >= 100


def test_library_has_no_libcuda_link_dependency():
    from uniter_b200 import _lib
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out          # loads on a CPU-only box; driver entry points are fetched lazily
    assert "libtorch" not in out            # plain C ABI, no torch types


def test_errors_are_reported_not_thrown(lib):
    # no device here: device_check must return a negative code and set the message
    rc = lib.ub200_device_check()
    if not torch.cuda.is_available():
        assert rc < 0
        assert len(lib.ub200_last_error_string()) > 0
    # NULL args -> UB200_EINVAL (-1), never a crash
    assert lib.ub200_gemm(None, None) == -1
    assert b"NULL" in lib.ub200_last_error_string()


def test_ctypes_mirrors_match_the_header_layout():
    """Compile a tiny C program against include/ub200.h and compare sizeof() with ctypes."""
    from uniter_b200 import _lib
    from uniter_b200.model import _EncoderDesc, _LayerGrads, _LayerWeights
    prog = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "ub200.h"
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(ub200_gemm_args), sizeof(ub200_attn_args),
             sizeof(ub200_ln_bwd_args), sizeof(ub200_layer_weights), sizeof(ub200_layer_grads),
             sizeof(ub200_encoder_desc), sizeof(ub200_adam_segment), sizeof(ub200_embed_colsum_args),
             offsetof(ub200_gemm_args, k_splits), offsetof(ub200_gemm_args, n_valid),
             offsetof(ub200_adam_segment, step_size), offsetof(ub200_embed_colsum_args, T),
             sizeof(ub200_peer_allreduce_args), offsetof(ub200_peer_allreduce_args, stage_bytes));
      return 0;
    }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    mine = [C.sizeof(_lib.GemmArgs), C.sizeof(_lib.AttnArgs), C.sizeof(_lib.LnBwdArgs),
            C.sizeof(_LayerWeights), C.sizeof(_LayerGrads), C.sizeof(_EncoderDesc),
            C.sizeof(_lib.AdamSegment), C.sizeof(_lib.EmbedColsumArgs),
            _lib.GemmArgs.k_splits.offset, _lib.GemmArgs.n_valid.offset,
            _lib.AdamSegment.step_size.offset, _lib.EmbedColsumArgs.T.offset,
            C.sizeof(_lib.PeerAllreduceArgs), _lib.PeerAllreduceArgs.stage_bytes.offset]
    assert sizes == mine, (sizes, mine)


def _tiny_cfg():
    from uniter_b200.model import UniterConfig
    return UniterConfig(2000, hidden_size=128, num_hidden_layers=2, num_attention_heads=2,
                        intermediate_size=512, max_position_embeddings=64)


def test_config_matches_reference_semantics(tmp_path):
    from uniter_b200.model import UniterConfig
    with pytest.raises(ValueError):
        UniterConfig(3.5)
    p = tmp_path / "c.json"
    p.write_text(json.dumps({"hidden_size": 768, "num_attention_heads": 12, "vocab_size": 28996,
                             "extra_key": 7}))
    c = UniterConfig.from_json_file(str(p))
    assert c.hidden_size == 768 and c.extra_key == 7        # every JSON key is copied (model/model.py:89-102)
    assert json.loads(c.to_json_string())["vocab_size"] == 28996
    with open(SCHEMA) as fh:
        configs = json.load(fh)["configs"]          # the reference's config/uniter-{base,large}.json
    assert sorted(configs) == ["uniter-base.json", "uniter-large.json"]
    for name, body in configs.items():
        path = tmp_path / name
        path.write_text(json.dumps(body))
        c = UniterConfig.from_json_file(str(path))
        assert c.hidden_size == 64 * c.num_attention_heads


def test_state_dict_schema_and_weight_decay_names():
    from uniter_b200.model import UniterModel
    from uniter_b200.synth import uniter_state_shapes
    m = UniterModel(_tiny_cfg(), 64)
    sd = m.state_dict()
    want = uniter_state_shapes(128, 2, 512, 2000, 64, 2, 64)
    assert set(sd) == set(want)
    assert all(tuple(sd[k].shape) == tuple(want[k]) for k in want)
    # q / k / v stay three separate parameters; pooler callable; dropout modules are real nn.Dropout
    names = dict(m.named_parameters())
    assert "encoder.layer.1.attention.self.key.weight" in names
    drops = [n for n, mod in m.named_modules() if isinstance(mod, torch.nn.Dropout)]
    assert len(drops) == 2 + 3 * 2
    # name-based no-decay grouping of optim/misc.py:14-22 still applies
    no_decay = ["bias", "LayerNorm.bias", "LayerNorm.weight"]
    nd = [n for n in names if any(x in n for x in no_decay)]
    assert "encoder.layer.0.output.LayerNorm.weight" in nd
    assert "img_embeddings.img_layer_norm.weight" not in nd   # the reference decays these; keep it


def test_from_pretrained_renames_and_errors(tmp_path):
    from uniter_b200.model import UniterModel
    cfgp = tmp_path / "cfg.json"
    cfgp.write_text(json.dumps({k: getattr(_tiny_cfg(), k) for k in
                                ("vocab_size", "hidden_size", "num_hidden_layers", "num_attention_heads",
                                 "intermediate_size", "hidden_act", "hidden_dropout_prob",
                                 "attention_probs_dropout_prob", "max_position_embeddings",
                                 "type_vocab_size", "initializer_range")}))
    src = UniterModel(_tiny_cfg(), 64)
    sd = {}
    for k, v in src.state_dict().items():      # TF-style names + "bert." prefix (model/model.py:166-199)
        k = k.replace("LayerNorm.weight", "LayerNorm.gamma").replace("LayerNorm.bias", "LayerNorm.beta")
        sd["bert." + k] = v.clone()
    m = UniterModel.from_pretrained(str(cfgp), sd, img_dim=64)
    for (k, a), (_, b) in zip(sorted(m.state_dict().items()), sorted(src.state_dict().items())):
        assert torch.equal(a, b), k
    bad = dict(src.state_dict())
    bad["pooler.dense.weight"] = torch.zeros(3, 3)
    with pytest.raises(RuntimeError):
        UniterModel.from_pretrained(str(cfgp), bad, img_dim=64)
    with pytest.raises(ValueError):
        UniterModel(object(), 64)


def test_forward_refuses_cpu_and_fp32():
    from uniter_b200.model import UniterModel
    from uniter_b200.synth import synth_batch
    m = UniterModel(_tiny_cfg(), 64)
    b = synth_batch(2, 3, 5, 2, 4, seed=1, img_dim=64, vocab_size=2000)
    with pytest.raises(RuntimeError, match="fp16/bf16"):
        m(b["input_ids"], b["position_ids"], b["img_feat"], b["img_pos_feat"], b["attn_masks"],
          b["gather_index"])


def test_qkv_packing_survives_dtype_casts():
    """query/key/value are re-homed as views of one [3H, H] buffer; .half()/.float() re-allocate
    them and the next _weight_table() call must re-pack (checked at the storage level on CPU by
    faking the dtype gate)."""
    from uniter_b200.model import UniterModel
    m = UniterModel(_tiny_cfg(), 64).half()
    att = m.encoder.layer[0].attention.self
    q0 = att.query.weight.detach().clone()
    # emulate what _weight_table does without touching CUDA
    H = 128
    buf = torch.cat([att.query.weight.data, att.key.weight.data, att.value.weight.data], 0)
    att.query.weight.data, att.key.weight.data, att.value.weight.data = buf[:H], buf[H:2 * H], buf[2 * H:]
    assert att.key.weight.data_ptr() == att.query.weight.data_ptr() + H * H * 2
    assert torch.equal(att.query.weight, q0)
    sd = m.state_dict()
    assert sd["encoder.layer.0.attention.self.key.weight"].shape == (H, H)
    m.load_state_dict(sd)          # in-place copies keep the packing
    assert att.key.weight.data_ptr() == att.query.weight.data_ptr() + H * H * 2


@pytest.mark.skipif(not ref_loader.available(), reason="reference sources not staged")
def test_reference_heads_accept_the_drop_in_model():
    """Monkey-patch model.model.UniterModel (the INTEGRATION.md recipe) and build the reference's
    own heads on top of it: constructor, init_weights, weight tying, and the state-dict keys and
    shapes the same heads have over the reference encoder (reference_schema.json)."""
    from tests.golden import make_goldens
    from uniter_b200.model import UniterModel
    rm, rvqa, rpre = ref_loader.load("model.model", "model.vqa", "model.pretrain")
    with open(SCHEMA) as fh:
        want = json.load(fh)
    orig = rm.UniterModel
    try:
        for mod in (rvqa, rpre):
            mod.UniterModel = UniterModel
        cfg = rm.UniterConfig(**make_goldens.TINY)
        vqa = rvqa.UniterForVisualQuestionAnswering(cfg, 64, 17)
        assert isinstance(vqa.uniter, UniterModel)
        pre = rpre.UniterForPretraining(cfg, 64, 11)
        assert isinstance(pre.uniter, UniterModel)
        assert pre.cls.predictions.decoder.weight is pre.uniter.embeddings.word_embeddings.weight
        assert pre.feat_regress.weight is pre.uniter.img_embeddings.img_linear.weight
        for tag, mod in (("vqa", vqa), ("pretraining", pre)):
            assert {k: list(v.shape) for k, v in mod.state_dict().items()} == want[tag], tag
    finally:
        rvqa.UniterModel = orig
        rpre.UniterModel = orig


def test_library_heads_keep_the_reference_schema():
    """The library's own heads (uniter_b200.heads) over our UniterModel: constructor, init_weights,
    weight tying, and the state-dict keys and shapes of the reference's heads over the reference
    encoder (reference_schema.json)."""
    from uniter_b200.heads import UniterForPretraining, UniterForVisualQuestionAnswering
    from uniter_b200.model import UniterModel
    with open(SCHEMA) as fh:
        want = json.load(fh)
    cfg = _tiny_cfg()
    vqa = UniterForVisualQuestionAnswering(cfg, 64, 17)
    assert isinstance(vqa.uniter, UniterModel)
    pre = UniterForPretraining(cfg, 64, 11)
    assert pre.cls.predictions.decoder.weight is pre.uniter.embeddings.word_embeddings.weight
    assert pre.feat_regress.weight is pre.uniter.img_embeddings.img_linear.weight
    for tag, mod in (("vqa", vqa), ("pretraining", pre)):
        got = {k: list(v.shape) for k, v in mod.state_dict().items()}
        assert got == want[tag], tag
    enc = {k[len("uniter."):]: v for k, v in want["pretraining"].items() if k.startswith("uniter.")}
    assert {k: list(v.shape) for k, v in UniterModel(cfg, 64).state_dict().items()} == enc


def test_prefix_pack_bookkeeping_matches_mask_derived_indices():
    """Host-side packing metadata (no device reads) == what the mask itself implies; with a token
    bucket (`T_pad`) the padding is one dummy sequence that no output position references."""
    from uniter_b200.model import _prefix_pack_host
    for lens, L, T_pad in (([56, 44], 56, None), ([1], 1, None), ([3, 7, 2, 7], 9, None),
                           ([5] * 64, 72, 384), ([0, 4, 0], 4, 8), ([3, 7, 2, 7], 9, 19)):
        B, T = len(lens), sum(lens)
        mask = torch.zeros(B, L, dtype=torch.long)
        for b, s in enumerate(lens):
            mask[b, :s] = 1
        host, o, T_out = _prefix_pack_host(lens, L, T_pad)
        Tp = T if T_pad is None else T_pad
        assert T_out == T
        assert host.dtype == torch.int32 and o["pack"] % 4 == 0 and o["inv"] % 4 == 0 and o["unpack"] % 4 == 0
        cu = host[o["cu"]:o["cu"] + B + 2]
        pack = host[o["pack"]:o["pack"] + Tp]
        inv = host[o["inv"]:o["inv"] + Tp]
        unpack = host[o["unpack"]:o["unpack"] + B * L + 1]
        assert cu.tolist() == [0] + torch.tensor(lens).cumsum(0).tolist() + [Tp]
        want_pack = mask.reshape(-1).nonzero().squeeze(1).to(torch.int32)
        assert torch.equal(pack[:T], want_pack) and torch.equal(inv[:T], want_pack)
        # dummy rows: computed from a valid position, invisible to the inverse map
        assert (inv[T:] == -1).all() and (pack[T:] == (want_pack[0] if T else 0)).all()
        want_unpack = torch.full((B * L + 1,), -1, dtype=torch.int32)
        want_unpack[want_pack.long()] = torch.arange(T, dtype=torch.int32)
        assert torch.equal(unpack, want_unpack) and unpack[-1] == -1
