"""GPU, SURVEY.md §8c G6: the task heads over the drop-in `uniter_b200.UniterModel`, forward and
backward on the device, against what the reference's own heads computed over the reference encoder
on CPU (tests/golden/heads_tiny.npz, reference_heads.npz, made by tests/golden/make_goldens.py).

  * test_unmodified_reference_*: the reference's OWN, UNMODIFIED heads (model/vqa.py,
    model/pretrain.py, model/itm.py staged in oracle/_ref by oracle/make_ref.py) built over our
    encoder — the INTEGRATION.md recipe (`model.<head>.UniterModel = ours`); they need the staged
    reference sources.
  * test_library_*: the library's own heads (uniter_b200.heads), self-contained.

North-star tolerance 1e-2 on logits in fp16; gradients against the CPU oracle or the stored
reference gradients.
"""
import pytest
import torch

from oracle import encoder_oracle as orc
from oracle import ref_loader
from tests import util
from tests.golden import make_goldens

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="reference sources not staged")


class _swap:
    """with _swap(rvqa, rpre): the reference modules construct OUR UniterModel."""

    def __init__(self, *mods):
        self.mods = mods

    def __enter__(self):
        from uniter_b200.model import UniterModel
        self.saved = [m.UniterModel for m in self.mods]
        for m in self.mods:
            m.UniterModel = UniterModel

    def __exit__(self, *a):
        for m, s in zip(self.mods, self.saved):
            m.UniterModel = s


def _tiny_ref_config(rm):
    c = util.TINY
    return rm.UniterConfig(c["vocab_size"], hidden_size=c["hidden_size"],
                           num_hidden_layers=c["num_hidden_layers"],
                           num_attention_heads=c["num_attention_heads"],
                           intermediate_size=c["intermediate_size"],
                           max_position_embeddings=c["max_position_embeddings"],
                           type_vocab_size=c["type_vocab_size"])


def _set_dropout_zero(model):
    """utils/misc.set_dropout (utils/misc.py:57-63) with p = 0: train mode made deterministic."""
    for _, module in model.named_modules():
        if isinstance(module, torch.nn.Dropout):
            module.p = 0.0


def _tensors(batch):
    return {k: v.cuda() for k, v in batch.items() if torch.is_tensor(v)}


def _seeded(mod, seed):
    """Per-key seeded weights over the module's own schema — the values the reference module held
    for the same keys when the goldens were made."""
    from uniter_b200.synth import seeded_state
    return seeded_state({k: tuple(v.shape) for k, v in mod.state_dict().items()}, seed=seed)


@needs_reference
def test_unmodified_reference_vqa_head_over_drop_in_encoder():
    from uniter_b200.model import UniterModel
    from uniter_b200.synth import seeded_state
    rm, rvqa = ref_loader.load("model.model", "model.vqa")
    g = util.load_golden("heads_tiny")
    with _swap(rvqa):
        vqa = rvqa.UniterForVisualQuestionAnswering(_tiny_ref_config(rm), 64, 17)
    assert isinstance(vqa.uniter, UniterModel)
    st = seeded_state({k: tuple(v.shape) for k, v in vqa.state_dict().items()}, seed=3)
    vqa.load_state_dict(st, strict=True)
    vqa = vqa.cuda().half().eval()
    batch = util.heads_batch()
    b = _tensors(batch)
    b["targets"] = torch.rand(3, 17, generator=torch.Generator().manual_seed(5)).cuda().half()
    logits = vqa(b, compute_loss=False)
    err = (logits.float().cpu() - torch.from_numpy(g["vqa_logits"])).abs().max().item()
    assert err <= 1e-2, err
    # backward of the reference's own loss (model/vqa.py:46-49) through the CUDA encoder
    loss = vqa(b, compute_loss=True)
    (loss.float().mean() * 256.0).backward()
    rs = {k: v.half().float().requires_grad_(True) for k, v in st.items()}
    enc = {k[len("uniter."):]: v for k, v in rs.items() if k.startswith("uniter.")}
    seq = orc.uniter_forward(enc, 2, 2, batch["input_ids"], batch["position_ids"],
                             batch["img_feat"].half().float(), batch["img_pos_feat"].half().float(),
                             batch["attn_masks"], batch["gather_index"], output_all_encoded_layers=False)
    ref_logits = orc.vqa_head(rs, orc.pooler(enc, seq))
    torch.nn.functional.binary_cross_entropy_with_logits(
        ref_logits, b["targets"].float().cpu(), reduction="none").mean().backward()
    params = dict(vqa.named_parameters())
    for name in ("uniter.encoder.layer.1.intermediate.dense.weight",
                 "uniter.encoder.layer.0.attention.self.value.weight", "uniter.pooler.dense.weight",
                 "uniter.img_embeddings.img_linear.weight", "vqa_output.0.weight"):
        got = params[name].grad.float().cpu() / 256.0
        want = rs[name].grad
        rel = ((got - want).norm() / (want.norm() + 1e-12)).item()
        assert rel <= 4e-2, (name, rel)


def test_library_vqa_head_matches_reference_logits_and_oracle_gradients():
    """OUR UniterForVisualQuestionAnswering (library pooler, torch classifier): logits against the
    reference heads' golden, gradients of the reference's loss against the CPU oracle."""
    from uniter_b200.heads import UniterForVisualQuestionAnswering
    from uniter_b200.model import UniterModel
    g = util.load_golden("heads_tiny")
    vqa = UniterForVisualQuestionAnswering(util.tiny_config(), 64, 17)
    assert isinstance(vqa.uniter, UniterModel)
    st = _seeded(vqa, seed=3)
    vqa.load_state_dict(st, strict=True)
    vqa = vqa.cuda().half().eval()
    batch = util.heads_batch()
    b = _tensors(batch)
    b["targets"] = torch.rand(3, 17, generator=torch.Generator().manual_seed(5)).cuda().half()
    logits = vqa(b, compute_loss=False)
    err = (logits.float().cpu() - torch.from_numpy(g["vqa_logits"])).abs().max().item()
    assert err <= 1e-2, err
    # backward of the reference's loss (model/vqa.py:46-49) through the CUDA encoder
    loss = vqa(b, compute_loss=True)
    (loss.float().mean() * 256.0).backward()
    rs = {k: v.half().float().requires_grad_(True) for k, v in st.items()}
    enc = {k[len("uniter."):]: v for k, v in rs.items() if k.startswith("uniter.")}
    seq = orc.uniter_forward(enc, 2, 2, batch["input_ids"], batch["position_ids"],
                             batch["img_feat"].half().float(), batch["img_pos_feat"].half().float(),
                             batch["attn_masks"], batch["gather_index"], output_all_encoded_layers=False)
    ref_logits = orc.vqa_head(rs, orc.pooler(enc, seq))
    torch.nn.functional.binary_cross_entropy_with_logits(
        ref_logits, b["targets"].float().cpu(), reduction="none").mean().backward()
    params = dict(vqa.named_parameters())
    for name in ("uniter.encoder.layer.1.intermediate.dense.weight",
                 "uniter.encoder.layer.0.attention.self.value.weight", "uniter.pooler.dense.weight",
                 "uniter.img_embeddings.img_linear.weight", "vqa_output.0.weight"):
        got = params[name].grad.float().cpu() / 256.0
        want = rs[name].grad
        rel = ((got - want).norm() / (want.norm() + 1e-12)).item()
        assert rel <= 4e-2, (name, rel)


@needs_reference
def test_unmodified_reference_pretraining_heads_over_drop_in_encoder():
    """UniterForPretraining.forward(batch, task) for mlm / itm / mrfr / mrc: the reference's own
    forward_* code (model/pretrain.py:107-229) over the CUDA encoder; MLM / ITM logits against the
    reference goldens, MRFR / MRC against the same reference heads over the
    reference encoder on CPU (reference_heads.npz)."""
    from uniter_b200.synth import seeded_state
    rm, rpre = ref_loader.load("model.model", "model.pretrain")
    g = util.load_golden("heads_tiny")
    cfg = _tiny_ref_config(rm)
    with _swap(rpre):
        pre = rpre.UniterForPretraining(cfg, 64, 11)
    assert pre.cls.predictions.decoder.weight is pre.uniter.embeddings.word_embeddings.weight
    assert pre.feat_regress.weight is pre.uniter.img_embeddings.img_linear.weight
    st = seeded_state({k: tuple(v.shape) for k, v in pre.state_dict().items()}, seed=4)
    pre.load_state_dict(st, strict=True)
    ref = util.load_golden("reference_heads")       # the reference heads over their own encoder
    pre = pre.cuda().half().eval()
    batch = util.heads_batch()
    b = _tensors(batch)
    with torch.no_grad():
        scores = pre(b, task="mlm", compute_loss=False)
    err = (scores.float().cpu() - torch.from_numpy(g["mlm_scores"])).abs().max().item()
    assert err <= 1e-2, ("mlm", err)
    bi = dict(b)
    bi["targets"] = torch.tensor([1, 0, 1]).cuda()
    bi["ot_inputs"] = None
    with torch.no_grad():
        itm, _ = pre(bi, task="itm", compute_loss=False)
    err = (itm.float().cpu() - torch.from_numpy(g["itm_scores"])).abs().max().item()
    assert err <= 1e-2, ("itm", err)
    # MRFR / MRC: masked regions (model/pretrain.py:135-154, :201-229)
    extra = make_goldens.pretrain_mrm_extra(batch)
    dev_extra = {k: (v.cuda().half() if v.is_floating_point() else v.cuda()) for k, v in extra.items()}
    for task in ("mrfr", "mrc"):
        want = torch.from_numpy(ref["pre/" + task])
        with torch.no_grad():
            got = pre(dict(b, **dev_extra), task=task, compute_loss=False)
        err = (got.float().cpu() - want).abs().max().item()
        assert got.shape == want.shape and err <= 1e-2, (task, err)


@needs_reference
def test_unmodified_reference_hard_negative_itm_over_drop_in_encoder():
    """model/itm.py:57-147 (UniterForImageTextRetrievalHardNeg): no-grad eval scoring of all pairs,
    top-k hard negatives, train-mode forward + backward on the selected rows — the reference's own
    class driving the CUDA encoder through model.train()/eval() toggles inside one step, against the
    rows the same class mined and the loss it computed over the reference encoder on CPU."""
    from uniter_b200.synth import seeded_state
    rm, ritm = ref_loader.load("model.model", "model.itm")
    golden = util.load_golden("reference_heads")
    cfg = _tiny_ref_config(rm)
    with _swap(ritm):
        mod = ritm.UniterForImageTextRetrievalHardNeg(cfg, 16, hard_size=3)
    st = seeded_state({k: tuple(v.shape) for k, v in mod.state_dict().items()}, seed=6)
    mod.load_state_dict(st, strict=True)
    mod = mod.cuda().half().train()
    _set_dropout_zero(mod)
    compared = 0
    for sf in ("t", "i"):
        batch, _ = make_goldens.hardneg_inputs(sf, seed=77)
        b = {k: v.cuda() for k, v in batch.items()}
        picked = {}
        orig = mod._get_hard_batch
        mod._get_hard_batch = lambda bt, sc, sfrom, _o=orig: picked.setdefault("gpu", _o(bt, sc, sfrom))
        mod.zero_grad(set_to_none=True)
        loss = mod(b, sample_from=sf, compute_loss=True)
        mod._get_hard_batch = orig
        assert loss.shape[0] == 1 and torch.isfinite(loss.float()).all()
        loss.float().mean().backward()
        gw = mod.uniter.encoder.layer[0].intermediate.dense.weight.grad
        assert gw is not None and torch.isfinite(gw.float()).all()
        # the same step through the reference class over the reference encoder (CPU fp32)
        key = "img_feat" if sf == "t" else "input_ids"
        g_rows = picked["gpu"][key].float().cpu()
        c_rows = torch.from_numpy(golden["hardneg/%s/%s" % (sf, key)])
        rloss = torch.from_numpy(golden["hardneg/%s/loss" % sf])
        if g_rows.shape == c_rows.shape and torch.equal(g_rows.half(), c_rows.half()):
            # same hard negatives mined (top-k over 16-bit scores can legitimately differ on near ties)
            assert (loss.float().cpu() - rloss).abs().max().item() <= 1e-2, sf
            compared += 1
    assert compared >= 1


def test_library_hard_negative_itm_matches_reference_rows_and_loss():
    """OUR UniterForImageTextRetrievalHardNeg (model/itm.py:57-147): no-grad eval scoring of all pairs,
    top-k hard negatives, train-mode forward + backward on the selected rows — the CUDA encoder
    through model.train()/eval() toggles inside one step — against the rows the reference class
    mined and the loss it computed on CPU."""
    from uniter_b200.heads import UniterForImageTextRetrievalHardNeg
    ref = util.load_golden("reference_heads")
    mod = UniterForImageTextRetrievalHardNeg(util.tiny_config(), 16, hard_size=3)
    mod.load_state_dict(_seeded(mod, seed=6), strict=True)
    mod = mod.cuda().half().train()
    _set_dropout_zero(mod)
    compared = 0
    for sf in ("t", "i"):
        batch, _ = make_goldens.hardneg_inputs(sf, seed=77)
        b = {k: v.cuda() for k, v in batch.items()}
        picked = {}
        orig = mod._get_hard_batch
        mod._get_hard_batch = lambda bt, sc, sfrom, _o=orig: picked.setdefault("gpu", _o(bt, sc, sfrom))
        mod.zero_grad(set_to_none=True)
        loss = mod(b, sample_from=sf, compute_loss=True)
        mod._get_hard_batch = orig
        assert loss.shape[0] == 1 and torch.isfinite(loss.float()).all()
        loss.float().mean().backward()
        gw = mod.uniter.encoder.layer[0].intermediate.dense.weight.grad
        assert gw is not None and torch.isfinite(gw.float()).all()
        key = "img_feat" if sf == "t" else "input_ids"
        g_rows = picked["gpu"][key].float().cpu()
        c_rows = torch.from_numpy(ref["hardneg/%s/%s" % (sf, key)])
        rloss = torch.from_numpy(ref["hardneg/%s/loss" % sf])
        if g_rows.shape == c_rows.shape and torch.equal(g_rows.half(), c_rows.half()):
            # same hard negatives mined (top-k over 16-bit scores can legitimately differ on near ties)
            assert loss.shape == rloss.shape
            assert (loss.float().cpu() - rloss).abs().max().item() <= 1e-2, sf
            compared += 1
    assert compared >= 1


@pytest.mark.parametrize("use_index", [True, False])
def test_library_pretraining_heads_match_the_reference_model(use_index):
    """OUR UniterForPretraining (every head on libub200: LibTransform / LibLinear / fused MLM head /
    library pooler) against the reference UniterForPretraining over the reference encoder on CPU fp32
    (weights rounded to fp16): logits of mlm / mrfr / mrc / itm within 1e-2 (north star),
    per-element losses, and gradients of a multi-task loss for the head parameters and both tied
    weights (decoder <-> word embeddings, feat_regress.weight <-> img_linear.weight)."""
    from uniter_b200.heads import UniterForPretraining
    ref = util.load_golden("reference_heads")
    mod = UniterForPretraining(util.tiny_config(), 64, 11)
    mod.load_state_dict(_seeded(mod, seed=4), strict=True)
    mod = mod.cuda().half().eval()
    base, mb, keys = make_goldens.library_pretrain_inputs(use_index)
    db = {k: mb[k].cuda() for k in keys}
    db["targets"] = torch.tensor([1, 0, 1, 1, 0]).cuda()
    plain_d = dict(db, img_feat=base["img_feat"].cuda())      # mlm / itm see unmasked regions
    total_d = 0.0
    for task in make_goldens.LIBRARY_PRETRAIN_TASKS:
        bd = plain_d if task in ("mlm", "itm") else db
        with torch.no_grad():
            got = mod(bd, task=task, compute_loss=False)
        want = torch.from_numpy(ref["library/%s/logits" % task])
        got = got[0] if isinstance(got, tuple) else got
        assert got.shape == want.shape, (task, got.shape, want.shape)
        err = (got.float().cpu() - want).abs().max().item()
        assert err <= 1e-2, (task, err)
        lw = torch.from_numpy(ref["library/%s/loss" % task])
        lg = mod(bd, task=task, compute_loss=True)
        lg = lg[0] if isinstance(lg, tuple) else lg
        assert lg.shape == lw.shape, (task, lg.shape, lw.shape)
        assert (lg.float().cpu() - lw).abs().max().item() <= 3e-2, task
        total_d = total_d + lg.float().mean()
    (total_d * 64.0).backward()
    gp = dict(mod.named_parameters())
    for name in make_goldens.LIBRARY_PRETRAIN_GRADS:
        rows = torch.from_numpy(ref["library/grad_rows/" + name])
        got = gp[name].grad.float().cpu()[rows] / 64.0
        want = torch.from_numpy(ref["library/grad/" + name])
        rel = ((got - want).norm() / (want.norm() + 1e-12)).item()
        assert rel <= 4e-2, (name, rel)
