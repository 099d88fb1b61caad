"""Generate golden vectors by running the UNMODIFIED reference modules on CPU (fp32).

    python tests/golden/make_goldens.py            # needs /root/reference (this container only)

The reference imports fine once `apex.normalization.fused_layer_norm.FusedLayerNorm` is shimmed
to torch.nn.LayerNorm (the only apex symbol model/*.py uses; same parameter names, same eps
argument, biased variance, fp32 statistics).  Weights are NOT stored: they are regenerated on
the test side from `uniter_b200.synth.seeded_state` (per-key seeded), and each golden file
records a checksum of the weights it was produced with.  Outputs are stored as fp32 .npz.

Cases (SURVEY.md §8c):
  tiny_*   H=128, 2 heads, 2 layers, I=512 — every tap, every output, full gradients
  c1a / c1b  BASELINE config[0]: UNITER-base 1 layer, B=2, 20 txt + 36 regions (and a ragged
             variant (20,36),(14,30)) — outputs, taps, gradient fingerprints
  *_adv    adversarial gather_index (permutation inside the valid range and the malformed index
           of data/itm.py:356-361) — embedding output, bit-exact row selection
  heads    VQA logits / MLM scores / ITM scores through the reference heads on top of the
           reference encoder
  reference_heads  MRFR / MRC outputs, the rows and loss of a hard-negative ITM step, and the
           logits, losses and gradients (see grad_rows) of a multi-task pre-training step, all through
           the reference heads (tests/test_reference_heads_gpu.py)
  reference_schema.json  state-dict keys and shapes of the reference heads, and the model configs
           the reference ships (tests/test_boundary_cpu.py)
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("UNITER_REFERENCE", "/root/reference")


def import_reference():
    apex = types.ModuleType("apex")
    norm = types.ModuleType("apex.normalization")
    fln = types.ModuleType("apex.normalization.fused_layer_norm")
    fln.FusedLayerNorm = torch.nn.LayerNorm
    apex.normalization = norm
    norm.fused_layer_norm = fln
    sys.modules.setdefault("apex", apex)
    sys.modules.setdefault("apex.normalization", norm)
    sys.modules.setdefault("apex.normalization.fused_layer_norm", fln)
    sys.path.insert(0, REF)
    import model.model as rm            # noqa: E402
    import model.vqa as rvqa            # noqa: E402
    import model.pretrain as rpre       # noqa: E402
    return rm, rvqa, rpre


def state_checksum(state):
    acc = 0.0
    for k in sorted(state):
        acc += float(state[k].double().abs().sum()) + 3.0 * float(state[k].double().sum())
    return np.float64(acc)


def grad_fingerprint(g, key):
    """(l2 norm, sum, 16 sampled entries) — compact stand-in for a full gradient tensor."""
    import hashlib
    h = int(hashlib.sha1(key.encode()).hexdigest()[:8], 16)
    gen = torch.Generator().manual_seed(h & 0x7FFFFFFF)
    flat = g.reshape(-1).double()
    idx = torch.randint(0, flat.numel(), (16,), generator=gen)
    return np.concatenate([[flat.norm().item(), flat.sum().item()], flat[idx].numpy()])


def run_case(rm, cfg_kw, img_dim, batch, out_path, full_grads, seed=0, adversarial=None):
    from uniter_b200.synth import seeded_state
    cfg = rm.UniterConfig(**cfg_kw)
    model = rm.UniterModel(cfg, img_dim)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    state = seeded_state(shapes, seed=seed)
    model.load_state_dict(state, strict=True)
    model.eval()  # dropout off: parity is only defined at p = 0

    gi = batch["gather_index"]
    if adversarial == "perm":
        g = torch.Generator().manual_seed(99)
        gi = gi.clone()
        for b in range(gi.size(0)):
            n = int(batch["attn_masks"][b].sum())
            gi[b, :n] = gi[b, :n][torch.randperm(n, generator=g)]
    elif adversarial == "malformed":
        # data/itm.py:356-361 passes a stale max_len: image slots index text-padding rows
        from uniter_b200.synth import get_gather_index
        Lt = batch["input_ids"].size(1)
        gi = get_gather_index(batch["txt_lens"], batch["num_bbs"], gi.size(0),
                              min(batch["txt_lens"]), gi.size(1))
        gi = gi.clamp(max=Lt + batch["img_feat"].size(1) - 1)

    taps = {}
    l0 = model.encoder.layer[0]
    hooks = [
        l0.attention.self.register_forward_hook(lambda m, i, o: taps.__setitem__("ctx", o.detach())),
        l0.attention.register_forward_hook(lambda m, i, o: taps.__setitem__("attn_out", o.detach())),
        l0.intermediate.register_forward_hook(lambda m, i, o: taps.__setitem__("ffn1", o.detach())),
        l0.register_forward_hook(lambda m, i, o: taps.__setitem__("layer_out", o.detach())),
    ]
    emb = model._compute_img_txt_embeddings(batch["input_ids"], batch["position_ids"],
                                            batch["img_feat"], batch["img_pos_feat"], gi)
    outs = model(batch["input_ids"], batch["position_ids"], batch["img_feat"],
                 batch["img_pos_feat"], batch["attn_masks"], gi, output_all_encoded_layers=True)
    for h in hooks:
        h.remove()
    pooled = model.pooler(outs[-1])
    maskf = batch["attn_masks"].float()
    loss = ((outs[-1] * maskf[..., None]) ** 2).sum() / maskf.sum() / outs[-1].size(-1)
    model.zero_grad()
    loss.backward()

    rec = {
        "weights_checksum": state_checksum(state),
        "gather_index": gi.numpy(),
        "embedding_output": emb.detach().numpy(),
        "pooled": pooled.detach().numpy(),
        "loss": np.float64(loss.item()),
    }
    for i, o in enumerate(outs):
        rec["layer_%d" % i] = o.detach().numpy()
    for k, v in taps.items():
        if k == "ffn1" and not full_grads:
            continue  # [B, L, 3072] is big; kept only for the tiny case
        rec["tap_" + k] = v.numpy()
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        if full_grads:
            rec["grad/" + name] = p.grad.numpy()
        rec["gfp/" + name] = grad_fingerprint(p.grad, name)
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024), "loss", loss.item())
    return model, state


def run_heads(rm, rvqa, rpre, out_path):
    """Head-level logits through the reference heads + reference encoder (tiny config)."""
    from uniter_b200.synth import seeded_state, synth_batch
    cfg_kw = TINY
    img_dim = 64
    batch = synth_batch(3, 5, 9, 4, 8, seed=7, img_dim=img_dim, vocab_size=cfg_kw["vocab_size_or_config_json_file"],
                        mlm_prob=0.3)
    rec = {}
    # --- VQA
    cfg = rm.UniterConfig(**cfg_kw)
    vqa = rvqa.UniterForVisualQuestionAnswering(cfg, img_dim, 17)
    st = seeded_state({k: tuple(v.shape) for k, v in vqa.state_dict().items()}, seed=3)
    vqa.load_state_dict(st, strict=True)
    vqa.eval()
    b = dict(batch)
    b["targets"] = torch.rand(3, 17, generator=torch.Generator().manual_seed(5))
    logits = vqa(b, compute_loss=False)
    rec["vqa_logits"] = logits.detach().numpy()
    rec["vqa_checksum"] = state_checksum(st)
    # --- pretraining heads (MLM, ITM)
    pre = rpre.UniterForPretraining(cfg, img_dim, 11)
    st = seeded_state({k: tuple(v.shape) for k, v in pre.state_dict().items()}, seed=4)
    pre.load_state_dict(st, strict=True)
    pre.eval()
    scores = pre(batch, task="mlm", compute_loss=False)
    rec["mlm_scores"] = scores.detach().numpy()
    b = dict(batch)
    b["targets"] = torch.tensor([1, 0, 1])
    b["ot_inputs"] = None
    itm, _ = pre(b, task="itm", compute_loss=False)
    rec["itm_scores"] = itm.detach().numpy()
    rec["pre_checksum"] = state_checksum(st)
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


def import_reference_data():
    """data/sampler.py, data/vqa.py, data/mlm.py import horovod / lmdb / lz4 / msgpack / (cy)toolz
    at module level; none of them is used by the sampler or the collate functions except
    cytoolz.partition_all and toolz.sandbox.unzip, shimmed here with their documented behaviour."""
    def shim(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    def partition_all(n, seq):
        seq = list(seq)
        for i in range(0, len(seq), n):
            yield tuple(seq[i:i + n])

    def unzip(seq):
        return tuple(zip(*list(seq)))

    hv = shim("horovod")
    hv.torch = shim("horovod.torch", rank=lambda: 0, size=lambda: 1)
    shim("cytoolz", partition_all=partition_all, concat=lambda x: [b for a in x for b in a], curry=lambda f: f)
    tz = shim("toolz")
    tz.sandbox = shim("toolz.sandbox", unzip=unzip)
    shim("lmdb")
    l4 = shim("lz4")
    l4.frame = shim("lz4.frame", compress=None, decompress=None)
    shim("msgpack")
    shim("msgpack_numpy", patch=lambda: None)
    shim("tqdm", tqdm=lambda x, **k: x)
    sys.path.insert(0, REF)
    import data.sampler as rsamp
    import data.vqa as rvqa_data
    import data.mlm as rmlm_data
    return rsamp, rvqa_data, rmlm_data


def batching_samples(seed, n, with_labels):
    """Per-sample tensors as the reference datasets' __getitem__ return them (data/vqa.py:30-42,
    data/mlm.py:62-94), seeded."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        tl = int(torch.randint(3, 12, (1,), generator=g))
        nbb = int(torch.randint(2, 9, (1,), generator=g))
        ids = torch.randint(1000, 2000, (tl,), generator=g)
        feat = torch.randn(nbb, 16, generator=g)
        pos = torch.rand(nbb, 7, generator=g)
        am = torch.ones(tl + nbb, dtype=torch.long)
        if with_labels:
            lab = torch.full((tl,), -1, dtype=torch.long)
            m = torch.rand(tl, generator=g) < 0.3
            lab[m] = ids[m]
            out.append((ids, feat, pos, am, lab))
        else:
            out.append((ids, feat, pos, am, torch.rand(5, generator=g)))
    return out


def run_batching(out_path):
    """The reference's own TokenBucketSampler and collate functions on seeded inputs."""
    import random
    rsamp, rvqa_data, rmlm_data = import_reference_data()
    rec = {}
    g = torch.Generator().manual_seed(17)
    lens = torch.randint(10, 120, (500,), generator=g).tolist()
    rec["lens"] = np.array(lens)
    random.seed(5)
    batches = list(iter(rsamp.TokenBucketSampler(lens, bucket_size=128, batch_size=1024, droplast=False)))
    rec["batches_flat"] = np.array([i for b in batches for i in b])
    rec["batches_len"] = np.array([len(b) for b in batches])
    random.seed(6)
    batches = list(iter(rsamp.TokenBucketSampler(lens, bucket_size=64, batch_size=800, droplast=True,
                                                 size_multiple=4)))
    rec["batches2_flat"] = np.array([i for b in batches for i in b])
    rec["batches2_len"] = np.array([len(b) for b in batches])
    for name, fn, lab in (("vqa", rvqa_data.vqa_collate, False), ("mlm", rmlm_data.mlm_collate, True)):
        b = fn(batching_samples(31, 6, lab))
        for k, v in b.items():
            rec["%s/%s" % (name, k)] = v.numpy()
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


class FakeTxtDB(object):
    """In-memory stand-in for TxtTokLmdb (data/data.py:176-230): only what the ITM datasets use."""

    def __init__(self, texts, txt2img, img2txts):
        self.texts, self.txt2img, self.img2txts = texts, txt2img, img2txts
        self.cls_, self.sep = 101, 102

    def __getitem__(self, id_):
        return {"input_ids": list(self.texts[id_])}

    def combine_inputs(self, *inputs):
        input_ids = [self.cls_]
        for ids in inputs:
            input_ids.extend(ids + [self.sep])
        return torch.tensor(input_ids)


class FakeImgDB(object):
    """Stand-in for DetectFeatLmdb: fname -> (feat [n, D], bb [n, 6] = x1,y1,x2,y2,w,h)."""

    def __init__(self, items):
        self.items = items

    def __getitem__(self, fname):
        return self.items[fname]


def itm_world(seed=5, n_img=9, txt_per_img=2, D=16):
    """A tiny seeded retrieval corpus: images, their captions, and the id maps the datasets use."""
    g = torch.Generator().manual_seed(seed)
    imgs, texts, txt2img, img2txts = {}, {}, {}, {}
    for i in range(n_img):
        fname = "img%02d" % i
        nbb = int(torch.randint(2, 8, (1,), generator=g))
        xy = torch.rand(nbb, 4, generator=g)
        bb = torch.cat([xy, (xy[:, 2:3] - xy[:, 0:1]).abs(), (xy[:, 3:4] - xy[:, 1:2]).abs()], 1)
        imgs[fname] = (torch.randn(nbb, D, generator=g), bb)
        img2txts[fname] = []
        for j in range(txt_per_img):
            tid = "t%02d_%d" % (i, j)
            tl = int(torch.randint(2, 8, (1,), generator=g))
            texts[tid] = torch.randint(1000, 2000, (tl,), generator=g).tolist()
            txt2img[tid] = fname
            img2txts[fname].append(tid)
    return FakeTxtDB(texts, txt2img, img2txts), FakeImgDB(imgs), sorted(texts.keys())


def mrm_samples(seed, n, soft, D=16, C=5):
    """Per-sample tuples as MrfrDataset / MrcDataset.__getitem__ return them (data/mrm.py:48-73,
    :141-173)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        tl = int(torch.randint(3, 9, (1,), generator=g))
        nb = int(torch.randint(2, 7, (1,), generator=g))
        ids = torch.randint(1000, 2000, (tl,), generator=g)
        f, p = torch.randn(nb, D, generator=g), torch.rand(nb, 7, generator=g)
        am = torch.ones(tl + nb, dtype=torch.long)
        m = torch.rand(nb, generator=g) < 0.4
        m[int(torch.randint(0, nb, (1,), generator=g))] = True
        tgt = torch.cat([torch.zeros(tl, dtype=torch.uint8), m.to(torch.uint8)])
        if soft:
            out.append((ids, f, p, torch.softmax(torch.randn(nb, C, generator=g), -1), am, m, tgt))
        else:
            out.append((ids, f, p, am, m, tgt))
    return out


def rank_samples(seed, n_anchor, n_pair, D=16):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_anchor):
        pairs = []
        for _ in range(n_pair):
            tl = int(torch.randint(3, 9, (1,), generator=g))
            nb = int(torch.randint(2, 7, (1,), generator=g))
            pairs.append((torch.randint(1000, 2000, (tl,), generator=g), torch.randn(nb, D, generator=g),
                          torch.rand(nb, 7, generator=g), torch.ones(tl + nb, dtype=torch.long)))
        out.append(pairs)
    return out


def run_itm_batching(out_path):
    """The reference's own ITM-ranking / MRM batch builders (data/itm.py:240-374, data/mrm.py:76-227)
    on seeded in-memory stores: itm_rank_collate, the two hard-negative datasets' __getitem__
    (negatives drawn from the global `random` state), mrfr_collate, mrc_collate."""
    import random
    import_reference_data()
    import data.itm as ritm
    import data.mrm as rmrm
    rec = {}

    def put(prefix, batch):
        for k, v in batch.items():
            rec["%s/%s" % (prefix, k)] = v.numpy() if torch.is_tensor(v) else np.array(v)

    put("rank", ritm.itm_rank_collate(rank_samples(41, 3, 3)))
    txt_db, img_db, ids = itm_world()
    for name, cls in (("hn_t", ritm.ItmRankDatasetHardNegFromText), ("hn_i", ritm.ItmRankDatasetHardNegFromImage)):
        ds = object.__new__(cls)                      # skip the LMDB-typed constructor
        ds.txt_db, ds.img_db, ds.ids = txt_db, img_db, ids
        ds.txt2img = {i: txt_db.txt2img[i] for i in ids}
        ds.img2txts = txt_db.img2txts
        ds.img_name_list = list(ds.img2txts.keys())
        ds.txt_name_list = list(ds.txt2img.keys())
        ds.neg_sample_size = 4
        for i in (0, 7):
            random.seed(100 + i)
            put("%s%d" % (name, i), ritm.itm_rank_hn_collate([ds[i]]))
    put("mrfr", rmrm.mrfr_collate(mrm_samples(51, 5, False)))
    put("mrc", rmrm.mrc_collate(mrm_samples(52, 5, True)))
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


def hardneg_inputs(sample_from, seed):
    """A 9-pair hard-negative batch as data/itm.py:270-361 builds it (one text x 9 images, or one
    image x 9 texts), plus random pair scores."""
    from uniter_b200.synth import get_gather_index
    g = torch.Generator().manual_seed(seed)
    n, D = 9, 16
    if sample_from == "t":
        tl = 6
        input_ids = torch.randint(1000, 2000, (1, tl), generator=g)
        num_bbs = torch.randint(2, 8, (n,), generator=g).tolist()
        img_feat = torch.zeros(n, max(num_bbs), D)
        img_pos = torch.zeros(n, max(num_bbs), 7)
        for i, nb in enumerate(num_bbs):
            img_feat[i, :nb] = torch.randn(nb, D, generator=g)
            img_pos[i, :nb] = torch.rand(nb, 7, generator=g)
        attn = torch.zeros(n, max(num_bbs) + tl, dtype=torch.long)
        for i, nb in enumerate(num_bbs):
            attn[i, :tl + nb] = 1
        gather = get_gather_index([tl] * n, num_bbs, n, tl, attn.size(1))
    else:
        nbb = 5
        txt_lens = torch.randint(3, 9, (n,), generator=g).tolist()
        input_ids = torch.zeros(n, max(txt_lens), dtype=torch.long)
        for i, tl in enumerate(txt_lens):
            input_ids[i, :tl] = torch.randint(1000, 2000, (tl,), generator=g)
        img_feat = torch.randn(1, nbb, D, generator=g)
        img_pos = torch.rand(1, nbb, 7, generator=g)
        attn = torch.zeros(n, max(txt_lens) + nbb, dtype=torch.long)
        for i, tl in enumerate(txt_lens):
            attn[i, :tl + nbb] = 1
        # data/itm.py:356-361 passes the LAST loop value of tl as max_len (the malformed index)
        gather = get_gather_index(txt_lens, [nbb] * n, n, txt_lens[-1], attn.size(1))
    batch = {"input_ids": input_ids, "position_ids": torch.arange(input_ids.size(1)).unsqueeze(0),
             "img_feat": img_feat, "img_pos_feat": img_pos, "attn_masks": attn, "gather_index": gather}
    scores = torch.randn(n, 1, generator=g)
    return batch, scores


def run_hardneg(rm, out_path):
    """Row selection of the reference's UniterForImageTextRetrievalHardNeg._get_hard_batch."""
    import model.itm as ritm
    cfg = rm.UniterConfig(**TINY)
    mod = ritm.UniterForImageTextRetrievalHardNeg(cfg, 16, hard_size=3)
    rec = {}
    for sf in ("t", "i"):
        batch, scores = hardneg_inputs(sf, seed=77)
        n = batch["attn_masks"].size(0)
        if sf == "t":
            batch["input_ids"] = batch["input_ids"].expand(n, -1)
        else:
            batch["img_feat"] = batch["img_feat"].expand(n, -1, -1)
            batch["img_pos_feat"] = batch["img_pos_feat"].expand(n, -1, -1)
        hb = mod._get_hard_batch(batch, scores, sf)
        for k, v in hb.items():
            rec["%s/%s" % (sf, k)] = v.numpy() if torch.is_tensor(v) else np.array(v)
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


def pretrain_mrm_extra(batch):
    """Masked-region inputs of the MRFR / MRC tasks (model/pretrain.py:135-154, :201-229) for one
    synth_batch, seeded: img_masks, img_mask_tgt, feat_targets (fp16-rounded), label_targets."""
    gen = torch.Generator().manual_seed(8)
    img_masks = torch.rand(batch["img_feat"].shape[:2], generator=gen) < 0.4
    for i, nb in enumerate(batch["num_bbs"]):
        img_masks[i, nb:] = False
    img_masks[0, 0] = True
    img_mask_tgt = torch.zeros_like(batch["attn_masks"], dtype=torch.bool)
    for i, tl in enumerate(batch["txt_lens"]):
        nb = batch["num_bbs"][i]
        img_mask_tgt[i, tl:tl + nb] = img_masks[i, :nb]
    n = int(img_masks.sum())
    return {"img_masks": img_masks, "img_mask_tgt": img_mask_tgt,
            "feat_targets": batch["img_feat"][img_masks].half().float(),
            "label_targets": torch.softmax(torch.randn(n, 11, generator=gen), -1)}


def library_pretrain_inputs(use_index):
    """(base batch, the same batch with masked regions, keys the heads read) of the multi-task
    pre-training comparison; without `use_index` the fixed-shape row lists are left out."""
    from uniter_b200.synth import synth_batch, synth_mrm
    base = synth_batch(5, 5, 9, 4, 8, seed=17, img_dim=64, vocab_size=2000, mlm_prob=0.3)
    mb = synth_mrm(base, mask_prob=0.3, label_dim=11, seed=3)
    keys = [k for k, v in mb.items() if torch.is_tensor(v)]
    if not use_index:
        keys = [k for k in keys if k not in ("mlm_index", "mlm_targets", "mrm_index", "mrm_valid", "mrm_inv_n")]
    return base, mb, keys


LIBRARY_PRETRAIN_TASKS = ("mlm", "mrfr", "mrc", "mrc-kl", "itm")
LIBRARY_PRETRAIN_GRADS = (
    "feat_regress.net.0.weight", "feat_regress.net.2.weight", "feat_regress.bias",
    "region_classifier.net.0.weight", "region_classifier.net.3.weight", "region_classifier.net.3.bias",
    "itm_output.weight", "itm_output.bias", "uniter.pooler.dense.weight", "uniter.pooler.dense.bias",
    "cls.predictions.transform.dense.weight", "cls.predictions.bias",
    "uniter.embeddings.word_embeddings.weight", "uniter.img_embeddings.img_linear.weight",
    "uniter.img_embeddings.mask_embedding.weight", "uniter.encoder.layer.1.output.dense.weight")


def grad_rows(g, key, whole=65536, budget=16384):
    """Rows of gradient `g` to store: every row when it holds <= `whole` entries (all but the
    word-embedding table), else `budget` entries: the largest-norm half (the rows the embedding
    lookup touches) plus a seeded sample of the rest (the tied decoder's dense part)."""
    import hashlib
    if g.dim() < 2 or g.numel() <= whole:
        return torch.arange(g.size(0))
    n = max(2, budget // g[0].numel())
    top = g.norm(dim=1).topk(n // 2)[1]
    rest = torch.ones(g.size(0), dtype=torch.bool)
    rest[top] = False
    gen = torch.Generator().manual_seed(int(hashlib.sha1(key.encode()).hexdigest()[:8], 16) & 0x7FFFFFFF)
    pick = rest.nonzero().squeeze(1)[torch.randperm(int(rest.sum()), generator=gen)[:n - n // 2]]
    return torch.cat([top, pick]).sort()[0]


def run_reference_heads(rm, out_path):
    """The reference's own task heads over the reference encoder (CPU fp32, weights rounded to fp16):
    what tests/test_reference_heads_gpu.py compares the drop-in heads on the GPU with."""
    import model.itm as ritm
    import model.pretrain as rpre
    from uniter_b200.synth import seeded_state, synth_batch

    def set_dropout_zero(m):
        for _, mod in m.named_modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0

    cfg = rm.UniterConfig(**TINY)
    rec = {}
    # --- pre-training heads, MRFR / MRC on the heads batch
    pre = rpre.UniterForPretraining(cfg, 64, 11)
    st = seeded_state({k: tuple(v.shape) for k, v in pre.state_dict().items()}, seed=4)
    pre.load_state_dict({k: v.half().float() for k, v in st.items()}, strict=True)
    pre.eval()
    batch = synth_batch(3, 5, 9, 4, 8, seed=7, img_dim=64, vocab_size=2000, mlm_prob=0.3)
    cb = {k: v for k, v in batch.items() if torch.is_tensor(v)}
    cb["img_feat"] = cb["img_feat"].half().float()
    cb["img_pos_feat"] = cb["img_pos_feat"].half().float()
    extra = pretrain_mrm_extra(batch)
    with torch.no_grad():
        for task in ("mrfr", "mrc"):
            rec["pre/" + task] = pre(dict(cb, **extra), task=task, compute_loss=False).numpy()
    # --- hard-negative ITM: rows mined and loss of one train step, both directions
    mod = ritm.UniterForImageTextRetrievalHardNeg(cfg, 16, hard_size=3)
    st = seeded_state({k: tuple(v.shape) for k, v in mod.state_dict().items()}, seed=6)
    mod.load_state_dict({k: v.half().float() for k, v in st.items()}, strict=True)
    mod.train()
    set_dropout_zero(mod)
    for sf in ("t", "i"):
        cbatch, _ = hardneg_inputs(sf, seed=77)
        cbatch["img_feat"] = cbatch["img_feat"].half().float()
        cbatch["img_pos_feat"] = cbatch["img_pos_feat"].half().float()
        picked = {}
        orig = mod._get_hard_batch
        mod._get_hard_batch = lambda bt, sc, sfrom, _o=orig: picked.setdefault("rows", _o(bt, sc, sfrom))
        loss = mod(cbatch, sample_from=sf, compute_loss=True)
        mod._get_hard_batch = orig
        key = "img_feat" if sf == "t" else "input_ids"
        rec["hardneg/%s/%s" % (sf, key)] = picked["rows"][key].float().numpy()
        rec["hardneg/%s/loss" % sf] = loss.detach().numpy()
    # --- multi-task pre-training step: logits, per-element losses, gradients of the summed loss
    ref = rpre.UniterForPretraining(cfg, 64, 11)
    st = seeded_state({k: tuple(v.shape) for k, v in ref.state_dict().items()}, seed=4)
    ref.load_state_dict({k: v.half().float() for k, v in st.items()}, strict=True)
    ref.eval()
    base, mb, keys = library_pretrain_inputs(use_index=False)
    cb = {k: (mb[k].half().float() if mb[k].is_floating_point() else mb[k]) for k in keys}
    cb["targets"] = torch.tensor([1, 0, 1, 1, 0])
    cb["ot_inputs"] = None
    plain = dict(cb, img_feat=base["img_feat"].half().float())
    total = 0.0
    for task in LIBRARY_PRETRAIN_TASKS:
        bc = plain if task in ("mlm", "itm") else cb
        with torch.no_grad():
            want = ref(bc, task=task, compute_loss=False)
        lw = ref(bc, task=task, compute_loss=True)
        want = want[0] if isinstance(want, tuple) else want
        lw = lw[0] if isinstance(lw, tuple) else lw
        rec["library/%s/logits" % task] = want.numpy()
        rec["library/%s/loss" % task] = lw.detach().numpy()
        total = total + lw.float().mean()
    total.backward()
    params = dict(ref.named_parameters())
    for name in LIBRARY_PRETRAIN_GRADS:
        g = params[name].grad
        rows = grad_rows(g, name)
        rec["library/grad_rows/" + name] = rows.numpy()
        rec["library/grad/" + name] = g[rows].numpy()
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


def run_reference_schema(rm, rvqa, rpre, out_path):
    """State-dict schema of the reference's own heads over the reference encoder and the model
    configs it ships (config/uniter-{base,large}.json)."""
    import json
    cfg = rm.UniterConfig(**TINY)
    rec = {"configs": {}}
    for name in ("uniter-base.json", "uniter-large.json"):
        with open(os.path.join(REF, "config", name)) as fh:
            rec["configs"][name] = json.load(fh)
    for tag, mod in (("vqa", rvqa.UniterForVisualQuestionAnswering(cfg, 64, 17)),
                     ("pretraining", rpre.UniterForPretraining(cfg, 64, 11))):
        rec[tag] = {k: list(v.shape) for k, v in mod.state_dict().items()}
    with open(out_path, "w") as fh:
        json.dump(rec, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


def run_adamw(out_path):
    """4 steps of the reference's own AdamW (optim/adamw.py) + clip_grad_norm_ on seeded fp32
    tensors: two param groups (decay 0.01 / 0), a linear-warmup lr per step, gradient clipping at
    2.0 (train_vqa.py:223-226 default --grad_norm 2.0)."""
    import warnings
    sys.path.insert(0, REF)
    from optim.adamw import AdamW
    g = torch.Generator().manual_seed(21)
    shapes = [(37, 16), (16,), (5, 8, 3), (129,)]
    params = [torch.nn.Parameter(torch.randn(s, generator=g) * 0.1) for s in shapes]
    opt = AdamW([{"params": [params[0], params[2]], "weight_decay": 0.01},
                 {"params": [params[1], params[3]], "weight_decay": 0.0}],
                lr=3e-4, betas=(0.9, 0.98))
    rec = {"n_params": np.array(len(shapes)), "betas": np.array([0.9, 0.98]), "eps": np.array(1e-6),
           "weight_decay": np.array([0.01, 0.0, 0.01, 0.0]), "max_norm": np.array(2.0)}
    for i, p in enumerate(params):
        rec["p0_%d" % i] = p.detach().numpy().copy()
    lrs = [1e-4, 2e-4, 3e-4, 2.5e-4]
    rec["lrs"] = np.array(lrs)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for t, lr in enumerate(lrs):
            for grp in opt.param_groups:
                grp["lr"] = lr
            for i, p in enumerate(params):
                scale = 30.0 if t == 1 else 1.0        # step 1 exceeds the clip threshold
                p.grad = torch.randn(p.shape, generator=g) * 0.05 * scale
                rec["g%d_%d" % (t, i)] = p.grad.numpy().copy()
            total = torch.nn.utils.clip_grad_norm_(params, 2.0)
            rec["norm%d" % t] = np.array(float(total))
            opt.step()
            for i, p in enumerate(params):
                rec["p%d_%d" % (t + 1, i)] = p.detach().numpy().copy()
    np.savez_compressed(out_path, **rec)
    print("wrote", out_path, "%.1f KB" % (os.path.getsize(out_path) / 1024))


TINY = dict(vocab_size_or_config_json_file=2000, hidden_size=128, num_hidden_layers=2,
            num_attention_heads=2, intermediate_size=512, hidden_act="gelu",
            hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
            max_position_embeddings=64, type_vocab_size=2, initializer_range=0.02)
BASE_L1 = dict(vocab_size_or_config_json_file=28996, hidden_size=768, num_hidden_layers=1,
               num_attention_heads=12, intermediate_size=3072, hidden_act="gelu",
               hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
               max_position_embeddings=512, type_vocab_size=2, initializer_range=0.02)


LARGE_L1 = dict(vocab_size_or_config_json_file=28996, hidden_size=1024, num_hidden_layers=1,
                num_attention_heads=16, intermediate_size=4096, hidden_act="gelu",
                hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
                max_position_embeddings=512, type_vocab_size=2, initializer_range=0.02)


def main():
    from uniter_b200.synth import synth_batch
    rm, rvqa, rpre = import_reference()
    torch.set_num_threads(8)
    # tiny: ragged batch of 4
    tb = synth_batch(4, 5, 12, 3, 9, seed=11, img_dim=64, vocab_size=2000)
    run_case(rm, TINY, 64, tb, os.path.join(HERE, "tiny.npz"), full_grads=True)
    run_case(rm, TINY, 64, tb, os.path.join(HERE, "tiny_adv_perm.npz"), full_grads=False,
             adversarial="perm")
    run_case(rm, TINY, 64, tb, os.path.join(HERE, "tiny_adv_malformed.npz"), full_grads=False,
             adversarial="malformed")
    # C1a: no padding; C1b: ragged
    c1a = synth_batch(2, 0, 0, 0, 0, seed=0, txt_lens=[20, 20], num_bbs=[36, 36])
    run_case(rm, BASE_L1, 2048, c1a, os.path.join(HERE, "c1a.npz"), full_grads=False)
    c1b = synth_batch(2, 0, 0, 0, 0, seed=0, txt_lens=[20, 14], num_bbs=[36, 30])
    run_case(rm, BASE_L1, 2048, c1b, os.path.join(HERE, "c1b.npz"), full_grads=False)
    # UNITER-large geometry (config/uniter-large.json: H 1024, 16 heads, I 4096), 1 layer, ragged
    lg = synth_batch(2, 0, 0, 0, 0, seed=3, txt_lens=[9, 6], num_bbs=[11, 14])
    run_case(rm, LARGE_L1, 2048, lg, os.path.join(HERE, "large_l1.npz"), full_grads=False)
    run_heads(rm, rvqa, rpre, os.path.join(HERE, "heads_tiny.npz"))
    run_hardneg(rm, os.path.join(HERE, "hardneg.npz"))
    run_reference_heads(rm, os.path.join(HERE, "reference_heads.npz"))
    run_reference_schema(rm, rvqa, rpre, os.path.join(HERE, "reference_schema.json"))
    run_adamw(os.path.join(HERE, "adamw.npz"))
    run_batching(os.path.join(HERE, "batching.npz"))
    run_itm_batching(os.path.join(HERE, "itm_batching.npz"))


if __name__ == "__main__":
    main()
