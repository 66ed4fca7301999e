"""Generate tests/golden/*.npz by running the UNMODIFIED reference modules (behind oracle/reference_shim.py)
on seeded inputs.  Runs only in the authoring container (needs /root/reference); the fixtures are committed.

    python -m oracle.make_golden            # writes tests/golden/

Weights are never stored: every fixture records the seeds from which `pigeon_b200.synthetic` regenerates
them bit-identically (torch CPU generator), so the files stay small.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import pandas as pd
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import golden  # noqa: E402
from oracle import reference_shim as rs  # noqa: E402
from pigeon_b200 import synthetic  # noqa: E402
from pigeon_b200.vit_engine import VitDims  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def hf_model(dims: VitDims, sd):
    from transformers import CLIPVisionConfig, CLIPVisionModel
    cfg = CLIPVisionConfig(hidden_size=dims.hidden, intermediate_size=dims.intermediate, num_hidden_layers=dims.layers,
                           num_attention_heads=dims.heads, image_size=dims.image_size, patch_size=dims.patch_size,
                           projection_dim=768, layer_norm_eps=dims.ln_eps, attn_implementation="eager")
    m = CLIPVisionModel(cfg)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    return m.eval()


def head_weights(C, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(C, D, generator=g) * 0.03, torch.randn(C, generator=g) * 0.01


def geo_fixture():
    from preprocessing import haversine, haversine_matrix, smooth_labels
    rng = np.random.default_rng(11)
    n, m = 64, 37
    x = np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1)
    y = np.stack([rng.uniform(-180, 180, n), rng.uniform(-90, 90, n)], 1)
    x[0], y[0] = [10.0, 20.0], [10.0, 20.0]            # zero distance
    x[1], y[1] = [0.0, 0.0], [180.0, 0.0]              # antipodes: pi * R
    x[2], y[2] = [-179.9, 89.9], [179.9, -89.9]
    c = np.stack([rng.uniform(-180, 180, m), rng.uniform(-90, 90, m)], 1)
    xt, yt, ct = torch.tensor(x), torch.tensor(y), torch.tensor(c)
    hm = haversine_matrix(xt, ct.t())
    np.savez(os.path.join(OUT, "geo.npz"), x=x, y=y, c=c,
             haversine=haversine(xt, yt).numpy(),
             haversine_f64_f32=haversine(xt, yt.float()).numpy(),   # the dtype mix ProtoRefiner produces (:198-201)
             haversine_matrix=hm.numpy(), smooth_labels=smooth_labels(hm).numpy())


def head_fixture(tmp):
    from models.super_guessr import SuperGuessr
    C, D, B = 1000, 1024, 6
    W, b = head_weights(C, D, seed=21)
    g = torch.Generator().manual_seed(22)
    emb4 = torch.randn(B, 4, D, generator=g) * 0.3
    emb1 = torch.randn(B, D, generator=g) * 0.3
    cells = synthetic.synthetic_geocells(C, 0)
    labels = torch.tensor(synthetic.synthetic_geocells(B, 5))
    labels_clf = torch.tensor([3, 999, 0, 17, 500, 250])
    out = {}
    with rs.chdir(tmp):
        for name, kw, emb in (("pano", dict(panorama=True, num_candidates=50), emb4),
                              ("pano_smooth", dict(panorama=True, num_candidates=5, should_smooth_labels=True), emb4),
                              ("single", dict(panorama=False, num_candidates=5), emb1),
                              ("single_from4", dict(panorama=False, num_candidates=7), emb4)):
            sg = SuperGuessr(None, **kw).eval()
            with torch.no_grad():
                sg.cell_layer.weight.copy_(W)
                sg.cell_layer.bias.copy_(b)
                o = sg(embedding=emb, labels=labels, labels_clf=labels_clf)
            # pandas' default CSV float parser is not round-trip exact: keep the table the reference actually loaded
            assert np.allclose(sg.lla_geocells.numpy(), cells, rtol=1e-12, atol=1e-12)
            out["centroids"] = sg.lla_geocells.detach().numpy().copy()
            out[f"{name}_loss"] = o.loss.numpy()
            out[f"{name}_preds_LLH"] = o.preds_LLH.numpy()
            out[f"{name}_preds_geocell"] = o.preds_geocell.numpy()
            out[f"{name}_topk_val"] = o.top5_geocells.values.numpy()
            out[f"{name}_topk_idx"] = o.top5_geocells.indices.numpy()
    np.savez(os.path.join(OUT, "head.npz"), emb4=emb4.numpy(), emb1=emb1.numpy(), labels=labels.numpy(),
             labels_clf=labels_clf.numpy(), meta=json.dumps(dict(C=C, D=D, w_seed=21, cells_seed=0)), **out)


def train_fixture(tmp):
    """Head-only fine-tune steps through the UNMODIFIED reference module + torch.optim.AdamW, the way
    training/train_eval_loop.py:187,215-221 drives it (model.train(); loss.backward(); gradient accumulation;
    optimizer.step(); optimizer.zero_grad()) with base_model=None (training on embeddings, train_modes on_embeddings)."""
    from models.super_guessr import SuperGuessr
    C, D, B, steps, acc, lr = 1000, 128, 8, 3, 2, 1e-3
    W, b = head_weights(C, D, seed=71)
    g = torch.Generator().manual_seed(72)
    emb = torch.randn(steps * acc, B, 4, D, generator=g) * 0.5
    labels = torch.tensor(np.stack([synthetic.synthetic_geocells(B, 80 + i) for i in range(steps * acc)]))
    labels_clf = torch.randint(0, C, (steps * acc, B), generator=g)
    out = {}
    with rs.chdir(tmp):
        gm = torch.Generator().manual_seed(73)
        labels_mt = torch.randn(steps * acc, B, 6, generator=gm)
        labels_climate = torch.nn.functional.one_hot(torch.randint(0, 28, (steps * acc, B), generator=gm), 28).float()
        labels_month = torch.randint(0, 12, (steps * acc, B), generator=gm)
        out.update(labels_mt=labels_mt.numpy(), labels_climate=labels_climate.numpy(), labels_month=labels_month.numpy())
        for name, smooth in (("smooth", True), ("index", False), ("multitask", True)):
            mt = name == "multitask"
            torch.manual_seed(74)      # the auxiliary heads keep nn.Linear's default init; the test rebuilds them from this seed
            sg = SuperGuessr(None, panorama=True, num_candidates=5, should_smooth_labels=smooth, embed_dim=D,
                             multi_task=mt).train()
            if mt:
                for hn in ("multi_task_head", "climate_layer", "month_layer"):
                    out[f"mt_init_{hn}_w"] = getattr(sg, hn).weight.detach().numpy().copy()
                    out[f"mt_init_{hn}_b"] = getattr(sg, hn).bias.detach().numpy().copy()
            with torch.no_grad():
                sg.cell_layer.weight.copy_(W)
                sg.cell_layer.bias.copy_(b)
            opt = torch.optim.AdamW(sg.parameters(), lr=lr)                       # train_eval_loop.py:187
            opt.zero_grad()
            losses = []
            for i in range(steps * acc):
                kw = dict(labels_multi_task=labels_mt[i], labels_climate=labels_climate[i], labels_month=labels_month[i]) if mt else {}
                o = sg(embedding=emb[i], labels=labels[i], labels_clf=labels_clf[i], **kw)
                o.loss.backward()
                losses.append(float(o.loss))
                if i % acc == acc - 1:                                            # :218-221
                    if i == acc - 1 and not mt:
                        out[f"{name}_grad_w_step1"] = sg.cell_layer.weight.grad.detach().numpy().copy()
                        out[f"{name}_grad_b_step1"] = sg.cell_layer.bias.grad.detach().numpy().copy()
                    opt.step()
                    opt.zero_grad()
                    if i == acc - 1 and not mt:
                        out[f"{name}_w_step1"] = sg.cell_layer.weight.detach().numpy().copy()
                        out[f"{name}_b_step1"] = sg.cell_layer.bias.detach().numpy().copy()
            out[f"{name}_losses"] = np.asarray(losses, dtype=np.float64)
            out[f"{name}_w_final"] = sg.cell_layer.weight.detach().numpy().copy()
            out[f"{name}_b_final"] = sg.cell_layer.bias.detach().numpy().copy()
            if mt:
                for hn in ("multi_task_head", "climate_layer", "month_layer"):
                    out[f"mt_final_{hn}_w"] = getattr(sg, hn).weight.detach().numpy().copy()
                    out[f"mt_final_{hn}_b"] = getattr(sg, hn).bias.detach().numpy().copy()
            out["centroids"] = sg.lla_geocells.detach().numpy().copy()
    golden.save("train_head", dict(emb=emb.numpy(), labels=labels.numpy(), labels_clf=labels_clf.numpy(), w0=W.numpy(),
                                   b0=b.numpy(), **out),
                dict(C=C, D=D, B=B, steps=steps, acc=acc, lr=lr, betas=[0.9, 0.999], eps=1e-8, weight_decay=0.01, w_seed=71, emb_seed=72))


def preprocess_fixture():
    """Images through the third-party code the reference calls for pre-processing: Pillow's BICUBIC resize and the
    PIL-backend CLIP image processor of the transformers installed here (the pinned 4.23.1 CLIPFeatureExtractor is the
    same pipeline; its formulas are restated in oracle/preprocess.py).  Smooth synthetic photos + noise, several aspect
    ratios, one up-scaling case, one that needs no resize."""
    from PIL import Image
    from transformers import CLIPImageProcessorPil
    from oracle import preprocess as op
    proc = CLIPImageProcessorPil(do_resize=True, size={"shortest_edge": 336}, resample=3, do_center_crop=True,
                                 crop_size={"height": 336, "width": 336}, do_rescale=True, rescale_factor=1 / 255,
                                 do_normalize=True, image_mean=list(op.CLIP_MEAN), image_std=list(op.CLIP_STD),
                                 do_convert_rgb=True)
    out = {}
    shapes = [(480, 640), (500, 375), (150, 210), (336, 400), (900, 1300)]
    for i, (h, w) in enumerate(shapes):
        img = synthetic.synthetic_photo(h, w, seed=91 + i)        # integer-only generator: regenerated by the tests
        pil = Image.fromarray(img)
        nh, nw = op.resized_shape(h, w)
        resized = np.asarray(pil.resize((nw, nh), resample=Image.BICUBIC))
        top, left = (nh - 336) // 2, (nw - 336) // 2
        crop = resized[top:top + 336, left:left + 336]
        px = proc(images=pil, return_tensors="np")["pixel_values"][0]
        assert np.array_equal(px, op.clip_preprocess(img)), "restated pipeline != HF PIL-backend processor"
        assert np.array_equal(crop, op.clip_preprocess(img, return_u8=True)[1])
        sha = lambda a: np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)
        out[f"img{i}_sha"] = sha(img)
        out[f"crop{i}_sha"] = sha(crop)                       # uint8 stage (Pillow), full tensor
        out[f"px{i}_sha"] = sha(px)                           # float32 stage (HF PIL-backend processor), full tensor
        out[f"crop{i}_sample"] = crop[::6].copy()
        out[f"px{i}_sample"] = px[:, ::12, ::7].copy()
    out["shapes"] = np.asarray(shapes)
    np.savez_compressed(os.path.join(OUT, "preprocess.npz"), **out)


def train_tower_fixture(tmp, name, dims: VitDims, n_views, sd_seed, px_seed, std, stride):
    """Gradients of the reference fine-tune step through the tower: the UNMODIFIED reference SuperGuessr over a HF
    CLIPVisionModel, loss.backward() under torch autograd in fp32 (training/train_eval_loop.py:215-216), every tower and
    head parameter trainable.  Views go through the non-panorama branch (super_guessr.py:388 hard-codes 336 x 336 in the
    panorama reshape).  Per parameter the fixture keeps the L2 norm and every `stride`-th element of the gradient."""
    from models.super_guessr import SuperGuessr
    C = 1000
    sd = synthetic.random_vit_state_dict(dims, seed=sd_seed, std=std)
    hf = hf_model(dims, sd)
    W, b = head_weights(C, dims.hidden, seed=33)
    g = torch.Generator().manual_seed(px_seed)
    px = torch.randn(n_views, 3, dims.image_size, dims.image_size, generator=g)
    labels = torch.tensor(synthetic.synthetic_geocells(n_views, 7))
    labels_clf = (torch.arange(n_views) * 13 + 5) % C
    with rs.chdir(tmp):
        sg = SuperGuessr(hf.base_model, panorama=False, should_smooth_labels=True, num_candidates=5).train()
    with torch.no_grad():
        sg.cell_layer.weight.copy_(W)
        sg.cell_layer.bias.copy_(b)
    for p_ in sg.parameters():
        p_.requires_grad_(p_.dtype == torch.float32)
    sg.lla_geocells.requires_grad_(False)
    o = sg(pixel_values=px, labels=labels, labels_clf=labels_clf)
    o.loss.backward()
    out = {}
    for n_, p_ in sg.named_parameters():
        if p_.grad is None:
            continue
        gflat = p_.grad.detach().reshape(-1).double()
        key = n_.replace("base_model.", "")
        out["norm/" + key] = np.asarray(float(gflat.norm()))
        out["sub/" + key] = gflat[::stride].float().numpy()
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"),
                        meta=json.dumps(dict(dims=dims.__dict__, sd_seed=sd_seed, std=std, px_seed=px_seed, n_views=n_views,
                                             C=C, w_seed=33, stride=stride)),
                        loss=np.asarray(float(o.loss)), labels=labels.numpy(), labels_clf=labels_clf.numpy(),
                        centroids=sg.lla_geocells.detach().numpy().copy(), **out)


def vit_fixture(tmp, name, dims: VitDims, sd_seed, n_samples, panorama, px_seed, std):
    """pixel_values -> reference SuperGuessr(HF CLIPVisionModel.base_model) -> ModelOutput; plus CLIPEmbedding."""
    from models.clip_embedder import CLIPEmbedding
    from models.super_guessr import SuperGuessr
    C = 1000
    sd = synthetic.random_vit_state_dict(dims, seed=sd_seed, std=std)
    hf = hf_model(dims, sd)
    W, b = head_weights(C, dims.hidden, seed=31)
    g = torch.Generator().manual_seed(px_seed)
    ch = 12 if panorama else 3
    px = torch.randn(n_samples, ch, dims.image_size, dims.image_size, generator=g)
    labels = torch.tensor(synthetic.synthetic_geocells(n_samples, 6))
    labels_clf = torch.arange(n_samples) * 7 % C
    with rs.chdir(tmp):
        sg = SuperGuessr(hf.base_model, panorama=panorama, freeze_base=True, num_candidates=50).eval()
    with torch.no_grad():
        sg.cell_layer.weight.copy_(W)
        sg.cell_layer.bias.copy_(b)
        if dims.image_size != 336:
            # super_guessr.py:388 hard-codes 336x336 in the panorama reshape; for the small geometry feed the
            # already-unfolded views through the non-panorama branch of the SAME reference forward.
            views = px.reshape(-1, 3, dims.image_size, dims.image_size)
            sg.panorama = False
            o = sg(pixel_values=views, labels=labels.repeat_interleave(ch // 3, 0), labels_clf=labels_clf.repeat_interleave(ch // 3))
            emb_views = o.embedding
        else:
            o = sg(pixel_values=px, labels=labels, labels_clf=labels_clf)
            emb_views = o.embedding
        ce = object.__new__(CLIPEmbedding)
        torch.nn.Module.__init__(ce)
        ce.device, ce.clip_model, ce.panorama = "cpu", hf, panorama
        views = px.reshape(-1, 3, dims.image_size, dims.image_size)
        ce_emb = ce.forward(views)                       # clip_embedder.py:79-89 -> :42-66
    np.savez(os.path.join(OUT, f"{name}.npz"),
             meta=json.dumps(dict(dims=dims.__dict__, sd_seed=sd_seed, std=std, px_seed=px_seed, n_samples=n_samples,
                                  panorama=panorama, C=C, w_seed=31, cells_seed=0)),
             embedding=emb_views.numpy(), clip_embedding=ce_emb.numpy(), loss=o.loss.numpy(),
             preds_LLH=o.preds_LLH.numpy(), preds_geocell=o.preds_geocell.numpy(),
             topk_val=o.top5_geocells.values.numpy(), topk_idx=o.top5_geocells.indices.numpy(),
             labels=labels.numpy(), labels_clf=labels_clf.numpy(), centroids=sg.lla_geocells.detach().numpy().copy())


class _DuckProtos:
    """protos[cell]: what the reference's per-cell HF Dataset (torch format) yields, for datasets>=3 where
    Dataset['embedding'] no longer returns a Tensor (SURVEY.md §8c): ['embedding'] -> Tensor, [i] -> row dict."""

    def __init__(self, ds):
        self.rows = [ds[i] for i in range(len(ds))]
        self.emb = torch.stack([r["embedding"] for r in self.rows])

    def __getitem__(self, k):
        return self.emb if isinstance(k, str) and k == "embedding" else self.rows[k]

    def __len__(self):
        return len(self.rows)


def refiner_fixture(tmp, name, C, P, D, B, kc, topk, members, T, maxref, seed):
    """Build the reference's on-disk inputs (HF DatasetDict + prototype CSV), run the UNMODIFIED ProtoRefiner
    constructor (bank building, proto_refiner.py:53-90,257-313,359-378) and forward (:121-255)."""
    import concurrent.futures as cf
    import datasets
    import models.proto_refiner as pr
    bank = synthetic.synthetic_bank(C, P, D, seed=seed, members_mean=members, empty_cells=3)
    n_train = bank["data_emb"].shape[0]
    tag = name or f"anon{seed}"
    ds_path, csv_path = os.path.join(tmp, f"hf_{tag}"), os.path.join(tmp, f"protos_{tag}.csv")
    # training embeddings as the reference stores them: (4, D) per sample (4-view panoramas) -> the refiner
    # averages views itself (:370-371).  Views are the stored mean +- a perturbation that cancels exactly.
    rng = np.random.default_rng(seed + 1)
    pert = rng.standard_normal((n_train, 2, D)).astype(np.float32) * 0.01
    e = bank["data_emb"]
    views = np.stack([e + pert[:, 0], e - pert[:, 0], e + pert[:, 1], e - pert[:, 1]], axis=1).astype(np.float32)
    ds = datasets.Dataset.from_dict({"embedding": views.tolist(), "labels": bank["data_lnglat"].tolist()})
    datasets.DatasetDict(train=ds.with_format("torch")).save_to_disk(ds_path)
    rows = []
    for c in range(C):
        for p in range(bank["cell_off"][c], bank["cell_off"][c + 1]):
            idx = bank["member_idx"][bank["member_off"][p]: bank["member_off"][p + 1]]
            rows.append(dict(geocell_idx=c, cluster=int(p - bank["cell_off"][c]), lng=float(bank["proto_lnglat"][p, 0]),
                             lat=float(bank["proto_lnglat"][p, 1]), count=int(len(idx)), indices=json.dumps([int(i) for i in idx])))
    pd.DataFrame(rows).to_csv(csv_path, index=False)

    class _Serial(cf.Executor):  # ProcessPoolExecutor(max_workers=64) stand-in: same calls, in-process
        def __init__(self, *a, **kw):
            pass

        def submit(self, fn, *a, **kw):
            f = cf.Future()
            try:
                f.set_result(fn(*a, **kw))
            except Exception as ex:  # noqa: BLE001
                f.set_exception(ex)
            return f

    real_pool = pr.ProcessPoolExecutor
    pr.ProcessPoolExecutor = _Serial
    try:
        ref = pr.ProtoRefiner(topk=topk, max_refinement=maxref, temperature=T, proto_path=csv_path, dataset_path=ds_path)
    finally:
        pr.ProcessPoolExecutor = real_pool
    ref.eval()
    ref.dataset = datasets.DatasetDict(train=ref.dataset["train"].with_format("torch"))
    # pack the bank FROM THE REFERENCE-BUILT prototypes (validates the CSR packing + prototype means)
    cells = []
    for c in range(C):
        d = ref.protos[c] if c < len(ref.protos) else None
        if d is None:
            cells.append(None)
            continue
        cells.append([dict(lng=float(r["lng"]), lat=float(r["lat"]), count=int(r["count"]),
                           indices=[int(i) for i in r["indices"]], embedding=r["embedding"].numpy()) for r in
                      (d[i] for i in range(len(d)))])
    while len(cells) < C:
        cells.append(None)
    from oracle.refiner import pack_bank
    data_emb = torch.stack([x for x in ref.dataset["train"]["embedding"]]).mean(1).numpy() if False else views.mean(axis=1)
    # the reference averages views with torch (.mean(dim=1), :250-251): reproduce with torch for bit-equality
    data_emb = torch.from_numpy(views).mean(dim=1).numpy()
    packed = pack_bank(cells, data_emb, bank["data_lnglat"])
    ref.protos = [None if d is None else _DuckProtos(d) for d in ref.protos] + [None] * (C - len(ref.protos))

    cand, probs = synthetic.synthetic_candidates(B, kc, C, seed=seed + 2)
    q = synthetic.synthetic_queries(packed, cand, views=4, seed=seed + 3)
    init = synthetic.synthetic_geocells(B, seed=seed + 4)
    qt, candt, probst = torch.from_numpy(q), torch.from_numpy(cand), torch.from_numpy(probs)
    with rs.device_redirect(), torch.no_grad():
        ref.max_refinement = 1e12
        _, ll0, _ = ref(qt, initial_preds=torch.from_numpy(init), candidate_cells=candt, candidate_probs=probst)
        init[::2] = ll0[::2].double().numpy() + 0.25      # both outcomes of the max-refinement gate
        ref.max_refinement = maxref
        _, ll, cell = ref(qt, initial_preds=torch.from_numpy(init), candidate_cells=candt, candidate_probs=probst)
        _, ll_np, cell_np = ref(qt, initial_preds=torch.from_numpy(init), candidate_cells=candt, candidate_probs=None)
    if name is not None:
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"),
                            meta=json.dumps(dict(C=C, P=P, D=D, B=B, kc=kc, topk=topk, members=members, T=T, maxref=maxref, seed=seed)),
                            emb=q, init=init, cand=cand, probs=probs, preds_LLH=ll.numpy(), preds_geocell=cell.numpy(),
                            preds_LLH_noprob=ll_np.numpy(), preds_geocell_noprob=cell_np.numpy(), **{f"bank_{k}": v for k, v in packed.items()})
    return ref, packed


def _reference_function(path, fn_name, namespace):
    """The UNMODIFIED source of one function of a reference file whose module cannot be imported here (accelerate /
    tensorboard are not installed), executed in `namespace` (stand-ins for the names the body uses from those imports)."""
    import ast
    src = open(os.path.join("/root/reference", path)).read()
    node = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == fn_name)
    exec(compile(ast.Module(body=[node], type_ignores=[]), os.path.join("/root/reference", path), "exec"), namespace)
    return namespace[fn_name]


def loops_fixture(tmp):
    """The callers of the hot path: the bodies of `evaluate_model` (training/train_eval_loop.py:35-161) and
    `compute_embeddings` (preprocessing/embed.py:16-43) run as they are, over the unmodified SuperGuessr / ProtoRefiner /
    CLIPEmbedding modules — pins batch order, ragged last batch, what is concatenated and what reaches `metrics` / disk."""
    import logging
    from typing import Any, Callable
    from torch.utils.data import DataLoader, Dataset
    from models.super_guessr import SuperGuessr
    from models.clip_embedder import CLIPEmbedding
    C, D, N, bs, topk = 1000, 128, 11, 4, 5
    ref, packed = refiner_fixture(tmp, None, C=C, P=1500, D=D, B=8, kc=10, topk=topk, members=1.5, T=1.6, maxref=1e6, seed=90)
    W, b = head_weights(C, D, seed=91)
    g = torch.Generator().manual_seed(92)
    cand, _ = synthetic.synthetic_candidates(N, topk, C, seed=93)
    emb = torch.from_numpy(synthetic.synthetic_queries(packed, cand, views=4, seed=94))          # [N, 4, D]
    # make the head prefer each sample's candidate cells, so that retrieval works on non-empty cells
    labels = synthetic.synthetic_geocells(N, 95)
    labels_clf = cand[:, 0].copy()

    class DS(Dataset):
        def __len__(self):
            return N

        def __getitem__(self, i):
            if isinstance(i, str):
                return {"labels": labels, "labels_clf": labels_clf}[i]
            return dict(embedding=emb[i], labels=torch.tensor(labels[i]), labels_clf=torch.tensor(labels_clf[i]))

    class Writer:
        def __init__(self):
            self.scalars = {}

        def add_scalar(self, k, v, step):
            self.scalars[k] = float(v)

    captured = {}

    def metrics(results):
        captured["results"] = results
        return {"Geocell_accuracy": float((results[1] == results[7]).mean())}

    def loader(ds, batch_size, **kw):
        return DataLoader(ds, batch_size, shuffle=kw.get("shuffle", False), num_workers=0)

    ns = dict(nn=torch.nn, Dataset=Dataset, Callable=Callable, Any=Any, TrainingArguments=object, ProtoRefiner=object,
              SummaryWriter=Writer, DataLoader=loader, tqdm=lambda x, **kw: x, torch=torch, np=np,
              logger=logging.getLogger("reference"), BenchmarkDataset=type("BenchmarkDataset", (), {}))
    evaluate_model = _reference_function("training/train_eval_loop.py", "evaluate_model", ns)
    with rs.chdir(tmp):
        sg = SuperGuessr(None, panorama=True, num_candidates=topk, embed_dim=D).eval()
    with torch.no_grad():
        sg.cell_layer.weight.copy_(W)
        sg.cell_layer.bias.copy_(b)
        for i in range(N):                       # the candidate cells of sample i score highest for its embedding
            sg.cell_layer.weight[cand[i]] += emb[i].mean(0) * (1.0 + 0.01 * torch.arange(topk))[:, None]

    class Args:
        per_device_eval_batch_size = bs

    out = {}
    for tag, refiner in (("refined", ref), ("plain", None)):
        w = Writer()
        with rs.device_redirect():
            ret = evaluate_model(sg, DS(), metrics, Args(), refiner=refiner, writer=w)
        r = captured["results"]
        out.update({f"eval_{tag}_preds": r[0], f"eval_{tag}_preds_geocell": r[1], f"eval_{tag}_top5": r[5],
                    f"eval_{tag}_return": np.float64(ret), f"eval_{tag}_loss_logged": np.float64(w.scalars["Loss/val"])})
        assert r[2] is None and r[3] is None and r[4] is None and np.array_equal(r[6], labels) and np.array_equal(r[7], labels_clf)

    # ---- compute_embeddings over the unmodified CLIPEmbedding (tiny random-init HF tower)
    dims = VitDims(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2)
    sd = synthetic.random_vit_state_dict(dims, seed=96, std=0.05)
    ce = object.__new__(CLIPEmbedding)
    torch.nn.Module.__init__(ce)
    ce.clip_model = hf_model(dims, sd)
    ce.device, ce.panorama = "cpu", False
    n_img, ebs = 9, 3                            # equal batches: np.save of the reference's LIST of batches needs them
    px = torch.randn(n_img, 3, 56, 56, generator=torch.Generator().manual_seed(97))
    order = torch.tensor([4, 0, 7, 2, 8, 1, 6, 3, 5])    # dataset order != index order: the consumer sorts by the saved index

    class EDS(Dataset):
        def __len__(self):
            return n_img

        def __getitem__(self, i):
            return px[order[i]], order[i]

    class Acc:
        is_local_main_process = True

        def gather(self, x):
            return x

    ens = dict(np=np, tqdm=lambda x, **kw: x, logger=logging.getLogger("reference"), AutoModel=object, DataLoader=DataLoader,
               Accelerator=object, enumerate=enumerate)
    compute_embeddings = _reference_function("preprocessing/embed.py", "compute_embeddings", ens)
    os.makedirs(os.path.join(tmp, "data", "landmark_embeddings"), exist_ok=True)
    with rs.chdir(tmp), torch.no_grad():
        compute_embeddings("golden", ce, DataLoader(EDS(), ebs, shuffle=False), Acc())
    saved = np.load(os.path.join(tmp, "data", "landmark_embeddings", "golden.npy"))
    saved_idx = np.load(os.path.join(tmp, "data", "landmark_embeddings", "golden_indices.npy"))
    # what preprocessing/dataset_preprocessing.py:296-300 makes of the two files
    arg = np.argsort(saved_idx.flatten()[:n_img])
    consumer = saved.reshape((-1, dims.hidden))[arg]
    out.update(embed_saved=saved, embed_saved_indices=saved_idx, embed_consumer_rows=consumer)
    golden.save("loops", dict(emb=emb.numpy(), labels=labels, labels_clf=labels_clf, cand=cand,
                              head_w=sg.cell_layer.weight.detach().numpy(), head_b=sg.cell_layer.bias.detach().numpy(),
                              centroids=sg.lla_geocells.detach().numpy(), **{f"bank_{k}": v for k, v in packed.items()}, **out),
                dict(C=C, D=D, N=N, bs=bs, topk=topk, head_seed=91, bank=dict(C=C, P=1500, D=D, members=1.5, seed=90, empty_cells=3),
                     embed=dict(n_img=n_img, bs=ebs, sd_seed=96, px_seed=97, std=0.05, order=order.tolist(),
                                dims=dict(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2))))


def tower_train_fixtures(tmp):
    small = VitDims(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2)
    train_tower_fixture(tmp, "train_tower_small", small, n_views=6, sd_seed=43, px_seed=44, std=0.05, stride=7)
    mid = VitDims(image_size=224, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2)
    train_tower_fixture(tmp, "train_tower_mid", mid, n_views=3, sd_seed=45, px_seed=46, std=0.05, stride=7)


def main():
    os.makedirs(OUT, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="pigeon_golden_")
    os.makedirs(os.path.join(tmp, "data"))
    cells = synthetic.synthetic_geocells(1000, 0)
    pd.DataFrame({"lng": cells[:, 0], "lat": cells[:, 1]}).to_csv(os.path.join(tmp, "data", "geocells_2203.csv"), index=False)
    rs.install()
    torch.set_num_threads(os.cpu_count())
    only = set(sys.argv[1:])          # e.g. `python -m oracle.make_golden train` regenerates one family
    if only:
        if "train" in only:
            train_fixture(tmp)
        if "preprocess" in only:
            preprocess_fixture()
        if "tower" in only:
            tower_train_fixtures(tmp)
        if "loops" in only:
            loops_fixture(tmp)
        return
    geo_fixture()
    head_fixture(tmp)
    train_fixture(tmp)
    preprocess_fixture()
    tower_train_fixtures(tmp)
    small = VitDims(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2)
    vit_fixture(tmp, "vit_small", small, sd_seed=41, n_samples=3, panorama=True, px_seed=42, std=0.05)
    vit_fixture(tmp, "vit_large_single", VitDims(), sd_seed=0, n_samples=1, panorama=False, px_seed=1, std=0.02)
    vit_fixture(tmp, "vit_large_pano", VitDims(), sd_seed=0, n_samples=2, panorama=True, px_seed=2, std=0.02)
    refiner_fixture(tmp, "refiner_count1", C=40, P=400, D=128, B=48, kc=10, topk=5, members=0.0, T=1.6, maxref=1000, seed=50)
    refiner_fixture(tmp, "refiner_members", C=30, P=200, D=128, B=40, kc=12, topk=12, members=5.0, T=0.6, maxref=100000, seed=60)
    loops_fixture(tmp)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
