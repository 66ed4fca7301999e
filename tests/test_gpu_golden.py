"""Parity of the PUBLIC modules (pigeon_b200.SuperGuessr / CLIPEmbedding / ProtoRefiner -> C ABI -> sm_100a
kernels) against tests/golden/*.npz, i.e. against outputs of the UNMODIFIED reference modules on the same inputs.

Tolerances: embeddings / logits-derived floats <= 1e-3 relative (BASELINE.json north_star); integer and index
outputs exact wherever the reference's own decision margin exceeds that floating-point budget."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 1e-3


def load(name):
    z = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
    return z, (json.loads(str(z["meta"])) if "meta" in z.files else {})


def head_weights(C, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(C, D, generator=g) * 0.03, torch.randn(C, generator=g) * 0.01


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _tower(meta, cuda):
    from pigeon_b200 import CLIPVisionTower, VitDims, synthetic
    dims = VitDims(**meta["dims"])
    tower = CLIPVisionTower(dims)
    sd = synthetic.random_vit_state_dict(dims, seed=meta["sd_seed"], std=meta["std"])
    missing, unexpected = tower.load_state_dict(sd, strict=True), None
    return tower, dims


def _pixels(meta, dims):
    g = torch.Generator().manual_seed(meta["px_seed"])
    ch = 12 if meta["panorama"] else 3
    return torch.randn(meta["n_samples"], ch, dims.image_size, dims.image_size, generator=g)


@pytest.mark.parametrize("name", ["vit_large_single", "vit_large_pano"])
def test_superguessr_pixels_to_geocells(cuda, name):
    """cfg1 of BASELINE.json (single 336x336 image, random-init ViT-L/14, 1000 geocells) and its 4-view variant."""
    from pigeon_b200 import SuperGuessr
    z, meta = load(name)
    tower, dims = _tower(meta, cuda)
    W, b = head_weights(meta["C"], dims.hidden, meta["w_seed"])
    sg = SuperGuessr(tower, panorama=meta["panorama"], freeze_base=True, num_candidates=50, geocells=z["centroids"])
    with torch.no_grad():
        sg.cell_layer.weight.copy_(W)
        sg.cell_layer.bias.copy_(b)
    sg.to(cuda).eval()
    px = _pixels(meta, dims)                                            # host tensor: the module moves it (H2D)
    out = sg(pixel_values=px, labels=torch.tensor(z["labels"]), labels_clf=torch.tensor(z["labels_clf"]))
    torch.cuda.synchronize()
    emb = out.embedding.cpu().numpy()
    assert emb.shape == z["embedding"].shape
    e = _rel(emb, z["embedding"])
    print(f"{name}: embedding rel-L2 vs reference = {e:.3e}")
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, "parity.log"), "a") as f:
            f.write(f"{name}: SuperGuessr(pixels) embedding rel-L2 vs UNMODIFIED reference golden = {e:.3e}; "
                    f"top-1 geocell identical; loss rel err {abs(out.loss.item() - float(z['loss'])) / float(z['loss']):.2e}\n")
    assert e < REL_TOL, e
    assert np.abs(emb - z["embedding"]).max() / np.abs(z["embedding"]).max() < 5e-3
    # top-1 geocell identical (the fixtures' top-1/top-2 probability margins are > 10x the error budget)
    margin = (z["topk_val"][:, 0] - z["topk_val"][:, 1]) / z["topk_val"][:, 0]
    assert (margin > 20 * REL_TOL).all(), margin
    assert np.array_equal(out.preds_geocell.cpu().numpy(), z["preds_geocell"])
    assert np.array_equal(out.preds_LLH.cpu().numpy(), z["preds_LLH"]) and out.preds_LLH.dtype == torch.float64
    np.testing.assert_allclose(out.top5_geocells.values.cpu().numpy(), z["topk_val"], rtol=5 * REL_TOL)
    np.testing.assert_allclose(out.loss.item(), z["loss"], rtol=REL_TOL)
    # candidate ORDER: identical down to the first pair of neighbours whose probabilities the reference itself separates by
    # less than the tolerance on the values (5 x 1e-3; deep in the top-50 the margins vanish); the top-5 the refiner
    # consumes must be inside
    idx, val = out.top5_geocells.indices.cpu().numpy(), z["topk_val"]
    gaps = (val[:, :-1] - val[:, 1:]) / val[:, :-1]
    safe = np.concatenate([np.ones_like(val[:, :1], dtype=bool), np.cumprod(gaps > 5 * REL_TOL, axis=1).astype(bool)], axis=1)
    assert safe[:, :5].all(), "fixture: the top-5 candidates must be separated by more than the tolerance"
    assert np.array_equal(idx[safe], z["topk_idx"][safe])
    assert set(map(tuple, np.sort(idx, 1))) == set(map(tuple, np.sort(z["topk_idx"], 1))) or (idx == z["topk_idx"]).mean() > 0.9


def test_clip_embedding_small_and_large(cuda):
    from pigeon_b200 import CLIPEmbedding
    for name in ("vit_small", "vit_large_single"):
        z, meta = load(name)
        tower, dims = _tower(meta, cuda)
        ce = CLIPEmbedding("unused", device="cuda", clip_model=tower)
        views = _pixels(meta, dims).reshape(-1, 3, dims.image_size, dims.image_size)
        emb = ce(views).cpu().numpy()
        assert emb.shape == z["clip_embedding"].shape
        assert _rel(emb, z["clip_embedding"]) < REL_TOL, (name, _rel(emb, z["clip_embedding"]))


@pytest.mark.parametrize("name,panorama,k,smooth,emb_key", [("pano", True, 50, False, "emb4"),
                                                           ("pano_smooth", True, 5, True, "emb4"),
                                                           ("single", False, 5, False, "emb1"),
                                                           ("single_from4", False, 7, False, "emb4")])
def test_superguessr_on_embeddings(cuda, name, panorama, k, smooth, emb_key):
    """`-b` not given: base_model=None, the head runs on precomputed embeddings (evaluate.py:36)."""
    from pigeon_b200 import SuperGuessr
    z, meta = load("head")
    W, b = head_weights(meta["C"], meta["D"], meta["w_seed"])
    sg = SuperGuessr(None, panorama=panorama, num_candidates=k, should_smooth_labels=smooth, geocells=z["centroids"])
    with torch.no_grad():
        sg.cell_layer.weight.copy_(W)
        sg.cell_layer.bias.copy_(b)
    sg.to(cuda).eval()
    out = sg(embedding=torch.tensor(z[emb_key]), labels=torch.tensor(z["labels"]), labels_clf=torch.tensor(z["labels_clf"]))
    assert np.array_equal(out.preds_geocell.cpu().numpy(), z[f"{name}_preds_geocell"])
    assert np.array_equal(out.preds_LLH.cpu().numpy(), z[f"{name}_preds_LLH"])
    assert np.array_equal(out.top5_geocells.indices.cpu().numpy(), z[f"{name}_topk_idx"])
    np.testing.assert_allclose(out.top5_geocells.values.cpu().numpy(), z[f"{name}_topk_val"], rtol=2e-5)
    np.testing.assert_allclose(out.loss.item(), z[f"{name}_loss"], rtol=2e-5)
    assert out.loss.dtype == torch.from_numpy(z[f"{name}_loss"]).dtype
    assert out.embedding.shape == z[emb_key].shape                      # un-averaged (B,4,D) in panorama mode (quirk 10)


def test_superguessr_serving_tuple_and_errors(cuda):
    from pigeon_b200 import SuperGuessr
    z, meta = load("head")
    sg = SuperGuessr(None, panorama=True, serving=True, num_candidates=5, geocells=z["centroids"]).to(cuda).eval()
    pred, topk, emb = sg(embedding=torch.tensor(z["emb4"]))
    assert pred.shape == (6, 2) and topk.values.shape == (6, 5) and topk.indices.dtype == torch.int64
    sg2 = SuperGuessr(None, panorama=True, num_candidates=5, geocells=z["centroids"]).to(cuda).eval()
    with pytest.raises(AttributeError):                                  # quirk 9: labels_clf required unless serving
        sg2(embedding=torch.tensor(z["emb4"]))
    with pytest.raises(AssertionError):
        sg2(pixel_values=None, embedding=None)


@pytest.mark.parametrize("name", ["refiner_count1", "refiner_members"])
def test_protorefiner_matches_reference(cuda, name):
    from pigeon_b200 import ProtoRefiner
    z, meta = load(name)
    bank = {k[5:]: z[k] for k in z.files if k.startswith("bank_")}
    ref = ProtoRefiner(topk=meta["topk"], max_refinement=meta["maxref"], temperature=meta["T"], protos=bank).eval()
    args = dict(initial_preds=torch.tensor(z["init"]), candidate_cells=torch.tensor(z["cand"]))
    loss, ll, cell = ref(torch.tensor(z["emb"]), candidate_probs=torch.tensor(z["probs"]), **args)
    assert loss is None and ll.dtype == torch.float32 and cell.dtype == torch.int64
    assert np.array_equal(cell.cpu().numpy(), z["preds_geocell"])
    assert np.array_equal(ll.cpu().numpy(), z["preds_LLH"])
    _, ll, cell = ref(torch.tensor(z["emb"]), candidate_probs=None, **args)
    assert np.array_equal(cell.cpu().numpy(), z["preds_geocell_noprob"])
    assert np.array_equal(ll.cpu().numpy(), z["preds_LLH_noprob"])
    with pytest.raises(AssertionError):                                  # proto_refiner.py:135-137
        ProtoRefiner(topk=99, protos=bank)(torch.tensor(z["emb"]), candidate_probs=None, **args)


def test_evaluate_model_loop_matches_direct_calls(cuda):
    """loops.evaluate_model (mirror of training/train_eval_loop.py:35-161) == per-batch direct calls."""
    from pigeon_b200 import ProtoRefiner, SuperGuessr
    from pigeon_b200.loops import evaluate_model
    z, meta = load("refiner_count1")
    zh, mh = load("head")
    bank = {k[5:]: z[k] for k in z.files if k.startswith("bank_")}
    D, C = bank["proto_emb"].shape[1], int(bank["cell_off"].shape[0]) - 1
    g = torch.Generator().manual_seed(5)
    n = 37
    emb = torch.randn(n, 4, D, generator=g) * 0.3
    labels = torch.rand(n, 2, generator=g, dtype=torch.float64) * 90
    labels_clf = torch.randint(0, C, (n,), generator=g)

    class DS(torch.utils.data.Dataset):
        def __len__(self):
            return n

        def __getitem__(self, i):
            if isinstance(i, str):
                return {"labels": labels.numpy(), "labels_clf": labels_clf.numpy()}[i]
            return dict(embedding=emb[i], labels=labels[i], labels_clf=labels_clf[i])

    cells = np.stack([np.linspace(-170, 170, C), np.linspace(-80, 80, C)], 1)
    sg = SuperGuessr(None, panorama=True, num_candidates=10, embed_dim=D, geocells=cells).to(cuda).eval()
    ref = ProtoRefiner(topk=5, max_refinement=1e6, temperature=1.6, protos=bank).eval()

    class Args:
        per_device_eval_batch_size = 16

    res = evaluate_model(sg, DS(), None, Args(), ref)
    out = sg(embedding=emb, labels=labels, labels_clf=labels_clf)
    _, ll, cell = ref(out.embedding, initial_preds=out.preds_LLH, candidate_cells=out.top5_geocells.indices,
                      candidate_probs=out.top5_geocells.values)
    assert np.array_equal(res["preds"], ll.cpu().numpy())
    assert np.array_equal(res["preds_geocell"], out.preds_geocell.cpu().numpy())
    assert np.array_equal(res["top_geocells"], out.top5_geocells.indices.cpu().numpy())
    np.testing.assert_allclose(res["loss"], out.loss.item(), rtol=1e-5)


def test_evaluate_model_loop_matches_reference_loop_golden(cuda):
    """loops.evaluate_model against tests/golden/loops.npz: the UNMODIFIED body of the reference's `evaluate_model`
    (training/train_eval_loop.py:35-161) run over the unmodified SuperGuessr + ProtoRefiner on an 11-sample dataset in
    batches of 4 (ragged last batch).  Pins batch order, what is concatenated, what `metrics` receives and the return."""
    from pigeon_b200 import ProtoRefiner, SuperGuessr
    from pigeon_b200.loops import evaluate_model
    from oracle import golden
    z, meta = golden.load("loops")
    N, bs, topk, D = meta["N"], meta["bs"], meta["topk"], meta["D"]
    emb, labels, labels_clf = torch.tensor(z["emb"]), z["labels"], z["labels_clf"]
    bank = {k[5:]: z[k] for k in z if k.startswith("bank_")}
    sg = SuperGuessr(None, panorama=True, num_candidates=topk, embed_dim=D, geocells=z["centroids"])
    with torch.no_grad():
        sg.cell_layer.weight.copy_(torch.tensor(z["head_w"]))
        sg.cell_layer.bias.copy_(torch.tensor(z["head_b"]))
    sg.to(cuda).eval()

    class DS(torch.utils.data.Dataset):
        def __len__(self):
            return N

        def __getitem__(self, i):
            if isinstance(i, str):
                return {"labels": labels, "labels_clf": labels_clf}[i]
            return dict(embedding=emb[i], labels=torch.tensor(labels[i]), labels_clf=torch.tensor(labels_clf[i]))

    class Args:
        per_device_eval_batch_size = bs

    captured = {}

    def metrics(results):
        captured["r"] = results
        return {"Geocell_accuracy": float((results[1] == results[7]).mean())}

    for tag, refiner in (("refined", ProtoRefiner(topk=topk, max_refinement=1e6, temperature=1.6, protos=bank).eval()), ("plain", None)):
        ret = evaluate_model(sg, DS(), metrics, Args(), refiner)
        r = captured["r"]
        assert len(r) == 11 and r[2] is None and r[3] is None and r[4] is None and r[8] is None
        assert np.array_equal(r[1], z[f"eval_{tag}_preds_geocell"])
        assert np.array_equal(r[5], z[f"eval_{tag}_top5"])
        assert np.array_equal(r[0], z[f"eval_{tag}_preds"]) and r[0].dtype == z[f"eval_{tag}_preds"].dtype
        assert np.array_equal(r[6], labels) and np.array_equal(r[7], labels_clf)
        assert ret == float(z[f"eval_{tag}_return"])
    # the loss the reference logs is sum_batches(loss_b * len(data)) / len(dataset) with len(data) = the number of COLUMNS of
    # the batch dict (3), train_eval_loop.py:81 — reproduce that figure from this path's per-batch losses
    logged = 0.0
    for lo in range(0, N, bs):
        o = sg(embedding=emb[lo:lo + bs], labels=torch.tensor(labels[lo:lo + bs]), labels_clf=torch.tensor(labels_clf[lo:lo + bs]))
        logged += float(o.loss) * 3
    np.testing.assert_allclose(logged / N, float(z["eval_refined_loss_logged"]), rtol=2e-5)


def test_compute_embeddings_matches_reference_loop_golden(cuda, tmp_path):
    """loops.compute_embeddings against the UNMODIFIED body of the reference's (preprocessing/embed.py:16-43) over the
    unmodified CLIPEmbedding: what lands on disk must give the reference's consumer (dataset_preprocessing.py:296-300:
    flatten the indices, reshape the embeddings to rows, sort by index) the same rows."""
    from pigeon_b200 import CLIPEmbedding, CLIPVisionTower, VitDims, synthetic
    from pigeon_b200.loops import compute_embeddings
    z, meta = load("loops")
    e = meta["embed"]
    dims = VitDims(**e["dims"])
    tower = CLIPVisionTower(dims)
    tower.load_state_dict(synthetic.random_vit_state_dict(dims, seed=e["sd_seed"], std=e["std"]))
    ce = CLIPEmbedding("unused", device="cuda", clip_model=tower.to(cuda))
    px = torch.randn(e["n_img"], 3, dims.image_size, dims.image_size, generator=torch.Generator().manual_seed(e["px_seed"]))
    order = torch.tensor(e["order"])

    class EDS(torch.utils.data.Dataset):
        def __len__(self):
            return e["n_img"]

        def __getitem__(self, i):
            return px[order[i]], order[i]

    compute_embeddings("golden", ce, torch.utils.data.DataLoader(EDS(), e["bs"], shuffle=False), save_dir=str(tmp_path))
    saved, idx = np.load(tmp_path / "golden.npy"), np.load(tmp_path / "golden_indices.npy")
    assert np.array_equal(idx.flatten(), z["embed_saved_indices"].flatten())          # same batch / row order on disk
    arg = np.argsort(idx.flatten()[: e["n_img"]])
    rows = saved.reshape((-1, dims.hidden))[arg]
    assert rows.shape == z["embed_consumer_rows"].shape
    assert _rel(rows, z["embed_consumer_rows"]) < REL_TOL
    assert _rel(saved.reshape(-1, dims.hidden), z["embed_saved"].reshape(-1, dims.hidden)) < REL_TOL


def test_bank_builder_matches_reference_prototypes(cuda):
    """pg_bank_build (GPU segmented mean) == the prototype embeddings the reference constructor computed
    (`_compute_protos_for_cell`, proto_refiner.py:359-378; packed into the golden by oracle/make_golden.py)."""
    from pigeon_b200 import bank as bank_mod
    z, meta = load("refiner_members")
    off, idx = z["bank_member_off"], z["bank_member_idx"]
    P = len(off) - 1
    cells = np.searchsorted(z["bank_cell_off"], np.arange(P), side="right") - 1
    indices = [idx[off[p]:off[p + 1]].tolist() for p in range(P)]
    # 4-view training embeddings whose view mean is the stored data_emb (two +/- perturbations cancel exactly in fp32)
    e = torch.from_numpy(z["bank_data_emb"])
    d1 = torch.randn(e.shape, generator=torch.Generator().manual_seed(3)) * 0.01
    views = torch.stack([e + d1, e - d1, e + 0.5 * d1, e - 0.5 * d1], dim=1)
    b = bank_mod.bank_from_arrays(cells, z["bank_proto_lnglat"], indices, views, z["bank_data_lnglat"],
                                  num_cells=len(z["bank_cell_off"]) - 1, device=cuda)
    assert np.array_equal(b["cell_off"], z["bank_cell_off"]) and np.array_equal(b["member_idx"], idx)
    np.testing.assert_allclose(b["data_emb"], z["bank_data_emb"], rtol=2e-6, atol=2e-7)
    np.testing.assert_allclose(b["proto_emb"], z["bank_proto_emb"], rtol=1e-5, atol=1e-6)
    assert np.array_equal(b["proto_count"], z["bank_proto_count"])


def test_checkpoint_round_trip_through_load_state(cuda, tmp_path):
    """`torch.save(model.state_dict())` (train_eval_loop.py:238) -> a fresh model -> `load_state(path)`
    (super_guessr.py:222-238, evaluate.py:45-46): same predictions bit for bit, unknown keys reported and skipped."""
    from pigeon_b200 import CLIPVisionTower, SuperGuessr, VitDims, synthetic
    dims = VitDims(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=2)
    cells = synthetic.synthetic_geocells(40, 0)

    def build(seed):
        tower = CLIPVisionTower(dims)
        tower.load_state_dict(synthetic.random_vit_state_dict(dims, seed=seed, std=0.05), strict=True)
        return SuperGuessr(tower, panorama=True, freeze_base=True, num_candidates=5, geocells=cells).to(cuda).eval()

    a, b = build(1), build(2)
    with torch.no_grad():
        a.cell_layer.weight.normal_(0, 0.05)
    px = torch.randn(3, 12, 56, 56, generator=torch.Generator().manual_seed(3)).to(cuda)
    lab = torch.tensor([1, 2, 3])
    oa = a(pixel_values=px, labels_clf=lab)
    ob = b(pixel_values=px, labels_clf=lab)
    assert not torch.equal(oa.embedding, ob.embedding)
    sd = a.state_dict()
    sd["not_a_parameter"] = torch.zeros(1)
    path = tmp_path / "head.model"
    torch.save(sd, path)
    b.load_state(str(path))                                  # prints the unknown key, copies the rest by name
    ob = b(pixel_values=px, labels_clf=lab)
    assert torch.equal(oa.embedding, ob.embedding) and torch.equal(oa.preds_geocell, ob.preds_geocell)
    assert torch.equal(oa.top5_geocells.values, ob.top5_geocells.values) and float(oa.loss) == float(ob.loss)


def test_multi_rank_outputs_equal_single_rank_bit_for_bit(cuda):
    """SURVEY.md §4-iii on NCCL: world-size-2 gathered outputs (replicated and cell-sharded bank) == single-rank outputs."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29579", os.path.join(root, "tools", "ddp_infer_check.py")],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
