"""Fine-tune step, head-only part (N1): pg_head_loss_grad / pg_head_backward / pg_adamw_step and the `train_model`
loop against the CPU oracle (oracle/train.py) and against tests/golden/train_head.npz, which holds what the UNMODIFIED
reference module + torch autograd + torch.optim.AdamW produced for the same micro-batches (oracle/make_golden.py)."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def G():
    from oracle import golden
    return golden.load("train_head")[0]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_loss_grad_matches_oracle(cuda, G, mode):
    from oracle import train as otrain
    from pigeon_b200._lib import check, current_stream_ptr, load, ptr
    lib = load()
    Cc, B = 1000, 8
    g = torch.Generator().manual_seed(mode)
    logits = (torch.randn(B, Cc, generator=g) * 3).to(cuda)
    cells = torch.tensor(G["centroids"], device=cuda)
    labels = torch.tensor(G["labels"][1], device=cuda)
    idx = torch.tensor(G["labels_clf"][1], device=cuda)
    soft = torch.rand(B, Cc, generator=g).to(cuda) * (torch.rand(B, Cc, generator=g).to(cuda) < 0.01)
    per = torch.empty(B, dtype=torch.float64, device=cuda)
    out = torch.empty(1, dtype=torch.float64, device=cuda)
    dl = torch.empty(B, Cc, dtype=torch.float32, device=cuda)
    check(lib.pg_head_loss_grad(ptr(logits), B, Cc, mode, ptr(idx) if mode == 0 else None, ptr(soft) if mode == 1 else None,
                                ptr(labels) if mode == 2 else None, ptr(cells) if mode == 2 else None, 65.0, 1.0, ptr(per),
                                ptr(out), ptr(dl), current_stream_ptr()), "pg_head_loss_grad")
    # oracle: identity "head" so that logits are the given ones
    x = logits.double().cpu().numpy()
    t = otrain._targets(Cc, labels.cpu().numpy(), soft.cpu().numpy() if mode == 1 else idx.cpu().numpy(),
                        G["centroids"], smooth=(mode == 2))
    m = x.max(1, keepdims=True)
    logp = x - (m + np.log(np.exp(x - m).sum(1, keepdims=True)))
    ref_loss = -(t * logp).sum() / B
    ref_g = (np.exp(logp) * t.sum(1, keepdims=True) - t) / B
    np.testing.assert_allclose(out.item(), ref_loss, rtol=1e-12)
    assert np.abs(dl.cpu().numpy() - ref_g).max() <= 1e-7 * max(1.0, np.abs(ref_g).max()) + 6e-8 * np.abs(ref_g).max()
    # and torch autograd on the same logits (soft-target CrossEntropyLoss, super_guessr.py:474)
    xl = logits.detach().cpu().double().requires_grad_(True)
    torch.nn.functional.cross_entropy(xl, torch.tensor(t)).backward()
    assert np.abs(dl.cpu().numpy() - xl.grad.numpy()).max() <= 2e-7 * np.abs(ref_g).max()


def test_loss_with_label_out_of_range_is_nan_not_a_wild_read(cuda):
    """include/pigeon_b200.h (pg_head_loss): a class index outside [0, C) poisons the loss and zeroes that gradient row."""
    from pigeon_b200._lib import check, current_stream_ptr, load, ptr
    lib = load()
    Cc, B = 130, 4
    logits = torch.randn(B, Cc, generator=torch.Generator().manual_seed(3)).to(cuda)
    idx = torch.tensor([5, Cc, -100, 7], dtype=torch.int64, device=cuda)
    per = torch.empty(B, dtype=torch.float64, device=cuda)
    out = torch.empty(1, dtype=torch.float64, device=cuda)
    dl = torch.full((B, Cc), 9.0, dtype=torch.float32, device=cuda)
    check(lib.pg_head_loss_grad(ptr(logits), B, Cc, 0, ptr(idx), None, None, None, 65.0, 1.0, ptr(per), ptr(out), ptr(dl),
                                current_stream_ptr()), "pg_head_loss_grad")
    torch.cuda.synchronize()
    assert torch.isnan(out).item()
    assert torch.isnan(per[1]).item() and torch.isnan(per[2]).item() and torch.isfinite(per[[0, 3]]).all()
    assert (dl[1] == 0).all() and (dl[2] == 0).all()
    ref = torch.nn.functional.cross_entropy(logits[[0, 3]].double().cpu(), idx[[0, 3]].cpu(), reduction="none")
    np.testing.assert_allclose(per[[0, 3]].cpu().numpy(), ref.numpy(), rtol=1e-12)


@pytest.mark.parametrize("B,Cc,D,acc", [(8, 1000, 128, 0), (37, 2076, 1024, 1), (256, 130, 768, 0)])
def test_head_backward_matches_fp64(cuda, B, Cc, D, acc):
    from pigeon_b200._lib import check, current_stream_ptr, load, ptr
    lib = load()
    g = torch.Generator().manual_seed(B)
    dl = (torch.randn(B, Cc, generator=g) * 0.01).to(cuda)
    x = (torch.randn(B, D, generator=g) * 0.5).to(cuda)
    w = (torch.randn(Cc, D, generator=g) * 0.03).to(cuda)
    dw0 = torch.randn(Cc, D, generator=g).to(cuda) * 0.01
    db0 = torch.randn(Cc, generator=g).to(cuda) * 0.01
    dw, db = dw0.clone(), db0.clone()
    dx = torch.empty(B, D, device=cuda)
    check(lib.pg_head_backward(ptr(dl), ptr(x), ptr(w), B, Cc, D, acc, ptr(dw), ptr(db), ptr(dx), current_stream_ptr()),
          "pg_head_backward")
    rw = dl.double().t() @ x.double() + (dw0.double() if acc else 0)
    rb = dl.double().sum(0) + (db0.double() if acc else 0)
    rx = dl.double() @ w.double()
    for got, ref in ((dw, rw), (db, rb), (dx, rx)):
        assert (got.double() - ref).abs().max().item() <= 2e-6 * ref.abs().max().item()


def test_adamw_matches_torch_and_oracle(cuda):
    from oracle import train as otrain
    from pigeon_b200.training import AdamW
    g = torch.Generator().manual_seed(9)
    p0 = torch.randn(1000 * 128 + 3, generator=g) * 0.05
    p_t = torch.nn.Parameter(p0.clone())
    p_o = torch.nn.Parameter(p0.clone().to(cuda))
    opt_t = torch.optim.AdamW([p_t], lr=1e-3)
    opt_o = AdamW([p_o], lr=1e-3)
    po, mo, vo = p0.numpy().copy(), np.zeros_like(p0.numpy()), np.zeros_like(p0.numpy())
    for t in range(1, 6):
        gr = torch.randn(p0.shape, generator=g) * 10.0 ** float(-t)
        p_t.grad = gr.clone()
        p_o.grad = gr.clone().to(cuda)
        opt_t.step()
        opt_o.step()
        po, mo, vo = otrain.adamw_step(po, gr.numpy(), mo, vo, t, 1e-3)
        assert np.abs(p_o.detach().cpu().numpy() - po).max() <= 2e-7
        assert (p_o.detach().cpu() - p_t.detach()).abs().max().item() <= 2e-7
    st = opt_o.state[id(p_o)]
    np.testing.assert_allclose(st["exp_avg"].cpu().numpy(), mo, rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(st["exp_avg_sq"].cpu().numpy(), vo, rtol=1e-6, atol=1e-20)


@pytest.mark.parametrize("name,smooth", [("smooth", True), ("index", False)])
def test_train_model_loop_matches_reference_run(cuda, G, name, smooth):
    """pigeon_b200.training.train_model on the golden micro-batches == the reference module trained by torch."""
    from pigeon_b200 import SuperGuessr
    from pigeon_b200.training import train_model
    meta = json.loads(str(G["meta"]))
    n_micro, B = meta["steps"] * meta["acc"], meta["B"]
    emb = torch.tensor(G["emb"]).reshape(n_micro * B, 4, meta["D"])
    labels = torch.tensor(G["labels"]).reshape(n_micro * B, 2)
    labels_clf = torch.tensor(G["labels_clf"]).reshape(n_micro * B)

    class DS(torch.utils.data.Dataset):
        def __len__(self):
            return n_micro * B

        def __getitem__(self, i):
            return dict(embedding=emb[i], labels=labels[i], labels_clf=labels_clf[i])

    class Args:
        learning_rate = meta["lr"]
        per_device_train_batch_size = B
        num_train_epochs = 1
        gradient_accumulation_steps = meta["acc"]

    sg = SuperGuessr(None, panorama=True, num_candidates=5, should_smooth_labels=smooth, embed_dim=meta["D"],
                     geocells=G["centroids"]).to(cuda)
    with torch.no_grad():
        sg.cell_layer.weight.copy_(torch.tensor(G["w0"]))
        sg.cell_layer.bias.copy_(torch.tensor(G["b0"]))

    # the DataLoader of train_model shuffles (train_eval_loop.py:188); the golden run is in order
    import pigeon_b200.training as T
    real = T.DataLoader
    T.DataLoader = lambda ds, bs, shuffle=False, **kw: real(ds, bs, shuffle=False)
    try:
        # first micro-batch pair by hand: gradients before the first optimizer step
        sg.train()
        for i in range(meta["acc"]):
            s = slice(i * B, (i + 1) * B)
            out = sg(embedding=emb[s], labels=labels[s], labels_clf=labels_clf[s])
            np.testing.assert_allclose(float(out.loss), G[f"{name}_losses"][i], rtol=1e-5)
            sg.backward(out.loss)
        gw, gb = G[f"{name}_grad_w_step1"], G[f"{name}_grad_b_step1"]          # gw: the golden's sampled elements
        assert np.abs(sg.cell_layer.weight.grad.cpu().numpy().reshape(-1)[G["sample"]] - gw).max() <= 1e-5 * np.abs(gw).max()
        assert np.abs(sg.cell_layer.bias.grad.cpu().numpy() - gb).max() <= 1e-5 * np.abs(gb).max()
        sg.cell_layer.weight.grad = None
        sg.cell_layer.bias.grad = None
        train_model(sg, {"train": DS()}, True, False, Args(), None)
    finally:
        T.DataLoader = real
    pick = lambda a: a.reshape(-1)[G["sample"]]
    for k, p, p0 in (("w_final", pick(sg.cell_layer.weight.detach().cpu().numpy()), pick(G["w0"])),
                     ("b_final", sg.cell_layer.bias.detach().cpu().numpy(), G["b0"])):
        ref = G[f"{name}_{k}"]
        move = np.abs(ref - p0).max()
        assert np.abs(p - ref).max() <= 2e-2 * move
        # the bulk of the entries agrees far tighter (only gradients of the order of eps amplify rounding)
        assert np.median(np.abs(p - ref)) <= 1e-4 * move
    # the trained head is the one inference uses afterwards (packed fp16 copy refreshed after optimizer steps)
    sg.eval()
    with torch.no_grad():
        o = sg(embedding=emb[:B], labels=labels[:B], labels_clf=labels_clf[:B])
    w, b = sg.cell_layer.weight.detach().double().cpu(), sg.cell_layer.bias.detach().double().cpu()
    ref_logits = emb[:B].double().mean(1) @ w.t() + b
    assert torch.equal(o.preds_geocell.cpu(), ref_logits.argmax(-1))


def test_training_forward_refuses_partly_frozen_block(cuda):
    """A block is trainable or frozen as a whole (the reference freezes whole layers, super_guessr.py:159-160); anything
    else fails loudly instead of silently dropping a gradient."""
    from pigeon_b200 import PigeonB200Error, SuperGuessr, synthetic
    from pigeon_b200.super_guessr import CLIPVisionTower
    from pigeon_b200.vit_engine import VitDims
    dims = VitDims(image_size=56, patch_size=14, hidden=256, heads=4, intermediate=512, layers=1)
    tower = CLIPVisionTower(dims)
    tower.load_state_dict(synthetic.random_vit_state_dict(dims, seed=1), strict=True)
    sg = SuperGuessr(tower, panorama=False, geocells=np.zeros((10, 2))).to(cuda).train()
    tower.vision_model.encoder.layers[0].mlp.fc1.weight.requires_grad = False
    with pytest.raises(PigeonB200Error):
        sg(pixel_values=torch.zeros(1, 3, 56, 56, device=cuda), labels_clf=torch.tensor([1]))
    with pytest.raises(NotImplementedError):                 # parameters the step has no backward for
        sg.lla_geocells.requires_grad = True
        tower.vision_model.encoder.layers[0].mlp.fc1.weight.requires_grad = True
        sg(pixel_values=torch.zeros(1, 3, 56, 56, device=cuda), labels_clf=torch.tensor([1]))


def test_multi_task_training_matches_reference_run(cuda, G):
    """multi_task=True: the geocell head through the kernels, the three auxiliary heads through torch autograd on the GPU,
    one AdamW over all of them == the unmodified reference trained by torch (tests/golden/train_head.npz, 'multitask')."""
    from pigeon_b200 import SuperGuessr
    from pigeon_b200.training import AdamW
    meta = json.loads(str(G["meta"]))
    n_micro, B, acc = meta["steps"] * meta["acc"], meta["B"], meta["acc"]
    sg = SuperGuessr(None, panorama=True, num_candidates=5, should_smooth_labels=True, embed_dim=meta["D"], multi_task=True,
                     geocells=G["centroids"]).to(cuda).train()
    heads = ("multi_task_head", "climate_layer", "month_layer")
    with torch.no_grad():
        sg.cell_layer.weight.copy_(torch.tensor(G["w0"]))
        sg.cell_layer.bias.copy_(torch.tensor(G["b0"]))
        for hn in heads:
            getattr(sg, hn).weight.copy_(torch.tensor(G[f"mt_init_{hn}_w"]))
            getattr(sg, hn).bias.copy_(torch.tensor(G[f"mt_init_{hn}_b"]))
    opt = AdamW(sg.parameters(), lr=meta["lr"])
    opt.zero_grad()
    for i in range(n_micro):
        out = sg(embedding=torch.tensor(G["emb"][i]), labels=torch.tensor(G["labels"][i]),
                 labels_clf=torch.tensor(G["labels_clf"][i]), labels_multi_task=torch.tensor(G["labels_mt"][i]),
                 labels_climate=torch.tensor(G["labels_climate"][i]), labels_month=torch.tensor(G["labels_month"][i]))
        np.testing.assert_allclose(float(out.loss), G["multitask_losses"][i], rtol=2e-5)
        sg.backward(out.loss)
        if i % acc == acc - 1:
            opt.step()
            opt.zero_grad()
    host = lambda p: p.detach().cpu().numpy()
    pick = lambda a: a.reshape(-1)[G["sample"]]
    pairs = [(pick(host(sg.cell_layer.weight)), G["multitask_w_final"], pick(G["w0"])),
             (host(sg.cell_layer.bias), G["multitask_b_final"], G["b0"])]
    for hn in heads:
        pairs.append((host(getattr(sg, hn).weight), G[f"mt_final_{hn}_w"], G[f"mt_init_{hn}_w"]))
        pairs.append((host(getattr(sg, hn).bias), G[f"mt_final_{hn}_b"], G[f"mt_init_{hn}_b"]))
    for p, ref, p0 in pairs:
        move = np.abs(ref - p0).max()
        assert np.abs(p - ref).max() <= 2e-2 * move
        assert np.median(np.abs(p - ref)) <= 1e-3 * move
