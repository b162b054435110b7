"""CPU: the oracle restatement (oracle/robust_unet_ref.py) against the committed golden vectors
that oracle/make_golden.py produced by running the unmodified reference (Main_Final.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import robust_unet_ref as R

GOLDEN_THREADS = 8       # torch.set_num_threads of oracle/make_golden.py


@pytest.fixture(autouse=True)
def golden_thread_count():
    """torch's CPU convolutions split their sums by the intra-op thread count, so the oracle reproduces the goldens bit for
    bit only with the thread count that wrote them, whatever the host's core count (elsewhere: up to 1.6e-4 on the eval
    probabilities of model_c4_b16_32x48)."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _run_model(g, training):
    n_channels, base, batch, h, w = [int(v) for v in g["config"]]
    sd = R.synthetic_state_dict(R.robust_unet_shapes(n_channels, 1, base), seed=0)
    x, y = R.synthetic_inputs(batch, n_channels, h, w, seed=123, blobby=True)
    masks = R.synthetic_drop_masks(batch, base, seed=7)
    return sd, x, y, masks, base


@pytest.mark.parametrize("name", ["model_c3_b16_32x32.npz", "model_c4_b16_32x48.npz", "model_c3_b64_64x64.npz",
                                  "model_c4_b64_64x96.npz"])
def test_model_eval_matches_reference_golden(golden_dir, name):
    g = _load(golden_dir, name)
    sd, x, y, _, _ = _run_model(g, False)
    with torch.no_grad():
        p = R.robust_unet_forward(sd, x, training=False)
    np.testing.assert_allclose(p.numpy(), g["probs_eval"], rtol=0, atol=2e-6)
    assert abs(R.bce_loss(p, y).item() - float(g["loss_eval"])) < 1e-4
    counts = R.confusion_counts(p.numpy(), y.numpy())
    ref_counts = R.confusion_counts(g["probs_eval"], y.numpy())
    assert (counts == ref_counts).all()
    for i in range(p.shape[0]):
        m = R.metrics_from_counts(*counts[i])
        for j, k in enumerate(g["metric_keys"]):
            assert abs(m[str(k)] - g["metrics_eval"][i, j]) < 1e-12


@pytest.mark.parametrize("name", ["model_c3_b16_32x32.npz", "model_c4_b16_32x48.npz", "model_c3_b64_64x64.npz",
                                  "model_c4_b64_64x96.npz"])
def test_model_train_step_matches_reference_golden(golden_dir, name):
    g = _load(golden_dir, name)
    sd, x, y, masks, _ = _run_model(g, True)
    names = [str(n) for n in g["param_names"]]
    for n in names:
        sd[n].requires_grad_(True)
    newbuf = {}
    p = R.robust_unet_forward(sd, x, training=True, drop_masks=masks, new_buffers=newbuf)
    loss = R.bce_dice_loss(p, y, 1.0, float(g["w_dice"]))
    loss.backward()
    np.testing.assert_allclose(p.detach().numpy(), g["probs_train"], rtol=0, atol=5e-6)
    assert abs(loss.item() - float(g["loss_train"])) < 1e-5
    for i, n in enumerate(names):
        s = g["grad_summary"][i]
        gr = sd[n].grad.double().flatten()
        tol = 1e-4 * max(s[0], 1e-6) + 1e-7
        assert abs(gr.norm().item() - s[0]) < tol, n
        head = gr[:8].numpy()
        np.testing.assert_allclose(head, s[2:2 + head.size], rtol=0, atol=1e-4 * max(s[0], 1e-6) + 1e-7, err_msg=n)
    for i, n in enumerate(g["buffer_names"]):
        s = g["buffer_summary"][i]
        assert abs(newbuf[str(n)].double().norm().item() - s[0]) < 1e-5 * max(s[0], 1.0), n


def test_module_goldens(golden_dir):
    g = _load(golden_dir, "modules.npz")
    # ResidualBlock
    shapes = {k[len("down1.1."):]: v for k, v in R.robust_unet_shapes(3, 1, 16).items() if k.startswith("down1.1.")}
    sd = {"b." + k: v for k, v in R.synthetic_state_dict(shapes, seed=3).items()}
    for k, v in sd.items():
        if v.is_floating_point() and "running" not in k:
            v.requires_grad_(True)
    x = torch.from_numpy(g["rb_x"]).requires_grad_(True)
    o = R.residual_block(sd, "b", x, True, torch.from_numpy(g["rb_mask"]))
    o.backward(torch.from_numpy(g["rb_gout"]))
    np.testing.assert_allclose(o.detach().numpy(), g["rb_out"], atol=2e-6, rtol=0)
    np.testing.assert_allclose(x.grad.numpy(), g["rb_gx"], atol=2e-5, rtol=1e-4)
    for k in g.files:
        if k.startswith("rb_g_"):
            np.testing.assert_allclose(sd["b." + k[5:]].grad.numpy(), g[k], atol=2e-5, rtol=1e-4, err_msg=k)
    # AttentionGate
    shapes = {k[len("att1."):]: v for k, v in R.robust_unet_shapes(3, 1, 32).items() if k.startswith("att1.")}
    sd = {"a." + k: v for k, v in R.synthetic_state_dict(shapes, seed=4).items()}
    for k, v in sd.items():
        if v.is_floating_point() and "running" not in k:
            v.requires_grad_(True)
    gg = torch.from_numpy(g["ag_g"]).requires_grad_(True)
    xx = torch.from_numpy(g["ag_x"]).requires_grad_(True)
    o = R.attention_gate(sd, "a", gg, xx, True)
    o.backward(torch.from_numpy(g["ag_gout"]))
    np.testing.assert_allclose(o.detach().numpy(), g["ag_out"], atol=2e-6, rtol=0)
    np.testing.assert_allclose(gg.grad.numpy(), g["ag_gg"], atol=2e-5, rtol=1e-4)
    np.testing.assert_allclose(xx.grad.numpy(), g["ag_gx"], atol=2e-5, rtol=1e-4)
    # DilatedBlock
    shapes = {k[len("bottleneck.1."):]: v for k, v in R.robust_unet_shapes(3, 1, 4).items() if k.startswith("bottleneck.1.")}
    sd = {"d." + k: v for k, v in R.synthetic_state_dict(shapes, seed=5).items()}
    xd = torch.from_numpy(g["db_x"]).requires_grad_(True)
    o = R.dilated_block(sd, "d", xd, True)
    o.backward(torch.from_numpy(g["db_gout"]))
    np.testing.assert_allclose(o.detach().numpy(), g["db_out"], atol=2e-6, rtol=0)
    np.testing.assert_allclose(xd.grad.numpy(), g["db_gx"], atol=2e-5, rtol=1e-4)


def test_metric_goldens(golden_dir):
    g = _load(golden_dir, "metrics.npz")
    counts = R.confusion_counts(g["pred"], g["target"])
    assert counts.sum(1).tolist() == [256] * 4
    for i in range(4):
        m = R.metrics_from_counts(*counts[i])
        for j, k in enumerate(g["metric_keys"]):
            assert abs(m[str(k)] - g["metrics"][i, j]) < 1e-12, (i, k)
    # empty/empty: accuracy 1, everything else 0 (SURVEY §8a)
    m = R.metrics_from_counts(*counts[2])
    assert m["accuracy"] == 1.0 and m["iou"] == 0.0 and m["f1_score"] == 0.0


def test_hsv_against_colorsys_and_cv2():
    import colorsys
    rng = np.random.RandomState(1)
    rgb = rng.rand(64, 3).astype(np.float32)
    rgb[:4] = [[0, 0, 0], [1, 1, 1], [0.5, 0.5, 0.5], [1, 0, 0]]
    hsv = R.rgb_to_hsv(rgb)
    for i in range(rgb.shape[0]):
        h, s, v = colorsys.rgb_to_hsv(*[float(c) for c in rgb[i]])
        assert abs(hsv[i, 0] - h * 360.0) < 1e-3 and abs(hsv[i, 1] - s) < 1e-5 and abs(hsv[i, 2] - v) < 1e-6
    cv2 = pytest.importorskip("cv2")
    ref = cv2.cvtColor(rgb.reshape(1, -1, 3), cv2.COLOR_RGB2HSV).reshape(-1, 3)
    np.testing.assert_allclose(hsv, ref, atol=2e-3, rtol=0)
