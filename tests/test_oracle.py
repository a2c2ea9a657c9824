"""CPU: the oracle restatements against the golden vectors produced by the reference itself
(tests/golden/make_golden.py).  No /root/reference needed."""
import os

import numpy as np
import pytest
import torch

from oracle.darknet_ref import RefDarknet, reorg_ref
from oracle import region_loss_ref as RL
from oracle.decode_ref import get_region_boxes_ref
from oracle.pnp_ref import pnp_ref, rodrigues_vec2mat, rodrigues_mat2vec, project
from singleshotpose_b200 import synth


def _ang(Ra, Rb):
    return np.degrees(np.arccos(np.clip((np.trace(Ra @ Rb.T) - 1) / 2, -1, 1)))


def test_region_loss_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "region_loss.npz"))
    out, tgt = torch.from_numpy(g["output"]), torch.from_numpy(g["target"])
    for epoch in (0, 20):
        o = out.clone().requires_grad_(True)
        loss, info = RL.region_loss_ref(o, tgt, epoch)
        loss.backward()
        assert float(loss) == pytest.approx(float(g["loss_e%d" % epoch]), rel=1e-6)
        np.testing.assert_allclose(o.grad.numpy(), g["grad_e%d" % epoch], rtol=1e-6, atol=1e-7)
        assert [info["nGT"], info["nCorrect"], info["nProposals"]] == list(g["counters_e%d" % epoch])
    np.testing.assert_allclose(info["tconf"].numpy(), g["tconf"], rtol=1e-6, atol=1e-8)
    np.testing.assert_array_equal(info["conf_mask"].numpy(), g["conf_mask_sqrt"])


def test_region_loss_epoch_gate_and_single_gt(golden_dir):
    g = np.load(os.path.join(golden_dir, "region_loss.npz"))
    p0, p20 = g["parts_e0"], g["parts_e20"]
    assert float(g["loss_e0"]) == pytest.approx(p0[0] + p0[1], rel=1e-6)          # conf term gated off
    assert float(g["loss_e20"]) == pytest.approx(p20.sum(), rel=1e-6)
    assert np.abs(g["grad_e0"][:, 18]).max() == 0.0                                # no conf gradient when gated


def test_decode_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "decode.npz"))
    box = get_region_boxes_ref(torch.from_numpy(g["output"]), 1, 9)
    np.testing.assert_array_equal(np.array([float(v) for v in box]), g["box"])


def test_pnp_oracle_matches_cv2_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "pnp.npz"))
    for tag in ("s0", "s1"):
        for i in range(0, 64, 4):
            R, t = pnp_ref(g["P3"], g["uv_" + tag][i], g["K"])
            assert _ang(R, g["R_" + tag][i]) < 1e-4                 # degrees
            assert np.abs(t.reshape(3) - g["t_" + tag][i]).max() * 1e3 < 1e-4   # mm


def test_pnp_oracle_matches_reference_golden_noisy(golden_dir):
    """sigma = 5 / 20 / 80 px and random-init-network keypoints: outputs of the reference's own pnp (make_golden_pnp_noise.py)"""
    g = np.load(os.path.join(golden_dir, "pnp_noise.npz"))
    for tag in ("s5", "s20", "s80", "net"):
        for i in range(0, 64, 8):
            R, t = pnp_ref(g["P3"], g["uv_" + tag][i], g["K"])
            assert _ang(R, g["R_" + tag][i]) < 1e-3, (tag, i)
            assert np.abs(t.reshape(3) - g["t_" + tag][i]).max() * 1e3 < 1e-3, (tag, i)


def test_eval_loop_oracle_recovers_planted_pose():
    """oracle/eval_ref.py (valid.py:123-183): planting the exact ground-truth keypoints in one confident cell gives zero errors"""
    import torch
    from oracle.eval_ref import evaluate_image_ref
    pr = synth.pnp_problems(1, sigma=0.0, seed=21)
    uvn = pr["uv"][0] / np.array([640.0, 480.0], np.float32)
    out = torch.zeros(1, 20, 13, 13)
    cx, cy = int(uvn[0, 0] * 13), int(uvn[0, 1] * 13)
    for k in range(9):
        vx, vy = uvn[k, 0] * 13 - cx, uvn[k, 1] * 13 - cy
        if k == 0:
            vx, vy = np.log(vx / (1 - vx)), np.log(vy / (1 - vy))
        out[0, 2 * k, cy, cx], out[0, 2 * k + 1, cy, cx] = float(vx), float(vy)
    out[0, 18, cy, cx] = 8.0
    tgt = np.zeros(21, np.float32); tgt[1:19] = uvn.reshape(-1)
    verts = np.concatenate([np.random.default_rng(0).uniform(-0.04, 0.04, size=(3, 50)), np.ones((1, 50))])
    r = evaluate_image_ref(out, tgt, verts, pr["P3"], synth.intrinsics())
    assert r["corner_err_px"] < 1e-2 and r["pixel_err"] < 1e-2 and r["angle_err_deg"] < 5e-2 and r["trans_err"] < 1e-4


def test_pnp_oracle_live_cv2():
    cv2 = pytest.importorskip("cv2")
    pr = synth.pnp_problems(8, sigma=1.0, seed=11)
    for i in range(8):
        _, rv, tv = cv2.solvePnP(pr["P3"], pr["uv"][i].reshape(-1, 1, 2), pr["K"], np.zeros((8, 1), np.float32))
        R, _ = cv2.Rodrigues(rv)
        Ro, to = pnp_ref(pr["P3"], pr["uv"][i], pr["K"])
        assert _ang(R, Ro) < 1e-4 and np.abs(tv - to).max() * 1e3 < 1e-4


def test_rodrigues_roundtrip_and_jacobian():
    rng = np.random.default_rng(0)
    for _ in range(20):
        r = rng.normal(size=3)
        r *= rng.uniform(0.01, 3.0) / np.linalg.norm(r)
        R, J = rodrigues_vec2mat(r, True)
        np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-12)
        np.testing.assert_allclose(rodrigues_mat2vec(R), r, atol=1e-9)
        num = np.stack([(rodrigues_vec2mat(r + 1e-6 * e) - rodrigues_vec2mat(r - 1e-6 * e)).reshape(9) / 2e-6
                        for e in np.eye(3)])
        np.testing.assert_allclose(J, num, atol=1e-7)


def test_projection_jacobian_numeric():
    pr = synth.pnp_problems(1, sigma=0, seed=2)
    M = pr["P3"].astype(np.float64); K = pr["K"].astype(np.float64)
    p = np.array([0.3, -0.5, 0.8, 0.05, -0.02, 0.9])
    _, J = project(M, p[:3], p[3:], K, jac=True)
    num = np.stack([(project(M, (p + 1e-6 * e)[:3], (p + 1e-6 * e)[3:], K)
                     - project(M, (p - 1e-6 * e)[:3], (p - 1e-6 * e)[3:], K)).reshape(-1) / 2e-6 for e in np.eye(6)], 1)
    np.testing.assert_allclose(J, num, rtol=1e-5, atol=1e-4)


def test_reorg_marvis_ordering():
    x = torch.arange(2 * 4 * 6 * 6, dtype=torch.float32).view(2, 4, 6, 6)
    y = reorg_ref(x, 2)
    for b, c, h, w, i, j in [(0, 0, 0, 0, 0, 0), (1, 3, 2, 1, 1, 0), (0, 2, 1, 2, 0, 1), (1, 1, 2, 2, 1, 1)]:
        assert y[b, (i * 2 + j) * 4 + c, h, w] == x[b, c, 2 * h + i, 2 * w + j]


@pytest.mark.timeout(600)
def test_network_oracle_matches_reference_golden(golden_dir, cfg_path):
    """Seeded default init + forward of the restated network == the reference's (bit for bit at
    generation time; 1e-5 here to allow a different CPU/BLAS on the test box)."""
    g = np.load(os.path.join(golden_dir, "net_b2.npz"))
    torch.manual_seed(0)
    model = RefDarknet(cfg_path)
    assert [n for n, _ in model.named_parameters()] == list(g["names"])
    model.train()
    x, tgt = synth.images(2, seed=0), synth.targets(2, seed=1)
    out = model(x)
    scale = np.abs(g["train_logits"]).max()
    assert np.abs(out.detach().numpy() - g["train_logits"]).max() / scale < 1e-4
    np.testing.assert_allclose(model.models[0][1].running_mean.numpy(), g["running_mean0"], rtol=1e-4, atol=1e-6)
    loss, _ = RL.region_loss_ref(out, tgt, 20)
    assert float(loss) == pytest.approx(float(g["loss"]), rel=1e-3)
    loss.backward()
    gn = np.array([p.grad.double().norm().item() for p in model.parameters()])
    np.testing.assert_allclose(gn, g["grad_norms"], rtol=2e-2)


def test_oracle_network_other_resolutions_match_reference_golden(cfg_path, golden_dir):
    """the oracle network at a multi-resolution training shape and a small one vs the reference's logits (make_golden.py main_multires).
    Bit for bit on the CPU that generated the goldens; another CPU's convolution kernels sum in another order (4e-6 of the largest
    logit measured on a second x86 host), hence 2e-5."""
    import torch
    from oracle.darknet_ref import RefDarknet
    from singleshotpose_b200 import synth
    g = np.load(os.path.join(golden_dir, "net_multires.npz"))
    torch.manual_seed(0)
    m = RefDarknet(cfg_path).train()
    for (h, w, seed) in ((352, 480, 5), (224, 224, 6)):
        with torch.no_grad():
            o = m(synth.images(1, h, w, seed=seed)).numpy()
        want = g["logits_%dx%d" % (h, w)]
        assert o.shape == want.shape
        assert np.abs(o - want).max() / np.abs(want).max() < 2e-5, (h, w)

