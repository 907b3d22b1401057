"""CPU: pins oracle/dquartic_oracle.py against vectors produced by the unmodified reference
(oracle/gen_golden.py -> tests/golden/*.npz)."""
import json
import os
import random

import numpy as np
import pytest
import torch

import dquartic_oracle as O

TINY = dict(dim=4, channels=1, dim_mults=[1, 2, 2, 3, 3, 4, 4], conditional=True, init_cond_channels=1,
            attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=320, simple=True)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_schedule_bit_exact(golden_dir):
    g = _load(golden_dir, "schedule.npz")
    for kind in ("cosine", "linear"):
        betas, alphas, ab = O.schedule_tables(1000, kind)
        assert np.array_equal(betas.numpy(), g[f"{kind}_betas"])
        assert np.array_equal(alphas.numpy(), g[f"{kind}_alphas"])
        assert np.array_equal(ab.numpy(), g[f"{kind}_alpha_bars"])
    _, _, ab = O.schedule_tables(1000, "cosine")
    assert np.array_equal(O.loss_weight_table(ab, "x0").numpy(), g["cosine_x0_loss_weight"])
    assert np.array_equal(O.ddim_timesteps(1000, 50).numpy(), g["steps50"])
    assert np.array_equal(O.ddim_timesteps(1000, 7).numpy(), g["steps7"])
    # known answers quoted in SURVEY.md §8 a1
    assert abs(float(ab[0]) - 0.99995869) < 1e-7 and abs(float(ab[499]) - 0.49384347) < 1e-7
    assert g["steps50"][:3].tolist() == [999, 978, 958] and g["steps50"][-3:].tolist() == [40, 20, 0]


def test_param_inventory_known_answers(golden_dir):
    info = json.load(open(os.path.join(golden_dir, "state_dict_keys.json")))
    for name in ("default", "notebook", "tiny"):
        shapes = O.param_shapes(info[name]["cfg"])
        ref = {k: tuple(s) for k, s in info[name]["keys"]}
        assert set(shapes) == set(ref)
        for k in ref:
            assert tuple(shapes[k]) == ref[k], k
        total = sum(int(np.prod(s)) for s in shapes.values())
        assert total == info[name]["total"]
        assert len(ref) == 396
    # torchinfo table in the reference's nbs/quantization_experiment.ipynb cell 14
    assert info["notebook"]["total"] == 1204739463 and info["notebook"]["trainable"] == 1204739455
    assert info["default"]["total"] == 1204738391


def test_unet_forward_matches_reference(golden_dir):
    g = _load(golden_dir, "unet_tiny.npz")
    P = O.det_params(TINY)
    with torch.no_grad():
        out = O.unet_forward(P, TINY, torch.from_numpy(g["x"]), torch.from_numpy(g["time"]),
                             torch.from_numpy(g["init_cond"]), torch.from_numpy(g["attn_cond"]))
    np.testing.assert_allclose(out.numpy(), g["out"], rtol=1e-4, atol=1e-5)


def test_train_step_loss_and_grads_match_reference(golden_dir):
    g = _load(golden_dir, "train_tiny.npz")
    gg = _load(golden_dir, "train_tiny_grads.npz")
    P = {k: v.clone().requires_grad_(not k.endswith("freqs")) for k, v in O.det_params(TINY).items()}
    _, _, ab = O.schedule_tables(1000, "cosine")
    loss, _ = O.train_loss(P, TINY, ab, torch.from_numpy(g["x0"]), torch.from_numpy(g["ms2_cond"]),
                           torch.from_numpy(g["ms1_cond"]), torch.from_numpy(g["t"]), torch.from_numpy(g["noise"]))
    assert abs(float(loss.detach()) - float(g["loss"])) < 1e-5 * max(1.0, abs(float(g["loss"])))
    loss.backward()
    names = [k for k in P if P[k].requires_grad]
    for k in names:
        ref = gg["grad:" + k]
        got = P[k].grad.numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= 2e-4 * scale + 1e-7, k
    grads = [P[k].grad for k in names]
    clipped, total = O.clip_grad_norm(grads)
    assert abs(float(total) - float(g["total_norm"])) < 1e-4 * float(g["total_norm"])
    # optimizer arithmetic is checked on the REFERENCE's gradients so that the first-step sign(g)-like
    # update (m / (sqrt(v) + eps) with |g| ~ eps) is not sensitive to 1e-4-level gradient differences
    lr = float(g["lr"])
    ref_grads = [torch.from_numpy(gg["grad:" + k]) for k in names]
    clipped, total = O.clip_grad_norm(ref_grads)
    assert abs(float(total) - float(g["total_norm"])) < 1e-5 * float(g["total_norm"])
    for k, gc in zip(names, clipped):
        if ("new:" + k) in g.files:
            p, m, v = O.adamw_step(P[k].detach(), gc, torch.zeros_like(gc), torch.zeros_like(gc), 1, lr)
            np.testing.assert_allclose(p.numpy(), g["new:" + k], rtol=1e-5, atol=1e-7)


def test_ddim_sample_matches_reference(golden_dir):
    g = _load(golden_dir, "sample_tiny.npz")
    P = O.det_params(TINY)
    _, _, ab = O.schedule_tables(1000, "cosine")
    xT, c2, c1 = (torch.from_numpy(g[k]) for k in ("x_T", "ms2_cond", "ms1_cond"))
    with torch.no_grad():
        for steps in (1, 6, 50):
            x, pn = O.ddim_sample(P, TINY, ab, xT, c2, c1, steps)
            ref = torch.from_numpy(g[f"x_{steps}"])
            cos = torch.nn.functional.cosine_similarity(x.flatten(1), ref.flatten(1), dim=1)
            assert float(cos.min()) > 0.99999, (steps, cos)
            np.testing.assert_allclose(x.numpy(), g[f"x_{steps}"], rtol=2e-3, atol=2e-3 * np.abs(g[f"x_{steps}"]).max())
            np.testing.assert_allclose(pn.numpy(), g[f"pred_noise_{steps}"], rtol=2e-3,
                                       atol=2e-3 * np.abs(g[f"x_{steps}"]).max())
        eps = O.unet_forward(P, TINY, xT[0:1], torch.tensor([500]), O.normalize(c2[0:1]), O.normalize(c1[0:1]))
        np.testing.assert_allclose(eps.numpy(), g["p500_eps"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(O.ddim_update(ab, xT[0:1], eps, 500).numpy(), g["p500_x"], rtol=1e-4, atol=1e-5)
        eps0 = O.unet_forward(P, TINY, xT[0:1], torch.tensor([0]), O.normalize(c2[0:1]), O.normalize(c1[0:1]))
        np.testing.assert_allclose(O.ddim_update(ab, xT[0:1], eps0, 0).numpy(), g["p0_x"], rtol=1e-4, atol=1e-5)


def test_pair_selection_and_minmax_bit_exact(golden_dir):
    g = _load(golden_dir, "data.npz")
    rng = random.Random(1234)
    used = set()
    seq = []
    for epoch in range(2):
        used.clear()
        for _ in range(64):
            seq.append(O.pair_draw(rng, 520, used))
    assert np.array_equal(np.array(seq, dtype=np.int64), g["pairs520"])
    ms2, ms1 = g["ms2_pool"], g["ms1_pool"]
    rng = random.Random(1234)
    used = set()
    for j in range(6):
        i1, i2 = O.pair_draw(rng, ms2.shape[0], used)
        a, b, c, d = O.minmax_pair(ms2[i1], ms1[i1], ms2[i2], ms1[i2])
        for nm, arr in zip(("ms2_1", "ms1_1", "ms2_2", "ms1_2"), (a, b, c, d)):
            assert np.array_equal(arr, g[f"item{j}:{nm}"]), (j, nm)
        mixed = O.mix(torch.from_numpy(a), torch.from_numpy(c)).numpy()
        assert np.array_equal(mixed, g[f"item{j}:mix"])


def test_lr_lambda_matches_formula():
    # model_interface.py:149-155 evaluated by hand
    assert O.lr_lambda(0, 5, 100) == pytest.approx(0.2)
    assert O.lr_lambda(4, 5, 100) == pytest.approx(1.0)
    assert O.lr_lambda(5, 5, 100) == pytest.approx(1.0)
    assert O.lr_lambda(100, 5, 100) == pytest.approx(1e-10)
