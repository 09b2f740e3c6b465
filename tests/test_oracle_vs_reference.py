"""CPU: the oracle against fixtures produced by the REFERENCE's own code.

tests/golden/ref_*.npz were written by tests/golden/make_ref_fixtures.py, which imports
/root/reference/ppvector/{models,loss,optimizer}/*.py UNMODIFIED under tests/paddle_shim (a paddle -> torch
stand-in; tests/paddle_shim/README.md lists every assumed op) and runs them in fp64 on the oracle's seeded
weights.  Agreement to 1e-10 ties the restatement in oracle/ to the reference graph; what stays assumed is the
semantics of the individual Paddle ops.
"""
import hashlib
import json

import numpy as np
import pytest
import torch

from oracle import campplus, ecapa, eres2net, head, resnet_se
from oracle import train as otrain

TOL = 1e-10
SEEDS = {"ecapa": 1000, "resnetse": 2000, "eres2net": 3000, "campplus": 4000}


def feats(model, T, B=2):
    g = torch.Generator().manual_seed(SEEDS[model] + T)
    f = torch.randn(B, T, 80, generator=g, dtype=torch.float64)
    return f - f.mean(1, keepdim=True)


def tap_slice(t):
    t = t.detach()
    idx = tuple(slice(0, min(n, 6)) for n in t.shape)
    return np.concatenate([t[idx].reshape(-1).numpy(), [float(t.abs().mean()), float(t.sum())]])


def close(a, b, tol=TOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b).max() / max(1.0, np.abs(b).max())
    assert err <= tol, err


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(f"{golden_dir}/ref_models.npz")


# ------------------------------------------------------------------------------------------------ backbones
@pytest.mark.parametrize("T", [98, 298])
def test_ecapa_matches_reference_code(ref, T):
    W = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    taps = {}
    emb = ecapa.ecapa_forward(feats("ecapa", T), W, taps=taps, layer_taps=True)
    close(emb.numpy(), ref[f"ecapa_T{T}_emb"])
    for k in ["blocks.0", "blocks.1.tdnn1", "blocks.1.res2net_block", "blocks.1.tdnn2", "blocks.1", "blocks.2", "blocks.3", "mfa", "asp"]:
        close(tap_slice(taps[k]), ref[f"ecapa_T{T}_tap_{k}"])


def test_ecapa_variants_match_reference_code(ref):
    f = feats("ecapa", 98)
    W = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    # lengths reach SEBlock and ASP (ecapa_tdnn.py:69-77, pooling.py:94-99)
    close(ecapa.ecapa_forward(f, W, lengths=torch.tensor([1.0, 0.6], dtype=torch.float64)).numpy(), ref["ecapa_T98_lengths_emb"])
    Wg = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, global_context=False)
    close(ecapa.ecapa_forward(f, Wg, global_context=False).numpy(), ref["ecapa_T98_noctx_emb"])
    # SERes2NetBlock shortcut conv (ecapa_tdnn.py:125-131)
    Ws = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, channels=(256, 384, 384, 384, 1152))
    close(ecapa.ecapa_forward(f, Ws).numpy(), ref["ecapa_T98_shortcut_emb"])


def test_non_asp_heads_raise_in_the_reference_and_pooling_modules_match(ref):
    # EcapaTdnn / ResNetSE with pooling_type SAP / TAP / TSP cannot run in the reference (double unsqueeze -> Conv1d on 4-D;
    # Linear on [N,C,1]); the pooling modules alone are pinned (pooling.py:8-66)
    for k in ("ecapa_SAP_raises", "ecapa_TAP_raises", "ecapa_TSP_raises", "resnetse_TAP_raises"):
        assert int(ref[k]) == 1
    g = torch.Generator().manual_seed(515)
    x = torch.randn(2, 1536, 50, generator=g, dtype=torch.float64)
    assert abs(float(x.sum()) - float(ref["pool_x_seed515_checksum"])) < 1e-9
    F = torch.nn.functional
    W = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64, pooling_type="SAP")
    a = torch.tanh(F.conv1d(x, W["asp.linear1.weight"], W["asp.linear1.bias"]))
    a = F.softmax(F.conv1d(a, W["asp.linear2.weight"], W["asp.linear2.bias"]), dim=2)
    close((a * x).sum(2, keepdim=True).numpy(), ref["pool_SAP_out"])
    close(x.mean(2, keepdim=True).numpy(), ref["pool_TAP_out"])
    close(torch.cat((x.mean(2), x.var(2, unbiased=True)), 1).unsqueeze(2).numpy(), ref["pool_TSP_out"])


@pytest.mark.parametrize("T", [98, 298])
def test_resnetse_matches_reference_code(ref, T):
    W = resnet_se.make_resnet_se_weights(seed=1000, dtype=torch.float64)
    taps = {}
    emb = resnet_se.resnet_se_forward(feats("resnetse", T), W, taps=taps)
    close(emb.numpy(), ref[f"resnetse_T{T}_emb"])
    for mine, theirs in [("conv1", "relu"), ("layer1", "layer1"), ("layer2", "layer2"), ("layer3", "layer3"), ("layer4", "layer4"),
                         ("asp", "pooling")]:
        close(tap_slice(taps[mine]), ref[f"resnetse_T{T}_tap_{theirs}"])


@pytest.mark.parametrize("T", [98, 298])
def test_eres2net_matches_reference_code(ref, T):
    W = eres2net.make_eres2net_weights(seed=1000, dtype=torch.float64)
    taps = {}
    emb = eres2net.eres2net_forward(feats("eres2net", T), W, taps=taps)
    close(emb.numpy(), ref[f"eres2net_T{T}_emb"])
    for mine, theirs in [("layer1", "layer1"), ("layer2", "layer2"), ("layer3", "layer3"), ("layer4", "layer4"),
                         ("fuse12", "fuse_mode12"), ("fuse123", "fuse_mode123"), ("fuse1234", "fuse_mode1234"), ("stats", "pooling")]:
        close(tap_slice(taps[mine]), ref[f"eres2net_T{T}_tap_{theirs}"])


@pytest.mark.parametrize("T", [98, 298])
def test_eres2netv2_matches_reference_code(ref, T):
    """ERes2NetV2 (eres2net.py:266-462): base_width 26 -> chunk widths 13 / 26 / 52 / 104, AFF blocks in layers 3-4, layer3_ds + fuse34"""
    W = eres2net.make_eres2net_weights(seed=1000, dtype=torch.float64, base_width=26, version=2)
    taps = {}
    emb = eres2net.eres2net_forward(feats("eres2net", T), W, taps=taps, base_width=26, version=2)
    close(emb.numpy(), ref[f"eres2netv2_T{T}_emb"])
    for mine, theirs in [("layer1", "layer1"), ("layer2", "layer2"), ("layer3", "layer3"), ("layer4", "layer4"), ("fuse34", "fuse34"),
                         ("stats", "pooling")]:
        close(tap_slice(taps[mine]), ref[f"eres2netv2_T{T}_tap_{theirs}"])


@pytest.mark.parametrize("T", [98, 298])
def test_campplus_matches_reference_code(ref, T):
    W = campplus.make_campplus_weights(seed=1000, dtype=torch.float64)
    taps = {}
    emb = campplus.campplus_forward(feats("campplus", T), W, taps=taps)
    close(emb.numpy(), ref[f"campplus_T{T}_emb"])
    for mine, theirs in [("head", "head"), ("tdnn", "xvector.tdnn"), ("block1", "xvector.block1"), ("transit1", "xvector.transit1"),
                         ("block2", "xvector.block2"), ("transit2", "xvector.transit2"), ("block3", "xvector.block3"),
                         ("transit3", "xvector.transit3"), ("stats", "xvector.stats")]:
        close(tap_slice(taps[mine]), ref[f"campplus_T{T}_tap_{theirs}"])


# ------------------------------------------------------------------------------------------------ head / loss
def test_head_and_aamloss_match_reference_code(ref_head):
    g = ref_head
    labels = torch.from_numpy(g["labels"])
    for margin, ls, easy in [(0.0, 0.0, False), (0.2, 0.0, False), (0.3, 0.1, False), (0.2, 0.0, True)]:
        e = torch.from_numpy(g["emb"]).requires_grad_(True)
        w = torch.from_numpy(g["W"]).requires_grad_(True)
        logits = head.cosine_logits(e, w)
        close(logits.detach().numpy(), g["logits"], 1e-12)
        loss = head.aam_loss(logits, labels, margin=margin, scale=32.0, easy_margin=easy, label_smoothing=ls)
        loss.backward()
        tag = f"m{margin}_ls{ls}_easy{int(easy)}"
        assert abs(loss.item() - float(g[f"loss_{tag}"])) < 1e-10
        close(e.grad.numpy(), g[f"demb_{tag}"])
        close(w.grad.numpy(), g[f"dW_{tag}"])
    p = head.aam_params(0.25)
    close([p["cos_m"], p["sin_m"], p["th"], p["mmm"]], g["update_0.25"], 1e-15)
    # AMLoss / ARMLoss / CELoss (loss/amloss.py, armloss.py, celoss.py)
    for kind, margin, ls in [("AM", 0.2, 0.0), ("AM", 0.35, 0.1), ("ARM", 0.2, 0.0), ("ARM", 0.1, 0.1), ("CE", 0.0, 0.0), ("CE", 0.0, 0.1)]:
        e = torch.from_numpy(g["emb"]).requires_grad_(True)
        w = torch.from_numpy(g["W"]).requires_grad_(True)
        loss = head.margin_head_loss(head.cosine_logits(e, w), labels, kind, margin=margin, scale=30.0, label_smoothing=ls)
        loss.backward()
        tag = f"{kind}_m{margin}_ls{ls}"
        assert abs(loss.item() - float(g[f"loss_{tag}"])) < 1e-10, tag
        close(e.grad.numpy(), g[f"demb_{tag}"])
        close(w.grad.numpy(), g[f"dW_{tag}"])
    # SphereFace2 (loss/sphereface2.py)
    for mt, margin, lam, t in [("C", 0.2, 0.7, 3), ("A", 0.15, 0.7, 3), ("C", 0.3, 0.5, 2)]:
        e = torch.from_numpy(g["emb"]).requires_grad_(True)
        w = torch.from_numpy(g["W"]).requires_grad_(True)
        loss = head.margin_head_loss(head.cosine_logits(e, w), labels, f"SF2{mt}{t}", margin=margin, scale=32.0, label_smoothing=lam)
        loss.backward()
        tag = f"SF2{mt}_m{margin}_l{lam}_t{t}"
        assert abs(loss.item() - float(g[f"loss_{tag}"])) < 1e-9 * max(1.0, abs(loss.item())), tag
        close(e.grad.numpy(), g[f"demb_{tag}"])
        close(w.grad.numpy(), g[f"dW_{tag}"])
    # SubCenterLoss (loss/subcenterloss.py) over K sub-centres per class
    for K, margin, ls, easy in [(3, 0.2, 0.0, False), (3, 0.3, 0.1, False), (2, 0.2, 0.0, True)]:
        e = torch.from_numpy(g["emb"]).requires_grad_(True)
        w = torch.from_numpy(g["W"][:, :156].copy()).requires_grad_(True)
        loss = head.margin_head_loss(head.cosine_logits(e, w), labels % (156 // K), f"SUB{K}{'e' if easy else ''}", margin=margin, scale=32.0,
                                     label_smoothing=ls)
        loss.backward()
        tag = f"SUB_K{K}_m{margin}_ls{ls}_easy{int(easy)}"
        assert abs(loss.item() - float(g[f"loss_{tag}"])) < 1e-10, tag
        close(e.grad.numpy(), g[f"demb_{tag}"])
        close(w.grad.numpy(), g[f"dW_{tag}"])


def test_train_step_matches_reference_code(golden_dir):
    """Train-mode forward (batch statistics), classifier, AAMLoss and autograd backward of the reference graph."""
    g = np.load(f"{golden_dir}/ref_train.npz")
    W = ecapa.make_ecapa_weights(seed=1000, dtype=torch.float64)
    loss, grads, new_stats, logits = otrain.train_step_grads(torch.from_numpy(g["feats"]), torch.from_numpy(g["labels"]), W,
                                                             torch.from_numpy(g["Wcls"]), margin=0.2, scale=32.0)
    assert abs(loss.item() - float(g["loss"])) < 1e-10
    close(logits.numpy(), g["logits"])
    close(grads["classifier.weight"].numpy(), g["grad_classifier.weight"], 1e-9)
    for k in g.files:
        if k.startswith("grad_") and k != "grad_classifier.weight":
            name = k[len("grad_"):]
            close(tap_slice(grads[name]), g[k], 1e-9)
            assert abs(float(grads[name].norm()) - float(g["gradnorm_" + name])) <= 1e-9 * max(1.0, float(g["gradnorm_" + name]))
        if k.startswith("stat_"):
            close(new_stats[k[len("stat_"):]].numpy(), g[k])


# ------------------------------------------------------------------------------------------------ schedules
def test_schedulers_match_reference_code(golden_dir):
    from ppvector.optimizer.scheduler import MarginScheduler, cosine_decay_with_warmup  # the product's host mirror
    g = np.load(f"{golden_dir}/ref_sched.npz")
    for name, kw in {"a": dict(learning_rate=1e-3, step_per_epoch=7, fix_epoch=6, warmup_epoch=2, min_lr=1e-5),
                     "b": dict(learning_rate=0.01, step_per_epoch=3, fix_epoch=10, warmup_epoch=5, min_lr=0.0)}.items():
        s = cosine_decay_with_warmup(**kw)
        vals = []
        for _ in range(len(g["lr_" + name])):
            vals.append(s.get_lr())
            s.step()
        close(vals, g["lr_" + name], 1e-15)

    class Crit:
        def update(self, margin):
            self.m = margin

    for name, kw in {"exp": dict(increase_start_epoch=3, fix_epoch=7, step_per_epoch=5, initial_margin=0.0, final_margin=0.3),
                     "lin": dict(increase_start_epoch=2, fix_epoch=4, step_per_epoch=4, initial_margin=0.1, final_margin=0.5,
                                 increase_type="linear")}.items():
        ms = MarginScheduler(criterion=Crit(), **kw)
        vals = []
        for i in range(len(g["margin_" + name])):
            ms.step()
            vals.append(ms.get_margin())
            inc0 = kw["increase_start_epoch"] * kw["step_per_epoch"]
            fix = kw["fix_epoch"] * kw["step_per_epoch"]
            want = otrain.margin_at(i, inc0, fix, kw["initial_margin"], kw["final_margin"], kw.get("increase_type", "exp"))
            assert abs(want - g["margin_" + name][i]) < 1e-15
        close(vals, g["margin_" + name], 1e-15)


# ------------------------------------------------------------------------------------------------ fixture provenance
def array_digest(a):
    """dtype, shape and SHA-256 of the bytes of one array (same recipe as tests/golden/make_ref_fixtures.py)."""
    a = np.ascontiguousarray(a)
    return {"dtype": a.dtype.str, "shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}


def test_fixtures_match_the_recorded_reference_run(golden_dir):
    """ref_digests.json holds the digest of every array the reference's own code computed when make_ref_fixtures.py last
    wrote the fixtures (its --check mode re-runs the reference and compares values).  The committed fixtures must be exactly
    those arrays: none was edited after that run."""
    want = json.load(open(f"{golden_dir}/ref_digests.json"))
    assert sorted(want) == ["ref_head.npz", "ref_models.npz", "ref_sched.npz", "ref_train.npz"]
    for fn, arrays in want.items():
        got = np.load(f"{golden_dir}/{fn}")
        assert sorted(got.files) == sorted(arrays), (fn, set(got.files) ^ set(arrays))
        for k, d in arrays.items():
            assert array_digest(got[k]) == d, (fn, k)
