"""SURVEY.md 8 (f1): the host classes as a drop-in ENCODER for the reference's own wrappers -- checked by running those wrappers.

Two test doubles make this possible on a CPU box: tests/fake_engine.py answers the C-ABI calls of the host classes with the
oracle (the product has no CPU path; the double exists so that the Python between the user and the C-ABI -- kwargs, ctypes
marshalling, attribute surface -- runs here), and oracle/tf_shim.py lets the reference's modules import without TensorFlow.

* host classes over the double: every stage entry goes through the real marshalling code and reproduces the oracle; what comes
  back answers `.numpy()` like the eager tensors the reference returns; `patch_embedding.layers[1].weights` exists;
* the reference's wrappers: the UNMODIFIED `simmim.SimMIM`, `mae.MAE`, `mpp.MPP` and `distill.DistillWrapper`, constructed
  around (a) the reference's own ViT and (b) our ViT carrying the same weights, with the same random stream, give the same
  loss, i.e. every attribute and call those wrappers make on their encoder (mae.py:32-38,49-69, simmim.py:74-80,88-125,
  mpp.py:149,200-212, distill.py:96-117) works on the drop-in and means the same thing.  tests/golden/make_wrapper_interactions.py
  checks that where the reference checkout exists and records run (a); the tests below replay it on the drop-in.
"""
import json
import os

import numpy as np
import pytest

import oracle
import fake_engine
from oracle import spec_numpy

KW = dict(image_size=64, patch_size=16, num_classes=10, dim=64, depth=2, heads=4, mlp_dim=128, dim_head=16)
CFG = oracle.make_config("vit", **KW)
W = oracle.stress_weights(CFG, 3)
IMG = oracle.make_image(CFG, 3, 4)


def _ours(cls_name="ViT", **extra):
    import vit_tensorflow_b200 as vb
    m = getattr(vb, cls_name)(**{**KW, **extra}, precision="fp32")
    m.set_weights_dict(W)
    return m


# ------------------------------------------------------------------------------------------ host classes over the double
def test_host_marshalling_reproduces_the_oracle_through_every_stage_entry():
    with fake_engine.installed() as fake:
        m = _ours()
        np.testing.assert_allclose(m(IMG, training=False), oracle.forward_numpy(IMG, W, CFG), atol=1e-6)
        small = oracle.make_image(CFG, 2, 5, h=32, w=48)                              # vit.py:165: fewer patches than positions
        np.testing.assert_allclose(m(small), oracle.forward_numpy(small, W, CFG), atol=1e-6)
        tok = m.forward_embed(IMG)
        np.testing.assert_allclose(tok, spec_numpy.embed_tokens(IMG, W, CFG), atol=1e-6)
        x = np.random.default_rng(0).standard_normal((2, 7, CFG["dim"])).astype(np.float32)
        np.testing.assert_allclose(m.transformer(x, training=False), spec_numpy.transformer_tokens(x, W, CFG), atol=1e-6)
        np.testing.assert_allclose(m.mlp_head(x), spec_numpy.head_logits(x, W, CFG), atol=1e-6)
        to_patch, patch_to_emb = m.patch_embedding.layers[:2]                        # mae.py:37
        p = to_patch(IMG, training=False)
        assert p.shape == (3, 16, 768) and patch_to_emb.weights[0].shape[0] == 768    # mae.py:38
        np.testing.assert_allclose(patch_to_emb(p, training=False), p.astype(np.float64) @ W["patch.kernel"] + W["patch.bias"], atol=1e-5)
        np.testing.assert_array_equal(m.patch_embedding(IMG), patch_to_emb(p))
        assert [c[0] for c in fake.calls][:4] == ["vb_create", "vb_finalize", "vb_forward", "vb_forward"]
        with pytest.raises(ValueError, match=r"expected \[batch, n, 64\]"):
            m.transformer(np.zeros((2, 7, 32), np.float32))                            # ADVICE round 1: no out-of-bounds host read


def test_results_answer_numpy_like_eager_tensors():
    """The wrappers call `.numpy()` on encoder outputs and on values derived from them (mae.py:63,66; simmim.py:119,125)."""
    with fake_engine.installed():
        m = _ours()
        out = m(IMG)
        for v in (out, m.transformer(np.zeros((1, 3, 64), np.float32)), m.patch_embedding.layers[0](IMG), m.pos_embedding, m.cls_token,
                  m.patch_embedding.layers[1](np.zeros((1, 2, 768), np.float32)) + m.pos_embedding[:, 1:3]):
            assert isinstance(v, np.ndarray) and type(v.numpy()) is np.ndarray and v.numpy().dtype == np.float32
        assert isinstance(out.max(), np.floating) and isinstance((out > 0).all(), (bool, np.bool_))   # reductions stay scalars
        with pytest.raises(ValueError):
            m.pos_embedding[0, 0, 0] = 1.0                                             # read-only view of the model's weight


def test_distillable_vit_over_the_double():
    with fake_engine.installed():
        m = _ours("DistillableViT")
        tok = np.random.default_rng(1).standard_normal((1, 1, CFG["dim"])).astype(np.float32)
        logits, dist = m(IMG, distill_token=tok, training=False)
        ref_l, ref_d = spec_numpy.forward_distill(IMG, tok, W, CFG)
        np.testing.assert_allclose(logits, ref_l, atol=1e-6)
        np.testing.assert_allclose(dist, ref_d, atol=1e-6)
        assert m.dim == 64 and m.num_classes == 10 and hasattr(logits, "numpy")       # distill.py:96-97


# ------------------------------------------------------------------------------------------ the reference's wrappers, replayed
# What the reference's unmodified wrappers did to the reference's own ViT -- every attribute read and every call, with its
# arguments and result -- is stored in tests/golden/wrapper_interactions__refshim.npz.  tests/golden/make_wrapper_interactions.py
# recorded it and, running each wrapper around our ViT as well, checked that the wrapper makes the same interactions there and
# ends with the same loss.  Here every interaction is replayed on our encoder and must give back what the reference's gave: the
# wrapper's computation is a function of those answers and its own seeded random stream, so equal answers are an equal loss.
REPLAY_TOL = 1e-5


def img_patches(img):
    """The images cut into 16 x 16 patches, 'b (h p1) (w p2) c -> b (h w) (p1 p2 c)' (one of the stored interactions' inputs)."""
    from einops import rearrange
    return rearrange(img, "b (h p1) (w p2) c -> b (h w) (p1 p2 c)", p1=16, p2=16)


@pytest.fixture(scope="module")
def interactions():
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "wrapper_interactions__refshim.npz"))
    return json.loads(str(z["meta"]))["wrappers"], {k: z[k] for k in z.files if k != "meta"}


def _replay(recorded, name, encoder):
    """Replays wrapper `name`'s recorded interactions on `encoder`; returns the number replayed."""
    wrappers, arrays = recorded
    known = {"img": IMG, "img_patches": img_patches(IMG), **{f"w:{k}": v for k, v in W.items()}}

    def arg(d):
        if "tuple" in d:
            return tuple(arg(e) for e in d["tuple"])
        if "py" in d:
            return tuple(d["py"]) if isinstance(d["py"], list) else d["py"]
        if "array" in d:
            return arrays[d["array"]]
        a = np.asarray(known[d["ref"]], dtype=np.float32)
        if "rows" in d:                               # each row: a row of the reference (>= 0) or one of the stored other rows
            base, other = a.reshape(-1, a.shape[-1]), arrays[d["other"]]
            a = np.stack([base[i] if i >= 0 else other[-1 - i] for i in arrays[d["rows"]]]).reshape(a.shape)
        return a

    def check(got, d, where):
        if "tuple" in d:
            assert isinstance(got, tuple) and len(got) == len(d["tuple"]), where
            for g, e in zip(got, d["tuple"]):
                check(g, e, where)
        elif "py" in d:
            assert (list(got) if isinstance(got, tuple) else got) == d["py"], (where, got, d["py"])
        else:
            want = arg(d)
            assert np.shape(got) == want.shape, where
            np.testing.assert_allclose(np.asarray(got, np.float32), want, rtol=0, atol=REPLAY_TOL, err_msg=str(where))

    events = wrappers[name]["events"]
    for i, e in enumerate(events):
        target = encoder
        for kind, step in e["path"]:
            target = getattr(target, step) if kind == "attr" else target[step]
        if e["op"] == "get":
            check(target, e["value"], (name, i, e["path"]))
            continue
        got = target(*[arg(a) for a in e["args"]], **{k: arg(v) for k, v in e["kwargs"].items()})
        check(got, e["result"], (name, i, e["path"]))
        if isinstance(got, np.ndarray):
            known[f"result:{i}"] = got                # later arguments built from this answer use ours, as the wrapper would
    return len(events)


def _replay_on_ours(interactions, name, cls_name="ViT"):
    with fake_engine.installed() as fake:
        n = _replay(interactions, name, _ours(cls_name))
        calls = [c[0] for c in fake.calls]
    assert n > 0 and calls == interactions[0][name]["engine_calls"]
    return calls


def test_live_simmim_over_the_dropin_encoder(interactions):
    """simmim.SimMIM around the drop-in (simmim.py:74-80,88-125): pos_embedding, patch_embedding.layers[:2] and their weights,
    to_patch / patch_to_emb / transformer on the wrapper's own inputs."""
    calls = _replay_on_ours(interactions, "simmim")
    assert calls == ["vb_create", "vb_finalize", "vb_to_patch", "vb_patch_to_emb", "vb_forward_tokens"]


def test_live_mae_over_the_dropin_encoder(interactions):
    calls = _replay_on_ours(interactions, "mae")
    assert calls[-1] == "vb_forward_tokens"                                         # the encoder saw only the unmasked quarter (mae.py:63-69)


def test_live_mpp_over_the_dropin_encoder(interactions):
    """mpp.py:200-212: Dense of `patch_embedding.layers[-1]` on masked patches, cls token, `pos_embedding[:, :(n + 1)]`, `dropout`,
    `transformer`."""
    calls = _replay_on_ours(interactions, "mpp")
    assert calls == ["vb_create", "vb_finalize", "vb_patch_to_emb", "vb_forward_tokens"]


def test_live_distill_wrapper_over_the_dropin_student(interactions):
    """distill.py:87-136: `student.dim`, `student.num_classes`, `student(img, distill_token=Variable, training=...)` ->
    (logits, distill_tokens).  (soft distillation only: the reference's hard branch feeds integer labels to
    categorical_crossentropy, distill.py:131-132, which fails on any encoder.)"""
    _replay_on_ours(interactions, "distill", "DistillableViT")


# ------------------------------------------------------------------------------------------ every host class over the double
@pytest.mark.parametrize("name", sorted(__import__("cases").SMALL))
def test_every_host_class_encodes_its_kwargs_losslessly(name):
    """kwargs -> VbConfig (`_create`) -> engine: decoding the VbConfig the host class built gives back exactly
    `oracle.make_config(kind, **kwargs)` (so nothing the reference's constructor takes is dropped on the way to the C-ABI), the
    weight list the engine reports is the oracle's (names, shapes, order) and the forward marshals the right buffers."""
    from cases import cfg_of
    from vit_tensorflow_b200 import from_config
    cfg = cfg_of(name)
    w = oracle.stress_weights(cfg, 3)
    img = oracle.make_image(cfg, 2, 4)
    with fake_engine.installed() as fake:
        m = from_config(cfg, precision="fp32")
        assert list(m.weight_specs().items()) == [(k, v[0]) for k, v in oracle.weight_specs(cfg).items()]
        decoded = fake.handles[m._h.value]["cfg"]
        raw = ("image_size", "patch_size", "patch_merge_layer")      # int-or-pair / None-or-int spellings of values the derived keys hold
        assert {k: v for k, v in decoded.items() if k not in raw} == {k: v for k, v in cfg.items() if k not in raw}
        m.set_weights_dict(w)
        np.testing.assert_allclose(m(img, training=False), oracle.forward_numpy(img, w, cfg), atol=1e-6)
        init = m.get_weights_dict()                                       # a fresh model's init follows the reference's distributions
        m2 = from_config(cfg, precision="fp32", seed=0)
        for k, v in m2.get_weights_dict().items():
            leaf = k.rsplit(".", 1)[-1]
            if leaf in ("bias", "beta"):
                assert not v.any()
            elif leaf == "gamma":
                assert (v == 1).all()
            elif leaf == "kernel":
                assert np.abs(v).max() <= np.sqrt(6.0 / sum(v.shape)) + 1e-6
        assert set(init) == set(m2.get_weights_dict())


def test_efficient_vit_and_t2t_with_injected_transformer_over_the_double():
    """efficient.py:12-55 / t2t.py:84-87: embed -> injected `transformer(tokens, training=...)` -> head, through the stage entries."""
    from vit_tensorflow_b200 import EfficientViT, T2TViT
    with fake_engine.installed():
        enc = _ours()
        ev = EfficientViT(image_size=64, patch_size=16, num_classes=10, dim=64, transformer=enc.transformer, precision="fp32")
        ev.set_weights_dict({k: v for k, v in W.items() if not k.startswith("layers.")})
        np.testing.assert_allclose(ev(IMG, training=False), oracle.forward_numpy(IMG, W, CFG), atol=1e-5)
        seen = []

        def probe(x, training=True):
            seen.append((x.shape, training))
            return x
        t2 = T2TViT(image_size=32, num_classes=10, dim=64, transformer=probe, t2t_layers=((3, 2), (3, 2)), precision="fp32")
        out = t2(oracle.make_image(dict(image_h=32, image_w=32, channels=3), 2, 1), training=False)
        assert out.shape == (2, 10) and seen == [((2, 65, 64), False)]
