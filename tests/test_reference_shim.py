"""The oracle pinned on the REFERENCE'S OWN CODE.

TensorFlow is not installable here, but the reference is pure Python over `tensorflow` + `einops`: oracle/tf_shim.py puts a
numpy implementation of the ~35 TensorFlow / Keras entry points it calls into sys.modules, and the unmodified modules of
the reference's vit_tensorflow package then run as written.  Three layers of checks:

1. the stand-in's primitives against PyTorch's independent operators (Dense / LayerNormalization eps 1e-3 / softmax / exact
   GELU / extract_patches SAME / Keras `training` plumbing) -- what remains ASSUMED about TensorFlow is exactly this list;
2. the reference's code, recorded: every model class of SURVEY.md section 8 (a) and (f), constructed by the reference's own
   `__init__`, weights loaded by Keras attribute path, `model(img, training=False)` == oracle.forward_numpy to 1e-12 in
   float64, and the reference's constructor / call signatures and constructor errors == ours.  What the reference returned is
   stored in tests/golden/reference_outputs__refshim.npz and reference_boundary.json (tests/golden/make_reference_outputs.py
   ran it), so these checks need no reference checkout;
3. the committed fixtures tests/golden/*__refshim.npz (the same outputs, stored so that they travel) == the oracle, for the
   small cases and for every BASELINE.json configuration at its own size.  The GPU tests compare the CUDA engine with these.
"""
import glob
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
from oracle import ref_torch, spec_numpy, tf_shim
from cases import (CALL_PAIRS, CTOR_ERROR_CASES, FULL, NO_DEFAULT, RANDOM_KINDS, RANDOM_SEEDS, README, REFERENCE_PAIRS, SMALL,
                   error_case_id, random_configuration)

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture
def f64():
    tf_shim.set_dtype(np.float64)
    yield
    tf_shim.set_dtype(np.float32)


# ------------------------------------------------------------------------------------------ 1. primitives vs torch
def test_shim_dense_layernorm_softmax_gelu_against_torch(f64):
    rng = np.random.default_rng(0)
    with tf_shim.installed() as tf:
        import tensorflow.keras.layers as nn
        x = rng.standard_normal((3, 7, 10))
        d = nn.Dense(units=6)
        d(x)                                                               # builds kernel [10, 6] + bias [6]
        k, b = rng.standard_normal((10, 6)), rng.standard_normal(6)
        d.set_weights([k, b])
        np.testing.assert_allclose(d(x), F.linear(torch.from_numpy(x), torch.from_numpy(k).T, torch.from_numpy(b)).numpy(), atol=1e-12)
        assert d.kernel.shape == (10, 6) and nn.Dense(units=4, use_bias=False)(x).shape == (3, 7, 4)
        ln = nn.LayerNormalization()
        ln(x)
        g, be = 1 + 0.3 * rng.standard_normal(10), rng.standard_normal(10)
        ln.set_weights([g, be])
        ref = F.layer_norm(torch.from_numpy(x), (10,), torch.from_numpy(g), torch.from_numpy(be), eps=1e-3).numpy()
        np.testing.assert_allclose(ln(x), ref, atol=1e-12)                 # Keras default epsilon = 1e-3 (NOT torch's 1e-5)
        assert np.abs(ln(x) - F.layer_norm(torch.from_numpy(x), (10,), torch.from_numpy(g), torch.from_numpy(be)).numpy()).max() > 1e-5
        np.testing.assert_allclose(nn.Softmax()(x), torch.softmax(torch.from_numpy(x), -1).numpy(), atol=1e-14)
        np.testing.assert_allclose(tf.nn.softmax(x, axis=-1), nn.Softmax()(x), atol=0)
        gelu = 0.5 * x * (1.0 + tf.math.erf(x / tf.cast(1.4142135623730951, x.dtype)))     # the reference's expression, vit.py:35
        np.testing.assert_allclose(gelu, F.gelu(torch.from_numpy(x)).numpy(), atol=1e-14)
        # tf.einsum ignores blanks; tf.matmul broadcasts batch dimensions (vit_with_patch_merger.py:51); tf.split in equal parts
        q = rng.standard_normal((2, 3, 5, 4))
        np.testing.assert_allclose(tf.einsum('b h i d, b h j d -> b h i j', q, q), torch.einsum('bhid,bhjd->bhij', torch.from_numpy(q), torch.from_numpy(q)).numpy(), atol=1e-12)
        m = tf.matmul(rng.standard_normal((4, 10)), tf.transpose(x, perm=[0, 2, 1]))
        assert m.shape == (3, 4, 7)
        a, b2, c = tf.split(x[..., :9], num_or_size_splits=3, axis=-1)
        assert a.shape == (3, 7, 3) and np.array_equal(np.concatenate([a, b2, c], -1), x[..., :9])


@pytest.mark.parametrize("H,W,k,s", [(32, 32, 7, 4), (8, 8, 3, 2), (9, 13, 3, 2), (7, 7, 3, 2), (16, 16, 3, 1), (5, 6, 7, 4)])
def test_shim_extract_patches_same_against_torch_unfold(f64, H, W, k, s):
    """tf.image.extract_patches(padding='SAME') (t2t.py:43) against F.unfold on an explicitly padded image: total padding
    max((ceil(in/s)-1)*s + k - in, 0), smaller half first; patch vector (row, col, channel)."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, H, W, 3))
    with tf_shim.installed() as tf:
        got = tf.image.extract_patches(x, sizes=[1, k, k, 1], strides=[1, s, s, 1], rates=[1, 1, 1, 1], padding='SAME')
    oh, ow = -(-H // s), -(-W // s)
    th, tw = max((oh - 1) * s + k - H, 0), max((ow - 1) * s + k - W, 0)
    xt = F.pad(torch.from_numpy(x).permute(0, 3, 1, 2), (tw // 2, tw - tw // 2, th // 2, th - th // 2))
    u = F.unfold(xt, kernel_size=k, stride=s)                               # [b, C*k*k, L], channel slowest
    u = u.reshape(2, 3, k, k, -1)[..., :].permute(0, 4, 2, 3, 1)            # [b, L', k, k, C]
    # unfold may produce more positions than ceil(in / s) when the padded extent allows: keep the first oh x ow grid
    L_h = (H + th - k) // s + 1
    L_w = (W + tw - k) // s + 1
    u = u.reshape(2, L_h, L_w, k * k * 3)[:, :oh, :ow]
    assert got.shape == (2, oh, ow, k * k * 3)
    np.testing.assert_array_equal(got, u.numpy())
    np.testing.assert_array_equal(got, spec_numpy.extract_patches_same(x, k, s))


def test_shim_extract_patches_reproduces_the_tensorflow_api_docs_example():
    """The worked example of the `tf.image.extract_patches` API documentation: a 10 x 10 image holding 1..100, 3 x 3 patches, stride 5.
    'VALID' gives the four patches below; with 'SAME' the output grid is ceil(10 / 5) = 2 as well and the total padding
    max((2 - 1) * 5 + 3 - 10, 0) = 0, so the result is the same -- a known answer for both the patch-vector order (row, column,
    channel) and the padding rule."""
    img = np.arange(1, 101, dtype=np.float32).reshape(1, 10, 10, 1)
    want = np.array([[[[1, 2, 3, 11, 12, 13, 21, 22, 23], [6, 7, 8, 16, 17, 18, 26, 27, 28]],
                      [[51, 52, 53, 61, 62, 63, 71, 72, 73], [56, 57, 58, 66, 67, 68, 76, 77, 78]]]], np.float32)
    with tf_shim.installed() as tf:
        for padding in ("VALID", "SAME"):
            got = tf.image.extract_patches(images=img, sizes=[1, 3, 3, 1], strides=[1, 5, 5, 1], rates=[1, 1, 1, 1], padding=padding)
            np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(spec_numpy.extract_patches_same(img, 3, 5), want)


def test_shim_keras_training_plumbing():
    """`training` resolution of Layer.__call__: explicit > enclosing call > the layer's own `call` default; Sequential forwards
    it to layers whose `call` names it (keras Sequential.call).  The reference relies on all three (vit.py:21,159-175)."""
    with tf_shim.installed():
        from tensorflow.keras import Sequential
        from tensorflow.keras.layers import Layer
        import tensorflow.keras.layers as nn
        seen = []

        class Probe(Layer):
            def call(self, x, training=True):
                seen.append(training)
                return x

        class NoArg(Layer):
            def call(self, x):
                return x

        class Outer(Layer):
            def __init__(self):
                super().__init__()
                self.inner = Sequential([Probe(), NoArg(), nn.Dropout(rate=0.5)])

            def call(self, x, training=True):
                return self.inner(x)                 # no explicit training: inherited from this call

        x = np.ones((4, 8), np.float32)
        o = Outer()
        assert np.array_equal(o(x, training=False), x) and seen == [False]
        y = o(x, training=True)
        assert seen == [False, True] and set(np.unique(y)) <= {0.0, 2.0} and (y == 0).any()
        o(x)                                         # nothing given anywhere: call-signature default (True)
        assert seen[-1] is True
        Probe()(x, training=False)
        assert seen[-1] is False


def test_shim_leaves_no_fake_tensorflow_behind():
    before = {n: sys.modules.get(n) for n in ("tensorflow", "tensorflow.keras", "einops.layers.tensorflow", "vit", "t2t")}
    with tf_shim.installed():
        import tensorflow as tf
        assert tf.__version__.endswith("numpy-shim")
    assert {n: sys.modules.get(n) for n in before} == before


# ------------------------------------------------------------------------------------------ 2. the reference's code, recorded
# What the reference's own classes returned for these inputs (tests/golden/make_reference_outputs.py ran them over the stand-in);
# the inputs are regenerated here from the same seeds.
@pytest.fixture(scope="module")
def recorded():
    z = np.load(os.path.join(GOLDEN, "reference_outputs__refshim.npz"))
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("gen", ["init_weights", "stress_weights"])
@pytest.mark.parametrize("name", sorted(SMALL))
def test_live_reference_equals_oracle(recorded, name, gen):
    case = SMALL[name]
    cfg = oracle.make_config(case["kind"], **{k: v for k, v in case.items() if k != "kind"})
    w = getattr(oracle, gen)(cfg, 21)
    img = oracle.make_image(cfg, 3, 22)
    got = recorded[f"oracle/{name}/{gen}"]
    ref = oracle.forward_numpy(img, w, cfg)
    assert got.dtype == np.float64 and got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12)
    np.testing.assert_allclose(ref_torch.forward(img, w, cfg), got, rtol=0, atol=5e-5)


def test_live_reference_smaller_image_and_tokens_entry(recorded):
    """vit.py:165 `pos_embedding[:, :(n + 1)]` on a smaller image, and `model.transformer(tokens)` at arbitrary n (what
    mae.py:69 / simmim.py:116 call) -- through the reference's own Transformer.call."""
    case = SMALL["vit_small"]
    cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
    w = oracle.stress_weights(cfg, 1)
    w64 = {k: v.astype(np.float64) for k, v in w.items()}
    img = oracle.make_image(cfg, 2, 3, h=32, w=48).astype(np.float64)
    x = np.random.default_rng(0).standard_normal((3, 9, cfg["dim"]))
    got, tok, pos = (recorded[f"tokens_entry/{k}"] for k in ("logits", "tokens", "pos"))   # pos: the wrappers' slicing (mae.py:54)
    np.testing.assert_allclose(got, oracle.forward_numpy(img, w, cfg), atol=1e-12)
    np.testing.assert_allclose(tok, spec_numpy.transformer_tokens(x, w, cfg), atol=1e-12)
    np.testing.assert_array_equal(pos, w64["pos_embedding"][:, 1:5])


@pytest.mark.parametrize("pool", ["cls", "mean"])
def test_live_reference_distillable_vit(recorded, pool):
    """distill.py:16-45 (DistillMixin.call) through the reference's DistillableViT."""
    case = dict(SMALL["vit_small"], pool=pool)
    cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
    w = oracle.stress_weights(cfg, 4)
    img = oracle.make_image(cfg, 2, 5).astype(np.float64)
    tok = np.random.default_rng(6).standard_normal((1, 1, cfg["dim"]))
    logits, dist, plain = (recorded[f"distill/{pool}/{k}"] for k in ("logits", "dist", "plain"))
    ref_l, ref_d = spec_numpy.forward_distill(img, tok, w, cfg)
    np.testing.assert_allclose(logits, ref_l, atol=1e-12)
    np.testing.assert_allclose(dist, ref_d, atol=1e-12)
    np.testing.assert_allclose(plain, oracle.forward_numpy(img, w, cfg), atol=1e-12)


def test_live_reference_efficient_vit_shell(recorded):
    """efficient.py:12-55 with the reference's own vit.Transformer injected: same logits as vit.ViT on the same weights."""
    case = SMALL["vit_small"]
    cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
    w = oracle.stress_weights(cfg, 7)
    img = oracle.make_image(cfg, 2, 8).astype(np.float64)
    np.testing.assert_allclose(recorded["efficient/logits"], oracle.forward_numpy(img, w, cfg), atol=1e-12)


def test_live_reference_dropout_is_identity_at_inference_and_random_in_training(recorded):
    """SURVEY.md 8 a15: with dropout > 0 the reference's `training=False` forward equals the dropout-free one; `training=True`
    (the signature default, vit.py:159) differs."""
    cfg = oracle.make_config("vit", **{k: v for k, v in SMALL["vit_small"].items() if k != "kind"})
    w = oracle.stress_weights(cfg, 9)
    img = oracle.make_image(cfg, 2, 10)
    inf, trn = recorded["dropout/inference"], recorded["dropout/training"]
    np.testing.assert_allclose(inf, oracle.forward_numpy(img, w, cfg), atol=2e-5)
    assert np.abs(trn - inf).max() > 1e-2


# ------------------------------------------------------------------------------------------ 3. committed fixtures
def _fixture(path):
    z = np.load(path)
    meta = json.loads(str(z["meta"]))
    case = meta["config"]
    for k in ("image_size", "patch_size", "t2t_layers"):            # json turned tuples into lists
        if isinstance(case.get(k), list):
            case[k] = tuple(tuple(e) if isinstance(e, list) else e for e in case[k])
    cfg = oracle.make_config(case["kind"], **{k: v for k, v in case.items() if k != "kind"})
    w = getattr(oracle, meta["weights"])(cfg, meta["weight_seed"])
    img = oracle.make_image(cfg, meta["batch"], meta["image_seed"])
    return z, cfg, w, img


def test_every_case_has_a_reference_fixture():
    have = {os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, "*__refshim.npz"))}
    want = {f"{n}__{g}__refshim.npz" for n in list(SMALL) + list(FULL) + list(README) for g in ("init_weights", "stress_weights")}
    assert want <= have, sorted(want - have)


@pytest.mark.parametrize("gen", ["init_weights", "stress_weights"])
@pytest.mark.parametrize("name", sorted(SMALL))
def test_reference_fixture_equals_oracle_small(name, gen):
    z, cfg, w, img = _fixture(os.path.join(GOLDEN, f"{name}__{gen}__refshim.npz"))
    ref = oracle.forward_numpy(img, w, cfg)
    np.testing.assert_allclose(z["logits_ref_f64"], ref, rtol=0, atol=1e-12)
    np.testing.assert_allclose(z["logits_ref_f32"], ref, rtol=0, atol=2e-5)
    np.testing.assert_allclose(np.load(os.path.join(GOLDEN, f"{name}__{gen}.npz"))["logits_f64"], z["logits_ref_f64"], rtol=0, atol=1e-12)


@pytest.mark.parametrize("gen", ["init_weights", "stress_weights"])
@pytest.mark.parametrize("name", sorted(FULL) + sorted(README))
def test_reference_fixture_equals_oracle_at_config_size(name, gen):
    """BASELINE.json configs[1..4] at their own width / depth / heads and the README's CrossViT / T2TViT examples at theirs, batch 2:
    the reference's code (float32) against the torch-CPU restatement the GPU config-size test uses as its checker."""
    z, cfg, w, img = _fixture(os.path.join(GOLDEN, f"{name}__{gen}__refshim.npz"))
    ref = ref_torch.forward(img, w, cfg)
    assert z["logits_ref_f32"].shape == ref.shape == (2, 1000)
    np.testing.assert_allclose(z["logits_ref_f32"], ref, rtol=0, atol=5e-5)


# ------------------------------------------------------------------------------------------ 4. the boundary (SURVEY.md 8b)
# The reference's signatures and constructor errors, as recorded from its own classes by tests/golden/make_reference_outputs.py.
@pytest.fixture(scope="module")
def boundary():
    with open(os.path.join(GOLDEN, "reference_boundary.json")) as fh:
        return json.load(fh)


def _params(recorded_params):
    """[(name, kind name, default)] of a recorded parameter list; defaults are stored as literals."""
    import ast
    import inspect
    return [(n, k, inspect.Parameter.empty if d == NO_DEFAULT else ast.literal_eval(d)) for n, k, d in recorded_params]


@pytest.mark.parametrize("ours,mod,theirs", REFERENCE_PAIRS)
def test_live_constructor_signature_equals_the_reference(boundary, ours, mod, theirs):
    """The drop-in boundary is the constructor + call surface (SURVEY.md 8b): every positional-or-keyword parameter of the
    reference's `__init__` -- name, position, default -- is one of ours; what we add (precision / device / seed) is keyword-only."""
    import inspect
    import vit_tensorflow_b200 as vb
    ref_params = _params(boundary["constructor"][f"{mod}.{theirs}"])
    our_params = list(inspect.signature(getattr(vb, ours).__init__).parameters.values())[1:]
    pos = [p for p in our_params if p.kind is inspect.Parameter.POSITIONAL_OR_KEYWORD]
    assert [(p.name, p.default) for p in pos] == [(n, d) for n, _, d in ref_params]
    extra = [p for p in our_params if p.kind is not inspect.Parameter.POSITIONAL_OR_KEYWORD]
    assert all(p.kind is inspect.Parameter.KEYWORD_ONLY for p in extra) and {p.name for p in extra} <= {"precision", "device", "seed"}


@pytest.mark.parametrize("ours,mod,theirs,kw", CTOR_ERROR_CASES)
def test_live_constructor_errors_equal_the_reference(boundary, ours, mod, theirs, kw):
    """Same error behaviour at the boundary: whatever the reference's constructor raises for these kwargs (type and message), ours
    raises too -- before any engine call, so this runs without a GPU."""
    import vit_tensorflow_b200 as vb
    ref_exc = boundary["constructor_errors"][error_case_id(ours, kw)]
    with pytest.raises(Exception) as our_exc:
        getattr(vb, ours)(**kw)
    t = type(our_exc.value)
    assert f"{t.__module__}.{t.__qualname__}" == ref_exc["type"] and str(our_exc.value) == ref_exc["message"]


@pytest.mark.parametrize("ours,mod,theirs", CALL_PAIRS)
def test_live_call_signature_equals_the_reference(boundary, ours, mod, theirs):
    """`model(img, training=True, **kwargs)` (vit.py:159): parameter names, order, defaults and the **kwargs catch-all of the
    reference's `call` are those of our `__call__` (which is also reachable as `.call`, as on a Keras model)."""
    import inspect
    import vit_tensorflow_b200 as vb
    ref = _params(boundary["call"][f"{mod}.{theirs}"])
    cls = getattr(vb, ours)
    mine = list(inspect.signature(cls.__call__).parameters.values())[1:]
    assert [(p.name, p.kind.name, p.default) for p in mine] == ref
    assert cls.call is cls.__call__ or inspect.signature(cls.call) == inspect.signature(cls.__call__)


# ------------------------------------------------------------------------------------------ 5. random configurations
@pytest.mark.parametrize("kind", RANDOM_KINDS)
def test_live_reference_equals_oracle_on_random_configurations(recorded, kind):
    """40 seeded random configurations per model class (cases.random_configuration): the reference's code == the float64 spec to
    1e-11 on each (the seeds are fixed, so a failure names a reproducible configuration)."""
    drawn = json.loads(str(recorded["meta"]))["random"]
    for seed in range(RANDOM_SEEDS):
        case, cfg = random_configuration(kind, seed)
        assert json.loads(json.dumps(case)) == drawn[f"{kind}/{seed}"], (seed, case)      # the recorded draw is this draw
        w = oracle.stress_weights(cfg, seed)
        img = oracle.make_image(cfg, 2, seed + 1)
        got = recorded[f"random/{kind}/{seed}"]
        ref = oracle.forward_numpy(img, w, cfg)
        assert got.shape == ref.shape, (seed, case)
        assert np.abs(got - ref).max() <= 1e-11 * max(1.0, np.abs(ref).max()), (seed, case, float(np.abs(got - ref).max()))
        if seed < 8:
            assert np.abs(ref_torch.forward(img, w, cfg) - got).max() <= 2e-4 * max(1.0, np.abs(ref).max()), (seed, case)
