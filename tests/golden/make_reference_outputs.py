"""What the reference's own code returns for the checks of tests/test_reference_shim.py, stored so that those checks run without
a reference checkout: the unmodified vit_tensorflow modules over the numpy TensorFlow stand-in of oracle/tf_shim.py.

    python tests/golden/make_reference_outputs.py --reference <vit-tensorflow checkout> [--force]

writes
    reference_outputs__refshim.npz  logits / token outputs of the reference's models for fixed seeds (float64 unless noted):
        oracle/<case>/<weights>            tests/cases.py SMALL cases, weight seed 21, image seed 22, batch 3
        tokens_entry/{logits,tokens,pos}   vit_small on a 32 x 48 image, `model.transformer(tokens)`, `pos_embedding[:, 1:5]`
        distill/<pool>/{logits,dist,plain} DistillableViT with a distill token, and without
        efficient/logits                   efficient.ViT around the reference's own vit.Transformer
        dropout/{inference,training}       float32, dropout 0.3 / emb_dropout 0.2, training=False / the default (True)
        random/<kind>/<seed>               tests/cases.py random_configuration(kind, seed), stress weights, batch 2
        meta                               JSON: the random configurations the logits belong to, and the generator
    reference_boundary.json         constructor / call signatures of the reference classes, and the exceptions its constructors
                                    raise for tests/cases.py CTOR_ERROR_CASES

The inputs are regenerated from their seeds by the tests; only the reference's outputs are stored.
"""
import importlib
import inspect
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import oracle  # noqa: E402
from oracle import ref_bind, tf_shim  # noqa: E402
from cases import (CALL_PAIRS, CTOR_ERROR_CASES, NO_DEFAULT, RANDOM_KINDS, RANDOM_SEEDS, REFERENCE_PAIRS, SMALL,  # noqa: E402
                   error_case_id, random_configuration)

OUTPUTS = os.path.join(HERE, "reference_outputs__refshim.npz")
BOUNDARY = os.path.join(HERE, "reference_boundary.json")


def encode_default(v):
    """A parameter default as text that ast.literal_eval turns back into an equal value."""
    import ast
    if v is inspect.Parameter.empty:
        return NO_DEFAULT
    assert ast.literal_eval(repr(v)) == v, v
    return repr(v)


def _logits(ref_dir, case, w, img, dtype=np.float64):
    kind, kw = ref_bind.ctor_kwargs(case)
    with tf_shim.installed(ref_dir):
        model = ref_bind.build_model(kind, kw, {k: v.astype(dtype) for k, v in w.items()}, img.astype(dtype))
        return ref_bind.to_numpy(model(img.astype(dtype), training=False))


def outputs(ref_dir):
    out, meta = {}, dict(generator="tests/golden/make_reference_outputs.py",
                         reference="vit_tensorflow (unmodified) over oracle/tf_shim.py", numpy=np.__version__, random={})
    tf_shim.set_dtype(np.float64)
    try:
        for name in sorted(SMALL):
            case = SMALL[name]
            cfg = oracle.make_config(case["kind"], **{k: v for k, v in case.items() if k != "kind"})
            for gen in ("init_weights", "stress_weights"):
                out[f"oracle/{name}/{gen}"] = _logits(ref_dir, case, getattr(oracle, gen)(cfg, 21), oracle.make_image(cfg, 3, 22))

        case = SMALL["vit_small"]
        cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
        w64 = {k: v.astype(np.float64) for k, v in oracle.stress_weights(cfg, 1).items()}
        img = oracle.make_image(cfg, 2, 3, h=32, w=48).astype(np.float64)
        kind, kw = ref_bind.ctor_kwargs(case)
        x = np.random.default_rng(0).standard_normal((3, 9, cfg["dim"]))
        with tf_shim.installed(ref_dir):
            model = ref_bind.build_model(kind, kw, w64, oracle.make_image(cfg, 1, 0).astype(np.float64))
            out["tokens_entry/logits"] = ref_bind.to_numpy(model(img, training=False))
            out["tokens_entry/tokens"] = ref_bind.to_numpy(model.transformer(x, training=False))
            out["tokens_entry/pos"] = ref_bind.to_numpy(model.pos_embedding[:, 1:5])

        for pool in ("cls", "mean"):
            case = dict(SMALL["vit_small"], pool=pool)
            cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
            w = oracle.stress_weights(cfg, 4)
            img = oracle.make_image(cfg, 2, 5).astype(np.float64)
            tok = np.random.default_rng(6).standard_normal((1, 1, cfg["dim"]))
            kind, kw = ref_bind.ctor_kwargs(case)
            with tf_shim.installed(ref_dir):
                import distill
                model = ref_bind.build_model("vit", kw, {k: v.astype(np.float64) for k, v in w.items()}, img, cls=distill.DistillableViT)
                logits, dist = model(img, distill_token=tok, training=False)
                out[f"distill/{pool}/logits"] = ref_bind.to_numpy(logits)
                out[f"distill/{pool}/dist"] = ref_bind.to_numpy(dist)
                out[f"distill/{pool}/plain"] = ref_bind.to_numpy(model(img, training=False))

        case = SMALL["vit_small"]
        cfg = oracle.make_config("vit", **{k: v for k, v in case.items() if k != "kind"})
        w = oracle.stress_weights(cfg, 7)
        img = oracle.make_image(cfg, 2, 8).astype(np.float64)
        with tf_shim.installed(ref_dir):
            import efficient
            import vit
            tr = vit.Transformer(cfg["dim"], cfg["depth"], cfg["heads"], cfg["dim_head"], cfg["mlp_dim"])
            kw = dict(image_size=case["image_size"], patch_size=case["patch_size"], num_classes=case["num_classes"], dim=case["dim"], transformer=tr)
            model = ref_bind.build_model("vit", kw, {k: v.astype(np.float64) for k, v in w.items()}, img, cls=efficient.ViT)
            out["efficient/logits"] = ref_bind.to_numpy(model(img, training=False))

        for kind in RANDOM_KINDS:
            for seed in range(RANDOM_SEEDS):
                case, cfg = random_configuration(kind, seed)
                meta["random"][f"{kind}/{seed}"] = case
                out[f"random/{kind}/{seed}"] = _logits(ref_dir, case, oracle.stress_weights(cfg, seed), oracle.make_image(cfg, 2, seed + 1))
    finally:
        tf_shim.set_dtype(np.float32)

    # float32, as the shim computes by default
    case = dict(SMALL["vit_small"], dropout=0.3, emb_dropout=0.2)
    cfg = oracle.make_config("vit", **{k: v for k, v in SMALL["vit_small"].items() if k != "kind"})
    w = oracle.stress_weights(cfg, 9)
    img = oracle.make_image(cfg, 2, 10)
    kind, kw = ref_bind.ctor_kwargs(case)
    with tf_shim.installed(ref_dir):
        model = ref_bind.build_model(kind, kw, w, img)
        out["dropout/inference"] = ref_bind.to_numpy(model(img, training=False))
        out["dropout/training"] = ref_bind.to_numpy(model(img))
    return out, meta


def boundary(ref_dir):
    d = dict(constructor={}, call={}, constructor_errors={})
    with tf_shim.installed(ref_dir):
        for _, mod, theirs in REFERENCE_PAIRS:
            params = list(inspect.signature(getattr(importlib.import_module(mod), theirs).__init__).parameters.values())[1:]
            d["constructor"][f"{mod}.{theirs}"] = [[p.name, p.kind.name, encode_default(p.default)] for p in params]
        for _, mod, theirs in CALL_PAIRS:
            params = list(inspect.signature(getattr(importlib.import_module(mod), theirs).call).parameters.values())[1:]
            d["call"][f"{mod}.{theirs}"] = [[p.name, p.kind.name, encode_default(p.default)] for p in params]
        for ours, mod, theirs, kw in CTOR_ERROR_CASES:
            try:
                getattr(importlib.import_module(mod), theirs)(**kw)
            except Exception as e:       # noqa: BLE001 -- whatever the reference raises is what is recorded
                t = type(e)
                d["constructor_errors"][error_case_id(ours, kw)] = dict(type=f"{t.__module__}.{t.__qualname__}", message=str(e))
            else:
                raise AssertionError(f"{mod}.{theirs}{kw} raised nothing")
    return d


def main():
    if "--reference" not in sys.argv:
        raise SystemExit(__doc__)
    ref_dir = os.path.join(sys.argv[sys.argv.index("--reference") + 1], "vit_tensorflow")
    if not os.path.isdir(ref_dir):
        raise SystemExit(f"{ref_dir} not found")
    if (os.path.exists(OUTPUTS) or os.path.exists(BOUNDARY)) and "--force" not in sys.argv:    # never rewritten silently
        raise SystemExit("fixtures exist; pass --force to regenerate them")
    out, meta = outputs(ref_dir)
    np.savez_compressed(OUTPUTS, meta=json.dumps(meta, sort_keys=True), **out)
    with open(BOUNDARY, "w") as fh:
        json.dump(boundary(ref_dir), fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(f"{OUTPUTS}: {len(out)} arrays, {os.path.getsize(OUTPUTS)} bytes; {BOUNDARY}: {os.path.getsize(BOUNDARY)} bytes")


if __name__ == "__main__":
    main()
