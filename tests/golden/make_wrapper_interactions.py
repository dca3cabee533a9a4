"""What the reference's own wrappers (simmim.SimMIM, mae.MAE, mpp.MPP, distill.DistillWrapper -- unmodified, over the numpy
TensorFlow stand-in of oracle/tf_shim.py) do to their encoder, stored so that tests/test_wrappers_over_dropin.py can check the
drop-in against it without a reference checkout.

    python tests/golden/make_wrapper_interactions.py --reference <vit-tensorflow checkout> [--force]

For each wrapper this runs, with the same weights and the same random stream, (a) the wrapper around the reference's own ViT and
(b) the wrapper around vit_tensorflow_b200.ViT / DistillableViT (engine calls answered by tests/fake_engine.py), each encoder
behind a recording proxy that logs every attribute the wrapper reads and every call it makes on the encoder: the path from the
encoder, the arguments and what came back.  It asserts that both runs make the same interactions with the same results and that
the wrapper's loss (MPP: the logits it computes from the encoder's output; DistillWrapper: its output) agrees, then stores run
(a) in wrapper_interactions__refshim.npz: `meta` (JSON, one event list per wrapper) and the arrays the events name.

An array the test can regenerate is stored as a reference to it: "img" (the test's input images), "img_patches" (those images
cut into 16 x 16 patches, 'b (h p1) (w p2) c -> b (h w) (p1 p2 c)'), "w:<name>" (a weight) or "result:<i>" (what event i
returned).  An argument most of whose rows (last axis) are rows of one of those is stored as that reference, the source row
of each of its rows and its other, distinct rows (MPP's masked input: the image's patches, some replaced by other patches of
the same image or by the mask token).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import oracle  # noqa: E402
import fake_engine  # noqa: E402
from oracle import ref_bind, tf_shim  # noqa: E402
from test_wrappers_over_dropin import CFG, IMG, KW, W, img_patches  # noqa: E402

OUT = os.path.join(HERE, "wrapper_interactions__refshim.npz")
TOL = 1e-5            # |ours - reference| on every value an interaction returns (float32 computations of the same function)


class Recorder:
    """Stands in for an encoder (or a part of it) and logs what the wrapper does with it."""

    def __init__(self, obj, path, log):
        object.__setattr__(self, "_obj", obj)
        object.__setattr__(self, "_path", path)
        object.__setattr__(self, "_log", log)

    def _wrap(self, value, path):
        if isinstance(value, np.ndarray) or np.isscalar(value) or value is None:
            self._log.append(dict(op="get", path=path, value=value))
            return value
        return Recorder(value, path, self._log)

    def __getattr__(self, name):
        return self._wrap(getattr(self._obj, name), self._path + [["attr", name]])

    def __getitem__(self, key):
        if isinstance(key, slice):
            return [self[i] for i in range(len(self._obj))[key]]
        i = key % len(self._obj)
        return self._wrap(self._obj[i], self._path + [["item", i]])

    def __len__(self):
        return len(self._obj)

    def __call__(self, *args, **kwargs):
        result = self._obj(*args, **kwargs)
        self._log.append(dict(op="call", path=self._path, args=list(args), kwargs=kwargs, result=result))
        return result


def _np(v):
    return np.asarray(v, dtype=np.float32) if isinstance(v, np.ndarray) else v


def _same_event(a, b):
    assert a["op"] == b["op"] and a["path"] == b["path"], (a["op"], a["path"], b["op"], b["path"])
    pairs = [(a["value"], b["value"])] if a["op"] == "get" else \
        list(zip(a["args"], b["args"])) + [(a["kwargs"][k], b["kwargs"][k]) for k in a["kwargs"]] + [(a["result"], b["result"])]
    assert a["op"] == "get" or sorted(a["kwargs"]) == sorted(b["kwargs"])
    for x, y in pairs:
        x, y = (list(x), list(y)) if isinstance(x, tuple) else ([x], [y])
        for u, v in zip(x, y):
            if isinstance(u, np.ndarray):
                assert u.shape == np.shape(v) and np.abs(_np(u) - _np(v)).max() <= TOL, (a["path"], np.abs(_np(u) - _np(v)).max())
            else:
                assert u == v, (a["path"], u, v)


class _Store:
    def __init__(self, name):
        self.name, self.arrays, self.known = name, {}, {"img": IMG, "img_patches": img_patches(IMG)}
        self.known.update({f"w:{k}": v for k, v in W.items()})

    def _put(self, tag, a):
        key = f"{self.name}/{len(self.arrays)}/{tag}"
        self.arrays[key] = a
        return key

    def value(self, v, is_result):
        if isinstance(v, tuple):
            return dict(tuple=[self.value(e, is_result) for e in v])
        if not isinstance(v, np.ndarray):
            return dict(py=list(v) if isinstance(v, tuple) else (v.item() if isinstance(v, np.generic) else v))
        a = _np(v)
        for token, k in self.known.items():
            if np.shape(k) == a.shape and np.array_equal(_np(k), a):
                return dict(ref=token)
        if not is_result and a.ndim >= 2:
            rows = a.reshape(-1, a.shape[-1])
            for token, k in self.known.items():
                if np.shape(k) != a.shape:
                    continue
                where = {r.tobytes(): i for i, r in reversed(list(enumerate(_np(k).reshape(-1, a.shape[-1]))))}
                extra = {}
                src = [where[r.tobytes()] if r.tobytes() in where else -1 - extra.setdefault(r.tobytes(), len(extra)) for r in rows]
                if len(extra) <= len(rows) // 4:
                    other = np.stack([np.frombuffer(b, np.float32) for b in extra]) if extra else np.zeros((0, a.shape[-1]), np.float32)
                    return dict(ref=token, rows=self._put("rows", np.array(src, np.int32)), other=self._put("other", other))
        return dict(array=self._put("array", a))

    def events(self, log):
        out = []
        for i, e in enumerate(log):
            if e["op"] == "get":
                out.append(dict(op="get", path=e["path"], value=self.value(e["value"], True)))
                continue
            ev = dict(op="call", path=e["path"], args=[self.value(a, False) for a in e["args"]],
                      kwargs={k: self.value(v, False) for k, v in e["kwargs"].items()}, result=self.value(e["result"], True))
            if isinstance(e["result"], np.ndarray):
                self.known[f"result:{i}"] = e["result"]
            out.append(ev)
        return out


def _ours(cls_name="ViT"):
    import vit_tensorflow_b200 as vb
    m = getattr(vb, cls_name)(**KW, precision="fp32")
    m.set_weights_dict(W)
    return m


def _wrapper_run(ref_dir, build, call, encoder):
    """One wrapper run around `encoder()` ("reference" or "ours"): (interaction log, wrapper value, engine calls)."""
    log = []
    with fake_engine.installed() as fake, tf_shim.installed(ref_dir):
        enc = ref_bind.build_model("vit", KW, W, IMG) if encoder == "reference" else _ours()
        tf_shim.set_seed(77)
        wrapper = build(Recorder(enc, [], log))
        tf_shim.set_seed(78)
        value = call(wrapper)
        return log, value, [c[0] for c in fake.calls]


def simmim(enc):
    import simmim as m
    return m.SimMIM(image_size=64, encoder=enc, masking_ratio=0.5)


def mae(enc):
    import mae as m
    return m.MAE(image_size=64, encoder=enc, decoder_dim=32, masking_ratio=0.75, decoder_depth=1, decoder_heads=2, decoder_dim_head=16)


def mpp(enc):
    import mpp as m
    w = m.MPP(image_size=64, transformer=enc, patch_size=16, mask_prob=0.15, random_patch_prob=0.30, replace_prob=0.50)
    w.loss = lambda logits, img, mask: (w.__dict__.setdefault("seen", []).append(np.asarray(logits)), np.asarray(logits).mean())[1]
    return w


def _distill_run(ref_dir, encoder):
    log = []
    labels = np.eye(10, dtype=np.float32)[[1, 4, 7]]
    with fake_engine.installed() as fake, tf_shim.installed(ref_dir):
        import distill
        teacher = ref_bind.build_model("vit", KW, oracle.init_weights(CFG, 9), IMG)
        student = ref_bind.build_model("vit", KW, W, IMG, cls=distill.DistillableViT) if encoder == "reference" else _ours("DistillableViT")
        distill.DistillableViT = Recorder                    # distill.py:91 checks the student's type against the names in its module
        tf_shim.set_seed(5)
        wrapper = distill.DistillWrapper(teacher=teacher, student=Recorder(student, [], log), temperature=3, alpha=0.5, hard=False)
        value = np.asarray(wrapper([IMG, labels], training=False), dtype=np.float64)
        return log, value, [c[0] for c in fake.calls]


def main():
    if "--reference" not in sys.argv:
        raise SystemExit(__doc__)
    ref_dir = os.path.join(sys.argv[sys.argv.index("--reference") + 1], "vit_tensorflow")
    if not os.path.isdir(ref_dir):
        raise SystemExit(f"{ref_dir} not found")
    if os.path.exists(OUT) and "--force" not in sys.argv:
        raise SystemExit("fixture exists; pass --force to regenerate it")
    call = lambda w: w(IMG, training=False)                       # noqa: E731
    meta, arrays = dict(generator="tests/golden/make_wrapper_interactions.py", wrappers={}), {}
    for name in ("simmim", "mae", "mpp", "distill"):
        if name == "distill":
            runs = {e: _distill_run(ref_dir, e) for e in ("reference", "ours")}
        else:
            get = (lambda w: (call(w), w.seen[0])[1]) if name == "mpp" else call     # MPP: the logits it computes from the encoder output
            runs = {e: _wrapper_run(ref_dir, globals()[name], get, e) for e in ("reference", "ours")}
        (ref_log, ref_value, ref_calls), (our_log, our_value, our_calls) = runs["reference"], runs["ours"]
        assert len(ref_log) == len(our_log), (name, len(ref_log), len(our_log))
        for a, b in zip(ref_log, our_log):
            _same_event(a, b)
        assert ref_calls == [] and np.isfinite(our_value).all()
        assert np.abs(np.asarray(our_value, np.float64) - np.asarray(ref_value, np.float64)).max() < (1e-6 if name in ("simmim", "mae") else 1e-5), name
        store = _Store(name)
        meta["wrappers"][name] = dict(events=store.events(ref_log), engine_calls=our_calls)
        arrays.update(store.arrays)
        print(f"{name}: {len(ref_log)} interactions, engine calls {our_calls}")
    np.savez_compressed(OUT, meta=json.dumps(meta, sort_keys=True), **arrays)
    print(f"{OUT}: {len(arrays)} arrays, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
