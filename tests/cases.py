"""Shared model configurations for the parity tests (small enough for the CPU oracle to finish in seconds)."""
import json

import numpy as np

import oracle

# BASELINE.json configs[0]: the numerics gate (C1).
C1 = dict(kind="vit", image_size=224, patch_size=16, num_classes=1000, dim=192, depth=1, heads=3, mlp_dim=768)

SMALL = {
    "vit_c1": C1,
    "vit_small": dict(kind="vit", image_size=64, patch_size=16, num_classes=10, dim=64, depth=2, heads=4, mlp_dim=128, dim_head=16),
    "vit_mean_rect": dict(kind="vit", image_size=(48, 64), patch_size=(8, 16), num_classes=7, dim=64, depth=1, heads=2,
                          mlp_dim=96, dim_head=32, pool="mean"),
    # widths that are multiples of neither 64 nor 8: every general (non-tcgen05, unaligned) kernel path of the bf16 engine
    "vit_odd_dims": dict(kind="vit", image_size=(40, 56), patch_size=8, num_classes=11, dim=50, depth=2, heads=3, mlp_dim=70,
                         dim_head=14, pool="mean"),
    "vit_noproj": dict(kind="vit", image_size=32, patch_size=8, num_classes=5, dim=64, depth=2, heads=1, mlp_dim=64, dim_head=64),
    "deepvit_small": dict(kind="deepvit", image_size=64, patch_size=16, num_classes=10, dim=64, depth=2, heads=4, mlp_dim=128, dim_head=16),
    "cait_small": dict(kind="cait", image_size=64, patch_size=16, num_classes=10, dim=64, depth=2, cls_depth=2, heads=4,
                       mlp_dim=128, dim_head=16),
    "crossvit_small": dict(kind="crossvit", image_size=64, num_classes=10, sm_dim=64, lg_dim=128, sm_patch_size=8,
                           lg_patch_size=16, sm_enc_depth=1, lg_enc_depth=2, sm_enc_heads=2, lg_enc_heads=2,
                           sm_enc_mlp_dim=64, lg_enc_mlp_dim=128, sm_enc_dim_head=32, lg_enc_dim_head=32,
                           cross_attn_depth=2, cross_attn_heads=2, cross_attn_dim_head=32, depth=2),
    "parallel_small": dict(kind="parallel_vit", image_size=64, patch_size=16, num_classes=10, dim=64, depth=2, heads=4, mlp_dim=128,
                           dim_head=16),
    "parallel_three_noproj": dict(kind="parallel_vit", image_size=32, patch_size=8, num_classes=5, dim=64, depth=2, heads=1,
                                  mlp_dim=64, dim_head=64, num_parallel_branches=3, pool="mean"),
    "merger_small": dict(kind="patch_merger_vit", image_size=64, patch_size=8, num_classes=10, dim=64, depth=4, heads=4, mlp_dim=128,
                         dim_head=16, patch_merge_layer=2, patch_merge_num_tokens=5),
    "merger_default_noproj": dict(kind="patch_merger_vit", image_size=(32, 48), patch_size=8, num_classes=6, dim=64, depth=2, heads=1,
                                  mlp_dim=96, dim_head=64),
    "t2t_small": dict(kind="t2t_vit", image_size=32, num_classes=10, dim=64, depth=2, heads=4, mlp_dim=128, dim_head=16,
                      t2t_layers=((3, 2), (3, 2))),
    "t2t_default_layers": dict(kind="t2t_vit", image_size=64, num_classes=7, dim=64, depth=1, heads=2, mlp_dim=64, dim_head=32,
                               pool="mean"),
    "crossvit_samedim": dict(kind="crossvit", image_size=32, num_classes=6, sm_dim=64, lg_dim=64, sm_patch_size=8,
                             lg_patch_size=16, sm_enc_depth=1, lg_enc_depth=1, sm_enc_heads=2, lg_enc_heads=2,
                             sm_enc_mlp_dim=64, lg_enc_mlp_dim=64, sm_enc_dim_head=32, lg_enc_dim_head=32,
                             cross_attn_depth=1, cross_attn_heads=2, cross_attn_dim_head=32, depth=1),
}

# Mid-size bf16 cases exercising the tcgen05 kernels at the real head / sequence geometry (n = 197, dh = 64).
MID = {
    "vit_mid": dict(kind="vit", image_size=224, patch_size=16, num_classes=1000, dim=256, depth=2, heads=4, mlp_dim=512),
    "parallel_mid": dict(kind="parallel_vit", image_size=224, patch_size=16, num_classes=100, dim=256, depth=2, heads=4, mlp_dim=512),
    "deepvit_mid": dict(kind="deepvit", image_size=224, patch_size=16, num_classes=100, dim=256, depth=2, heads=4, mlp_dim=512),
    "merger_mid": dict(kind="patch_merger_vit", image_size=224, patch_size=16, num_classes=100, dim=256, depth=4, heads=4, mlp_dim=512,
                       patch_merge_layer=2),
    "t2t_mid": dict(kind="t2t_vit", image_size=224, num_classes=100, dim=256, depth=2, heads=4, mlp_dim=512),
    "cait_mid": dict(kind="cait", image_size=224, patch_size=16, num_classes=100, dim=192, depth=2, cls_depth=2, heads=4,
                     mlp_dim=384, dim_head=48),
}

# BASELINE.json configs[1..4] (batch replaced by 2: the path has no cross-image op, see test_batch_independence)
FULL = {
    "c2_vit_b16_224": dict(kind="vit", image_size=224, patch_size=16, num_classes=1000, dim=768, depth=12, heads=12, mlp_dim=3072),
    "c3_deepvit_1024x24": dict(kind="deepvit", image_size=224, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16,
                               mlp_dim=4096),
    "c4_cait_s36_dh48": dict(kind="cait", image_size=224, patch_size=16, num_classes=1000, dim=384, depth=36, cls_depth=2, heads=8,
                             mlp_dim=1536, dim_head=48),
    "c4_cait_s36_dh64": dict(kind="cait", image_size=224, patch_size=16, num_classes=1000, dim=384, depth=36, cls_depth=2, heads=8,
                             mlp_dim=1536, dim_head=64),
    "c5_vit_l16_384": dict(kind="vit", image_size=384, patch_size=16, num_classes=1000, dim=1024, depth=24, heads=16, mlp_dim=4096),
}

# The reference README's usage examples of the two hot-path model classes BASELINE.json has no configuration for (CrossViT: SURVEY.md 8
# a14, README.md:327-345; T2TViT: 8 f3, README.md:208-216), at their own size, batch 2 -- the configurations bench.py --config
# crossvit_readme / t2t_readme time.
README = {
    "crossvit_readme": dict(kind="crossvit", image_size=256, num_classes=1000, depth=4, sm_dim=192, sm_patch_size=16, sm_enc_depth=2,
                            sm_enc_heads=8, sm_enc_mlp_dim=2048, lg_dim=384, lg_patch_size=64, lg_enc_depth=3, lg_enc_heads=8,
                            lg_enc_mlp_dim=2048, cross_attn_depth=2, cross_attn_heads=8),
    "t2t_readme": dict(kind="t2t_vit", image_size=224, num_classes=1000, dim=512, depth=5, heads=8, mlp_dim=512,
                       t2t_layers=((7, 4), (3, 2), (3, 2))),
}


# The drop-in classes and the reference classes they stand for: (our class, reference module, reference class).
REFERENCE_PAIRS = [("ViT", "vit", "ViT"), ("DeepViT", "deepvit", "DeepViT"), ("CaiT", "cait", "CaiT"), ("CrossViT", "cross_vit", "CrossViT"),
                   ("ParallelViT", "parallel_vit", "ViT"), ("T2TViT", "t2t", "T2TViT"), ("PatchMergerViT", "vit_with_patch_merger", "ViT"),
                   ("EfficientViT", "efficient", "ViT"), ("PatchMerger", "vit_with_patch_merger", "PatchMerger")]
CALL_PAIRS = REFERENCE_PAIRS + [("DistillableViT", "distill", "DistillableViT")]

# Constructor kwargs every one of which the reference's constructor rejects: (our class, reference module, reference class, kwargs).
CTOR_ERROR_CASES = [
    ("ViT", "vit", "ViT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32)),
    ("ViT", "vit", "ViT", dict(image_size=32, patch_size=16, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32, pool="max")),
    ("ViT", "vit", "ViT", dict(image_size=(32, 40), patch_size=(16, 16), num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32)),
    ("DeepViT", "deepvit", "DeepViT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32)),
    ("DeepViT", "deepvit", "DeepViT", dict(image_size=32, patch_size=16, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32, pool="sum")),
    ("CaiT", "cait", "CaiT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, depth=1, cls_depth=1, heads=2, mlp_dim=32)),
    ("CrossViT", "cross_vit", "CrossViT", dict(image_size=30, num_classes=4, sm_dim=32, lg_dim=32)),
    ("ParallelViT", "parallel_vit", "ViT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32)),
    ("T2TViT", "t2t", "T2TViT", dict(image_size=32, num_classes=4, dim=32)),
    ("T2TViT", "t2t", "T2TViT", dict(image_size=32, num_classes=4, dim=32, depth=1, heads=2, mlp_dim=32, pool="max")),
    ("PatchMergerViT", "vit_with_patch_merger", "ViT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, depth=2, heads=2, mlp_dim=32)),
    ("EfficientViT", "efficient", "ViT", dict(image_size=30, patch_size=16, num_classes=4, dim=32, transformer=None)),
    ("EfficientViT", "efficient", "ViT", dict(image_size=32, patch_size=16, num_classes=4, dim=32, transformer=None, pool="max")),
]

NO_DEFAULT = "<no default>"       # how tests/golden/reference_boundary.json spells a parameter without a default


def error_case_id(ours, kw):
    """The key of a CTOR_ERROR_CASES entry in tests/golden/reference_boundary.json."""
    return f"{ours} {json.dumps(kw, sort_keys=True)}"


RANDOM_KINDS = ["vit", "deepvit", "cait", "crossvit", "parallel_vit", "patch_merger_vit", "t2t_vit"]
RANDOM_SEEDS = 40


def random_case(kind, rng):
    """A random small constructor-kwargs set of `kind` (every shape-changing argument drawn, incl. the branches the hand-picked
    cases might miss: rectangular images, heads == 1 with dim_head == dim (no out-projection, vit.py:53), equal CrossViT widths
    (no ProjectInOut Dense, cross_vit.py:124), PatchMerger after the first / last layer, T2T kernel / stride combinations)."""
    heads = int(rng.choice([1, 2, 3]))
    dim_head = int(rng.choice([4, 8]))
    dim = heads * dim_head if (heads == 1 and rng.random() < 0.5) else int(rng.choice([8, 12, 20]))
    base = dict(num_classes=int(rng.integers(2, 7)), dim=dim, depth=int(rng.integers(1, 4)), heads=heads, mlp_dim=int(rng.choice([8, 24])),
                dim_head=dim_head)
    if kind in ("vit", "parallel_vit", "patch_merger_vit"):
        ph, pw = int(rng.choice([2, 4])), int(rng.choice([2, 4]))
        case = dict(kind=kind, image_size=(ph * int(rng.integers(1, 4)), pw * int(rng.integers(1, 4))), patch_size=(ph, pw), **base)
        if kind != "patch_merger_vit":
            case["pool"] = str(rng.choice(["cls", "mean"]))
        if kind == "parallel_vit":
            case["num_parallel_branches"] = int(rng.integers(1, 4))
        if kind == "patch_merger_vit":
            case["depth"] = int(rng.integers(2, 5))
            case["patch_merge_layer"] = int(rng.integers(1, case["depth"] + 1)) if rng.random() < 0.7 else None
            case["patch_merge_num_tokens"] = int(rng.integers(1, 5))
        return case
    if kind in ("deepvit", "cait"):
        p = int(rng.choice([2, 4]))
        case = dict(kind=kind, image_size=p * int(rng.integers(1, 4)), patch_size=p, **base)
        if kind == "deepvit":
            case["pool"] = str(rng.choice(["cls", "mean"]))
        else:
            case["cls_depth"] = int(rng.integers(1, 3))
        return case
    if kind == "t2t_vit":
        layers = tuple((int(rng.choice([3, 5])), int(rng.choice([1, 2]))) for _ in range(int(rng.integers(1, 3))))
        return dict(kind=kind, image_size=int(rng.choice([6, 8, 9])), t2t_layers=layers, pool=str(rng.choice(["cls", "mean"])), **base)
    if kind == "crossvit":
        sm_dim = int(rng.choice([8, 12]))
        lg_dim = sm_dim if rng.random() < 0.4 else int(rng.choice([16, 20]))
        return dict(kind=kind, image_size=16, num_classes=int(rng.integers(2, 6)), sm_dim=sm_dim, lg_dim=lg_dim, sm_patch_size=int(rng.choice([4, 8])),
                    lg_patch_size=int(rng.choice([8, 16])), sm_enc_depth=int(rng.integers(1, 3)), lg_enc_depth=int(rng.integers(1, 3)),
                    sm_enc_heads=int(rng.choice([1, 2])), lg_enc_heads=int(rng.choice([1, 2])), sm_enc_mlp_dim=8, lg_enc_mlp_dim=12,
                    sm_enc_dim_head=4, lg_enc_dim_head=8, cross_attn_depth=int(rng.integers(1, 3)), cross_attn_heads=int(rng.choice([1, 3])),
                    cross_attn_dim_head=4, depth=int(rng.integers(1, 3)))
    raise ValueError(kind)


def random_configuration(kind, seed):
    """(case, cfg) of random configuration `seed` of `kind`.  T2T draws the reference cannot run are redrawn: the reference sizes
    pos_embedding with a conv formula (t2t.py:14-15,66,76) but tokenises with SAME padding (:43); when the formula comes out short
    its own call fails at :102 -- not a configuration anyone can run."""
    rng = np.random.default_rng(1000 * seed + len(kind))
    while True:
        case = random_case(kind, rng)
        cfg = oracle.make_config(kind, **{k: v for k, v in case.items() if k != "kind"})
        if kind != "t2t_vit":
            return case, cfg
        gh, gw = oracle.t2t_token_grid(cfg)[-1]
        if cfg["num_patches"] >= gh * gw:
            return case, cfg


def cfg_of(name):
    d = dict({**SMALL, **MID}[name])
    return oracle.make_config(d.pop("kind"), **d)


def bf16_round(x):
    x = np.ascontiguousarray(x, np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)
