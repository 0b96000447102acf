"""parse_config: reference flags/defaults/precedence; the reference's own yaml files load unchanged.

The reference's yaml files and the flag table of its own parse_config are recorded in
tests/golden/ref_config_golden.json (tests/golden/make_ref_host_golden.py)."""
import json
import os

import pytest

from cape_b200.config_parser import model_params, parse_config

REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_config_golden.json")


def _ref_golden():
    with open(REF_GOLDEN) as f:
        return json.load(f)

AFFINE_YAML = """dataset: dataset_male_4clotypes
name: CAPE-affineconv_nz64_pose32_clotype32_male
lambda_latent: 0.0008
lambda_edge: 1.0
num_conv_layers: 8
nf: 64
nz: 64
nz_cond: 32
nz_cond2: 32
pose_type: rot
cond_encoder: 0
reduce_dim: 64
lr: 0.008
use_res_block: 0
use_res_block_dec: 1
affine: 1
num_epochs: 60
lr_warmup: 1
decay_every: 2
gender: male
mode: demo
vis_demo: 1
some_unknown_key: 7
"""


def test_yaml_and_cli_precedence(tmp_path):
    f = tmp_path / "c.yaml"
    f.write_text(AFFINE_YAML)
    args, d = parse_config(["--config", str(f)])
    assert args.nz == 64 and args.affine == 1 and args.lr == 0.008 and args.mode == "demo"
    assert args.batch_size == 16 and args.Kd == 3 and args.regularization == 2e-3      # argparse defaults
    assert d is vars(args)
    args, _ = parse_config(["--config", str(f), "--nz", "32", "--mode", "train", "--unknown_flag", "1"])
    assert args.nz == 32 and args.mode == "train"                                      # CLI > file
    p = model_params(args, n_train=1000)
    assert p["F"] == [64, 64, 128, 128, 256, 256, 512, 512] and p["K"] == [2] * 8      # --K is ignored (main.py:65)
    assert p["cond_dim"] == 126 and p["affine"] is True and p["decay_steps"] == 2 * 1000 / 16
    assert "mode" not in p and "nf" not in p


def test_defaults_without_file(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)                      # no configs/default_config.yaml here
    args, _ = parse_config([])
    assert args.nz == 18 and args.use_res_block_dec == 1 and args.optimizer == "sgd"
    with pytest.raises(FileNotFoundError):
        parse_config(["--config", "missing.yaml"])


def test_reference_configs_load_unchanged(tmp_path):
    configs = _ref_golden()["configs"]
    assert len(configs) == 8
    for fn, text in sorted(configs.items()):
        (tmp_path / fn).write_text(text)
        args, _ = parse_config(["--config", str(tmp_path / fn)])
        if fn.startswith("CAPE-affineconv_nz64"):
            assert (args.nz, args.nz_cond, args.nz_cond2, args.affine) == (64, 32, 32, 1)
        if fn.startswith("CAPE_nz18"):
            assert (args.nz, args.nz_cond, args.nz_cond2, args.affine) == (18, 24, 8, 0)


def test_param_store_low_part_views():
    """ParamStore.lo_of: the tf32 low-part buffer is addressed through the same views as the parameters."""
    import torch
    from cape_b200.network import ParamStore
    specs = {"a/weights": (6, 8), "a/bias": (8,), "b/weights": (3, 5)}
    ps = ParamStore(specs, list(specs), torch.device("cpu"))
    ps.flat.copy_(torch.arange(ps.size, dtype=torch.float32))
    ps.lo.copy_(-ps.flat)
    w = ps.w("b/weights")
    lo = ps.lo_of(w)
    assert lo is not None and lo.shape == w.shape and torch.equal(lo, -w)
    v = ps.w("a/weights").view(6, 8)
    assert torch.equal(ps.lo_of(v), -v)
    assert ps.lo_of(torch.zeros(4)) is None                     # not a view of this store


def test_weight_gradient_operand_choice():
    """choose_dw_mode on the layer shapes of the shipped config (levels 6890/3445/1723/862)."""
    from cape_b200.network import choose_dw_mode as m
    assert m(3, 64, 2, 6890, 6890, False) == "gather"            # enc conv1: thin input
    assert m(64, 64, 2, 6890, 3445, True) == "aside"             # enc conv2: pooled -> contract over the coarse rows
    assert m(64, 128, 2, 3445, 3445, True) == "aside"            # enc conv3: widening, same level -> narrower side is x
    assert m(512, 512, 2, 862, 862, True) == "aside"             # enc conv8: K*Fout > 512
    assert m(512, 256, 2, 862, 862, True) == "gside"             # dec aff1: narrowing, all terms in one pass
    assert m(256, 256, 2, 862, 1723, True) == "gside"            # dec aff2: un-pooling -> contract over the coarse rows
    assert m(32, 3, 2, 6890, 6890, True) == "gather"             # dec outputs: thin output (role-swapped thin kernel)
    assert m(64, 64, 3, 3445, 1723, True) == "aside"             # disc conv2
    assert m(128, 128, 2, 862, 862, False) == "aside"            # no data gradient requested -> no G-side stash
    assert m(64, 64, 2, 6890, 3445, True, stash=False) == "gather"


def test_layer_forms_of_the_shipped_config():
    """choose_forms (fused / basis-first / contract-first) on the nz64 layer shapes, and its overrides."""
    from cape_b200.network import choose_forms as f
    env = {}
    # encoder conv2 (pooled 64 -> 64, precise): basis-first forward; the data gradient stays fused (64 wide)
    assert f(64, 0, 64, 2, 6890, 3445, False, True, "aside", True, False, "enc/conv2", env) == ("basis", "fused")
    # encoder conv3 (64 -> 128): the gradient narrows -> contract first; conv6 (pooled, 256 wide) too; conv8 (K*F > 512) not
    assert f(64, 0, 128, 2, 3445, 3445, False, True, "aside", True, False, "enc/conv3", env) == ("basis", "contract")
    assert f(256, 0, 256, 2, 1723, 862, False, True, "aside", True, False, "enc/conv6", env) == ("basis", "contract")
    assert f(512, 0, 512, 2, 862, 862, False, True, "aside", True, False, "enc/conv8", env) == ("basis", "fused")
    # decoder: un-pooling affine blocks contract first, same-level ones stay fused; a precise one contracts first too
    # (the wide un-pooling block also takes its data gradient basis-first, the narrower ones stay fused)
    assert f(256, 64, 128, 2, 862, 1723, True, True, "gside", False, False, "dec/aff3", env) == ("contract", "basis")
    assert f(128, 64, 64, 2, 1723, 3445, True, True, "gside", False, False, "dec/aff5", env) == ("contract", "fused")
    assert f(512, 64, 256, 2, 862, 862, True, True, "gside", False, False, "dec/aff1", env) == ("fused", "fused")
    assert f(512, 64, 256, 2, 862, 862, True, True, "gside", True, False, "dec/aff1", env)[0] == "contract"
    # an affine block that WIDENS (32 -> 64: generated 4-layer hierarchies) has two upstream gradients: its data gradient
    # must not take the single-tensor contract-first form, not even on request
    assert f(32, 64, 64, 2, 3445, 3445, True, True, "aside", False, False, "dec/aff2", env) == ("fused", "fused")
    assert f(32, 64, 64, 2, 3445, 3445, True, True, "aside", False, False, "dec/aff2", {"CAPE_DX_MODE": "contract"})[1] == "fused"
    # discriminator (not precise, K = 3, pooled): basis-first forward (the fused kernel's 19-tap gather loses to gather
    # launch + plain contraction), contract-first data gradient where the layer pools and narrows; the first layer
    # carries the condition channels and stays fused
    assert f(64, 0, 128, 3, 1723, 862, False, True, "aside", False, False, "disc/conv3", env) == ("basis", "contract")
    assert f(64, 0, 64, 3, 3445, 1723, False, True, "aside", False, False, "disc/conv2", env) == ("basis", "fused")
    assert f(3, 64, 64, 3, 6890, 3445, False, False, "gather", False, False, "disc/conv1", env) == ("fused", "fused")
    # thin layers and 1x1 convs (identity operators only) never split
    assert f(3, 0, 64, 2, 6890, 6890, False, False, "gather", True, False, "enc/conv1", env) == ("fused", "fused")
    assert f(512, 0, 64, 1, 862, 862, False, True, "gside", True, True, "enc/1x1", env) == ("fused", "fused")
    # overrides: global and per layer; ineligible requests are ignored
    assert f(64, 0, 128, 2, 3445, 3445, False, True, "aside", True, False, "enc/conv3", {"CAPE_FWD_MODE": "fused"})[0] == "fused"
    assert f(512, 0, 512, 2, 862, 862, False, True, "aside", True, False, "enc/conv8",
             {"CAPE_MODES": "enc/conv8:dx=contract,enc/conv7:fwd=fused"}) == ("basis", "contract")
    assert f(512, 64, 256, 2, 862, 862, True, True, "gside", False, False, "dec/aff1", {"CAPE_FWD_MODE": "basis"})[0] == "fused"


def test_flag_inventory_is_the_references():
    """Every flag the reference's own parse_config declares (config_parser.py:11-63) -- name, type, default, choices --
    against the table this package parses with.  The reference needs `configargparse` (not installed): its table was
    recorded by a stand-in that captured its add_argument calls while its unmodified parse_config ran."""
    from cape_b200 import config_parser as ours
    g = _ref_golden()
    cf = g["config_flag"]
    assert cf["name"] == "config" and cf["is_config_file"] and cf["default"] == ours.DEFAULT_CONFIG
    ref = [tuple(r) for r in g["flags"]]
    mine = [(n, t.__name__, d, None if ours._CHOICES.get(n) is None else list(ours._CHOICES[n]))
            for n, t, d, _ in ours._SPEC]
    assert [r[0] for r in ref] == [m[0] for m in mine]                       # same flags, same order
    for r, m in zip(ref, mine):
        assert r == m, (r, m)
    # and the defaults our parser hands out when neither a file nor a flag sets them
    a, _ = ours.parse_config(["--config", os.devnull])
    for n, _, default, _ in ref:
        assert getattr(a, n) == default, n
