"""CPU suite (-m "not gpu"): the oracle against the golden fixtures generated from the real reference
(oracle/gen_golden.py), and the C-ABI library's symbol table against include/deepliif_b200.h."""
import glob
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import nets, pixel

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = 2e-5   # fp32 oracle vs fp32 reference (different CPU kernels / thread counts may reorder sums)


def _load(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    return z, json.loads(str(z["meta"]))


def _x(meta, c=3):
    g = torch.Generator().manual_seed(meta["x_seed"])
    return torch.rand((meta["n"], c, meta["hw"], meta["hw"]), generator=g) * 2 - 1


RESNET_CASES = ["resnet9_batch_zero_64", "resnet9_inst_zero_64", "resnet9_batch_reflect_64", "resnet2_inst_reflect_32"]


@pytest.mark.parametrize("name", RESNET_CASES)
def test_resnet_oracle_matches_reference_golden(name):
    z, m = _load(name)
    cfg = m["cfg"]
    sd = nets.make_state_dict(nets.resnet_param_shapes(3, 3, 64, cfg["n_blocks"], cfg["norm"], cfg["use_dropout"],
                                                       cfg["padding_type"]), m["seed"], m["init"])
    with torch.no_grad():
        y = nets.resnet_forward(_x(m), sd, norm_mode="sample", **cfg).numpy()
    assert np.abs(y - z["y"]).max() <= TOL


def test_resnet_oracle_full_size_subsample():
    z, m = _load("resnet9_inst_zero_512")
    cfg = m["cfg"]
    sd = nets.make_state_dict(nets.resnet_param_shapes(3, 3, 64, 9, cfg["norm"], cfg["use_dropout"], cfg["padding_type"]),
                              m["seed"], m["init"])
    torch.set_num_threads(min(32, os.cpu_count()))
    with torch.no_grad():
        y = nets.resnet_forward(_x(m), sd, norm_mode="sample", **cfg).numpy()
    assert np.abs(y[:, :, ::8, ::8] - z["y"]).max() <= TOL
    assert abs(float(y.astype(np.float64).sum()) - m["sum"]) <= 1e-2 * max(1.0, abs(m["sum"]))


@pytest.mark.parametrize("name", ["unet256_batch_256", "unet128_inst_128"])
def test_unet_oracle_matches_reference_golden(name):
    z, m = _load(name)
    sd = nets.make_state_dict(nets.unet_param_shapes(m["num_downs"], 64, 3, 3, m["norm"]), m["seed"], m["init"])
    with torch.no_grad():
        y = nets.unet_forward(_x(m), sd, num_downs=m["num_downs"], norm=m["norm"], norm_mode="sample").numpy()
    s = m["subsample"]
    assert np.abs(y[:, :, ::s, ::s] - z["y"]).max() <= TOL


@pytest.mark.parametrize("name", ["dbasic_batch_128", "dn4_inst_128"])
def test_discriminator_oracle_matches_reference_golden(name):
    z, m = _load(name)
    sd = nets.make_state_dict(nets.nlayer_d_param_shapes(m["n_layers"], 64, 6, m["norm"]), m["seed"], m["init"])
    with torch.no_grad():
        y = nets.nlayer_d_forward(_x(m, 6), sd, n_layers=m["n_layers"], norm=m["norm"], norm_mode="batch").numpy()
    assert np.abs(y - z["y"]).max() <= TOL


def test_pixel_oracle_bit_exact():
    z = np.load(os.path.join(GOLD, "pixel_ends.npz"))
    assert np.array_equal(pixel.transform(z["img"]), z["transform"])
    assert np.array_equal(pixel.tensor2im(z["f"]), z["tensor2im"])
    assert np.array_equal(pixel.create_posneg_mask(z["seg"], 120), z["mask"])
    # edge cases of the threshold rule (postprocessing.py:184-188)
    seg = np.array([[[60, 80, 61], [61, 80, 60], [60, 81, 61], [60, 0, 60], [255, 0, 255], [0, 0, 0]]], np.uint8)
    assert pixel.create_posneg_mask(seg).tolist() == [[150, 200, 50, 50, 200, 50]]


def test_resnet_gflop_matches_survey():
    assert abs(nets.resnet_gflop(512) - 396.41) < 0.05


def test_state_dict_keys_match_survey_counts():
    assert len(nets.resnet_param_shapes(norm="batch", use_dropout=True)) == 140
    assert len(nets.resnet_param_shapes(norm="instance", use_dropout=False)) == 48
    assert len(nets.unet_param_shapes(9, norm="batch")) == 94


def test_library_exports_every_declared_symbol(lib_built):
    """The C-ABI .so loads on a CPU-only box and exports exactly what include/deepliif_b200.h declares."""
    from deepliif_b200 import _lib
    lib = _lib.load()
    assert lib.dlb_version() >= 100
    hdr = open(os.path.join(os.path.dirname(GOLD), "..", "include", "deepliif_b200.h")).read()
    declared = set(re.findall(r"\b(dlb_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    for name in declared:
        assert hasattr(lib, name), name


def test_conv_out_shape_matches_pytorch(lib_built):
    from deepliif_b200 import ops
    for (H, R, st, pad, tr, op) in [(512, 7, 1, 3, False, 0), (512, 3, 2, 1, False, 0), (128, 3, 2, 1, True, 1),
                                    (64, 4, 2, 1, True, 0), (64, 4, 1, 1, False, 0), (63, 4, 1, 1, False, 0)]:
        d = ops.conv_desc(1, H, H, 8, 8, R, R, st, pad, tr, op)
        x = torch.zeros(1, 8, H, H)
        if tr:
            ref = torch.nn.functional.conv_transpose2d(x, torch.zeros(8, 8, R, R), stride=st, padding=pad, output_padding=op)
        else:
            ref = torch.nn.functional.conv2d(x, torch.zeros(8, 8, R, R), stride=st, padding=pad)
        assert ops.conv_out_shape(d) == tuple(ref.shape[2:])


def test_no_product_import_of_oracle():
    """The product package must never import the oracle (tier rule)."""
    root = os.path.join(os.path.dirname(GOLD), "..", "deepliif_b200")
    for path in glob.glob(os.path.join(root, "**", "*.py"), recursive=True):
        src = open(path).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), path


def test_tilegrid_matches_reference_tiler_golden():
    """TileGrid (batched tiles + stitch) against origins / stitched result recorded from the reference's InferenceTiler
    (util/__init__.py:244-316), incl. ragged sizes, images smaller than a tile, and the last-tile clamp."""
    from deepliif_b200.util import TileGrid, image_variance_gray
    z = np.load(os.path.join(GOLD, "tiler.npz"))
    rng = np.random.default_rng(7)
    # replay gen_golden's random stream up to the tiler section
    rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8); rng.random((1, 3, 64, 64), dtype=np.float32)
    rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8)
    ci = 0
    while f"c{ci}_cfg" in z:
        h, w, ts, ov = [int(v) for v in z[f"c{ci}_cfg"]]
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(img[::23, ::17], z[f"c{ci}_img"])
        g = TileGrid(img, ts, ov)
        assert np.array_equal(np.array(g.origins, dtype=np.int32), z[f"c{ci}_origins"])
        tiles = g.tiles().astype(np.int32)
        res_tiles = np.stack([((t * 7 + n * 13) % 256).astype(np.uint8) for n, t in enumerate(tiles)])
        res = g.stitch(res_tiles)
        assert res.shape[:2] == (h, w)
        assert np.array_equal(res[::23, ::17], z[f"c{ci}_res_sub"]) and int(res.astype(np.int64).sum()) == int(z[f"c{ci}_res_sum"][0])
        ci += 1
    assert ci == 7
    for im, v in zip(z["var_imgs"], z["var_vals"]):
        assert abs(image_variance_gray(im) - float(v)) < 1e-6


def test_options_round_trip_and_test_mode_defaults(tmp_path):
    """train_opt.txt written by print_options is re-read in test mode with the reference's back-compat defaults."""
    from deepliif_b200.options import Options, print_options
    d = dict(model="DeepLIIF", name="m", checkpoints_dir=str(tmp_path), gpu_ids=(0,), modalities_no=4, seg_gen=True,
             input_no=1, phase="train", norm="batch", net_g="resnet_9blocks", net_gs="unet_512", padding="zero", no_dropout=False)
    print_options(Options(d_params=d, mode="train"), save=True)
    mdir = tmp_path / "m"
    for k in ["G1", "G2", "G3", "G4", "G51", "G52", "G53", "G54", "G55"]:       # legacy Zenodo naming
        (mdir / f"latest_net_{k}.pth").write_bytes(b"")
    opt = Options(path_file=str(mdir / "train_opt.txt"), mode="test")
    assert opt.mod_id_seg == "5" and opt.input_id == 1
    assert opt.modalities_names == ["IHC", "Hema", "DAPI", "Lap2", "Marker"] and opt.seg_weights == [0.5, 0, 0, 0, 0.5]
    assert opt.is_train is False and opt.scale_size == 512 and opt.n_layers_D == 4 and opt.lambda_L1 == 100
    assert opt.checkpoints_dir == str(tmp_path) and opt.name == "m"


def test_unknown_names_raise_like_the_reference():
    from deepliif_b200.models import networks
    with pytest.raises(NotImplementedError):
        networks.define_G(3, 3, 64, "nonsense")
    with pytest.raises(NotImplementedError):
        networks.define_D(6, 64, "nonsense")
    with pytest.raises(NotImplementedError):
        networks.get_norm_layer("nonsense")


def test_lr_schedulers_match_reference_golden():
    """get_scheduler (networks.py:55-81) stepped per epoch: linear / step / cosine sequences equal the reference's."""
    from deepliif_b200.models.networks import get_scheduler
    from oracle.gen_golden import SCHED_CASES, lr_sequence
    z = np.load(os.path.join(GOLD, "schedulers.npz"))
    for i, case in enumerate(SCHED_CASES):
        assert np.array_equal(lr_sequence(get_scheduler, case), z[f"c{i}"]), case


def test_same_seed_gives_the_reference_initial_weights():
    """define_G / define_D + init_weights consume torch's RNG exactly as the reference does (networks.py:84-238): under
    the same seed every tensor of a fresh network equals the reference's (keys, order and values)."""
    import json
    from deepliif_b200.models import networks
    from oracle.gen_golden import INIT_CASES, init_signature
    z = np.load(os.path.join(GOLD, "init_weights.npz"))
    for i, case in enumerate(INIT_CASES):
        keys, sig = init_signature(networks, case)
        assert keys == json.loads(bytes(z[f"c{i}_keys"]).decode()), case
        ref = json.loads(bytes(z[f"c{i}_sig"]).decode())
        assert sig == ref, (case, [k for k, a, b in zip(keys, sig, ref) if a != b][:8])


def test_test_mode_options_equal_the_reference(tmp_path):
    """Options(path_file, mode='test') on a directory written by this package's trainer: every attribute equals what the
    reference's Options derives from the same files (new GS0.. naming and legacy G51.. naming)."""
    import json
    from deepliif_b200.options import Options
    from oracle.gen_golden import options_as_json, options_model_dir
    z = np.load(os.path.join(GOLD, "options_test_mode.npz"))
    for tag, legacy in (("new", False), ("legacy", True)):
        root = str(tmp_path / tag)
        os.makedirs(root)
        mdir = options_model_dir(root, legacy)
        got = json.loads(options_as_json(Options(path_file=os.path.join(mdir, "train_opt.txt"), mode="test"), root))
        want = json.loads(bytes(z[tag]).decode())
        assert got == want, {k: (got.get(k), want.get(k)) for k in set(got) | set(want) if got.get(k) != want.get(k)}


def test_image_variance_gray_drops_saturated_pixels_like_the_reference():
    """is_empty()'s statistic: the variance is taken over the luma values that are neither 0 nor 255 (0 if none)."""
    from deepliif_b200.util import image_variance_gray
    z = np.load(os.path.join(GOLD, "variance.npz"))
    for im, v, e in zip(z["imgs"], z["var"], z["empty"]):
        got = image_variance_gray(im)
        assert abs(got - float(v)) < 1e-9 * max(1.0, abs(float(v)))
        assert (got < 9) == bool(e)


def test_ctypes_signatures_match_the_header_prototypes(lib_built):
    """Every prototype in include/deepliif_b200.h against the ctypes table the host code calls through: same number of
    arguments and the same argument class (pointer / int / float / unsigned 64-bit incl. size_t / signed 64-bit) in every position — a binding
    that drifts from the header corrupts the call frame silently."""
    import ctypes as C
    from deepliif_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(GOLD), "..", "include", "deepliif_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    hdr = re.sub(r"//[^\n]*", " ", hdr)
    protos = re.findall(r"\b([A-Za-z_][A-Za-z0-9_ \*]*?)\b(dlb_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", hdr)
    assert len(protos) >= 40

    def klass_c(decl):
        d = " ".join(decl.split())
        if "*" in d or "dlb_stream_t" in d:
            return "ptr"
        if "size_t" in d:
            return "u64"                  # ctypes aliases c_size_t and c_ulonglong on LP64
        if "float" in d:
            return "float"
        if "unsigned long long" in d:
            return "u64"
        if "long long" in d:
            return "i64"
        if re.search(r"\bint\b", d):
            return "int"
        raise AssertionError(f"unclassified parameter: {decl!r}")

    def klass_py(t):
        if t in (C.c_void_p, C.c_char_p) or hasattr(t, "contents") or (isinstance(t, type) and issubclass(t, C._Pointer)):
            return "ptr"
        return {C.c_size_t: "u64", C.c_float: "float", C.c_ulonglong: "u64", C.c_longlong: "i64", C.c_int: "int"}[t]

    seen = set()
    for ret, name, params in protos:
        seen.add(name)
        params = params.strip()
        cparams = [] if params in ("", "void") else [p for p in params.split(",")]
        restype, argtypes = _lib.SIGNATURES[name]
        assert len(cparams) == len(argtypes), (name, len(cparams), len(argtypes))
        for i, (cp, at) in enumerate(zip(cparams, argtypes)):
            assert klass_c(cp) == klass_py(at), (name, i, cp.strip(), at)
    assert seen == set(_lib.SIGNATURES)
