"""End-to-end boundary test: a reference-format model directory (train_opt.txt + latest_net_*.pth) goes through
create_model / init_nets / infer_modalities / `deepliif test`, and the stitched uint8 outputs are compared with the
oracle's cascade (DeepLIIF_model.py:175-203 + tensor2im) on the same weights."""
import json
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import nets, pixel

pytestmark = pytest.mark.gpu


def _write_model_dir(root, net_g="resnet_9blocks", net_gs="unet_512", n_blocks=9):
    from deepliif_b200.options import Options, print_options
    d = dict(model="DeepLIIF", name="m", checkpoints_dir=str(root), gpu_ids=(0,), input_nc=3, output_nc=3, ngf=64, ndf=64,
             net_g=net_g, net_gs=net_gs, net_d="n_layers", norm="batch", no_dropout=False, padding="zero", init_type="normal",
             init_gain=0.02, modalities_no=4, seg_gen=True, input_no=1, scale_size=512, phase="train",
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25],
             loss_G_weights=[0.2] * 5, loss_D_weights=[0.2] * 5, mod_id_seg="S")
    opt = Options(d_params=d, mode="train")
    print_options(opt, save=True)
    mdir = os.path.join(str(root), "m")
    sds = {}
    g_shapes = nets.resnet_param_shapes(3, 3, 64, n_blocks, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(9, 64, 3, 3, "batch") if net_gs == "unet_512" else \
        nets.resnet_param_shapes(3, 3, 64, n_blocks, "batch", True, "reflect")
    for i in range(1, 5):
        sds[f"G{i}"] = nets.make_state_dict(g_shapes, 50 + i, "stress")
    for i in range(5):
        sds[f"GS{i}"] = nets.make_state_dict(s_shapes, 60 + i, "stress")
    for k, sd in sds.items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    return mdir, sds


def _oracle_cascade(x, sds, net_gs, weights=(0.2, 0.2, 0.2, 0.2, 0.2)):
    torch.set_num_threads(min(32, os.cpu_count()))
    cfg = dict(n_blocks=9, norm="batch", use_dropout=True, padding_type="zero", norm_mode="sample")
    with torch.no_grad():
        run_g = lambda t, sd: nets.resnet_forward(t, sd, **cfg)
        if net_gs == "unet_512":
            run_s = lambda t, sd: nets.unet_forward(t, sd, num_downs=9, norm="batch", norm_mode="sample")
        else:
            run_s = lambda t, sd: nets.resnet_forward(t, sd, **{**cfg, "padding_type": "reflect"})
        return nets.deepliif_forward(x, [sds[f"G{i}"] for i in range(1, 5)], [sds[f"GS{i}"] for i in range(5)],
                                     list(weights), run_g, run_s)


def test_infer_modalities_matches_oracle_cascade(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from deepliif_b200.models import infer_modalities
    mdir, sds = _write_model_dir(tmp_path)
    rng = np.random.default_rng(11)
    # smooth-ish synthetic IHC tile (variance >> empty-tile threshold)
    img = (rng.random((512, 512, 3)) * 255).astype(np.uint8)
    images, scoring = infer_modalities(Image.fromarray(img), 512, mdir, return_seg_intermediate=True)
    assert set(images) == {"mod1-Hema", "mod2-DAPI", "mod3-Lap2", "mod4-Marker", "Seg", "mod0-IHC_s", "mod1-Hema_s",
                           "mod2-DAPI_s", "mod3-Lap2_s", "mod4-Marker_s", "SegOverlaid", "SegRefined"}
    x = torch.from_numpy(pixel.transform(img))
    mods, parts, seg = _oracle_cascade(x, sds, "unet_512")
    worst = 0
    for name, ref in [("mod1-Hema", mods[0]), ("mod2-DAPI", mods[1]), ("mod3-Lap2", mods[2]), ("mod4-Marker", mods[3]),
                      ("Seg", seg), ("mod0-IHC_s", parts[0]), ("mod4-Marker_s", parts[4])]:
        got = np.asarray(images[name]).astype(np.int32)
        want = pixel.tensor2im(ref.numpy()).astype(np.int32)
        diff = np.abs(got - want)
        frac = float((diff > 0).mean())
        print(f"{name}: uint8 mismatches {frac * 100:.3f}% (max |d| {diff.max()})")
        # fp32 outputs agree to ~1e-4, so a uint8 can differ by at most 1 LSB where (x+1)/2*255 straddles an integer
        assert diff.max() <= 1 and frac < 0.02
        worst = max(worst, frac)
    mask_ref = pixel.create_posneg_mask(pixel.tensor2im(seg.numpy()))
    mask_got = pixel.create_posneg_mask(np.asarray(images["Seg"]))
    mism = int((mask_ref != mask_got).sum())
    print(f"posneg mask pixel mismatches vs oracle-from-fp32: {mism} of {mask_ref.size}")
    # measured on B200: 0 of 262144 (the 1e-4 fp32 differences straddle no mask threshold on this fixture); pinned, not a band
    assert mism == 0
    # explicit seg_weights (what `deepliif test` passes down from train_opt.txt, cli.py:878): same parts, other weights
    w2 = [0.25, 0.15, 0.25, 0.1, 0.25]
    images2, _ = infer_modalities(Image.fromarray(img), 512, mdir, seg_weights=w2)
    seg2 = pixel.seg_aggregate([p.numpy() for p in parts], w2)
    d2 = np.abs(np.asarray(images2["Seg"]).astype(np.int32) - pixel.tensor2im(seg2).astype(np.int32))
    assert d2.max() <= 1 and float((d2 > 0).mean()) < 0.02
    assert np.abs(np.asarray(images2["Seg"]).astype(np.int32) - np.asarray(images["Seg"]).astype(np.int32)).max() > 1
    # postprocess (models/__init__.py:582-591): integer work on the stitched uint8 images -> bit-exact vs the oracle
    from oracle import cells
    ov, rf, sc = cells.compute_final_results(img, np.asarray(images["Seg"]), np.asarray(images["mod4-Marker"]), "40x")
    assert scoring == sc and list(scoring) == ["num_total", "num_pos", "num_neg", "percent_pos", "seg_thresh", "size_thresh",
                                               "size_thresh_upper", "marker_thresh"]
    assert np.array_equal(np.asarray(images["SegOverlaid"]), ov) and np.array_equal(np.asarray(images["SegRefined"]), rf)


def test_cli_test_command_writes_outputs(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from click.testing import CliRunner
    from deepliif_b200.cli import cli
    mdir, _ = _write_model_dir(tmp_path)
    inp, out = tmp_path / "in", tmp_path / "out"
    inp.mkdir()
    rng = np.random.default_rng(12)
    Image.fromarray((rng.random((600, 700, 3)) * 255).astype(np.uint8)).save(inp / "roi.png")
    r = CliRunner().invoke(cli, ["test", "--input-dir", str(inp), "--output-dir", str(out), "--tile-size", "512",
                                 "--model-dir", mdir, "--gpu-ids", "0"])
    assert r.exit_code == 0, r.output
    files = sorted(os.listdir(out))
    assert "roi_Seg.png" in files and "roi_mod4-Marker.png" in files and "roi.json" in files
    assert "roi_SegOverlaid.png" in files and "roi_SegRefined.png" in files
    assert Image.open(out / "roi_Seg.png").size == (700, 600)
    assert "num_total" in json.load(open(out / "roi.json"))


def test_cli_train_then_test_round_trip(tmp_path):
    """`deepliif train` on a tiny synthetic aligned dataset (default topology: ResNet modality generators, UNet seg
    generators, dropout on, seg_gen) writes reference-format checkpoints + train_opt.txt that `deepliif test` loads."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from click.testing import CliRunner
    from deepliif_b200.cli import cli
    root = tmp_path / "data"
    (root / "train").mkdir(parents=True)
    rng = np.random.default_rng(3)
    for i in range(2):       # row of 6 tiles: IHC | Hema | DAPI | Lap2 | Marker | Seg (512 high: scale_size is read off it)
        Image.fromarray((rng.random((512, 6 * 512, 3)) * 255).astype(np.uint8)).save(root / "train" / f"s{i}.png")
    ck = tmp_path / "ck"
    r = CliRunner().invoke(cli, ["train", "--dataroot", str(root), "--name", "exp", "--checkpoints-dir", str(ck), "--gpu-ids", "0",
                                 "--batch-size", "2", "--net-g", "resnet_2blocks", "--net-gs", "unet_128", "--n-epochs", "1",
                                 "--n-epochs-decay", "0", "--save-epoch-freq", "1", "--print-freq", "1", "--num-threads", "2",
                                 "--preprocess", "resize_and_crop", "--load-size", "144", "--crop-size", "128",
                                 "--seed", "0"])
    assert r.exit_code == 0, r.output[-3000:]
    files = set(os.listdir(ck / "exp"))
    for k in ["G1", "G4", "GS0", "GS4", "D1", "DS4"]:
        assert f"latest_net_{k}.pth" in files, files
    assert "train_opt.txt" in files and "loss_log.txt" in files and "1_net_G1.pth" in files
    assert "G_L1_1" in r.output and "D_real_S" in r.output
    from deepliif_b200.options import Options
    topt = Options(path_file=str(ck / "exp" / "train_opt.txt"), mode="test")
    assert topt.scale_size == 512 and topt.input_no == 1 and topt.seg_weights == [0.25, 0.15, 0.25, 0.1, 0.25]
    inp, out = tmp_path / "in", tmp_path / "out"
    inp.mkdir()
    Image.fromarray((rng.random((200, 300, 3)) * 255).astype(np.uint8)).save(inp / "roi.png")
    r = CliRunner().invoke(cli, ["test", "--input-dir", str(inp), "--output-dir", str(out), "--tile-size", "128",
                                 "--model-dir", str(ck / "exp"), "--gpu-ids", "0"])
    assert r.exit_code == 0, r.output[-3000:]
    assert Image.open(out / "roi_Seg.png").size == (300, 200)


def test_empty_tiles_skip_the_networks(tmp_path):
    """run_wrapper semantics (models/__init__.py:399-443): a tile whose gray variance is < 9 is not inferred; its
    modality outputs are the configured background colours and its Seg output is black."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from deepliif_b200.models import get_opt, init_nets, run_batch
    mdir, _ = _write_model_dir(tmp_path)
    opt = get_opt(mdir)
    nets_ = init_nets(mdir, True, opt)
    rng = np.random.default_rng(2)
    tiles = np.stack([(rng.random((512, 512, 3)) * 255).astype(np.uint8), np.full((512, 512, 3), 201, np.uint8)])
    res = run_batch(tiles, nets_, opt, opt.seg_weights)
    for j, k in enumerate(["G1", "G2", "G3", "G4"]):
        assert (res[k][1] == np.array(opt.background_colors[j], np.uint8)).all()
        assert res[k][0].std() > 1.0
    assert (res["GS"][1] == 0).all() and res["GS"][0].std() > 1.0


class _Stub(torch.nn.Module):
    """A torch module with the reference's parameter names (what `deepliif serialize` traces, cli.py:800-811)."""

    def __init__(self, sd):
        super().__init__()
        for k, v in sd.items():
            mod, parts = self, k.split(".")
            for p in parts[:-1]:
                if p not in mod._modules:
                    mod.add_module(p, torch.nn.Module())
                mod = mod._modules[p]
            mod.register_parameter(parts[-1], torch.nn.Parameter(v.clone()))

    def forward(self, x):
        return x + 0


def test_legacy_names_and_serialized_pt_dirs_load_identically(tmp_path):
    """SURVEY 8f row 4: (i) legacy Zenodo naming latest_net_G51..G55 and (ii) a `deepliif serialize` directory of
    TorchScript archives G1.pt.. give the same images as the S-named .pth directory with the same weights."""
    from deepliif_b200.models import infer_modalities, init_nets
    mdir, sds = _write_model_dir(tmp_path, net_g="resnet_2blocks", net_gs="unet_128", n_blocks=2)
    # _write_model_dir builds 9-block / unet_512 shapes: rewrite the files for the small topology
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 2, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(7, 64, 3, 3, "batch")
    sds = {**{f"G{i}": nets.make_state_dict(g_shapes, 50 + i, "stress") for i in range(1, 5)},
           **{f"GS{i}": nets.make_state_dict(s_shapes, 60 + i, "stress") for i in range(5)}}
    for k, sd in sds.items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    legacy, serialized = str(tmp_path / "legacy"), str(tmp_path / "serialized")
    for d in (legacy, serialized):
        os.makedirs(d)
        with open(os.path.join(mdir, "train_opt.txt")) as f, open(os.path.join(d, "train_opt.txt"), "w") as g:
            g.writelines(l for l in f if "mod_id_seg" not in l and "input_id" not in l)
    for k, sd in sds.items():
        old = k if not k.startswith("GS") else f"G5{int(k[2:]) + 1}"
        torch.save(sd, os.path.join(legacy, f"latest_net_{old}.pth"))
        keep = {n: v for n, v in sd.items() if not n.endswith(("running_mean", "running_var", "num_batches_tracked"))}
        torch.jit.trace(_Stub(keep), torch.zeros(1)).save(os.path.join(serialized, f"{k}.pt"))
    rng = np.random.default_rng(21)
    img = Image.fromarray((rng.random((256, 256, 3)) * 255).astype(np.uint8))
    base, _ = infer_modalities(img, 256, mdir, return_seg_intermediate=True)
    for d, eager in ((legacy, True), (serialized, False)):
        init_nets.cache_clear()
        got, _ = infer_modalities(img, 256, d, eager_mode=eager, return_seg_intermediate=True)
        assert set(got) == set(base)
        for k in base:
            assert np.array_equal(np.asarray(got[k]), np.asarray(base[k])), (d, k)


def test_infer_modalities_matches_reference_end_to_end_golden(tmp_path):
    """tests/golden/e2e_infer_modalities.npz = the reference's own infer_modalities (tiling, per-tile cascade, stitching,
    naming, postprocess) on a seeded 600 x 700 region, reading a model directory written by this package's trainer
    options.  Same directory + image here: names, shapes and the scoring dict must be equal, every uint8 image within
    1 LSB (fp32 outputs agree to ~1e-4, so a pixel can straddle a quantisation step)."""
    from deepliif_b200 import training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.models import infer_modalities
    from deepliif_b200.options import print_options
    from oracle.gen_golden import e2e_image, e2e_state_dicts
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "e2e_infer_modalities.npz"))
    p = dict(TRAIN_DEFAULTS, dataroot=str(tmp_path), checkpoints_dir=str(tmp_path), name="m", gpu_ids=(0,),
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25])
    print_options(training.build_options(p), save=True)
    mdir = os.path.join(str(tmp_path), "m")
    for k, sd in e2e_state_dicts().items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    images, scoring = infer_modalities(Image.fromarray(e2e_image()), 512, mdir, return_seg_intermediate=True)
    assert sorted(images) == json.loads(bytes(gold["names"]).decode())
    assert json.dumps(scoring, sort_keys=True) == bytes(gold["scoring"]).decode()
    for k, im in images.items():
        a = np.asarray(im)
        assert list(a.shape) == gold[f"{k}__shape"].tolist(), k
        d = np.abs(a[::7, ::5].astype(np.int32) - gold[f"{k}__sub"].astype(np.int32))
        frac = float((d > 0).mean())
        print(f"{k}: max |d| {d.max()} LSB, {100 * frac:.3f}% of the sampled bytes differ")
        assert d.max() <= 1 and frac < 0.02, k


def _golden_model_dir(tmp_path):
    from deepliif_b200 import training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.options import print_options
    from oracle.gen_golden import e2e_state_dicts
    p = dict(TRAIN_DEFAULTS, dataroot=str(tmp_path), checkpoints_dir=str(tmp_path), name="m", gpu_ids=(0,),
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25])
    print_options(training.build_options(p), save=True)
    mdir = os.path.join(str(tmp_path), "m")
    for k, sd in e2e_state_dicts().items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    return mdir


def _compare_u8(name, got, ref, max_frac):
    d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    frac = float((d > 0).mean())
    print(f"{name}: max |d| {d.max()} LSB, {100 * frac:.4f}% of {d.size} bytes differ")
    assert d.max() <= 1 and frac <= max_frac, name
    return int((d > 0).sum())


def test_real_sample_tile_matches_the_reference_golden(tmp_path):
    """BASELINE config 1: the reference's infer_modalities on the REAL tile Datasets/Sample_Dataset/test_cli/22_2.png
    (tests/golden/real_tile_22_2.npz carries its pixels as lossless WebP and the reference outputs).  Same pixels -> this
    package: names, shapes, is_empty statistic and scoring equal; overlays and the posneg mask compared at FULL
    resolution, Seg and Marker on every 2nd pixel of every 2nd row, the other outputs on every 4th of every 4th."""
    import io
    from deepliif_b200.models import infer_modalities
    from deepliif_b200.util import image_variance_gray, is_empty
    from oracle import pixel
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "real_tile_22_2.npz"))
    img = Image.open(io.BytesIO(gold["webp"].tobytes())).convert("RGB")
    assert img.size == (512, 512)
    assert abs(image_variance_gray(np.asarray(img)) - float(gold["variance"])) <= 1e-9 * float(gold["variance"])
    assert is_empty(np.asarray(img)) == bool(gold["is_empty"]) == False          # noqa: E712  (real tissue: not an empty tile)
    mdir = _golden_model_dir(tmp_path)
    images, scoring = infer_modalities(img, 512, mdir, return_seg_intermediate=True)
    assert sorted(images) == json.loads(bytes(gold["names"]).decode())
    assert json.dumps(scoring, sort_keys=True) == bytes(gold["scoring"]).decode()
    for k, im in images.items():
        a = np.asarray(im)
        assert list(a.shape) == gold[f"{k}__shape"].tolist(), k
        if k in ("SegOverlaid", "SegRefined"):
            ref = gold[f"{k}__full"] if k == "SegRefined" else np.asarray(img) + gold[f"{k}__minus_input"]
            # integer post-processing of Seg / Marker images that themselves differ by isolated LSBs
            bad = int((a != ref).any(axis=-1).sum())
            print(f"{k}: {bad} of {a.shape[0] * a.shape[1]} pixels differ from the reference")
            assert bad <= 0.001 * a.shape[0] * a.shape[1]
        else:
            st = 2 if k in ("Seg", "mod4-Marker") else 4
            _compare_u8(k, a[::st, ::st], gold[f"{k}__sub{st}"], 0.004)
    # the thresholded uint8 segmentation mask (north_star: bit-exact) on the real tile, against the reference's Seg image
    m_ref = gold["Seg__mask"]
    m_got = pixel.create_posneg_mask(np.asarray(images["Seg"]))
    mism = int((m_ref != m_got).sum())
    print(f"posneg mask on the real tile: {mism} of {m_ref.size} pixels differ from the reference's")
    assert mism <= 2


def test_wsi_region_overlap56_matches_the_reference_golden(tmp_path):
    """BASELINE config 3: the reference's inference() at tile_size=512, overlap_size=56 on a real 1000 x 600 region of
    Sample_Large_Tissues/ROI_7.png (6 tiles; its pixels travel in tests/golden/wsi_region_overlap56.npz as lossless
    WebP), plus the InferenceTiler tile counts of all five ROIs at overlap 56 and 32 against TileGrid."""
    import io
    from deepliif_b200.models import get_opt, inference
    from deepliif_b200.util import TileGrid
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "wsi_region_overlap56.npz"))
    counts = json.loads(bytes(gold["roi_tile_counts"]).decode())
    assert len(counts) == 5
    for name, c in counts.items():
        W_, H_ = c["size"]
        blank = np.zeros((H_, W_, 3), np.uint8)
        assert len(TileGrid(blank, 512, 56).tiles()) == c["tiles_overlap56"], name
        assert len(TileGrid(blank, 512, 32).tiles()) == c["tiles_overlap32"], name
    assert sum(c["tiles_overlap56"] for c in counts.values()) == 102 and sum(c["tiles_overlap32"] for c in counts.values()) == 83
    img = Image.open(io.BytesIO(gold["webp"].tobytes())).convert("RGB")
    assert len(TileGrid(np.asarray(img), 512, 56).tiles()) == int(gold["n_tiles"]) == 6
    mdir = _golden_model_dir(tmp_path)
    opt = get_opt(mdir)
    images = inference(img, tile_size=512, overlap_size=56, model_path=mdir, opt=opt, seg_weights=opt.seg_weights)
    assert sorted(images) == json.loads(bytes(gold["names"]).decode())
    for k, im in images.items():
        a = np.asarray(im)
        assert list(a.shape) == gold[f"{k}__shape"].tolist(), k
        st = 4 if k in ("Seg", "mod4-Marker") else 8
        _compare_u8(k, a[::st, ::st], gold[f"{k}__sub{st}"], 0.004)


def test_serialize_command_writes_a_packed_directory_that_test_reads(tmp_path):
    """`deepliif serialize` (SURVEY 8f row 4): the output directory holds <name>.pt files with the fp32 weights plus the
    repacked tensor-core operand planes, and gives the same images as the .pth directory it was made from."""
    from click.testing import CliRunner
    from deepliif_b200.cli import cli
    from deepliif_b200.models import infer_modalities, init_nets
    from deepliif_b200.models.serialized import FORMAT
    mdir, _ = _write_model_dir(tmp_path, net_g="resnet_2blocks", net_gs="unet_128", n_blocks=2)
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 2, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(7, 64, 3, 3, "batch")
    sds = {**{f"G{i}": nets.make_state_dict(g_shapes, 50 + i, "stress") for i in range(1, 5)},
           **{f"GS{i}": nets.make_state_dict(s_shapes, 60 + i, "stress") for i in range(5)}}
    for k, sd in sds.items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    out = str(tmp_path / "packed")
    init_nets.cache_clear()
    r = CliRunner().invoke(cli, ["serialize", "--model-dir", mdir, "--output-dir", out])
    assert r.exit_code == 0, r.output
    blob = torch.load(os.path.join(out, "G1.pt"), weights_only=True)
    assert blob["format"] == FORMAT and blob["arch"]["kind"] == "resnet"
    w = sds["G1"]["model.4.weight"]                                   # 64 -> 128 3x3 stride-2 conv
    pk = blob["packed"]["model.4"]
    assert tuple(pk["hi"].shape) == (9, 128, 64) and pk["hi"].dtype == torch.bfloat16
    ref = w.permute(2, 3, 0, 1).reshape(9, 128, 64)
    assert torch.equal(pk["hi"], ref.to(torch.bfloat16))
    assert torch.equal(pk["lo"], (ref - ref.to(torch.bfloat16).float()).to(torch.bfloat16))
    rng = np.random.default_rng(23)
    img = Image.fromarray((rng.random((256, 256, 3)) * 255).astype(np.uint8))
    init_nets.cache_clear()
    base, _ = infer_modalities(img, 256, mdir)
    init_nets.cache_clear()
    got, _ = infer_modalities(img, 256, out, eager_mode=False)
    assert set(got) == set(base)
    for k in base:
        assert np.array_equal(np.asarray(got[k]), np.asarray(base[k])), k


def test_infer_images_pipeline_equals_per_image_inference(tmp_path):
    """models.infer_images (tiling / upload / stitching pipelined across images, side-stream is_empty) returns, image by
    image and in order, exactly what infer_tiles returns — including an image with an empty (constant) tile."""
    from deepliif_b200.models import get_opt, infer_images, infer_tiles, init_nets
    mdir, _ = _write_model_dir(tmp_path, net_g="resnet_2blocks", net_gs="unet_128", n_blocks=2)
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 2, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(7, 64, 3, 3, "batch")
    for k, sd in {**{f"G{i}": nets.make_state_dict(g_shapes, 50 + i, "stress") for i in range(1, 5)},
                  **{f"GS{i}": nets.make_state_dict(s_shapes, 60 + i, "stress") for i in range(5)}}.items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    init_nets.cache_clear()
    opt = get_opt(mdir)
    opt.scale_size = 256
    netd = init_nets(mdir, True, opt)
    rng = np.random.default_rng(31)
    imgs = []
    for (h, w) in ((300, 520), (256, 256), (700, 300), (512, 512), (260, 900)):
        a = (rng.random((h, w, 3)) * 255).astype(np.uint8)
        imgs.append(Image.fromarray(a))
    blank = np.full((300, 520, 3), 200, np.uint8); blank[:, 260:] = (rng.random((300, 260, 3)) * 255).astype(np.uint8)
    imgs.append(Image.fromarray(blank))                                          # left tile is empty (variance 0)
    ref = [infer_tiles(im, 256, 16, netd, opt, seg_weights=opt.seg_weights, want_parts=False) for im in imgs]
    got = list(infer_images(imgs, 256, 16, netd, opt, seg_weights=opt.seg_weights, want_parts=False, depth=2))
    assert [i for i, _ in got] == list(range(len(imgs)))
    for (_, g_), r_ in zip(got, ref):
        assert sorted(g_) == sorted(r_)
        for k in r_:
            assert np.array_equal(np.asarray(g_[k]), np.asarray(r_[k])), k
