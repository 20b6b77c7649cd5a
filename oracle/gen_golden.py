"""Generate tests/golden/*.npz by running the REAL reference modules (this container only).

    python -m oracle.gen_golden

For every case: build a seeded state_dict with oracle.nets.make_state_dict (own deterministic
procedure), load it (strict) into the module returned by the reference's own
define_G / define_D (/root/reference/deepliif/models/networks.py:142-238), switch it to the
reference's inference mode (eval + disable_batchnorm_tracking_stats, util/__init__.py:743-755),
run it per sample at N=1 (reference inference semantics) on a seeded input, and store
(input seed, config, output[, subsampled]) as a small fixture.  The same script asserts the
functional oracle (oracle/nets.py) reproduces the reference output to <= 2e-5 max-abs before a
fixture is written, so a committed fixture always pins the oracle.
"""
import json
import os
import sys

import numpy as np
import torch

from . import nets, pixel
from .ref_shim import import_reference, reference_networks

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def seeded_input(seed, n, c, h, w):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((n, c, h, w), generator=g) * 2 - 1


def ref_eval(net, x):
    import deepliif.util as U
    net.eval()
    U.disable_batchnorm_tracking_stats(net)
    with torch.no_grad():
        return torch.cat([net(x[i:i + 1]) for i in range(x.shape[0])])


def save(name, **arrs):
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
    print("wrote", name, {k: getattr(v, "shape", None) for k, v in arrs.items()})


CELL_CASES = [   # (H, W, seed, resolution, kwargs of compute_final_results)
    (200, 260, 1, "40x", dict()),
    (160, 300, 2, "20x", dict(marker_thresh="default", size_thresh_upper=400, large_noise_thresh="default")),
    (128, 128, 3, "40x", dict(od_thresh_lower=20, od_thresh_upper=330, size_thresh=None)),
    (96, 140, 4, "10x", dict(seg_thresh=90, noise_thresh=0, size_thresh=3, marker_thresh=100)),
    (512, 512, 5, "40x", dict(marker_thresh="default")),
    (64, 64, 6, "40x", dict(no_marker=True)),
]


def cells_fixture():
    """Cell post-processing fixture: the reference's own numba functions (deepliif/postprocessing.py) on seeded
    synthetic images; every stage of compute_final_results (:1223-1304) is stored, and the restatement in
    oracle/cells.py is asserted equal before the file is written."""
    import_reference()
    import deepliif.postprocessing as P
    from . import cells as C
    arrs = {}
    for ci, (H, W, seed, res, kw) in enumerate(CELL_CASES):
        kw = dict(kw)
        orig, seg, marker = C.synth_case(H, W, seed)
        marker_in = None if kw.pop("no_marker", False) else marker
        # stage by stage with the reference functions (body of compute_final_results)
        lnt = P.calculate_large_noise_thresh(kw.get("large_noise_thresh"), res)
        use_od = kw.get("od_thresh_lower") is not None or kw.get("od_thresh_upper") is not None
        m0 = P.create_posneg_mask(seg, kw.get("seg_thresh", 120))
        m1 = m0.copy(); P.mark_background(m1)
        mask, cellsinfo, defaults = P.get_cells_info(seg, orig if use_od else marker_in, res, kw.get("noise_thresh", 4),
                                                     kw.get("seg_thresh", 120), lnt, use_od=use_od)
        cells = np.array([[c[0], int(c[1]), int(c[2]), c[3], c[4], c[5], c[6]] for c in cellsinfo], dtype=np.int64).reshape(-1, 7)
        overlay, refined, scoring = P.compute_final_results(orig, seg, marker_in, res, **kw)
        # the same through the restatement
        st = {}
        o2, r2, s2 = C.compute_final_results(orig, seg, marker_in, res, stages=st, **kw)
        assert np.array_equal(C.mark_background(m0), m1), f"case {ci}: mark_background differs"
        c2 = np.array([[c[0], int(c[1]), int(c[2]), c[3], c[4], c[5], c[6]] for c in st["cells"]], dtype=np.int64).reshape(-1, 7)
        assert np.array_equal(c2, cells), f"case {ci}: cell list differs"
        assert st["defaults"] == {k: int(v) for k, v in defaults.items()}, (ci, st["defaults"], defaults)
        assert np.array_equal(o2, overlay) and np.array_equal(r2, refined), f"case {ci}: final images differ"
        assert json.dumps(s2, sort_keys=True) == json.dumps(scoring, sort_keys=True), (ci, s2, scoring)
        print("cells case", ci, "n_cells", len(cellsinfo), scoring)
        arrs[f"c{ci}_bg"] = m1
        arrs[f"c{ci}_cells"] = cells
        arrs[f"c{ci}_defaults"] = np.array([defaults.get("size_thresh", -1), defaults.get("marker_thresh", -1)], dtype=np.int64)
        arrs[f"c{ci}_scoring"] = np.frombuffer(json.dumps(scoring, sort_keys=True).encode(), dtype=np.uint8)
        if H * W <= 200 * 300:
            arrs[f"c{ci}_overlay"] = overlay; arrs[f"c{ci}_refined"] = refined
        else:
            arrs[f"c{ci}_refined_sub"] = refined[::3, ::5].copy()
            arrs[f"c{ci}_sums"] = np.array([int(overlay.astype(np.int64).sum()), int(refined.astype(np.int64).sum()),
                                            int((refined.astype(np.int64) * (np.arange(W)[None, :, None] + 1)).sum())])
    save("cells", **arrs)


DATASET_CASES = [("resize_and_crop", 48, 32, False), ("resize_and_crop", 40, 40, True), ("crop", 48, 24, False),
                 ("scale_width_and_crop", 52, 36, False), ("none", 48, 48, False)]


def dataset_rows(n=3, h=40, w=44, k=6, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, k * w, 3), dtype=np.uint8) for _ in range(n)]


def dataset_opt(root, pre, ls, cs, nf):
    class O:
        pass
    o = O()
    o.dataroot, o.preprocess, o.max_dataset_size, o.load_size, o.crop_size, o.direction = root, pre, None, ls, cs, "AtoB"
    o.input_nc = o.output_nc = 3
    o.no_flip, o.modalities_no, o.seg_no, o.input_no, o.seg_gen, o.model = nf, 4, 1, 1, True, "DeepLIIF"
    return o


def checksum(a):
    a = a.astype(np.int64).ravel()
    return np.array([a.sum(), (a * (np.arange(a.size) % 8191 + 1)).sum()], dtype=np.int64)


def dataset_fixture():
    """Training data path: the reference's AlignedDataset (deepliif/data/aligned_dataset.py:36-113) on seeded row
    images with `random.seed(100 + index)` before each item; stored as uint8 (its fp32 output is exactly
    (u8/255 - 0.5)/0.5, inverted here) — checksums of every item plus a subsample."""
    import random
    import tempfile
    from PIL import Image
    import_reference()
    from deepliif.data.aligned_dataset import AlignedDataset as RefDS
    root = tempfile.mkdtemp()
    os.makedirs(os.path.join(root, "train"))
    for i, row in enumerate(dataset_rows()):
        Image.fromarray(row).save(os.path.join(root, "train", f"s{i}.png"))
    arrs = {}
    for ci, (pre, ls, cs, nf) in enumerate(DATASET_CASES):
        ds = RefDS(dataset_opt(root, pre, ls, cs, nf))
        for i in range(len(ds)):
            random.seed(100 + i)
            r = ds[i]
            t = torch.stack([r["A"]] + r["B"]).numpy()                       # [k,3,H,W] fp32
            u8 = np.rint((t * 0.5 + 0.5) * 255).astype(np.uint8).transpose(0, 2, 3, 1)
            assert np.array_equal(np.concatenate([pixel.transform(u8[j]) for j in range(u8.shape[0])]), t)
            arrs[f"c{ci}_i{i}_sum"] = checksum(u8)
            arrs[f"c{ci}_i{i}_shape"] = np.array(u8.shape)
            arrs[f"c{ci}_i{i}_sub"] = u8[:, ::3, ::3].copy()
    save("aligned_dataset", **arrs)


E2E_IMAGE = (600, 700, 31)          # H, W, seed of the synthetic IHC region (2 x 2 tiles of 512 with overlap 32)


def e2e_image():
    """Seeded, smooth-ish synthetic RGB region (low-pass noise: tiles are far from is_empty())."""
    H, W, seed = E2E_IMAGE
    rng = np.random.default_rng(seed)
    small = rng.integers(0, 256, size=(H // 8 + 2, W // 8 + 2, 3)).astype(np.float32)
    img = np.kron(small, np.ones((8, 8, 1), np.float32))[:H, :W]
    img = 0.75 * img + 0.25 * rng.integers(0, 256, size=(H, W, 3)).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def e2e_state_dicts():
    """The nine generators of the default topology with the seeds tests/test_inference_api_gpu.py::_write_model_dir uses."""
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 9, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(9, 64, 3, 3, "batch")
    sds = {f"G{i}": nets.make_state_dict(g_shapes, 50 + i, "stress") for i in range(1, 5)}
    sds.update({f"GS{i}": nets.make_state_dict(s_shapes, 60 + i, "stress") for i in range(5)})
    return sds


def e2e_fixture():
    """End-to-end pin: the reference's own `infer_modalities` (deepliif/models/__init__.py:613-660: InferenceTiler, run_dask
    per tile, stitching, output naming, postprocess) on a seeded 600 x 700 region with a model directory whose
    train_opt.txt was written by deepliif_b200.options (format interchange) and whose nine .pth files hold the seeded
    state_dicts above.  Stored: per output image a subsample + checksums, and the scoring dict."""
    import tempfile
    from PIL import Image
    import_reference()
    import deepliif.models as RM
    from deepliif_b200 import training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.options import print_options
    root = tempfile.mkdtemp()
    # exactly what `python -m deepliif_b200.cli train` writes (CLI defaults), read back below by the reference
    p = dict(TRAIN_DEFAULTS, dataroot=root, checkpoints_dir=root, name="m", gpu_ids=(0,),
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25])
    print_options(training.build_options(p), save=True)
    mdir = os.path.join(root, "m")
    for k, sd in e2e_state_dicts().items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    img = Image.fromarray(e2e_image())
    torch.set_num_threads(os.cpu_count())
    images, scoring = RM.infer_modalities(img, 512, mdir, eager_mode=True, return_seg_intermediate=True)
    arrs = {"names": np.frombuffer(json.dumps(sorted(images)).encode(), dtype=np.uint8),
            "scoring": np.frombuffer(json.dumps(scoring, sort_keys=True).encode(), dtype=np.uint8)}
    for k, im in images.items():
        a = np.asarray(im)
        arrs[f"{k}__sub"] = a[::7, ::5].copy()
        arrs[f"{k}__sum"] = checksum(a)
        arrs[f"{k}__shape"] = np.array(a.shape)
    print("e2e outputs:", sorted(images), scoring)
    save("e2e_infer_modalities", **arrs)


def _e2e_model_dir():
    """The model directory of the e2e fixtures: train_opt.txt written by this package's trainer options, nine seeded .pth."""
    import tempfile
    from deepliif_b200 import training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.options import print_options
    root = tempfile.mkdtemp()
    p = dict(TRAIN_DEFAULTS, dataroot=root, checkpoints_dir=root, name="m", gpu_ids=(0,),
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25])
    print_options(training.build_options(p), save=True)
    mdir = os.path.join(root, "m")
    for k, sd in e2e_state_dicts().items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    return mdir


REAL_TILE = "/root/reference/Datasets/Sample_Dataset/test_cli/22_2.png"          # BASELINE config 1's tile
REAL_ROI = ("/root/reference/Sample_Large_Tissues/ROI_7.png", (120, 200, 1120, 800))   # BASELINE config 3: crop box (l, t, r, b)


def webp_lossless(img):
    """The image as lossless WebP bytes: the same pixels as a PNG in about two thirds of the space."""
    import io
    from PIL import Image
    buf = io.BytesIO()
    img.save(buf, format="WEBP", lossless=True, quality=100, method=6)
    data = buf.getvalue()
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGB")), np.asarray(img))
    return np.frombuffer(data, dtype=np.uint8)


def realtile_fixture():
    """BASELINE configs[0]: the reference's `deepliif test` body (infer_modalities, cli.py:833-919) on the REAL sample tile
    Datasets/Sample_Dataset/test_cli/22_2.png — PIL decode, transform, is_empty on real content, the nine generators, seg
    aggregation, tensor2im, postprocess.  The tile's pixels travel inside the fixture as lossless WebP.  Stored at full
    resolution: the posneg mask of Seg, SegRefined, and SegOverlaid as its difference from the tile (mostly zero); Seg
    and Marker 2x subsampled, the other outputs 4x; sums of every output."""
    import io
    from PIL import Image
    import_reference()
    import deepliif.models as RM
    import deepliif.postprocessing as RP
    import deepliif.util as RU
    mdir = _e2e_model_dir()
    webp = webp_lossless(Image.open(REAL_TILE).convert("RGB"))
    img = Image.open(io.BytesIO(webp.tobytes())).convert("RGB")
    torch.set_num_threads(os.cpu_count())
    images, scoring = RM.infer_modalities(img, 512, mdir, eager_mode=True, return_seg_intermediate=True)
    arrs = {"webp": webp,
            "names": np.frombuffer(json.dumps(sorted(images)).encode(), dtype=np.uint8),
            "scoring": np.frombuffer(json.dumps(scoring, sort_keys=True).encode(), dtype=np.uint8),
            "variance": np.array(RU.image_variance_gray(img)), "is_empty": np.array(bool(RM.is_empty(img))),
            "Seg__mask": RP.create_posneg_mask(np.asarray(images["Seg"]), 120)}
    assert np.array_equal(arrs["Seg__mask"], pixel.create_posneg_mask(np.asarray(images["Seg"])))
    for k, im in images.items():
        a = np.asarray(im)
        if k == "SegRefined":
            arrs[f"{k}__full"] = a.copy()
        elif k == "SegOverlaid":
            arrs[f"{k}__minus_input"] = a - np.asarray(img)            # uint8, modulo 256
        else:
            st = 2 if k in ("Seg", "mod4-Marker") else 4
            arrs[f"{k}__sub{st}"] = a[::st, ::st].copy()
        arrs[f"{k}__sum"] = checksum(a)
        arrs[f"{k}__shape"] = np.array(a.shape)
    print("real tile outputs:", sorted(images), scoring)
    save("real_tile_22_2", **arrs)


def wsi_fixture():
    """BASELINE configs[2]: the reference's inference() (models/__init__.py:464-579: InferenceTiler, run_dask per tile,
    stitching) at tile_size=512, overlap_size=56 on a REAL 1000 x 600 region of Sample_Large_Tissues/ROI_7.png (6 tiles),
    plus the InferenceTiler tile counts of all five ROIs at overlap 56 and 32.  Stored: the region as lossless WebP, Seg
    and Marker 4x subsampled + sums, the other outputs 8x subsampled + sums."""
    import io
    from PIL import Image
    import_reference()
    import deepliif.models as RM
    import deepliif.util as RU
    mdir = _e2e_model_dir()
    path, box = REAL_ROI
    webp = webp_lossless(Image.open(path).convert("RGB").crop(box))
    img = Image.open(io.BytesIO(webp.tobytes())).convert("RGB")
    torch.set_num_threads(os.cpu_count())
    opt = RM.get_opt(mdir)
    images = RM.inference(img, tile_size=512, overlap_size=56, model_path=mdir, eager_mode=True, opt=opt,
                          seg_weights=opt.seg_weights)
    counts = {}
    import glob
    for f in sorted(glob.glob(os.path.join(os.path.dirname(path), "*.png"))):
        im = Image.open(f).convert("RGB")
        counts[os.path.basename(f)] = {"size": list(im.size),
                                       "tiles_overlap56": sum(1 for _ in RU.InferenceTiler(im, 512, 56)),
                                       "tiles_overlap32": sum(1 for _ in RU.InferenceTiler(im, 512, 32))}
    arrs = {"webp": webp, "names": np.frombuffer(json.dumps(sorted(images)).encode(), dtype=np.uint8),
            "roi_tile_counts": np.frombuffer(json.dumps(counts, sort_keys=True).encode(), dtype=np.uint8),
            "n_tiles": np.array(sum(1 for _ in RU.InferenceTiler(img, 512, 56)))}
    for k, im in images.items():
        a = np.asarray(im)
        st = 4 if k in ("Seg", "mod4-Marker") else 8
        arrs[f"{k}__sub{st}"] = a[::st, ::st].copy()
        arrs[f"{k}__sum"] = checksum(a)
        arrs[f"{k}__shape"] = np.array(a.shape)
    print("wsi region outputs:", sorted(images), "tiles:", int(arrs["n_tiles"]), counts)
    save("wsi_region_overlap56", **arrs)


TRAIN_CASE = dict(modalities_no=2, seg_gen=True, net_g="resnet_2blocks", net_gs="unet_128", norm="batch", no_dropout=True,
                  padding="zero", batch_size=1, hw=128)


def train_state_dicts(case=TRAIN_CASE):
    """Seeded state_dicts for every network of the small training topology (names as DeepLIIF_model.py:72-113)."""
    n, norm = case["modalities_no"], case["norm"]
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 2, norm, not case["no_dropout"], case["padding"])
    s_shapes = nets.unet_param_shapes(7, 64, 3, 3, norm)
    d_shapes = nets.nlayer_d_param_shapes(4, 64, 6, norm)
    sds = {}
    for i in range(n):
        sds[f"G{i + 1}"] = nets.make_state_dict(g_shapes, 700 + i, "reference")
        sds[f"D{i + 1}"] = nets.make_state_dict(d_shapes, 720 + i, "reference")
    for i in range(n + 1):
        sds[f"GS{i}"] = nets.make_state_dict(s_shapes, 740 + i, "reference")
        sds[f"DS{i}"] = nets.make_state_dict(d_shapes, 760 + i, "reference")
    return sds


def train_batch(case=TRAIN_CASE):
    hw, B, n = case["hw"], case["batch_size"], case["modalities_no"]
    return {"A": seeded_input(800, B, 3, hw, hw), "B": [seeded_input(801 + i, B, 3, hw, hw) for i in range(n + 1)],
            "A_paths": ["synthetic"] * B}


def train_params(root, case=TRAIN_CASE):
    from deepliif_b200.cli import TRAIN_DEFAULTS
    return dict(TRAIN_DEFAULTS, dataroot=root, checkpoints_dir=root, name="t", gpu_ids=(),
                **{k: v for k, v in case.items() if k != "hw"})


def train_step_fixture():
    """One `optimize_parameters()` of the reference's own DeepLIIFModel (DeepLIIF_model.py:431-467) on CPU: seeded weights
    in all ten networks (2 ResNet G, 3 UNet seg G, 5 PatchGAN D), a seeded batch, VGG term patched to zero (it needs a
    downloaded VGG19; lambda_feat is not part of the north star).  Stored: the 14 losses and the post-step values of two
    small weight tensors per optimizer."""
    import tempfile
    import_reference()
    N = reference_networks()
    import deepliif.models as RM
    from deepliif_b200 import training

    class NoVGG(torch.nn.Module):
        def forward(self, x, y):
            return torch.zeros((), device=x.device)
    N.VGGLoss = lambda *a, **k: NoVGG()
    root = tempfile.mkdtemp()
    opt = training.build_options(train_params(root))
    opt.gpu_ids = []
    torch.manual_seed(0)
    model = RM.create_model(opt)
    model.setup(opt)
    for name, sd in train_state_dicts().items():
        getattr(model, "net" + name).load_state_dict(sd)
    model.set_input(train_batch())
    model.optimize_parameters()
    losses = {k: float(v) for k, v in model.get_current_losses().items()}
    print("reference losses:", losses)
    arrs = {"losses": np.frombuffer(json.dumps(losses, sort_keys=True).encode(), dtype=np.uint8)}
    for name, key in (("G1", "model.1.weight"), ("GS0", "model.model.0.weight"), ("D1", "model.0.weight"), ("DS2", "model.0.weight")):
        arrs[f"{name}__{key}"] = getattr(model, "net" + name).state_dict()[key].detach().numpy().copy()
        # the gradient the reference's Adam consumed (still in .grad after the step): lets the tests separate gradient
        # parity (floating point) from optimizer parity (our fused Adam on THIS gradient must land on the same weights)
        arrs[f"{name}__{key}__grad"] = dict(getattr(model, "net" + name).named_parameters())[key].grad.detach().numpy().copy()
    # BatchNorm2d buffers after the step (momentum 0.1, unbiased batch variance; a discriminator is run three times per
    # step — fake, real, fake-for-G — and moves its statistics three times): what the reference writes into its .pth files
    for name, key in (("G1", "model.2"), ("G1", "model.5"), ("GS0", "model.model.1.model.2"), ("D1", "model.3"), ("DS2", "model.6")):
        sd_ = getattr(model, "net" + name).state_dict()
        for suffix in ("running_mean", "running_var", "num_batches_tracked"):
            arrs[f"{name}__{key}.{suffix}"] = sd_[f"{key}.{suffix}"].detach().numpy().copy()
    save("train_step", **arrs)


def options_model_dir(root, legacy=False):
    """A model directory as `deepliif_b200.cli train` leaves it (train_opt.txt from the CLI defaults + empty checkpoint
    files: only their names matter for Options(mode='test'))."""
    from deepliif_b200 import training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.options import print_options
    p = dict(TRAIN_DEFAULTS, dataroot=root, checkpoints_dir=root, name="m", gpu_ids=(0,),
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25])
    print_options(training.build_options(p), save=True)
    mdir = os.path.join(root, "m")
    names = ["G1", "G2", "G3", "G4"] + ([f"G5{i}" for i in range(1, 6)] if legacy else [f"GS{i}" for i in range(5)])
    for k in names:
        open(os.path.join(mdir, f"latest_net_{k}.pth"), "wb").close()
    return mdir


def options_as_json(opt, root):
    d = {k: (list(v) if isinstance(v, tuple) else v) for k, v in vars(opt).items() if k not in ("checkpoints_dir", "dataroot")}
    return json.dumps(d, sort_keys=True, default=str).replace(root, "<root>")


def options_fixture():
    """Options(path_file=train_opt.txt, mode='test') (deepliif/options/__init__.py:76-217): every attribute the reference
    derives for inference (scale_size, mod_id_seg / input_id from the checkpoint names, modalities_names, seg_weights,
    is_train/phase overrides ...) for a new-style (GS0..) and a legacy (G51..) directory."""
    import tempfile
    import_reference()
    from deepliif.options import Options as RefOptions
    arrs = {}
    for tag, legacy in (("new", False), ("legacy", True)):
        root = tempfile.mkdtemp()
        mdir = options_model_dir(root, legacy)
        arrs[tag] = np.frombuffer(options_as_json(RefOptions(path_file=os.path.join(mdir, "train_opt.txt"), mode="test"), root).encode(),
                                  dtype=np.uint8)
    save("options_test_mode", **arrs)


def variance_images():
    """Tiles that exercise is_empty()'s rule of dropping saturated luma (0 / 255) before the variance: pure white, white
    with a dark speck, light grey with black dots, half black / half white, near-white noise, plain noise, one grey level."""
    rng = np.random.default_rng(17)
    t = []
    t.append(np.full((32, 32, 3), 255, np.uint8))
    a = np.full((32, 32, 3), 255, np.uint8); a[:4, :4] = rng.integers(90, 110, (4, 4, 3)); t.append(a)
    b = np.full((32, 32, 3), 240, np.uint8); b[::7, ::5] = 0; t.append(b)
    c = np.zeros((32, 32, 3), np.uint8); c[:, 16:] = 255; t.append(c)
    t.append(rng.integers(250, 256, (32, 32, 3)).astype(np.uint8))
    t.append(rng.integers(0, 256, (32, 32, 3)).astype(np.uint8))
    t.append(np.full((32, 32, 3), 128, np.uint8))
    d = rng.integers(0, 256, (32, 32, 3)).astype(np.uint8); d[rng.random((32, 32)) < 0.3] = 255; d[rng.random((32, 32)) < 0.2] = 0; t.append(d)
    return np.stack(t)


def variance_fixture():
    """image_variance_gray (deepliif/util/__init__.py:478-485) and is_empty (models/__init__.py:391-396) of those tiles."""
    from PIL import Image
    import_reference()
    from deepliif.util import image_variance_gray as ref_var
    from deepliif.models import is_empty
    imgs = variance_images()
    save("variance", imgs=imgs, var=np.array([float(ref_var(Image.fromarray(v))) for v in imgs]),
         empty=np.array([bool(is_empty(Image.fromarray(v))) for v in imgs]))


INIT_CASES = [("G", "resnet_9blocks", "batch", True), ("G", "unet_512", "batch", True), ("G", "resnet_6blocks", "instance", False),
              ("D", "n_layers", "batch", 4), ("D", "basic", "instance", 3)]


def init_signature(networks_module, case, seed=3):
    """Per-tensor SHA-256 of the raw values of a freshly initialised network under torch.manual_seed(seed).  Exact, unlike
    a floating-point sum, whose last bits depend on how many threads torch splits the reduction over."""
    import hashlib
    kind, arch, norm, extra = case
    torch.manual_seed(seed)
    if kind == "G":
        net = networks_module.define_G(3, 3, 64, arch, norm, extra, "normal", 0.02, [], "zero")
    else:
        net = networks_module.define_D(6, 64, arch, extra, norm, "normal", 0.02, [])
    sd = net.state_dict()
    keys = list(sd)
    sig = [hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest() for v in sd.values()]
    return keys, sig


def init_fixture():
    """define_G / define_D + init_weights (networks.py:84-238): same seed -> the same initial weights, tensor by tensor."""
    N = reference_networks()
    arrs = {}
    for i, case in enumerate(INIT_CASES):
        keys, sig = init_signature(N, case)
        arrs[f"c{i}_keys"] = np.frombuffer(json.dumps(keys).encode(), dtype=np.uint8)
        arrs[f"c{i}_sig"] = np.frombuffer(json.dumps(sig).encode(), dtype=np.uint8)
    save("init_weights", **arrs)


SCHED_CASES = [dict(lr_policy="linear", n_epochs=3, n_epochs_decay=4, epoch_count=1, lr_decay_iters=50),
               dict(lr_policy="linear", n_epochs=100, n_epochs_decay=100, epoch_count=98, lr_decay_iters=50),
               dict(lr_policy="step", n_epochs=3, n_epochs_decay=4, epoch_count=1, lr_decay_iters=2),
               dict(lr_policy="cosine", n_epochs=5, n_epochs_decay=4, epoch_count=1, lr_decay_iters=50)]


def lr_sequence(get_scheduler, case, epochs=9, lr=2e-4):
    class O:
        pass
    o = O()
    for k, v in case.items():
        setattr(o, k, v)
    w = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([w], lr=lr)
    sch = get_scheduler(opt, o)
    out = [opt.param_groups[0]["lr"]]
    for _ in range(epochs):
        opt.step(); sch.step()
        out.append(opt.param_groups[0]["lr"])
    return np.asarray(out, dtype=np.float64)


def scheduler_fixture():
    """Learning-rate sequences of the reference's get_scheduler (networks.py:55-81), stepped once per epoch as
    BaseModel.update_learning_rate does (base_model.py:132-141)."""
    N = reference_networks()
    save("schedulers", **{f"c{i}": lr_sequence(N.get_scheduler, c) for i, c in enumerate(SCHED_CASES)})


TRAIN_CLI_CASES = [
    # (dataset: tile size, tiles per row, number of rows), CLI overrides
    (dict(tile=64, k=6, rows=3), dict()),
    (dict(tile=64, k=6, rows=3), dict(seg_weights="0.3,0.1,0.2,0.1,0.3", loss_weights_g="0.1,0.2,0.3,0.2,0.2", seed=7, padding="reflect",
                                     modalities_names="IHC, Hema,DAPI,Lap2,Marker", net_g="resnet_9blocks", preprocess="resize_and_crop",
                                     load_size=72, crop_size=64, epoch_count=1, no_flip=True)),
    (dict(tile=32, k=5, rows=2), dict(modalities_no=2, net_g="resnet_6blocks,resnet_9blocks", net_gs="unet_256", batch_size=3)),
    (dict(tile=32, k=5, rows=2), dict(modalities_no=4, seg_gen=False, net_d="basic", norm="instance", no_dropout=True)),
]


def train_cli_dataset(root, tile, k, rows, seed=5):
    """Row images for the CLI prologue: the seg tile (last one) is black with a bright square, so that the background colour
    estimate finds empty 32 x 32 boxes; the other tiles are smooth colour fields plus noise."""
    from PIL import Image
    rng = np.random.default_rng(seed)
    os.makedirs(os.path.join(root, "train"), exist_ok=True)
    for r in range(rows):
        row = np.zeros((tile, tile * k, 3), np.uint8)
        for j in range(k - 1):
            base = rng.integers(40, 220, size=3)
            row[:, j * tile:(j + 1) * tile] = np.clip(base + rng.integers(-12, 13, size=(tile, tile, 3)), 0, 255)
        seg = np.zeros((tile, tile, 3), np.uint8)
        seg[tile // 2:, tile // 2:] = rng.integers(60, 250, size=(tile - tile // 2, tile - tile // 2, 3))
        row[:, (k - 1) * tile:] = seg
        Image.fromarray(row).save(os.path.join(root, "train", f"r{r}.png"))


def options_snapshot(opt, root):
    skip = ("checkpoints_dir", "dataroot", "local_rank", "precision", "cuda_graph")
    d = {k: (list(v) if isinstance(v, tuple) else v) for k, v in vars(opt).items() if k not in skip}
    def conv(o):
        if isinstance(o, np.integer):
            return int(o)
        return [int(x) for x in o] if hasattr(o, "__iter__") else str(o)
    return json.dumps(d, sort_keys=True, default=conv).replace(root, "<root>")


def train_cli_fixture():
    """The option prologue of the reference's `deepliif train` (cli.py:213-386): the command's callback runs with its click
    defaults + the overrides above on a synthetic dataroot until it calls print_options(opt, save=True); the attributes of
    that Options object are the fixture."""
    import importlib
    import tempfile
    import_reference()
    sys.path.insert(0, "/root/reference")
    rcli = importlib.import_module("cli")

    class Captured(Exception):
        pass

    def capture(opt, save=False):
        raise Captured(opt)
    rcli.print_options = capture
    arrs = {}
    for ci, (ds, over) in enumerate(TRAIN_CLI_CASES):
        root = tempfile.mkdtemp()
        train_cli_dataset(root, **ds)
        kw = {p.name: (p.default if not callable(p.default) else p.default()) for p in rcli.cli.commands["train"].params}
        kw.update(dataroot=root, checkpoints_dir=root, name="exp", gpu_ids=())
        kw.update(over)
        try:
            rcli.cli.commands["train"].callback(**kw)
            raise RuntimeError("print_options was not reached")
        except Captured as c:
            arrs[f"c{ci}"] = np.frombuffer(options_snapshot(c.args[0], root).encode(), dtype=np.uint8)
    save("train_cli_options", **arrs)


def main():
    if "traincli" in sys.argv[1:]:
        return train_cli_fixture()
    if "variance" in sys.argv[1:]:
        return variance_fixture()
    if "options" in sys.argv[1:]:
        return options_fixture()
    if "init" in sys.argv[1:]:
        return init_fixture()
    if "sched" in sys.argv[1:]:
        return scheduler_fixture()
    if "train" in sys.argv[1:]:
        return train_step_fixture()
    if "realtile" in sys.argv[1:]:
        return realtile_fixture()
    if "wsi" in sys.argv[1:]:
        return wsi_fixture()
    if "e2e" in sys.argv[1:]:
        return e2e_fixture()
    if "cells" in sys.argv[1:]:
        return cells_fixture()
    if "dataset" in sys.argv[1:]:
        return dataset_fixture()
    torch.set_num_threads(os.cpu_count())
    N = reference_networks()
    import_reference()
    cases = []

    # ---- ResnetGenerator -------------------------------------------------------------------
    for name, cfg, hw, n, seed, init in [
        ("resnet9_batch_zero_64", dict(n_blocks=9, norm="batch", use_dropout=True, padding_type="zero"), 64, 2, 11, "stress"),
        ("resnet9_inst_zero_64", dict(n_blocks=9, norm="instance", use_dropout=False, padding_type="zero"), 64, 2, 12, "stress"),
        ("resnet9_batch_reflect_64", dict(n_blocks=9, norm="batch", use_dropout=False, padding_type="reflect"), 64, 1, 13, "stress"),
        ("resnet2_inst_reflect_32", dict(n_blocks=2, norm="instance", use_dropout=True, padding_type="reflect"), 32, 2, 14, "stress"),
        ("resnet9_batch_zero_512", dict(n_blocks=9, norm="batch", use_dropout=True, padding_type="zero"), 512, 1, 0, "reference"),
        ("resnet9_inst_zero_512", dict(n_blocks=9, norm="instance", use_dropout=False, padding_type="zero"), 512, 1, 1, "reference"),
    ]:
        shapes = nets.resnet_param_shapes(3, 3, 64, cfg["n_blocks"], cfg["norm"], cfg["use_dropout"], cfg["padding_type"])
        sd = nets.make_state_dict(shapes, seed, init)
        net = N.define_G(3, 3, 64, f"resnet_{cfg['n_blocks']}blocks", cfg["norm"], cfg["use_dropout"],
                         "normal", 0.02, [], cfg["padding_type"])
        assert list(net.state_dict().keys()) == list(sd.keys()), "state_dict key order mismatch"
        net.load_state_dict(sd, strict=True)
        x = seeded_input(1000 + seed, n, 3, hw, hw)
        y_ref = ref_eval(net, x)
        y_orc = nets.resnet_forward(x, sd, norm_mode="sample", **cfg)
        err = (y_ref - y_orc).abs().max().item()
        print(f"{name}: oracle-vs-reference max|d| = {err:.3e}")
        assert err <= 2e-5, name
        y = y_ref.numpy()
        if hw > 128:
            y = y[:, :, ::8, ::8]          # strided subsample keeps the fixture small
        save(name, y=y.astype(np.float32), meta=np.array(json.dumps(
            dict(arch="resnet", cfg=cfg, hw=hw, n=n, seed=seed, init=init, x_seed=1000 + seed,
                 subsample=8 if hw > 128 else 1, mean_abs=float(y_ref.abs().mean()),
                 sum=float(y_ref.double().sum())))))

    # ---- UnetGenerator ---------------------------------------------------------------------
    for name, netG, nd, norm, hw, n, seed in [
        ("unet256_batch_256", "unet_256", 8, "batch", 256, 1, 21),
        ("unet512_batch_512", "unet_512", 9, "batch", 512, 1, 22),
        ("unet128_inst_128", "unet_128", 7, "instance", 128, 2, 23),
    ]:
        shapes = nets.unet_param_shapes(nd, 64, 3, 3, norm)
        sd = nets.make_state_dict(shapes, seed, "stress")
        net = N.define_G(3, 3, 64, netG, norm, True, "normal", 0.02, [])
        assert list(net.state_dict().keys()) == list(sd.keys()), "unet key order mismatch"
        net.load_state_dict(sd, strict=True)
        x = seeded_input(1000 + seed, n, 3, hw, hw)
        y_ref = ref_eval(net, x)
        y_orc = nets.unet_forward(x, sd, num_downs=nd, norm=norm, norm_mode="sample")
        err = (y_ref - y_orc).abs().max().item()
        print(f"{name}: oracle-vs-reference max|d| = {err:.3e}")
        assert err <= 2e-5, name
        y = y_ref.numpy()
        sub = 4 if hw > 128 else 1
        save(name, y=y[:, :, ::sub, ::sub].astype(np.float32), meta=np.array(json.dumps(
            dict(arch="unet", num_downs=nd, norm=norm, hw=hw, n=n, seed=seed, init="stress",
                 x_seed=1000 + seed, subsample=sub, sum=float(y_ref.double().sum())))))

    # ---- NLayerDiscriminator (training-mode batch statistics, N=2) ---------------------------
    for name, netD, nl, norm, hw, n, seed in [
        ("dbasic_batch_128", "basic", 3, "batch", 128, 2, 31),
        ("dn4_inst_128", "n_layers", 4, "instance", 128, 2, 32),
    ]:
        shapes = nets.nlayer_d_param_shapes(nl, 64, 6, norm)
        sd = nets.make_state_dict(shapes, seed, "stress")
        net = N.define_D(6, 64, netD, nl, norm, "normal", 0.02, [])
        assert list(net.state_dict().keys()) == list(sd.keys()), "D key order mismatch"
        net.load_state_dict(sd, strict=True)
        net.train()
        x = seeded_input(1000 + seed, n, 6, hw, hw)
        with torch.no_grad():
            y_ref = net(x)
        y_orc = nets.nlayer_d_forward(x, sd, n_layers=nl, norm=norm, norm_mode="batch")
        err = (y_ref - y_orc).abs().max().item()
        print(f"{name}: oracle-vs-reference max|d| = {err:.3e}")
        assert err <= 2e-5, name
        save(name, y=y_ref.numpy().astype(np.float32), meta=np.array(json.dumps(
            dict(arch="nlayer_d", n_layers=nl, norm=norm, hw=hw, n=n, seed=seed, init="stress",
                 x_seed=1000 + seed))))

    # ---- pixel ends: transform / tensor2im / create_posneg_mask ------------------------------
    from deepliif.data import transform as ref_transform
    from deepliif.util.util import tensor2im as ref_tensor2im
    from deepliif.postprocessing import create_posneg_mask as ref_mask
    from PIL import Image
    rng = np.random.default_rng(7)
    img = rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8)
    t_ref = ref_transform(Image.fromarray(img)).numpy()
    assert np.array_equal(t_ref, pixel.transform(img)), "transform restatement differs"
    f = (rng.random((1, 3, 64, 64), dtype=np.float32) * 2 - 1).astype(np.float32)
    u8_ref = ref_tensor2im(torch.from_numpy(f))
    assert np.array_equal(u8_ref, pixel.tensor2im(f)), "tensor2im restatement differs"
    seg = rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8)
    m_ref = ref_mask(seg, 120)
    assert np.array_equal(m_ref, pixel.create_posneg_mask(seg, 120)), "posneg restatement differs"
    save("pixel_ends", img=img, transform=t_ref.astype(np.float32), f=f, tensor2im=u8_ref,
         seg=seg, mask=m_ref)
    # ---- InferenceTiler geometry + is_empty variance (deepliif/util/__init__.py:129-331, 478-485) ------------------
    from deepliif.util import InferenceTiler, image_variance_gray as ref_var
    tiler_cases = [(995, 1250, 512, 32), (600, 512, 512, 32), (300, 400, 512, 32), (1100, 1300, 512, 56), (512, 512, 512, 32),
                   (513, 1025, 256, 16), (2207, 2662, 512, 32)]
    arrs = {}
    for ci, (h, w, ts, ov) in enumerate(tiler_cases):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        tiler = InferenceTiler(Image.fromarray(img), ts, ov)
        origins, n = [], 0
        for tile in tiler:
            origins.append((tiler.x, tiler.y))
            t = np.asarray(tile).astype(np.int32)
            tiler.stitch({"a": Image.fromarray(((t * 7 + n * 13) % 256).astype(np.uint8))})   # tile-dependent result
            n += 1
        res = np.asarray(tiler.results()["a"])
        arrs[f"c{ci}_cfg"] = np.array([h, w, ts, ov]); arrs[f"c{ci}_img_seed"] = np.array([ci])
        arrs[f"c{ci}_origins"] = np.array(origins, dtype=np.int32)
        arrs[f"c{ci}_res_sub"] = res[::23, ::17].copy(); arrs[f"c{ci}_res_sum"] = np.array([int(res.astype(np.int64).sum())])
        arrs[f"c{ci}_img"] = img[::23, ::17].copy()          # spot check of the regenerated input
    var_imgs = rng.integers(0, 256, (4, 32, 32, 3), dtype=np.uint8)
    var_imgs[1] = 200; var_imgs[2] = (var_imgs[2] // 64) + 100
    arrs["var_imgs"] = var_imgs
    arrs["var_vals"] = np.array([ref_var(Image.fromarray(v)) for v in var_imgs])
    save("tiler", **arrs)
    cells_fixture()
    dataset_fixture()
    e2e_fixture()
    train_step_fixture()
    scheduler_fixture()
    init_fixture()
    options_fixture()
    variance_fixture()
    train_cli_fixture()
    print("all fixtures written to", OUT)


if __name__ == "__main__":
    sys.exit(main())
