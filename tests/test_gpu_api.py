"""GPU tests of the reference-facing Python API (LENS, run_inference, recallAtK) on the bundled
example data (committed as fixtures by tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

NS = (1, 5, 10, 15, 20, 25)


def reference_recall_here(D, GTtol):
    """What the reference's recallAtK returns in THIS environment (numpy's default argsort decides the
    ties, metrics.py:218), restated by the oracle."""
    return [round(O.recall_at_k(D, GTtol, K=n), 2) for n in NS]


def check_recall(model, R, D, GTtol, golden_R=None):
    """R (what evaluate returned) is the reference's list; the GPU tie rule and the kernel's tie bounds are
    exposed next to it.  The golden list was produced by the reference itself in the build container: it
    must be reproduced wherever numpy orders the ties the same way (checked with the oracle)."""
    here = reference_recall_here(D, GTtol)
    assert R == here
    if golden_R is not None and here == [round(float(r), 2) for r in golden_R]:
        assert R == [round(float(r), 2) for r in golden_R]
    assert model.recall_gpu == [round(O.recall_at_k(D, GTtol, K=n, kind="stable"), 2) for n in NS]
    bounds = [tuple(round(x, 2) for x in O.recall_bounds(D, GTtol, n)) for n in NS]
    assert model.recall_bounds == bounds
    for r, g, (lo, hi) in zip(R, model.recall_gpu, bounds):
        assert lo - 1e-9 <= r <= hi + 1e-9 and lo - 1e-9 <= g <= hi + 1e-9


def write_png_u8(path, frame):
    from torchvision.io import write_png
    write_png(torch.from_numpy(frame)[None].contiguous(), path)


@pytest.fixture()
def example_tree(tmp_path, golden):
    """Recreate the reference's on-disk layout (dataset PNGs + CSV + GT + .pth) from a golden npz."""
    def make(name, dataset, camera, reference, query):
        g = golden(name)
        root = tmp_path / "lens"
        qdir = root / "dataset" / dataset / camera / query
        rdir = root / "dataset" / dataset / camera / reference
        os.makedirs(qdir), os.makedirs(rdir), os.makedirs(root / "models"), os.makedirs(root / "output")
        names = []
        for i, fr in enumerate(g["frames"]):
            n = f"image_{i:04d}.png"
            write_png_u8(str(qdir / n), fr)
            names.append(n)
        with open(root / "dataset" / (query + ".csv"), "w") as f:
            f.write("Image_name,index\n" + "".join(f"{n},{i}\n" for i, n in enumerate(names)))
        np.save(root / "dataset" / dataset / camera / f"{reference}_{query}_GT.npy", g["GT"])
        F, I = g["W_feat"].shape
        P = g["W_out"].shape[0]
        sd = {"feature_layer.thr": torch.zeros(1, F), "feature_layer.w.weight": torch.from_numpy(g["W_feat"]),
              "output_layer.thr": torch.zeros(1, P), "output_layer.w.weight": torch.from_numpy(g["W_out"])}
        torch.save(sd, root / "models" / f"{reference}_LENS_IN{I}_FN{F}_DB{P}.pth")
        return g, root
    return make


def test_run_inference_example(example_tree, monkeypatch):
    """python main.py --sim_mat --matching on the bundled example: same similarity matrix, same
    sequence-matched matrix, same Recall@N list as the reference's own run (0.63 / 0.84 / ...), with the
    GPU tie rule's list and the kernel-computed tie bounds exposed as attributes."""
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    monkeypatch.chdir(root.parent)
    args = default_args(matching=True, sim_mat=True, data_dir=str(root / "dataset") + "/")
    args.quiet = True
    model = LENS(args)
    name = generate_model_name(model)
    assert name == "example-reference_LENS_IN100_FN200_DB100.pth"
    R = run_inference(model, name, models_dir=str(root / "models"))
    assert np.array_equal(model.similarity.cpu().numpy(), g["S"].astype(np.float32))
    assert np.array_equal(model.dist_matrix_seq, g["D"])
    assert np.array_equal(model.GTtol, g["GTtol"])
    check_recall(model, R, g["D"], g["GTtol"], golden_R=g["R"])
    assert os.path.exists(os.path.join(model.output_folder, "lens.log"))


def test_run_inference_brisevent_all_queries(example_tree, monkeypatch):
    """The second bundled model end to end through run_inference with the reference's own command line
    (--dims 7 --roi_dim 7 -> kernel 1, centre index -1 wraps; --sequence_length 4; 724 queries x 641
    places).  The similarity matrix differs from the reference's own run in exactly the entries where the
    oracle does (a spike that the BLAS summation order of the reference moves across a query boundary);
    D, GTtol and Recall@N are the reference's."""
    from lens_b200.config import build_parser, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    g, root = example_tree("brisevent", "brisevent", "davis346", "sunset2", "sunset1")
    argv = [str(a) for a in g["argv"]]
    args = build_parser().parse_args(argv)
    assert (args.dataset, args.camera, args.reference, args.query) == ("brisevent", "davis346", "sunset2", "sunset1")
    args.data_dir = str(root / "dataset") + "/"
    args.quiet = True
    monkeypatch.chdir(root.parent)
    model = LENS(args)
    assert model.kernel_size == 1 and int(args.sequence_length) == int(g["sequence_length"])
    R = run_inference(model, generate_model_name(model), models_dir=str(root / "models"))
    S = model.similarity.cpu().numpy()
    assert S.shape == (724, 641)
    # oracle on the same frames: bit-equal to the GPU, and its differences from the reference's golden S
    # (2 of 464 084 counts, by one spike) are the GPU's differences
    roi, k, T = int(g["roi_dim"]), int(g["roi_dim"]) // int(g["dims"]), int(g["timebin"])
    onet = O.OracleSNN(g["W_feat"], g["W_out"], O.raster_uniforms(T, roi, k), T)
    So = onet.run_streams(O.pool(g["frames"], k)[None])[0]
    assert np.array_equal(S, So)
    diff = np.argwhere(S != g["S"].astype(np.float32))
    assert len(diff) <= 2 and np.all(np.abs(S - g["S"].astype(np.float32)) <= 1)
    L = int(g["sequence_length"])
    D_or = O.seqmatch(So.astype(np.float64), L)
    assert np.array_equal(model.dist_matrix_seq, D_or)
    # the sequence-matched matrix differs from the reference's only on the diagonals through those entries
    dD = np.argwhere(model.dist_matrix_seq != g["D"])
    assert len(dD) <= L * len(diff)
    for r, q in dD:
        assert any(0 <= qq - q < L and pp - r == qq - q for qq, pp in diff)
    assert np.array_equal(model.GTtol, g["GTtol"])
    check_recall(model, R, D_or, g["GTtol"], golden_R=g["R"])


def test_seam_loop_equals_fast_path(example_tree, monkeypatch):
    """The reference's per-query loop through `sinabs_model(spikes)` (run_model.py:234-241) and the
    batched run_streams fast path give the same similarity rows."""
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS
    from lens_b200.src.dataset import CustomImageDataset, ProcessImage
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    monkeypatch.chdir(root.parent)
    args = default_args(matching=False, data_dir=str(root / "dataset") + "/", query_places=6)
    args.quiet = True
    model = LENS(args)
    model.load_model(str(root / "models" / generate_model_name(model)))
    ds = CustomImageDataset(model.dataset_file, model.query_dir, model.kernel_size, transform=ProcessImage(),
                            skip=1, max_samples=6, is_spiking=True, time_window=model.timebin)
    model.build_network()
    rows = []
    for i in range(len(ds)):
        spikes, label, _, _ = ds[i]                       # [T, 1, roi, roi] float raster (reference format)
        assert label == i
        out = model.sinabs_model(spikes.cuda())            # [T, P]
        rows.append(out.sum(dim=0))
    S_loop = torch.stack(rows).cpu().numpy()
    assert np.array_equal(S_loop, g["S"][:6].astype(np.float32))
    model.build_network()                                  # fresh state
    S_fast = model.similarity_matrix(ds).cpu().numpy()
    assert np.array_equal(S_fast, S_loop)


def test_recallAtK_signature(golden):
    from lens_b200.src.metrics import recallAtK
    g = golden("config1")
    D, GT = g["D"], g["GTtol"]
    for K in (1, 5, 25):
        assert abs(recallAtK(D, GT, K=K) - O.recall_at_k(D, GT, K=K)) < 1e-12      # the reference's value
    soft = np.roll(GT, 1, axis=0) | GT
    assert abs(recallAtK(D, GT, GTsoft=soft, K=5) - O.recall_at_k(D, GT, GTsoft=soft, K=5)) < 1e-12
    with pytest.raises(AssertionError):
        recallAtK(D, GT[:-1], K=1)


def test_sequence_length_zero_branch(example_tree, monkeypatch):
    """sequence_length = 0 keeps the raw similarity matrix (run_model.py:254)."""
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    monkeypatch.chdir(root.parent)
    args = default_args(matching=True, sequence_length=0, data_dir=str(root / "dataset") + "/")
    args.quiet = True
    model = LENS(args)
    R = run_inference(model, generate_model_name(model), models_dir=str(root / "models"))
    S = g["S"].astype(np.float64)
    assert np.array_equal(model.dist_matrix_seq, S)
    GTtol = O.make_gt_tol(g["GT"], 0, 3)
    check_recall(model, R, S, GTtol)


def test_createPR_matches_reference(golden):
    """CUDA createPR (matching='single') == the reference's own lists on both bundled runs."""
    from lens_b200.src.metrics import createPR
    for name in ("config1", "brisevent"):
        g = golden(name)
        P, R = createPR(g["D"].T, g["GTtol"].T, None, matching="single", n_thresh=100)
        assert np.array_equal(np.array(P, dtype=np.float64), g["PR_P"], equal_nan=True)
        assert np.array_equal(np.array(R, dtype=np.float64), g["PR_R"], equal_nan=True)


def test_createPR_multi_matches_reference(golden):
    """CUDA createPR(matching='multi'), the reference's default mode: the reference's own lists on both bundled
    runs (n_thresh 100 and 7), with a soft ground truth, and on a small matrix full of ties."""
    from lens_b200.src.metrics import createPR
    pm = golden("pr_multi")

    def same(got, key):
        P, R = got
        assert np.array_equal(np.array(P, dtype=np.float64), pm[key + "/P"], equal_nan=True), key
        assert np.array_equal(np.array(R, dtype=np.float64), pm[key + "/R"], equal_nan=True), key
    for name in ("config1", "brisevent"):
        g = golden(name)
        S, GT = g["D"].T, g["GTtol"].T
        for n in (100, 7):
            same(createPR(S, GT, None, matching="multi", n_thresh=n), f"{name}/n{n}")
        same(createPR(S, GT, None, GTsoft=np.roll(GT, 1, axis=1) | GT, matching="multi", n_thresh=50), f"{name}/soft")
    same(createPR(pm["random/S"], pm["random/GT"], None, n_thresh=20), "random")      # 'multi' is the default


def test_pr_curve_flag(example_tree, monkeypatch):
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    monkeypatch.chdir(root.parent)
    args = default_args(matching=True, PR_curve=True, data_dir=str(root / "dataset") + "/")
    args.quiet = True
    model = LENS(args)
    run_inference(model, generate_model_name(model), models_dir=str(root / "models"))
    assert np.array_equal(np.array(model.lens_PR["Precision"], dtype=np.float64), g["PR_P"], equal_nan=True)
    assert np.array_equal(np.array(model.lens_PR["Recall"], dtype=np.float64), g["PR_R"], equal_nan=True)


def test_sad_baseline_matches_reference(golden):
    """SAD baseline (lens/src/sad.py) on the GPU: 1/distance matrix, PR lists and Recall@N equal to the
    reference's own run_sad outputs on both bundled datasets."""
    from lens_b200 import ops
    from lens_b200.src.sad import sad_distance_matrix
    from lens_b200.src.metrics import createPR, recallAtK
    for name in ("config1", "brisevent"):
        g = golden(name)
        L = int(g["sequence_length"])
        q = torch.from_numpy(g["frames"].reshape(g["frames"].shape[0], -1))
        r = torch.from_numpy(g["ref_frames"].reshape(g["ref_frames"].shape[0], -1))
        D = sad_distance_matrix(q, r, L)
        sim = ops.reciprocal(D.contiguous()).cpu().numpy()
        if "sad_sim" in g.files:
            assert np.array_equal(sim, g["sad_sim"])
        else:                   # a large matrix is stored as the SHA-256 of its float32 bytes (make_golden.py)
            assert sim.dtype == np.float32 and sim.shape == g["D"].shape
            assert hashlib.sha256(sim.tobytes()).hexdigest() == str(g["sad_sim_sha256"])
        P, R = createPR(sim, g["GTtol"], None, datatype="SAD", matching="single", n_thresh=100)
        assert np.array_equal(np.array(P, dtype=np.float64), g["sad_P"], equal_nan=True)
        assert np.array_equal(np.array(R, dtype=np.float64), g["sad_R"], equal_nan=True)
        rec = [round(recallAtK(sim, g["GTtol"], K=n), 2) for n in NS]
        here = reference_recall_here(sim, g["GTtol"])
        assert rec == here
        if here == [round(float(r), 2) for r in g["sad_recall"]]:
            assert rec == [round(float(r), 2) for r in g["sad_recall"]]
        for mine, ref, n in zip(rec, g["sad_recall"], NS):
            lo, hi = O.recall_bounds(sim, g["GTtol"], n)
            assert round(lo, 2) - 1e-9 <= mine <= round(hi, 2) + 1e-9
            assert round(lo, 2) - 1e-9 <= ref <= round(hi, 2) + 1e-9


def test_sad_flag(example_tree, monkeypatch, golden):
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    # the reference frames live next to the query frames in the reference's layout
    rdir = root / "dataset" / "example" / "davis128" / "example-reference"
    for i, fr in enumerate(g["ref_frames"]):
        write_png_u8(str(rdir / f"image_{i:04d}.png"), fr)
    monkeypatch.chdir(root.parent)
    args = default_args(matching=True, PR_curve=True, sad=True, data_dir=str(root / "dataset") + "/")
    args.quiet = True
    model = LENS(args)
    run_inference(model, generate_model_name(model), models_dir=str(root / "models"))
    assert np.array_equal(np.array(model.sad_PR["Precision"], dtype=np.float64), g["sad_P"], equal_nan=True)
    assert len(model.sad_Recall) == 6


def test_online_matcher_matches_reference_arithmetic():
    """OnlineMatcher (run_speck.py:155-226 on the GPU) against the oracle state machine and scipy."""
    from scipy.signal import convolve2d
    from lens_b200.online import OnlineMatcher
    rng = np.random.default_rng(21)
    for P, L in [(100, 4), (1000, 2), (37, 5), (8, 1)]:
        gpu, cpu = OnlineMatcher(P, L), O.OnlineMatcherOracle(P, L)
        n_match = 0
        for i in range(40):
            counts = rng.integers(0, 12, size=P).astype(np.float32)
            a, b = gpu.push(torch.from_numpy(counts).cuda()), cpu.push(counts)
            assert (a is None) == (b is None)
            if a is not None:
                n_match += 1
                assert np.array_equal(a[0].cpu().numpy(), b[0])
                assert np.array_equal(a[1].cpu().numpy(), b[1])
                seq = gpu.sequence.cpu().numpy()
                ref = convolve2d(seq.T, np.eye(L, dtype=np.float32), mode="same") / L
                assert np.array_equal(a[1].cpu().numpy(), ref)
        assert n_match == 2
        assert np.array_equal(gpu.similarity_matrix().cpu().numpy(), cpu.matrix.T)


def test_evaluate_option_space(example_tree, monkeypatch):
    """LENS.evaluate with other --sequence_length / --GT_tolerance values == the reference's own run on
    the bundled example (tests/golden/options.npz): D, GTtol and Recall@N identical;
    --sequence_length 1 fails with the reference's assertion."""
    from lens_b200.config import default_args, generate_model_name
    from lens_b200.run_model import LENS, run_inference
    opt = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "options.npz"))
    g, root = example_tree("config1", "example", "davis128", "example-reference", "example-query")
    monkeypatch.chdir(root.parent)
    for L, tol in opt["variants"]:
        key = f"L{L}_tol{tol}"
        args = default_args(matching=True, sim_mat=True, data_dir=str(root / "dataset") + "/",
                            sequence_length=int(L), GT_tolerance=int(tol))
        args.quiet = True
        model = LENS(args)
        name = generate_model_name(model)
        if str(opt[key + "/error"]):
            with pytest.raises(AssertionError, match="same shape"):
                run_inference(model, name, models_dir=str(root / "models"))
            continue
        R = run_inference(model, name, models_dir=str(root / "models"))
        assert np.array_equal(np.asarray(model.dist_matrix_seq, dtype=np.float32), opt[key + "/D"]), key
        assert np.array_equal(model.GTtol, opt[key + "/GTtol"]), key
        check_recall(model, R, np.asarray(model.dist_matrix_seq), model.GTtol, golden_R=opt[key + "/R"])
        for want, K in zip(opt[key + "/R"], NS):
            lo, hi = O.recall_bounds(opt[key + "/D"], model.GTtol, K)
            assert round(lo, 2) <= want <= round(hi, 2), (key, K)
