#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by running the REAL reference code.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

What runs for real (imported unmodified from /root/reference):
  lens/run_model.py   LENS.__init__, run_inference, LENS.evaluate (:122-338)
  lens/src/dataset.py CustomImageDataset/ProcessImage (PNG -> /255 -> seed-50 raster)
  lens/src/blitnet.py SNNLayer (weight container)
  lens/src/metrics.py recallAtK
  lens/src/loggers.py model_logger
What is stubbed because the wheels are not installable here (no network):
  sinabs     -> tests/golden/sinabs_stub.py (torch restatement of IAFSqueeze/from_model)
  matplotlib, seaborn, prettytable, skimage -> inert fakes (plots/tables only)
The reference tree is read-only, so the script runs from a scratch directory whose
`lens/models` and `lens/dataset` are symlinks into /root/reference and whose
`lens/output` is real.

Outputs (committed): config1.npz (bundled example model + data) and brisevent.npz
(bundled sunset2 model, sunset1 queries) holding inputs (frames, weights, GT) and
the reference outputs (similarity matrix S, sequence-matched D, GTtol, Recall@N,
final membrane potentials, hidden-layer spike statistics).  Every fixture stays under
1 MB: the members are LZMA-compressed, and a SAD similarity matrix of more than
SAD_SIM_MAX_ENTRIES entries is stored as the SHA-256 of its float32 bytes (C order).
"""
import argparse
import hashlib
import os
import sys
import tempfile
import types
import zipfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
SAD_SIM_MAX_ENTRIES = 100_000


def savez_lzma(path, **arrays):
    """np.savez with LZMA-compressed members (np.load reads them like any other .npz)."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            with z.open(k + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


class _Anything:
    """Object that swallows any attribute access / call (for plotting fakes)."""
    def __getattr__(self, k):
        return _Anything()

    def __call__(self, *a, **k):
        return _Anything()

    def __iter__(self):
        return iter((_Anything(), _Anything()))


def _fake_module(name, **attrs):
    m = types.ModuleType(name)
    def _ga(k):
        if k.startswith("__"):
            raise AttributeError(k)
        return _Anything()
    m.__getattr__ = _ga  # type: ignore
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def install_fakes():
    sys.path.insert(0, HERE)
    import sinabs_stub
    sinabs_stub.install()
    mpl = _fake_module("matplotlib")
    mpl.pyplot = _fake_module("matplotlib.pyplot")
    _fake_module("seaborn")

    class PrettyTable:
        field_names = None

        def add_row(self, r):
            self.row = r

        def __str__(self):
            return f"{self.field_names} {getattr(self, 'row', None)}"
    _fake_module("prettytable", PrettyTable=PrettyTable)
    sk = _fake_module("skimage")

    def imread(path):
        from PIL import Image
        return np.array(Image.open(path))
    sk.io = _fake_module("skimage.io", imread=imread)
    return sinabs_stub


def imread_u8(path):
    from PIL import Image
    return np.array(Image.open(path))


def run_case(stub, name, argv, out_path, full_steps=2):
    import main as ref_main  # /root/reference/main.py (argparse surface)
    from lens.run_model import LENS, run_inference
    import lens.run_model as rm
    import sinabs.from_torch as ft

    # ---- parse with the reference's own argparse definitions
    captured = {}
    orig_init = ref_main.initialize_and_run_model
    ref_main.initialize_and_run_model = lambda a: captured.setdefault("args", a)
    old_argv = sys.argv
    sys.argv = ["main.py"] + argv
    try:
        ref_main.parse_network()
    finally:
        sys.argv = old_argv
        ref_main.initialize_and_run_model = orig_init
    args = captured["args"]
    from lens.tools import checker
    checker.check_args(args)

    # ---- hooks: keep a handle on the converted network, record layer outputs
    holder = {}
    real_from_model = stub.from_model

    def from_model(*a, **k):
        net = real_from_model(*a, **k)
        holder["net"] = net
        for m in net.spiking_model:
            if isinstance(m, stub.IAFSqueeze):
                m.record = []
        return net
    rm.from_model = from_model
    ft.from_model = from_model

    rec = {}
    real_recall = rm.recallAtK

    def recallAtK(S, GT, GTsoft=None, K=1):
        rec["D"] = np.array(S)
        rec["GTtol"] = np.array(GT)
        return real_recall(S, GT, GTsoft, K=K)
    rm.recallAtK = recallAtK

    model = LENS(args)
    model_name = ref_main.generate_model_name(model)
    torch.set_num_threads(1)
    R = run_inference(model, model_name)

    net = holder["net"]
    iafs = [m for m in net.spiking_model if isinstance(m, stub.IAFSqueeze)]
    assert len(iafs) == 3
    T = args.timebin
    s0 = [r for r in iafs[0].record]
    s1 = [r for r in iafs[1].record]
    s2 = [r for r in iafs[2].record]
    Q = len(s2)
    S = np.stack([r.sum(0).reshape(-1).numpy() for r in s2]).astype(np.float64)
    hidden_counts = np.stack([r.sum(0).reshape(-1).numpy() for r in s1]).astype(np.int32)
    in_counts = np.stack([r.sum(0).reshape(-1).numpy() for r in s0]).astype(np.int32)
    assert S.shape == (args.query_places, args.reference_places)
    # IAF#0 must be the identity on the (binary) sub-sampled raster
    hidden_hist = np.bincount(torch.cat(s1).reshape(-1).to(torch.int64).numpy(), minlength=8)
    out_hist = np.bincount(torch.cat(s2).reshape(-1).to(torch.int64).numpy(), minlength=8)

    # ---- inputs as fixtures
    import pandas as pd
    from torchvision.io import read_image
    df = pd.read_csv(model.dataset_file)
    names = list(df.iloc[::args.filter, 0][:args.query_places])
    frames = np.stack([read_image(os.path.join(model.query_dir, n)).numpy()[0] for n in names])
    sd = torch.load(os.path.join("./lens/models", model_name), weights_only=True, map_location="cpu")
    GT = np.load(os.path.join(args.data_dir, args.dataset, args.camera,
                              args.reference + "_" + args.query + "_GT.npy"))
    torch.manual_seed(50)
    U = torch.rand(T, args.roi_dim * args.roi_dim)
    # precision-recall curve exactly as run_model.py:321 calls it (figure goes to the fake matplotlib)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        PR_P, PR_R = rm.createPR(rec["D"].T, rec["GTtol"].T, model.output_folder, matching="single", n_thresh=100)
    # SAD baseline exactly as run_model.py:330 calls it (lens/src/sad.py, skimage.io.imread -> PIL)
    import lens.src.sad as sad_mod
    sad_rec = {}
    real_cpr = sad_mod.createPR

    def spy_createPR(S, GTm, *a, **k):
        sad_rec["sim"] = np.array(S)
        return real_cpr(S, GTm, *a, **k)
    sad_mod.createPR = spy_createPR
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sad_PR, sad_Recall = sad_mod.run_sad(model.reference_dir, model.query_dir, rec["GTtol"], model.output_folder,
                                             args.sequence_length)
    ref_files = sorted(os.listdir(model.reference_dir), key=sad_mod.natural_sort_key)
    ref_frames = np.stack([imread_u8(os.path.join(model.reference_dir, f)) for f in ref_files if f.endswith(".png")])
    qry_files = sorted(os.listdir(model.query_dir), key=sad_mod.natural_sort_key)
    sad_query_frames_equal = len([f for f in qry_files if f.endswith(".png")])
    h = hashlib.sha256()
    for r in s2:
        h.update(r.to(torch.uint8).numpy().tobytes())
    sad_sim = sad_rec["sim"].astype(np.float32)
    if sad_sim.size > SAD_SIM_MAX_ENTRIES:
        sad = dict(sad_sim_sha256=hashlib.sha256(sad_sim.tobytes()).hexdigest())
    else:
        sad = dict(sad_sim=sad_sim)

    savez_lzma(
        out_path,
        argv=np.array(argv),
        dims=args.dims, roi_dim=args.roi_dim, timebin=T, sequence_length=args.sequence_length,
        GT_tolerance=args.GT_tolerance, reference_places=args.reference_places,
        query_places=args.query_places, feature_multiplier=args.feature_multiplier,
        frames=frames.astype(np.uint8),
        W_feat=sd["feature_layer.w.weight"].numpy(), W_out=sd["output_layer.w.weight"].numpy(),
        GT=GT.astype(np.uint8),
        U_sha256=hashlib.sha256(U.numpy().tobytes()).hexdigest(),
        S=S.astype(np.uint16), D=rec["D"].astype(np.float32), GTtol=rec["GTtol"].astype(np.uint8),
        R=np.array(R, dtype=np.float64),
        PR_P=np.array(PR_P, dtype=np.float64), PR_R=np.array(PR_R, dtype=np.float64),
        ref_frames=ref_frames.astype(np.uint8), n_query_files=sad_query_frames_equal,
        **sad, sad_recall=np.array(sad_Recall, dtype=np.float64),
        sad_P=np.array(sad_PR["Precision"], dtype=np.float64), sad_R=np.array(sad_PR["Recall"], dtype=np.float64),
        v0=iafs[0].v_mem.reshape(-1).numpy(), v1=iafs[1].v_mem.reshape(-1).numpy(),
        v2=iafs[2].v_mem.reshape(-1).numpy(),
        hidden_counts=hidden_counts.astype(np.uint16), in_counts=in_counts.astype(np.uint16),
        hidden_hist=hidden_hist, out_hist=out_hist,
        hidden_steps=torch.stack(s1[:full_steps]).to(torch.uint8).numpy(),
        out_steps=torch.stack(s2[:full_steps]).to(torch.uint8).numpy(),
        out_steps_sha256=h.hexdigest(),
    )
    assert S.max() < 65536
    print(f"[{name}] Q={Q} S.shape={S.shape} S.max={S.max()} S.mean={S.mean():.3f} R={R}")
    print(f"[{name}] hidden spike histogram {hidden_hist.tolist()} output {out_hist.tolist()}")
    return R


def run_options(stub, out_path):
    """The tail of evaluate() (sequence matching, GT slicing/dilation, Recall@N) for other option values:
    the reference's whole run_inference on the bundled example with --sequence_length / --GT_tolerance varied.
    Stores D (what the reference hands to recallAtK), GTtol and R per variant, or the exception it raises."""
    import main as ref_main
    from lens.run_model import LENS, run_inference
    import lens.run_model as rm
    out = {}
    variants = [(0, 3), (1, 3), (2, 0), (2, 1), (3, 3), (4, 2), (10, 3), (25, 5)]
    for L, tol in variants:
        argv = ["--sim_mat", "--matching", "--nocuda", "--sequence_length", str(L), "--GT_tolerance", str(tol)]
        captured = {}
        orig_init = ref_main.initialize_and_run_model
        ref_main.initialize_and_run_model = lambda a: captured.setdefault("args", a)
        old_argv = sys.argv
        sys.argv = ["main.py"] + argv
        try:
            ref_main.parse_network()
        finally:
            sys.argv = old_argv
            ref_main.initialize_and_run_model = orig_init
        args = captured["args"]
        rec = {}
        real_recall = rm.recallAtK

        def recallAtK(S, GT, GTsoft=None, K=1, rec=rec, real_recall=real_recall):
            rec["D"] = np.array(S)
            rec["GTtol"] = np.array(GT)
            return real_recall(S, GT, GTsoft, K=K)
        rm.recallAtK = recallAtK
        key = f"L{L}_tol{tol}"
        try:
            model = LENS(args)
            torch.set_num_threads(1)
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                R = run_inference(model, ref_main.generate_model_name(model))
            out[key + "/D"] = rec["D"].astype(np.float32)
            out[key + "/GTtol"] = rec["GTtol"].astype(np.uint8)
            out[key + "/R"] = np.array(R, dtype=np.float64)
            out[key + "/error"] = np.array("")
            print(f"[options {key}] D{rec['D'].shape} GTtol{rec['GTtol'].shape} R={R}")
        except Exception as e:          # noqa: BLE001 - the outcome itself is the fixture
            out[key + "/error"] = np.array(type(e).__name__ + ": " + str(e)[:200])
            print(f"[options {key}] raised {type(e).__name__}: {e}")
        finally:
            rm.recallAtK = real_recall
    out["variants"] = np.array(variants)
    np.savez_compressed(out_path, **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    stub = install_fakes()
    sys.path.insert(0, REF)
    work = tempfile.mkdtemp(prefix="lens_golden_")
    os.makedirs(os.path.join(work, "lens", "output"))
    os.symlink(os.path.join(REF, "lens", "models"), os.path.join(work, "lens", "models"))
    os.symlink(os.path.join(REF, "lens", "dataset"), os.path.join(work, "lens", "dataset"))
    os.chdir(work)
    cases = {
        "config1": ["--sim_mat", "--matching", "--nocuda"],
        "brisevent": ["--dataset", "brisevent", "--camera", "davis346", "--reference", "sunset2",
                      "--query", "sunset1", "--dims", "7", "--roi_dim", "7",
                      "--feature_multiplier", "1.3", "--reference_places", "641",
                      "--query_places", "724", "--sequence_length", "4", "--matching", "--nocuda"],
    }
    for name, argv in cases.items():
        if a.only and a.only != name:
            continue
        run_case(stub, name, argv, os.path.join(HERE, name + ".npz"))
    if not a.only or a.only == "options":
        run_options(stub, os.path.join(HERE, "options.npz"))


if __name__ == "__main__":
    main()
