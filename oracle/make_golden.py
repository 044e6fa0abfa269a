"""TEST INFRASTRUCTURE — generates tests/golden/*.npz and gtsfm_bases.json by running the UNMODIFIED reference in the build container.

    python -m oracle.make_golden            # needs /root/reference; not runnable on the GPU box

For every hot-path row it (1) runs the reference module (oracle/ref_modules.py) with the seeded weights of
gtsfm_b200/synthetic.py on seeded inputs, (2) runs the CPU restatement in oracle/*_ref.py on the same inputs and
asserts they agree (the "pin"), (3) writes the reference's outputs as the committed fixture.  The fixtures store
outputs (and inputs only where they cannot be regenerated from a seed: the two lund-door frames).
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from gtsfm_b200 import synthetic as syn  # noqa: E402
from oracle import lightglue_ref, ref_modules, superglue_ref, superpoint_ref, verifier_ref  # noqa: E402

OUT = ROOT / "tests" / "golden"
LUND = ref_modules.REF / "tests" / "data" / "set1_lund_door" / "images"


def versions():
    import cv2

    return dict(torch=torch.__version__, numpy=np.__version__, cv2=cv2.__version__)


def load_lund_gray(idx: int) -> np.ndarray:
    """Loader semantics: PIL decode, cubic resize so the short side is 760 (loader_base.py:160-200,
    utils/images.py:102-129,150-220), then the wrapper's gray conversion."""
    import cv2
    from PIL import Image

    rgb = np.asarray(Image.open(LUND / f"DSC_{idx:04d}.JPG").convert("RGB"))
    h, w = rgb.shape[:2]
    if min(h, w) > 760:
        if h <= w:
            nh, nw = 760, int(np.round(w * 760 / float(h)))
        else:
            nw, nh = 760, int(np.round(h * 760 / float(w)))
        rgb = cv2.resize(rgb, (nw, nh), interpolation=cv2.INTER_CUBIC)
    gray = cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY)
    assert np.array_equal(gray, superpoint_ref.rgb_to_gray_u8(rgb)), "gray restatement differs from cv2"
    return gray


def run_ref_superpoint(model, gray_u8):
    x = torch.from_numpy(gray_u8.astype(np.float32) / 255.0)[None, None]
    with torch.no_grad():
        out = model({"image": x})
    return (out["keypoints"][0].numpy(), out["scores"][0].numpy(), np.ascontiguousarray(out["descriptors"][0].numpy().T))


def golden_superpoint():
    sd = syn.superpoint_state_dict(0)
    model = ref_modules.ref_superpoint(sd)
    cases = {
        "tiny": superpoint_ref.rgb_to_gray_u8(syn.synthetic_frame(0, 120, 160)),
        "odd": superpoint_ref.rgb_to_gray_u8(syn.synthetic_frame(3, 203, 317)),  # not divisible by 8
        "vga": superpoint_ref.rgb_to_gray_u8(syn.synthetic_frame(1, 480, 640)),
        "lund1": load_lund_gray(1),
        "lund2": load_lund_gray(2),
    }
    feats = {}
    for name, gray in cases.items():
        kp, sc, desc = run_ref_superpoint(model, gray)
        kp2, sc2, desc2 = superpoint_ref.superpoint_forward(gray.astype(np.float32) / 255.0, sd)
        assert np.array_equal(kp, kp2) and np.array_equal(sc, sc2), f"superpoint restatement != reference on {name}"
        err = float(np.abs(desc - desc2).max())
        assert err <= 1e-6, (name, err)
        # wrapper top-k (gtsfm/.../superpoint.py:90, keypoints.py:101-110)
        sel = np.argpartition(-sc, 5000)[:5000] if len(kp) > 5000 else np.arange(len(kp))
        stride = max(1, len(kp) // 256)
        fx = dict(
            keypoints=kp.astype(np.int16), scores=sc, topk_sel=sel.astype(np.int32),
            desc_rows=np.arange(0, len(kp), stride, dtype=np.int32), desc=desc[::stride].copy(),
            desc_checksum=np.float64(desc.astype(np.float64).sum()), restatement_desc_err=np.float64(err),
            **{f"v_{k}": np.array(v) for k, v in versions().items()},
        )
        if name.startswith("lund"):
            fx["gray"] = gray
        if name == "tiny":
            fx["desc_full"] = desc
        np.savez_compressed(OUT / f"superpoint_{name}.npz", **fx)
        feats[name] = (kp, sc, desc, gray.shape)
        if name == "lund1":
            feats["lund1_gray"] = gray
        print(f"superpoint {name}: {gray.shape} N={len(kp)} restatement desc err {err:.2e}")
    return feats


def run_ref_lightglue(model, kp0, d0, kp1, d1, shape0, shape1):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))[None]
    data = {  # lightglue_matcher.py:82-99
        "image0": {"keypoints": t(kp0), "descriptors": t(d0), "image": torch.empty(1, 1, shape0[0], shape0[1])},
        "image1": {"keypoints": t(kp1), "descriptors": t(d1), "image": torch.empty(1, 1, shape1[0], shape1[1])},
    }
    with torch.no_grad():
        out = model(data)
    return out["matches"][0].numpy(), int(out["stop"]), out["prune0"][0].numpy(), out["prune1"][0].numpy(), out["scores"][0].numpy()


def golden_lightglue(feats):
    cases = [("full", 5, 300, 350), ("full", 6, 1024, 900), ("prune", 7, 700, 640), ("stop", 8, 512, 512),
             ("prune", 9, 37, 5), ("stop", 10, 2048, 1900)]
    for profile, seed, n0, n1 in cases:
        sd = syn.lightglue_state_dict(2, profile)
        model = ref_modules.ref_lightglue(sd)
        kp0, sc0, d0, kp1, sc1, d1, gt = syn.synthetic_features(seed, n0, n1)
        m, stop, pr0, pr1, ms = run_ref_lightglue(model, kp0, d0, kp1, d1, (480, 640), (480, 640))
        tr = {}
        m2 = lightglue_ref.lightglue_match(kp0, d0, kp1, d1, sd, trace=tr)
        assert np.array_equal(m, m2), f"lightglue restatement != reference ({profile},{seed}): {len(m)} vs {len(m2)}"
        assert tr["stop"] == stop
        assert len(m) >= 0.25 * min(n0, n1) or n1 < 10, (profile, seed, len(m))
        np.savez_compressed(OUT / f"lightglue_{profile}_{seed}.npz", matches=m, stop=stop, sizes=tr["sizes"],
                            prune0=pr0.astype(np.int8), prune1=pr1.astype(np.int8), mscores=ms,
                            seed=seed, n0=n0, n1=n1, profile=profile)
        print(f"lightglue {profile} seed {seed} ({n0},{n1}): K={len(m)} stop={stop} sizes={tr['sizes'].tolist()[-1]}")
    # real-image features: lund door pair through the wrapper top-k
    sd = syn.lightglue_state_dict(2, "sharp")
    model = ref_modules.ref_lightglue(sd)
    (kpa, sca, da, sha), (kpb, scb, db, shb) = feats["lund1"], feats["lund2"]
    sela = np.argpartition(-sca, 5000)[:5000] if len(kpa) > 5000 else np.arange(len(kpa))
    selb = np.argpartition(-scb, 5000)[:5000] if len(kpb) > 5000 else np.arange(len(kpb))
    m, stop, *_ = run_ref_lightglue(model, kpa[sela], da[sela], kpb[selb], db[selb], sha, shb)
    m2 = lightglue_ref.lightglue_match(kpa[sela], da[sela], kpb[selb], db[selb], sd)
    assert np.array_equal(m, m2)
    np.savez_compressed(OUT / "lightglue_lund_1_2.npz", matches=m, stop=stop, profile="sharp")
    print(f"lightglue lund 1-2: K={len(m)} stop={stop}")
    # two overlapping crops of lund1 (offsets are multiples of 8, so interior features coincide): a detect -> top-k ->
    # match chain with many true matches; inputs are derivable from superpoint_lund1.npz's gray.
    sp_sd = syn.superpoint_state_dict(0)
    gray = feats["lund1_gray"]
    ca, cb = gray[0:1000, 0:700], gray[40:1040, 24:724]
    fa = superpoint_ref.detect_and_describe(ca, sp_sd, 5000)
    fb = superpoint_ref.detect_and_describe(cb, sp_sd, 5000)
    for profile in ("sharp",):
        sd = syn.lightglue_state_dict(2, profile)
        model = ref_modules.ref_lightglue(sd)
        m, stop, *_ = run_ref_lightglue(model, fa[0], fa[2], fb[0], fb[2], ca.shape, cb.shape)
        m2 = lightglue_ref.lightglue_match(fa[0], fa[2], fb[0], fb[2], sd)
        assert np.array_equal(m, m2)
        good = np.abs((fa[0][m[:, 0]] - fb[0][m[:, 1]]) - [24, 40]).max(1) < 0.5
        np.savez_compressed(OUT / f"pipeline_lund_crops_{profile}.npz", matches=m, stop=stop, kp_a=fa[0].astype(np.int16),
                            kp_b=fb[0].astype(np.int16), sc_a=fa[1], sc_b=fb[1], profile=profile)
        print(f"pipeline lund crops {profile}: Na={len(fa[0])} Nb={len(fb[0])} K={len(m)} geometrically right {good.sum()} stop={stop}")


def golden_superglue():
    sd = syn.superglue_state_dict(1)
    model = ref_modules.ref_superglue(sd, weights="outdoor", sinkhorn_iterations=20, descriptor_dim=256)
    for seed, n0, n1 in [(5, 300, 350), (6, 1024, 900), (9, 40, 3)]:
        kp0, sc0, d0, kp1, sc1, d1, gt = syn.synthetic_features(seed, n0, n1)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))[None]
        data = {"keypoints0": t(kp0), "keypoints1": t(kp1), "descriptors0": t(d0.T), "descriptors1": t(d1.T),
                "scores0": t(sc0), "scores1": t(sc1), "image0": torch.empty(1, 1, 480, 640), "image1": torch.empty(1, 1, 480, 640)}
        with torch.no_grad():
            pred = model(data)
        m0 = pred["matches0"][0].numpy()
        valid = m0 > -1
        rows = np.hstack([np.arange(n0)[valid].reshape(-1, 1), np.arange(n1)[m0[valid]].reshape(-1, 1)]).astype(np.uint32)
        rows2 = superglue_ref.superglue_match(kp0, sc0, d0, kp1, sc1, d1, (480, 640, 3), (480, 640, 3), sd)
        assert np.array_equal(rows, rows2), f"superglue restatement != reference (seed {seed}): {len(rows)} vs {len(rows2)}"
        np.savez_compressed(OUT / f"superglue_{seed}.npz", matches=rows, mscores=pred["matching_scores0"][0].numpy()[valid],
                            seed=seed, n0=n0, n1=n1)
        print(f"superglue seed {seed} ({n0},{n1}): K={len(rows)}")


def golden_verifier():
    import cv2

    for seed, k, ratio in [(1, 200, 0.5), (2, 1000, 0.8), (3, 2000, 0.3), (4, 500, 0.6)]:
        kp1, kp2, matches, K, R, t, is_in = verifier_ref.synthetic_two_view(seed, k, ratio)
        Rc, tc, rows, r, E = verifier_ref.verify_cv2(kp1, kp2, matches, K, K, True, 4.0)
        Rf, tf, rowsf, rf, Ef = verifier_ref.verify_cv2(kp1, kp2, matches, K, K, False, 4.0)
        np.savez_compressed(OUT / f"verifier_{seed}.npz", seed=seed, k=k, ratio=ratio, R_gt=R, t_gt=t, is_inlier=is_in,
                            R_cv=Rc, t_cv=tc, rows_cv=rows, ratio_cv=r, E_cv=E,
                            R_cvF=Rf, t_cvF=tf, rows_cvF=rowsf, ratio_cvF=rf, cv2_version=cv2.__version__)
        print(f"verifier seed {seed} K={k}: cv2 E inliers {len(rows)} (gt {is_in.sum()}), rot err "
              f"{verifier_ref.rot_angle_deg(R, Rc):.3f} deg, F inliers {len(rowsf)}")


def golden_verifier_argoverse():
    """The reference's own known-answer test for this path (tests/frontend/verifier/test_verifier_argoverse.py:32-104): 20
    hand-labelled correspondences of an Argoverse front-centre image pair, the log's intrinsics, the expected relative pose
    (Euler zyx [-0.37, 32.47, -0.42] deg +-1, i1ti2 [0.21, -0.0024, 0.976] +-0.01) at a 0.5 px threshold.  The labelled
    points (test DATA of the reference, 20 x 4 numbers) are stored as a fixture together with what cv2 returns for them."""
    import pickle

    import cv2

    src = Path("/root/reference/tests/data/argoverse/labeled_correspondences/argoverse_315975640448534784__315975643412234000.pkl")
    with open(src, "rb") as f:
        d = pickle.load(f)
    uv1 = np.stack([np.array(d["x1"]), np.array(d["y1"])], -1).astype(np.float32)  # test_verifier_argoverse.py:51-52
    uv2 = np.stack([np.array(d["x2"]), np.array(d["y2"])], -1).astype(np.float32)
    K = (1392.1069298937407, 980.1759848618066, 604.3534182680304)  # fx, px, py (:62-70), k1 = k2 = 0
    matches = np.stack([np.arange(len(uv1)), np.arange(len(uv1))], -1).astype(np.int64)
    R, t, rows, ratio, E = verifier_ref.verify_cv2(uv1, uv2, matches, K, K, True, 0.5)
    np.savez_compressed(OUT / "verifier_argoverse.npz", uv1=uv1, uv2=uv2, K=np.array(K), thr_px=0.5,
                        euler_zyx_deg_gt=np.array([-0.37, 32.47, -0.42]), i1ti2_gt=np.array([0.21, -0.0024, 0.976]),
                        euler_tol_deg=1.0, t_tol=0.01, R_cv=R, t_cv=t, rows_cv=rows, cv2_version=cv2.__version__)
    e, tt = verifier_ref.pose_to_euler_zyx_and_i1ti2(R, t)
    print(f"verifier argoverse: cv2 euler zyx {np.round(e, 2)}, i1ti2 {np.round(tt, 3)}, inliers {len(rows)}/20")


# ---- round 2: the configurations the bench times and north_star names ------------------------------------------------
def golden_lightglue_bench():
    """(a) The BENCHED matcher configuration: 5000 x 5000 keypoints, 'bench' weights, 9 full layers, nothing pruned.
    Inputs regenerate from a seed (bit-identical on the GPU box), so match indices must be EXACTLY the reference's."""
    sd = syn.lightglue_state_dict(2, "bench")
    model = ref_modules.ref_lightglue(sd)
    for seed, n0, n1 in [(11, 5000, 5000), (12, 1024, 1024)]:
        kp0, sc0, d0, kp1, sc1, d1, gt = syn.synthetic_features(seed, n0, n1)
        m, stop, pr0, pr1, ms = run_ref_lightglue(model, kp0, d0, kp1, d1, (480, 640), (480, 640))
        tr = {}
        m2 = lightglue_ref.lightglue_match(kp0, d0, kp1, d1, sd, trace=tr)
        assert np.array_equal(m, m2) and tr["stop"] == stop == 9, (len(m), len(m2), stop)
        assert (tr["sizes"] == np.array([n0, n1])).all(), "bench weights must not prune"
        np.savez_compressed(OUT / f"lightglue_bench_{seed}.npz", matches=m.astype(np.int32), stop=stop, sizes=tr["sizes"], mscores=ms,
                            seed=seed, n0=n0, n1=n1, profile="bench")
        print(f"lightglue bench seed {seed} ({n0},{n1}): K={len(m)} stop={stop}")
    # the bench's own detect -> match chain: two frames of the bench sequence, wrapper top-k, 'bench' weights
    frames, cal = syn.synthetic_sequence(8, 480, 640)
    sp_sd = syn.superpoint_state_dict(0)
    fa = superpoint_ref.detect_and_describe(frames[0], sp_sd, 5000)
    fb = superpoint_ref.detect_and_describe(frames[5], sp_sd, 5000)
    m, stop, *_ = run_ref_lightglue(model, fa[0], fa[2], fb[0], fb[2], (480, 640), (480, 640))
    m2 = lightglue_ref.lightglue_match(fa[0], fa[2], fb[0], fb[2], sd)
    assert np.array_equal(m, m2) and stop == 9
    good = np.abs((fa[0][m[:, 0]] - fb[0][m[:, 1]]) - [40, 8]).max(1) < 0.5
    np.savez_compressed(OUT / "pipeline_bench_seq_0_5.npz", matches=m.astype(np.int32), stop=stop, kp_a=fa[0].astype(np.int16),
                        kp_b=fb[0].astype(np.int16), sc_a=fa[1], sc_b=fb[1], profile="bench", frames=np.array([0, 5]))
    print(f"pipeline bench seq 0-5: Na={len(fa[0])} Nb={len(fb[0])} K={len(m)} geometrically right {int(good.sum())} stop={stop}")


def golden_superpoint_mp1():
    """(b) SuperPoint on a 1024 x 1024 frame (BASELINE configs[2], SURVEY cfg-B)."""
    sd = syn.superpoint_state_dict(0)
    model = ref_modules.ref_superpoint(sd)
    gray = superpoint_ref.rgb_to_gray_u8(syn.synthetic_frame(2, 1024, 1024))
    kp, sc, desc = run_ref_superpoint(model, gray)
    kp2, sc2, desc2 = superpoint_ref.superpoint_forward(gray.astype(np.float32) / 255.0, sd)
    assert np.array_equal(kp, kp2) and np.array_equal(sc, sc2)
    err = float(np.abs(desc - desc2).max())
    assert err <= 1e-6, err
    sel = np.argpartition(-sc, 5000)[:5000] if len(kp) > 5000 else np.arange(len(kp))
    stride = max(1, len(kp) // 256)
    np.savez_compressed(OUT / "superpoint_mp1.npz", keypoints=kp.astype(np.int16), scores=sc, topk_sel=sel.astype(np.int32),
                        desc_rows=np.arange(0, len(kp), stride, dtype=np.int32), desc=desc[::stride].copy(),
                        desc_checksum=np.float64(desc.astype(np.float64).sum()), restatement_desc_err=np.float64(err),
                        **{f"v_{k}": np.array(v) for k, v in versions().items()})
    print(f"superpoint mp1: {gray.shape} N={len(kp)} restatement desc err {err:.2e}")


def golden_superglue_large():
    """(c) SuperGlue at 2048 and 5000 keypoints (Sinkhorn over 16.8 / 100 MB matrices)."""
    sd = syn.superglue_state_dict(1, "sharp")
    model = ref_modules.ref_superglue(sd, weights="outdoor", sinkhorn_iterations=20, descriptor_dim=256)
    for seed, n0, n1 in [(12, 2048, 1900), (13, 5000, 5000)]:
        kp0, sc0, d0, kp1, sc1, d1, gt = syn.synthetic_features(seed, n0, n1)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))[None]
        data = {"keypoints0": t(kp0), "keypoints1": t(kp1), "descriptors0": t(d0.T), "descriptors1": t(d1.T),
                "scores0": t(sc0), "scores1": t(sc1), "image0": torch.empty(1, 1, 480, 640), "image1": torch.empty(1, 1, 480, 640)}
        with torch.no_grad():
            pred = model(data)
        m0 = pred["matches0"][0].numpy()
        valid = m0 > -1
        rows = np.hstack([np.arange(n0)[valid].reshape(-1, 1), np.arange(n1)[m0[valid]].reshape(-1, 1)]).astype(np.uint32)
        rows2 = superglue_ref.superglue_match(kp0, sc0, d0, kp1, sc1, d1, (480, 640, 3), (480, 640, 3), sd)
        assert np.array_equal(rows, rows2), f"superglue restatement != reference (seed {seed}): {len(rows)} vs {len(rows2)}"
        np.savez_compressed(OUT / f"superglue_{seed}.npz", matches=rows, mscores=pred["matching_scores0"][0].numpy()[valid],
                            seed=seed, n0=n0, n1=n1, profile="sharp")
        print(f"superglue seed {seed} ({n0},{n1}): K={len(rows)}")


def golden_lund_door():
    """(d) BASELINE configs[0]: all 12 lund-door images (loader resize to short side 760) and the 66 exhaustive pairs through
    SuperPoint (max 5000 keypoints, wrapper argpartition) -> LightGlue ('sharp' weights).  Stores the resized gray frames
    (inputs that cannot be regenerated from a seed), every detection, the reference's top-k selection and per-pair matches."""
    sp_sd = syn.superpoint_state_dict(0)
    lg_sd = syn.lightglue_state_dict(2, "sharp")
    sp_model = ref_modules.ref_superpoint(sp_sd)
    lg_model = ref_modules.ref_lightglue(lg_sd)
    img, feats = {}, []
    for i in range(1, 13):
        gray = load_lund_gray(i)
        kp, sc, desc = run_ref_superpoint(sp_model, gray)
        kp2, sc2, desc2 = superpoint_ref.superpoint_forward(gray.astype(np.float32) / 255.0, sp_sd)
        assert np.array_equal(kp, kp2) and np.array_equal(sc, sc2) and np.abs(desc - desc2).max() <= 1e-6
        sel = np.argpartition(-sc, 5000)[:5000] if len(kp) > 5000 else np.arange(len(kp))
        img[f"gray_{i}"] = gray
        img[f"kp_{i}"] = kp.astype(np.int16)
        img[f"sc_{i}"] = sc
        img[f"sel_{i}"] = sel.astype(np.int32)
        img[f"desc_{i}"] = desc[sel][::20].copy()  # every 20th selected descriptor (250 rows)
        feats.append((kp[sel], desc[sel], gray.shape))
        print(f"lund image {i}: {gray.shape} N={len(kp)}")
    np.savez_compressed(OUT / "lund_door_images.npz", **img, **{f"v_{k}": np.array(v) for k, v in versions().items()})
    out = {}
    n_matches = []
    for a in range(12):
        for b in range(a + 1, 12):
            (kpa, da, sha), (kpb, db, shb) = feats[a], feats[b]
            m, stop, *_ = run_ref_lightglue(lg_model, kpa, da, kpb, db, sha, shb)
            if (a + b) % 7 == 0:  # restatement pinned on a subset (the rest is the unmodified reference alone)
                assert np.array_equal(m, lightglue_ref.lightglue_match(kpa, da, kpb, db, lg_sd))
            out[f"m_{a + 1}_{b + 1}"] = m.astype(np.int16)
            out[f"stop_{a + 1}_{b + 1}"] = np.int32(stop)
            n_matches.append(len(m))
            print(f"lund pair {a + 1}-{b + 1}: K={len(m)} stop={stop}", flush=True)
    np.savez_compressed(OUT / "lund_door_66pairs.npz", **out, profile="sharp")
    print(f"lund door: 66 pairs, matches per pair min/median/max {min(n_matches)}/{int(np.median(n_matches))}/{max(n_matches)}")


def retriever_descriptors(n=130, dim=512, seed=7):
    """A walk through descriptor space: neighbours in the sequence are similar (like NetVLAD over a video), unit norm."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal(dim)
    out = []
    for _ in range(n):
        base = base + 0.35 * rng.standard_normal(dim)
        v = base + 0.1 * rng.standard_normal(dim)
        out.append((v / np.linalg.norm(v)).astype(np.float32))
    return np.stack(out)


def golden_retriever():
    """The reference's SimilarityRetriever (gtsfm/retriever/similarity_retriever.py) on seeded descriptors; matplotlib, dask
    and gtsam are not installed, and gtsfm.evaluation.metrics (type names in retriever_base.py only) pulls in h5py / open3d,
    so those are replaced by empty stand-ins: the retriever module and its base are the reference's own code."""
    import types

    class _Stub(types.ModuleType):
        def __getattr__(self, n):
            if n.startswith("__"):
                raise AttributeError(n)
            return type(n, (), {"__init__": lambda self, *a, **k: None})

    for name in ("gtsam", "gtsam.noiseModel", "dask", "dask.distributed", "distributed", "matplotlib", "matplotlib.pyplot", "gtsfm.evaluation.metrics"):
        sys.modules.setdefault(name, _Stub(name))
    sys.path.insert(0, "/root/reference")
    from gtsfm.retriever.similarity_retriever import SimilarityRetriever

    g = retriever_descriptors()
    out = {"descriptors": g}
    cases = [(5, 0.1), (200, 0.3), (2, -1.0), (10, 0.55)]
    for c, (k, ms) in enumerate(cases):
        r = SimilarityRetriever(num_matched=k, min_score=ms)
        pairs = r.get_image_pairs([d for d in g], [f"{i}.jpg" for i in range(len(g))])
        out[f"pairs_{c}"] = np.asarray(pairs, np.int32).reshape(-1, 2)
        out[f"case_{c}"] = np.asarray([k, ms], np.float64)
        if c == 0:
            out["sim"] = r._latest_similarity_matrix.numpy()
        print("retriever case", c, k, ms, len(pairs))
    out["versions"] = versions()
    np.savez_compressed(OUT / "retriever.npz", **out)


def netvlad_images(shapes=((96, 128), (120, 168), (96, 128))):
    """Seeded RGB frames as the (3, H, W) float32 [0, 1] tensors the reference's batch transform produces."""
    return [np.ascontiguousarray(syn.synthetic_frame(40 + i, h, w).transpose(2, 0, 1)).astype(np.float32) / np.float32(255.0)
            for i, (h, w) in enumerate(shapes)]


def golden_netvlad():
    """thirdparty/hloc/netvlad.py's NetVLAD.forward (unmodified) on seeded weights.  The constructor downloads and parses a
    MATLAB checkpoint (netvlad.py:94-160), impossible offline, so the module is assembled exactly as :104-113 does - vgg16
    features[:-2], NetVLADLayer(), Linear(32768, 4096) - and given `synthetic.netvlad_state_dict` instead."""
    import torch.nn as nn
    import torchvision.models as models

    import types

    class _Stub(types.ModuleType):  # dask is only imported by gtsfm.utils.logger; not installed offline
        def __getattr__(self, n):
            if n.startswith("__"):
                raise AttributeError(n)
            return type(n, (), {"__init__": lambda self, *a, **k: None})

    for name in ("dask", "dask.distributed", "distributed"):
        sys.modules.setdefault(name, _Stub(name))
    sys.path.insert(0, "/root/reference")
    from thirdparty.hloc.netvlad import NetVLAD, NetVLADLayer

    sd = syn.netvlad_state_dict(3)
    m = NetVLAD.__new__(NetVLAD)
    nn.Module.__init__(m)
    backbone = list(models.vgg16().children())[0]
    m.backbone = nn.Sequential(*list(backbone.children())[:-2])
    m.netvlad = NetVLADLayer()
    m.whiten = nn.Linear(m.netvlad.output_dim, 4096)
    missing = m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items() if k != "mean"}, strict=True)
    m.preprocess = {"mean": sd["mean"], "std": np.array([1, 1, 1], dtype=np.float32)}
    m.eval()
    out = {"versions": versions()}
    imgs = netvlad_images()
    with torch.no_grad():
        for i, im in enumerate(imgs):
            d = m({"image": torch.from_numpy(im)[None]})["global_descriptor"].numpy()[0]
            out[f"desc_{i}"] = d
            out[f"shape_{i}"] = np.asarray(im.shape[1:], np.int32)
            print("netvlad", i, im.shape, float(np.linalg.norm(d)), d[:4])
        both = m({"image": torch.from_numpy(np.stack([imgs[0], imgs[2]]))})["global_descriptor"].numpy()
    out["desc_batch_0_2"] = both
    print("missing keys:", missing, "cos(0,2) =", float(out["desc_0"] @ out["desc_2"]), "cos(0,1) =", float(out["desc_0"] @ out["desc_1"]))
    np.savez_compressed(OUT / "netvlad.npz", **out)


GTSFM_BASES_SCRIPT = """
import inspect, json, sys, types
sys.path.insert(0, sys.argv[1])
class _Stub(types.ModuleType):  # gtsam / dask / hydra are not installable offline; nothing recorded here comes from them
    def __getattr__(self, n):
        if n.startswith("__"): raise AttributeError(n)
        return type(n, (), {"__init__": lambda self, *a, **k: None})
for name in ("gtsam", "gtsam.noiseModel", "dask", "dask.distributed", "distributed", "hydra", "hydra.utils", "omegaconf"):
    sys.modules[name] = _Stub(name)
sys.modules["gtsam"].noiseModel = sys.modules["gtsam.noiseModel"]
from gtsfm.common.image import Image
from gtsfm.common.keypoints import Keypoints
from gtsfm.frontend.detector_descriptor.detector_descriptor_base import DetectorDescriptorBase
from gtsfm.frontend.matcher.matcher_base import MatcherBase
from gtsfm.frontend.verifier.verifier_base import VerifierBase
from gtsfm.ui.gtsfm_process import GTSFMProcess

def params(f):
    return [[p.name, None if p.default is p.empty else repr(p.default)] for p in inspect.signature(f).parameters.values()]

def methods(cls):
    return {n: params(f) for n, f in vars(cls).items() if inspect.isfunction(f) and (not n.startswith("_") or n == "__init__")}

def base_state(cls, *args):  # the attributes the base's own __init__ sets for these constructor arguments
    stub = type("Probe", (cls,), {n: (lambda *a, **k: None) for n in cls.__abstractmethods__})
    return {k: repr(v) for k, v in vars(stub(*args)).items()}

bases, plugins = {}, {}
for cls in (DetectorDescriptorBase, MatcherBase, VerifierBase):
    bases[cls.__name__] = dict(module=cls.__module__, init=params(cls.__init__) if "__init__" in vars(cls) else None,
                               abstract={n: params(getattr(cls, n)) for n in sorted(cls.__abstractmethods__)})
plugins["B200SuperPointDetectorDescriptor"] = dict(base="DetectorDescriptorBase", state=base_state(DetectorDescriptorBase, 5000))
plugins["B200LightGlueMatcher"] = dict(base="MatcherBase", state=base_state(MatcherBase))
plugins["B200SuperGlueMatcher"] = dict(base="MatcherBase", state=base_state(MatcherBase))
probe = type("B200Ransac", (VerifierBase,), {n: (lambda *a, **k: None) for n in VerifierBase.__abstractmethods__})
plugins["B200Ransac"] = dict(base="VerifierBase", state=base_state(VerifierBase, True, 4), repr=repr(probe(True, 4)))
out = dict(bases=bases, plugins=plugins,
           process=dict(module=GTSFMProcess.__module__, name=GTSFMProcess.__name__, abstract=sorted(GTSFMProcess.__abstractmethods__)),
           keypoints=dict(module=Keypoints.__module__, methods=methods(Keypoints)),
           image=dict(module=Image.__module__, methods=methods(Image)))
print(json.dumps(out, indent=1, sort_keys=True))
"""


def golden_gtsfm_bases():
    """The reference's plugin API (the abstract bases GTSfM's front end instantiates through Hydra, Keypoints, Image): module
    paths, abstract methods and their parameters, what each base's __init__ stores, and the verifier repr that keys GTSfM's
    two-view cache.  Read in a subprocess, with empty stand-ins for gtsam / dask / hydra, so they never reach this process."""
    import subprocess

    r = subprocess.run([sys.executable, "-c", GTSFM_BASES_SCRIPT, str(ref_modules.REF)], capture_output=True, text=True,
                       check=True)
    (OUT / "gtsfm_bases.json").write_text(r.stdout)


def main():
    assert ref_modules.available(), "/root/reference is required"
    OUT.mkdir(parents=True, exist_ok=True)
    torch.set_num_threads(8)
    if len(sys.argv) > 1:  # e.g. `python -m oracle.make_golden lightglue_bench superpoint_mp1 superglue_large lund_door`
        for name in sys.argv[1:]:
            globals()[f"golden_{name}"]()
        return
    feats = golden_superpoint()
    golden_lightglue(feats)
    golden_superglue()
    golden_verifier()
    golden_verifier_argoverse()
    golden_lightglue_bench()
    golden_superpoint_mp1()
    golden_superglue_large()
    golden_lund_door()
    golden_retriever()
    golden_netvlad()
    golden_gtsfm_bases()


if __name__ == "__main__":
    main()
