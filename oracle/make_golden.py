"""Generate tests/golden/*.pt from the UNMODIFIED reference (run in the build container only).

    python oracle/make_golden.py --reference <checkout of microsoft/MoGe>      # writes tests/golden/

For every case the script (1) builds the reference `moge.model.v2.MoGeModel(**cfg)`, loads the seeded
synthetic state dict from moge_b200.synthetic with strict=True (pins key names and shapes), (2) runs the
reference `forward()` / `infer()` in fp32 on CPU, (3) asserts that oracle/moge_port.py reproduces it,
and (4) stores the reference outputs (not the port's) as the golden fixture.  Inputs are regenerated
from the seed by the tests (moge_b200.synthetic.synthetic_images), so only outputs are stored.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "utils3d_shim"))

import torch  # noqa: E402

from moge_b200.configs import model_config  # noqa: E402
from moge_b200.synthetic import make_state_dict, synthetic_images, synthetic_point_map  # noqa: E402
from oracle import moge_port  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

FORWARD_CASES = [
    # name, size, with_normal, seed, (B,H,W), num_tokens, store_stride
    ("vits_b1_126x168_t192", "vits", True, 0, (1, 126, 168), 192, 1),
    ("vits_b2_140x98_t117", "vits", True, 1, (2, 140, 98), 117, 1),
    ("vits_b1_70x70_t1369_native", "vits", True, 2, (1, 70, 70), 1369, 1),
    ("vits_b1_224x224_default", "vits", True, 3, (1, 224, 224), None, 2),      # BASELINE.json configs[0]
    ("vitb_b1_98x154_t150_nonormal", "vitb", False, 4, (1, 98, 154), 150, 1),
    ("vitl_b1_112x140_t120", "vitl", True, 5, (1, 112, 140), 120, 1),
]

# Round-2 cases: (name, size, with_normal, seed, (B,H,W), num_tokens, stride, options)
#   options: well_posed (synthetic.make_state_dict(well_posed=True): the focal/shift solve is well-conditioned, so the five
#   infer() outputs are comparable end to end), remap (overrides cfg['remap_output']), autocast (store the reference's own
#   16-bit deviation as the yardstick; costs two more reference passes)
CASES_R2 = [
    # the benchmarked shape (BASELINE.json configs[1]/[3]): ViT-L, 518x518, 37x37 native grid
    ("vitl_b1_518x518_t1369_wp", "vitl", True, 10, (1, 518, 518), 1369, 4, {"well_posed": True, "autocast": True}),
    # 35x35 grid -> 490 px: the antialiased DOWN-sampling branch of the input resize (modules.py:121)
    ("vitl_b1_518x518_t1200_wp", "vitl", True, 11, (1, 518, 518), 1200, 4, {"well_posed": True}),
    # API default: 3600 tokens, 60x60 grid, 840 px
    ("vitl_b1_518x518_default_wp", "vitl", True, 12, (1, 518, 518), None, 4, {"well_posed": True}),
    # mixed-aspect shapes of BASELINE.json configs[2] (grids 19x37 and 37x19)
    ("vitl_b1_518x1036_t700_wp", "vitl", True, 13, (1, 518, 1036), 700, 6, {"well_posed": True}),
    ("vitl_b1_1036x518_t700_wp", "vitl", True, 14, (1, 1036, 518), 700, 6, {"well_posed": True}),
    # large input, down-sampled by more than 2x on both axes (wide antialias filter), ViT-B (configs[4] family)
    ("vitb_b1_1024x768_t1200_wp", "vitb", True, 15, (1, 1024, 768), 1200, 8, {"well_posed": True}),
    # well-posed small cases (fast) incl. batch 2
    ("vits_b2_126x168_t192_wp", "vits", True, 16, (2, 126, 168), 192, 2, {"well_posed": True, "autocast": True}),
    # remap_output variants (v2.py:122-136)
    ("vits_b1_98x126_t120_linear", "vits", True, 17, (1, 98, 126), 120, 1, {"remap": "linear"}),
    ("vits_b1_98x126_t120_sinh", "vits", True, 18, (1, 98, 126), 120, 1, {"remap": "sinh"}),
    ("vits_b1_98x126_t120_sinh_exp", "vits", True, 19, (1, 98, 126), 120, 1, {"remap": "sinh_exp"}),
]

# Stride of the stored infer() outputs where it differs from the forward() stride.  The tests feed the whole forward() maps
# of these cases to the focal/shift solve and post-processing (the engine's kernels and the oracle port's), so those stay at
# stride 1; the infer() maps are sampled so that every golden file stays below 1 MB.
INFER_STRIDE = {"vits_b1_126x168_t192": 2, "vits_b2_140x98_t117": 3}


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the unmodified reference (microsoft/MoGe)")
    ap.add_argument("--only", default=None, help="comma-separated substrings: generate only the cases whose name contains one")
    ap.add_argument("--skip-focal", action="store_true")
    a = ap.parse_args()
    only = a.only.split(",") if a.only else None
    sys.path.insert(1, os.path.abspath(a.reference))
    from moge.model.v2 import MoGeModel as RefModel                                   # the real reference
    from moge.utils.geometry_torch import recover_focal_shift as ref_recover
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    for case in [c + ({},) for c in FORWARD_CASES] + CASES_R2:
        name, size, with_normal, seed, (B, H, W), tokens, stride, opt = case
        if only and not any(o in name for o in only):
            continue
        cfg = model_config(size, with_normal)
        if "remap" in opt:
            cfg["remap_output"] = opt["remap"]
        sd = make_state_dict(cfg, seed, well_posed=opt.get("well_posed", False))
        ref = RefModel(**cfg).eval()
        missing = ref.load_state_dict(sd, strict=True)
        assert not missing.missing_keys and not missing.unexpected_keys
        img = synthetic_images(B, H, W, seed)
        nt = tokens if tokens is not None else int(1200 + (9 / 9) * (3600 - 1200))
        with torch.no_grad():
            fwd = ref.forward(img, nt)
            inf = ref.infer(img, num_tokens=tokens, use_fp16=False)
            # the reference's OWN 16-bit deviation on these weights (CPU autocast), the yardstick for the engine's tolerance
            dev16 = {}
            for tag, dt_ in ((("fp16", torch.float16), ("bf16", torch.bfloat16)) if opt.get("autocast", name in [c[0] for c in FORWARD_CASES]) else ()):
                with torch.autocast("cpu", dtype=dt_):
                    f16 = ref.forward(img, nt)
                dev16[tag] = {k: rel_l2(f16[k].float(), fwd[k]) for k in fwd}
        pf = moge_port.forward(cfg, sd, img, nt)
        pi = moge_port.infer(cfg, sd, img, num_tokens=tokens)
        report = {}
        for k in fwd:
            report["fwd." + k] = rel_l2(pf[k], fwd[k])
            assert report["fwd." + k] < 2e-5, (name, k, report)
        m = inf["mask"]
        assert bool((pi["mask"] == m).float().mean() > 0.9999), name
        both = m & pi["mask"]
        for k in ("points", "depth", "normal"):
            if k in inf:
                report["inf." + k] = rel_l2(pi[k][both], inf[k][both])
                assert report["inf." + k] < 1e-4, (name, k, report)
        report["inf.intrinsics"] = rel_l2(pi["intrinsics"], inf["intrinsics"])
        assert report["inf.intrinsics"] < 1e-4, (name, report)
        print(name, {k: f"{v:.2e}" for k, v in report.items()}, "mask_frac", float(m.float().mean()))
        print("   reference autocast deviation:", {t: {k: f"{v:.1e}" for k, v in d.items()} for t, d in dev16.items()})
        sl = (slice(None), slice(None, None, stride), slice(None, None, stride))
        istride = INFER_STRIDE.get(name, stride)
        isl = (slice(None), slice(None, None, istride), slice(None, None, istride))
        gold = {
            "meta": {"size": size, "with_normal": with_normal, "seed": seed, "shape": (B, H, W), "num_tokens": tokens,
                     "stride": stride, "infer_stride": istride, "port_vs_reference": report, "options": dict(opt),
                     "reference_autocast_deviation": dev16},
            "forward": {k: (v[sl].contiguous() if v.dim() >= 3 else v) for k, v in fwd.items()},
            "infer": {k: (v[isl].contiguous() if v.dim() >= 3 and k != "intrinsics" else v) for k, v in inf.items()},
        }
        torch.save(gold, os.path.join(OUT, name + ".pt"))

    if a.skip_focal or only:
        return
    # focal / shift recovery on synthetic well-posed point maps (SURVEY.md 8c cut point 2)
    cases = []
    for i, (H, W, f_true, s_true, noise, mask_mode, given_focal) in enumerate([
        (96, 128, 1.1, 0.35, 0.0, "all", False),
        (120, 90, 0.7, -0.2, 0.01, "random", False),
        (64, 64, 1.6, 0.8, 0.02, "half", False),
        (150, 200, 0.9, 0.1, 0.005, "random", True),
        (77, 113, 1.3, 0.5, 0.01, "none", False),        # mask all-false -> (1, 0) fallback
        (518, 518, 1.0, 0.25, 0.01, "random", False),
        (80, 100, 2.5, 1.5, 0.0, "single", False),       # 1 valid sample -> fallback
    ]):
        pts, mask = synthetic_point_map(2, H, W, f_true, s_true, noise, mask_mode, seed=100 + i)
        focal_in = torch.full((2,), f_true) * torch.tensor([1.0, 1.05]) if given_focal else None
        f, s = ref_recover(pts, mask, focal=focal_in)
        pf_, ps_ = moge_port.recover_focal_shift(pts, mask, focal=focal_in)
        assert torch.allclose(pf_, f, rtol=1e-6, atol=1e-7) and torch.allclose(ps_, s, rtol=1e-6, atol=1e-7), (i, f, pf_, s, ps_)
        cases.append({"args": (2, H, W, f_true, s_true, noise, mask_mode, 100 + i), "focal_in": focal_in,
                      "focal": f, "shift": s})
        print("focal case", i, f.tolist(), s.tolist())
    torch.save(cases, os.path.join(OUT, "recover_focal_shift.pt"))


if __name__ == "__main__":
    main()
