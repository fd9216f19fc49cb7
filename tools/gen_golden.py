"""Generate tests/golden/*.npz by running the UNMODIFIED reference (CPU, via
tools/refshim.py) on seeded synthetic inputs.  Build-container only.

    python tools/gen_golden.py

Golden files hold outputs only (inputs are regenerated from the seed by
visiondepth3d_b200.synth), plus versions of the third-party libs used.
"""
import os
import sys
import threading

import numpy as np

sys.path.insert(0, os.path.dirname(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import refshim  # noqa: E402
from tests.util import save_golden  # noqa: E402
from visiondepth3d_b200.synth import synth_frame  # noqa: E402

OUT = os.path.join(os.path.dirname(__file__), "..", "tests", "golden")


class Var:
    def __init__(self, v):
        self.v = v

    def get(self):
        return self.v


def run_pixel_shift(r3d, torch, w, h, iw, ih, n_frames, kind, **kw):
    """pixel_shift_cuda on n_frames consecutive frames (floating-window state carries)."""
    refshim.reset_singletons(r3d)
    out = {}
    for i in range(n_frames):
        fr, dp = synth_frame(i, iw, ih, kind)
        ft = r3d.frame_to_tensor(fr)
        dt = r3d.depth_to_tensor(dp)
        l, r, s = r3d.pixel_shift_cuda(ft, dt, w, h, 4.5, -1.5, -6.0, return_shift_map=True, **kw)
        out[f"left{i}"] = l
        out[f"right{i}"] = r
        out[f"shift{i}"] = s.numpy().astype(np.float16 if False else np.float32)
    return out


def run_loop(r3d, torch, cv2, src_w, src_h, n_frames, kind, rp):
    """Drive the body of render_sbs_3d in memory by writing lossless-ish input is not
    possible (codecs are lossy) -> we run the real render_sbs_3d with cv2 capture
    monkey-patched to an in-memory frame source and the writer to a collector."""
    refshim.reset_singletons(r3d)
    frames = [synth_frame(i, src_w, src_h, kind) for i in range(n_frames)]

    class Cap:
        def __init__(self, which):
            self.which = which
            self.pos = 0

        def isOpened(self):
            return True

        def get(self, prop):
            if prop == cv2.CAP_PROP_FRAME_COUNT:
                return float(n_frames)
            if prop == cv2.CAP_PROP_FPS:
                return 24.0
            if prop == cv2.CAP_PROP_POS_FRAMES:
                return float(self.pos)
            return 0.0

        def set(self, prop, v):
            if prop == cv2.CAP_PROP_POS_FRAMES:
                self.pos = int(v)
            return True

        def read(self):
            if self.pos >= n_frames:
                return False, None
            f = frames[self.pos][self.which].copy()
            self.pos += 1
            return True, f

        def release(self):
            pass

    collected = []

    class Writer:
        def __init__(self, *a, **k):
            pass

        def isOpened(self):
            return True

        def write(self, f):
            collected.append(f.copy())

        def release(self):
            pass

    real_cap, real_wr = cv2.VideoCapture, cv2.VideoWriter
    cv2.VideoCapture = lambda path: Cap(0 if path == "rgb" else 1)
    cv2.VideoWriter = Writer
    try:
        r3d.render_sbs_3d(
            "rgb", "depth", "out.avi", "XVID", 24.0, rp["output_width"], rp["output_height"],
            4.5, -1.5, -6.0, rp["sharpness_factor"], rp["output_format"], Var(rp.get("aspect_name", "Default (16:9)")),
            r3d.aspect_ratios, rp["dof_strength"],
            feather_strength=rp["feather_strength"], blur_ksize=rp["blur_ksize"],
            use_subject_tracking=rp["use_subject_tracking"],
            use_floating_window=rp["use_floating_window"],
            max_pixel_shift_percent=0.02, suspend_flag=threading.Event(),
            cancel_flag=threading.Event(),
            preserve_original_aspect=rp["preserve_original_aspect"],
            zero_parallax_strength=rp["zero_parallax_strength"],
            color_saturation=rp.get("color_saturation", 1.0),
            color_contrast=rp.get("color_contrast", 1.0),
            color_brightness=rp.get("color_brightness", 0.0),
            **{k: rp[k] for k in ("enable_edge_masking", "enable_feathering",
                                  "convergence_strength", "enable_dynamic_convergence", "ipd_factor",
                                  "parallax_balance", "depth_pop_gamma", "fg_pop_multiplier") if k in rp},
        )
    finally:
        cv2.VideoCapture, cv2.VideoWriter = real_cap, real_wr
    return {f"final{i}": f for i, f in enumerate(collected)}


def main():
    mods = refshim.load_reference(("render_3d",))
    r3d = mods["render_3d"]
    import cv2
    import torch
    import torchvision
    torch.set_num_threads(os.cpu_count())
    os.makedirs(OUT, exist_ok=True)
    meta = dict(torch=torch.__version__, torchvision=torchvision.__version__, cv2=cv2.__version__,
                numpy=np.__version__)

    # A. pixel_shift_cuda, identity resize, GUI-style params, 3 consecutive frames
    g = run_pixel_shift(r3d, torch, 320, 180, 320, 180, 3, "smooth",
                        blur_ksize=9, feather_strength=10.0, zero_parallax_strength=0.01)
    save_golden(os.path.join(OUT, "ps_smooth_320x180.npz"), **g, **meta)
    # B. 2x upsample inside pixel_shift (Half-SBS style), no floating window
    g = run_pixel_shift(r3d, torch, 320, 180, 160, 90, 2, "smooth",
                        blur_ksize=5, feather_strength=4.0, enable_floating_window=False,
                        convergence_strength=0.5)
    np.savez_compressed(os.path.join(OUT, "ps_up2_320x180.npz"), **g, **meta)
    # C. noise content (adversarial LSB), edge masking off, even blur ksize
    g = run_pixel_shift(r3d, torch, 192, 108, 192, 108, 1, "noise",
                        blur_ksize=4, feather_strength=10.0, enable_edge_masking=False,
                        use_subject_tracking=False)
    np.savez_compressed(os.path.join(OUT, "ps_noise_192x108.npz"), **g, **meta)

    # D. full loop, Half-SBS (config-2 shape scaled down 6x: 320x180 source)
    base = dict(output_width=320, output_height=180, sharpness_factor=0.2, output_format="Half-SBS",
                dof_strength=0.0, feather_strength=10.0, blur_ksize=9, use_subject_tracking=True,
                use_floating_window=True, preserve_original_aspect=False, zero_parallax_strength=0.01)
    g = run_loop(r3d, torch, cv2, 320, 180, 6, "smooth", base)
    np.savez_compressed(os.path.join(OUT, "loop_halfsbs_320x180.npz"), **g, **meta)
    # E. full loop, Full-SBS preserve aspect (config-3 shape scaled down), DOF on + colour grade
    rp = dict(base, output_format="Full-SBS", preserve_original_aspect=True, dof_strength=2.0,
              color_saturation=1.1, color_contrast=1.05, color_brightness=0.02)
    g = run_loop(r3d, torch, cv2, 320, 180, 5, "smooth", rp)
    np.savez_compressed(os.path.join(OUT, "loop_fullsbs_dof_320x180.npz"), **g, **meta)
    # F. anaglyph + interlaced formats, render defaults (no tracking)
    rp = dict(base, output_format="Red-Cyan Anaglyph", preserve_original_aspect=True,
              use_subject_tracking=False, use_floating_window=False, feather_strength=0.0, blur_ksize=1)
    g = run_loop(r3d, torch, cv2, 256, 144, 3, "smooth", rp)
    np.savez_compressed(os.path.join(OUT, "loop_anaglyph_256x144.npz"), **g, **meta)
    rp = dict(rp, output_format="Passive Interlaced")
    g = run_loop(r3d, torch, cv2, 256, 144, 3, "smooth", rp)
    np.savez_compressed(os.path.join(OUT, "loop_interlaced_256x144.npz"), **g, **meta)
    # G. heal_missing_pixels (dead code in the reference's loop, named by north_star): standalone op
    rng = np.random.default_rng(21)
    H, W = 90, 160
    yy, xx = np.mgrid[0:H, 0:W]
    warped = np.stack([(xx / W), (yy / H), ((xx + yy) % 32) / 32.0]).astype(np.float32)
    warped[:, 30:60, 50:90] = rng.random((3, 30, 40), dtype=np.float32)
    orig = np.clip(warped + 0.1 * rng.standard_normal(warped.shape).astype(np.float32), 0, 1).astype(np.float32)
    edge = (rng.random((1, H, W), dtype=np.float32) > 0.9).astype(np.float32)
    outs = {}
    for name, em in (("none", None), ("edge", edge)):
        outs["heal_" + name] = r3d.heal_missing_pixels(
            torch.from_numpy(warped), None, torch.from_numpy(orig),
            torch.from_numpy(em) if em is not None else None, 0.5).numpy()
    np.savez_compressed(os.path.join(OUT, "heal_160x90.npz"), warped=warped, orig=orig, edge=edge, **outs)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def gen_vr():
    """H. VR format: 1600x900 eyes -> pad_to_aspect_ratio(1440, 1600) = non-integer INTER_AREA (x1.111) + black
    bars, hstack to 2880x1600.  Separate entry (`python tools/gen_golden.py vr`) so the earlier fixtures stay
    byte-identical.  Stored per frame: every 3rd row / column of the image band (the rest of the 2880x1600 frame is
    black), the band position, and a sha256 of the whole frame."""
    import hashlib
    mods = refshim.load_reference(("render_3d",))
    r3d = mods["render_3d"]
    import cv2
    import torch
    import torchvision
    torch.set_num_threads(os.cpu_count())
    meta = dict(torch=torch.__version__, torchvision=torchvision.__version__, cv2=cv2.__version__,
                numpy=np.__version__)
    rp = dict(output_width=1600, output_height=900, sharpness_factor=0.2, output_format="VR",
              dof_strength=0.0, feather_strength=10.0, blur_ksize=9, use_subject_tracking=True,
              use_floating_window=True, preserve_original_aspect=False, zero_parallax_strength=0.01)
    g = run_loop(r3d, torch, cv2, 320, 180, 3, "smooth", rp)
    out = {}
    for k, f in g.items():
        assert f.shape == (1600, 2880, 3), f.shape
        rows = np.nonzero(f.reshape(1600, -1).any(axis=1))[0]
        y0, y1 = int(rows.min()), int(rows.max()) + 1
        out[k + "_band"] = f[y0:y1:3, ::3]
        out[k + "_y0"] = np.int32(y0)
        out[k + "_y1"] = np.int32(y1)
        out[k + "_sha256"] = np.frombuffer(hashlib.sha256(f.tobytes()).digest(), dtype=np.uint8)
    p = os.path.join(OUT, "loop_vr_320x180.npz")
    np.savez_compressed(p, **out, **meta)
    print(p, os.path.getsize(p), {k: v.shape for k, v in out.items() if k.endswith("_band")})


def gen_extra():
    """I-K. loop cases that pin the crop / aspect / fractional-fit branches of render_sbs_3d
    (`python tools/gen_golden.py extra`; the earlier fixtures stay byte-identical)."""
    mods = refshim.load_reference(("render_3d",))
    r3d = mods["render_3d"]
    import cv2
    import torch
    import torchvision
    torch.set_num_threads(os.cpu_count())
    meta = dict(torch=torch.__version__, torchvision=torchvision.__version__, cv2=cv2.__version__,
                numpy=np.__version__)
    base = dict(output_width=320, output_height=180, sharpness_factor=0.2, output_format="Half-SBS",
                dof_strength=0.0, feather_strength=10.0, blur_ksize=9, use_subject_tracking=True,
                use_floating_window=True, preserve_original_aspect=False, zero_parallax_strength=0.01)
    # I. 4:3 source against the 16:9 target: centre crop of the height (1244-1248)
    g = run_loop(r3d, torch, cv2, 320, 240, 3, "smooth", base)
    np.savez_compressed(os.path.join(OUT, "loop_crop43_320x240.npz"), **g, **meta)
    # J. CinemaScope 2.39:1 target on a 16:9 source: crop + 430x180 warp + 215x180 eyes
    g = run_loop(r3d, torch, cv2, 320, 180, 3, "smooth", dict(base, aspect_name="CinemaScope (2.39:1)"))
    np.savez_compressed(os.path.join(OUT, "loop_scope239_320x180.npz"), **g, **meta)
    # K. preserve_original_aspect with an odd width: 321 -> 160 per eye = fractional INTER_AREA (x2.00625)
    g = run_loop(r3d, torch, cv2, 321, 180, 3, "smooth", dict(base, preserve_original_aspect=True))
    np.savez_compressed(os.path.join(OUT, "loop_halfsbs_odd_321x180.npz"), **g, **meta)
    # L. the remaining loop-level controls: IPD factor, fixed convergence, edge masking off, sharpness factor 0 (still a
    #    5/-1 kernel), and the parallax/pop controls the loop accepts but does not forward to pixel_shift_cuda
    g = run_loop(r3d, torch, cv2, 320, 180, 4, "smooth",
                 dict(base, sharpness_factor=0.0, ipd_factor=0.8, convergence_strength=0.3,
                      enable_dynamic_convergence=False, enable_edge_masking=False, parallax_balance=0.6,
                      depth_pop_gamma=0.7, fg_pop_multiplier=1.4))
    np.savez_compressed(os.path.join(OUT, "loop_controls_320x180.npz"), **g, **meta)
    # M. DOF on the Half-SBS path: the normalised depth (160x90) is upsampled to the eye size for apply_dof_cuda
    g = run_loop(r3d, torch, cv2, 320, 180, 3, "smooth", dict(base, dof_strength=1.5))
    np.savez_compressed(os.path.join(OUT, "loop_dof_halfsbs_320x180.npz"), **g, **meta)
    # N. pixel_shift_cuda with every shaping / balance control off its default (the preview path passes them)
    g = run_pixel_shift(r3d, torch, 256, 144, 256, 144, 2, "smooth",
                        blur_ksize=5, feather_strength=20.0, convergence_strength=0.3, enable_dynamic_convergence=False,
                        depth_pop_gamma=0.7, depth_pop_mid=0.4, depth_stretch_lo=0.1, depth_stretch_hi=0.9,
                        fg_pop_multiplier=1.5, bg_push_multiplier=0.9, subject_lock_strength=0.5,
                        parallax_balance=0.6, max_pixel_shift_percent=0.03, zero_parallax_strength=0.02)
    np.savez_compressed(os.path.join(OUT, "ps_controls_256x144.npz"), **g, **meta)
    print("ps_controls_256x144.npz", os.path.getsize(os.path.join(OUT, "ps_controls_256x144.npz")))
    for f in ("loop_crop43_320x240.npz", "loop_scope239_320x180.npz", "loop_halfsbs_odd_321x180.npz",
              "loop_controls_320x180.npz", "loop_dof_halfsbs_320x180.npz"):
        z = np.load(os.path.join(OUT, f))
        print(f, os.path.getsize(os.path.join(OUT, f)), {k: z[k].shape for k in z.files if k.startswith("final")})


def _sparse(f, step):
    import hashlib
    return f[::step, ::step].copy(), np.frombuffer(hashlib.sha256(f.tobytes()).digest(), dtype=np.uint8)


def gen_natural():
    """Q. the "natural" synthetic set (visiondepth3d_b200/synth.py: band-limited fields + texture, values off the
    k/255 truncation grid) through pixel_shift_cuda and the full loop with sharpening on, plus the two BASELINE sizes
    (1080p Half-SBS, 4K Full-SBS) stored as every 7th / 16th row and column + sha256 of the full frame
    (`python tools/gen_golden.py natural`)."""
    mods = refshim.load_reference(("render_3d",))
    r3d = mods["render_3d"]
    import cv2
    import torch
    import torchvision
    torch.set_num_threads(os.cpu_count())
    meta = dict(torch=torch.__version__, torchvision=torchvision.__version__, cv2=cv2.__version__,
                numpy=np.__version__)
    base = dict(output_width=320, output_height=180, sharpness_factor=0.2, output_format="Half-SBS",
                dof_strength=0.0, feather_strength=10.0, blur_ksize=9, use_subject_tracking=True,
                use_floating_window=True, preserve_original_aspect=False, zero_parallax_strength=0.01)
    g = run_pixel_shift(r3d, torch, 320, 180, 320, 180, 3, "natural",
                        blur_ksize=9, feather_strength=10.0, zero_parallax_strength=0.01)
    save_golden(os.path.join(OUT, "ps_natural_320x180.npz"), **g, **meta)
    g = run_loop(r3d, torch, cv2, 320, 180, 5, "natural", base)
    np.savez_compressed(os.path.join(OUT, "loop_natural_halfsbs_320x180.npz"), **g, **meta)
    g = run_loop(r3d, torch, cv2, 320, 180, 4, "natural", dict(base, output_format="Full-SBS", preserve_original_aspect=True))
    np.savez_compressed(os.path.join(OUT, "loop_natural_fullsbs_320x180.npz"), **g, **meta)
    # BASELINE sizes
    g = run_loop(r3d, torch, cv2, 1920, 1080, 3, "natural", dict(base, output_width=1920, output_height=1080))
    out = {}
    for k, f in g.items():
        assert f.shape == (1080, 1920, 3), f.shape
        out[k + "_s7"], out[k + "_sha256"] = _sparse(f, 7)
    np.savez_compressed(os.path.join(OUT, "loop_natural_1080p_halfsbs.npz"), **out, **meta)
    g = run_loop(r3d, torch, cv2, 3840, 2160, 2, "natural",
                 dict(base, output_width=3840, output_height=2160, output_format="Full-SBS", preserve_original_aspect=True))
    out = {}
    for k, f in g.items():
        assert f.shape == (2160, 7680, 3), f.shape
        out[k + "_s16"], out[k + "_sha256"] = _sparse(f, 16)
    np.savez_compressed(os.path.join(OUT, "loop_natural_4k_fullsbs.npz"), **out, **meta)
    for f in ("ps_natural_320x180.npz", "loop_natural_halfsbs_320x180.npz", "loop_natural_fullsbs_320x180.npz",
              "loop_natural_1080p_halfsbs.npz", "loop_natural_4k_fullsbs.npz"):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def gen_depth_gray():
    """O. convert_depth_to_grayscale (core/render_depth.py:585-611) on the input kinds it accepts
    (`python tools/gen_golden.py depthgray`): tensor / ndarray, 2-D, [C,H,W], [H,W,C], flat and NaN frames."""
    # core/render_depth.py drags in diffusers / DepthCrafter at import; run just this (unmodified) function by
    # compiling its definition out of the reference file at generation time -- nothing is copied into the repo
    import ast
    import types
    import torch
    from PIL import Image
    path = os.path.join(refshim.REF_ROOT, "core", "render_depth.py")
    tree = ast.parse(open(path).read(), filename=path)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "convert_depth_to_grayscale"]
    ns = {"np": np, "torch": torch, "Image": Image}
    exec(compile(ast.Module(body=fn, type_ignores=[]), path, "exec"), ns)
    rd = types.SimpleNamespace(convert_depth_to_grayscale=ns["convert_depth_to_grayscale"])
    rng = np.random.default_rng(77)
    base = (rng.standard_normal((24, 32)) * 3.0 + 5.0).astype(np.float32)
    inputs = {
        "hw": base,
        "chw1": base[None],
        "chw3": np.stack([base, base * 0.5, base + 1.0]).astype(np.float32),
        "hwc1": base[..., None],
        "hwc3": np.stack([base, base * 0.5, base + 1.0], axis=-1).astype(np.float32),
        "flat": np.full((24, 32), 2.5, dtype=np.float32),
        "nan": np.where(rng.random((24, 32)) < 0.05, np.nan, base).astype(np.float32),
        "f64": base.astype(np.float64) * 1e-3,
        "neg": -base,
    }
    out = {}
    for k, v in inputs.items():
        out["in_" + k] = v
        out["np_" + k] = rd.convert_depth_to_grayscale(v.copy())
        out["pt_" + k] = rd.convert_depth_to_grayscale(torch.from_numpy(v.copy()))
    p = os.path.join(OUT, "depth_gray.npz")
    np.savez_compressed(p, **out)
    print(p, os.path.getsize(p))


def gen_signatures():
    """P. the call surface of the boundary (SURVEY 8(b)): parameter names, order and defaults of the reference's
    hot-path functions (`python tools/gen_golden.py signatures`) -> tests/golden/signatures.json."""
    import inspect
    import json
    mods = refshim.load_reference(("render_3d",))
    r3d = mods["render_3d"]
    names = ["pixel_shift_cuda", "render_sbs_3d", "format_3d_output", "generate_anaglyph_3d", "apply_sharpening",
             "pad_to_aspect_ratio", "frame_to_tensor", "depth_to_tensor", "tensor_to_frame", "heal_missing_pixels"]
    out = {}
    for n in names:
        sig = inspect.signature(getattr(r3d, n))
        out[n] = [[p.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
                  for p in sig.parameters.values()]
    out["aspect_ratios"] = {k: float(v) for k, v in r3d.aspect_ratios.items()}
    p = os.path.join(OUT, "signatures.json")
    json.dump(out, open(p, "w"), indent=1, sort_keys=True)
    print(p, os.path.getsize(p))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "signatures":
        gen_signatures()
    elif len(sys.argv) > 1 and sys.argv[1] == "depthgray":
        gen_depth_gray()
    elif len(sys.argv) > 1 and sys.argv[1] == "extra":
        gen_extra()
    elif len(sys.argv) > 1 and sys.argv[1] == "vr":
        gen_vr()
    elif len(sys.argv) > 1 and sys.argv[1] == "natural":
        gen_natural()
    else:
        main()
