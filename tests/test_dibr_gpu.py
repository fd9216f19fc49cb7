"""GPU: the CUDA path (through the C ABI / the drop-in Python surface) against the oracle
on seeded inputs, against the reference goldens, and through size-independent properties
at BASELINE sizes.

Tolerances (north_star): uint8 eyes <= 1 LSB; float intermediates <= 1e-3.

Every oracle / golden comparison runs in both DIBR arithmetic modes (include/vd3d.h: vd3d_set_exact):
  "fast"  (the default, what bench.py times): persistent stats kernel + fused render kernel, fp32 hardware
          pow/exp, separable box sums.  Gated at eyes <= 1 LSB with <= 0.5 % of bytes off by one, shift map and
          scalars <= 2e-5 (50x inside the north-star 1e-3).
  "exact" one kernel per reference op, correctly rounded transcendentals: follows the oracle's rounding op for
          op, gated at <= 0.2 % one-LSB flips / 1e-5 / 1e-6 (in practice bit-identical).
Full frames after apply_sharpening may amplify an isolated one-LSB flip up to 7.7 LSB (kernel centre 5.2/1.2...):
gated at <= 8 LSB with <= 0.2 % (exact) / 0.5 % (fast) of bytes off by more than one.
"""
import os

import numpy as np
import pytest

from oracle import dibr as O
from tests.util import (BIG_NATURAL, LOOP_CASES, LOOP_CASES_EXTRA, LOOP_NATURAL, PS_CASES, PS_CASES_EXTRA, PS_NATURAL,
                        load_golden, u8_diff)
from visiondepth3d_b200.synth import synth_frame

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    from visiondepth3d_b200 import render_3d
    return render_3d


MODES = ["fast", "exact"]


@pytest.fixture
def mode(request, R):
    m = getattr(request, "param", "fast")
    R._ctx().set_exact(m == "exact")
    yield m
    R._ctx().set_exact(False)


def _tol(mode, kind="noise"):
    """(scalar abs tol, shift abs tol, eye bytes that may differ by one LSB, packed-frame bytes that may differ at all,
    packed-frame bytes that may differ by more than one, max LSB on packed frames).

    Every u8 eye is gated at <= 1 LSB (north_star).  How MANY bytes sit on the other side of a truncation boundary is
    a property of the content: the warped value of locally flat / ramp content lands exactly on k/255, where a 1e-7
    change of any float intermediate flips the LSB (tools/diag_fast2.py: the fp32 pow accounts for 0.14 % of the bytes
    of the natural set, the separable box sum for 0.2 %; the oracle itself is 0.05 % / 2-3 % away from the real
    reference for the same reason, tests/test_oracle_golden.py).  Downstream, the reference's lossy identity colour
    grade can turn a one-LSB flip into two and apply_sharpening (centre 4.33, neighbours -0.83) spreads it over five
    pixels with up to 2 x 7.7 LSB at the centre -- hence the packed-frame budgets."""
    if mode == "exact":
        return (1e-6, 1e-5, 0.002, 0.01, 0.002, 8)
    if kind == "smooth":
        return (2e-5, 2e-5, 0.05, 0.30, 0.10, 16)
    return (2e-5, 2e-5, 0.01, 0.05, 0.012, 16)


def _ps(R, fr, dp, w, h, kw, infos=None):
    ft, dt = O.bgr_to_rgb01(fr), O.depth_bgr_to_01(dp)
    return R.pixel_shift_cuda(ft, dt, w, h, kw.get("fg", 4.5), kw.get("mg", -1.5), kw.get("bg", -6.0),
                              _info=infos, **{k: v for k, v in kw.items() if k not in ("fg", "mg", "bg")})


def _oracle_kw(kw):
    m = dict(kw)
    for a, b in (("fg", "fg_shift"), ("mg", "mg_shift"), ("bg", "bg_shift")):
        if a in m:
            m[b] = m.pop(a)
    return m


SIZES = [(320, 180, 320, 180), (157, 93, 157, 93), (320, 180, 160, 90), (256, 144, 100, 60), (64, 40, 64, 40)]
PARAMS = [
    dict(blur_ksize=9, feather_strength=10.0, zero_parallax_strength=0.01),
    dict(blur_ksize=4, feather_strength=3.0, enable_floating_window=False, convergence_strength=0.5),
    dict(blur_ksize=1, feather_strength=0.0),
    dict(enable_feathering=False, enable_edge_masking=False, use_subject_tracking=False),
    dict(blur_ksize=5, feather_strength=20.0, convergence_strength=0.3, enable_dynamic_convergence=False,
         depth_pop_gamma=0.7, depth_pop_mid=0.4, depth_stretch_lo=0.1, depth_stretch_hi=0.9,
         fg_pop_multiplier=1.5, bg_push_multiplier=0.9, subject_lock_strength=0.5, parallax_balance=0.6),
]


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("pi", range(len(PARAMS)))
@pytest.mark.parametrize("kind", ["smooth", "noise"])
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_pixel_shift_vs_oracle(R, size, pi, kind, mode):
    ts, tsh, tf0 = _tol(mode, kind)[:3]
    w, h, iw, ih = size
    kw = PARAMS[pi]
    R.reset_temporal_state()
    gs = O.GlobalState()
    p = O.ShiftParams(**_oracle_kw(kw))
    for i in range(2):  # two frames: the floating-window tracker carries state
        fr, dp = synth_frame(i, iw, ih, kind)
        infos = []
        l, r, s = _ps(R, fr, dp, w, h, kw, infos)
        ol, orr, os_, parts = O.pixel_shift(gs, O.bgr_to_rgb01(fr), O.depth_bgr_to_01(dp), w, h, p,
                                            return_parts=True)
        inf = infos[0]
        assert inf.subj_raw == pytest.approx(float(parts["subj_raw"]), abs=ts)
        assert inf.stretch_lo == pytest.approx(float(parts["lo"]), abs=ts)
        assert inf.stretch_hi == pytest.approx(float(parts["hi"]), abs=ts)
        assert inf.subj_shaped == pytest.approx(float(parts["subj"]), abs=2e-5)
        assert inf.zero_parallax_offset == pytest.approx(parts["zpo"], abs=1e-7 if mode == "exact" else 1e-6)
        assert np.abs(s.numpy() - os_).max() <= tsh
        for mine, ref in ((l, ol), (r, orr)):
            mx, f0, f1 = u8_diff(mine, ref)
            assert mx <= 1 and f0 <= tf0, (size, pi, kind, i, mode, mx, f0)


@pytest.mark.parametrize("name", sorted(PS_CASES) + sorted(PS_CASES_EXTRA))
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_pixel_shift_vs_reference_golden(R, golden_dir, name, mode):
    c = {**PS_CASES, **PS_CASES_EXTRA}[name]
    g = load_golden(os.path.join(golden_dir, name))
    R.reset_temporal_state()
    for i in range(c["n"]):
        fr, dp = synth_frame(i, c["iw"], c["ih"], c["kind"])
        l, r, s = _ps(R, fr, dp, c["w"], c["h"], c["kw"])
        assert np.abs(s.numpy() - g[f"shift{i}"]).max() <= 1e-3
        for mine, ref in ((l, g[f"left{i}"]), (r, g[f"right{i}"])):
            mx, f0, f1 = u8_diff(mine, ref)
            assert mx <= 1, (name, i, mx)


@pytest.mark.parametrize("name", sorted(PS_NATURAL))
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_pixel_shift_natural_vs_reference(R, golden_dir, name, mode):
    """CUDA path against the UNMODIFIED reference on content off the k/255 grid: eyes <= 1 LSB, < 0.3 % flips."""
    c = PS_NATURAL[name]
    g = load_golden(os.path.join(golden_dir, name))
    R.reset_temporal_state()
    for i in range(c["n"]):
        fr, dp = synth_frame(i, c["iw"], c["ih"], c["kind"])
        l, r, s = _ps(R, fr, dp, c["w"], c["h"], c["kw"])
        assert np.abs(s.numpy() - g[f"shift{i}"]).max() <= 2e-5
        for mine, ref in ((l, g[f"left{i}"]), (r, g[f"right{i}"])):
            mx, f0, f1 = u8_diff(mine, ref)
            assert mx <= 1 and f0 <= (0.003 if mode == "exact" else 0.01), (name, mode, i, mx, f0)


@pytest.mark.parametrize("name", sorted(LOOP_NATURAL) + sorted(BIG_NATURAL))
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_render_loop_natural_vs_reference(R, golden_dir, name, mode):
    """Full chain (sharpening on) against the unmodified reference: natural content at 320x180 and at the two
    BASELINE sizes (1080p Half-SBS, 4K Full-SBS; sparse samples of the reference's frames)."""
    big = name in BIG_NATURAL
    c = BIG_NATURAL[name] if big else LOOP_NATURAL[name]
    g = np.load(os.path.join(golden_dir, name))
    rp, _ = _rp(R, c["rp"], c["sw"], c["sh"])
    R.reset_temporal_state()
    for j, i in enumerate(range(1, c["n"])):
        fr, dp = synth_frame(i, c["sw"], c["sh"], c["kind"])
        out = R.render_frame(fr, dp, rp)
        ref = g[f"final{j}_{c['key']}"] if big else g[f"final{j}"]
        mine = out[::c["step"], ::c["step"]] if big else out
        assert mine.shape == ref.shape
        mx, f0, f1 = u8_diff(mine, ref)
        _, _, _, tf0, tf1, tmx = _tol(mode, "natural")
        assert mx <= tmx and f1 <= tf1 and f0 <= tf0, (name, mode, j, mx, f0, f1)


def _rp(R, d, w, h):
    o = O.RenderParams(**d)
    return R.make_render_params(
        o.output_width, o.output_height, o.fg_shift, o.mg_shift, o.bg_shift, o.sharpness_factor,
        o.output_format, o.aspect_ratio, o.dof_strength, o.feather_strength, o.blur_ksize,
        o.use_subject_tracking, o.use_floating_window, o.max_pixel_shift_percent,
        o.preserve_original_aspect, o.zero_parallax_strength, o.enable_edge_masking, o.enable_feathering,
        o.original_video_width, o.original_video_height, o.convergence_strength,
        o.enable_dynamic_convergence, o.ipd_factor, o.color_saturation, o.color_contrast,
        o.color_brightness), o


@pytest.mark.parametrize("name", sorted(LOOP_CASES) + sorted(LOOP_CASES_EXTRA))
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_render_loop_vs_oracle_and_golden(R, golden_dir, name, mode):
    ts, _, _, tf0, tf1, tmx = _tol(mode, "smooth")
    c = {**LOOP_CASES, **LOOP_CASES_EXTRA}[name]
    g = np.load(os.path.join(golden_dir, name))
    rp, orp = _rp(R, c["rp"], c["sw"], c["sh"])
    R.reset_temporal_state()
    gs, cs = O.GlobalState(), O.ClipState()
    for j, i in enumerate(range(1, c["n"])):
        fr, dp = synth_frame(i, c["sw"], c["sh"], c["kind"])
        out, inf = R.render_frame(fr, dp, rp, want_info=True)
        ref, parts = O.render_frame(gs, cs, fr, dp, orp, return_parts=True)
        assert out.shape == ref.shape
        assert inf.dyn_scale == pytest.approx(parts["dyn"], abs=1e-6)
        assert inf.focal_depth == pytest.approx(parts["focal"], abs=ts)
        assert inf.stable_zero == pytest.approx(parts["stable_zero"], abs=1e-7 if mode == "exact" else 1e-6)
        assert inf.bar_width == parts["bar"]
        assert inf.pct_lo == pytest.approx(float(gs.pct_lo), abs=1e-6)
        assert inf.pct_hi == pytest.approx(float(gs.pct_hi), abs=1e-6)
        mx, f0, f1 = u8_diff(out, ref)
        assert mx <= tmx and f1 <= tf1 and f0 <= tf0, (name, mode, j, mx, f0, f1)
        mx, f0, f1 = u8_diff(out, g[f"final{j}"])  # vs the real reference: see test_oracle_golden docstring
        assert mx <= max(12, tmx) and f1 <= max(0.03, tf1), (name, mode, j, mx, f0, f1)


def test_render_clip_equals_frame_by_frame(R):
    import ctypes as C
    from visiondepth3d_b200 import _lib
    rp, _ = _rp(R, LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], 320, 180)
    frames = [synth_frame(i, 320, 180, "smooth") for i in range(5)]
    R.reset_temporal_state()
    single = [R.render_frame(f, d, rp) for f, d in frames]
    R.reset_temporal_state()
    ctx = _lib.default_context(0)
    n = len(frames)
    outs = [np.empty_like(single[0]) for _ in range(n)]
    fp = (C.c_void_p * n)(*[f.ctypes.data for f, _ in frames])
    dp = (C.c_void_p * n)(*[d.ctypes.data for _, d in frames])
    op = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
    ctx.check(ctx.lib.vd3d_render_clip(ctx.h, n, fp, dp, 3, 180, 320, C.byref(rp), op, _lib.MEM_HOST, None))
    for a, b in zip(single, outs):
        assert np.array_equal(a, b)


def test_stage_sharpen_and_dof(R):
    rng = np.random.default_rng(3)
    fr = rng.integers(0, 256, (97, 131, 3), dtype=np.uint8)
    for f in (0.0, 0.2, 1.0, 2.5):
        assert np.array_equal(R.apply_sharpening(fr, f), O.sharpen(fr, f))
    d = rng.random((1, 97, 131), dtype=np.float32)
    for sig in (2.0, 1.0, 3.5):
        out = R.dof_grade_frame(fr, d, 0.4, sig, 1.1, 1.05, 0.02)
        t = O.color_grade(O.apply_dof(O.bgr_to_rgb01(fr), d, 0.4, max_sigma=sig), 1.1, 1.05, 0.02)
        mx, f0, f1 = u8_diff(out, O.rgb01_to_bgr8(t))
        assert mx <= 1 and f0 <= 0.002, (sig, mx, f0)
    # DOF off: colour grade only, including the reference's lossy identity grade
    out = R.dof_grade_frame(fr, None, 0.0, 0.0, 1.0, 1.0, 0.0)
    assert np.array_equal(out, O.rgb01_to_bgr8(O.color_grade(O.bgr_to_rgb01(fr), 1.0, 1.0, 0.0)))
    # depth at another resolution is resized like core/render_3d.py:1347-1350
    d2 = rng.random((1, 49, 66), dtype=np.float32)
    out = R.dof_grade_frame(fr, d2, 0.5, 2.0)
    t = O.color_grade(O.apply_dof(O.bgr_to_rgb01(fr), O.resize_bilinear(d2, 97, 131), 0.5, max_sigma=2.0))
    mx, f0, _ = u8_diff(out, O.rgb01_to_bgr8(t))
    assert mx <= 1 and f0 <= 0.002


@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_edge_cases(R, mode):
    def same(a, b):
        if mode == "exact":
            return np.array_equal(a, b)
        mx, f0, f1 = u8_diff(a, b)
        return a.shape == b.shape and mx <= 16 and f1 <= 0.10

    # flat depth: both percentile guards trip (core/render_3d.py:252-253, 538-540), subject fallback 0.5
    fr = np.full((90, 160, 3), 128, dtype=np.uint8)
    dp = np.full((90, 160, 3), 77, dtype=np.uint8)
    rp, orp = _rp(R, dict(LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], output_width=160, output_height=90), 160, 90)
    R.reset_temporal_state()
    gs, cs = O.GlobalState(), O.ClipState()
    for _ in range(2):
        out, inf = R.render_frame(fr, dp, rp, want_info=True)
        ref = O.render_frame(gs, cs, fr, dp, orp)
        assert same(out, ref)
    assert gs.pct_lo is None and inf.pct_lo == 0.0
    # black and white frames
    for v in (0, 255):
        fr[:] = v
        dp[:] = v
        R.reset_temporal_state()
        gs, cs = O.GlobalState(), O.ClipState()
        assert same(R.render_frame(fr, dp, rp), O.render_frame(gs, cs, fr, dp, orp))
    # single-channel depth == grey BGR depth
    f2, d2 = synth_frame(2, 160, 90, "smooth")
    R.reset_temporal_state()
    a = R.render_frame(f2, d2, rp)
    R.reset_temporal_state()
    b = R.render_frame(f2, np.ascontiguousarray(d2[..., 0]), rp)
    assert np.array_equal(a, b)
    # aspect crop (4:3 source into a 16:9 target) follows core/render_3d.py:1236-1248
    f3, d3 = synth_frame(1, 200, 150, "smooth")
    rp3, orp3 = _rp(R, dict(LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], output_width=192, output_height=108), 200, 150)
    R.reset_temporal_state()
    gs, cs = O.GlobalState(), O.ClipState()
    out = R.render_frame(f3, d3, rp3)
    ref = O.render_frame(gs, cs, f3, d3, orp3)
    mx, f0, f1 = u8_diff(out, ref)
    assert out.shape == ref.shape and mx <= _tol(mode, "smooth")[5] and f1 <= _tol(mode, "smooth")[4]


_FULL_SIZE_ORACLE = {}


@pytest.mark.parametrize("cfg", ["1080p_halfsbs", "4k_fullsbs"])
@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_full_size_properties(R, cfg, mode):
    """BASELINE sizes: oracle comparison on one frame (seconds on CPU) plus properties."""
    if cfg == "1080p_halfsbs":
        sw, sh = 1920, 1080
        d = dict(output_width=1920, output_height=1080, output_format="Half-SBS", sharpness_factor=0.2,
                 feather_strength=10.0, blur_ksize=9, use_subject_tracking=True, use_floating_window=True,
                 zero_parallax_strength=0.01)
    else:
        sw, sh = 3840, 2160
        d = dict(output_format="Full-SBS", preserve_original_aspect=True, sharpness_factor=0.2,
                 feather_strength=10.0, blur_ksize=9, use_subject_tracking=True, use_floating_window=True,
                 zero_parallax_strength=0.01)
    rp, orp = _rp(R, d, sw, sh)
    fr, dp = synth_frame(1, sw, sh, "smooth")
    R.reset_temporal_state()
    out, inf = R.render_frame(fr, dp, rp, want_info=True)
    if cfg not in _FULL_SIZE_ORACLE:  # the CPU oracle takes a minute at 4K: computed once for both modes
        gs, cs = O.GlobalState(), O.ClipState()
        ref, parts = O.render_frame(gs, cs, fr, dp, orp, return_parts=True)
        _FULL_SIZE_ORACLE[cfg] = (ref, parts, float(gs.pct_lo))
    ref, parts, pct_lo = _FULL_SIZE_ORACLE[cfg]
    assert out.shape == ref.shape == ((1080, 1920, 3) if cfg == "1080p_halfsbs" else (2160, 7680, 3))
    assert inf.dyn_scale == pytest.approx(parts["dyn"], abs=1e-6)
    assert inf.pct_lo == pytest.approx(pct_lo, abs=1e-6)
    mx, f0, f1 = u8_diff(out, ref)
    _, _, _, tf0, tf1, tmx = _tol(mode, "smooth")
    assert mx <= tmx and f1 <= tf1 and f0 <= tf0, (mode, mx, f0, f1)
    # property: zero shifts -> both eyes identical
    d0 = dict(d, fg_shift=0.0, mg_shift=0.0, bg_shift=0.0, use_subject_tracking=False, use_floating_window=False)
    rp0, _ = _rp(R, d0, sw, sh)
    R.reset_temporal_state()
    o0 = R.render_frame(fr, dp, rp0)
    half = o0.shape[1] // 2
    assert np.array_equal(o0[:, :half], o0[:, half:])
    # property: determinism / idempotent state reset
    R.reset_temporal_state()
    assert np.array_equal(R.render_frame(fr, dp, rp), out)


def test_format_3d_output_on_gpu(R):
    rng = np.random.default_rng(11)
    l = rng.integers(0, 256, (45, 67, 3), dtype=np.uint8)
    r = rng.integers(0, 256, (45, 67, 3), dtype=np.uint8)
    assert np.array_equal(R.format_3d_output(l, r, "Full-SBS"), np.hstack((l, r)))
    assert np.array_equal(R.format_3d_output(l, r, "Half-SBS"), np.hstack((l, r)))
    assert np.array_equal(R.generate_anaglyph_3d(l, r), O.anaglyph(l, r))
    assert np.array_equal(R.format_3d_output(l, r, "Passive Interlaced"), O.format_output(l, r, "Passive Interlaced"))


def test_state_handoff_makes_sharding_exact(R):
    """SURVEY 8(e): chunk B rendered on another context after importing the state that a stats-only
    pass over chunk A produced must equal sequential rendering bit for bit."""
    from visiondepth3d_b200 import _lib
    rp, _ = _rp(R, LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], 320, 180)
    frames = [synth_frame(i, 320, 180, "smooth") for i in range(9)]
    main = _lib.default_context(0)
    main.reset()
    seq = [R.render_frame(f, d, rp, ctx=main) for f, d in frames]
    a, b = _lib.Context(0), _lib.Context(0)
    a.reset()
    for f, d in frames[:5]:
        R.advance_state(f, d, rp, ctx=a)        # no rendering on "rank 0" for this check
    blob = a.export_state()
    b.import_state(blob)
    for i in range(5, 9):
        out = R.render_frame(frames[i][0], frames[i][1], rp, ctx=b)
        assert np.array_equal(out, seq[i]), i
    # and the exporter itself can continue rendering from its own state
    assert np.array_equal(R.render_frame(frames[5][0], frames[5][1], rp, ctx=a), seq[5])
    a.close()
    b.close()


def test_heal_missing_pixels(R, golden_dir):
    g = np.load(os.path.join(golden_dir, "heal_160x90.npz"))
    for key, em in (("heal_none", None), ("heal_edge", g["edge"])):
        out = R.heal_missing_pixels(g["warped"], None, g["orig"], em, 0.5)
        assert np.abs(out - g[key]).max() <= 1e-6  # vs the reference function's own output
        assert np.array_equal(out, O.heal_missing_pixels(g["warped"], g["orig"], em, 0.5))
    rng = np.random.default_rng(4)
    w = rng.random((3, 37, 53), dtype=np.float32)
    o = rng.random((3, 37, 53), dtype=np.float32)
    assert np.array_equal(R.heal_missing_pixels(w, None, o, None, 0.8), O.heal_missing_pixels(w, o, None, 0.8))


def _clip(ctx, rp, frames, h, w):
    import ctypes as C
    from visiondepth3d_b200 import _lib
    n = len(frames)
    rp_, _ = rp
    from visiondepth3d_b200 import render_3d as R_
    pl = R_.plan_sizes(w, h, rp_)
    outs = [np.empty(R_.output_shape(rp_, pl), dtype=np.uint8) for _ in range(n)]
    fp = (C.c_void_p * n)(*[f.ctypes.data for f, _ in frames])
    dp = (C.c_void_p * n)(*[d.ctypes.data for _, d in frames])
    op = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
    ctx.check(ctx.lib.vd3d_render_clip(ctx.h, n, fp, dp, 3, h, w, C.byref(rp_), op, _lib.MEM_HOST, None))
    return outs


@pytest.mark.parametrize("mode", MODES, indirect=True)
def test_graph_replay_survives_other_entry_points(R, mode):
    """ADVICE r1: captured frame graphs bake in device pointers and host-cached tables (linspace axes, INTER_AREA
    tables, workspaces).  Another entry point at another size in between must not leave stale graphs behind:
    clip(A) -> render_frame(B) / pixel_shift(B) / fit_eye -> clip(A) equals the same sequence launched eagerly."""
    from visiondepth3d_b200 import _lib
    ctx = _lib.default_context(0)
    rpA = _rp(R, LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], 320, 180)
    rpB = _rp(R, dict(LOOP_CASES["loop_halfsbs_320x180.npz"]["rp"], output_width=256, output_height=144,
                      output_format="Full-SBS", preserve_original_aspect=True), 256, 144)
    fa = [synth_frame(i, 320, 180, "smooth") for i in range(16)]
    fb, db = synth_frame(3, 256, 144, "smooth")
    img = np.random.default_rng(5).integers(0, 256, (270, 480, 3), dtype=np.uint8)

    def sequence():
        R.reset_temporal_state()
        res = _clip(ctx, rpA, fa[:8], 180, 320)          # 3 eager frames, then captured graphs
        res.append(R.render_frame(fb, db, rpB[0]))        # other size: axes, workspaces, state planes
        l, r, s = _ps(R, fb, db, 400, 226, dict(blur_ksize=5, feather_strength=4.0))
        res += [l, r]
        res.append(R.pad_to_aspect_ratio(img, 360, 400))  # INTER_AREA tables
        res += _clip(ctx, rpA, fa[8:], 180, 320)
        return res

    ctx.check(ctx.lib.vd3d_set_graphs(ctx.h, 1))
    with_graphs = sequence()
    ctx.check(ctx.lib.vd3d_set_graphs(ctx.h, 0))
    try:
        eager = sequence()
    finally:
        ctx.check(ctx.lib.vd3d_set_graphs(ctx.h, 1))
    assert len(with_graphs) == len(eager)
    for k, (a, b) in enumerate(zip(with_graphs, eager)):
        assert np.array_equal(a, b), k
