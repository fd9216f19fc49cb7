"""Shared helpers for the parity tests."""
import io
import zipfile

import numpy as np


def u8_diff(a, b):
    d = np.abs(a.astype(np.int32) - b.astype(np.int32))
    return int(d.max()), float((d > 0).mean()), float((d > 1).mean())


def save_golden(path, **arrays):
    """Lossless fixture writer for full-frame eyes: an .npz with LZMA-compressed members, and every HxWx3 uint8 image
    stored planar and differenced along x then y (mod 256) under `<key>_dxy`.  That predictor keeps three 320x180
    frames of natural content (eyes + float32 shift maps) under 1 MB, where plain np.savez_compressed needs 1.5 MB."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            a = np.asarray(a)
            if a.dtype == np.uint8 and a.ndim == 3 and a.shape[2] == 3:
                p = a.transpose(2, 0, 1).astype(np.int16)
                a = np.diff(np.diff(p, axis=2, prepend=0), axis=1, prepend=0).astype(np.uint8)
                k += "_dxy"
            buf = io.BytesIO()
            np.lib.format.write_array(buf, a, allow_pickle=False)
            z.writestr(k + ".npy", buf.getvalue())


def load_golden(path):
    """Arrays of a save_golden fixture as a dict, images restored bit-exactly (a plain .npz loads unchanged)."""
    out = {}
    with np.load(path) as g:
        for k in g.files:
            a = g[k]
            if k.endswith("_dxy"):
                k = k[:-4]
                a = np.cumsum(np.cumsum(a, axis=1, dtype=np.uint8), axis=2, dtype=np.uint8)
                a = np.ascontiguousarray(a.transpose(1, 2, 0))
            out[k] = a
    return out


# Parameter sets used by tools/gen_golden.py (kept in one place so the oracle and the
# CUDA path are driven exactly like the reference was).
PS_CASES = {
    "ps_smooth_320x180.npz": dict(w=320, h=180, iw=320, ih=180, n=3, kind="smooth",
                                  kw=dict(blur_ksize=9, feather_strength=10.0, zero_parallax_strength=0.01)),
    "ps_up2_320x180.npz": dict(w=320, h=180, iw=160, ih=90, n=2, kind="smooth",
                               kw=dict(blur_ksize=5, feather_strength=4.0, enable_floating_window=False,
                                       convergence_strength=0.5)),
    "ps_noise_192x108.npz": dict(w=192, h=108, iw=192, ih=108, n=1, kind="noise",
                                 kw=dict(blur_ksize=4, feather_strength=10.0, enable_edge_masking=False,
                                         use_subject_tracking=False)),
}

# oracle-vs-reference only for now (CPU); add to the GPU golden test once run on a B200
PS_CASES_EXTRA = {
    # tools/gen_golden.py extra: every shaping / balance control of pixel_shift_cuda off its default
    "ps_controls_256x144.npz": dict(w=256, h=144, iw=256, ih=144, n=2, kind="smooth",
                                    kw=dict(blur_ksize=5, feather_strength=20.0, convergence_strength=0.3,
                                            enable_dynamic_convergence=False, depth_pop_gamma=0.7, depth_pop_mid=0.4,
                                            depth_stretch_lo=0.1, depth_stretch_hi=0.9, fg_pop_multiplier=1.5,
                                            bg_push_multiplier=0.9, subject_lock_strength=0.5, parallax_balance=0.6,
                                            max_pixel_shift_percent=0.03, zero_parallax_strength=0.02)),
}

_BASE = dict(output_width=320, output_height=180, sharpness_factor=0.2, output_format="Half-SBS",
             dof_strength=0.0, feather_strength=10.0, blur_ksize=9, use_subject_tracking=True,
             use_floating_window=True, preserve_original_aspect=False, zero_parallax_strength=0.01)
LOOP_CASES = {
    "loop_halfsbs_320x180.npz": dict(sw=320, sh=180, n=6, kind="smooth", rp=dict(_BASE)),
    "loop_fullsbs_dof_320x180.npz": dict(
        sw=320, sh=180, n=5, kind="smooth",
        rp=dict(_BASE, output_format="Full-SBS", preserve_original_aspect=True, dof_strength=2.0,
                color_saturation=1.1, color_contrast=1.05, color_brightness=0.02)),
    "loop_anaglyph_256x144.npz": dict(
        sw=256, sh=144, n=3, kind="smooth",
        rp=dict(_BASE, output_format="Red-Cyan Anaglyph", preserve_original_aspect=True,
                use_subject_tracking=False, use_floating_window=False, feather_strength=0.0, blur_ksize=1)),
    "loop_interlaced_256x144.npz": dict(
        sw=256, sh=144, n=3, kind="smooth",
        rp=dict(_BASE, output_format="Passive Interlaced", preserve_original_aspect=True,
                use_subject_tracking=False, use_floating_window=False, feather_strength=0.0, blur_ksize=1)),
}

# VR fixture (tools/gen_golden.py vr): 2880x1600 frames, stored as every 3rd row/column of the image band + sha256
VR_CASE = dict(file="loop_vr_320x180.npz", sw=320, sh=180, n=3, kind="smooth",
               rp=dict(_BASE, output_width=1600, output_height=900, output_format="VR"))

# Extra loop fixtures (tools/gen_golden.py extra): crop / aspect / fractional-fit branches of render_sbs_3d.
# Oracle-vs-reference only (CPU); the CUDA path is compared with the oracle on the same branches in test_dibr_gpu.py.
LOOP_CASES_EXTRA = {
    "loop_crop43_320x240.npz": dict(sw=320, sh=240, n=3, kind="smooth", rp=dict(_BASE)),
    "loop_scope239_320x180.npz": dict(sw=320, sh=180, n=3, kind="smooth", rp=dict(_BASE, aspect_ratio=2.39)),
    "loop_halfsbs_odd_321x180.npz": dict(sw=321, sh=180, n=3, kind="smooth",
                                         rp=dict(_BASE, preserve_original_aspect=True)),
    # the reference was ALSO given parallax_balance=0.6, depth_pop_gamma=0.7, fg_pop_multiplier=1.4 here: render_sbs_3d
    # accepts them but does not forward them to pixel_shift_cuda (SURVEY appendix A), so they must not change the output
    "loop_controls_320x180.npz": dict(
        sw=320, sh=180, n=4, kind="smooth",
        rp=dict(_BASE, sharpness_factor=0.0, ipd_factor=0.8, convergence_strength=0.3,
                enable_dynamic_convergence=False, enable_edge_masking=False)),
    "loop_dof_halfsbs_320x180.npz": dict(sw=320, sh=180, n=3, kind="smooth", rp=dict(_BASE, dof_strength=1.5)),
}

# "natural" set (tools/gen_golden.py natural): band-limited content whose warped values are generic reals instead of
# sitting on the k/255 truncation boundaries of the ramps.  Against the unmodified reference the eyes are <= 1 LSB with
# < 0.1 % one-LSB flips (torch's Sleef powf/expf differ from IEEE by <= 1 ulp), and full frames -- sharpening ON, which
# amplifies an isolated flip up to 7.7 LSB -- have < 0.1 % of bytes off by more than one (2-3 % on the smooth set).
PS_NATURAL = {
    "ps_natural_320x180.npz": dict(w=320, h=180, iw=320, ih=180, n=3, kind="natural",
                                   kw=dict(blur_ksize=9, feather_strength=10.0, zero_parallax_strength=0.01)),
}
LOOP_NATURAL = {
    "loop_natural_halfsbs_320x180.npz": dict(sw=320, sh=180, n=5, kind="natural", rp=dict(_BASE)),
    "loop_natural_fullsbs_320x180.npz": dict(sw=320, sh=180, n=4, kind="natural",
                                             rp=dict(_BASE, output_format="Full-SBS", preserve_original_aspect=True)),
}
# BASELINE sizes against the unmodified reference: every `step`-th row / column of each output frame + sha256
BIG_NATURAL = {
    "loop_natural_1080p_halfsbs.npz": dict(sw=1920, sh=1080, n=3, kind="natural", step=7, key="s7",
                                           rp=dict(_BASE, output_width=1920, output_height=1080)),
    "loop_natural_4k_fullsbs.npz": dict(sw=3840, sh=2160, n=2, kind="natural", step=16, key="s16",
                                        rp=dict(_BASE, output_width=3840, output_height=2160, output_format="Full-SBS",
                                                preserve_original_aspect=True)),
}
