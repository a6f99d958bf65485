"""Density images of a run: the B200 counterpart of the reference's Density_Image.py (SURVEY.md §8(f) item 3).

Density_Image.py loads a 9-column `save<N>.txt`, keeps |x|,|y|,|z| < 100, samples the cubic-spline density on
a 120^3 grid with a fixed h = 1.25 through a KD-tree and sums the grid along z (Density_Image.py:64-145).
Here the image is the line-of-sight integral itself, taken on the device from the resident particles with their
own smoothing lengths (`sph_column_density`), either from a live engine or from a save file:

    python -m summersph_b200.density_image save275.txt --variable --size 100 --pixels 512 --out save275.pgm

Writes a binary PGM (8-bit, log scale like a colour-mapped imshow of a disc) and, with --npy, the raw FP64 image.
With --slice OFFSET the image is instead the density on the plane `axis = OFFSET` (a cross-section, what SPLASH-style
slice plots show), sampled at the pixel centres with `sph_interpolate`.
There is no CPU path: the projection and the interpolation run in the CUDA engine.
"""
import argparse
import numpy as np

from ._abi import default_params, MODE_FIXED_H, MODE_VARIABLE_H


def column_density(engine, axis="z", size=100.0, pixels=512):
    """Square frame |u|,|v| < size (Density_Image.py:64), `pixels` x `pixels`."""
    return engine.column_density(axis, (-size, size, -size, size), (pixels, pixels))


_FRAME_AXES = {"x": (1, 2), "y": (2, 0), "z": (0, 1)}       # image axes (u, v) of each view axis, as sph_column_density


def density_slice(engine, axis="z", offset=0.0, size=100.0, pixels=512):
    """Density on the plane `axis = offset` at the pixel centres of the frame of `column_density` (|u|,|v| < size,
    `pixels` x `pixels`, rows along v): `sph_interpolate` column rho."""
    ax = {0: "x", 1: "y", 2: "z"}.get(axis, axis)
    iu, iv = _FRAME_AXES[ax]
    size, pixels = float(size), int(pixels)
    c = -size + (np.arange(pixels) + 0.5) * ((size - -size) / pixels)      # pixel centres, as sph_column_density places them
    pts = np.empty((pixels * pixels, 3))
    pts[:, "xyz".index(ax)] = float(offset)
    pts[:, iu] = np.tile(c, pixels)
    pts[:, iv] = np.repeat(c, pixels)
    return engine.interpolate(pts, n_out=1)["rho"].reshape(pixels, pixels)


def to_gray(img, log=True, decades=4.0):
    """8-bit grey levels: log10 scale over `decades` below the maximum (linear if log=False); empty pixels are 0."""
    img = np.asarray(img, dtype=float)
    top = float(np.nanmax(img)) if img.size else 0.0
    if not top > 0.0:
        return np.zeros(img.shape, np.uint8)
    if log:
        with np.errstate(divide="ignore", invalid="ignore"):
            lv = (np.log10(img / top) + decades) / decades
        lv = np.where(img > 0.0, lv, 0.0)
    else:
        lv = img / top
    return np.uint8(np.clip(np.nan_to_num(lv), 0.0, 1.0) * 255.0 + 0.5)


def save_pgm(path, img, log=True, decades=4.0):
    """Binary PGM with the image ordinate pointing up (imshow origin='lower', Density_Image.py:147)."""
    g = to_gray(img, log, decades)[::-1]
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (g.shape[1], g.shape[0]))
        f.write(np.ascontiguousarray(g).tobytes())


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("save_file")
    ap.add_argument("--variable", action="store_true", help="10-column save of the variable-h program (uses column 10 as h)")
    ap.add_argument("--h-fixed", type=float, default=None, help="fixed-h mode: smoothing length (default: the engine's 2.5; Density_Image.py uses 1.25)")
    ap.add_argument("--axis", default="z", choices=["x", "y", "z"])
    ap.add_argument("--size", type=float, default=100.0)
    ap.add_argument("--pixels", type=int, default=512)
    ap.add_argument("--out", default=None)
    ap.add_argument("--npy", default=None)
    ap.add_argument("--slice", type=float, default=None, metavar="OFFSET",
                    help="write the density on the plane axis = OFFSET instead of the column density")
    ap.add_argument("--device", type=int, default=0)
    a = ap.parse_args(argv)
    from .engine import Engine
    from .textio import read_data_from_file
    p = default_params(MODE_VARIABLE_H if a.variable else MODE_FIXED_H)
    if a.h_fixed is not None:
        p.h_fixed = a.h_fixed
    b, s = read_data_from_file(a.save_file, p)
    with Engine(p, device=a.device) as e:
        e.upload(b, s)
        if a.slice is None:
            img = column_density(e, a.axis, a.size, a.pixels)
        else:
            img = density_slice(e, a.axis, a.slice, a.size, a.pixels)
    out = a.out or (a.save_file.rsplit(".", 1)[0] + ".pgm")
    save_pgm(out, img)
    if a.npy:
        np.save(a.npy, img)
    if a.slice is None:
        print(f" wrote {out}: {a.pixels} x {a.pixels}, sum * pixel area = {img.sum() * (2 * a.size / a.pixels) ** 2!r} (mass in frame)")
    else:
        print(f" wrote {out}: {a.pixels} x {a.pixels} density slice {a.axis} = {a.slice!r}, max {img.max()!r}")


if __name__ == "__main__":
    main()
