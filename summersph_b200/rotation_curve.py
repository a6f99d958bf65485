"""Rotation curves of a disc: the circular speed the gravitational field asks for against the speed the gas has.

For each ring of radius R in the plane z = `z` (`per_ring` points at azimuths (k + 1/2) 2 pi / per_ring around the z
axis through the origin):
  v_c      = sqrt(max(0, R <-g . R_hat>)), g = gas + sinks, averaged over the ring (`sph_gravity_at`, h = h_fixed)
  v_c_gas, v_c_sink: the same with the gas part or the sink part of g alone (inside a disc the gas beyond R can pull
             outward, so v_c_gas is 0 there and v_c falls below v_c_sink)
  v_phi    = the density-weighted ring mean of the gas azimuthal velocity, sum rho v_phi / sum rho (0 where no gas),
             from the mass-weighted velocity of `sph_interpolate` at the same points
The difference between v_phi and v_c is the pressure support (and whatever else the gas feels).  From a save file:

    python -m summersph_b200.rotation_curve save275.txt --variable --rmin 10 --rmax 100 --rings 46 --per-ring 256

prints one row per ring.  There is no CPU path: both fields are evaluated in the CUDA engine.
"""
import argparse
import numpy as np

from ._abi import default_params, MODE_FIXED_H, MODE_VARIABLE_H

COLUMNS = ("R", "v_c", "v_c_gas", "v_c_sink", "v_phi")


def ring_points(radii, per_ring=256, z=0.0):
    """(len(radii) * per_ring, 3) points, ring by ring, and the azimuths of one ring."""
    R = np.asarray(radii, dtype=float).reshape(-1)
    phi = (np.arange(int(per_ring)) + 0.5) * (2.0 * np.pi / int(per_ring))
    pts = np.empty((len(R), len(phi), 3))
    pts[:, :, 0] = R[:, None] * np.cos(phi)[None, :]
    pts[:, :, 1] = R[:, None] * np.sin(phi)[None, :]
    pts[:, :, 2] = float(z)
    return pts.reshape(-1, 3), phi


def rotation_curve(engine, radii, per_ring=256, z=0.0):
    """dict of arrays over the rings: R, v_c, v_c_gas, v_c_sink, v_phi (see the module docstring)."""
    R = np.asarray(radii, dtype=float).reshape(-1)
    pts, phi = ring_points(R, per_ring, z)
    shape = (len(R), len(phi))
    g = engine.gravity_at(pts, n_out=8)
    f = engine.interpolate(pts, n_out=3)
    c, s = np.cos(phi)[None, :], np.sin(phi)[None, :]

    def vc(gx, gy):      # sqrt(R <-g . R_hat>) over each ring
        inward = -(gx.reshape(shape) * c + gy.reshape(shape) * s).mean(1)
        return np.sqrt(np.maximum(0.0, R * inward))

    rho = f["rho"].reshape(shape)
    vphi = -f["vx"].reshape(shape) * s + f["vy"].reshape(shape) * c
    w = rho.sum(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        vphi_mean = np.where(w > 0.0, (rho * vphi).sum(1) / w, 0.0)
    return {"R": R,
            "v_c": vc(g["gx_gas"] + g["gx_sink"], g["gy_gas"] + g["gy_sink"]),
            "v_c_gas": vc(g["gx_gas"], g["gy_gas"]),
            "v_c_sink": vc(g["gx_sink"], g["gy_sink"]),
            "v_phi": vphi_mean}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("save_file")
    ap.add_argument("--variable", action="store_true", help="10-column save of the variable-h program (uses column 10 as h)")
    ap.add_argument("--h-fixed", type=float, default=None, help="fixed-h mode: smoothing length (default: the engine's 2.5)")
    ap.add_argument("--rmin", type=float, default=10.0)
    ap.add_argument("--rmax", type=float, default=100.0)
    ap.add_argument("--rings", type=int, default=46)
    ap.add_argument("--per-ring", type=int, default=256)
    ap.add_argument("--z", type=float, default=0.0)
    ap.add_argument("--out", default=None, help="also write the table to this file (whitespace-separated, one row per ring)")
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
        rc = rotation_curve(e, np.linspace(a.rmin, a.rmax, a.rings), a.per_ring, a.z)
    table = np.stack([rc[k] for k in COLUMNS], 1)
    head = " ".join(f"{k:>22s}" for k in COLUMNS)
    rows = [" ".join(f"{v:22.15e}" for v in row) for row in table]
    print(head)
    print("\n".join(rows))
    if a.out:
        with open(a.out, "w") as f:
            f.write("# " + head[2:] + "\n" + "\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
