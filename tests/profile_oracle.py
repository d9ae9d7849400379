"""Numpy reference for the area-weighted height change by model level (TEST INFRASTRUCTURE), built only from
``oracle.steric``.

``profile[t, z] = -1/rhozero * nansum_col(m * w * dz * delta_rho[t, z]) / nansum_col(w)``: ``delta_rho`` and ``dz``
are those of the local branch (``steric.py:150-166``, ``derived.py:249-325``), ``m`` is the surface mask of the
reference volume (``steric.py:166``) and ``w`` the column weights, ``areacello`` by default, a NaN weight counting
as 0.  A NaN term is skipped.
"""

import numpy as np

from oracle import steric as osteric


def steric_profile(thetao, so, z_l, z_i, deptho, reference, weights=None, rhozero=1035.0, patm=101325.0, eos="Wright",
                   variant="steric"):
    """Returns ``(profile[t, z], scale[t, z])``; ``scale`` is ``|coef| * nansum_col|m * w * dz * delta_rho| /
    nansum_col(w)``, the size of the terms a profile value sums (the yardstick of a rounding tolerance)."""
    _, delta_rho = osteric.steric_local(thetao, so, z_l, z_i, deptho, reference, rhozero=rhozero, patm=patm, eos=eos,
                                        variant=variant)
    dz = osteric.calc_dz(z_l, z_i, deptho)
    w = np.asarray(reference["areacello"] if weights is None else weights, dtype=np.float64)
    m = ~np.isnan(reference["volcello"][0])
    terms = (m * np.nan_to_num(w, nan=0.0))[None, None] * dz[None] * delta_rho
    coef = -1.0 / rhozero
    total = np.nansum(w)
    return coef * np.nansum(terms, axis=(2, 3)) / total, abs(coef) * np.nansum(np.abs(terms), axis=(2, 3)) / total
