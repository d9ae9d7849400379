"""Numpy reference for the local height by depth layer (TEST INFRASTRUCTURE), built only from ``oracle.steric``.

Layer ``b`` is the local branch of ``steric.py:150-166`` with ``calc_dz(z_l, z_i, deptho, top=edges[b],
bottom=edges[b+1])`` (``derived.py:249-325``) in place of ``calc_dz(z_l, z_i, deptho)``: the skipna column sum of
``dz * delta_rho`` times ``-1/rhozero``, masked where the reference volume of the surface cell is missing.
"""

import numpy as np

from oracle import steric as osteric


def steric_local_layers(
    thetao, so, z_l, z_i, deptho, reference, edges, rhozero=1035.0, patm=101325.0, eos="Wright", variant="steric"
):
    """``edges[-1]`` may be ``None`` (to the sea floor).  Returns ``eta[t, layer, y, x]``."""
    _, delta_rho = osteric.steric_local(thetao, so, z_l, z_i, deptho, reference, rhozero=rhozero, patm=patm, eos=eos,
                                        variant=variant)
    wet = ~np.isnan(reference["volcello"])
    out = []
    for top, bottom in zip(edges[:-1], edges[1:]):
        dz = osteric.calc_dz(z_l, z_i, deptho, top=top, bottom=bottom)
        eta = (-1.0 / rhozero) * np.nansum(dz[None] * delta_rho, axis=1)
        out.append(np.where(wet[0][None], eta, np.nan))
    return np.stack(out, axis=1)
