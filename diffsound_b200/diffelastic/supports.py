"""Stiffness helpers for elastic supports (DiffSoundObj.set_supports)."""


def pad_stiffness(youngs, poisson, thickness):
    """(k_n, k_t) per unit area (N/m^3) of a thin elastic pad of Young's modulus `youngs`, Poisson's ratio `poisson` and
    thickness `thickness` (m) bonded to a rigid ground: the constrained (oedometric) modulus over the thickness,
    E (1 - nu) / ((1 + nu) (1 - 2 nu) t), and the shear modulus over the thickness, E / (2 (1 + nu) t).  Floats or
    broadcastable torch tensors; differentiable in all three."""
    k_n = youngs * (1 - poisson) / ((1 + poisson) * (1 - 2 * poisson) * thickness)
    k_t = youngs / (2 * (1 + poisson) * thickness)
    return k_n, k_t
