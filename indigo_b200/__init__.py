"""
indigo_b200 -- B200 (sm_100a) execution backend for indigo's `Backend` interface.

    from indigo_b200 import B200Backend            # standalone (mirror of the reference interface)
    import indigo_b200; indigo_b200.register()      # plugs into an installed `indigo`
    B = indigo.backends.get_backend('b200')

Importing this package does not touch CUDA; the shared library is loaded (and
its absence reported, loudly) when a backend is constructed.
"""
__all__ = ["B200Backend", "get_backend", "register", "sense_operator", "sense_operator_fused", "normal_operator",
           "pipe_menon_dcf", "toeplitz_normal", "wavelet_operator", "l1wavelet_recon", "spectral_norm", "calibration_kspace", "espirit_maps", "CoilTeam"]


def __getattr__(name):
    if name == "B200Backend":
        from .backend import B200Backend
        return B200Backend
    if name in ("sense_operator", "normal_operator", "sqrt_dcf", "pipe_menon_dcf"):
        from . import sense
        return getattr(sense, name)
    if name == "sense_operator_fused":
        from .fused import sense_operator_fused
        return sense_operator_fused
    if name == "toeplitz_normal":
        from .fused import toeplitz_normal
        return toeplitz_normal
    if name in ("wavelet_operator", "l1wavelet_recon", "spectral_norm"):
        from . import wavelet
        return getattr(wavelet, name)
    if name in ("calibration_kspace", "espirit_maps"):
        from . import espirit
        return getattr(espirit, name)
    if name == "CoilTeam":
        from .team import CoilTeam
        return CoilTeam
    if name == "register":
        from .refcompat import register
        return register
    raise AttributeError(name)


def get_backend(name='b200', **init):
    """Mirror of indigo.backends.get_backend (backends/__init__.py:44-64) for this package."""
    if name != 'b200':
        raise ValueError("unrecognized backend: %s" % name)
    from .backend import B200Backend
    return B200Backend(**init)
