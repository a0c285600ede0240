"""pymf.NNDSVD on B200: Non-negative Double SVD initialisation (pymf/nndsvd.py:24-115).

The reference class is ``NMF`` with ``update_w`` replaced by the SVD-based construction of
Boutsidis & Gallopoulos and ``update_h`` a no-op; ``factorize`` always runs exactly one
"iteration".  Its product, ``.W`` / ``.H``, is meant to be copied into an ``NMF`` object as the
starting point of the multiplicative updates (class docstring of the reference, :56-66).  Here
the construction runs in libpymfb (``pymfb_nndsvd``, kernels_svd.cuh): the top-k singular triplets of
``data`` by subspace iteration on the device-resident matrix, the second SVD in closed form.
"""
import numpy as np

from .nmf import NMF

__all__ = ["NNDSVD"]


class NNDSVD(NMF):
    """
    NNDSVD(data, num_bases=4)

    Drop-in for ``pymf.nndsvd.NNDSVD``: after ``factorize()``, ``W`` (data_dimension x num_bases) and
    ``H`` (num_bases x num_samples) hold the non-negative double SVD factors and ``ferr`` the Frobenius
    error ``|data - W*H|``.  ``singular_values`` (extra) holds the leading singular values of ``data``,
    ``svd_sweeps`` the subspace-iteration sweeps it took and ``svd_path`` the kernel family of its passes over
    ``data`` ("simt": fp32 CUDA cores, "tc": 3xTF32 tensor cores; ``path=`` forces one).  ``num_bases`` <= 200.

    With ``process_group`` (column-sharded ``data``, as for ``NMF``) every rank gets the same ``W``,
    ``singular_values`` and ``svd_sweeps`` and its own columns of ``H``: the blocks of what the unsharded data gives,
    ready for a sharded ``NMF`` on the same shards.

    >>> init = NNDSVD(data, num_bases=8); init.factorize()
    >>> mdl = NMF(data, num_bases=8); mdl.W = init.W; mdl.H = init.H; mdl.factorize(niter=50)
    """

    def __init__(self, data, num_bases=4, **kw):
        # path= selects the family of the SVD passes; the engine's own NMF kernels (the error pass) keep their default
        self._svd_path_opt = kw.pop("path", None) or "auto"
        if kw.get("sparse"):
            raise TypeError("NNDSVD of sparse data is not supported: pass a dense array")
        super(NNDSVD, self).__init__(data, num_bases, **kw)

    @staticmethod
    def _native_hooks():
        return NNDSVD

    def init_w(self):                                                    # pymf/nndsvd.py:70-71
        self.W = np.zeros((self._data_dimension, self._num_bases))

    def init_h(self):                                                    # pymf/nndsvd.py:73-74
        self.H = np.zeros((self._num_bases, self._n_local))              # this rank's columns (all of them unsharded)

    def update_h(self):                                                  # pymf/nndsvd.py:76-77
        pass

    def update_w(self):                                                  # pymf/nndsvd.py:79-108
        eng = self._sync_to_device()
        eng.set_nndsvd_path(self._svd_path_opt)
        self.singular_values, self.svd_sweeps = eng.nndsvd()
        self.svd_path = eng.nndsvd_path
        self._mark_device_newer("W")
        self._mark_device_newer("H")

    def factorize(self, niter=1, show_progress=False,
                  compute_w=True, compute_h=True, compute_err=True):
        # "enforce certain default values, otherwise it won't work" (pymf/nndsvd.py:110-115): one pass, W and H
        import logging
        self._logger.setLevel(logging.INFO if show_progress else logging.ERROR)
        if "W" not in self._factors:
            self.init_w()
        if "H" not in self._factors:
            self.init_h()
        self._factorize_template(1, True, True, compute_err)
