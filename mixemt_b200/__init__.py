"""mixemt_b200 -- B200-native numeric core for svohr/mixemt.

Two functions of the reference are replaced, with unchanged signatures:

    mixemt.preprocess.build_em_matrix   ->  mixemt_b200.preprocess.build_em_matrix
    mixemt.em.run_em (+ em_step)        ->  mixemt_b200.em.run_em / em_step

``install()`` assigns them onto an imported ``mixemt`` package so that the
unmodified CLI, assemble.py and stats.py run on top (see INTEGRATION.md).
Importing this package loads the CUDA shared library and fails loudly when it
has not been built; there is no CPU fallback.
"""
from . import _lib  # noqa: F401  (loads libmixemt_b200.so or raises)
from . import consumers, em, preprocess, runtime  # noqa: F401
from .em import run_em, em_step, init_props, converged  # noqa: F401
from .bootstrap import bootstrap_props, BootstrapResult  # noqa: F401
from .preprocess import build_em_matrix, HapVarBaseMatrix  # noqa: F401

__version__ = "0.1.0"


def install(mixemt_pkg=None, with_consumers=False):
    """Monkeypatch the reference's hot-path entry points (SURVEY.md 8b).

    ``with_consumers=True`` also replaces the functions that walk the N x H
    matrices right after the fit (SURVEY.md 8f N2/N3) with their device-side
    forms from :mod:`mixemt_b200.consumers`; together with resident mode
    (``MIXEMT_B200_RESIDENT=1``) the matrices are then read where they live."""
    if mixemt_pkg is None:
        import mixemt as mixemt_pkg  # the unmodified reference
    mixemt_pkg.preprocess.build_em_matrix = preprocess.build_em_matrix
    mixemt_pkg.em.run_em = em.run_em
    mixemt_pkg.em.em_step = em.em_step
    if with_consumers:
        mixemt_pkg.preprocess.reduce_em_matrix = consumers.reduce_em_matrix
        mixemt_pkg.assemble._find_contribs_from_reads = consumers.find_contribs_from_reads
        mixemt_pkg.assemble.assign_read_indexes = consumers.assign_read_indexes
    return mixemt_pkg
