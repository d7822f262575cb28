"""illico_b200 -- B200-native asymptotic Wilcoxon rank-sum (Mann-Whitney U) tests.

Drop-in for the one hot path of remydubois/illico: ``asymptotic_wilcoxon(adata, ...)`` and the six
batch dispatchers under it, plus ``rank_genes(adata, ...)`` (each group's genes ranked by score, selected on the GPU) and ``ttest(adata, ...)``
(Welch's t-test, scanpy's ``method="t-test"``) and ``rank_genes_groups(adata, ...)`` (a drop-in for scanpy's, writing
``adata.uns``) with its marker filter ``filter_rank_genes_groups(adata, ...)``, computed by hand-written sm_100a CUDA kernels behind a C ABI
(``include/illico_b200.h``).  There is no CPU fallback.
"""
__version__ = "0.1.0"

__all__ = ["asymptotic_wilcoxon", "filter_rank_genes_groups", "rank_genes", "rank_genes_groups", "ttest", "register_into_reference", "__version__"]


def __getattr__(name):
    # lazy: importing the package (e.g. for illico_b200.synth or illico_b200.build) must not need torch/CUDA
    if name == "asymptotic_wilcoxon":
        from .asymptotic_wilcoxon import asymptotic_wilcoxon as fn

        globals()["asymptotic_wilcoxon"] = fn  # rebind: the submodule import bound the module to this name
        return fn
    if name == "rank_genes":
        from .asymptotic_wilcoxon import asymptotic_wilcoxon as aw
        from .ranking import rank_genes as fn

        # (importing .ranking imports the .asymptotic_wilcoxon submodule, which binds the module to that name)
        globals().update(asymptotic_wilcoxon=aw, rank_genes=fn)
        return fn
    if name == "ttest":
        from .asymptotic_wilcoxon import asymptotic_wilcoxon as aw
        from .ttest import ttest as fn

        # (importing .ttest binds the .ttest submodule to this name, and the .asymptotic_wilcoxon module to its own)
        globals().update(asymptotic_wilcoxon=aw, ttest=fn)
        return fn
    if name in ("rank_genes_groups", "filter_rank_genes_groups"):
        from .asymptotic_wilcoxon import asymptotic_wilcoxon as aw
        from .scanpy_compat import filter_rank_genes_groups, rank_genes_groups

        # (importing .scanpy_compat imports .asymptotic_wilcoxon, which binds that module to its name)
        globals().update(asymptotic_wilcoxon=aw, rank_genes_groups=rank_genes_groups,
                         filter_rank_genes_groups=filter_rank_genes_groups)
        return globals()[name]
    if name == "register_into_reference":
        from .registry import register_into_reference as fn

        return fn
    raise AttributeError(name)
