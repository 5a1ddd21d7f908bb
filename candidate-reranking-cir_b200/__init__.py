"""B200-native stage-II candidate re-ranker (and the stage-I cosine/top-K feeding it).

The directory name carries a hyphen (it mirrors the reference repo's name), so import it
through the root-level alias module::

    import cir_b200 as cir
    model = cir.blip_stage2(state_dict=sd)

All math runs in the hand-written sm_100a CUDA library ``csrc/libcir_b200.so`` behind the
C-ABI declared in ``include/cir_b200.h``; there is no CPU or PyTorch fallback.
"""
from . import synthetic  # noqa: F401  (pure-CPU helpers; safe without the CUDA library)

__all__ = ["synthetic"]


def __getattr__(name):
    # Heavy modules (they dlopen the CUDA library) load lazily so that ``synthetic`` stays
    # importable on machines without the built extension.
    import importlib
    if name in ("native", "engine", "schedule", "blip", "blip_stage1", "blip_stage2", "validate",
                "validate_stage2", "distributed", "topk_file", "checkpoint", "build", "online"):
        return importlib.import_module(f"{__name__}.{name}")
    for mod in ("blip_stage1", "blip_stage2"):
        if name in ("BLIP_Retrieval", "BLIP_NLVR"):
            m = importlib.import_module(f"{__name__}.{'blip_stage1' if name == 'BLIP_Retrieval' else 'blip_stage2'}")
            return getattr(m, name)
    raise AttributeError(name)
