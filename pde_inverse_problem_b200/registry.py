"""Mirror of registry.py:1-32 (same names, same dispatch)."""
from .example_problems.fokker_planck_example import FokkerPlanck
from .example_problems.fokker_planck_example_GMM import FokkerPlanckGMM
from .example_problems.kinetic_fokker_planck_example_OU import KineticFokkerPlanck as KFPOU
from .example_problems.kinetic_fokker_planck_example_GMM import KineticFokkerPlanck as KFPGMM
from .example_problems.kinetic_mckean_vlasov_example_quadratic import KineticMcKeanVlasov as KMVOU
from .methods.consistency import ConsistencyBased

FokkerPlanckPotential = {
    "Quadratic": FokkerPlanck,
    "GMM": FokkerPlanckGMM,
}

KineticFokkerPlanckPotential = {
    "Quadratic": KFPOU,
    "GMM": KFPGMM,
}

KineticMcKeanVlasovPotential = {
    "Quadratic": KMVOU,
}


def get_pde_instance(cfg):
    if cfg.pde_instance.name == "Fokker-Planck":
        # any potential other than "GMM" is the reference's overdamped OU instance
        return FokkerPlanckPotential.get(cfg.pde_instance.get("potential"), FokkerPlanck)
    elif cfg.pde_instance.name == "Kinetic-Fokker-Planck":
        return KineticFokkerPlanckPotential[cfg.pde_instance.potential]
    elif cfg.pde_instance.name == "Kinetic-McKean-Vlasov":
        return KineticMcKeanVlasovPotential[cfg.pde_instance.potential]
    else:
        # the reference *returns* the exception class here (registry.py:26); raising is the evident intent
        raise NotImplementedError(cfg.pde_instance.name)


def get_method(cfg):
    if cfg.solver.name == "ConsistencyBased":
        return ConsistencyBased
    else:
        raise NotImplementedError
