"""sos-radiative-transfer_b200 -- B200-native Successive-Orders-of-Scattering engine.

Drop-in for the SOS_AER hot path of Guillaume-SOULIER/SOS-Radiative-Transfer: the reference's
I1_NumInt / Jn_NumInt / In_NumInt signatures and SOS_Aer_main_specular / SOS_Aer_main_lambertian
drivers, NumPy arrays in and out, computed by hand-written sm_100a CUDA kernels behind a C ABI
(include/sos_b200.h).  There is no CPU fallback.

The directory name is not a Python identifier; import it as `import sos_b200` (alias module at
the repository root) or with importlib.import_module("sos-radiative-transfer_b200").
"""
from . import _lib
from ._lib import SosError
from .grid import mu_grid, tau_profile, extrapolation_width, aerosol_rows
from .phase import phase_matrices, phase_P, phase_P0, phase_table, phase_modes, phase_exact
from . import brdf
from .brdf import BRDF_NODES, BRDF_MU_MIN, rossli_kernels, brdf_modes, brdf_beam
from . import ocean
from .ocean import cox_munk, glint_modes, glint_beam
from . import mie
from .mie import EVA_AEROSOL, WILDFIRE_AEROSOL
from .engine import SosEngine, ScenarioCoefficients, SolveResult
from .api import I1_NumInt, Jn_NumInt, In_NumInt, mu_approx_In, clear_cache
from . import multi_gpu
from . import graphe
from .graphe import (graphe_diffusivity, graphe_flux, graphe_heating_rate, graphe_successive_dif, graphe_flux_up_down,
                     successive_diffusivity)
from .multi_gpu import PeerFields, PeerBuffers, LayerShardedSolver, MuShardedSolver, mu_blocks, shard_scenarios, gather_scenario_results, allgather_columns, shard_range
from .drivers import (Scenario, DriverResult, BatchSolver, solve_scenarios, SOS_Aer_main_specular,
                      SOS_Aer_main_lambertian, SOS_Aer_radiative_forcing, SOS_Aer_critical_albedo,
                      critical_albedo_sweep, EVA, WILDFIRE, clear_caches)
from .azimuth import AzimuthalResult, solve_azimuthal

__all__ = [
    "SosError", "mu_grid", "tau_profile", "extrapolation_width", "aerosol_rows", "phase_matrices", "phase_P", "phase_P0", "phase_table", "phase_modes", "phase_exact",
    "brdf", "BRDF_NODES", "BRDF_MU_MIN", "rossli_kernels", "brdf_modes", "brdf_beam", "ocean", "cox_munk", "glint_modes", "glint_beam", "mie", "EVA_AEROSOL", "WILDFIRE_AEROSOL",
    "SosEngine", "ScenarioCoefficients", "SolveResult", "I1_NumInt", "Jn_NumInt", "In_NumInt",
    "mu_approx_In", "clear_cache", "Scenario", "DriverResult", "BatchSolver", "solve_scenarios",
    "MuShardedSolver", "LayerShardedSolver", "PeerFields", "PeerBuffers", "mu_blocks", "shard_scenarios", "gather_scenario_results", "allgather_columns", "shard_range",
    "SOS_Aer_main_specular", "SOS_Aer_main_lambertian", "SOS_Aer_radiative_forcing", "SOS_Aer_critical_albedo", "critical_albedo_sweep", "EVA", "WILDFIRE", "clear_caches",
    "AzimuthalResult", "solve_azimuthal",
    "graphe", "graphe_diffusivity", "graphe_flux", "graphe_heating_rate", "graphe_successive_dif", "graphe_flux_up_down", "successive_diffusivity",
]
