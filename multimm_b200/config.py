"""SimulationConfig — the reference's flag set (src/multimm/config.py:94-312) re-hosted without
``openmm.unit``.  Same field names, defaults, coercions and validation behaviour, so a
``config.ini`` written for MultiMM means the same thing here:

* quantities are ``"<float> <unit-expr>"`` strings (config.py:24-49) -> units.Quantity;
* booleans accept true/1/y/yes and false/0/n/no/""/none (config.py:65-77);
* CHROM is normalised to ``chrN`` or None (config.py:82-91);
* empty / "none" strings become None for Optional fields and for LOOPS_PATH, which makes a
  missing loops file a pydantic ValidationError (config.py:103-125, tests/test_run_validation.py:18-24).

New meaning for two existing fields: PLATFORM accepts "B200"; the OpenMM platform names (CUDA,
OpenCL, CPU, Reference, HIP — every ini the reference ships says OpenCL) are taken as the
preference they are in the reference (model.py:862-871) and run on the B200 engine with a logged
warning; anything else is a ValueError.  There is no CPU path.  DEVICE, which the
reference declares but never reads (config.py:131), selects the CUDA device index.
"""
from __future__ import annotations

import os
from enum import Enum
from typing import Any, Optional

from pydantic import BaseModel, BeforeValidator, TypeAdapter, WithJsonSchema, create_model, model_validator
from typing_extensions import Annotated

from .units import Quantity, parse_quantity

_PKG = os.path.dirname(os.path.abspath(__file__))


class InitialStructureType(str, Enum):
    """enums.py:4-13"""

    RW = "rw"
    CONFINED_RW = "confined_rw"
    KNOT = "knot"
    SELF_AVOIDING_RW = "self_avoiding_rw"
    CIRCLE = "circle"
    HELIX = "helix"
    SPIRAL = "spiral"
    SPHERE = "sphere"
    HILBERT = "hilbert"


def _to_quantity(v: Any) -> Quantity:
    if isinstance(v, Quantity):
        return v
    if isinstance(v, str):
        return parse_quantity(v)
    raise ValueError(f"Cannot cast {type(v)} to Quantity")


def _to_bool(v: Any) -> bool:
    if isinstance(v, bool):
        return v
    if isinstance(v, (int, float)):
        return bool(v)
    if isinstance(v, str):
        low = v.strip().lower()
        if low in ("true", "1", "y", "yes"):
            return True
        if low in ("false", "0", "n", "no", "", "none"):
            return False
    raise ValueError(f"Cannot cast {v} to boolean")


def _to_chrom(v: Any) -> Optional[str]:
    if v is None:
        return None
    text = str(v).strip()
    if not text or text.lower() == "none":
        return None
    return text if text.startswith("chr") else f"chr{text}"


Q = Annotated[Quantity, BeforeValidator(_to_quantity),
              WithJsonSchema({"type": "string", "description": "'<float> <unit expression>', e.g. '0.1 nanometer'"})]
B = Annotated[bool, BeforeValidator(_to_bool)]
Chrom = Annotated[Optional[str], BeforeValidator(_to_chrom)]

# name -> (type, default).  Order follows the reference so config_auto.ini dumps line up.
_FIELDS: dict[str, tuple[Any, Any]] = {
    "PLATFORM": (str, "B200"),
    "CPU_THREADS": (Optional[int], None),
    "DEVICE": (str, ""),
    "MODELLING_LEVEL": (str, ""),
    "INITIAL_STRUCTURE_PATH": (str, ""),
    "BUILD_INITIAL_STRUCTURE": (B, True),
    "INITIAL_STRUCTURE_TYPE": (InitialStructureType, InitialStructureType.HILBERT),
    "GENERATE_ENSEMBLE": (B, False),
    "COMPARTMENT_FLIP_PROB": (float, 0.0),
    "COMPARTMENT_NOISE_STD": (float, 0.0),
    "N_ENSEMBLE": (Optional[int], None),
    "DOWNSAMPLING_PROB": (float, 1.0),
    # accepted for config.ini compatibility and never read: the reference's ff.xml defines one atom
    # type and no forces (SURVEY 2); the bead mass is loaders.BEAD_MASS
    "FORCEFIELD_PATH": (str, ""),
    "N_BEADS": (int, 50000),
    "COMPARTMENT_PATH": (Optional[str], None),
    "LOOPS_PATH": (str, ""),
    "GENE_TSV": (str, os.path.join(_PKG, "data", "hg38_gtf_annotations.tsv")),
    "GENE_NAME": (str, ""),
    "GENE_ID": (str, ""),
    "GENE_WINDOW": (int, 100000),
    "ATACSEQ_PATH": (Optional[str], None),
    "OUT_PATH": (str, "results"),
    "LOC_START": (Optional[int], None),
    "LOC_END": (Optional[int], None),
    "CHROM": (Chrom, None),
    "SHUFFLE_CHROMS": (B, False),
    "SHUFFLING_SEED": (int, 0),
    "SAVE_PLOTS": (B, True),
    "POL_USE_HARMONIC_BOND": (B, True),
    "POL_HARMONIC_BOND_R0": (Q, "0.1 nanometer"),
    "POL_HARMONIC_BOND_K": (Q, "300000.0 kilojoules_per_mole/nanometer**2"),
    "POL_USE_HARMONIC_ANGLE": (B, True),
    "POL_HARMONIC_ANGLE_R0": (Q, "3.141592653589793 radian"),
    "POL_HARMONIC_ANGLE_CONSTANT_K": (Q, "100.0 kilojoules_per_mole/radian**2"),
    "LE_USE_HARMONIC_BOND": (B, True),
    "LE_FIXED_DISTANCES": (B, False),
    "LE_HARMONIC_BOND_R0": (Q, "0.1 nanometer"),
    "LE_HARMONIC_BOND_K": (Q, "30000.0 kilojoules_per_mole/nanometer**2"),
    "EV_USE_EXCLUDED_VOLUME": (B, True),
    "EV_EPSILON": (float, 100.0),
    "EV_R_SMALL": (float, 0.05),
    "EV_POWER": (float, 6.0),
    "SC_USE_SPHERICAL_CONTAINER": (B, False),
    "SC_RADIUS1": (Optional[Q], None),
    "SC_RADIUS2": (Optional[Q], None),
    "SC_SCALE": (float, 1000.0),
    "CHB_USE_CHROMOSOMAL_BLOCKS": (B, False),
    "CHB_KC": (float, 0.3),
    "CHB_DE": (float, 1e-4),
    "COB_USE_COMPARTMENT_BLOCKS": (B, False),
    "COB_DISTANCE": (Optional[Q], None),
    "COB_EA": (float, 1.0),
    "COB_EB": (float, 2.0),
    "SCB_USE_SUBCOMPARTMENT_BLOCKS": (B, False),
    "SCB_DISTANCE": (Optional[Q], None),
    "SCB_EA1": (float, 1.0),
    "SCB_EA2": (float, 1.33),
    "SCB_EB1": (float, 1.66),
    "SCB_EB2": (float, 2.0),
    "IBL_USE_B_LAMINA_INTERACTION": (B, False),
    "IBL_SCALE": (float, 400.0),
    "CF_USE_CENTRAL_FORCE": (B, False),
    "CF_STRENGTH": (float, 20.0),
    "NUC_DO_INTERPOLATION": (B, False),
    "MAX_NUCS_PER_BEAD": (int, 4),
    "NUC_RADIUS": (float, 0.1),
    "POINTS_PER_NUC": (int, 20),
    "PHI_NORM": (float, 0.6283185307179586),
    "SIM_RUN_MD": (B, False),
    "SIM_N_STEPS": (int, 10000),
    "SIM_ERROR_TOLERANCE": (float, 0.01),
    "SIM_AMD_ALPHA": (float, 100.0),
    "SIM_AMD_E": (float, 1000.0),
    "SIM_SAMPLING_STEP": (int, 100),
    "SIM_INTEGRATOR_TYPE": (str, "langevin"),
    "SIM_INTEGRATOR_STEP": (Q, "1 femtosecond"),
    "SIM_FRICTION_COEFF": (float, 0.5),
    "SIM_SET_INITIAL_VELOCITIES": (B, False),
    "SIM_TEMPERATURE": (Q, "310 kelvin"),
    "TRJ_FRAMES": (int, 2000),
    "EV_FORCE_TYPE": (str, "powerlaw"),
    "COB_FORCE_TYPE": (str, "gaussian"),
    "SCB_FORCE_TYPE": (str, "gaussian"),
    "BLAMINA_FORCE_TYPE": (str, "sin"),
    "LE_LOOP_FORCE_TYPE": (str, "harmonic"),
    "CHB_FORCE_TYPE": (str, "polynomial"),
    "CENTRAL_FORCE_TYPE": (str, "harmonic"),
    # engine extensions (not in the reference)
    "PAIR_CUTOFF": (float, 0.0),          # nm; 0 = exact all-pairs (the reference's NoCutoff)
    "MIN_COARSE_CUTOFF": (float, 0.0),    # nm; > 0: minimise with cut-off forces first, then finish on the exact potential
    "MIN_COARSE_FAR_FIELD": (str, "clusters"),  # coarse stage only: CHB and the EV tail beyond the cut-off between cluster centroids ("clusters"), or the exact CHB pass and no tail ("exact")
    "MIN_COARSE_TOLERANCE": (float, 1.0),  # first coarse round converges to this fraction of MIN_TOLERANCE; x 0.7 per further round
    "MIN_COARSE_ROUNDS": (int, 4),         # coarse -> exact-probe rounds before the exact stage runs unbounded
    "MIN_EXACT_PROBE_ITERATIONS": (int, 30),  # bound of the exact stage in all rounds but the last
    "MIN_COARSE_MAX_ITERATIONS": (int, 20000),  # bound of the coarse stage (a truncated potential may never meet the tolerance)
    "MIN_TOLERANCE": (float, 10.0),       # kJ/mol/nm, OpenMM's minimizeEnergy default
    "MIN_MAX_ITERATIONS": (int, 0),       # 0 = until converged (OpenMM default)
}

# Contact-map settings (multimm_b200.contacts; not in the reference).  They are accepted from the ini and
# the command line like the fields above and validated the same way, but kept as model extras that exist
# only when given: a config without them has exactly the reference's field set plus the engine knobs above,
# and dumps (config_auto.ini, parameters.txt) exactly as before.  Read them with contact_setting().
CONTACT_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_CONTACTS": (B, False),          # count contacts of the minimised structure (analysis/contacts.npz; ensembles: ensemble_contacts.npz)
    "CONTACT_RADIUS": (float, 0.2),       # nm; a bead pair closer than this is a contact (2 x the default bond length)
    "CONTACT_RESOLUTION": (int, 0),       # bp per bin of the contact map; 0 = about 1000 bins over the modelled genome or region
}
# The fine (sparse) contact map, kept the same way; effective only with SAVE_CONTACTS.
CONTACT_FINE_FIELDS: dict[str, tuple[Any, Any]] = {
    "CONTACT_FINE_RESOLUTION": (int, 0),  # bp per bin of the sparse map (contacts_fine.npz); 0 = off
}
# Mean-distance maps and radial profiles (multimm_b200.distances), kept the same way.
DISTANCE_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_DISTANCES": (B, False),         # distance sums of the minimised structure (analysis/distances.npz; ensembles: ensemble_distances.npz)
    "DISTANCE_RESOLUTION": (int, 0),      # bp per bin of the distance map; 0 = about 1000 bins, at most 4096 bins
}
# Trajectory maps: the maps above summed over structures sampled during MD (files *_md.npz), kept the same way.
# Which maps are sampled follows SAVE_CONTACTS, CONTACT_FINE_RESOLUTION and SAVE_DISTANCES.
MD_SAMPLE_FIELDS: dict[str, tuple[Any, Any]] = {
    "MD_SAMPLE_STEP": (int, 0),           # MD steps between two structures added to the trajectory maps; 0 = off
}
# Loop readout (multimm_b200.loops), kept the same way: per-loop contact frequencies and anchor distances and
# aggregate peak analysis of the rows of LOOPS_PATH; the contact test uses CONTACT_RADIUS, and MD_SAMPLE_STEP
# also samples it.
LOOP_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_LOOPS": (B, False),             # measure the input loops in the minimised structure (analysis/loops.npz; ensembles: ensemble_loops.npz)
    "LOOP_APA_WINDOW": (int, 10),         # beads on each side of an anchor in the APA window, in [0, 25]
}
# Three-way contact maps (multimm_b200.triplets), kept the same way: bead triples in mutual contact, binned in
# genomic coordinates; the contact test uses CONTACT_RADIUS, and MD_SAMPLE_STEP also samples them.
TRIPLET_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_TRIPLETS": (B, False),          # three-way contacts of the minimised structure (analysis/triplets.npz; ensembles: ensemble_triplets.npz)
    "TRIPLET_RESOLUTION": (int, 0),       # bp per bin of the three-way map; 0 = about 1000 bins, at most 2^20 bins
}
# Locus dynamics of MD runs (multimm_b200.dynamics), kept the same way: mean squared displacements per genomic bin
# and of the loop anchors, and loop lifetimes, over the structures MD_SAMPLE_STEP samples; the loop state uses
# CONTACT_RADIUS.
DYNAMICS_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_DYNAMICS": (B, False),          # MSDs and loop lifetimes of the MD samples (analysis/dynamics.npz; ensembles: ensemble_dynamics.npz)
    "DYNAMICS_RESOLUTION": (int, 0),      # bp per bin of the per-bin MSD; 0 = about 1000 bins, at most 2^22 bins
    "DYNAMICS_MAX_LAG": (int, 64),        # largest lag in samples, a power of two in [1, 4096]; lags 1, 2, 4, ..., max
}
# Distance distributions per genomic bin pair (multimm_b200.disthist), kept the same way: bead pairs counted per
# distance cell between the edges; MD_SAMPLE_STEP also samples them.
DISTANCE_HIST_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_DISTANCE_HIST": (B, False),     # distance histograms of the minimised structure (analysis/distance_hist.npz; ensembles: ensemble_distance_hist.npz)
    "DISTANCE_HIST_RESOLUTION": (int, 0), # bp per bin; 0 = about 1000 bins; B (B + 1) / 2 x (edges + 1) <= 2^27 counters
    "DISTANCE_HIST_EDGES": (str, "0.1,0.15,0.2,0.3,0.5,0.7,1,1.5,2,3,5,7,10,15,20,30,50,70,100"),  # cell edges in nm, comma-separated, strictly increasing, 1 to 63
}
# Genome architecture mapping (multimm_b200.gam), kept the same way: bins co-detected in random thin slices of each
# structure; MD_SAMPLE_STEP also samples it.
GAM_FIELDS: dict[str, tuple[Any, Any]] = {
    "SAVE_GAM": (B, False),               # GAM co-segregation of the minimised structure (analysis/gam.npz; ensembles: ensemble_gam.npz)
    "GAM_RESOLUTION": (int, 0),           # bp per bin; 0 = about 1000 bins; B (B + 1) / 2 <= 2^27
    "GAM_SLICES": (int, 1024),            # slices per structure, in [1, 65536]
    "GAM_SLICE_FRACTION": (float, 0.025), # slice thickness over the envelope diameter, in (0, 1]
}
EXTRA_FIELDS = {**CONTACT_FIELDS, **CONTACT_FINE_FIELDS, **DISTANCE_FIELDS, **MD_SAMPLE_FIELDS, **LOOP_FIELDS,
                **TRIPLET_FIELDS, **DYNAMICS_FIELDS, **DISTANCE_HIST_FIELDS, **GAM_FIELDS}
_CONTACT_ADAPTERS = {name: TypeAdapter(ftype) for name, (ftype, _) in EXTRA_FIELDS.items()}


def contact_setting(args, name: str):
    """Value of a CONTACT_FIELDS, CONTACT_FINE_FIELDS, DISTANCE_FIELDS, MD_SAMPLE_FIELDS, LOOP_FIELDS,
    TRIPLET_FIELDS, DYNAMICS_FIELDS, DISTANCE_HIST_FIELDS or GAM_FIELDS setting of `args`, its default where it
    was not given."""
    extra = getattr(args, "__pydantic_extra__", None) or {}
    return extra.get(name, EXTRA_FIELDS[name][1])


class _Base(BaseModel):
    model_config = {
        "arbitrary_types_allowed": True,
        "populate_by_name": True,
        "validate_assignment": True,
        "validate_default": True,
        "extra": "allow",  # for EXTRA_FIELDS only: every other unknown key is dropped in _blank_to_none
    }

    @model_validator(mode="before")
    @classmethod
    def _blank_to_none(cls, data: Any) -> Any:
        """'' / 'none' -> None where the field may be None (and for LOOPS_PATH, which may not:
        that is what turns a missing loops file into a ValidationError)."""
        if not isinstance(data, dict):
            return data
        out = {}
        for key, val in data.items():
            if key in EXTRA_FIELDS:
                if val is not None:  # given: validated like a field (ValueError -> ValidationError)
                    out[key] = _CONTACT_ADAPTERS[key].validate_python(val)
                continue
            if key not in _FIELDS:  # unknown keys are ignored, as pydantic's default does
                continue
            if isinstance(val, str) and val.strip().lower() in ("", "none"):
                ftype = _FIELDS.get(key, (str, None))[0]
                nullable = type(None) in getattr(ftype, "__args__", ()) or ftype is Chrom
                out[key] = None if (key == "LOOPS_PATH" or nullable) else ""
            else:
                out[key] = val
        return out


SimulationConfig = create_model(
    "SimulationConfig", __base__=_Base, **{name: (ftype, default) for name, (ftype, default) in _FIELDS.items()})
SimulationConfig.__doc__ = __doc__
