"""legenddsp.jl_b200 -- B200-native (sm_100a) implementation of the LegendDSP.jl `dsp_icpc` hot path.

Public surface (mirrors the reference's names, /root/reference/src/LegendDSP.jl:35-58 for this path):
    DSPConfig, get_fltpars                         src/types.jl, src/utils.jl
    dsp_icpc(data, config, τ, pars_filter)         src/dsp_icpc.jl:62
    dsp_trap/cusp/zac_rt_optimization, dsp_trap/cusp/zac_ft_optimization, dsp_sg_optimization
                                                   src/dsp_filter_optimization.jl:102-441
    dsp_puls, dsp_decay_times                      src/dsp_puls.jl:29, src/dsp_decaytime.jl:11
    extremestats, saturation, tailstats, get_wvf_maximum, thresholdstats(_mad), IntersectMaximum
                                                   the per-waveform primitives, broadcast over waveform arrays

All compute happens in the in-tree CUDA library (csrc/ -> liblgdsp_b200.so) behind the C ABI of
include/lgdsp_b200.h.  Importing this package does not need a GPU; calling a compute function does.
"""
from . import _abi
from ._abi import COLUMNS, COL, INT_COLUMNS, NCOL, UNITS
from .config import (DSPConfig, Q, RddspPolicy, DEFAULT_POLICY, LibBuilders, example_config, tiefree_config,
                     get_fltpars, grid_values, ns, us, resolve_icpc_params, resolve_compressed_params, resolve_sweep_params,
                     trap_variants,
                     trap_sweep_variants, cuspzac_sweep_variants, sg_sweep_variants, SweepVariants, params_summary)
from ._lib import Handle, LgdspError, load_library, LIB_PATH, EXPORTED_SYMBOLS
from .dsp_icpc import (RDWaveforms, TABLE_COLUMNS, COMPRESSED_COLUMNS, dsp_icpc, dsp_icpc_rows, rows_to_table, get_handle,
                       dsp_icpc_compressed, compressed_to_table)
from .dsp_filter_optimization import (dsp_trap_rt_optimization, dsp_trap_ft_optimization, dsp_trap_rtft_grid,
                                      dsp_cusp_rt_optimization, dsp_zac_rt_optimization, dsp_cusp_ft_optimization,
                                      dsp_zac_ft_optimization, dsp_sg_optimization, dsp_sg_optimization_compressed, dsp_qc_flt_optimization,
                                      dsp_qc_flt_optimization_compressed, dsp_qdrift_flt_optimization)
from .dsp_sipm import (dsp_sipm, dsp_sipm_compressed, sipm_rows, sipm_to_table, resolve_sipm_params, example_sipm_config, SIPM_TABLE,
                       VectorOfVectors, IntersectMaximum, MultiIntersect, thresholdstats, thresholdstats_mad)
from .dsp_puls import dsp_puls, dsp_puls_compressed, dsp_decay_times, resolve_puls_params, PULS_COLUMNS
from .stats import extremestats, saturation, tailstats, get_wvf_maximum
from .codec import EncodedWaveforms, encode_waveforms, decode_data, RADWARE_SIGCOMPRESS, ULEB128_ZIGZAG_DIFF
from . import synth, sharding, codec

__all__ = [
    "DSPConfig", "Q", "ns", "us", "RddspPolicy", "example_config", "tiefree_config", "get_fltpars", "grid_values",
    "resolve_icpc_params", "resolve_sweep_params", "trap_variants", "params_summary",
    "Handle", "LgdspError", "load_library", "RDWaveforms", "TABLE_COLUMNS", "dsp_icpc", "dsp_icpc_rows",
    "rows_to_table", "dsp_trap_rt_optimization", "dsp_trap_ft_optimization", "dsp_trap_rtft_grid",
    "dsp_cusp_rt_optimization", "dsp_zac_rt_optimization", "dsp_cusp_ft_optimization", "dsp_zac_ft_optimization",
    "dsp_sg_optimization", "dsp_puls", "dsp_decay_times", "resolve_puls_params", "PULS_COLUMNS", "trap_sweep_variants", "cuspzac_sweep_variants", "sg_sweep_variants",
    "dsp_icpc_compressed", "compressed_to_table", "COMPRESSED_COLUMNS", "resolve_compressed_params",
    "dsp_qc_flt_optimization", "dsp_qc_flt_optimization_compressed", "dsp_qdrift_flt_optimization",
    "dsp_puls_compressed", "dsp_sipm_compressed", "dsp_sg_optimization_compressed",
    "dsp_sipm", "sipm_rows", "sipm_to_table", "resolve_sipm_params", "example_sipm_config", "SIPM_TABLE", "VectorOfVectors",
    "IntersectMaximum", "MultiIntersect", "thresholdstats", "thresholdstats_mad",
    "extremestats", "saturation", "tailstats", "get_wvf_maximum",
    "EncodedWaveforms", "encode_waveforms", "decode_data", "RADWARE_SIGCOMPRESS", "ULEB128_ZIGZAG_DIFF", "codec",
    "synth", "sharding", "COLUMNS", "COL", "INT_COLUMNS", "NCOL", "UNITS",
]
