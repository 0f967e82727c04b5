"""B200-native `advance_mu_t` (WRF acoustic small step): CUDA kernels for sm_100a behind the reference
subroutine's argument list.  See DESIGN.md; the C ABI is include/wrfb200.h."""
from ._lib import (EAST, FIELD_ID, FIELDS, FIELDS_1D, FIELDS_2D, FIELDS_3D, KERNEL_AUTO, KERNEL_COLUMN,
                   KERNEL_PIPE, KERNEL_TILE, NORTH, SOUTH, TRANSFER_DIRECT, TRANSFER_MIXED, TRANSFER_STAGED, WEST,
                   WrfB200Error, lib)
from .advance_mu_t import (INPUT_FIELDS, OUTPUT_FIELDS, Grid, Patch, acoustic_loop, advance_mu_t, call_with_fields,
                           compare, default_devices, default_last_kernel, default_last_transfer, host_split_plan, set_default_devices,
                           set_shared_tiles, shared_tiles, synth_fields)

__all__ = ["advance_mu_t", "call_with_fields", "Grid", "Patch", "synth_fields", "compare", "lib", "acoustic_loop", "default_last_kernel",
           "default_last_transfer",
           "set_default_devices", "default_devices", "host_split_plan", "set_shared_tiles", "shared_tiles",
           "FIELDS", "FIELDS_3D", "FIELDS_2D", "FIELDS_1D", "FIELD_ID", "INPUT_FIELDS", "OUTPUT_FIELDS",
           "KERNEL_AUTO", "KERNEL_COLUMN", "KERNEL_TILE", "KERNEL_PIPE", "TRANSFER_DIRECT", "TRANSFER_MIXED", "TRANSFER_STAGED", "WEST", "EAST", "SOUTH", "NORTH", "WrfB200Error"]
