// kernels.cuh -- sm_100a device code of the batched commit-index engine.
//
// Every kernel here is HBM-bound u64 index arithmetic over the SoA arena
// (DESIGN.md); there is no floating point and no tensor-core work on this path.
// Reference semantics (file:line relative to the raft-rs checkout) are cited at
// each step; bit-exactness against oracle/raft_oracle.c is the contract.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "raftgpu.h"
#include "wire_format.h"
#include "quorum_select.h"

namespace raftgpu {

#include "k_common.cuh"
#include "k_recompute.cuh"
#include "k_apply.cuh"
#include "k_tile.cuh"
#include "k_tile_compact.cuh"
#include "k_control.cuh"
#include "k_wire.cuh"
#include "k_read.cuh"

}  // namespace raftgpu
