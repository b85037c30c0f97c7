// Stream of one position of a draw batch (stream contract: philox.cuh; StreamId: engine.h).
#pragma once

#include "engine.h"
#include "philox.cuh"

namespace bl {

// Position `obs` of the batch draws from (seed, obs0 + obs); with id.chain_len > 0 the batch holds independent chains
// side by side, and position obs is observation obs0 + obs mod chain_len of chain obs / chain_len, keyed by seed + chain
// (a batch of chains holds fewer than 2^31 positions).
__device__ __forceinline__ void open_batch_stream(PhiloxSource &src, const StreamId &id, int64_t obs)
{
    if (id.chain_len) {
        const uint32_t ch = (uint32_t)obs / id.chain_len;
        src.open(id.seed + ch, id.obs0 + ((uint32_t)obs - ch * id.chain_len), id.call_id);
    } else {
        src.open(id.seed, id.obs0 + (uint64_t)obs, id.call_id);
    }
}

}  // namespace bl
