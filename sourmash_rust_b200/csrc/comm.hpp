// comm.hpp -- multi-GPU exchange steps of the path over NCCL, inside the library (comm.cu).
#pragma once
#include <functional>
#include <vector>

#include "collection.hpp"

namespace smb200 {

constexpr int COMM_ID_BYTES = 128;  // sizeof(ncclUniqueId)

void comm_unique_id(uint8_t out[COMM_ID_BYTES]);                            // ncclGetUniqueId, on one rank
void comm_init(const uint8_t id[COMM_ID_BYTES], int rank, int world);       // collective
void comm_destroy();
int comm_rank();
int comm_world();
int comm_nccl_version();

// every rank's rows, in rank order, on every rank (collective)
SketchCollection *collection_allgather(SketchCollection &local);
// rows of `local` x all ranks' rows; returns the gathered collection (collective).  The join's hash table over the
// local rows is built while the gather is in flight.
SketchCollection *compare_matrix_allgather(SketchCollection &local, int mode, uint32_t *common, uint32_t *size, double *ratio,
                                           uint64_t ld, bool out_on_device);
// mh := merge of every rank's mh, folded in rank order (collective)
void comm_allmerge(KmerMinHash &mh);
// LinearIndex::find over an index partitioned by rank; same result on every rank (collective)
uint64_t linear_find_sharded(SketchCollection &index_part, SketchCollection &queries, int mode, double threshold,
                             uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap);

}  // namespace smb200
