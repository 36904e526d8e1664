// rfx_shard.h -- shared by rfx_shard.cu (peer memory plumbing, sharded counting) and rfx_shard_graph.cu (sharded graph stages).
#pragma once
#include "rfx_internal.h"

namespace rfx {

// at offset 0 of every rank's arena: barrier flags written by the peers, values published by the owner
// The published block is double buffered: a rank that has passed the barrier of exchange e may already be writing the values
// of exchange e + 1 while a slower peer still reads those of e (it cannot get two exchanges ahead: e + 1 has a barrier too).
struct ShardCtl {
    unsigned long long flags[RFX_MAX_RANKS];
    unsigned long long pub[2][RFX_PUB_SLOTS];
    unsigned long long flags2[RFX_MAX_RANKS];  // barriers taken INSIDE a kernel (the fused pointer-jumping rounds), own epoch counter
};

// what rfx_shard_export hands out (RFX_SHARD_HANDLE_BYTES = 128)
struct ShardBlob {
    unsigned char handle[64];  // cudaIpcMemHandle_t of the arena
    unsigned long long arena_bytes;
    int rank, device;
    long long pid;             // same process: use `ptr`, no IPC
    unsigned long long ptr;
    unsigned char pad[32];
};
static_assert(sizeof(ShardBlob) == 128, "handle blob is 128 bytes");

struct PeerBases {
    uint8_t* base[RFX_MAX_RANKS];
    int n, me;
};

// values one exchange can carry: slot 0 of the published block is the caller's status
constexpr int PUB_VALS = RFX_PUB_SLOTS - 1;

// everybody's values of the last exchange: value i of rank r (the caller's host values, then its device counters)
struct PubVals {
    unsigned long long v[RFX_MAX_RANKS][PUB_VALS];
    int world = 0;
    unsigned long long at(int r, int i) const { return v[r][i]; }
    unsigned long long sum(int i) const {
        unsigned long long s = 0;
        for (int r = 0; r < world; r++) s += v[r][i];
        return s;
    }
};

PeerBases peer_bases(const Ctx* c);
int shard_barrier(Ctx* c);                       // enqueue a cross-GPU barrier on the context's stream
int shard_check(Ctx* c, const char* what);       // synchronise the stream, report a barrier that timed out
// Publish the status `rc` (RFX_OK or the code this rank fails with), n host values `mine` and n_dev device counters
// dstat[dev_slots[i]] (copied on the stream), barrier, read everybody's values back into `all`.  If any rank published a
// failure, every rank returns the code of the lowest failing rank: a rank that fails still takes part, and its peers do not
// wait for it in the next barrier.
int shard_exchange(Ctx* c, int rc, int n, const unsigned long long* mine, PubVals& all, int n_dev = 0, const int* dev_slots = nullptr);
void shard_graph_release(Ctx* c);
void shard_graph_reset(Ctx* c);  // forget the graph stages' arena buffers (rfx_reset)
void shard_graph_stats(Ctx* c, rfx_shard_stats_t* out);
void shard_graph_set_contigs_global(Ctx* c, uint64_t n_contigs, uint64_t n_bases);  // rfx_shard_stats after a stage that replaced the contigs
void free_all_buffers(Ctx* c);

}  // namespace rfx
