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

// slots of ShardCtl::pub
enum {
    PUB_INSTANCES = 0,
    PUB_SLAB_REC = 1,   // 9 slots: slab records, slab counts, slab cap, overflow records, overflow offsets, n overflow, bins, instances, status
    PUB_TABLE = 1,      // rfx_shard_table, 3 + RFX_MAX_RANKS slots (never in use together with PUB_SLAB_REC)
    PUB_GRAPH = 12,     // rfx_shard_graph.cu: GPub
    PUB_END = RFX_PUB_SLOTS
};

PeerBases peer_bases(const Ctx* c);
int shard_barrier(Ctx* c);                       // enqueue a cross-GPU barrier on the context's stream
int shard_check(Ctx* c, const char* what);       // synchronise the stream, report a barrier that timed out
// publish slots [first, first + n) (host values `mine`, then n_dev device counters dstat[dev_slots[i]] copied on the stream into slots dev_first + i),
// barrier, read everybody's slots back: all[r * RFX_PUB_SLOTS + slot]
int shard_exchange(Ctx* c, int first, int n, const unsigned long long* mine, unsigned long long* all /* [RFX_MAX_RANKS * RFX_PUB_SLOTS] */, int n_dev = 0,
                   const int* dev_slots = nullptr, int dev_first = 0);
void shard_graph_release(Ctx* c);
void shard_graph_reset(Ctx* c);  // forget the graph stages' arena buffers (rfx_reset)
void shard_graph_stats(Ctx* c, rfx_shard_stats_t* out);
void free_all_buffers(Ctx* c);

}  // namespace rfx
