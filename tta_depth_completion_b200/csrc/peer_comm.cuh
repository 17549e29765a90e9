// Peer-memory exchanges of the shared-model mode (BASELINE.json configs[4]; the reference runs it as DDP + SyncBatchNorm,
// src/msg_chn_model_adapt.py:480,555-556 and src/tta_main.py:101-111,327,354).  What crosses the GPUs per step is tiny -- the 2 C
// BatchNorm sums of ten BatchNorm calls and one 296 KB gradient buffer -- so every exchange is ONE-SHOT over NVLink peer memory, inside
// the kernel that needs the result, and the whole step stays one CUDA graph (no NCCL call, no host round trip):
//
//   * every rank owns one cudaMalloc'ed block (flags | arrival counters | epoch | two parities of data slots), mapped into every peer
//     through CUDA IPC (ptta_comm_*);
//   * an exchange `xid`: every block of the kernel writes its part of the rank's slot, the LAST block to arrive (device counter) publishes
//     the slot by storing the step tag into flag[xid][rank] of EVERY peer (st.release.sys), all blocks spin on the rank's own flag row
//     (ld.acquire.sys) until every rank has published, then read the peers' slots with volatile loads and combine them IN RANK ORDER --
//     every rank computes bit-identical sums, so the replicas cannot drift apart;
//   * tags are a per-rank epoch counter advanced at the end of every step (all ranks run the same step sequence); data slots alternate
//     between two parities, so a fast rank two exchanges ahead never overwrites what a slow rank still reads (it cannot get further
//     ahead: the exchange in between needs the slow rank's flag).
//
// The kernels that spin are small, launched on ONE stream in shared mode, so all their blocks are resident.  The NLSPN entry points
// enforce PTTA_COMM_MAX_SPIN_BLOCKS (37): a BatchNorm finalize has cdiv(C, 32) <= 32 blocks (C <= 1024, the slot size), the NLSPN
// flat-buffer Adam 23.
//
// Capacity: PTTA_COMM_MAX_XID exchanges per step; one NLSPN step uses 125 (80 BatchNorm forwards: 36 + 36 encoder
// layers of the real and the zero-image pass, 5 decoder, 3 head; 44 BatchNorm backwards; 1 gradient all-reduce).
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"

namespace ptta {

#define PTTA_COMM_MAX_RANKS 8
#define PTTA_COMM_MAX_XID 256
#define PTTA_COMM_MAX_SPIN_BLOCKS 37         // blocks of one spinning kernel (all resident on 148 SMs with the step on one stream)
#define PTTA_COMM_BN_DOUBLES 2048            // per BatchNorm exchange slot: 2 x up to 1024 channels

struct PeerComm {
    int world = 1, rank = 0;
    unsigned char* base[PTTA_COMM_MAX_RANKS] = {};   // every rank's block as mapped HERE (base[rank] = the local block)
    size_t grad_floats = 0;                          // capacity of the gradient slot
};

// block layout
__host__ __device__ inline size_t comm_flags_off() { return 0; }                                                          // uint32 [XID][RANKS]
__host__ __device__ inline size_t comm_counters_off() { return (size_t)PTTA_COMM_MAX_XID * PTTA_COMM_MAX_RANKS * 4; }        // uint32 [XID]
__host__ __device__ inline size_t comm_epoch_off() { return comm_counters_off() + (size_t)PTTA_COMM_MAX_XID * 4; }           // uint32
__host__ __device__ inline size_t comm_error_off() { return comm_epoch_off() + 4; }                                         // uint32: exchange that timed out + 1
__host__ __device__ inline size_t comm_data_off() { return (comm_error_off() + 4 + 4095) / 4096 * 4096; }                 // 12288
__host__ __device__ inline size_t comm_bn_slot_off(int parity, int xid) {
    return comm_data_off() + ((size_t)parity * PTTA_COMM_MAX_XID + xid) * PTTA_COMM_BN_DOUBLES * sizeof(double);
}
__host__ __device__ inline size_t comm_grad_off(int parity, size_t grad_floats) {
    return comm_data_off() + (size_t)2 * PTTA_COMM_MAX_XID * PTTA_COMM_BN_DOUBLES * sizeof(double) + (size_t)parity * grad_floats * sizeof(float);
}
inline size_t comm_block_bytes(size_t grad_floats) { return comm_grad_off(2, grad_floats) + 256; }

__device__ __forceinline__ uint32_t comm_tag(const PeerComm& c) {
    return *reinterpret_cast<const volatile uint32_t*>(c.base[c.rank] + comm_epoch_off()) + 1u;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Called by ALL threads of ALL blocks of the kernel after the block has written its part of the local slot.
__device__ __forceinline__ void comm_publish_and_wait(const PeerComm& c, int xid, uint32_t tag) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t* counters = reinterpret_cast<uint32_t*>(c.base[c.rank] + comm_counters_off());
        const unsigned nblocks = gridDim.x * gridDim.y * gridDim.z;
        const unsigned t = atomicAdd(&counters[xid], 1u);
        if (t == nblocks - 1) {                              // the whole slot of this rank is written
            counters[xid] = 0;                               // next use: next step
            __threadfence_system();
            for (int r = 0; r < c.world; ++r)
                st_release_sys(reinterpret_cast<uint32_t*>(c.base[r] + comm_flags_off()) + xid * PTTA_COMM_MAX_RANKS + c.rank, tag);
        }
        const uint32_t* mine = reinterpret_cast<const uint32_t*>(c.base[c.rank] + comm_flags_off()) + xid * PTTA_COMM_MAX_RANKS;
        // a peer that never arrives (a rank died, or the ranks issued their exchanges in different orders) must not hang the GPU: after
        // ~4 s the wait gives up and records the exchange id; the host reads it with ptta_comm_error() and the step's results are void
        const long long t0 = clock64();
        for (int r = 0; r < c.world; ++r) {
            while ((int32_t)(ld_acquire_sys(mine + r) - tag) < 0) {
                if (clock64() - t0 > 8000000000LL) {
                    *reinterpret_cast<volatile uint32_t*>(c.base[c.rank] + comm_error_off()) = (uint32_t)xid + 1u;
                    break;
                }
            }
        }
    }
    __syncthreads();
}

__device__ __forceinline__ double ld_volatile_f64(const double* p) { return *reinterpret_cast<const volatile double*>(p); }
__device__ __forceinline__ float ld_volatile_f32(const float* p) { return *reinterpret_cast<const volatile float*>(p); }

// sums of one BatchNorm call over ALL ranks (SyncBatchNorm semantics of the shared-model mode): the owner threads publish the rank's
// (sum, sum of squares) / (sum dy, sum dy xhat) per channel, wait for every rank, and add the ranks' values in rank order.  Called by
// ALL threads of ALL blocks of the kernel (comm_publish_and_wait is a rendezvous); C <= PTTA_COMM_BN_DOUBLES / 2.
__device__ __forceinline__ void bn_sums_all_ranks(const PeerComm& comm, int xid, int C, bool owner, int ch, double& a, double& b) {
    const uint32_t tag = comm_tag(comm);
    const size_t off = comm_bn_slot_off((int)(tag & 1u), xid);
    if (owner) {
        double* slot = reinterpret_cast<double*>(comm.base[comm.rank] + off);
        slot[ch] = a; slot[C + ch] = b;
    }
    comm_publish_and_wait(comm, xid, tag);
    if (owner) {
        a = 0.0; b = 0.0;
        for (int r = 0; r < comm.world; ++r) {
            const double* slot = reinterpret_cast<const double*>(comm.base[r] + off);
            a += ld_volatile_f64(slot + ch); b += ld_volatile_f64(slot + C + ch);
        }
    }
}

}  // namespace ptta

// host handle of the C ABI (include/ptta_b200.h `ptta_comm_*`): the device-side view every engine entry point passes to its kernels,
// the local block and the peers' mapped blocks
struct ptta_comm {
    ptta::PeerComm dev;
    void* local = nullptr;
    void* opened[PTTA_COMM_MAX_RANKS] = {};
    size_t bytes = 0;
};
