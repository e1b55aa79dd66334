// contact.h — collision response kernels (contact.cu).
#pragma once

#include <algorithm>

#include "engine.h"

namespace pies {

struct ClusterView {   // device view of this substep's contact clusters and their entries (contact.cu)
  const uint32_t* nClusters = nullptr;
  const uint32_t* start = nullptr;
  const uint32_t* nodes = nullptr;
  const uint32_t* entStart = nullptr;
  const uint32_t* entryOf = nullptr; // per sorted entry (grouped by cluster, list order inside): its index in the list
  const uint64_t* keys = nullptr;    // per sorted entry: ranks of its four nodes inside the cluster (10 bits each) << 24 | cluster
  const uint32_t* midList = nullptr; // clusters of 33 .. kMidClusterMax nodes
};

struct ClusterTables {  // what reblock.cu produced for this substep
  const uint32_t* nClusters = nullptr;  // device count
  const uint32_t* start = nullptr;      // cluster -> first position in nodes
  const uint32_t* nodes = nullptr;      // touched nodes sorted by cluster
  const uint32_t* clusterOf = nullptr;  // node -> cluster
  const uint32_t* rankOf = nullptr;     // node -> position inside its cluster (== lane inside a small cluster)
  const uint8_t* gsClass = nullptr;     // node -> 0 / 1 (small cluster) / 3 (mid cluster) / 2 (large cluster)
  uint32_t nTouched = 0;
  const uint32_t* midList = nullptr;    // mid clusters (device list)
  const uint32_t* nMidDev = nullptr;    // device count of mid clusters
  const uint32_t* hostCounts = nullptr; // pinned: [0] mid clusters, [1] large clusters, valid once countsReady fired
  cudaEvent_t countsReady = nullptr;
};

struct ContactWork {
  DevBuf<uint32_t> sweepCounters;  // one chunk counter per ordered dataflow sweep of the substep
  DevBuf<float4> contribC;         // 4 per distinct point-triangle contact
  DevBuf<uint64_t> keys, tmpKeys;
  DevBuf<uint32_t> lanes, tmpVals, entStart, sortHist, scanScratch;
  ClusterView view;
  const uint8_t* gsClass = nullptr;
  const uint32_t* hostCounts = nullptr;
  const uint32_t* nMidDev = nullptr;
  cudaEvent_t countsReady = nullptr;
  uint32_t nTri = 0, sweepsUsed = 0, clusterBound = 0;
  bool haveClusters = false;
  // the one-CTA-per-cluster sweeps of the mid-size clusters run beside the warp-per-cluster sweeps of the small ones
  // (disjoint clusters, hence disjoint nodes): a handful of long-running CTAs next to thousands of short warps
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  ~ContactWork() {
    if (fork) cudaEventDestroy(fork);
    if (join) cudaEventDestroy(join);
    if (side) cudaStreamDestroy(side);
  }
};

// Once per substep, after detection: resets the chunk counters of the ordered sweeps.
int prepareContactSweeps(ContactWork& w, cudaStream_t s, const ContactLists& c);
// After reblock.cu: groups the entries by contact cluster for the in-warp sweeps.  Returns launches or -1.
int prepareClusterSweeps(ContactWork& w, cudaStream_t s, const ContactLists& c, const ClusterTables& t);
// Per PD iteration: collision projections (local step) and their RHS contributions.
int launchContactProject(cudaStream_t s, const ContactLists& c, const float4* q, float thickness, float4* contribC);
// nodes: the n nodes to assemble (null = 0 .. n-1)
int launchGatherRhsContacts(cudaStream_t s, uint32_t n, const uint32_t* nodes, const float4* msn, const int* incPtr,
                            const uint32_t* inc, const float4* contrib, const ContactLists& c, const float4* contribC,
                            const float4* q, float4* snap, float4* rhs);
// End of substep: ordered stabilisation sweeps (list order per node, see contact.cu) and the friction pass.
int launchStabilize(cudaStream_t s, ContactWork& w, const ContactLists& c, uint32_t n, float4* q, float4* prev,
                    const float4* snap, float thickness, uint32_t iterations);
int launchFriction(cudaStream_t s, ContactWork& w, const ContactLists& c, uint32_t n, const float4* q, float4* vel,
                   float friction, float staticThreshold);

}  // namespace pies
