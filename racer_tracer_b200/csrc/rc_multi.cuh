// rc_multi.cuh — exchange step of a multi-device render inside one process
// (the reference is a single process; SURVEY §8(e)).
//
//   tile split    every device traces a disjoint set of interleaved tiles.  With peer
//                 access in both directions the megakernel of device k stores its
//                 pixels STRAIGHT INTO device 0's accumulation buffer over NVLink as
//                 each tile finishes (compute and gather in one kernel; device 0 only
//                 waits on an event).  Without it every device fills its own
//                 zero-initialised buffer and device 0 pulls them out of peer memory
//                 (or a staging copy) and adds them.
//   sample split  every device holds a partial sum of ALL pixels; the buffers
//                 are summed onto device 0 with ncclReduce (NCCL is loaded
//                 lazily with dlopen so a 1-GPU host needs no NCCL at all).
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <string>
#include <vector>

#define RC_MULTI_MAX_DEV 16

struct PeerList {
    const float* src[RC_MULTI_MAX_DEV];
    int n;
};

// dst[i] += sum_k src_k[i]; src_k are peer-mapped device pointers
__global__ void peer_gather_add_kernel(float* __restrict__ dst, PeerList peers, size_t n4) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 acc = d4[i];
        for (int k = 0; k < peers.n; ++k) {
            float4 v = reinterpret_cast<const float4*>(peers.src[k])[i];
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        d4[i] = acc;
    }
}

__global__ void tail_add_kernel(float* __restrict__ dst, PeerList peers, size_t begin, size_t n) {
    size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float acc = dst[i];
    for (int k = 0; k < peers.n; ++k) acc += peers.src[k][i];
    dst[i] = acc;
}

typedef void* nccl_comm_t;
struct NcclApi {
    void* lib = nullptr;
    int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};

struct MultiState {
    size_t n_dev = 0;
    bool peer_ok = false;               // device 0 can read every other device's memory
    bool peer_write_ok = false;         // every other device can write device 0's memory
    std::vector<cudaEvent_t> done;      // per device: tracing finished
    float* staging = nullptr;           // device 0, used when peer access is unavailable
    size_t staging_n = 0;
    NcclApi nccl;
    std::vector<nccl_comm_t> comms;
    std::string err;
};

inline const char* multi_error(const MultiState& m) { return m.err.c_str(); }

template <class DevOf>
int multi_init(MultiState& m, size_t n_dev, DevOf device_of) {
    m.n_dev = n_dev;
    if (n_dev <= 1) return 0;
    if (n_dev > RC_MULTI_MAX_DEV) return -1;
    m.peer_ok = true;
    for (size_t k = 1; k < n_dev; ++k) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, device_of(0), device_of(k)) != cudaSuccess || !can) { m.peer_ok = false; continue; }
        cudaSetDevice(device_of(0));
        cudaError_t e = cudaDeviceEnablePeerAccess(device_of(k), 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        if (e != cudaSuccess) { cudaGetLastError(); m.peer_ok = false; }
    }
    m.peer_write_ok = m.peer_ok;
    for (size_t k = 1; k < n_dev && m.peer_write_ok; ++k) {
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, device_of(k), device_of(0)) != cudaSuccess || !can) { m.peer_write_ok = false; break; }
        cudaSetDevice(device_of(k));
        cudaError_t e = cudaDeviceEnablePeerAccess(device_of(0), 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        if (e != cudaSuccess) { cudaGetLastError(); m.peer_write_ok = false; }
    }
    m.done.resize(n_dev);
    for (size_t k = 0; k < n_dev; ++k) {
        cudaSetDevice(device_of(k));
        if (cudaEventCreateWithFlags(&m.done[k], cudaEventDisableTiming) != cudaSuccess) return -3;
    }
    return 0;
}

inline void multi_destroy(MultiState& m) {
    for (auto c : m.comms) if (c && m.nccl.CommDestroy) m.nccl.CommDestroy(c);
    m.comms.clear();
    for (auto e : m.done) if (e) cudaEventDestroy(e);
    m.done.clear();
    if (m.staging) cudaFree(m.staging);
    m.staging = nullptr;
    if (m.nccl.lib) dlclose(m.nccl.lib);
    m.nccl.lib = nullptr;
}

template <class DevOf>
int multi_nccl_init(MultiState& m, DevOf device_of) {
    if (!m.comms.empty()) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        m.nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (m.nccl.lib) break;
    }
    if (!m.nccl.lib) { m.err = "libnccl.so.2 not found (needed for the sample-split reduce)"; return -6; }
#define RC_SYM(field, name)                                                       \
    *(void**)(&m.nccl.field) = dlsym(m.nccl.lib, name);                           \
    if (!m.nccl.field) { m.err = std::string("NCCL symbol missing: ") + name; return -6; }
    RC_SYM(CommInitAll, "ncclCommInitAll");
    RC_SYM(CommDestroy, "ncclCommDestroy");
    RC_SYM(Reduce, "ncclReduce");
    RC_SYM(GroupStart, "ncclGroupStart");
    RC_SYM(GroupEnd, "ncclGroupEnd");
    RC_SYM(GetErrorString, "ncclGetErrorString");
#undef RC_SYM
    std::vector<int> devs(m.n_dev);
    for (size_t k = 0; k < m.n_dev; ++k) devs[k] = device_of(k);
    m.comms.assign(m.n_dev, nullptr);
    int rc = m.nccl.CommInitAll(m.comms.data(), (int)m.n_dev, devs.data());
    if (rc != 0) { m.err = std::string("ncclCommInitAll: ") + m.nccl.GetErrorString(rc); m.comms.clear(); return -6; }
    return 0;
}

// Device 0's stream waits for the other devices' (all a direct tile split needs: they stored into its buffer themselves).
template <class StreamOf, class DevOf>
int multi_join(MultiState& m, StreamOf stream_of, DevOf device_of) {
    for (size_t k = 1; k < m.n_dev; ++k) {
        cudaSetDevice(device_of(k));
        if (cudaEventRecord(m.done[k], stream_of(k)) != cudaSuccess) { m.err = "event record failed"; return -3; }
    }
    cudaSetDevice(device_of(0));
    for (size_t k = 1; k < m.n_dev; ++k)
        if (cudaStreamWaitEvent(stream_of(0), m.done[k], 0) != cudaSuccess) { m.err = "stream wait failed"; return -3; }
    return 0;
}

// Sum (sample split) or gather (tile split) every device's buffer onto dst0.
template <class AccumOf, class StreamOf, class DevOf>
int multi_gather(MultiState& m, int split, size_t n, float* dst0, AccumOf accum_of, StreamOf stream_of, DevOf device_of) {
    if (m.n_dev <= 1) return 0;
    if (split == 1 /* RC_SPLIT_SAMPLES */) {
        int rc = multi_nccl_init(m, device_of);
        if (rc != 0) return rc;
        const int ncclFloat32 = 7, ncclSum = 0;
        rc = m.nccl.GroupStart();
        for (size_t k = 0; rc == 0 && k < m.n_dev; ++k) {
            cudaSetDevice(device_of(k));
            const float* send = k == 0 ? dst0 : accum_of(k);
            rc = m.nccl.Reduce(send, dst0, n, ncclFloat32, ncclSum, 0, m.comms[k], stream_of(k));
        }
        int rc2 = m.nccl.GroupEnd();
        if (rc == 0) rc = rc2;
        if (rc != 0) { m.err = std::string("ncclReduce: ") + m.nccl.GetErrorString(rc); return -6; }
        // device 0's stream now carries the reduced buffer; later work is enqueued on it
        cudaSetDevice(device_of(0));
        return 0;
    }
    // tile split: device 0 waits for the others, then pulls their buffers
    int rc = multi_join(m, stream_of, device_of);
    if (rc != 0) return rc;
    PeerList pl;
    pl.n = 0;
    if (m.peer_ok) {
        for (size_t k = 1; k < m.n_dev; ++k) pl.src[pl.n++] = accum_of(k);
    } else {
        // no peer mapping: stage each buffer on device 0 with cudaMemcpyPeerAsync
        if (m.staging_n < n * (m.n_dev - 1)) {
            if (m.staging) cudaFree(m.staging);
            if (cudaMalloc(&m.staging, n * (m.n_dev - 1) * sizeof(float)) != cudaSuccess) { m.err = "staging alloc failed"; return -3; }
            m.staging_n = n * (m.n_dev - 1);
        }
        for (size_t k = 1; k < m.n_dev; ++k) {
            float* dst = m.staging + (k - 1) * n;
            if (cudaMemcpyPeerAsync(dst, device_of(0), accum_of(k), device_of(k), n * sizeof(float), stream_of(0)) != cudaSuccess) {
                m.err = "cudaMemcpyPeerAsync failed";
                return -3;
            }
            pl.src[pl.n++] = dst;
        }
    }
    size_t n4 = n / 4;
    if (n4 > 0) peer_gather_add_kernel<<<148 * 4, 256, 0, stream_of(0)>>>(dst0, pl, n4);
    if (n4 * 4 < n) tail_add_kernel<<<1, 32, 0, stream_of(0)>>>(dst0, pl, n4 * 4, n);
    if (cudaGetLastError() != cudaSuccess) { m.err = "gather kernel launch failed"; return -3; }
    return 0;
}
