// Sample-sharded mode (SURVEY 8e, secondary partitioning): every rank holds a slice of the histogram rows and
// ALL node problems; per objective/gradient pass the partial sums are combined with one NCCL all-reduce of the
// int64 gradient accumulators (exact, order-independent) and one of the fp64 objective sums, over NVLink.
// NCCL is resolved at run time (dlopen of the libnccl.so.2 already loaded by torch, or the system one), so
// libgml_b200.so carries no link-time dependency on it.
#include <dlfcn.h>

#include <cstring>

#include "common.cuh"

// The handful of NCCL declarations this file needs, restated so that the library builds without NCCL headers (NCCL is
// a run-time dependency of the multi-GPU modes only; values as in nccl.h 2.x, whose ABI has kept them stable).
extern "C" {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;
typedef enum { ncclInt64 = 4, ncclFloat64 = 8 } ncclDataType_t;
typedef enum { ncclSum = 0, ncclMax = 2 } ncclRedOp_t;
}

namespace gml {

struct Comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
};

namespace {

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
};

NcclApi& api() {
    static NcclApi a;
    if (a.lib) return a;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        a.lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD);      // the copy torch already mapped, if any
        if (a.lib) break;
    }
    for (const char* n : names) {
        if (a.lib) break;
        a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    }
    GML_REQUIRE(a.lib != nullptr, "sample-sharded mode needs NCCL (libnccl.so.2 not found)");
    a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(a.lib, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(a.lib, "ncclCommInitRank"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(a.lib, "ncclCommDestroy"));
    a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(dlsym(a.lib, "ncclAllReduce"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(a.lib, "ncclGetErrorString"));
    a.GroupStart = reinterpret_cast<decltype(a.GroupStart)>(dlsym(a.lib, "ncclGroupStart"));
    a.GroupEnd = reinterpret_cast<decltype(a.GroupEnd)>(dlsym(a.lib, "ncclGroupEnd"));
    GML_REQUIRE(a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllReduce && a.GroupStart && a.GroupEnd, "incomplete NCCL library");
    return a;
}

void nccl_check(ncclResult_t rc, const char* what) {
    if (rc == ncclSuccess) return;
    const char* msg = api().GetErrorString ? api().GetErrorString(rc) : "?";
    set_error(std::string(what) + " failed: " + msg);
    throw CudaError{GML_B200_ECUDA};
}

__global__ void rescale_weights_kernel(double* w64, float* w32, int64_t n, double factor) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double w = w64[k] * factor;
    w64[k] = w; w32[k] = (float)w;
}

}  // namespace

void comm_unique_id(uint8_t* out128) {
    ncclUniqueId id;
    nccl_check(api().GetUniqueId(&id), "ncclGetUniqueId");
    static_assert(sizeof(id) == 128, "unexpected ncclUniqueId size");
    memcpy(out128, &id, 128);
}

Comm* comm_create(const uint8_t* id128, int rank, int world) {
    GML_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank / world size");
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    Comm* c = new Comm();
    c->rank = rank; c->world = world;
    nccl_check(api().CommInitRank(&c->comm, world, id, rank), "ncclCommInitRank");
    return c;
}

void comm_destroy(Comm* c) {
    if (!c) return;
    if (c->comm) api().CommDestroy(c->comm);
    delete c;
}

// several collectives issued between start / end go out as ONE NCCL launch
void comm_group_start(Comm* c) { if (c && c->world > 1) nccl_check(api().GroupStart(), "ncclGroupStart"); }
void comm_group_end(Comm* c) { if (c && c->world > 1) nccl_check(api().GroupEnd(), "ncclGroupEnd"); }

void comm_allreduce_sum_i64(Comm* c, long long* buf, size_t n, cudaStream_t st) {
    if (!c || c->world == 1) return;
    nccl_check(api().AllReduce(buf, buf, n, ncclInt64, ncclSum, c->comm, st), "ncclAllReduce(int64)");
}
void comm_allreduce_sum_f64(Comm* c, double* buf, size_t n, cudaStream_t st) {
    if (!c || c->world == 1) return;
    nccl_check(api().AllReduce(buf, buf, n, ncclFloat64, ncclSum, c->comm, st), "ncclAllReduce(f64 sum)");
}
void comm_allreduce_max_f64(Comm* c, double* buf, size_t n, cudaStream_t st) {
    if (!c || c->world == 1) return;
    nccl_check(api().AllReduce(buf, buf, n, ncclFloat64, ncclMax, c->comm, st), "ncclAllReduce(f64 max)");
}

// max over the ranks of a small non-negative status code: lets every rank leave together when one of them failed
// before a collective phase (a rank that skipped the phase would leave the others waiting for ever)
int comm_agree_max(Comm* c, int value, cudaStream_t st) {
    if (!c || c->world == 1) return value;
    DevBuf<double> d;
    d.alloc(1);
    const double v = (double)value;
    double out = v;
    GML_CUDA(cudaMemcpyAsync(d.p, &v, sizeof(double), cudaMemcpyHostToDevice, st));
    comm_allreduce_max_f64(c, d.p, 1, st);
    GML_CUDA(cudaMemcpyAsync(&out, d.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    return (int)out;
}

// Make the weights of a locally normalised histogram slice global: w = c / M_global, wmax = max over ranks.
void comm_globalize_histogram(Comm* c, Histogram& h, cudaStream_t st) {
    if (!c || c->world == 1) { h.M_local = h.M; h.K_total = (double)h.K; return; }
    // idempotent: a second call on the same upload starts again from the rank's own mass (the weights currently hold
    // c / M_global, i.e. they are rescaled by M_global_old / M_global_new = 1)
    const double own_mass = h.M_local > 0.0 ? h.M_local : h.M;
    const double w_norm = h.M;                                   // what the resident weights are normalised by
    DevBuf<double> s;
    s.alloc(3);
    const double local[3] = {own_mass, (double)h.K, h.wmax * w_norm};   // sum of counts, rows, max count
    GML_CUDA(cudaMemcpyAsync(s.p, local, sizeof(local), cudaMemcpyHostToDevice, st));
    comm_allreduce_sum_f64(c, s.p, 2, st);
    comm_allreduce_max_f64(c, s.p + 2, 1, st);
    double glob[3];
    GML_CUDA(cudaMemcpyAsync(glob, s.p, sizeof(glob), cudaMemcpyDeviceToHost, st));
    GML_CUDA(cudaStreamSynchronize(st));
    rescale_weights_kernel<<<(unsigned)ceil_div(h.Kp, 256), 256, 0, st>>>(h.w64.p, h.w32.p, h.Kp, w_norm / glob[0]);
    GML_LAUNCHED();
    h.M_local = own_mass;
    h.M = glob[0];
    h.K_total = glob[1];
    h.wmax = glob[2] / glob[0];
}

}  // namespace gml
