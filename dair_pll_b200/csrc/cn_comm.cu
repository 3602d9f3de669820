// Peer-memory communicator of the data-parallel step (C ABI: include/dair_pll_b200.h, "data-parallel
// exchange").  The reference has no distributed code at all (SURVEY.md section 2); the sharded step needs ONE
// exchange -- the sum over ranks of the 15-double parameter gradient and the loss sum (section 8(e)) -- and this
// file sets up the buffers through which the reduction kernels perform it themselves (cn_comm.cuh).
#include <cuda_runtime.h>

#include <cstring>
#include <new>

#include "../../include/dair_pll_b200.h"
#include "cn_comm.cuh"
#include "cn_launch.cuh"

namespace {

struct Comm {
  int rank = 0, world = 1, device = 0;
  cn::CommBuf* local = nullptr;
  cn::CommBuf* peers[cn::COMM_MAX_WORLD] = {};
  bool opened[cn::COMM_MAX_WORLD] = {};
  cn::CommDev* dev = nullptr;
};

__global__ void comm_allreduce_kernel(cn::CommDev* C, double* buf, int n, double scale) {
  __shared__ double v[cn::COMM_MAX_ELEMS];
  if (threadIdx.x < n) v[threadIdx.x] = buf[threadIdx.x];
  cn::comm_allreduce_block(C, v, n);
  if (threadIdx.x < n) buf[threadIdx.x] = v[threadIdx.x] * scale;
}

}  // namespace

extern "C" {

size_t dpll_comm_handle_bytes(void) { return sizeof(cudaIpcMemHandle_t); }

int dpll_comm_create(int32_t rank, int32_t world, void** comm_out, void* handle_out) {
  if (!comm_out || !handle_out || world < 1 || world > cn::COMM_MAX_WORLD || rank < 0 || rank >= world) return DPLL_EINVAL;
  Comm* c = new (std::nothrow) Comm();
  if (!c) return DPLL_EINVAL;
  c->rank = rank; c->world = world;
  cudaError_t e = cudaGetDevice(&c->device);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->local), sizeof(cn::CommBuf));
  if (e == cudaSuccess) e = cudaMemset(c->local, 0, sizeof(cn::CommBuf));
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->dev), sizeof(cn::CommDev));
  if (e == cudaSuccess) e = cudaMemset(c->dev, 0, sizeof(cn::CommDev));
  cudaIpcMemHandle_t h;
  std::memset(&h, 0, sizeof(h));
  if (e == cudaSuccess && world > 1) e = cudaIpcGetMemHandle(&h, c->local);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    if (c->local) cudaFree(c->local);
    if (c->dev) cudaFree(c->dev);
    delete c;
    return (int)e;
  }
  std::memcpy(handle_out, &h, sizeof(h));
  *comm_out = c;
  return DPLL_OK;
}

int dpll_comm_connect(void* comm, const void* handles) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c || (!handles && c->world > 1)) return DPLL_EINVAL;
  cn::CommDev host;
  std::memset(&host, 0, sizeof(host));
  host.rank = c->rank; host.world = c->world;
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) { c->peers[r] = c->local; }
    else {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, static_cast<const char*>(handles) + (size_t)r * sizeof(h), sizeof(h));
      void* p = nullptr;
      cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) return (int)e;
      c->peers[r] = static_cast<cn::CommBuf*>(p);
      c->opened[r] = true;
    }
    host.peer[r] = c->peers[r];
  }
  cudaError_t e = cudaMemcpy(c->dev, &host, sizeof(host), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return e == cudaSuccess ? DPLL_OK : (int)e;
}

int dpll_comm_destroy(void* comm) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c) return DPLL_EINVAL;
  for (int r = 0; r < c->world; ++r)
    if (c->opened[r]) cudaIpcCloseMemHandle(c->peers[r]);
  if (c->local) cudaFree(c->local);
  if (c->dev) cudaFree(c->dev);
  delete c;
  return DPLL_OK;
}

void* dpll_comm_device_state(void* comm) { return comm ? static_cast<Comm*>(comm)->dev : nullptr; }

int dpll_comm_error(void* comm) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c) return DPLL_EINVAL;
  cn::CommDev host;
  cudaError_t e = cudaMemcpy(&host, c->dev, sizeof(host), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return (int)e;
  return host.error ? DPLL_ECOMM : DPLL_OK;
}

int dpll_comm_allreduce_f64(void* comm, double* buf, int32_t n, double scale, void* stream) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c || !buf || n < 0 || n > cn::COMM_MAX_ELEMS) return DPLL_EINVAL;
  if (n == 0) return DPLL_OK;
  comm_allreduce_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(c->dev, buf, n, scale);
  return cn::launch_status();
}

}  // extern "C"
