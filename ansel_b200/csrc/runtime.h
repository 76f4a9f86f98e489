// Internal runtime of libb200iop.so: error reporting, device binding, per-thread device scratch.
// Stands where the reference's OpenCL runtime does (src/common/opencl.c: dt_opencl_*), sized for
// one process driving 1..8 B200s.  Nothing here is visible through include/b200iop.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "../../include/b200iop.h"

namespace b200
{
// thread-local last-error text (b200_last_error)
void set_error(const char *fmt, ...);
int fail(int code, const char *fmt, ...);

#define B200_CUDA_TRY(expr)                                                                       \
  do                                                                                              \
  {                                                                                               \
    cudaError_t _e = (expr);                                                                      \
    if(_e != cudaSuccess)                                                                         \
      return ::b200::fail(B200_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,             \
                          cudaGetErrorString(_e));                                                \
  } while(0)

// Select the device a piece asks for (pipe->devid analogue); < 0 keeps the current device.
int bind_device(int devid);
int sm_count();

// Grow-only device scratch owned by the calling thread on the current device.  `slot` names an
// independent buffer (modules needing several temporaries use several slots).  Freed by
// b200_shutdown() or thread exit.  This is the shim's own device scratch, the counterpart of
// dt_opencl_alloc_device_buffer(); host-side tiling accounting never sees it (SURVEY 8b).
int scratch(int slot, size_t bytes, void **ptr);
enum
{
  SLOT_IN = 0,
  SLOT_OUT = 1,
  SLOT_TMP0 = 2,
  SLOT_TMP1 = 3,
  SLOT_TMP2 = 4,
  SLOT_TMP3 = 5,
  SLOT_SMALL = 6,
  SLOT_COUNT = 12
};

// Host <-> device transfer for the process() (host pointer) entry points.  Pinned or registered
// host memory goes straight over PCIe; pageable memory is staged through two pinned buffers so
// the copy into staging overlaps the DMA.
int copy_h2d(void *dst, const void *src, size_t bytes, cudaStream_t stream);
int copy_d2h(void *dst, const void *src, size_t bytes, cudaStream_t stream);

// per-thread non-blocking stream used by the *_process_host entry points
int host_stream(cudaStream_t *s);

// Launch timing of the headline kernels (b200_kernel_timing, b200_kernel_timing_read): when enabled, a pair of CUDA
// events brackets the launch on the stream it goes to.  One `if` per launch when disabled.
enum
{
  TIMED_NLM = 0,
  TIMED_RCD = 1,
  TIMED_COUNT = 2
};
bool timing_enabled();
// Records the start event of a new pair and returns its index (-1: not recorded); `generation` identifies the recording
// the pair belongs to, so an end mark after a b200_kernel_timing() clear records nothing.
int timing_start(int which, cudaStream_t stream, unsigned *generation);
void timing_end(int which, int index, unsigned generation, cudaStream_t stream);
struct timed_launch
{ // brackets the statement(s) between construction and destruction; the end goes into this launch's own pair, whatever
  // other threads time meanwhile
  int which, index;
  unsigned generation;
  cudaStream_t stream;
  timed_launch(int w, cudaStream_t s) : which(w), index(-1), generation(0), stream(s)
  {
    if(timing_enabled()) index = timing_start(which, stream, &generation);
  }
  ~timed_launch()
  {
    if(index >= 0) timing_end(which, index, generation, stream);
  }
};

// false before b200_init() and after b200_shutdown(): the CUDA context may be gone, per-thread state is not freed then
bool runtime_alive();

// Device copy of three tone curves (3 * B200_LUT_SAMPLES floats), cached per device by `identity` and `side`
// (0 = decoding / source, 1 = encoding / target); identity 0 = upload every time.  color.cu.
int device_curves(const float *const host[3], uint64_t identity, int side, cudaStream_t stream, const float **out);
} // namespace b200
