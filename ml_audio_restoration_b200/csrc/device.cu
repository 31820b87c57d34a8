// Per-device host state shared by the launchers: SM count and one-time kernel attributes.
// Function attributes (cudaFuncSetAttribute) and the SM count belong to a device / context, not to the process: one
// process may drive several GPUs (RestorationPipeline(device="cuda:1") next to "cuda:0"), so every "done once" flag here
// is kept per device.
#include <atomic>

#include "ar_common.cuh"

namespace ar {

int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev < 0 ? 0 : dev;
}

bool DeviceOnce::pending() const {
  const int dev = current_device();
  return dev >= MAX_DEVICES || !(bits.load(std::memory_order_acquire) >> dev & 1ull);
}
void DeviceOnce::done() {
  const int dev = current_device();
  if (dev < MAX_DEVICES) bits.fetch_or(1ull << dev, std::memory_order_release);
}

int sm_count() {
  static std::atomic<int> n[DeviceOnce::MAX_DEVICES];   // zero-initialised
  const int dev = current_device();
  int v = dev < DeviceOnce::MAX_DEVICES ? n[dev].load(std::memory_order_relaxed) : 0;
  if (v == 0) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (v <= 0) v = 148;
    if (dev < DeviceOnce::MAX_DEVICES) n[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

}  // namespace ar
