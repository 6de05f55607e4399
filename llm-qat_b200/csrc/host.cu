// host.cu — host-buffer entry points: the same fake-quant forward + STE
// backward, called with HOST pointers (pinned for full speed).  This is the
// end-to-end shape of the reference's call when tensors live on the CPU
// (SymQuantizer.apply / .backward, utils_quant.py:37-87): copy in, run, copy out.
//
// Rows are independent, so the tensor is cut into row chunks that flow through
// a three-stage pipeline — H2D(x, g) | K1/K2 + K3 | D2H(y, gx) — overlapping
// both PCIe directions with the kernels.  One stream per direction: measured on
// the B200 box, two concurrent copies in the SAME direction (x beside g) drop the
// link from 41 to 33 GB/s per direction.  The
// ceiling is the link itself: 47 GB/s per direction with both directions busy
// (tests/gpu_pcie_probe.py); this pipeline sustains 42 (profiles/r02_e2e_sweep.json: 7.75 ms per configs[1]
// step with both inputs copied ahead of the kernels at 8 MB, 7.50 ms with the split schedule at 16 MB).
// Everything is ordered
// after prior work on the caller's stream and the caller's stream waits for the
// last D2H, so stream semantics are those of a single asynchronous call.
#define QAT_PDL_FAMILY 9   // bit of QAT_B200_PDL_MASK (common.cuh)
#include <vector>

#include "common.cuh"

namespace qat {
namespace {

struct Pipe {
  cudaStream_t in = nullptr, out = nullptr;   // one stream per PCIe direction
  std::vector<cudaEvent_t> ev;
  int device = -1;
  cudaEvent_t event(size_t i) {
    while (ev.size() <= i) {
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
      ev.push_back(e);
    }
    return ev[i];
  }
};

// one pipe per host thread and device; streams/events are the only persistent
// resources the library creates (include/qat_b200.h "Ownership").
Pipe* get_pipe() {
  static thread_local std::vector<Pipe> pipes;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  for (auto& p : pipes)
    if (p.device == dev) return &p;
  Pipe p;
  p.device = dev;
  if (cudaStreamCreateWithFlags(&p.in, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
  if (cudaStreamCreateWithFlags(&p.out, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
  pipes.push_back(p);
  return &pipes.back();
}

constexpr int64_t kChunkBytes = 16ll << 20;   // per tensor per chunk

template <bool SYM>
int fwd_bwd_host(const void* x_host, const void* g_host, void* y_host, void* gx_host, float lo,
                 float hi, int64_t rows, int64_t cols, int dtype, int bits, void* scratch,
                 size_t scratch_bytes, void* stream) {
  QAT_CHECK_ARG(dtype == QAT_F32 || dtype == QAT_BF16, "dtype must be QAT_F32 or QAT_BF16 (got %d)", dtype);
  QAT_CHECK_ARG(rows >= 0 && cols >= 0, "negative shape");
  if (rows == 0 || cols == 0) return QAT_OK;
  QAT_CHECK_ARG(x_host != nullptr && y_host != nullptr, "x_host / y_host is NULL");
  const bool bwd = g_host != nullptr;
  QAT_CHECK_ARG(!bwd || gx_host != nullptr, "gx_host is NULL but g_host is given");
  const size_t need = qat_host_scratch_bytes(rows, cols, dtype, bwd ? 1 : 0);
  if (scratch == nullptr || scratch_bytes < need) {
    set_error("host entry point needs %zu bytes of device scratch (got %zu)", need, scratch_bytes);
    return QAT_ERR_WORKSPACE;
  }
  if (qat_fwd_workspace_bytes(rows, cols, dtype) != 0) {
    set_error("host entry points handle register-resident rows only (cols=%lld too long)", (long long)cols);
    return QAT_ERR_UNSUPPORTED;
  }
  Pipe* pipe = get_pipe();
  if (pipe == nullptr) return cuda_fail(cudaGetLastError(), "creating pipeline streams");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);

  const int64_t esz = dtype == QAT_F32 ? 4 : 2;
  const int64_t row_bytes = cols * esz;
  // device rows start 16-byte aligned so the vector path is taken whenever the
  // row pitch allows; tensors are laid out back to back, each 256-byte aligned.
  const int64_t tensor_bytes = ((rows * row_bytes + 255) / 256) * 256;
  char* dx = reinterpret_cast<char*>(scratch);
  char* dy = dx + tensor_bytes;
  char* dg = dy + tensor_bytes;
  char* dgx = dg + tensor_bytes;

  // Chunk schedule: steady-state chunks of ~16 MB per tensor (smaller ones are
  // bound by the host's enqueue rate), but the first and last chunks ramp
  // 1/8, 1/4, 1/2 of that: the D2H direction idles while the first chunk goes
  // in, and the H2D direction while the last one comes out, so short end
  // chunks cut those two bubbles from ~0.3 ms to ~0.04 ms per call.
  int64_t chunk_rows = kChunkBytes / (row_bytes > 0 ? row_bytes : 1);
  if (chunk_rows < 1) chunk_rows = 1;
  // keep chunk starts 16-byte aligned for any row pitch
  int64_t align_rows = 1;
  while ((align_rows * row_bytes) % 16 != 0) ++align_rows;
  auto round_rows = [&](int64_t r) { return ((r < 1 ? 1 : r) + align_rows - 1) / align_rows * align_rows; };
  chunk_rows = round_rows(chunk_rows);
  std::vector<int64_t> bounds;  // chunk c covers rows [bounds[c], bounds[c+1])
  {
    const int64_t ramp[3] = {round_rows(chunk_rows / 8), round_rows(chunk_rows / 4), round_rows(chunk_rows / 2)};
    const int64_t ramp_total = ramp[0] + ramp[1] + ramp[2];
    bounds.push_back(0);
    if (rows >= 2 * ramp_total + chunk_rows) {
      int64_t r = 0;
      for (int i = 0; i < 3; ++i) bounds.push_back(r += ramp[i]);
      const int64_t steady_end = rows - ramp_total;
      while (steady_end - r > chunk_rows + chunk_rows / 2) bounds.push_back(r += chunk_rows);
      if (steady_end > r) bounds.push_back(r = steady_end);
      for (int i = 2; i >= 1; --i) bounds.push_back(r += ramp[i]);
      bounds.push_back(rows);
    } else {
      for (int64_t r = chunk_rows; r < rows; r += chunk_rows) bounds.push_back(r);
      bounds.push_back(rows);
    }
  }
  const int64_t nchunks = (int64_t)bounds.size() - 1;

  cudaError_t e;
#define QAT_TRY(call)                                  \
  do {                                                 \
    e = (call);                                        \
    if (e != cudaSuccess) return cuda_fail(e, #call);  \
  } while (0)

  cudaEvent_t ev_start = pipe->event(0);
  if (ev_start == nullptr) return cuda_fail(cudaGetLastError(), "cudaEventCreate");
  QAT_TRY(cudaEventRecord(ev_start, st));
  QAT_TRY(cudaStreamWaitEvent(pipe->in, ev_start, 0));
  QAT_TRY(cudaStreamWaitEvent(pipe->out, ev_start, 0));

  // Within a chunk the forward needs x only: x goes in, K1/K2 runs and y starts its way back while g is still
  // going in; then K3 and gx.  The outbound direction so trails the inbound one by HALF a chunk (one tensor's
  // slice), which lets the copies be twice as long for the same pipeline granularity.
  cudaStream_t s_in = pipe->in, s_out = pipe->out;
  const char* src[2] = {reinterpret_cast<const char*>(x_host), reinterpret_cast<const char*>(g_host)};
  char* dst_dev[2] = {dx, dg};
  const char* src_dev[2] = {dy, dgx};
  char* dst[2] = {reinterpret_cast<char*>(y_host), reinterpret_cast<char*>(gx_host)};
  for (int64_t c = 0; c < nchunks; ++c) {
    const int64_t r0 = bounds[c];
    const int64_t nr = bounds[c + 1] - r0;
    const int64_t off = r0 * row_bytes, bytes = nr * row_bytes;
    cudaEvent_t ev_in[2] = {pipe->event(1 + 4 * c), pipe->event(2 + 4 * c)};
    cudaEvent_t ev_k[2] = {pipe->event(3 + 4 * c), pipe->event(4 + 4 * c)};
    if (ev_in[0] == nullptr || ev_in[1] == nullptr || ev_k[0] == nullptr || ev_k[1] == nullptr)
      return cuda_fail(cudaGetLastError(), "cudaEventCreate");
    auto copy_in = [&](int l) -> cudaError_t {
      cudaError_t ce = cudaMemcpyAsync(dst_dev[l] + off, src[l] + off, bytes, cudaMemcpyHostToDevice, s_in);
      if (ce == cudaSuccess) ce = cudaEventRecord(ev_in[l], s_in);
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(st, ev_in[l], 0);
      return ce;
    };
    auto copy_out = [&](int l) -> cudaError_t {   // after the kernel(s) enqueued on st so far
      cudaError_t ce = cudaEventRecord(ev_k[l], st);
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s_out, ev_k[l], 0);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(dst[l] + off, src_dev[l] + off, bytes, cudaMemcpyDeviceToHost, s_out);
      return ce;
    };
    auto forward = [&]() -> int {
      return SYM ? qat_sym_fwd(dx + off, dy + off, nullptr, QAT_CODES_NONE, nullptr, nullptr, nullptr, lo, hi, nr, cols,
                               dtype, bits, nullptr, 0, st)
                 : qat_asym_fwd(dx + off, dy + off, nullptr, QAT_CODES_NONE, nullptr, nullptr, nullptr, lo, hi, nr, cols,
                                dtype, bits, nullptr, 0, st);
    };
    int rc;
    QAT_TRY(copy_in(0));
    if ((rc = forward()) != QAT_OK) return rc;
    QAT_TRY(copy_out(0));
    if (bwd) {
      QAT_TRY(copy_in(1));
      if ((rc = qat_ste_bwd(dg + off, dx + off, dgx + off, nullptr, lo, hi, nr * cols, dtype, st)) != QAT_OK) return rc;
      QAT_TRY(copy_out(1));
    }
  }
  {
    cudaEvent_t ev_done = pipe->event(1 + 4 * nchunks);
    if (ev_done == nullptr) return cuda_fail(cudaGetLastError(), "cudaEventCreate");
    QAT_TRY(cudaEventRecord(ev_done, s_out));
    QAT_TRY(cudaStreamWaitEvent(st, ev_done, 0));
  }
#undef QAT_TRY
  return QAT_OK;
}

}  // namespace
}  // namespace qat

extern "C" {

size_t qat_host_scratch_bytes(int64_t rows, int64_t cols, int dtype, int with_backward) {
  if (rows <= 0 || cols <= 0) return 0;
  const int64_t esz = dtype == QAT_F32 ? 4 : 2;
  const int64_t tensor_bytes = ((rows * cols * esz + 255) / 256) * 256;
  return (size_t)tensor_bytes * (with_backward ? 4 : 2);
}

int qat_sym_fwd_bwd_host(const void* x_host, const void* g_host, void* y_host, void* gx_host,
                         float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                         int bits, void* dev_scratch, size_t dev_scratch_bytes, void* stream) {
  return qat::fwd_bwd_host<true>(x_host, g_host, y_host, gx_host, clip_lo, clip_hi, rows, cols,
                                 dtype, bits, dev_scratch, dev_scratch_bytes, stream);
}

int qat_asym_fwd_bwd_host(const void* x_host, const void* g_host, void* y_host, void* gx_host,
                          float clip_lo, float clip_hi, int64_t rows, int64_t cols, int dtype,
                          int bits, void* dev_scratch, size_t dev_scratch_bytes, void* stream) {
  return qat::fwd_bwd_host<false>(x_host, g_host, y_host, gx_host, clip_lo, clip_hi, rows, cols,
                                  dtype, bits, dev_scratch, dev_scratch_bytes, stream);
}

}  // extern "C"
