// C ABI of libugnet.so: handle management, single-op entry points and the program executor.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include "engine.h"

namespace ug {

int set_error(ug_engine* h, int code, const char* fmt, ...) {
  if (h) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    h->last_error = buf;
  }
  return code;
}

int check_cuda(ug_engine* h, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return UG_OK;
  return set_error(h, UG_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

}  // namespace ug

using namespace ug;

struct PreparedOp {
  int kind;
  ConvLaunch conv;  // valid when kind == UG_OP_CONV
  StemLaunch stem;  // valid when kind == UG_OP_STEM
  ug_op op;         // descriptor copy for the other kinds
};

struct ug_program_s {
  std::vector<PreparedOp> ops;
};

static int run_simple(ug_engine* h, const ug_op* op, cudaStream_t s) {
  switch (op->kind) {
    case UG_OP_POOL: return launch_pool(h, &op->u.pool, s);
    case UG_OP_LAYERNORM: return launch_layernorm(h, &op->u.ln, s);
    case UG_OP_ATTN: return launch_attention(h, &op->u.attn, s);
    case UG_OP_CHANSTATS: return launch_chanstats(h, &op->u.stats, s);
    case UG_OP_GATE: return launch_gate(h, &op->u.gate, s);
    case UG_OP_BBOX: return launch_bbox(h, &op->u.bbox, s);
    case UG_OP_CROPRESIZE: return launch_cropresize(h, &op->u.crop, s);
    case UG_OP_HEAD: return launch_head(h, &op->u.head, s);
    case UG_OP_RESIZE: return launch_resize_u8(h, &op->u.resize, s);
    case UG_OP_WAVELET: return launch_wavelet(h, &op->u.wavelet, s);
    case UG_OP_S2D: return launch_s2d_pack(h, &op->u.s2d, s);
    case UG_OP_RESIZE_RAGGED: return launch_resize_ragged(h, &op->u.resize_ragged, s);
    case UG_OP_WAVELET_RAGGED: return launch_wavelet_ragged(h, &op->u.wavelet_ragged, s);
    case UG_OP_CAM: return launch_cam(h, &op->u.cam, s);
    case UG_OP_SOURCE_FRAME: return launch_source_frame(h, &op->u.source_frame, s);
    default: return set_error(h, UG_EINVAL, "unknown op kind %d", op->kind);
  }
}

static int run_prepared(ug_engine* h, const PreparedOp& po, cudaStream_t s) {
  if (po.kind == UG_OP_CONV) return conv_launch(h, &po.conv, s);
  if (po.kind == UG_OP_STEM) return stem_launch(h, &po.stem, s);
  return run_simple(h, &po.op, s);
}

extern "C" {

int ug_version(void) { return UG_VERSION; }

int ug_create(int device, ug_handle* out) {
  if (!out) return UG_EINVAL;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return UG_ECUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return UG_ECUDA;
  if (prop.major != 10) return UG_EUNSUPPORTED;  // sm_100a only: there is no fallback path
  ug_engine* h = new (std::nothrow) ug_engine();
  if (!h) return UG_ENOMEM;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  *out = h;
  return UG_OK;
}

int ug_destroy(ug_handle h) {
  if (h) {
    DeviceGuard guard(h);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (int i = 0; i < 2; ++i) {
      if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
      if (h->ev_free[i]) cudaEventDestroy(h->ev_free[i]);
    }
  }
  delete h;
  return UG_OK;
}

const char* ug_last_error(ug_handle h) { return h ? h->last_error.c_str() : "null handle"; }
long long ug_launch_count(ug_handle h) { return h ? h->launches : 0; }

int ug_conv(ug_handle h, const ug_conv_desc* d, void* stream) {
  if (!h || !d) return UG_EINVAL;
  DeviceGuard guard(h);
  ConvLaunch L;
  int rc = conv_prepare(h, d, &L);
  if (rc != UG_OK) return rc;
  return conv_launch(h, &L, static_cast<cudaStream_t>(stream));
}

int ug_stem(ug_handle h, const ug_stem_desc* d, void* stream) {
  if (!h || !d) return UG_EINVAL;
  DeviceGuard guard(h);
  StemLaunch L;
  int rc = stem_prepare(h, d, &L);
  if (rc != UG_OK) return rc;
  return stem_launch(h, &L, static_cast<cudaStream_t>(stream));
}

#define UG_SIMPLE_ENTRY(name, type, fn)                         \
  int name(ug_handle h, const type* d, void* stream) {          \
    if (!h || !d) return UG_EINVAL;                             \
    DeviceGuard guard(h);                                       \
    return fn(h, d, static_cast<cudaStream_t>(stream));         \
  }
UG_SIMPLE_ENTRY(ug_pool, ug_pool_desc, launch_pool)
UG_SIMPLE_ENTRY(ug_layernorm, ug_layernorm_desc, launch_layernorm)
UG_SIMPLE_ENTRY(ug_attention, ug_attn_desc, launch_attention)
UG_SIMPLE_ENTRY(ug_chanstats, ug_chanstats_desc, launch_chanstats)
UG_SIMPLE_ENTRY(ug_gate, ug_gate_desc, launch_gate)
UG_SIMPLE_ENTRY(ug_bbox, ug_bbox_desc, launch_bbox)
UG_SIMPLE_ENTRY(ug_cropresize, ug_cropresize_desc, launch_cropresize)
UG_SIMPLE_ENTRY(ug_head, ug_head_desc, launch_head)
UG_SIMPLE_ENTRY(ug_resize_u8, ug_resize_desc, launch_resize_u8)
UG_SIMPLE_ENTRY(ug_wavelet, ug_wavelet_desc, launch_wavelet)
UG_SIMPLE_ENTRY(ug_s2d_pack, ug_s2d_desc, launch_s2d_pack)
UG_SIMPLE_ENTRY(ug_resize_ragged, ug_resize_ragged_desc, launch_resize_ragged)
UG_SIMPLE_ENTRY(ug_wavelet_ragged, ug_wavelet_ragged_desc, launch_wavelet_ragged)
UG_SIMPLE_ENTRY(ug_cam, ug_cam_desc, launch_cam)
UG_SIMPLE_ENTRY(ug_source_frame, ug_source_frame_desc, launch_source_frame)

int ug_program_create(ug_handle h, const ug_op* ops, int n_ops, ug_program* out) {
  if (!h || !ops || n_ops <= 0 || !out) return UG_EINVAL;
  *out = nullptr;
  ug_program_s* p = new (std::nothrow) ug_program_s();
  if (!p) return UG_ENOMEM;
  p->ops.resize(n_ops);
  for (int i = 0; i < n_ops; ++i) {
    PreparedOp& po = p->ops[i];
    po.kind = ops[i].kind;
    po.op = ops[i];
    if (po.kind == UG_OP_CONV) {
      int rc = conv_prepare(h, &ops[i].u.conv, &po.conv);
      if (rc != UG_OK) {
        std::string msg = h->last_error;
        set_error(h, rc, "op %d: %s", i, msg.c_str());
        delete p;
        return rc;
      }
    } else if (po.kind == UG_OP_STEM) {
      int rc = stem_prepare(h, &ops[i].u.stem, &po.stem);
      if (rc != UG_OK) {
        std::string msg = h->last_error;
        set_error(h, rc, "op %d: %s", i, msg.c_str());
        delete p;
        return rc;
      }
    } else if (po.kind < UG_OP_CONV || po.kind > UG_OP_SOURCE_FRAME) {
      delete p;
      return set_error(h, UG_EINVAL, "op %d: unknown kind %d", i, po.kind);
    }
  }
  *out = p;
  return UG_OK;
}

int ug_program_run(ug_handle h, ug_program p, void* stream) {
  if (!h || !p) return UG_EINVAL;
  DeviceGuard guard(h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (size_t i = 0; i < p->ops.size(); ++i) {
    const PreparedOp& po = p->ops[i];
    int rc = run_prepared(h, po, s);
    if (rc != UG_OK) {
      std::string msg = h->last_error;
      return set_error(h, rc, "op %zu: %s", i, msg.c_str());
    }
  }
  return UG_OK;
}

int ug_program_run_timed(ug_handle h, ug_program p, void* stream, float* ms_per_op) {
  if (!h || !p || !ms_per_op) return UG_EINVAL;
  DeviceGuard guard(h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = p->ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev)
    if (cudaEventCreate(&e) != cudaSuccess) return set_error(h, UG_ECUDA, "cudaEventCreate failed");
  int rc = UG_OK;
  cudaEventRecord(ev[0], s);
  for (size_t i = 0; i < n && rc == UG_OK; ++i) {
    const PreparedOp& po = p->ops[i];
    rc = run_prepared(h, po, s);
    cudaEventRecord(ev[i + 1], s);
  }
  if (rc == UG_OK) rc = check_cuda(h, cudaStreamSynchronize(s), "stream synchronize");
  if (rc == UG_OK)
    for (size_t i = 0; i < n; ++i) cudaEventElapsedTime(&ms_per_op[i], ev[i], ev[i + 1]);
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

int ug_program_num_launches(ug_program p) { return p ? (int)p->ops.size() : 0; }

int ug_program_destroy(ug_handle h, ug_program p) {
  (void)h;
  delete p;
  return UG_OK;
}

int ug_program_run_host(ug_handle h, ug_program p, const ug_copy* h2d, int n_h2d, const ug_copy* d2h, int n_d2h,
                        void* stream) {
  if (!h || !p) return UG_EINVAL;
  DeviceGuard guard(h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int i = 0; i < n_h2d; ++i) {
    int rc = check_cuda(h, cudaMemcpyAsync(h2d[i].dst, h2d[i].src, h2d[i].bytes, cudaMemcpyHostToDevice, s), "H2D copy");
    if (rc != UG_OK) return rc;
  }
  int rc = ug_program_run(h, p, stream);
  if (rc != UG_OK) return rc;
  for (int i = 0; i < n_d2h; ++i) {
    rc = check_cuda(h, cudaMemcpyAsync(d2h[i].dst, d2h[i].src, d2h[i].bytes, cudaMemcpyDeviceToHost, s), "D2H copy");
    if (rc != UG_OK) return rc;
  }
  return check_cuda(h, cudaStreamSynchronize(s), "stream synchronize");
}

int ug_program_run_host_pipelined(ug_handle h, ug_program p, const ug_copy* h2d, void* const* stage0,
                                  void* const* stage1, int n_h2d, const ug_copy* d2h, int n_d2h, void* stream) {
  const bool direct = !stage0 && !stage1;  // see ugnet.h: the caller alternates two programs with their own inputs
  if (!h || !p || (n_h2d > 0 && (!h2d || (!direct && (!stage0 || !stage1))))) return UG_EINVAL;
  DeviceGuard guard(h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!h->copy_stream) {
    int rc = check_cuda(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking), "copy stream");
    for (int i = 0; i < 2 && rc == UG_OK; ++i) {
      rc = check_cuda(h, cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming), "event");
      if (rc == UG_OK) rc = check_cuda(h, cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming), "event");
    }
    if (rc != UG_OK) return rc;
  }
  const int slot = (int)(h->pipelined_steps & 1);
  void* const* stage = direct ? nullptr : (slot ? stage1 : stage0);
  // copy stream: wait until the step that last used this slot no longer reads it, then H2D into the slot
  if (h->pipelined_steps >= 2) cudaStreamWaitEvent(h->copy_stream, h->ev_free[slot], 0);
  for (int i = 0; i < n_h2d; ++i) {
    void* dst = direct ? h2d[i].dst : stage[i];
    int rc = check_cuda(h, cudaMemcpyAsync(dst, h2d[i].src, h2d[i].bytes, cudaMemcpyHostToDevice, h->copy_stream), "H2D copy");
    if (rc != UG_OK) return rc;
  }
  cudaEventRecord(h->ev_h2d[slot], h->copy_stream);
  cudaStreamWaitEvent(s, h->ev_h2d[slot], 0);
  if (!direct) {
    // compute stream: staging slot -> the program's input buffers (device to device); the slot is free after that
    for (int i = 0; i < n_h2d; ++i) {
      int rc = check_cuda(h, cudaMemcpyAsync(h2d[i].dst, stage[i], h2d[i].bytes, cudaMemcpyDeviceToDevice, s), "D2D copy");
      if (rc != UG_OK) return rc;
    }
    cudaEventRecord(h->ev_free[slot], s);
  }
  int rc = ug_program_run(h, p, stream);
  if (rc != UG_OK) return rc;
  if (direct) cudaEventRecord(h->ev_free[slot], s);  // the program reads its input buffers until its last kernels
  for (int i = 0; i < n_d2h; ++i) {
    rc = check_cuda(h, cudaMemcpyAsync(d2h[i].dst, d2h[i].src, d2h[i].bytes, cudaMemcpyDeviceToHost, s), "D2H copy");
    if (rc != UG_OK) return rc;
  }
  h->pipelined_steps++;
  return UG_OK;
}

}  // extern "C"
