// Development hooks (libugnet_dev.so only; declared in include/ugnet_dev.h): the launch-plan queries of the conv and
// memory-bound ops.  Not part of the product library.
#include <algorithm>
#include <cstring>
#include <vector>
#include "engine.h"
#include "../../include/ugnet_dev.h"

using namespace ug;

extern "C" {

int ug_conv_instances(int kernel, ug_conv_instance_t* out, int cap) {
  std::vector<ug_conv_instance_t> rows;
  switch (kernel) {
    case UG_CONV_KERNEL_ONETILE:
    case UG_CONV_KERNEL_PERSISTENT:
      for (int act : {UG_ACT_NONE, UG_ACT_RELU, UG_ACT_GELU}) rows.push_back({act, -1, -1, -1, -1, -1});
      break;
    case UG_CONV_KERNEL_MULTI:
    case UG_CONV_KERNEL_MULTI_PAIR: {
      // every row of the multi table, so that ug_conv_launch_info's `instance` indexes it; rows of the other kind are
      // told apart by `pair`
#define UG_MULTI_ROW(A, T, M, K, RT, P) rows.push_back({A, T, M, K, RT, P});
      UG_MULTI_INSTANCES(UG_MULTI_ROW)
#undef UG_MULTI_ROW
      break;
    }
    case UG_CONV_KERNEL_PAIR:
#define UG_PAIR_ROW(M, RT) rows.push_back({UG_ACT_RELU, 9, M, -1, RT, 1});
      UG_PAIR_INSTANCES(UG_PAIR_ROW)
#undef UG_PAIR_ROW
      break;
    default: return UG_EINVAL;
  }
  for (int i = 0; out && i < (int)rows.size() && i < cap; ++i) out[i] = rows[i];
  return (int)rows.size();
}

int ug_conv_launch_info(ug_handle h, const ug_conv_desc* d, ug_conv_launch_info_t* out) {
  if (!h || !d || !out) return UG_EINVAL;
  DeviceGuard guard(h);
  ConvLaunch L;
  const int rc = conv_prepare(h, d, &L);
  if (rc != UG_OK) return rc;
  ug_conv_launch_info_t& o = *out;
  memset(&o, 0, sizeof(o));
  o.kernel = (int)L.kernel;
  o.instance = L.instance;
  std::vector<ug_conv_instance_t> rows(64);
  const int n = ug_conv_instances(o.kernel, rows.data(), (int)rows.size());
  if (L.instance < 0 || L.instance >= n) return set_error(h, UG_EINVAL, "conv_launch_info: instance %d out of range", L.instance);
  o.inst = rows[L.instance];
  const ConvKParams& p = L.p;
  const bool multi = L.kernel == ConvKernel::Multi || L.kernel == ConvKernel::MultiPair;
  const bool pair_grid = L.kernel == ConvKernel::MultiPair || L.kernel == ConvKernel::Pair;
  o.BN = p.BN; o.n_tiles = p.n_tiles; o.TW = p.TW; o.TH = p.TH; o.TN = p.TN;
  o.kchunks = p.kchunks;
  o.sa = p.stages; o.obufs = p.obufs; o.acc_stages = p.acc_stages;
  o.pool = p.pool; o.stats = p.stats_sum != nullptr; o.split = p.n_split != 0; o.up = p.up;
  if (multi) {
    o.strip = L.mp.strip; o.rowtaps = L.mp.rowtaps != 0; o.row_halo = L.mp.rowtaps == 2;
    o.b_resident = L.mp.b_resident; o.sb = L.mp.sb;
  }
  if (L.kernel == ConvKernel::Pair) {
    o.streams = L.pp.streams; o.n_quads = L.pp.n_quads;
  }
  o.block = (int)L.block;
  // the pair kernels launch on at most the co-resident cluster count (launch_pairs)
  o.grid = pair_grid ? (int)std::min(L.grid.x, 2u * (unsigned)max_cluster_pairs(h)) : (int)(L.grid.x * L.grid.y);
  o.smem = (long long)L.smem;
  o.m_tiles = p.m_tiles;
  o.item_tiles = L.item_tiles;
  o.units = pair_grid ? o.grid / 2 : o.grid;
  if (multi) o.items = (long long)L.mp.m_super * p.n_tiles;
  else if (L.kernel == ConvKernel::Pair) o.items = L.pp.n_quads;
  else o.items = (long long)p.m_tiles * p.n_tiles;
  o.rounds = (int)((o.items + o.units - 1) / o.units);
  o.last_round_items = o.items - (long long)(o.rounds - 1) * o.units;
  o.tiles_past_end = (o.items / p.n_tiles) * L.item_tiles - p.m_tiles;
  if (L.kernel == ConvKernel::OneTile || L.kernel == ConvKernel::Persistent) o.tiles_past_end = 0;
  return UG_OK;
}

static_assert((int)MemKernel::Pool == UG_MEMOP_KERNEL_POOL && (int)MemKernel::LayerNorm == UG_MEMOP_KERNEL_LAYERNORM &&
                  (int)MemKernel::CropResize == UG_MEMOP_KERNEL_CROPRESIZE && (int)MemKernel::Head == UG_MEMOP_KERNEL_HEAD,
              "MemKernel and UG_MEMOP_KERNEL_* must list the kernels in the same order");

int ug_memop_launch_info(ug_handle h, const ug_op* op, ug_memop_launch_info_t* out) {
  if (!h || !op || !out) return UG_EINVAL;
  DeviceGuard guard(h);
  ug_memop_launch_info_t& o = *out;
  memset(&o, 0, sizeof(o));
  o.launches = 1;
  if (op->kind == UG_OP_STEM) {
    StemLaunch L;
    const int rc = stem_prepare(h, &op->u.stem, &L);
    if (rc != UG_OK) return rc;
    o.kernel = UG_MEMOP_KERNEL_STEM;
    o.variant = -1;
    o.grid_x = (int)L.grid;
    o.grid_y = 1;
    o.block = (int)L.block;
    o.smem = (long long)L.smem;
    return UG_OK;
  }
  MemLaunch L;
  int rc;
  switch (op->kind) {
    case UG_OP_POOL: rc = plan_pool(h, &op->u.pool, &L); break;
    case UG_OP_LAYERNORM: rc = plan_layernorm(h, &op->u.ln, &L); break;
    case UG_OP_ATTN: rc = plan_attention(h, &op->u.attn, &L); break;
    case UG_OP_CHANSTATS: rc = plan_chanstats(h, &op->u.stats, &L); break;
    case UG_OP_GATE: rc = plan_gate(h, &op->u.gate, &L); break;
    case UG_OP_BBOX: rc = plan_bbox(h, &op->u.bbox, &L); break;
    case UG_OP_CROPRESIZE: rc = plan_cropresize(h, &op->u.crop, &L); break;
    case UG_OP_HEAD: rc = plan_head(h, &op->u.head, &L); break;
    case UG_OP_S2D: rc = plan_s2d_pack(h, &op->u.s2d, &L); break;
    default: return set_error(h, UG_EINVAL, "memop_launch_info: op kind %d is not a memory-bound op", op->kind);
  }
  if (rc != UG_OK) return rc;
  o.kernel = (int)L.kernel;
  o.variant = L.variant;
  o.grid_x = (int)L.grid.x;
  o.grid_y = (int)L.grid.y;
  o.block = (int)L.block;
  o.smem = (long long)L.smem;
  if (L.kernel == MemKernel::Gate) o.launches = 2;
  return UG_OK;
}

}  // extern "C"
