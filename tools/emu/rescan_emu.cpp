// rescan_emu.cpp — the rescan diff (csrc/kvg_rescan.cuh: k_rescan_merge<RsPci|RsMdev>, k_rescan_keys), compiled
// for the CPU from its real source on top of warp_emu.h.  The launch sequence is the one of rescan_diff
// (csrc/api/kvg_api_rescan.inc), with one CTA per tile: the emulator runs blocks one after another, so a
// persistent grid's look-back would wait for a block that never runs.
#define KVG_HOST_EMU 1
#include "warp_emu.h"
#include "kvgpu.h"
namespace kvg {
#include "emu_order.inc"
}
#include "../../kubevirt-gpu-device-plugin_b200/csrc/kvg_rescan.cuh"

using namespace kvg;

namespace {
// state the context keeps between rescans: the key flags (they travel with their key list) and the look-back
// words; neither is ever cleared by the harness
std::vector<uint8_t> g_mark[2][2];  // [buffer][map]
int g_cur = 0;
std::vector<uint64_t> g_state, g_kstate;
uint32_t g_epoch = 0;
}  // namespace

extern "C" {

// keys[m] = {old keys, new keys}, nkeys[m] = {n old, n new}; outputs sized by the caller:
// surv_out = {added u32[nb], removed uint4[U*na], moved u32[nb]}, key_out[m][q] u32[max(n old, n new)],
// b_next uint4[U*nb], kb_next[m] u32[n new]; ctrl_out receives the RescanCtrl words.
int emu_rescan(int mdev, const uint4* a, uint32_t na, const uint4* b, uint32_t nb, const uint32_t* const* keys,
               const uint32_t* nkeys, uint32_t* added, uint4* removed, uint32_t* moved, uint32_t* const* key_out,
               uint4* b_next, uint32_t* const* kb_next, uint32_t* ctrl_out) {
  const int cur = g_cur, nx = cur ^ 1;
  for (int m = 0; m < 2; m++)  // grown zero-filled, like a fresh device allocation
    for (int s = 0; s < 2; s++)
      g_mark[s ? nx : cur][m].resize(std::max<size_t>(g_mark[s ? nx : cur][m].size(), nkeys[2 * m + s] + 1), 0);
  const uint32_t tiles = (na + nb + RS_TILE - 1) / RS_TILE;
  uint32_t ktiles = 0;
  for (int m = 0; m < 2; m++) ktiles = std::max(ktiles, (nkeys[2 * m] + nkeys[2 * m + 1] + RS_TILE - 1) / RS_TILE);
  if (g_state.size() < 3 * (tiles + 1)) g_state.resize(3 * (tiles + 1), 0);
  if (g_kstate.size() < 6 * (ktiles + 1)) g_kstate.resize(6 * (ktiles + 1), 0);
  RescanCtrl ctrl;
  memset(&ctrl, 0xee, sizeof ctrl);  // poisoned: every count is written by the kernels
  ctrl.bad = 0;
  const uint32_t epoch = ++g_epoch;
  RsMergeArgs g;
  g.a = a;
  g.na = na;
  g.b = b;
  g.nb = nb;
  g.b_next = b_next;
  for (int m = 0; m < 2; m++) {
    g.okeys[m] = keys[2 * m];
    g.nok[m] = nkeys[2 * m];
    g.nkeys[m] = keys[2 * m + 1];
    g.nnk[m] = nkeys[2 * m + 1];
    g.omark[m] = g_mark[cur][m].data();
    g.nmark[m] = g_mark[nx][m].data();
  }
  g.added = added;
  g.removed = removed;
  g.moved = moved;
  g.ctrl = &ctrl;
  g.state = g_state.data();
  g.stride = tiles + 1;
  if (mdev)
    emu_launch(k_rescan_merge<RsMdev>, dim3(std::max(1u, tiles), 1), KVG_BLOCK, g, epoch);
  else
    emu_launch(k_rescan_merge<RsPci>, dim3(std::max(1u, tiles), 1), KVG_BLOCK, g, epoch);
  RsKeysArgs2 kk;
  for (int m = 0; m < 2; m++) {
    RsKeysArgs& k = kk.m[m];
    k.a = keys[2 * m];
    k.na = nkeys[2 * m];
    k.b = keys[2 * m + 1];
    k.nb = nkeys[2 * m + 1];
    k.b_next = kb_next[m];
    k.amark = g_mark[cur][m].data();
    k.bmark = g_mark[nx][m].data();
    for (int q = 0; q < 3; q++) k.out[q] = key_out[3 * m + q];
    k.state = g_kstate.data() + (size_t)m * 3 * (ktiles + 1);
    k.stride = ktiles + 1;
  }
  emu_launch(k_rescan_keys, dim3(std::max(1u, ktiles), 2), KVG_BLOCK, kk, &ctrl, epoch);
  memcpy(ctrl_out, &ctrl, sizeof ctrl);
  g_cur = nx;
  return ctrl.bad == epoch ? 1 : 0;
}

// every key flag of both buffers is zero (the kernels clean up after themselves)
int emu_rescan_flags_clear(void) {
  for (auto& buf : g_mark)
    for (auto& v : buf)
      for (uint8_t f : v)
        if (f) return 0;
  return 1;
}

}
