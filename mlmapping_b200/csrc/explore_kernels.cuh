// Exploration-frontier mode (use_exploration_frontiers): the reference's update_observation
// (src/map_local.cpp:7-33), frontier bookkeeping and release pass (:208-232).
//
// update_observation is called when a cell turns from 'u' to 'f' in the miss pass, in miss_idx_set
// iteration order, and looks at the CURRENT state of the 6 neighbours, so the result depends on that
// order.  It is still data parallel: a 'u' cell with misses turns 'f' at its first miss cell in iteration
// order; a neighbour is still 'u' at that moment iff it was 'u' after the hit pass and either has no miss
// cell or its own first miss cell comes later.  The iteration order of the unordered_set<size_t> is the same
// (bucket activation, insert stamp) rule as for the hit map (identity hash), so "comes earlier" is a
// comparison of two 64-bit keys staged per voxel.
#pragma once
#include "frame_kernels.cuh"
#include "order_kernels.cuh"

namespace mlm {

__device__ __forceinline__ bool inside_exp_bd(const MapParams &P, double x, double y, double z) {  // map_local.h:160-165
  return x >= P.bd[0] && x < P.bd[1] && y >= P.bd[2] && y < P.bd[3] && z >= P.bd[4] && z < P.bd[5];
}

// per miss cell: key = (activation stamp of its bucket, its own stamp); the voxel keeps the largest key
// (= the miss cell that the descending iteration reaches first)
__device__ __forceinline__ void miss_tkey_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  const FrameCounters *fc = D.fc[F.parity];
  const int n = fc->n_miss_list;
  const uint32_t *am = D.act_miss[F.parity];
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const unsigned long long key = ((unsigned long long)am[D.miss_bucket[j]] << 32) | D.miss_t[j];
    atomicMax(&D.lvg_tkey[D.miss_lv[j]], key);
  }
}

// subbox_neighbors row i of cell (g, sub): +z,-z,+y,-y,+x,-x (src/map_local.cpp:78-120)
__device__ __forceinline__ void nb_of(const MapParams &P, int dir, const int g[3], int sub, int gn[3], int &subn, int dl[3]) {
  int c[3] = {sub % P.n, (sub / P.n) % P.n, sub / (P.n * P.n)};
  gn[0] = g[0];
  gn[1] = g[1];
  gn[2] = g[2];
  dl[0] = dl[1] = dl[2] = 0;
  const int axis = 2 - (dir >> 1), step = (dir & 1) ? -1 : 1;
  dl[axis] = step;
  c[axis] += step;
  if (c[axis] >= P.n) {
    gn[axis] += 1;
    c[axis] = 0;
  } else if (c[axis] < 0) {
    gn[axis] -= 1;
    c[axis] = P.n - 1;
  }
  subn = (c[2] * P.n + c[1]) * P.n + c[0];
}

// pass A: the miss cell that turns its voxel from 'u' to 'f' evaluates update_observation: remembers which
// neighbour becomes a frontier cell, allocates neighbour subboxes exactly like allocate_ram would.
__device__ __forceinline__ void explore_a_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  FrameCounters *fc = D.fc[F.parity];
  const int n = fc->n_miss_list;
  const uint32_t *am = D.act_miss[F.parity];
  const int dxy = P.lvg_dim_xy;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    D.miss_choice[j] = -1;
    const int lv = D.miss_lv[j];
    const unsigned long long key = ((unsigned long long)am[D.miss_bucket[j]] << 32) | D.miss_t[j];
    if (key != D.lvg_tkey[lv]) continue;  // not the first miss cell of its voxel
    // the voxel
    int c[3] = {lv % dxy + F.lvg_base[0], (lv / dxy) % dxy + F.lvg_base[1], lv / (dxy * dxy) + F.lvg_base[2]};
    int g[3], l[3];
    for (int a = 0; a < 3; a++) {
      g[a] = floor_div(c[a], P.n);
      l[a] = c[a] - g[a] * P.n;
    }
    const int sub = (l[2] * P.n + l[1]) * P.n + l[0];
    const int ls = lsg_index(P, F, g);
    const int block = ls >= 0 ? __ldcg(&D.lsg_block[ls]) : -3;
    if (block < 0) continue;                                             // allocate_ram false
    if (D.pool_occ[(size_t)block * P.cell_stride + sub] != 'u') continue;  // only 'u' -> 'f' observes
    // p_w of THIS miss cell (src/map_local.cpp:180,198)
    const int idx = D.miss_idx[j];
    const int zk = idx / (P.nRho * P.nPhi), rem = idx - zk * (P.nRho * P.nPhi);
    const int pk = rem / P.nRho, rk = rem - pk * P.nRho;
    const double2 cxy = __ldg(&P.centre_xy[pk * P.nRho + rk]);
    const double pw[3] = {cxy.x + F.t_wa[0], cxy.y + F.t_wa[1], __ldg(&P.centre_z[zk]) + F.t_wa[2]};
    if (!inside_exp_bd(P, pw[0], pw[1], pw[2])) continue;
    // observed_subboxes.emplace(glb_idx)
    if (__ldcg(&D.obs_flag[ls]) == 0 && atomicExch(&D.obs_flag[ls], 1) == 0) D.obs_list[atomicAdd(&fc->n_obs, 1)] = ls;
    const unsigned long long my_key = key;
    for (int i = 0; i < 6; i++) {
      int gn[3], subn, dl[3];
      nb_of(P, i, g, sub, gn, subn, dl);
      // pt_w_nb = pt_w + nbr_disp_real[i]: one axis gets +-d_sub, the others + 0
      const double pn[3] = {pw[0] + (double)dl[0] * P.d_sub, pw[1] + (double)dl[1] * P.d_sub, pw[2] + (double)dl[2] * P.d_sub};
      if (!inside_exp_bd(P, pn[0], pn[1], pn[2])) continue;
      uint64_t hkey;
      if (!pack_glb(gn, hkey)) {
        fc->error = kErrRange;
        continue;
      }
      // allocate_ram(glb_idx_nb): find, or create (a fresh subbox is all 'u')
      uint32_t slot = ht_hash(hkey) & P.ht_mask;
      int val = kBlockPending, created = -1;
      bool found = false;
      for (uint32_t probe = 0; probe <= P.ht_mask; probe++) {
        uint64_t k = D.ht_key[slot];
        if (k == kEmptyKey) {
          unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(&D.ht_key[slot]),
                                             (unsigned long long)kEmptyKey, (unsigned long long)hkey);
          if (old == kEmptyKey) {
            int top = atomicSub(D.free_top, 1) - 1;
            if (top < 0) {
              atomicAdd(D.free_top, 1);
              D.ht_val[slot] = kBlockUnusable;
              fc->error = kErrPool;
            } else {
              created = D.free_stack[top];
              D.ht_val[slot] = created;
              atomicAdd(&fc->n_new_blocks, 1);
            }
            val = kBlockPending;  // created in this pass: every cell 'u'
            found = true;
            break;
          }
          k = (uint64_t)old;
        }
        if (k == hkey) {
          val = D.ht_val[slot];
          found = true;
          break;
        }
        slot = (slot + 1) & P.ht_mask;
      }
      if (!found) {
        fc->error = kErrPool;
        continue;
      }
      if (val == kBlockCollapsed || val == kBlockUnusable) continue;  // allocate_ram returns false
      bool is_u = true;
      if (val >= 0) {
        is_u = D.pool_occ[(size_t)val * P.cell_stride + subn] == 'u';   // state after the hit pass
        if (is_u) {
          // ... and not yet turned 'f' by a miss cell that the iteration reaches before mine
          const int cn[3] = {c[0] + dl[0], c[1] + dl[1], c[2] + dl[2]};
          const int lx = cn[0] - F.lvg_base[0], ly = cn[1] - F.lvg_base[1], lz = cn[2] - F.lvg_base[2];
          if ((unsigned)lx < (unsigned)P.lvg_dim_xy && (unsigned)ly < (unsigned)P.lvg_dim_xy && (unsigned)lz < (unsigned)P.lvg_dim_z) {
            const int lvn = (lz * P.lvg_dim_xy + ly) * P.lvg_dim_xy + lx;
            if (D.lvg[lvn].y > 0 && D.lvg_tkey[lvn] > my_key) is_u = false;
          }
        }
      }
      if (is_u) {
        // frontier[glb_nb].emplace(sub_nb): at once when the neighbour's block is known here (nobody reads the frontier
        // words during this pass); a subbox another thread is creating right now is left to pass B
        const int blk = val >= 0 ? val : created;
        if (blk >= 0) atomicOr(&D.pool_front[(size_t)blk * P.front_words + (subn >> 5)], 1u << (subn & 31));
        else D.miss_choice[j] = (signed char)i;
        break;
      }
    }
  }
}

// pass B: frontier[glb_nb].emplace(sub_nb) for the choices pass A could not place itself (all subboxes exist now)
__device__ __forceinline__ void explore_b_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  const FrameCounters *fc = D.fc[F.parity];
  const int n = fc->n_miss_list;
  const int dxy = P.lvg_dim_xy;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const int i = D.miss_choice[j];
    if (i < 0) continue;
    const int lv = D.miss_lv[j];
    int c[3] = {lv % dxy + F.lvg_base[0], (lv / dxy) % dxy + F.lvg_base[1], lv / (dxy * dxy) + F.lvg_base[2]};
    int g[3], l[3];
    for (int a = 0; a < 3; a++) {
      g[a] = floor_div(c[a], P.n);
      l[a] = c[a] - g[a] * P.n;
    }
    int gn[3], subn, dl[3];
    nb_of(P, i, g, (l[2] * P.n + l[1]) * P.n + l[0], gn, subn, dl);
    const int val = ht_find(P, D, gn);
    if (val >= 0) atomicOr(&D.pool_front[(size_t)val * P.front_words + (subn >> 5)], 1u << (subn & 31));
  }
}

// release pass (src/map_local.cpp:208-232): one warp per observed subbox; collapse if the frontier is empty
// and all occupancy chars are equal.  The block returns to the free stack in its initial state; element 0 of
// the three vectors stays readable through the per-slot arrays.
__device__ __forceinline__ void release_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  FrameCounters *fc = D.fc[F.parity];
  const int lane = lane_id();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n = fc->n_obs;
  for (int o = warp; o < n; o += nwarps) {
    const int ls = D.obs_list[o];
    if (lane == 0) D.obs_flag[ls] = 0;
    int lx = ls % P.lsg_dim_xy, ly = (ls / P.lsg_dim_xy) % P.lsg_dim_xy, lz = ls / (P.lsg_dim_xy * P.lsg_dim_xy);
    int g[3] = {lx + F.lsg_base[0], ly + F.lsg_base[1], lz + F.lsg_base[2]};
    uint32_t slot;
    const int block = ht_find_slot(P, D, g, slot);
    if (block < 0) continue;  // absent or already collapsed (occupancy.size() == 1)
    const size_t base = (size_t)block * P.cell_stride;
    // (no short-circuit: the loads of a lane are independent and all in flight together)
    bool ok = true;
    for (int w = lane; w < P.front_words; w += 32) ok &= D.pool_front[(size_t)block * P.front_words + w] == 0;
    const char first = D.pool_occ[base];
    if ((base & 3) == 0) {
      const uint32_t first4 = 0x01010101u * (uint32_t)(unsigned char)first;
      const uint32_t *occ4 = reinterpret_cast<const uint32_t *>(D.pool_occ + base);
      const int n4 = P.cells >> 2;
      for (int i = lane; i < n4; i += 32) ok &= occ4[i] == first4;
      for (int i = (n4 << 2) + lane; i < P.cells; i += 32) ok &= D.pool_occ[base + i] == first;
    } else {
      for (int i = lane; i < P.cells; i += 32) ok &= D.pool_occ[base + i] == first;
    }
    if (!__all_sync(0xffffffffu, ok)) continue;
    if (lane == 0) {
      D.col_occ[slot] = first;
      D.col_inf[slot] = D.pool_inf[base];
      D.col_lo[slot] = D.pool_lo[base];
      D.ht_val[slot] = kBlockCollapsed;
      atomicAdd(&fc->n_released, 1);
    }
    __syncwarp();
    for (int i = lane; i < P.cell_stride; i += 32) {
      D.pool_occ[base + i] = 'u';
      D.pool_inf[base + i] = 'u';
      D.pool_lo[base + i] = 0.f;
    }
    for (int w = lane; w < P.front_words; w += 32) D.pool_front[(size_t)block * P.front_words + w] = 0;
    __syncwarp();
    if (lane == 0) {
      __threadfence();
      D.free_stack[atomicAdd(D.free_top, 1)] = block;  // recycled: ready for the next allocate_ram
    }
  }
}

__global__ void __launch_bounds__(256) k_miss_finalize(MapParams P, DeviceBuffers D, FrameParams F) { miss_finalize_body(P, D, F); }
__global__ void __launch_bounds__(256) k_miss_tkey(MapParams P, DeviceBuffers D, FrameParams F) { miss_tkey_body(P, D, F); }
__global__ void __launch_bounds__(256) k_explore_a(MapParams P, DeviceBuffers D, FrameParams F) { explore_a_body(P, D, F); }
__global__ void __launch_bounds__(256) k_explore_b(MapParams P, DeviceBuffers D, FrameParams F) { explore_b_body(P, D, F); }
__global__ void __launch_bounds__(256) k_release(MapParams P, DeviceBuffers D, FrameParams F) { release_body(P, D, F); }

// ---- the exploration-mode frame as ONE cooperative launch (the k_frame of frame_kernels.cuh with the six exploration
// passes behind further device-wide barriers).  A frame whose hit map or miss set would cross a libstdc++ rehash is
// detected after staging, on the device: every CTA returns with the staging intact, the frame is flagged (overflow) and
// the host re-sequences and runs the passes as stand-alone kernels (run_frame_complete in mlmap_capi.cu).
template <int kMode>
__global__ void __launch_bounds__(kColThreads, 1) k_frame_explore(MapParams P, DeviceBuffers D, FrameParams F) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  const int G = (int)gridDim.x;
  FrameCounters *fc = D.fc[F.parity];
  MLM_FRAME_WALL(0);
  {
    const int n_tiles = (F.n_total + F.tile_pts - 1) / F.tile_pts;
    for (int t = blockIdx.x; t < max(n_tiles, 1); t += G) {
      project_tile<kMode>(P, D, F, t, reinterpret_cast<int *>(s_raw));
      __syncthreads();
    }
  }
  MLM_FRAME_WALL(1);
  grid_arrive(D.grid_bar);
  load_col_tables(P, s_raw);   // the projection is done with shared memory (the loop's last barrier)
  grid_wait(D.grid_bar, G);
  MLM_FRAME_WALL(2);
  column_phase(P, D, F, s_raw, true);
  MLM_FRAME_WALL(3);
  grid_barrier(D.grid_bar, 2 * G);
  MLM_FRAME_WALL(4);
  if (blockIdx.x == 0 && threadIdx.x == 0) *D.col_queue = 0;
  miss_finalize_body(P, D, F);    // split layouts: stamps of the sensor-row miss cells (read again behind the next barriers)
  if (__ldcg(&fc->n_hit) > (int)F.bucket_count || __ldcg(&fc->n_miss_list) > (int)F.bucket_count_miss) {
    frame_bail(D, fc, F);
    return;
  }
  fuse_body<1>(P, D, F);          // hits (the frame-local voxel grid stays intact)
  MLM_FRAME_WALL(5);
  grid_barrier(D.grid_bar, 3 * G);
  miss_tkey_body(P, D, F);        // first miss cell of every voxel in set iteration order
  MLM_FRAME_WALL(6);
  grid_barrier(D.grid_bar, 4 * G);
  explore_a_body(P, D, F);        // update_observation: neighbour choices, neighbour subboxes allocated
  MLM_FRAME_WALL(9);
  grid_barrier(D.grid_bar, 5 * G);
  // frontier inserts pass A left over: neighbours in subboxes another thread was creating at that moment.  Such a subbox
  // did not exist when the frame was staged, so no voxel of it is touched this frame and the miss pass erases no
  // frontier bit in it: the two passes share a phase
  explore_b_body(P, D, F);
  MLM_FRAME_WALL(10);
  fuse_body<2, false>(P, D, F);   // misses
  MLM_FRAME_WALL(11);
  grid_barrier(D.grid_bar, 6 * G);
  release_body(P, D, F);          // collapse pass over the observed subboxes
  MLM_FRAME_WALL(12);
  frame_finish(P, D, F, fc, __ldcg(&fc->n_hit));
}

}  // namespace mlm
