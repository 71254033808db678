// rectify_ring.cuh -- scheduling and producer side shared by the staged rectification kernels.
//
// Persistent CTAs fed from a global ticket counter.  A work unit is one tile (strip x, tile y)
// of a GROUP of consecutive frames, numbered x fastest, and units are handed out in that order to
// whichever CTA is free: at any instant the device works on a window of consecutive units, so tiles that
// share source lines (the halos of neighbouring strips) are fetched within microseconds of each
// other and the second fetch hits L2.  Static schedules (long private walks, round-robin) let
// the CTAs drift apart and were measured to read 1.5x the frame from DRAM
// (profiles/r1_rectify.md).
//
// Producer warp, per unit: take a ticket (one ticket ahead, so the atomic's latency is hidden),
// decode it, read the tile header and the q2 terms from the plan, wait for a free stage, publish
// {position, header, q2} in the stage's slot and issue ONE cp.async.bulk.tensor.  A ticket past
// the last unit is published as a stop marker.  The last producer to leave resets the counter.
#pragma once

namespace cc {

__device__ __forceinline__ void ring_init(SmemRing* ring, int stages) {
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&ring->full[s], 1);
            mbar_init(&ring->empty[s], kWarps);
        }
        mbar_fence_init();
    }
    __syncthreads();
}

// the producer waits for a free stage parked on the barrier's own suspend-time hint (a polling loop of
// try_wait + nanosleep was 8 % of all executed warp instructions of the u8 kernel, ncu round 2)
__device__ __forceinline__ void producer_wait(uint64_t* bar, uint32_t parity) {
    mbar_wait_parked<2000>(bar, parity);
}

__device__ __forceinline__ uint32_t take_ticket(RectSched* sched, int lane_id) {
    uint32_t u = 0;
    if (lane_id == 0) u = atomicAdd(&sched->next, 1u);
    return __shfl_sync(0xffffffffu, u, 0);
}

// PXB: multiplier from TileHdr.x0 to the tensor-map coordinate (1: f32c1 texels, and u8c3 whose x0 already is a byte offset).
// A unit is (strip x, tile y, frame group): the producer publishes one slot per FRAME of the
// group -- pos = (x, y, frame, number of frames of the unit on its first frame, else 0) -- the
// consumers read the slot on a unit's first frame only and count the frames down.
// NF: frames per ring stage (2: a stage holds the boxes of two consecutive frames of the unit -- one at
// the odd end of a unit -- so the consumers pay one hand-over per pair)
// VIEWS: frames with different views in one launch -- the third unit coordinate counts (view, frame group of
// the view), the view's tables start at view * tiles / view * sz2, and the view index travels in the header.
// The launch may cover a window of the group's frames (TileCfg.w0 / g0, g.nframes = its length): the frame
// index published to the consumers and given to TMA is relative to the window, the view stays the group's.
template <bool EXACT, int TL, int PXB, int NF = 1, bool VIEWS = false>
__device__ __forceinline__ void producer_loop(const CUtensorMap* tmap, const RectGeom& g, const TileCfg& cfg,
                                              const TileHdr* __restrict__ plan,
                                              const double* __restrict__ q2tab, RectSched* sched,
                                              SmemRing* ring, uint8_t* stage_mem, int lane_id) {
    if (lane_id == 0) tma_prefetch_desc(tmap);
    const uint64_t policy = l2_evict_last();
    int s = 0;
    uint32_t phase = 1;                            // a fresh barrier passes a parity-1 wait
    uint32_t u_next = take_ticket(sched, lane_id);
    for (;;) {
        const uint32_t u = u_next;
        if (u >= cfg.units) break;
        const int x = (int)(u % (uint32_t)cfg.strips);
        const uint32_t r = u / (uint32_t)cfg.strips;
        const int y = (int)(r % (uint32_t)cfg.ntiles2);
        int f0 = (int)(r / (uint32_t)cfg.ntiles2) * cfg.fg;
        int f1 = min(f0 + cfg.fg, g.nframes);
        const TileHdr* hdr_v = plan;
        const double* q2_v = q2tab;
        [[maybe_unused]] uint32_t view = 0;
        if (VIEWS) {
            const uint32_t grp = cfg.g0 + r / (uint32_t)cfg.ntiles2;
            view = grp / (uint32_t)cfg.gpv;
            f0 = (int)view * cfg.fpv + (int)(grp - view * (uint32_t)cfg.gpv) * cfg.fg;
            f1 = min(f0 + cfg.fg, ((int)view + 1) * cfg.fpv);
            // the frame window (TileCfg.w0): frames of the group -> frames of the launch
            f0 = max(f0, cfg.w0) - cfg.w0;
            f1 = min(f1, cfg.w0 + g.nframes) - cfg.w0;
            hdr_v = plan + (size_t)view * cfg.tiles;
            q2_v = q2tab + (size_t)view * g.sz2;
        }
        const uint32_t* hp = reinterpret_cast<const uint32_t*>(hdr_v + x * cfg.ntiles2 + y);
        uint32_t hword = 0;
        if (lane_id < 12) hword = __ldg(hp + lane_id);            // the 48-byte header, one word per lane
        if (VIEWS && lane_id == 11) hword = view;
        [[maybe_unused]] double q2a = 0, q2b = 0;
        if (EXACT) {
            const int b = y * TL + lane_id;
            q2a = __ldg(q2_v + min(b, g.sz2 - 1));
            if (TL > 32) q2b = __ldg(q2_v + min(b + 32, g.sz2 - 1));
        }
        u_next = take_ticket(sched, lane_id);
        const int x0 = __shfl_sync(0xffffffffu, (int)hword, 8), y0 = __shfl_sync(0xffffffffu, (int)hword, 9);
        for (int f = f0; f < f1; f += NF) {
            producer_wait(&ring->empty[s], phase);
            if (f == f0) {                                        // the map inputs travel with the first frame
                if (lane_id < 12) reinterpret_cast<uint32_t*>(&ring->hdr[s])[lane_id] = hword;
                if (EXACT) {
                    if (lane_id < TL) ring->q2[s][lane_id] = q2a;
                    if (TL > 32) ring->q2[s][lane_id + 32] = q2b;
                }
            }
            if (lane_id == 12) ring->pos[s] = make_int4(x, y, f, f == f0 ? f1 - f0 : 0);   // .w: frames of the unit, on its first frame
            __syncwarp();
            if (lane_id == 0) {
                const int nload = min(NF, f1 - f);             // the odd end of a unit: one box
                mbar_arrive_expect_tx(&ring->full[s], (uint32_t)cfg.box_bytes * nload);
#pragma unroll
                for (int j = 0; j < NF; ++j) {
                    if (j >= nload) break;
                    uint8_t* box = stage_mem + ((size_t)s * NF + j) * cfg.box_bytes;
                    tma_load_3d_hint(box, tmap, &ring->full[s], x0 * PXB, y0, f + j, policy);
                }
            }
            if (++s == cfg.stages) { s = 0; phase ^= 1; }
        }
    }
    // stop marker
    producer_wait(&ring->empty[s], phase);
    if (lane_id == 0) { ring->pos[s] = make_int4(0, 0, -1, 0); mbar_arrive(&ring->full[s]); }
    // every producer has taken its last ticket before it counts itself out
    if (lane_id == 0 && atomicAdd(&sched->done, 1u) == gridDim.x - 1) {
        sched->next = 0;
        sched->done = 0;
    }
}

}  // namespace cc
