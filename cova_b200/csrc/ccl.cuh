// Connected-component labelling + bounding boxes + bincode, one CTA per mask, entirely in shared memory.
//
// Reference: cova-rs/gst-plugins/src/bboxcc/process.rs:5-49 (cv::connectedComponentsWithStats, 8-connectivity,
// CV_32S; keep CC_STAT_AREA >= threshold; Bbox::new(left, top, width, height)) and
// cova-rs/bbox/src/bbox.rs:17-29,84-86 (area = width*height; bincode: u64 count + 24 bytes per box).
//
// Design (not OpenCV's two-pass scan): the mask is reduced to one 4-bit code per 2x2-aligned block
// (all pixels of a 2x2 block are mutually 8-adjacent, so a block is the natural union-find node).
// Blocks are merged with a lock-free atomicMin union-find in shared memory; because links always go
// from the larger to the smaller block index, a component's root IS its first block in raster order,
// which is exactly OpenCV's label order (SURVEY.md section 8 row A7) - so ranking the roots with a
// block-wide prefix sum reproduces the reference's label numbers and box order with no sort.
// Horizontal runs of blocks are linked by a warp ballot before the union-find (depth-1 trees), which removes the
// O(run length) chains: all-ones 720p masks 2.58 ms -> 0.65 ms per 8192 masks, diagonal checkerboard 1.72 -> 0.43 ms
// (tools/ccl_timing.py, B200).
#pragma once
#include <type_traits>

#include <cooperative_groups.h>

#include "common.cuh"

namespace cova {

struct CclArgs {
    const uint8_t *masks;     // [n][H][W]
    int H, W, nbx, nby;       // nbx = ceil(W/2), nby = ceil(H/2)
    int area_thresh;          // u32 property reinterpreted as i32 like imp.rs:248
    const int *thresh;        // optional [n]: per-mask area_thresh (a batch whose streams have their own cc-threshold)
    uint8_t *blob;            // bincode output arena
    unsigned long long blob_cap;
    unsigned long long *cursor;   // [0] bytes reserved so far, [1] overflow flag
    unsigned long long *offsets;  // [n]
    unsigned long long *lens;     // [n]
    int32_t *labels;          // optional [n][H][W]
    int32_t *stats;           // optional [n][(nb+1)*5]
    int32_t *n_labels;        // optional [n]
    FastDiv div_nbx;          // block index -> (by, bx) of a thread's first block; later blocks advance by (step_by, step_bx)
    int step_by, step_bx;     // blockDim.x / nbx, blockDim.x % nbx
    // merge phase "tile scan" (0 = concurrent union-find over all foreground blocks): the grid of blocks is cut into tiles
    // of 32 columns x tile_rows rows, about one per warp
    int scan, tiles_x, tiles_y, tile_rows;
    FastDiv div_tile_rows;
};

// (by, bx) of block b + blockDim.x from those of block b
#define COVA_CCL_ADVANCE(by, bx) do { bx += A.step_bx; by += A.step_by; if (bx >= A.nbx) { bx -= A.nbx; by++; } } while (0)

// Shared-memory layouts.  WIDE: parent (i32) + per-block statistics [min x, min y, max x, max y, area] (i32 each) +
// block code (u8) = 25 bytes per 2x2 block.  At 4K (8160 blocks) that is 204 KB, i.e. one CTA per SM for a kernel that
// waits on shared-memory pointer chases, not on bandwidth.  COMPACT: parent u16 (block indices are below 65535), min x |
// min y and max x | max y as 16-bit pairs in one word each, area u16 (at most 4 pixels per block) = 13 bytes per block:
// 106 KB at 4K, two CTAs (64 warps) per SM.  16-bit parents are updated with compare-and-swap loops, the packed
// statistics with a CAS that is skipped when the box would not grow (on a large component almost every update is a
// no-op).  The wide layout keeps the native 32-bit atomics; the host picks COMPACT when the wide one would not leave room
// for a second CTA.
__host__ __device__ inline size_t ccl_smem_bytes(int nb, int threads, bool compact) {
    const size_t per_block = compact ? (size_t)((nb + 1) / 2 * 2) * 2 * 2 + (size_t)nb * 8    // parent u16 + area u16 (even count), mn + mx u32
                                     : (size_t)nb * 6 * sizeof(int);
    // + block codes (u8) + the per-warp lists of foreground blocks (u16, ceil(nb / threads) * threads entries) + scan scratch
    const size_t list = (size_t)((nb + threads - 1) / threads) * threads * 2;
    return per_block + (size_t)((nb + 15) / 16) * 16 + (list + 15) / 16 * 16 + (size_t)(threads / 32 + 4) * sizeof(int);
}

template <bool COMPACT>
struct CclMem {
    using PT = typename std::conditional<COMPACT, unsigned short, int>::type;
    static constexpr int kNone = COMPACT ? 0xFFFF : -1;          // parent of a background block (never equals a block index)
    PT *parent;
    int *stat;                 // WIDE: [block][5]
    uint32_t *mn, *mx;         // COMPACT: min x | min y << 16, max x | max y << 16
    unsigned short *area;      // COMPACT
    uint8_t *code;
    unsigned short *list;      // per-warp lists of foreground blocks (bit 15: the block was lane 0 of its 32-block segment)
    int *scan;

    __device__ __forceinline__ CclMem(unsigned char *base, int nb, int nt) {
        if constexpr (COMPACT) {
            const int nbe = (nb + 1) / 2 * 2;
            parent = reinterpret_cast<PT *>(base);
            area = reinterpret_cast<unsigned short *>(base) + nbe;
            mn = reinterpret_cast<uint32_t *>(area + nbe);
            mx = mn + nb;
            code = reinterpret_cast<uint8_t *>(mx + nb);
            stat = nullptr;
        } else {
            parent = reinterpret_cast<PT *>(base);
            stat = reinterpret_cast<int *>(base) + nb;
            code = reinterpret_cast<uint8_t *>(stat + 5 * nb);
            mn = mx = nullptr; area = nullptr;
        }
        list = reinterpret_cast<unsigned short *>(code + ((nb + 15) / 16) * 16);
        scan = reinterpret_cast<int *>(reinterpret_cast<unsigned char *>(list) + ((size_t)((nb + nt - 1) / nt) * nt * 2 + 15) / 16 * 16);
    }
    // ---- parent[]: every concurrent access is an atomic or a volatile load
    __device__ __forceinline__ int load(int i) const { return (int)reinterpret_cast<volatile PT *>(parent)[i]; }
    __device__ __forceinline__ void lower(int j, int r) const {            // parent[j] = min(parent[j], r)
        if constexpr (COMPACT) {
            unsigned short cur = reinterpret_cast<volatile PT *>(parent)[j];
            while ((int)cur > r) {
                const unsigned short old = atomicCAS(&parent[j], cur, (unsigned short)r);
                if (old == cur) break;
                cur = old;
            }
        } else {
            atomicMin(&parent[j], r);
        }
    }
    __device__ __forceinline__ int cas(int a, int b) const {                // link root a under b if a is still a root
        if constexpr (COMPACT) return (int)atomicCAS(&parent[a], (unsigned short)a, (unsigned short)b);
        else return atomicCAS(&parent[a], a, b);
    }
    __device__ __forceinline__ int find(int i) const {
        int p;
        while ((p = load(i)) != i) i = p;
        return i;
    }
    // Find with path compression.  parent[] only ever DECREASES and always names a block of the same (eventual) component:
    // links go from a ROOT to a smaller index (compare-and-swap: an edge, once made, is never replaced by another edge), and a
    // compression moves a parent to one of its own ancestors.  All ancestors a block ever has lie on one chain, ordered by
    // index, so "the smaller of the current parent and a root seen a moment ago" is always a valid ancestor whatever other
    // threads do meanwhile, no cycle can form (parent[j] < j for every non-root).  Without compression a dense mask builds
    // one link per block row (the run heads of consecutive rows chain up) and every find of a block in row r walks r links:
    // 41 % of the kernel's stall samples at 4K sat in that loop (profiles/r2c_ccl_lines.txt).
    __device__ __forceinline__ int find_compress(int i) const {
        int r = load(i);
        if (r == i) return i;
        int p, hops = 0;
        while ((p = load(r)) != r) { r = p; hops++; }
        if (hops) {
            int j = i;                                   // second walk: everything on the path now points at r
            while ((p = load(j)) > r) {
                lower(j, r);
                j = p;
            }
        }
        return r;
    }
    __device__ __forceinline__ void unite(int a, int b) const {
        while (true) {
            a = find_compress(a);
            b = find_compress(b);
            if (a == b) return;
            if (a < b) { int t = a; a = b; b = t; }
            // Link the larger ROOT under the smaller one - compare-and-swap, not atomicMin: an atomicMin on an `a` that has
            // meanwhile been linked elsewhere would REPLACE that committed edge (the displaced pair is re-united by this
            // thread's next iteration, but a concurrent compression that has already seen the new edge can short-cut across
            // it before that happens, and the re-union then finds nothing left to do - one component too many, once in a few
            // hundred dense masks).
            const int old = cas(a, b);
            if (old == a) return;
            a = old;
        }
    }
    // ---- statistics (live at roots; only foreground blocks can be roots)
    __device__ __forceinline__ void stat_init(int b) const {
        if constexpr (COMPACT) { mn[b] = 0xFFFFFFFFu; mx[b] = 0u; area[b] = 0; }
        else { int *sb = stat + 5 * b; sb[0] = 0x7fffffff; sb[1] = 0x7fffffff; sb[2] = -1; sb[3] = -1; sb[4] = 0; }
    }
    __device__ __forceinline__ void stat_add(int r, int x0, int y0, int x1, int y1, int cnt) const {
        if constexpr (COMPACT) {
            uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&mn[r]);
            while (true) {
                const uint32_t want = min(cur & 0xFFFFu, (uint32_t)x0) | (min(cur >> 16, (uint32_t)y0) << 16);
                if (want == cur) break;                                  // the box already covers this block
                const uint32_t old = atomicCAS(&mn[r], cur, want);
                if (old == cur) break;
                cur = old;
            }
            cur = *reinterpret_cast<volatile uint32_t *>(&mx[r]);
            while (true) {
                const uint32_t want = max(cur & 0xFFFFu, (uint32_t)x1) | (max(cur >> 16, (uint32_t)y1) << 16);
                if (want == cur) break;
                const uint32_t old = atomicCAS(&mx[r], cur, want);
                if (old == cur) break;
                cur = old;
            }
            // two u16 areas per word; a component has at most 4 * nb < 65536 pixels, so a half never carries into its neighbour
            atomicAdd(reinterpret_cast<unsigned int *>(area) + (r >> 1), (unsigned int)cnt << (16 * (r & 1)));
        } else {
            int *sr = stat + 5 * r;
            atomicMin(&sr[0], x0); atomicMax(&sr[2], x1);
            atomicMin(&sr[1], y0); atomicMax(&sr[3], y1);
            atomicAdd(&sr[4], cnt);
        }
    }
    __device__ __forceinline__ int stat_area(int b) const { return COMPACT ? (int)area[b] : stat[5 * b + 4]; }
    __device__ __forceinline__ void stat_get(int b, int &x0, int &y0, int &x1, int &y1) const {
        if constexpr (COMPACT) { x0 = (int)(mn[b] & 0xFFFFu); y0 = (int)(mn[b] >> 16); x1 = (int)(mx[b] & 0xFFFFu); y1 = (int)(mx[b] >> 16); }
        else { const int *sb = stat + 5 * b; x0 = sb[0]; y0 = sb[1]; x1 = sb[2]; y1 = sb[3]; }
    }
    // the area slot of a root becomes the root -> label map once the boxes are out
    __device__ __forceinline__ void set_label(int b, int label) const { if constexpr (COMPACT) area[b] = (unsigned short)label; else stat[5 * b + 4] = label; }
    __device__ __forceinline__ int label(int b) const { return COMPACT ? (int)area[b] : stat[5 * b + 4]; }
};

// Phases 1 and 2 over one CTA's grid of blocks - the whole mask in ccl_bbox_kernel, one band of it in ccl_cluster_kernel.
// Afterwards parent[] is a forest over the grid whose roots are the first blocks (raster order) of its components, and
// my_list / the return value are the calling warp's list of foreground blocks.
template <bool COMPACT>
__device__ __forceinline__ int ccl_codes_and_merge(const CclArgs &A, const CclMem<COMPACT> &M, const uint8_t *m, int nb,
                                                   unsigned short *&my_list) {
    const int tid = threadIdx.x, nt = blockDim.x;
    uint8_t *code = M.code;
    // 1. 2x2 block codes: bit0 (0,0) bit1 (0,1) bit2 (1,0) bit3 (1,1).  Horizontal runs are linked here, without
    //    union-find: consecutive lanes hold consecutive blocks, so a warp ballot of "not connected to my west
    //    neighbour" gives every block the first block of its run inside the warp's 32-block segment as parent
    //    (depth 1).  Without this a run of n blocks is a chain of n links that every later find walks.
    const int lane = tid & 31;
    // no per-block division: (by, bx) of the thread's first block once, then incremental
    const int by_first = A.nbx > 1 ? (int)fast_div((uint32_t)tid, A.div_nbx) : tid;
    const int bx_first = tid - by_first * A.nbx;
    const bool w_even = (A.W & 1) == 0;          // then every 2x2 block row is one aligned 16-bit load
    // Foreground blocks are also appended to a list private to the warp (ballot + popcount, no cross-warp scan): the merge
    // and statistics passes below then run over lists of foreground blocks only, with full warps - on the masks the network
    // produces three blocks in four are background, and a warp that carries one foreground lane through a find loop pays
    // for 32.  A warp owns the 32-block segments base + 32*wid .. of every pass over the grid, i.e. a fine interleave of the
    // whole mask, so the lists are balanced.
    const int iters = (nb + nt - 1) / nt;
    my_list = M.list + (size_t)(tid >> 5) * iters * 32;
    int n_fg = 0;                                    // warp-uniform: entries in my_list
    int run_by = by_first, run_bx = bx_first;
    for (int base = 0; base < nb; base += nt) {
        const int b = base + tid;
        const int by = run_by, bx = run_bx;
        COVA_CCL_ADVANCE(run_by, run_bx);
        int c = 0;
        if (b < nb) {
            const int y = 2 * by, x = 2 * bx;
            const uint8_t *r0 = m + (unsigned)(y * A.W + x);           // one mask is far below 2^31 pixels: 32-bit offset
            const bool y1 = y + 1 < A.H;
            // plain (coherent) loads: under programmatic dependent launch the mask is written while this grid is
            // already resident, which rules out the read-only data path
            if (w_even) {
                const unsigned v0 = *reinterpret_cast<const unsigned short *>(r0);
                const unsigned v1 = y1 ? *reinterpret_cast<const unsigned short *>(r0 + A.W) : 0u;
                c = ((v0 & 0xffu) ? 1 : 0) | ((v0 >> 8) ? 2 : 0) | ((v1 & 0xffu) ? 4 : 0) | ((v1 >> 8) ? 8 : 0);
            } else {
                const bool x1 = x + 1 < A.W;
                c = (r0[0] != 0) ? 1 : 0;
                if (x1 && r0[1] != 0) c |= 2;
                if (y1 && r0[A.W] != 0) c |= 4;
                if (x1 && y1 && r0[A.W + 1] != 0) c |= 8;
            }
        }
        const int cw = __shfl_up_sync(0xffffffffu, c, 1);
        const bool west = lane > 0 && bx > 0 && (c & 0x5) && (cw & 0xA);       // my left column / its right column
        const unsigned starts = __ballot_sync(0xffffffffu, !west);              // bit 0 is always set
        if (b < nb) {
            const int start_lane = 31 - __clz((int)(starts & (0xffffffffu >> (31 - lane))));
            code[b] = (uint8_t)c;
            // (the tile scan makes its own runs per tile row: there every foreground block starts as its own root)
            M.parent[b] = (typename CclMem<COMPACT>::PT)(c ? (A.scan ? b : b - lane + start_lane) : CclMem<COMPACT>::kNone);
            if (c) M.stat_init(b);
        }
        const unsigned fg = __ballot_sync(0xffffffffu, c != 0);
        if (c) my_list[n_fg + __popc(fg & ((1u << lane) - 1u))] = (unsigned short)(b | (lane == 0 ? 0x8000 : 0));
        n_fg += __popc(fg);
    }
    __syncthreads();

    // 2. merge.
    if (A.scan) {
        // 2a. TILE SCAN.  A warp walks its tile (32 columns, lane = column) row by row.  Inside a row, runs come from one
        //     ballot; a run takes over the smallest root among the labels of the upper-row blocks it touches (north, north-
        //     west, north-east: shuffles of the previous row's registers, one short find each), spread over the run by a
        //     segmented min-scan of shuffles; only when a run touches two DIFFERENT roots is there a union to make.  Every
        //     block then points straight at its run's label.  No block-level union per adjacency, no divergent find loops
        //     over whole warps: on a dense 4K mask the old phase 2 was 70 % of the kernel (profiles/r2c_ccl_lines.txt).
        //     Links across tile borders are left to 2b.  Roots are still "the smallest block index of the component", so
        //     the label order contract (OpenCV's) is untouched.
        const int nwarps = nt >> 5, wid = tid >> 5;
        constexpr int kInf = 0x7fffffff;
        for (int tile = wid; tile < A.tiles_x * A.tiles_y; tile += nwarps) {
            const int ty = tile / A.tiles_x, tx = tile - ty * A.tiles_x;
            const int x = tx * 32 + lane;
            const bool inx = x < A.nbx;
            const int y_end = min(A.nby, (ty + 1) * A.tile_rows);
            int cu = 0, lu = kInf;                       // code and label of the block above (previous row of this tile)
            for (int y = ty * A.tile_rows; y < y_end; y++) {
                const int b = y * A.nbx + x;
                const int c = inx ? code[b] : 0;
                const int cl = __shfl_up_sync(0xffffffffu, c, 1);
                const int cul = __shfl_up_sync(0xffffffffu, cu, 1), cur = __shfl_down_sync(0xffffffffu, cu, 1);
                const int lul = __shfl_up_sync(0xffffffffu, lu, 1), lur = __shfl_down_sync(0xffffffffu, lu, 1);
                const bool west = lane > 0 && (c & 0x5) && (cl & 0xA);
                const unsigned starts = __ballot_sync(0xffffffffu, !west);                 // bit 0 is always set
                const int start_lane = 31 - __clz((int)(starts & (0xffffffffu >> (31 - lane))));
                const unsigned above = lane < 31 ? (starts & ~((2u << lane) - 1u)) : 0u;   // run starts to my right
                const int end_lane = above ? __ffs((int)above) - 2 : 31;
                int r0 = kInf, r1 = kInf, r2 = kInf;
                if (c) {
                    if ((c & 0x3) && (cu & 0xC)) r0 = M.find(lu);                           // north
                    if (lane > 0 && (c & 0x1) && (cul & 0x8)) r1 = M.find(lul);             // north-west
                    if (lane < 31 && (c & 0x2) && (cur & 0x4)) r2 = M.find(lur);            // north-east
                }
                int v = min(r0, min(r1, r2));
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {                                         // segmented min-scan from the run's first lane
                    const int o = __shfl_up_sync(0xffffffffu, v, d);
                    if (lane - d >= start_lane) v = min(v, o);
                }
                const int run_min = __shfl_sync(0xffffffffu, v, end_lane);
                int lab = kInf;
                if (c) {
                    if (run_min == kInf) {
                        lab = b - lane + start_lane;                                       // a run nothing above touches: its first block
                    } else {
                        lab = run_min;
                        if (r0 != kInf && r0 != run_min) M.unite(r0, run_min);
                        if (r1 != kInf && r1 != run_min) M.unite(r1, run_min);
                        if (r2 != kInf && r2 != run_min) M.unite(r2, run_min);
                    }
                    if (lab != b) M.lower(b, lab);
                }
                cu = c; lu = lab;
            }
        }
        __syncthreads();
        // 2b. links across tile borders, by the concurrent union-find: the first row of every row of tiles (north, north-west,
        //     north-east), the first column of every column of tiles (west, north-west), the last column (north-east)
        //     The border blocks are enumerated by geometry (a few hundred of the thousands of foreground blocks; walking the
        //     whole foreground list for them cost a quarter of the kernel on dense 4K masks): first the rows that start a row
        //     of tiles, then the two columns on either side of every vertical tile border.
        {
            const int n_row = (A.tiles_y - 1) * A.nbx, n_col = (A.tiles_x - 1) * 2 * A.nby;
            for (int i = tid; i < n_row + n_col; i += nt) {
                int by, bx;
                bool row0 = false, col0 = false, col31 = false;
                if (i < n_row) {
                    const int t = A.nbx > 1 ? (int)fast_div((uint32_t)i, A.div_nbx) : i;
                    by = (t + 1) * A.tile_rows; bx = i - t * A.nbx;
                    row0 = true;
                    col0 = bx > 0 && (bx & 31) == 0; col31 = (bx & 31) == 31 && bx + 1 < A.nbx;
                } else {
                    const int e = i - n_row, t = e / (2 * A.nby), rem = e - t * 2 * A.nby;      // one division per border block
                    by = rem >> 1;
                    bx = (t + 1) * 32 - (rem & 1);                                              // column 31 of tile t, column 0 of tile t+1
                    if (rem & 1) col31 = bx + 1 < A.nbx; else col0 = true;
                    if (by > 0 && (A.tile_rows == 1 || by - (int)fast_div((uint32_t)by, A.div_tile_rows) * A.tile_rows == 0)) continue;   // done as a row block
                }
                if (by >= A.nby || bx >= A.nbx) continue;
                const int b = by * A.nbx + bx;
                const int c = code[b];
                if (!c) continue;
                if (col0 && (c & 0x5) && (code[b - 1] & 0xA)) M.unite(b, b - 1);
                if (by > 0) {
                    const int u = b - A.nbx;
                    if (row0 && (c & 0x3) && (code[u] & 0xC)) M.unite(b, u);
                    if ((row0 || col0) && bx > 0 && (c & 0x1) && (code[u - 1] & 0x8)) M.unite(b, u - 1);
                    if ((row0 || col31) && bx + 1 < A.nbx && (c & 0x2) && (code[u + 1] & 0x4)) M.unite(b, u + 1);
                }
            }
        }
        __syncthreads();
    } else {
    // 2 (alternative). merge with the raster-preceding neighbour blocks: north, north-west, north-east, and west across a warp
    //    segment boundary (lane 0 could not see its west neighbour in step 1)
    for (int k = lane; k < n_fg; k += 32) {
        const int e = my_list[k], b = e & 0x7fff;
        const int c = code[b];
        const int by = A.nbx > 1 ? (int)fast_div((uint32_t)b, A.div_nbx) : b, bx = b - by * A.nbx;
        const int cw = bx > 0 ? code[b - 1] : 0;
        const bool west_b = (c & 0x5) && (cw & 0xA);                                           // b-1 ~ b along the row
        if ((e & 0x8000) && west_b) M.unite(b, b - 1);
        if (by > 0) {
            const int u = b - A.nbx;
            const int cu = code[u];
            const int cuw = bx > 0 ? code[u - 1] : 0, cue = bx + 1 < A.nbx ? code[u + 1] : 0;
            const bool n = (c & 0x3) && (cu & 0xC);                                            // north: my top row / its bottom row
            const bool west_u = (cu & 0x5) && (cuw & 0xA), west_ue = (cue & 0x5) && (cu & 0xA);   // u-1 ~ u, u ~ u+1
            const bool n_w = west_b && (cw & 0x3) && (cuw & 0xC);                              // b ~ b-1 and b-1 has its own north link
            // Links that other links imply are skipped (every union costs two finds).  All links of the phase are in place
            // at its closing barrier, so transitivity may lean on links other threads make:
            //   north:      b ~ b-1 ~ u-1 ~ u   when the west neighbour has a north link and the two north blocks are joined
            //               - on a dense mask only the first block of every run-to-run contact is left;
            //   north-west: b ~ u ~ u-1, or b ~ b-1 ~ u-1;     north-east: b ~ u ~ u+1
            const bool do_n = n && !(n_w && west_u);
            const bool nw = (c & 0x1) && (cuw & 0x8) && !(n && west_u) && !n_w;
            const bool ne = (c & 0x2) && (cue & 0x4) && !(n && west_ue);
            if (do_n) M.unite(b, u);
            if (nw) M.unite(b, u - 1);
            if (ne) M.unite(b, u + 1);
        }
    }
    __syncthreads();

    }
    return n_fg;
}

template <bool COMPACT>
__global__ void ccl_bbox_kernel(CclArgs A) {
    extern __shared__ __align__(16) unsigned char ccl_smem[];
    const int nb = A.nbx * A.nby;
    const CclMem<COMPACT> M(ccl_smem, nb, (int)blockDim.x);
    uint8_t *code = M.code;
    int *scan = M.scan;
    __shared__ unsigned long long s_off;

    const int frame = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    pdl_launch_dependents();
    pdl_wait();              // the mask comes from the preceding kernel of the stream (common.cuh, "Programmatic dependent launch")
    const uint8_t *m = A.masks + (size_t)frame * A.H * A.W;
    const int thresh = A.thresh ? __ldg(A.thresh + frame) : A.area_thresh;

    unsigned short *my_list;
    const int n_fg = ccl_codes_and_merge<COMPACT>(A, M, m, nb, my_list);
    const int lane = tid & 31;

    // 3. flatten + per-root statistics.  parent[b] is lowered to the root while other threads may still walk through b in
    //    their own find: they read either b's old parent (an ancestor) or its root and reach the same root either way.
    //    (compute-sanitizer --tool racecheck: clean.)
    //    A component that covers much of the mask would put thousands of atomics on the same five words, one after the
    //    other (a 4K all-ones mask: 8160 x 5).  When at least a quarter of a warp shares the root of its first lane those
    //    lanes are combined first (ballot + redux, one lane speaks); a full match.any over all roots was also tried and
    //    costs the many-small-components masks more than it saves (720p network masks 0.155 -> 0.183 ms).
    for (int k0 = 0; k0 < n_fg; k0 += 32) {                         // warp-uniform trip count
        const int k = k0 + lane;
        const bool live = k < n_fg;
        int r = -1 - lane, x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1, cnt = 0;     // dead lanes: a group of their own
        if (live) {
            const int b = my_list[k] & 0x7fff;
            const int c = code[b];
            const int by = A.nbx > 1 ? (int)fast_div((uint32_t)b, A.div_nbx) : b, bx = b - by * A.nbx;
            r = M.find(b);
            M.lower(b, r);
            x0 = 2 * bx + ((c & 0x5) ? 0 : 1); x1 = 2 * bx + ((c & 0xA) ? 1 : 0);
            y0 = 2 * by + ((c & 0x3) ? 0 : 1); y1 = 2 * by + ((c & 0xC) ? 1 : 0);
            cnt = __popc(c);
        }
        const int r_lead = __shfl_sync(0xffffffffu, r, 0);         // lane 0 is live in every iteration
        const unsigned grp = __ballot_sync(0xffffffffu, r == r_lead);
        bool speak = live;
        if (__popc(grp) >= 8) {                                     // warp-uniform
            if (r == r_lead) {
                x0 = __reduce_min_sync(grp, x0); y0 = __reduce_min_sync(grp, y0);
                x1 = __reduce_max_sync(grp, x1); y1 = __reduce_max_sync(grp, y1);
                cnt = __reduce_add_sync(grp, cnt);
                speak = lane == 0;
            }
        }
        if (speak) M.stat_add(r, x0, y0, x1, y1, cnt);
    }
    __syncthreads();

    // 4. rank the roots in block-raster order: hi16 = all components, lo16 = components passing the filter
    const int ipt = (nb + nt - 1) / nt;
    const int b0 = min(tid * ipt, nb), b1 = min(b0 + ipt, nb);
    int cnt = 0;
    for (int b = b0; b < b1; b++)
        if ((int)M.parent[b] == b) cnt += 0x10000 + (M.stat_area(b) >= thresh ? 1 : 0);
    int incl = cnt;
    const int wid = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) scan[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int nw = nt >> 5;
        int v = lane < nw ? scan[lane] : 0, s = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int u = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += u;
        }
        if (lane < nw) scan[lane] = s - v;   // exclusive warp offsets
        if (lane == 31) scan[nw] = s;        // grand total
    }
    __syncthreads();
    const int total = scan[nt >> 5];
    const int n_all = total >> 16, n_keep = total & 0xffff;
    int excl = scan[wid] + incl - cnt;

    // 5. reserve the output range
    const unsigned long long need = 8ull + 24ull * (unsigned long long)n_keep;
    if (tid == 0) {
        unsigned long long off = atomicAdd(A.cursor, need);
        s_off = off;
        A.offsets[frame] = off;
        A.lens[frame] = need;
        if (off + need > A.blob_cap) atomicExch(A.cursor + 1, 1ull);
        if (A.n_labels) A.n_labels[frame] = n_all + 1;
    }
    __syncthreads();
    const unsigned long long off = s_off;
    const bool fits = off + need <= A.blob_cap;
    if (tid == 0 && fits) *reinterpret_cast<unsigned long long *>(A.blob + off) = (unsigned long long)n_keep;
    int32_t *st = A.stats ? A.stats + (size_t)frame * (nb + 1) * 5 : nullptr;
    if (st && tid < 5) st[tid] = 0;

    // 6. emit boxes in label order; turn the area slot into the root -> label map
    int rank_all = excl >> 16, rank_keep = excl & 0xffff;
    for (int b = b0; b < b1; b++) {
        if ((int)M.parent[b] != b) continue;
        int x0, y0, x1, y1;
        M.stat_get(b, x0, y0, x1, y1);
        const int w = x1 - x0 + 1, h = y1 - y0 + 1, ar = M.stat_area(b);
        rank_all++;
        if (st) {
            int32_t *s5 = st + (size_t)rank_all * 5;
            s5[0] = x0; s5[1] = y0; s5[2] = w; s5[3] = h; s5[4] = ar;
        }
        if (ar >= thresh) {
            if (fits) {
                uint32_t *rec = reinterpret_cast<uint32_t *>(A.blob + off + 8 + 24ull * rank_keep);
                float fw = (float)w, fh = (float)h;
                rec[0] = __float_as_uint((float)x0);
                rec[1] = __float_as_uint((float)y0);
                rec[2] = __float_as_uint(fw);
                rec[3] = __float_as_uint(fh);
                rec[4] = __float_as_uint(fw * fh);   // bbox.rs:23
                rec[5] = 0u;                         // track_id, timestamp, class_id, confidence = None
            }
            rank_keep++;
        }
        M.set_label(b, rank_all);
    }
    if (!A.labels) return;
    __syncthreads();
    int32_t *lab = A.labels + (size_t)frame * A.H * A.W;
    for (int p = tid; p < A.H * A.W; p += nt) {
        int y = p / A.W, x = p - y * A.W;
        int b = (y >> 1) * A.nbx + (x >> 1);
        lab[p] = (m[p] != 0) ? M.label((int)M.parent[b]) : 0;
    }
}

inline int ccl_threads_for(int nb) { return nb <= 1024 ? 256 : (nb <= 4096 ? 512 : 1024); }

// =====================================================================================================================
// Thread-block-cluster CCL for masks whose blocks do not fit one CTA's shared memory (8K video: 480 x 270 macroblocks =
// 32,400 blocks, 876 KB in the wide layout).  One cluster of k CTAs per mask; rank r owns the block rows
// [r * rows, min((r + 1) * rows, nby)), a band that is itself a grid of the single-CTA kind (at 8K: 4 bands of at most
// 34 x 240 = 8,160 blocks, exactly the 4K problem).  Phases 1-2 run per band with ccl_codes_and_merge on band-local
// indices; then the parents become GLOBAL block indices (band offset + local index) and everything else works on the
// whole mask through distributed shared memory: the seams between bands are linked by the same lock-free union-find
// (compare-and-swap links of the larger root under the smaller, compression only towards ancestors), so a component's
// root is still its first block in raster order over the whole mask and the label order stays OpenCV's with no sort.
// Every CTA lays its shared memory out for a full band (CclMem of rows * nbx blocks), the last one included, so a
// global index g lives at offset g - q * band_nb of rank q = g / band_nb's arrays, at the same addresses in every CTA.
// =====================================================================================================================
struct CclClusterArgs {
    CclArgs band[2];          // [0]: ranks 0 .. k-2 (`rows` block rows, 2 * rows pixel rows), [1]: the last rank
    int H;                    // pixel rows of the whole mask
    int nb;                   // blocks of the whole mask
    int rows, band_nb;        // block rows and blocks of every band but the last
    FastDiv div_band;         // by band_nb (when band_nb >= 2)
};

namespace ccl_cluster_detail {
namespace cg = cooperative_groups;

// union-find and statistics over the global block indices of the cluster's mask; every access may land in a peer CTA
struct Global {
    cg::cluster_group cl;
    int *parent, *stat;       // this CTA's arrays (the same offsets in every CTA of the cluster)
    int band_nb;
    FastDiv div_band;

    __device__ __forceinline__ int owner(int g) const { return band_nb > 1 ? (int)fast_div((uint32_t)g, div_band) : g; }
    __device__ __forceinline__ int *par(int g) const {
        const int q = owner(g);
        return cl.map_shared_rank(parent, (unsigned)q) + (g - q * band_nb);
    }
    __device__ __forceinline__ int *st(int g) const {
        const int q = owner(g);
        return cl.map_shared_rank(stat, (unsigned)q) + 5 * (g - q * band_nb);
    }
    __device__ __forceinline__ int load(int g) const { return *reinterpret_cast<volatile int *>(par(g)); }
    __device__ __forceinline__ int find(int g) const {
        int p;
        while ((p = load(g)) != g) g = p;
        return g;
    }
    // CclMem::find_compress / unite over the whole mask: the same invariants (see there)
    __device__ __forceinline__ int find_compress(int i) const {
        int r = load(i);
        if (r == i) return i;
        int p, hops = 0;
        while ((p = load(r)) != r) { r = p; hops++; }
        if (hops) {
            int j = i;
            while ((p = load(j)) > r) {
                atomicMin(par(j), r);
                j = p;
            }
        }
        return r;
    }
    __device__ __forceinline__ void unite(int a, int b) const {
        while (true) {
            a = find_compress(a);
            b = find_compress(b);
            if (a == b) return;
            if (a < b) { int t = a; a = b; b = t; }
            const int old = atomicCAS(par(a), a, b);
            if (old == a) return;
            a = old;
        }
    }
    __device__ __forceinline__ void stat_add(int r, int x0, int y0, int x1, int y1, int cnt) const {
        int *sr = st(r);
        atomicMin(&sr[0], x0); atomicMax(&sr[2], x1);
        atomicMin(&sr[1], y0); atomicMax(&sr[3], y1);
        atomicAdd(&sr[4], cnt);
    }
    __device__ __forceinline__ int label(int g) const { return st(g)[4]; }
};
}  // namespace ccl_cluster_detail

__global__ void ccl_cluster_kernel(const __grid_constant__ CclClusterArgs C) {
    namespace cg = cooperative_groups;
    extern __shared__ __align__(16) unsigned char ccl_smem[];
    __shared__ unsigned long long s_off;
    __shared__ int s_cnt[2];            // roots of this band: all, passing the area filter (read by the peers)
    __shared__ int s_base[4];           // components of the earlier bands (all, kept) and of the whole mask (all, kept)
    const cg::cluster_group cl = cg::this_cluster();
    const int rank = (int)cl.block_rank(), k = (int)cl.num_blocks();
    const CclArgs &A = C.band[rank == k - 1 ? 1 : 0];
    const int nb = A.nbx * A.nby;                      // blocks of this band
    const CclMem<false> M(ccl_smem, C.band_nb, (int)blockDim.x);
    int *scan = M.scan;
    const ccl_cluster_detail::Global G{cl, M.parent, M.stat, C.band_nb, C.div_band};

    const int frame = blockIdx.x / k;                  // a cluster is k consecutive CTAs along x
    const int tid = threadIdx.x, nt = blockDim.x;
    const int row0 = rank * C.rows, off = row0 * A.nbx;
    pdl_launch_dependents();
    pdl_wait();
    const uint8_t *m = A.masks + (size_t)frame * C.H * A.W + (size_t)2 * row0 * A.W;
    const int thresh = A.thresh ? __ldg(A.thresh + frame) : A.area_thresh;

    // 1-2. codes, runs and merge inside the band, on band-local indices (in-band links never leave the band)
    unsigned short *my_list;
    const int n_fg = ccl_codes_and_merge<false>(A, M, m, nb, my_list);
    const int lane = tid & 31;
    for (int i = lane; i < n_fg; i += 32) M.parent[my_list[i] & 0x7fff] += off;    // -> global indices, order kept
    cl.sync();                                         // also: every peer has started, its shared memory may be touched

    // 2c. seams: this band's first block row against the last row of the band above (north, north-west, north-east)
    if (rank > 0) {
        const uint8_t *up = cl.map_shared_rank(M.code, (unsigned)(rank - 1)) + (C.rows - 1) * A.nbx;
        for (int bx = tid; bx < A.nbx; bx += nt) {
            const int c = M.code[bx];
            if (!c) continue;
            const int g = off + bx, gu = off - A.nbx + bx;
            if ((c & 0x3) && (up[bx] & 0xC)) G.unite(g, gu);
            if (bx > 0 && (c & 0x1) && (up[bx - 1] & 0x8)) G.unite(g, gu - 1);
            if (bx + 1 < A.nbx && (c & 0x2) && (up[bx + 1] & 0x4)) G.unite(g, gu + 1);
        }
    }
    cl.sync();

    // 3. flatten + statistics into the owner CTA's slots (as in ccl_bbox_kernel; the warp combining matters more here:
    //    a component across a seam would otherwise send thousands of remote atomics to the same five words)
    for (int k0 = 0; k0 < n_fg; k0 += 32) {
        const int kk = k0 + lane;
        const bool live = kk < n_fg;
        int r = -1 - lane, x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1, cnt = 0;
        if (live) {
            const int b = my_list[kk] & 0x7fff;
            const int c = M.code[b];
            const int by = A.nbx > 1 ? (int)fast_div((uint32_t)b, A.div_nbx) : b, bx = b - by * A.nbx;
            r = G.find(off + b);
            atomicMin(&M.parent[b], r);
            x0 = 2 * bx + ((c & 0x5) ? 0 : 1); x1 = 2 * bx + ((c & 0xA) ? 1 : 0);
            y0 = 2 * (row0 + by) + ((c & 0x3) ? 0 : 1); y1 = 2 * (row0 + by) + ((c & 0xC) ? 1 : 0);
            cnt = __popc(c);
        }
        const int r_lead = __shfl_sync(0xffffffffu, r, 0);
        const unsigned grp = __ballot_sync(0xffffffffu, r == r_lead);
        bool speak = live;
        if (__popc(grp) >= 8) {
            if (r == r_lead) {
                x0 = __reduce_min_sync(grp, x0); y0 = __reduce_min_sync(grp, y0);
                x1 = __reduce_max_sync(grp, x1); y1 = __reduce_max_sync(grp, y1);
                cnt = __reduce_add_sync(grp, cnt);
                speak = lane == 0;
            }
        }
        if (speak) G.stat_add(r, x0, y0, x1, y1, cnt);
    }
    cl.sync();

    // 4. rank this band's roots (hi16 all, lo16 kept: a band has fewer than 2^15 blocks), then across the cluster in 32 bits
    const int ipt = (nb + nt - 1) / nt;
    const int b0 = min(tid * ipt, nb), b1 = min(b0 + ipt, nb);
    int cnt = 0;
    for (int b = b0; b < b1; b++)
        if (M.parent[b] == off + b) cnt += 0x10000 + (M.stat[5 * b + 4] >= thresh ? 1 : 0);
    int incl = cnt;
    const int wid = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) scan[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int nw = nt >> 5;
        int v = lane < nw ? scan[lane] : 0, s = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int u = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += u;
        }
        if (lane < nw) scan[lane] = s - v;
        if (lane == 31) { s_cnt[0] = s >> 16; s_cnt[1] = s & 0xffff; }
    }
    cl.sync();
    const int excl = scan[wid] + incl - cnt;
    if (tid == 0) {
        int all_before = 0, keep_before = 0, n_all = 0, n_keep = 0;
        for (int q = 0; q < k; q++) {
            const int *pc = cl.map_shared_rank(s_cnt, (unsigned)q);
            const int a = pc[0], kp = pc[1];
            if (q < rank) { all_before += a; keep_before += kp; }
            n_all += a; n_keep += kp;
        }
        s_base[0] = all_before; s_base[1] = keep_before; s_base[2] = n_all; s_base[3] = n_keep;
        // 5. rank 0 reserves the mask's output range and publishes its offset into every CTA of the cluster
        if (rank == 0) {
            const unsigned long long need = 8ull + 24ull * (unsigned long long)n_keep;
            const unsigned long long o = atomicAdd(A.cursor, need);
            A.offsets[frame] = o;
            A.lens[frame] = need;
            if (o + need > A.blob_cap) atomicExch(A.cursor + 1, 1ull);
            if (A.n_labels) A.n_labels[frame] = n_all + 1;
            if (o + need <= A.blob_cap) *reinterpret_cast<unsigned long long *>(A.blob + o) = (unsigned long long)n_keep;
            for (int q = 0; q < k; q++) *cl.map_shared_rank(&s_off, (unsigned)q) = o;
        }
    }
    cl.sync();
    const unsigned long long off_out = s_off;
    const unsigned long long need = 8ull + 24ull * (unsigned long long)s_base[3];
    const bool fits = off_out + need <= A.blob_cap;
    int32_t *st = A.stats ? A.stats + (size_t)frame * (C.nb + 1) * 5 : nullptr;
    if (st && rank == 0 && tid < 5) st[tid] = 0;

    // 6. emit this band's boxes at its base; the area slot of a root becomes the root -> label map
    int rank_all = s_base[0] + (excl >> 16), rank_keep = s_base[1] + (excl & 0xffff);
    for (int b = b0; b < b1; b++) {
        if (M.parent[b] != off + b) continue;
        int x0, y0, x1, y1;
        M.stat_get(b, x0, y0, x1, y1);
        const int w = x1 - x0 + 1, h = y1 - y0 + 1, ar = M.stat_area(b);
        rank_all++;
        if (st) {
            int32_t *s5 = st + (size_t)rank_all * 5;
            s5[0] = x0; s5[1] = y0; s5[2] = w; s5[3] = h; s5[4] = ar;
        }
        if (ar >= thresh) {
            if (fits) {
                uint32_t *rec = reinterpret_cast<uint32_t *>(A.blob + off_out + 8 + 24ull * rank_keep);
                float fw = (float)w, fh = (float)h;
                rec[0] = __float_as_uint((float)x0);
                rec[1] = __float_as_uint((float)y0);
                rec[2] = __float_as_uint(fw);
                rec[3] = __float_as_uint(fh);
                rec[4] = __float_as_uint(fw * fh);   // bbox.rs:23
                rec[5] = 0u;
            }
            rank_keep++;
        }
        M.set_label(b, rank_all);
    }
    if (!A.labels) return;             // no CTA reads a peer's shared memory after the last barrier
    cl.sync();                         // every label map of the cluster is written
    int32_t *lab = A.labels + (size_t)frame * C.H * A.W + (size_t)2 * row0 * A.W;
    for (int p = tid; p < A.H * A.W; p += nt) {
        int y = p / A.W, x = p - y * A.W;
        int b = (y >> 1) * A.nbx + (x >> 1);
        lab[p] = (m[p] != 0) ? G.label(M.parent[b]) : 0;
    }
    cl.sync();                         // no CTA leaves while a peer may still read its label map
}

}  // namespace cova
