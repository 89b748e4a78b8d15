// scan3d_internal.h -- context layout and kernel launcher declarations (not part of the ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/scan3d.h"
#include "scan3d_device_buffer.h"
#include "scan3d_math.cuh"
#include "scan3d_results.h"

#define S3D_PLANE_MASK_H 10   // internal: valid_map_horizontal when the stage API is used

namespace s3h {
struct Cell;                  // common/scan3d_fill_math.h
}

namespace s3d {
// tensor maps of the last few capture stacks (a map depends on the stack's address and the tile size only)
struct TensorMapCache {
    static constexpr int SLOTS = 8;
    const uint8_t* stack[SLOTS] = {};
    int box[SLOTS] = {};
    alignas(64) CUtensorMap map[SLOTS];
    int next = 0;
};

// Each stage on the merged model owns its device scratch in a workspace below.  The workspace's functions, defined next
// to the stage's kernels, grow the scratch, clear what the kernels need cleared and launch.  A function or launcher
// with an int64_t* launches argument adds the kernels it launches to *launches.

// the voxel-grid merge's hash table (scan3d_voxel_kernels.cu)
constexpr uint32_t VOXEL_NO_SLOT = 0xffffffffu;   // no slot / no ordinal yet
// the integer sums of one voxel (zero-initialised); first_inv = ~(index of the first point within the current add)
struct VoxelSlot {
    unsigned long long q[3];   // positions inside the voxel, Q steps
    unsigned long long m[3];   // normals, Q steps, two's complement
    unsigned long long c[3];   // colours
    uint32_t n, first_inv;
};
struct VoxelState {
    unsigned long long dropped;
    uint32_t occupied;         // slots taken = distinct voxels inserted
    uint32_t overflow;         // an ordinal >= max_voxels was assigned
    uint32_t total[2];         // voxels with an ordinal, after an even / odd number of adds (chunks)
    uint32_t chunk_new;        // new voxels of the current add (chunk)
    uint32_t pad;
};
struct VoxelTable {
    unsigned long long* keys;  // [cap], s3v::EMPTY_KEY = free
    VoxelSlot* acc;            // [cap]
    uint32_t* ordinal;         // [cap], VOXEL_NO_SLOT until assigned
    uint32_t* ord2slot;        // [max_voxels]
    VoxelState* state;
    uint32_t cap, max_voxels;
    double S;                  // (double)voxel_size
};
// One voxel hash table and its kernels' view: the merge's accumulator and the simplification's clusters.
struct VoxelStore {
    DeviceBuffer<unsigned long long> keys;
    DeviceBuffer<VoxelSlot> acc;
    DeviceBuffer<uint32_t> ordinal;
    DeviceBuffer<uint32_t> ord2slot;
    DeviceBuffer<VoxelState> state;
    VoxelTable view{};
    // an empty table for max_voxels voxels of edge S: grown, the view set, keys and ordinals 0xff, sums and state 0
    cudaError_t reset(uint32_t max_voxels, double S, int sm_count, cudaStream_t st);
};

// the alignment's cell index of the model (scan3d_align_kernels.cu)
struct AlignIndex {
    unsigned long long* keys;  // [cap], s3v::EMPTY_KEY = free; key = s3v::pack_key of the cell
    uint2* cells;              // [cap] (points in the cell, end of its range in entries)
    uint32_t* model_slot;      // [max_voxels] cell slot of each voxel, VOXEL_NO_SLOT = not in the model
    float4* entries;           // [2 max_voxels] per model point: (x, y, z, ordinal bits), (nx, ny, nz, 0)
    uint32_t* cursor;          // [1]
    uint32_t cap;
};
// the device state of one alignment run
struct AlignState {
    double T[12];              // current estimate [R | t], row-major
    double rms_first, rms_last;
    long long pairs_first, pairs_last;
    int iterations, status, done, rounds;   // updates applied, scan3d_align_result.status, run ended, solves run
    int overflow;              // the voxel accumulator overflowed (read when the index is built)
    uint32_t n_src;            // the ctx route's point count (read when the index is built)
};
struct AlignRun {
    double T0[12];             // T_init
    double S;                  // cell edge
    double r2;                 // max_distance^2
    double stop_rotation, stop_translation;
    int max_iterations;
};
// The alignment's cell index of the merged model, the state of one run and the match partials.  The model is the first
// min(total, max_voxels) voxel outputs (xyz, nrm [max_voxels][3]) of t, total = t.state->total[par].
struct AlignWorkspace {
    DeviceBuffer<unsigned long long> keys;   // [2 max_voxels]
    DeviceBuffer<uint2> cells;               // [2 max_voxels]
    DeviceBuffer<uint32_t> model_slot;       // [max_voxels]
    DeviceBuffer<float4> entries;            // [2 max_voxels]
    DeviceBuffer<uint32_t> cursor;           // [1]
    DeviceBuffer<double> partials;           // [sums + 1][blocks]
    DeviceBuffer<AlignState> state;
    AlignIndex view{};
    // the index of cell edge run.S, 3 launches: cell keys and counts (which also initialises state from run, the voxel
    // overflow flag and, when n_dev is set, the source count), cell ranges, scatter of the model points
    cudaError_t index(const VoxelTable& t, int par, const float* xyz, const float* nrm, const AlignRun& run,
                      const uint32_t* n_dev, int sm_count, cudaStream_t st, int64_t* launches);
    // the index, then one match + one solve launch per iteration.  The source is src[i * stride] for i * stride < n,
    // n = min(*n_dev, n_max) when n_dev is set, else n_max; the grid depends on n_max and stride only.
    cudaError_t align(const VoxelTable& t, int par, const float* xyz, const float* nrm, const AlignRun& run,
                      const float* src, const uint32_t* n_dev, long long n_max, int stride, int sm_count,
                      cudaStream_t st, int64_t* launches);
};

// the surface extraction's lattice table (scan3d_surface_kernels.cu), one slot per distinct lattice point
struct SurfaceState {
    unsigned long long undefined;  // lattice points without a model point within max_distance
    uint32_t occupied;             // slots taken = distinct lattice points
    uint32_t overflow;             // an insert found no free slot, or a vertex ordinal reached max_points
    uint32_t vertices, faces;
};
struct SurfaceTable {
    unsigned long long* keys;      // [cap] s3v::pack_key of the lattice point, s3v::EMPTY_KEY = free
    unsigned long long* owner;     // [cap] min(27 o + k) of a candidate cell, ~0 = not a candidate
    double* f;                     // [cap] corner value
    uint32_t* nearest;             // [cap] ordinal of the nearest model point, VOXEL_NO_SLOT = f undefined
    uint32_t* vert;                // [cap] VOXEL_NO_SLOT = not an active cell, else its vertex ordinal
    SurfaceState* state;
    uint32_t cap, max_points;
    double S;                      // (double)voxel_size
};
// A triangle surface.  The context holds two: the held surface and the spare set, which the stage that replaces the
// held surface writes before the two are swapped.
struct SurfaceMesh {
    DeviceBuffer<float> xyz, nrm;  // [vertices][3]
    DeviceBuffer<uint8_t> rgb;     // [vertices][3]
    DeviceBuffer<int32_t> tri;     // [faces][3]
    int64_t vertices = 0, faces = 0;
    cudaError_t grow(size_t nv, size_t nf)
    {
        const cudaError_t e = grow_group(Grow(xyz, 3 * nv), Grow(nrm, 3 * nv), Grow(rgb, 3 * nv));
        return e != cudaSuccess ? e : tri.ensure(3 * nf);
    }
    // positions and normals only: the smoothing writes nothing else
    cudaError_t grow_positions(size_t nv) { return grow_group(Grow(xyz, 3 * nv), Grow(nrm, 3 * nv)); }
};
// The lattice table and the vertex scratch of the surface extraction.
struct SurfaceWorkspace {
    DeviceBuffer<unsigned long long> keys, owner;  // [cap]
    DeviceBuffer<double> f;                        // [cap]
    DeviceBuffer<uint32_t> nearest, vert;          // [cap]
    DeviceBuffer<SurfaceState> state;
    DeviceBuffer<uint8_t> flags;                   // [27 max_voxels] (o, k) owns an active cell
    DeviceBuffer<uint32_t> flag_counts;            // [cdiv(27 max_voxels, POINT_BLOCK) + 1]
    DeviceBuffer<uint32_t> vert_slot;              // [max_points] lattice slot of each vertex
    DeviceBuffer<uint32_t> face_counts;            // [cdiv(max_points, vertex block) + 1] faces per block, then offsets
    SurfaceTable view{};
    // 8 launches after ix was built from t's model with cell edge s3l::cell_edge(max_distance): candidate cells (27 per
    // model voxel, with their order key), their other 7 corners, the corner values, the (o, k) flags of active cells,
    // k_count + k_scan over them (the vertex ordinals), vertex assignment with the faces per block of vertices, and the
    // scan of those; state->vertices and state->faces are then known
    cudaError_t count(const AlignIndex& ix, const VoxelTable& t, int par, const float* vox_nrm, float max_distance,
                      uint32_t max_points, int sm_count, cudaStream_t st, int64_t* launches);
    // 1 launch: the vertices (xyz, normals, rgb) and faces into out
    cudaError_t emit(const uint8_t* vox_rgb, uint32_t vertices, SurfaceMesh& out, cudaStream_t st, int64_t* launches);
};

// the connected components of a triangle mesh (scan3d_components_kernels.cu)
struct ComponentsState {
    unsigned long long threshold;  // K of the keep rule: component c is kept when eligible and its key is >= K
    uint32_t components;           // of the mesh
    uint32_t kept, largest;        // components kept; the most faces of one component
    uint32_t vertices, faces;      // kept
    uint32_t bad;                  // a face index outside [0, vertices)
    uint32_t pad;
};
// The union-find scratch and the component table.
struct ComponentsWorkspace {
    DeviceBuffer<uint32_t> parent;       // [vertices] union-find forest, then each vertex's root
    DeviceBuffer<uint8_t> flags;         // [vertices] root flags, then the vertices' keep flags
    DeviceBuffer<uint32_t> vert_counts;  // [cdiv(vertices, POINT_BLOCK) + 1] block offsets of the flags
    DeviceBuffer<int32_t> label;         // [vertices] component ids, then the kept vertices' new indices
    DeviceBuffer<uint32_t> comp_v;       // [vertices] per component: vertices, faces, kept flag
    DeviceBuffer<uint32_t> comp_f;
    DeviceBuffer<uint8_t> kept;
    DeviceBuffer<uint8_t> keep_f;        // [faces]
    DeviceBuffer<uint32_t> face_counts;  // [cdiv(faces, POINT_BLOCK) + 1]
    DeviceBuffer<ComponentsState> state;
    // 7 launches for n vertices and n_faces faces [n_faces][3]: parent = v, union per face, find per vertex with the
    // root flags, k_count + k_scan over them (state->components), the roots' ids, every vertex's id into out [n].  Any
    // n below 2^31 and n_faces below 2^32, 0 included.
    cudaError_t labels(const int32_t* faces, uint32_t n_faces, uint32_t n, int32_t* out, cudaStream_t st,
                       int64_t* launches);
    // 14 launches on the mesh of in: its labels, then vertices and faces per component, the selection
    // (state->threshold, kept, largest), the keep flags, k_count + k_scan over each of the vertex flags
    // (state->vertices) and the face flags (state->faces)
    cudaError_t select(const SurfaceMesh& in, unsigned long long min_faces, unsigned long long max_components,
                       cudaStream_t st, int64_t* launches);
    // 2 launches after select: the kept vertices of in into out (their new indices into label), then the kept faces,
    // remapped
    cudaError_t emit(const SurfaceMesh& in, SurfaceMesh& out, cudaStream_t st, int64_t* launches);
};

// the surface simplification (scan3d_decimate_kernels.cu); the clusters are a second VoxelStore
struct DecimateState {
    uint32_t collapsed;            // faces with two corners in one cluster
    uint32_t fallbacks;            // clusters placed at their mean after a failed solve
    uint32_t faces;                // kept faces
    uint32_t zero;                 // stays 0: the vertex count of an empty surface's voxel add
};
struct DecimateWorkspace {
    VoxelStore clusters;                    // edge H, max_voxels = the vertex count
    DeviceBuffer<uint32_t> point_slot;      // [vertices] cluster slot of each vertex
    DeviceBuffer<uint8_t> vert_flags;       // [vertices]
    DeviceBuffer<uint32_t> vert_counts;     // [cdiv(vertices, POINT_BLOCK) + 1]
    DeviceBuffer<unsigned long long> quad;  // [vertices][10] quadric sums per cluster ordinal (int64 two's complement)
    DeviceBuffer<int32_t> ctri;             // [faces][3] cluster ordinals of the corners
    DeviceBuffer<uint32_t> table;           // [2 faces] face indices, VOXEL_NO_SLOT = free
    DeviceBuffer<uint32_t> slot_of;         // [faces] table slot of each face, VOXEL_NO_SLOT = collapsed
    DeviceBuffer<uint8_t> keep;             // [faces]
    DeviceBuffer<uint32_t> face_counts;     // [cdiv(faces, POINT_BLOCK) + 1]
    DeviceBuffer<DecimateState> state;
    // 12 launches for the surface in: the merge's voxel add over its vertices into the clusters, the face quadrics
    // with the cluster triples, the duplicate-face table, the keep flags, k_count + k_scan over them (state->faces),
    // then the vertices of the clusters (clusters.state->total[1] of them) and the kept faces into out, which holds
    // in's counts
    cudaError_t run(const SurfaceMesh& in, double H, SurfaceMesh& out, int sm_count, cudaStream_t st,
                    int64_t* launches);
};

// the surface smoothing (scan3d_smooth_kernels.cu); the undirected edges are a hash of (min << 32 | max) keys
struct SmoothState {
    unsigned long long max_move;   // bits of the largest displacement (a non-negative double, so the bits order it)
    uint32_t exp_field;            // the largest biased float exponent field of the coordinates
    uint32_t bad;                  // a coordinate not finite or a face index outside [0, vertices): SCAN3D_ERR_ARG
    uint32_t overflow;             // a free vertex over a limit of common/scan3d_smooth_math.h: SCAN3D_ERR_CONFIG
    uint32_t held, isolated;       // vertices on an edge whose count is not 2; vertices without a neighbour
    uint32_t entries;              // neighbour row entries (the sum of the degrees)
};
struct SmoothWorkspace {
    DeviceBuffer<unsigned long long> keys;  // [6 faces] the edge table
    DeviceBuffer<uint32_t> sides;           // [6 faces]
    DeviceBuffer<uint32_t> rows;            // [6 faces]
    DeviceBuffer<uint32_t> degree;          // [vertices]
    DeviceBuffer<uint8_t> held;             // [vertices]
    DeviceBuffer<uint32_t> block_counts;    // [cdiv(vertices, POINT_BLOCK) + 1]
    DeviceBuffer<uint32_t> cursor;          // [vertices]
    DeviceBuffer<long long> q[2];           // [vertices][3]
    DeviceBuffer<unsigned long long> nsum;  // [vertices][3]
    DeviceBuffer<SmoothState> state;
    // 7 + passes + 2 launches for n vertices (xyz, nrm may be null) and nf faces [nf][3], nf < 2^32 / 6: the exponent
    // max and the finiteness check over the vertices, the sides into the edge table, the degrees and held flags per
    // edge, the degree sums per POINT_BLOCK vertices, their k_scan, the row starts with the fixed-point positions, the
    // neighbour rows; then one gather per pass (k = lambda, or lambda and mu alternating when mu != 0); then the face
    // normals and the write of xyz_out / nrm_out (nrm_out may be null), which writes nothing when the state holds an
    // error.  xyz_out may be xyz and nrm_out nrm.
    cudaError_t run(const float* xyz, const float* nrm, const int32_t* faces, uint32_t n, uint32_t nf, int passes,
                    double lambda, double mu, float* xyz_out, float* nrm_out, cudaStream_t st, int64_t* launches);
};

// the hole filling (scan3d_fill_kernels.cu; common/scan3d_fill_math.h has the arithmetic); the undirected edges are
// the smoothing's table of (min << 32 | max) keys
struct FillState {
    unsigned long long cells64;    // the DP cells of every hole, exact (the scan's 32-bit total may wrap)
    uint32_t bad;                  // a coordinate not finite or a face index outside [0, vertices): SCAN3D_ERR_ARG
    uint32_t boundary;             // hole edges (edges of count 1)
    uint32_t holes, loop_edges, cells;   // the scans' totals: holes, their edges, their DP cells
    uint32_t filled, added;        // holes filled, faces added (a scan total)
    uint32_t pad;
};
struct FillBuffers;
struct FillHole {
    uint32_t v0, n;                // smallest vertex, edges
    uint32_t vert;                 // first of its vertices (and stack entries)
    uint32_t cell;                 // first of its DP cells
};
struct FillWorkspace {
    DeviceBuffer<unsigned long long> keys;  // [6 faces] the edge table
    DeviceBuffer<uint32_t> sides, face;     // [6 faces] sides per edge; the face of a side on it
    DeviceBuffer<uint32_t> out_n, in_n;     // [vertices] hole edges leaving / entering the vertex
    DeviceBuffer<uint32_t> next, rim;       // [vertices] head and rim face of the hole edge leaving the vertex
    DeviceBuffer<uint32_t> len;             // [vertices] edges of the hole whose smallest vertex this is, else 0
    DeviceBuffer<uint32_t> block_counts;    // [3][cdiv(vertices, POINT_BLOCK) + 1] holes, edges and cells per block
    DeviceBuffer<FillHole> holes;           // [holes]
    DeviceBuffer<uint32_t> hole_faces;      // [holes] faces the hole adds
    DeviceBuffer<uint32_t> face_counts;     // [cdiv(holes, POINT_BLOCK) + 1] faces added per block of holes
    DeviceBuffer<uint32_t> verts, stack;    // [loop edges] the holes' vertices; the emission's stacks
    DeviceBuffer<s3h::Cell> cells;          // [cells]
    DeviceBuffer<FillState> state;
    uint32_t table = 0, stride = 0;         // the edge table's slots and block_counts' stride of the last count
    FillBuffers view();
    // 6 launches for n vertices and nf faces [nf][3], nf < 2^32 / 6, holes of at most max_edges edges: the sides into
    // the edge table (with the face-index check), the hole edges per edge of count 1, the walk per vertex (with the
    // finiteness check) that flags each hole's smallest vertex with the per-block sums, and k_scan over the holes, their
    // edges and their cells; state->bad, boundary, holes, loop_edges and cells64 are then known
    cudaError_t count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, uint32_t max_edges,
                      cudaStream_t st, int64_t* launches);
    // 4 launches after count and a synchronisation that read st: the holes and their vertices, the DP (one block per
    // hole), k_scan over the faces added per block of holes (state->added), and the emission of the added faces into
    // out, which writes nothing when state->added > capacity
    cudaError_t fill(const FillState& counts, const float* xyz, const int32_t* faces, uint32_t n, int32_t* out,
                     uint64_t capacity, cudaStream_t st, int64_t* launches);
};

// the non-manifold repair (scan3d_repair_kernels.cu; common/scan3d_repair_math.h has the face key and the edge rule);
// the undirected edges are the smoothing's table of (min << 32 | max) keys, the fans a union-find over face corners
struct RepairState {
    uint32_t bad;                  // a coordinate not finite or a face index outside [0, vertices): SCAN3D_ERR_ARG
    uint32_t degenerate, duplicate;
    uint32_t nonmanifold_edges, nonmanifold_faces;
    uint32_t split;                // vertices with more than one fan
    uint32_t added, faces;         // the scans' totals: new vertices, kept faces
    uint32_t boundary, inconsistent;
};
struct RepairBuffers;
struct RepairWorkspace {
    DeviceBuffer<unsigned long long> keys;  // [6 faces] the edge table
    DeviceBuffer<uint32_t> sides, kept_n;   // [6 faces] faces on each edge after steps 1-2; kept faces on it
    DeviceBuffer<unsigned long long> best;  // [6 faces][3] largest face key per direction, largest other than f1
    DeviceBuffer<uint32_t> pair;            // [6 faces][2] the kept faces of an edge with at most 2 of them
    DeviceBuffer<uint32_t> triples;         // [2 faces] the duplicate table: face indices, VOXEL_NO_SLOT = free
    DeviceBuffer<uint32_t> triple_slot;     // [faces] table slot of each face
    DeviceBuffer<unsigned long long> key;   // [faces] K(f)
    DeviceBuffer<uint32_t> side_slot;       // [faces][3] edge-table slot of each side
    DeviceBuffer<uint8_t> status;           // [faces] 1 = survives steps 1-2
    DeviceBuffer<uint8_t> keep;             // [faces] kept
    DeviceBuffer<uint32_t> face_counts;     // [cdiv(faces, POINT_BLOCK) + 1]
    DeviceBuffer<uint32_t> parent;          // [3 faces] union-find over corners, then each corner's root
    DeviceBuffer<uint8_t> fresh;            // [3 faces] the corner is the smallest of a fan that gets a new vertex
    DeviceBuffer<uint32_t> corner_counts;   // [cdiv(3 faces, POINT_BLOCK) + 1]
    DeviceBuffer<uint32_t> new_id;          // [3 faces] the new vertex of a fan, at its smallest corner
    DeviceBuffer<uint32_t> first, fans;     // [vertices] smallest kept corner; new fans
    DeviceBuffer<int32_t> source;           // [added] the surface route's source vertices
    DeviceBuffer<RepairState> state;
    uint32_t table = 0, dup_table = 0;      // slots of the edge and duplicate tables of the last count
    RepairBuffers view();
    // 10 launches for n vertices and nf faces [nf][3], 3 nf < 2^31, flags SCAN3D_REPAIR_*: the finiteness check, the
    // face-index check, the degenerate faces and the duplicate table; the surviving faces' keys and sides into the
    // edge table; the largest key other than f1 per edge; the drop flags with the kept faces' sides and smallest
    // corners; per edge the counts and the unions of the corners; the roots with the fresh flags; k_count + k_scan over
    // the fresh flags (state->added) and over the keep flags (state->faces).  Every count of state is then known.
    cudaError_t count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, int flags, cudaStream_t st,
                      int64_t* launches);
    // 2 launches after count and a synchronisation that read st: the new vertices (their sources into source_out and,
    // when xyz_out is set, their xyz, normal and rgb bytes after the first n vertices of out), then the kept faces,
    // remapped, into faces_out
    cudaError_t emit(const int32_t* faces, uint32_t n, uint32_t nf, int flags, int32_t* faces_out, int32_t* source_out,
                     const float* xyz, const float* nrm, const uint8_t* rgb, float* xyz_out, float* nrm_out,
                     uint8_t* rgb_out, cudaStream_t st, int64_t* launches);
};

// the coherent orientation and the measures (scan3d_orient_kernels.cu; common/scan3d_orient_math.h has the
// arithmetic); the undirected edges are the smoothing's table of (min << 32 | max) keys, the 2-colouring a union-find
// over the nodes 2 f (f as wound) and 2 f + 1 (f flipped)
struct OrientState {
    unsigned long long volume[2], area[2];   // int128 sums of the volume and area terms (low word, high word)
    uint32_t box_lo[3], box_hi[3];           // s3o::order_key of the referenced vertices' bounding box
    uint32_t exp_field;            // the largest double exponent field of an offset from the centre
    uint32_t bad;                  // a coordinate not finite or a face index outside [0, vertices): SCAN3D_ERR_ARG
    uint32_t degenerate, referenced;
    uint32_t edges, boundary, nonmanifold, inconsistent;
    uint32_t patches;              // a scan total
    uint32_t closed, nonorientable, flipped, flipped_normals, inconsistent_after;
};
struct OrientBuffers;
struct OrientWorkspace {
    DeviceBuffer<unsigned long long> keys;  // [6 faces] the edge table
    DeviceBuffer<uint32_t> sides;           // [6 faces] faces on each edge
    DeviceBuffer<uint32_t> pair;            // [6 faces][2] the first two faces of each edge
    DeviceBuffer<uint32_t> side_slot;       // [faces][3] edge-table slot of each side
    DeviceBuffer<uint8_t> status;           // [faces] indices in range, not degenerate
    DeviceBuffer<uint32_t> parent;          // [2 faces] union-find over the face nodes
    DeviceBuffer<uint32_t> root;            // [faces] find(2 f)
    DeviceBuffer<uint8_t> is_root;          // [faces] the smallest face of its patch
    DeviceBuffer<uint32_t> face_counts;     // [cdiv(faces, POINT_BLOCK) + 1]
    DeviceBuffer<uint32_t> size, npos;      // [faces] per patch (at its smallest face): faces, faces of sigma = +1
    DeviceBuffer<unsigned long long> v0;    // [faces][2] per patch: int128 sum of sigma D
    DeviceBuffer<uint8_t> open, nonorientable;   // [faces] per patch
    DeviceBuffer<uint8_t> flip;             // [faces]
    DeviceBuffer<uint8_t> ref, kept;        // [vertices] in a face that is not degenerate; in one that keeps its winding
    DeviceBuffer<OrientState> state;
    uint32_t table = 0;                     // slots of the edge table of the last count
    OrientBuffers view();
    // 7 launches for n vertices and nf faces [nf][3], 6 nf < 2^32: the face-index check with the degenerate faces, the
    // referenced vertices and the sides into the edge table; the finiteness check with the bounding box; per edge the
    // counts and the unions, per vertex the exponent of the offsets; per face the roots, the patch counters and the
    // volume and area sums; k_count + k_scan over the roots (state->patches); per face the flips, per patch the closed
    // and non-orientable counts, per edge the inconsistent edges left.  Every count of state but flipped_normals is
    // then known.
    cudaError_t count(const float* xyz, const int32_t* faces, uint32_t n, uint32_t nf, cudaStream_t st,
                      int64_t* launches);
    // 1 launch after count on the same stream: the flips into faces and, when nrm is set, the negated normals
    // (state->flipped_normals); nothing is written when state->bad is set
    cudaError_t apply(int32_t* faces, float* nrm, uint32_t n, uint32_t nf, cudaStream_t st, int64_t* launches);
};
}  // namespace s3d

// Every device buffer the context owns is a DeviceBuffer: scan3d_destroy frees them all by deleting the context.
struct scan3d_ctx {
    template <class T>
    using Buf = s3d::DeviceBuffer<T>;

    scan3d_config cfg{};
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    std::string err;
    int64_t launches = 0;

    // calibration
    bool has_calib = false;
    bool fast_div_ok = false;      // see scan3d_math.cuh div_const
    scan3d_calib hcal{};
    s3d::DeviceCalib dcal{};
    Buf<double2> cam_lut;          // [H][W] (u',v') of the local rows, only if the camera is distorted
    Buf<double2> proj_lut;         // [PH][PW], only if the projector is distorted
    Buf<double> atan_tab;          // hi[33] then lo[33]
    Buf<double> code_term;         // [2^max(M_v, M_h)] the unwrap term of every fringe order
    float* pts_ext = nullptr;      // scan3d_set_points_buffer: caller-owned (possibly peer) destination of the points
    Buf<uint8_t> pattern_profiles; // scan3d_generate_patterns: 1-D profiles of both directions' patterns
    bool have_profiles[2] = {false, false};
    Buf<uint8_t> roi_eff;          // SCAN3D_FLAG_MODULATION_MASK: ROI && modulation criterion of the current direction
    Buf<uint8_t> roi_eff_h;        // ... single-pass entry: the horizontal direction's plane (roi_eff = the vertical one's)
    Buf<uint8_t> roi_strict;       // SCAN3D_FLAG_STRICT_REFERENCE: (ROI == 1) && N in {3, 4}, whole frame
    Buf<double> nstep_w;           // sin[64] then cos[64] (generic-N extension)
    Buf<short2> undist_xy[2];      // cv::undistort's fixed-point map of the camera [0] / projector [1]
    Buf<uint16_t> undist_frac[2];  // (scan3d_undistort_frames; built on first use per calibration)

    // planes (row-major [H][W])
    Buf<float> wrapped[2];
    Buf<float> unwrapped[2];
    Buf<int16_t> code[2];
    Buf<uint8_t> mask[2];
    Buf<uint8_t> valid;
    Buf<int2> cpmap;
    Buf<double> xyz;               // lazily allocated by scan3d_triangulate

    // compacted points
    Buf<float> pts;                // [H*W][3]
    Buf<uint32_t> pix;             // [H*W]   (only with SCAN3D_FLAG_POINT_PIXELS / stage API)
    Buf<uint8_t> rgb;              // [H*W][3] (only when a texture is set)
    Buf<uint8_t> texture;          // [H][W][3] BGR
    Buf<uint32_t> d_count;         // [1]
    Buf<uint32_t> block_counts;    // stage-API compaction scratch
    Buf<unsigned long long> tile_state;  // fused kernel decoupled look-back
    Buf<uint8_t> tile_flags;             // fused kernel work list (see k_tile_flags)
    Buf<int> tile_list;
    Buf<unsigned long long> trace;       // SCAN3D_TRACE=1: per-CTA pipeline timeline
    uint32_t epoch = 0;
    s3d::TensorMapCache tmaps;

    // staging for the host-buffer entries
    Buf<uint8_t> d_stack;
    Buf<uint8_t> d_roi;
    Buf<uint8_t> d_undist;         // scan3d_reconstruct_raw: the undistorted stack

    // scan3d_build_mesh (allocated on the first build)
    Buf<int32_t> mesh_idx;         // [H*W] point index of each pixel, -1 = invalid
    Buf<uint32_t> mesh_counts;     // face counts / offsets per block of POINT_BLOCK pixels
    Buf<uint32_t> mesh_totals;     // [2] points, faces
    Buf<int32_t> mesh_faces;       // [2(W-1)(H-1)][3]
    Buf<float> mesh_normals;       // [H*W][3]

    // scan3d_voxel_begin: the merge accumulator (independent of the points; reallocated when a begin asks for more)
    s3d::VoxelStore vox;
    uint64_t vox_bound = 0;        // upper bound of the points added since begin (W*H per ctx add, n per dev add)
    uint32_t vox_chunks = 0;       // adds (chunks of <= W*H points) since begin
    Buf<uint32_t> vox_point_slot;         // [H*W] per-point scratch of an add
    Buf<uint8_t> vox_flags;               // [H*W]
    Buf<float> vox_xyz;                   // [max_voxels][3] outputs of scan3d_voxel_finish
    Buf<float> vox_nrm;                   // [max_voxels][3]
    Buf<uint8_t> vox_rgb;                 // [max_voxels][3]
    Buf<uint32_t> vox_cnt;                // [max_voxels]

    // The stages on the merged model.  Each owns its device scratch, allocates it on first use, grows it on demand
    // and clears what its kernels need cleared.
    s3d::AlignWorkspace aln;              // scan3d_align_to_voxels*, and the model index of scan3d_voxel_surface
    s3d::SurfaceWorkspace lattice;        // scan3d_voxel_surface
    s3d::ComponentsWorkspace cc;          // scan3d_voxel_surface_components, scan3d_mesh_components_dev
    s3d::DecimateWorkspace dec;           // scan3d_voxel_surface_decimate
    s3d::SmoothWorkspace smooth;          // scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev
    s3d::FillWorkspace fill;              // scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev
    s3d::RepairWorkspace repair;          // scan3d_voxel_surface_repair, scan3d_mesh_repair_dev
    s3d::OrientWorkspace orient;          // scan3d_voxel_surface_orient / _measure, scan3d_mesh_orient_dev / _measure_dev

    // the held voxel surface, and the spare set that components, decimate, smooth, fill and repair write before they
    // swap it in
    s3d::SurfaceMesh surface, spare;
    int64_t cc_components = 0;
    // since the held surface was extracted: a repair dropped faces or split vertices, or an orientation flipped faces;
    // a fill added faces after that.  The decimation's quadric bound needs one hole per cell, which holds unless both
    // happened (common/scan3d_repair_math.h, common/scan3d_orient_math.h).
    bool srf_repaired = false, srf_filled_after_repair = false;

    int cta_limit = 0;             // scan3d_set_cta_limit

    // scan3d_set_registration
    bool reg_on = false;
    float reg_R[16] = {}, reg_t[3] = {};

    // which of the results above are current (scan3d_results.h)
    s3d::Results results;
};

// the C entries' error returns: a failed CUDA call names itself in ctx->err
#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return SCAN3D_ERR_CUDA;                                                       \
        }                                                                                 \
    } while (0)

namespace s3d {

inline int fail(scan3d_ctx* ctx, int code, const char* msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

struct Shape {
    int W, H;         // local frame
    int row0, H_total;
    int PW, PH;
};

inline Shape shape_of(const scan3d_config& c)
{
    Shape s;
    s.W = c.W; s.H = c.H; s.row0 = c.row0;
    s.H_total = c.H_total > 0 ? c.H_total : c.H;
    s.PW = c.PW; s.PH = c.PH;
    return s;
}

// ---- stage-wise kernels (any W, H) ----
cudaError_t launch_mask(const Shape& s, const uint8_t* roi_full, uint8_t* mask, cudaStream_t st);
cudaError_t launch_expand_patterns(const uint8_t* profiles, int profile_len, int n_patterns, uint8_t* out, int PW, int PH,
                                   int dir, cudaStream_t st);
cudaError_t launch_strict_roi(const uint8_t* roi, uint8_t* roi_eff, size_t n, int N, cudaStream_t st);
cudaError_t launch_modulation_roi(const Shape& s, const uint8_t* fringe, const uint8_t* roi, uint8_t* roi_eff, cudaStream_t st);
cudaError_t launch_wrapped(const Shape& s, int N, const uint8_t* fringe, const uint8_t* roi_full,
                           float* wrapped, const double* atan_tab, const double* nstep_w,
                           bool libdevice, cudaStream_t st);
cudaError_t launch_unwrap(const Shape& s, int dir, int M, const uint8_t* gray, const uint8_t* inv,
                          float* wrapped, const uint8_t* mask, int16_t* code, float* unwrapped,
                          cudaStream_t st);
cudaError_t launch_cpmap(const Shape& s, int fw_v, int fw_h, const float* unw_v, const float* unw_h,
                         const uint8_t* mask_v, const uint8_t* mask_h, int2* cpmap, uint8_t* valid,
                         cudaStream_t st);
cudaError_t launch_triangulate(const Shape& s, const DeviceCalib& cal, const double2* cam_lut,
                               const double2* proj_lut, const int2* cpmap, const uint8_t* valid,
                               double* xyz, cudaStream_t st);
cudaError_t launch_undistort_lut(const double* K9_k5_dev_unused, const DeviceCalib& cal, bool projector,
                                 int W, int H, int row0, double2* lut, cudaStream_t st);
// Raster-order point offsets of the valid plane, 2 launches (k_count, k_scan): block_counts[b] = number of valid
// pixels before block b of POINT_BLOCK pixels, *total = all of them.  An empty plane takes one block (total 0).
constexpr int POINT_BLOCK = 1024;
cudaError_t launch_point_offsets(const uint8_t* valid, size_t plane, uint32_t* block_counts, uint32_t* total,
                                 cudaStream_t st);
// exclusive scan of counts[n] in place by one CTA (k_scan), *total = the sum; 1 launch
cudaError_t launch_block_scan(uint32_t* counts, int n, uint32_t* total, cudaStream_t st);

// rank of this thread's flag among the flags of its POINT_BLOCK block (every thread of the block calls it); with the
// block offsets of launch_point_offsets this places a flagged item at its compacted position
__device__ __forceinline__ uint32_t block_rank(bool flag)
{
    __shared__ uint32_t wsum[POINT_BLOCK / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) wsum[w] = __popc(b);
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < w; k++) before += wsum[k];
    return before + __popc(b & ((1u << lane) - 1));
}
// 3 launches: count, scan, scatter.  pix / rgb / texture may be null.
cudaError_t launch_compact(const Shape& s, const double* xyz, const uint8_t* valid,
                           const uint8_t* texture, uint32_t* block_counts, float* pts, uint32_t* pix,
                           uint8_t* rgb, uint32_t* d_count, cudaStream_t st, int* n_launches);

// ---- fused single-pass kernel (W % 16 == 0, N in {3,4,5,8}) ----
struct FusedArgs {
    const uint8_t* stack;   // [NF][H][W]
    const uint8_t* roi;     // [H_total][W]
    const uint8_t* roi2;    // modulation criterion: the horizontal direction's effective ROI (roi = the vertical one's)
    const uint8_t* roi_list;   // ... and the caller's ROI, a superset of both: the work list is built from it
    float* unw_v; float* unw_h;
    int16_t* code_v; int16_t* code_h;
    uint8_t* valid;         // final valid (dirs==2) or mask (dirs==1)
    int2* cpmap;
    float* pts; uint32_t* pix; uint8_t* rgb; const uint8_t* texture;
    uint32_t* d_count;
    unsigned long long* tile_state;
    uint8_t* tile_flags;          // [n_tiles] tile holds at least one ROI pixel
    int* tile_list;               // [n_tiles] ids of those tiles, raster order
    int* n_list;                  // [1]; n_list[n_tiles + 8] is the counter the CTAs draw work-list positions from
    int reg_on;                   // fold register_point_clouds' transform into the point store (scan3d_set_registration)
    float reg_R[16], reg_t[3];
    int ctas_per_sm;              // 0 = all the kernel can have; else the launch takes at most this many CTA slots per SM
    TensorMapCache* tmap_cache;   // host pointer (the launcher's cache of tensor maps; unused on the device)
    unsigned long long* trace;    // optional timeline buffer (SCAN3D_TRACE), else null
    const double2* cam_lut; const double2* proj_lut;
    const double* atan_tab;
    const double* code_term;      // [2^max(M_v, M_h)] code*2.0*Pi per fringe order (fill_code_term_table)
    uint32_t epoch;
    int W, H, row0, H_total, PW, PH;
    int N, M_v, M_h, fw_v, fw_h;
    double fw_v_d, fw_h_d;        // the fringe widths as doubles (5/compute_correspondance.cpp:648: fw * (Phi / 2Pi) in double)
    int n_tiles;
};
int fused_num_tiles(const scan3d_config& c);

// the single-pass kernel (scan3d_fused_kernel7.cu)
bool fused7_supported(const scan3d_config& c);
bool fused7_folds_registration(const scan3d_config& c);
cudaError_t launch_fused7(const scan3d_config& c, const FusedArgs& a, const DeviceCalib& cal,
                          int sm_count, cudaStream_t st);

// ---- either side of the path (scan3d_aux_kernels.cu) ----
cudaError_t launch_undistort_map(const double K[9], const double d[5], int W, int H, short2* map_xy, uint16_t* map_frac,
                                 cudaStream_t st);
cudaError_t launch_remap_frames(const uint8_t* src, uint8_t* dst, const short2* map_xy, const uint16_t* map_frac, int W,
                                int H, int n_frames, int sm_count, cudaStream_t st);
cudaError_t launch_roi_fill(const uint8_t* outline, int W, int H, uint8_t* roi, uint8_t* filled, cudaStream_t st);
cudaError_t launch_register_points(const float* src, float* dst, long long n, const float R[16], float tx, float ty,
                                   float tz, int sm_count, cudaStream_t st);

// ---- camera-grid mesh (scan3d_mesh_kernels.cu) ----
// 6 launches: point offsets (k_count, k_scan), pixel -> point index plane, face counts per block, their scan, faces +
// normals.  idx [W*H], block_counts [cdiv(W*H, POINT_BLOCK)], face_counts [same], totals [2] (points, faces); faces
// [2(W-1)(H-1)][3], normals [W*H][3].
cudaError_t launch_mesh(const uint8_t* valid, const float* pts, int W, int H, float max_edge, int32_t* idx,
                        uint32_t* block_counts, uint32_t* face_counts, uint32_t* totals, int32_t* faces, float* normals,
                        cudaStream_t st, int64_t* launches);

// ---- voxel-grid merge (scan3d_voxel_kernels.cu; common/scan3d_voxel_math.h has the arithmetic) ----
// 5 launches for `plane` points (the ctx add reads the point count from n_dev, <= plane): insert, flag, k_count +
// k_scan over the flags, assign.  point_slot and flags [plane], block_counts [cdiv(plane, POINT_BLOCK)]; par = number
// of adds (chunks) since begin, mod 2.  nrm / rgb may be null (zeros).
cudaError_t launch_voxel_add(const VoxelTable& t, const float* xyz, const float* nrm, const uint8_t* rgb,
                             const uint32_t* n_dev, uint32_t plane, uint32_t* point_slot, uint8_t* flags,
                             uint32_t* block_counts, int par, cudaStream_t st, int64_t* launches);
// 1 launch: the merged voxels in first-point order into xyz / nrm [max_voxels][3], rgb [max_voxels][3], cnt
cudaError_t launch_voxel_finish(const VoxelTable& t, int par, float* xyz, float* nrm, uint8_t* rgb, uint32_t* cnt,
                                int sm_count, cudaStream_t st);

// ---- debug / self-test ----
cudaError_t launch_debug_atan2(const double* y, const double* x, float* out, int n, int mode,
                               const double* atan_tab, cudaStream_t st);

cudaError_t launch_debug_divcheck(unsigned long long* bad, cudaStream_t st);


}  // namespace s3d
