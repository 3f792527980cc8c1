// mesh.cu — marching cubes on the device-resident layer (SURVEY.md §8f N4).
//
// What the callers do right after the merge: voxgraph::SubmapVisuals::saveAndPubCombinedMesh ->
// voxblox::MeshIntegrator<TsdfVoxel>::generateMesh over the projected map
// (coxgraph/src/server/visualizer/server_visualizer.cpp:123-126) and generateSubmapMesh on the
// client (coxgraph/src/client/map_server.cpp:126-130).  Meshing here means the global layer
// (~50 KB per block) never has to leave HBM: only the triangles do.
//
// Semantics follow upstream voxblox mesh/mesh_integrator.h + mesh/marching_cubes.h ([EXT]):
//   * per block, cubes in the reference's order: interior (x, y, z loops, z fastest, indices
//     0..14), max-X plane (z, y), max-Y plane (z, x < 15), max-Z plane (y < 15, x < 15);
//   * a cube is meshed iff all 8 corners are observed (weight > min_weight); border cubes read
//     the +x/+y/+z neighbour blocks and are skipped when one is missing;
//   * vertices by linear interpolation along sign-changing edges (midpoint when |sdf1 - sdf2| <
//     1e-6), three per triangle in table order reversed, normal = normalised cross product,
//     colour = the voxel containing the vertex (clamped index in the block found from the vertex
//     coordinates when it lies outside this block).
// One CTA per block: the block plus its +1 halo is staged in shared memory (17^3 distances and
// weights), every thread classifies 16 consecutive cubes of the reference order, a block-wide
// scan numbers the triangles, and the vertices land at their final position — the output is
// byte-identical whatever the launch geometry.  Two passes (count, then write) with a scan over
// the blocks in between give every block its vertex range in (z, y, x) block order.
// cg_layer_mesh_sharded runs the same kernel over one rank's owned layer of a sharded global map;
// only the block lookup differs (ShardedBlocks: the +x/+y/+z neighbours and the colour block may
// live on a peer rank and are read from its pool over NVLink).
#include <cub/cub.cuh>

#include <algorithm>

#include "cg_internal.cuh"

namespace cg {

__device__ const int8_t kTriTable[256][16] = {
    {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 8, 3, 9, 8, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 1, 2, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 2, 10, 0, 2, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 8, 3, 2, 10, 8, 10, 9, 8, -1, -1, -1, -1, -1, -1, -1},
    {3, 11, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 11, 2, 8, 11, 0, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 11, 2, 1, 9, 11, 9, 8, 11, -1, -1, -1, -1, -1, -1, -1},
    {3, 10, 1, 11, 10, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 10, 1, 0, 8, 10, 8, 11, 10, -1, -1, -1, -1, -1, -1, -1},
    {3, 9, 0, 3, 11, 9, 11, 10, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 8, 10, 10, 8, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 7, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 3, 0, 7, 3, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 1, 9, 4, 7, 1, 7, 3, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 4, 7, 3, 0, 4, 1, 2, 10, -1, -1, -1, -1, -1, -1, -1},
    {9, 2, 10, 9, 0, 2, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1},
    {2, 10, 9, 2, 9, 7, 2, 7, 3, 7, 9, 4, -1, -1, -1, -1},
    {8, 4, 7, 3, 11, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 4, 7, 11, 2, 4, 2, 0, 4, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 1, 8, 4, 7, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1},
    {4, 7, 11, 9, 4, 11, 9, 11, 2, 9, 2, 1, -1, -1, -1, -1},
    {3, 10, 1, 3, 11, 10, 7, 8, 4, -1, -1, -1, -1, -1, -1, -1},
    {1, 11, 10, 1, 4, 11, 1, 0, 4, 7, 11, 4, -1, -1, -1, -1},
    {4, 7, 8, 9, 0, 11, 9, 11, 10, 11, 0, 3, -1, -1, -1, -1},
    {4, 7, 11, 4, 11, 9, 9, 11, 10, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, 0, 8, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 5, 4, 1, 5, 0, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 5, 4, 8, 3, 5, 3, 1, 5, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 9, 5, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 1, 2, 10, 4, 9, 5, -1, -1, -1, -1, -1, -1, -1},
    {5, 2, 10, 5, 4, 2, 4, 0, 2, -1, -1, -1, -1, -1, -1, -1},
    {2, 10, 5, 3, 2, 5, 3, 5, 4, 3, 4, 8, -1, -1, -1, -1},
    {9, 5, 4, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 11, 2, 0, 8, 11, 4, 9, 5, -1, -1, -1, -1, -1, -1, -1},
    {0, 5, 4, 0, 1, 5, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1},
    {2, 1, 5, 2, 5, 8, 2, 8, 11, 4, 8, 5, -1, -1, -1, -1},
    {10, 3, 11, 10, 1, 3, 9, 5, 4, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 5, 0, 8, 1, 8, 10, 1, 8, 11, 10, -1, -1, -1, -1},
    {5, 4, 0, 5, 0, 11, 5, 11, 10, 11, 0, 3, -1, -1, -1, -1},
    {5, 4, 8, 5, 8, 10, 10, 8, 11, -1, -1, -1, -1, -1, -1, -1},
    {9, 7, 8, 5, 7, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 3, 0, 9, 5, 3, 5, 7, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 7, 8, 0, 1, 7, 1, 5, 7, -1, -1, -1, -1, -1, -1, -1},
    {1, 5, 3, 3, 5, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 7, 8, 9, 5, 7, 10, 1, 2, -1, -1, -1, -1, -1, -1, -1},
    {10, 1, 2, 9, 5, 0, 5, 3, 0, 5, 7, 3, -1, -1, -1, -1},
    {8, 0, 2, 8, 2, 5, 8, 5, 7, 10, 5, 2, -1, -1, -1, -1},
    {2, 10, 5, 2, 5, 3, 3, 5, 7, -1, -1, -1, -1, -1, -1, -1},
    {7, 9, 5, 7, 8, 9, 3, 11, 2, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 7, 9, 7, 2, 9, 2, 0, 2, 7, 11, -1, -1, -1, -1},
    {2, 3, 11, 0, 1, 8, 1, 7, 8, 1, 5, 7, -1, -1, -1, -1},
    {11, 2, 1, 11, 1, 7, 7, 1, 5, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 8, 8, 5, 7, 10, 1, 3, 10, 3, 11, -1, -1, -1, -1},
    {5, 7, 0, 5, 0, 9, 7, 11, 0, 1, 0, 10, 11, 10, 0, -1},
    {11, 10, 0, 11, 0, 3, 10, 5, 0, 8, 0, 7, 5, 7, 0, -1},
    {11, 10, 5, 7, 11, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {10, 6, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 1, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 8, 3, 1, 9, 8, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 5, 2, 6, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 5, 1, 2, 6, 3, 0, 8, -1, -1, -1, -1, -1, -1, -1},
    {9, 6, 5, 9, 0, 6, 0, 2, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 9, 8, 5, 8, 2, 5, 2, 6, 3, 2, 8, -1, -1, -1, -1},
    {2, 3, 11, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 0, 8, 11, 2, 0, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 2, 3, 11, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 1, 9, 2, 9, 11, 2, 9, 8, 11, -1, -1, -1, -1},
    {6, 3, 11, 6, 5, 3, 5, 1, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 11, 0, 11, 5, 0, 5, 1, 5, 11, 6, -1, -1, -1, -1},
    {3, 11, 6, 0, 3, 6, 0, 6, 5, 0, 5, 9, -1, -1, -1, -1},
    {6, 5, 9, 6, 9, 11, 11, 9, 8, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 4, 7, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 3, 0, 4, 7, 3, 6, 5, 10, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 5, 10, 6, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1},
    {10, 6, 5, 1, 9, 7, 1, 7, 3, 7, 9, 4, -1, -1, -1, -1},
    {6, 1, 2, 6, 5, 1, 4, 7, 8, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 5, 5, 2, 6, 3, 0, 4, 3, 4, 7, -1, -1, -1, -1},
    {8, 4, 7, 9, 0, 5, 0, 6, 5, 0, 2, 6, -1, -1, -1, -1},
    {7, 3, 9, 7, 9, 4, 3, 2, 9, 5, 9, 6, 2, 6, 9, -1},
    {3, 11, 2, 7, 8, 4, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 4, 7, 2, 4, 2, 0, 2, 7, 11, -1, -1, -1, -1},
    {0, 1, 9, 4, 7, 8, 2, 3, 11, 5, 10, 6, -1, -1, -1, -1},
    {9, 2, 1, 9, 11, 2, 9, 4, 11, 7, 11, 4, 5, 10, 6, -1},
    {8, 4, 7, 3, 11, 5, 3, 5, 1, 5, 11, 6, -1, -1, -1, -1},
    {5, 1, 11, 5, 11, 6, 1, 0, 11, 7, 11, 4, 0, 4, 11, -1},
    {0, 5, 9, 0, 6, 5, 0, 3, 6, 11, 6, 3, 8, 4, 7, -1},
    {6, 5, 9, 6, 9, 11, 4, 7, 9, 7, 11, 9, -1, -1, -1, -1},
    {10, 4, 9, 6, 4, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 10, 6, 4, 9, 10, 0, 8, 3, -1, -1, -1, -1, -1, -1, -1},
    {10, 0, 1, 10, 6, 0, 6, 4, 0, -1, -1, -1, -1, -1, -1, -1},
    {8, 3, 1, 8, 1, 6, 8, 6, 4, 6, 1, 10, -1, -1, -1, -1},
    {1, 4, 9, 1, 2, 4, 2, 6, 4, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 1, 2, 9, 2, 4, 9, 2, 6, 4, -1, -1, -1, -1},
    {0, 2, 4, 4, 2, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 3, 2, 8, 2, 4, 4, 2, 6, -1, -1, -1, -1, -1, -1, -1},
    {10, 4, 9, 10, 6, 4, 11, 2, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 2, 2, 8, 11, 4, 9, 10, 4, 10, 6, -1, -1, -1, -1},
    {3, 11, 2, 0, 1, 6, 0, 6, 4, 6, 1, 10, -1, -1, -1, -1},
    {6, 4, 1, 6, 1, 10, 4, 8, 1, 2, 1, 11, 8, 11, 1, -1},
    {9, 6, 4, 9, 3, 6, 9, 1, 3, 11, 6, 3, -1, -1, -1, -1},
    {8, 11, 1, 8, 1, 0, 11, 6, 1, 9, 1, 4, 6, 4, 1, -1},
    {3, 11, 6, 3, 6, 0, 0, 6, 4, -1, -1, -1, -1, -1, -1, -1},
    {6, 4, 8, 11, 6, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 10, 6, 7, 8, 10, 8, 9, 10, -1, -1, -1, -1, -1, -1, -1},
    {0, 7, 3, 0, 10, 7, 0, 9, 10, 6, 7, 10, -1, -1, -1, -1},
    {10, 6, 7, 1, 10, 7, 1, 7, 8, 1, 8, 0, -1, -1, -1, -1},
    {10, 6, 7, 10, 7, 1, 1, 7, 3, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 6, 1, 6, 8, 1, 8, 9, 8, 6, 7, -1, -1, -1, -1},
    {2, 6, 9, 2, 9, 1, 6, 7, 9, 0, 9, 3, 7, 3, 9, -1},
    {7, 8, 0, 7, 0, 6, 6, 0, 2, -1, -1, -1, -1, -1, -1, -1},
    {7, 3, 2, 6, 7, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 11, 10, 6, 8, 10, 8, 9, 8, 6, 7, -1, -1, -1, -1},
    {2, 0, 7, 2, 7, 11, 0, 9, 7, 6, 7, 10, 9, 10, 7, -1},
    {1, 8, 0, 1, 7, 8, 1, 10, 7, 6, 7, 10, 2, 3, 11, -1},
    {11, 2, 1, 11, 1, 7, 10, 6, 1, 6, 7, 1, -1, -1, -1, -1},
    {8, 9, 6, 8, 6, 7, 9, 1, 6, 11, 6, 3, 1, 3, 6, -1},
    {0, 9, 1, 11, 6, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 8, 0, 7, 0, 6, 3, 11, 0, 11, 6, 0, -1, -1, -1, -1},
    {7, 11, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 6, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 1, 9, 8, 3, 1, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1},
    {10, 1, 2, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 3, 0, 8, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1},
    {2, 9, 0, 2, 10, 9, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1},
    {6, 11, 7, 2, 10, 3, 10, 8, 3, 10, 9, 8, -1, -1, -1, -1},
    {7, 2, 3, 6, 2, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 0, 8, 7, 6, 0, 6, 2, 0, -1, -1, -1, -1, -1, -1, -1},
    {2, 7, 6, 2, 3, 7, 0, 1, 9, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 2, 1, 8, 6, 1, 9, 8, 8, 7, 6, -1, -1, -1, -1},
    {10, 7, 6, 10, 1, 7, 1, 3, 7, -1, -1, -1, -1, -1, -1, -1},
    {10, 7, 6, 1, 7, 10, 1, 8, 7, 1, 0, 8, -1, -1, -1, -1},
    {0, 3, 7, 0, 7, 10, 0, 10, 9, 6, 10, 7, -1, -1, -1, -1},
    {7, 6, 10, 7, 10, 8, 8, 10, 9, -1, -1, -1, -1, -1, -1, -1},
    {6, 8, 4, 11, 8, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 6, 11, 3, 0, 6, 0, 4, 6, -1, -1, -1, -1, -1, -1, -1},
    {8, 6, 11, 8, 4, 6, 9, 0, 1, -1, -1, -1, -1, -1, -1, -1},
    {9, 4, 6, 9, 6, 3, 9, 3, 1, 11, 3, 6, -1, -1, -1, -1},
    {6, 8, 4, 6, 11, 8, 2, 10, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 3, 0, 11, 0, 6, 11, 0, 4, 6, -1, -1, -1, -1},
    {4, 11, 8, 4, 6, 11, 0, 2, 9, 2, 10, 9, -1, -1, -1, -1},
    {10, 9, 3, 10, 3, 2, 9, 4, 3, 11, 3, 6, 4, 6, 3, -1},
    {8, 2, 3, 8, 4, 2, 4, 6, 2, -1, -1, -1, -1, -1, -1, -1},
    {0, 4, 2, 4, 6, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 2, 3, 4, 2, 4, 6, 4, 3, 8, -1, -1, -1, -1},
    {1, 9, 4, 1, 4, 2, 2, 4, 6, -1, -1, -1, -1, -1, -1, -1},
    {8, 1, 3, 8, 6, 1, 8, 4, 6, 6, 10, 1, -1, -1, -1, -1},
    {10, 1, 0, 10, 0, 6, 6, 0, 4, -1, -1, -1, -1, -1, -1, -1},
    {4, 6, 3, 4, 3, 8, 6, 10, 3, 0, 3, 9, 10, 9, 3, -1},
    {10, 9, 4, 6, 10, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 5, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 4, 9, 5, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 0, 1, 5, 4, 0, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1},
    {11, 7, 6, 8, 3, 4, 3, 5, 4, 3, 1, 5, -1, -1, -1, -1},
    {9, 5, 4, 10, 1, 2, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1},
    {6, 11, 7, 1, 2, 10, 0, 8, 3, 4, 9, 5, -1, -1, -1, -1},
    {7, 6, 11, 5, 4, 10, 4, 2, 10, 4, 0, 2, -1, -1, -1, -1},
    {3, 4, 8, 3, 5, 4, 3, 2, 5, 10, 5, 2, 11, 7, 6, -1},
    {7, 2, 3, 7, 6, 2, 5, 4, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, 0, 8, 6, 0, 6, 2, 6, 8, 7, -1, -1, -1, -1},
    {3, 6, 2, 3, 7, 6, 1, 5, 0, 5, 4, 0, -1, -1, -1, -1},
    {6, 2, 8, 6, 8, 7, 2, 1, 8, 4, 8, 5, 1, 5, 8, -1},
    {9, 5, 4, 10, 1, 6, 1, 7, 6, 1, 3, 7, -1, -1, -1, -1},
    {1, 6, 10, 1, 7, 6, 1, 0, 7, 8, 7, 0, 9, 5, 4, -1},
    {4, 0, 10, 4, 10, 5, 0, 3, 10, 6, 10, 7, 3, 7, 10, -1},
    {7, 6, 10, 7, 10, 8, 5, 4, 10, 4, 8, 10, -1, -1, -1, -1},
    {6, 9, 5, 6, 11, 9, 11, 8, 9, -1, -1, -1, -1, -1, -1, -1},
    {3, 6, 11, 0, 6, 3, 0, 5, 6, 0, 9, 5, -1, -1, -1, -1},
    {0, 11, 8, 0, 5, 11, 0, 1, 5, 5, 6, 11, -1, -1, -1, -1},
    {6, 11, 3, 6, 3, 5, 5, 3, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 9, 5, 11, 9, 11, 8, 11, 5, 6, -1, -1, -1, -1},
    {0, 11, 3, 0, 6, 11, 0, 9, 6, 5, 6, 9, 1, 2, 10, -1},
    {11, 8, 5, 11, 5, 6, 8, 0, 5, 10, 5, 2, 0, 2, 5, -1},
    {6, 11, 3, 6, 3, 5, 2, 10, 3, 10, 5, 3, -1, -1, -1, -1},
    {5, 8, 9, 5, 2, 8, 5, 6, 2, 3, 8, 2, -1, -1, -1, -1},
    {9, 5, 6, 9, 6, 0, 0, 6, 2, -1, -1, -1, -1, -1, -1, -1},
    {1, 5, 8, 1, 8, 0, 5, 6, 8, 3, 8, 2, 6, 2, 8, -1},
    {1, 5, 6, 2, 1, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 3, 6, 1, 6, 10, 3, 8, 6, 5, 6, 9, 8, 9, 6, -1},
    {10, 1, 0, 10, 0, 6, 9, 5, 0, 5, 6, 0, -1, -1, -1, -1},
    {0, 3, 8, 5, 6, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {10, 5, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 5, 10, 7, 5, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 5, 10, 11, 7, 5, 8, 3, 0, -1, -1, -1, -1, -1, -1, -1},
    {5, 11, 7, 5, 10, 11, 1, 9, 0, -1, -1, -1, -1, -1, -1, -1},
    {10, 7, 5, 10, 11, 7, 9, 8, 1, 8, 3, 1, -1, -1, -1, -1},
    {11, 1, 2, 11, 7, 1, 7, 5, 1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 1, 2, 7, 1, 7, 5, 7, 2, 11, -1, -1, -1, -1},
    {9, 7, 5, 9, 2, 7, 9, 0, 2, 2, 11, 7, -1, -1, -1, -1},
    {7, 5, 2, 7, 2, 11, 5, 9, 2, 3, 2, 8, 9, 8, 2, -1},
    {2, 5, 10, 2, 3, 5, 3, 7, 5, -1, -1, -1, -1, -1, -1, -1},
    {8, 2, 0, 8, 5, 2, 8, 7, 5, 10, 2, 5, -1, -1, -1, -1},
    {9, 0, 1, 5, 10, 3, 5, 3, 7, 3, 10, 2, -1, -1, -1, -1},
    {9, 8, 2, 9, 2, 1, 8, 7, 2, 10, 2, 5, 7, 5, 2, -1},
    {1, 3, 5, 3, 7, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 7, 0, 7, 1, 1, 7, 5, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 3, 9, 3, 5, 5, 3, 7, -1, -1, -1, -1, -1, -1, -1},
    {9, 8, 7, 5, 9, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {5, 8, 4, 5, 10, 8, 10, 11, 8, -1, -1, -1, -1, -1, -1, -1},
    {5, 0, 4, 5, 11, 0, 5, 10, 11, 11, 3, 0, -1, -1, -1, -1},
    {0, 1, 9, 8, 4, 10, 8, 10, 11, 10, 4, 5, -1, -1, -1, -1},
    {10, 11, 4, 10, 4, 5, 11, 3, 4, 9, 4, 1, 3, 1, 4, -1},
    {2, 5, 1, 2, 8, 5, 2, 11, 8, 4, 5, 8, -1, -1, -1, -1},
    {0, 4, 11, 0, 11, 3, 4, 5, 11, 2, 11, 1, 5, 1, 11, -1},
    {0, 2, 5, 0, 5, 9, 2, 11, 5, 4, 5, 8, 11, 8, 5, -1},
    {9, 4, 5, 2, 11, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 5, 10, 3, 5, 2, 3, 4, 5, 3, 8, 4, -1, -1, -1, -1},
    {5, 10, 2, 5, 2, 4, 4, 2, 0, -1, -1, -1, -1, -1, -1, -1},
    {3, 10, 2, 3, 5, 10, 3, 8, 5, 4, 5, 8, 0, 1, 9, -1},
    {5, 10, 2, 5, 2, 4, 1, 9, 2, 9, 4, 2, -1, -1, -1, -1},
    {8, 4, 5, 8, 5, 3, 3, 5, 1, -1, -1, -1, -1, -1, -1, -1},
    {0, 4, 5, 1, 0, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 4, 5, 8, 5, 3, 9, 0, 5, 0, 3, 5, -1, -1, -1, -1},
    {9, 4, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 11, 7, 4, 9, 11, 9, 10, 11, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 4, 9, 7, 9, 11, 7, 9, 10, 11, -1, -1, -1, -1},
    {1, 10, 11, 1, 11, 4, 1, 4, 0, 7, 4, 11, -1, -1, -1, -1},
    {3, 1, 4, 3, 4, 8, 1, 10, 4, 7, 4, 11, 10, 11, 4, -1},
    {4, 11, 7, 9, 11, 4, 9, 2, 11, 9, 1, 2, -1, -1, -1, -1},
    {9, 7, 4, 9, 11, 7, 9, 1, 11, 2, 11, 1, 0, 8, 3, -1},
    {11, 7, 4, 11, 4, 2, 2, 4, 0, -1, -1, -1, -1, -1, -1, -1},
    {11, 7, 4, 11, 4, 2, 8, 3, 4, 3, 2, 4, -1, -1, -1, -1},
    {2, 9, 10, 2, 7, 9, 2, 3, 7, 7, 4, 9, -1, -1, -1, -1},
    {9, 10, 7, 9, 7, 4, 10, 2, 7, 8, 7, 0, 2, 0, 7, -1},
    {3, 7, 10, 3, 10, 2, 7, 4, 10, 1, 10, 0, 4, 0, 10, -1},
    {1, 10, 2, 8, 7, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 1, 4, 1, 7, 7, 1, 3, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 1, 4, 1, 7, 0, 8, 1, 8, 7, 1, -1, -1, -1, -1},
    {4, 0, 3, 7, 4, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 8, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 10, 8, 10, 11, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 9, 3, 9, 11, 11, 9, 10, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 10, 0, 10, 8, 8, 10, 11, -1, -1, -1, -1, -1, -1, -1},
    {3, 1, 10, 11, 3, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 11, 1, 11, 9, 9, 11, 8, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 9, 3, 9, 11, 1, 2, 9, 2, 11, 9, -1, -1, -1, -1},
    {0, 2, 11, 8, 0, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 2, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 8, 2, 8, 10, 10, 8, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 10, 2, 0, 9, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 8, 2, 8, 10, 0, 1, 8, 1, 10, 8, -1, -1, -1, -1},
    {1, 10, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 3, 8, 9, 1, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 9, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 3, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1}
};
__constant__ int kMcEdge[12][2] = {{0, 1}, {1, 2}, {2, 3}, {3, 0}, {4, 5}, {5, 6},
                                   {6, 7}, {7, 4}, {0, 4}, {1, 5}, {2, 6}, {3, 7}};

constexpr int kMcThreads = 256;
constexpr int kMcTile = kVps + 1;
constexpr int kMcTileVox = kMcTile * kMcTile * kMcTile;
constexpr int kMcPerThread = kVoxelsPerBlock / kMcThreads;  // 16 cubes of consecutive rank

// position of the rank-th cube of MeshIntegrator::extractBlockMesh
__device__ __forceinline__ void mc_cube_of_rank(int r, int& x, int& y, int& z) {
  constexpr int kIn = (kVps - 1) * (kVps - 1) * (kVps - 1);  // 3375 interior cubes
  constexpr int kX = kIn + kVps * kVps;                      // + max-X plane
  constexpr int kY = kX + kVps * (kVps - 1);                 // + max-Y plane
  if (r < kIn) {
    x = r / ((kVps - 1) * (kVps - 1));
    y = (r / (kVps - 1)) % (kVps - 1);
    z = r % (kVps - 1);
  } else if (r < kX) {
    const int q = r - kIn;
    x = kVps - 1;
    z = q / kVps;
    y = q % kVps;
  } else if (r < kY) {
    const int q = r - kX;
    y = kVps - 1;
    z = q / (kVps - 1);
    x = q % (kVps - 1);
  } else {
    const int q = r - kY;
    z = kVps - 1;
    y = q / (kVps - 1);
    x = q % (kVps - 1);
  }
}
__device__ __forceinline__ int mc_tile_index(int x, int y, int z, int corner) {
  // cube_index_offsets_: corner i at (x + ox, y + oy, z + oz)
  const int ox = ((corner + 1) >> 1) & 1, oy = (corner >> 1) & 1, oz = corner >> 2;
  return (x + ox) + kMcTile * ((y + oy) + kMcTile * (z + oz));
}
// MarchingCubes::interpolateVertex
__device__ __forceinline__ V3 mc_interpolate(V3 v1, V3 v2, float sdf1, float sdf2) {
  const float diff = sdf1 - sdf2;
  if (fabsf(diff) >= 1e-6f) {
    const float t = sdf1 / diff;
    return v1 + (v2 - v1) * t;
  }
  return (v1 + v2) * 0.5f;
}

// How the kernel finds a block: find() turns a key into a reference (-1: no such block), planes()
// a reference into the block's distance plane (weight and colour planes follow, kVoxelsPerBlock
// words apart).  cg_layer_mesh looks in the layer's own hash: the reference is the pool slot.
struct LocalBlocks {
  __device__ __forceinline__ int find(const LayerView& L, uint64_t key) const {
    return L.find_slot(key);
  }
  __device__ __forceinline__ const float* planes(const LayerView& L, int ref) const {
    return L.dist_plane(ref);
  }
};

template <bool kWrite, class Blocks>
__global__ void __launch_bounds__(kMcThreads)
k_mesh_blocks(LayerView L, Blocks blocks, const uint64_t* __restrict__ sorted_keys,
              const uint32_t* __restrict__ sorted_slots, uint32_t num_blocks, float min_weight,
              int use_color, int only_updated, uint32_t* __restrict__ counts,
              const uint32_t* __restrict__ vertex_begin, float* __restrict__ vertices,
              float* __restrict__ normals, uint32_t* __restrict__ colors) {
  __shared__ float s_d[kMcTileVox];
  __shared__ float s_w[kMcTileVox];
  __shared__ int s_nb[8];
  __shared__ uint32_t s_warp[kMcThreads / 32];
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t b = blockIdx.x; b < num_blocks; b += gridDim.x) {
    const int slot = static_cast<int>(sorted_slots[b]);
    if (only_updated && !L.updated[slot]) {  // uniform for the CTA
      if (!kWrite && threadIdx.x == 0) counts[b] = 0;
      continue;
    }
    int bx, by, bz;
    unpack_block_key(sorted_keys[b], bx, by, bz);
    __syncthreads();  // previous block done with the tile
    if (threadIdx.x < 8) {
      const int k = threadIdx.x;
      s_nb[k] = k == 0 ? slot
                       : blocks.find(L, pack_block_key(bx + (k & 1), by + ((k >> 1) & 1), bz + (k >> 2)));
    }
    __syncthreads();
    for (int t = threadIdx.x; t < kMcTileVox; t += kMcThreads) {
      const int x = t % kMcTile, y = (t / kMcTile) % kMcTile, z = t / (kMcTile * kMcTile);
      const int nb = s_nb[(x >> 4) | ((y >> 4) << 1) | ((z >> 4) << 2)];
      float d = 0.0f, w = -1.0f;  // a missing neighbour block: the corner is not observed
      if (nb != -1) {
        const int lin = (x & 15) + kVps * ((y & 15) + kVps * (z & 15));
        const float* p = blocks.planes(L, nb);
        d = p[lin];
        w = p[kVoxelsPerBlock + lin];
      }
      s_d[t] = d;
      s_w[t] = w;
    }
    __syncthreads();
    // classify this thread's 16 cubes: configuration index (0 when a corner is unobserved)
    uint32_t cfg_pack[kMcPerThread / 4];
    uint32_t tris = 0;
#pragma unroll
    for (int j = 0; j < kMcPerThread; ++j) {
      int x, y, z;
      mc_cube_of_rank(threadIdx.x * kMcPerThread + j, x, y, z);
      uint32_t cfg = 0;
      bool observed = true;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int t = mc_tile_index(x, y, z, i);
        observed = observed && (s_w[t] > min_weight);  // utils::getSdfIfValid
        cfg |= (s_d[t] < 0.0f ? 1u : 0u) << i;
      }
      if (!observed) cfg = 0;
      if ((j & 3) == 0) cfg_pack[j >> 2] = 0;
      cfg_pack[j >> 2] |= cfg << (8 * (j & 3));
      int nt = 0;
      while (nt < 15 && kTriTable[cfg][nt] >= 0) nt += 3;
      tris += nt / 3;
    }
    // block-wide exclusive scan of the triangle counts
    uint32_t incl = tris;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(full, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t before = incl - tris, total = 0;
#pragma unroll
    for (int k = 0; k < kMcThreads / 32; ++k) {
      if (k < warp) before += s_warp[k];
      total += s_warp[k];
    }
    if (!kWrite) {
      if (threadIdx.x == 0) counts[b] = 3 * total;
      continue;
    }
    if (tris == 0) continue;
    // ---- write this thread's triangles at their final position
    size_t out = static_cast<size_t>(vertex_begin[b]) + 3 * static_cast<size_t>(before);
    const V3 origin = V3{static_cast<float>(bx) * L.block_size, static_cast<float>(by) * L.block_size,
                         static_cast<float>(bz) * L.block_size};
#pragma unroll 1
    for (int j = 0; j < kMcPerThread; ++j) {
      const uint32_t cfg = (cfg_pack[j >> 2] >> (8 * (j & 3))) & 255u;
      if (kTriTable[cfg][0] < 0) continue;
      int x, y, z;
      mc_cube_of_rank(threadIdx.x * kMcPerThread + j, x, y, z);
      const V3 coords = origin + V3{center_coord(x, L.voxel_size), center_coord(y, L.voxel_size),
                                    center_coord(z, L.voxel_size)};
      float sdf[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) sdf[i] = s_d[mc_tile_index(x, y, z, i)];
      auto corner = [&](int i) {
        const int ox = ((i + 1) >> 1) & 1, oy = (i >> 1) & 1, oz = i >> 2;
        return coords + V3{static_cast<float>(ox) * L.voxel_size, static_cast<float>(oy) * L.voxel_size,
                           static_cast<float>(oz) * L.voxel_size};
      };
      auto edge_vertex = [&](int e) {
        const int a = kMcEdge[e][0], c = kMcEdge[e][1];
        float sa = 0.0f, sc = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {  // register array: select, do not index
          if (i == a) sa = sdf[i];
          if (i == c) sc = sdf[i];
        }
        return mc_interpolate(corner(a), corner(c), sa, sc);
      };
      for (int c = 0; c < 15 && kTriTable[cfg][c] >= 0; c += 3) {
        V3 p[3];
        p[0] = edge_vertex(kTriTable[cfg][c + 2]);
        p[1] = edge_vertex(kTriTable[cfg][c + 1]);
        p[2] = edge_vertex(kTriTable[cfg][c]);
        const V3 n = normalized3(cross3(p[1] - p[0], p[2] - p[0]));
#pragma unroll
        for (int k = 0; k < 3; ++k, ++out) {
          vertices[3 * out] = p[k].x;
          vertices[3 * out + 1] = p[k].y;
          vertices[3 * out + 2] = p[k].z;
          normals[3 * out] = n.x;
          normals[3 * out + 1] = n.y;
          normals[3 * out + 2] = n.z;
          uint32_t col = kDefaultColor;
          if (use_color) {  // MeshIntegrator::updateMeshColor: nearest voxel
            const V3 rel = p[k] - origin;
            const int vx = grid_index(rel.x, L.voxel_size_inv), vy = grid_index(rel.y, L.voxel_size_inv),
                      vz = grid_index(rel.z, L.voxel_size_inv);
            int cs = slot, cx = vx, cy = vy, cz = vz;
            if (static_cast<unsigned>(vx) >= kVps || static_cast<unsigned>(vy) >= kVps ||
                static_cast<unsigned>(vz) >= kVps) {
              // getBlockPtrByCoordinates(vertex)->getVoxelByCoordinates(vertex)
              const int nbx = grid_index(p[k].x, L.block_size_inv), nby = grid_index(p[k].y, L.block_size_inv),
                        nbz = grid_index(p[k].z, L.block_size_inv);
              cs = blocks.find(L, pack_block_key(nbx, nby, nbz));
              const V3 no = V3{static_cast<float>(nbx) * L.block_size, static_cast<float>(nby) * L.block_size,
                               static_cast<float>(nbz) * L.block_size};
              const V3 nr = p[k] - no;
              cx = max(min(grid_index(nr.x, L.voxel_size_inv), kVps - 1), 0);
              cy = max(min(grid_index(nr.y, L.voxel_size_inv), kVps - 1), 0);
              cz = max(min(grid_index(nr.z, L.voxel_size_inv), kVps - 1), 0);
            }
            if (cs != -1) {
              const int lin = cx + kVps * (cy + kVps * cz);
              const float* p = blocks.planes(L, cs);
              if (p[kVoxelsPerBlock + lin] > min_weight)
                col = reinterpret_cast<const uint32_t*>(p)[2 * kVoxelsPerBlock + lin];
            }
          }
          colors[out] = col;
        }
      }
    }
  }
}

__global__ void k_mesh_unpack_idx(const uint64_t* __restrict__ keys, uint32_t n,
                                  int32_t* __restrict__ idx) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x, y, z;
  unpack_block_key(keys[i], x, y, z);
  idx[3 * i] = x;
  idx[3 * i + 1] = y;
  idx[3 * i + 2] = z;
}

}  // namespace cg

using namespace cg;

template <bool kWrite, class Blocks>
static void launch_mesh(unsigned grid, cudaStream_t s, const cg_layer* L, const Blocks& blocks,
                        const uint64_t* keys, const uint32_t* slots, uint32_t n, float min_weight,
                        int32_t use_color, int32_t only_updated, uint32_t* counts,
                        const uint32_t* begin, float* vertices, float* normals, uint32_t* colors) {
  k_mesh_blocks<kWrite, Blocks><<<grid, kMcThreads, 0, s>>>(L->v, blocks, keys, slots, n, min_weight,
                                                            use_color, only_updated, counts, begin,
                                                            vertices, normals, colors);
}

// Runs both passes; the result stays in the context's buffers (mc_*, stage_b) until the next call.
// `sharded` (cg_layer_mesh_sharded): blocks this rank does not hold are looked up across the ranks.
// The collective opening comes after the local scratch is reserved, and from there every exit
// passes the closing barrier, so no rank leaves while a peer still waits for it.  The one host
// synchronisation reads the vertex total and the duplicate-key word together.
static int32_t mesh_to_device(const cg_layer* L, float min_weight, int32_t use_color,
                              int32_t only_updated, bool sharded, size_t* n_blocks,
                              size_t* n_vertices) {
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t n = static_cast<size_t>(L->num_blocks);
  *n_blocks = n;
  *n_vertices = 0;
  ctx->mc_blocks = 0;
  ctx->mc_total = 0;
  if (n == 0 && !sharded) return CG_OK;  // a rank without blocks still takes part in the exchange
  const uint64_t* keys = nullptr;
  const uint32_t* slots = nullptr;
  int32_t rc;
  if (n > 0 && (rc = sort_blocks(L, &keys, &slots))) return rc;
  // counts [n + 1] | vertex_begin [n + 1] | duplicate key (sharded: 8-byte aligned, read back with
  // the total that ends vertex_begin)
  CG_CUDA(ctx->mc_counts.reserve((2 * (n + 1) + 2) * sizeof(uint32_t)));
  CG_CUDA(ctx->mc_index.reserve(n * 3 * sizeof(int32_t)));
  uint32_t* counts = ctx->mc_counts.as<uint32_t>();
  uint32_t* begin = counts + (n + 1);
  unsigned long long* dup_key = reinterpret_cast<unsigned long long*>(counts + 2 * (n + 1));
  size_t tmp = 0;
  CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, counts, begin, static_cast<int>(n + 1), s));
  CG_CUDA(ctx->cub_tmp.reserve(tmp));
  const unsigned grid = static_cast<unsigned>(std::min<size_t>(n, static_cast<size_t>(ctx->num_sms) * 16));
  ShardedBlocks sb{};
  if (sharded && (rc = sharded_mesh_open(L, dup_key, &sb))) return rc;
  const uint32_t nb = static_cast<uint32_t>(n);
  rc = [&]() -> int32_t {
    CG_CUDA(cudaMemsetAsync(counts + n, 0, sizeof(uint32_t), s));
    if (n > 0) {
      ctx->own_launches += 2;
      if (sharded)
        launch_mesh<false>(grid, s, L, sb, keys, slots, nb, min_weight, use_color, only_updated,
                           counts, nullptr, nullptr, nullptr, nullptr);
      else
        launch_mesh<false>(grid, s, L, LocalBlocks{}, keys, slots, nb, min_weight, use_color,
                           only_updated, counts, nullptr, nullptr, nullptr, nullptr);
      k_mesh_unpack_idx<<<grid_for(n, 256), 256, 0, s>>>(keys, nb, ctx->mc_index.as<int32_t>());
    }
    CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, tmp, counts, begin, static_cast<int>(n + 1), s));
    uint32_t back[3] = {0u, 0u, 0u};  // total, duplicate key (low, high word)
    CG_CUDA(cudaMemcpyAsync(back, begin + n, (sharded ? 3 : 1) * sizeof(uint32_t),
                            cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    CG_CUDA(cudaGetLastError());
    const uint32_t total = back[0];
    const unsigned long long dup = (static_cast<unsigned long long>(back[2]) << 32) | back[1];
    if (sharded && dup != kEmptyKey) {  // the same key map on every rank: every rank stops here
      int x, y, z;
      unpack_block_key(dup, x, y, z);
      set_error("cg_layer_mesh_sharded: block (%d, %d, %d) is held by more than one rank", x, y, z);
      return CG_ERR_INVALID_ARG;
    }
    if (total > 0) {
      CG_CUDA(ctx->mc_vertices.reserve(static_cast<size_t>(total) * 3 * sizeof(float)));
      CG_CUDA(ctx->mc_normals.reserve(static_cast<size_t>(total) * 3 * sizeof(float)));
      CG_CUDA(ctx->mc_colors.reserve(static_cast<size_t>(total) * sizeof(uint32_t)));
      ctx->own_launches += 1;
      float* v = ctx->mc_vertices.as<float>();
      float* nrm = ctx->mc_normals.as<float>();
      uint32_t* col = ctx->mc_colors.as<uint32_t>();
      if (sharded)
        launch_mesh<true>(grid, s, L, sb, keys, slots, nb, min_weight, use_color, only_updated,
                          counts, begin, v, nrm, col);
      else
        launch_mesh<true>(grid, s, L, LocalBlocks{}, keys, slots, nb, min_weight, use_color,
                          only_updated, counts, begin, v, nrm, col);
      CG_CUDA(cudaGetLastError());
    }
    ctx->mc_blocks = n;
    ctx->mc_total = total;
    *n_vertices = total;
    return CG_OK;
  }();
  if (sharded) {
    const int32_t rb = sharded_mesh_close(ctx);
    if (rc == CG_OK) rc = rb;
  }
  return rc;
}

static int32_t mesh_fetch(cg_context* ctx, size_t capacity_blocks, size_t capacity_vertices,
                          int32_t* block_idx, uint32_t* vertex_begin, float* vertices,
                          float* normals, uint8_t* colors) {
  cudaStream_t s = ctx->stream;
  const size_t n = ctx->mc_blocks, total = ctx->mc_total;
  if ((block_idx || vertex_begin) && capacity_blocks < n) {
    set_error("cg_layer_mesh: capacity %zu < %zu blocks", capacity_blocks, n);
    return CG_ERR_INVALID_ARG;
  }
  if ((vertices || normals || colors) && capacity_vertices < total) {
    set_error("cg_layer_mesh: capacity %zu < %zu vertices", capacity_vertices, total);
    return CG_ERR_INVALID_ARG;
  }
  if (n == 0) {
    if (vertex_begin) vertex_begin[0] = 0;
    return CG_OK;
  }
  if (vertex_begin)
    CG_CUDA(cudaMemcpyAsync(vertex_begin, ctx->mc_counts.as<uint32_t>() + (n + 1),
                            (n + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  if (block_idx)
    CG_CUDA(cudaMemcpyAsync(block_idx, ctx->mc_index.p, n * 3 * sizeof(int32_t),
                            cudaMemcpyDeviceToHost, s));
  if (total > 0) {
    if (vertices)
      CG_CUDA(cudaMemcpyAsync(vertices, ctx->mc_vertices.p, total * 12, cudaMemcpyDeviceToHost, s));
    if (normals)
      CG_CUDA(cudaMemcpyAsync(normals, ctx->mc_normals.p, total * 12, cudaMemcpyDeviceToHost, s));
    if (colors)
      CG_CUDA(cudaMemcpyAsync(colors, ctx->mc_colors.p, total * 4, cudaMemcpyDeviceToHost, s));
  }
  CG_CUDA(cudaStreamSynchronize(s));
  return CG_OK;
}

extern "C" {

int32_t cg_layer_mesh(const cg_layer* L, float min_weight, int32_t use_color, int32_t only_updated,
                      size_t capacity_blocks, size_t capacity_vertices, int32_t* block_idx,
                      uint32_t* vertex_begin, float* vertices, float* normals, uint8_t* colors,
                      size_t* num_blocks_out, size_t* num_vertices_out) {
  if (!L) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(L->ctx->device));
  size_t nb = 0, nv = 0;
  int32_t rc = mesh_to_device(L, min_weight, use_color, only_updated, false, &nb, &nv);
  if (num_blocks_out) *num_blocks_out = nb;
  if (num_vertices_out) *num_vertices_out = nv;
  if (rc) return rc;
  if (!block_idx && !vertex_begin && !vertices && !normals && !colors) return CG_OK;
  return mesh_fetch(L->ctx, capacity_blocks, capacity_vertices, block_idx, vertex_begin, vertices,
                    normals, colors);
}

int32_t cg_layer_mesh_sharded(const cg_layer* owned, float min_weight, int32_t use_color,
                              int32_t only_updated, size_t capacity_blocks, size_t capacity_vertices,
                              int32_t* block_idx, uint32_t* vertex_begin, float* vertices,
                              float* normals, uint8_t* colors, size_t* num_blocks_out,
                              size_t* num_vertices_out) {
  if (!owned) return CG_ERR_INVALID_ARG;
  if (!owned->ctx->comm) {
    set_error("cg_layer_mesh_sharded: call cg_comm_init first");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(owned->ctx->device));
  size_t nb = 0, nv = 0;
  int32_t rc = mesh_to_device(owned, min_weight, use_color, only_updated, true, &nb, &nv);
  if (num_blocks_out) *num_blocks_out = nb;
  if (num_vertices_out) *num_vertices_out = nv;
  if (rc) return rc;
  if (!block_idx && !vertex_begin && !vertices && !normals && !colors) return CG_OK;
  return mesh_fetch(owned->ctx, capacity_blocks, capacity_vertices, block_idx, vertex_begin,
                    vertices, normals, colors);
}

int32_t cg_mesh_fetch(cg_context* ctx, size_t capacity_blocks, size_t capacity_vertices,
                      int32_t* block_idx, uint32_t* vertex_begin, float* vertices, float* normals,
                      uint8_t* colors) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(ctx->device));
  return mesh_fetch(ctx, capacity_blocks, capacity_vertices, block_idx, vertex_begin, vertices,
                    normals, colors);
}

}  // extern "C"
