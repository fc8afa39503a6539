// Local node numbering of a tet and of its faces, shared by the boundary / strike kernels (gains.cu) and the support
// kernels (support.cu).  Local P2 order is the reference's [v0, m01, v1, m12, v2, m02, m03, m13, m23, v3]
// (shape_func.P2_NODES); face f of a tet is the face opposite corner f.
#pragma once
#include <cstdint>

namespace ds {

namespace {

// local node of tet corner j (shape_func.CORNER_LOCAL)
__device__ __forceinline__ int corner_local(int order, int j) { return order == 1 ? j : (j == 3 ? 9 : 2 * j); }

// the (l, m) barycentric pair of P2 node a (shape_func.P2_NODES): l == m a corner, else the mid-edge node of (l, m)
__constant__ signed char c_p2_l[10] = {0, 0, 1, 1, 2, 2, 0, 1, 2, 3};
__constant__ signed char c_p2_m[10] = {0, 1, 1, 2, 2, 0, 3, 3, 3, 3};

// The tet-local nodes of face f: its three corners (ascending corner index), then for P2 its three mid-edge nodes
// (ascending local index).  Returns the count, 3 or 6.
__device__ __forceinline__ int face_local_nodes(int order, int f, int (&ln)[6]) {
    int q = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (j != f) ln[q++] = corner_local(order, j);
    if (order == 1) return 3;
#pragma unroll
    for (int a = 0; a < 10; ++a)
        if (c_p2_l[a] != c_p2_m[a] && c_p2_l[a] != f && c_p2_m[a] != f) ln[q++] = a;
    return 6;
}

}  // namespace

}  // namespace ds
