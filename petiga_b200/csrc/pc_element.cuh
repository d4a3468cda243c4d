// pc_element.cuh -- per-element rules of the reference that several quadrature kernels restate, written once.
//
//   element_id, closure_index   IGANextElement and the element's node map          src/petigaelem.c:388-395,703-719
//   inverse_map                 InverseMap, order 1                                src/petigamapinv.f90.in:28-31
//   value_offset                where IGAElementAssembleMat's entry lands           src/petigaelem.c:1525-1559
//                               (its column position is seg_position, pc_layout.h)
// The Dirichlet/Neumann lists and the element fix-up are still written out in each kernel: moved here, they changed the
// register allocation of some instantiations (DESIGN 3.1).  Tuned restatements stay where they are: the affine scatter of
// quad_sf_kernel, the packed positions and aggregate fix-up of the third-generation and separable kernels, and the
// reciprocal inverse of sf3_geom_kernel.
#pragma once
#include "pc_device.h"

namespace pc {

// IGANextElement (src/petigaelem.c:388-395): local element index -> element coordinates, axis 0 fastest
__host__ __device__ __forceinline__ void element_id(const DevAxis ax[3], int elem, int ID[3]) {
  for (int d = 0; d < 3; d++) {
    const int c = elem % ax[d].ew;
    elem /= ax[d].ew;
    ID[d] = c + ax[d].es;
  }
}

// element->mapping[a] (src/petigaelem.c:703-719): ghost-box index of local node ai = (a0, a1, a2) of element ID.
// Axes >= DIM have one node in the ghost box and add nothing.
template <int DIM>
__host__ __device__ __forceinline__ int closure_index(const DevAxis ax[3], const int ID[3], const int ai[3]) {
  const int g0 = ax[0].offset[ID[0]] + ai[0] - ax[0].gs;
  const int g1 = (DIM > 1) ? ax[1].offset[ID[1]] + ai[1] - ax[1].gs : 0;
  const int g2 = (DIM > 2) ? ax[2].offset[ID[2]] + ai[2] - ax[2].gs : 0;
  return g0 + ax[0].gw * (g1 + ax[1].gw * g2);
}

// InverseMap, order 1 (src/petigamapinv.f90.in:28-31): from X1[i][d] = dX_i/du_d writes E[d][i] = du_d/dx_i (entries
// d, i < DIM) and returns det X1.  Every entry is a cofactor divided by det: results depend on that rounding.
template <int DIM>
__host__ __device__ __forceinline__ double inverse_map(const double X1[3][3], double E[3][3]) {
  if (DIM == 1) {
    E[0][0] = 1.0 / X1[0][0];
    return X1[0][0];
  }
  if (DIM == 2) {
    const double det = X1[0][0] * X1[1][1] - X1[0][1] * X1[1][0];
    E[0][0] = X1[1][1] / det; E[0][1] = -X1[0][1] / det; E[1][0] = -X1[1][0] / det; E[1][1] = X1[0][0] / det;
    return det;
  }
  const double a00 = X1[0][0], a01 = X1[0][1], a02 = X1[0][2], a10 = X1[1][0], a11 = X1[1][1], a12 = X1[1][2], a20 = X1[2][0], a21 = X1[2][1], a22 = X1[2][2];
  const double det = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
  E[0][0] = (a11 * a22 - a12 * a21) / det; E[0][1] = -(a01 * a22 - a02 * a21) / det; E[0][2] = (a01 * a12 - a02 * a11) / det;
  E[1][0] = -(a10 * a22 - a12 * a20) / det; E[1][1] = (a00 * a22 - a02 * a20) / det; E[1][2] = -(a00 * a12 - a02 * a10) / det;
  E[2][0] = (a10 * a21 - a11 * a20) / det; E[2][1] = -(a00 * a21 - a01 * a20) / det; E[2][2] = (a00 * a11 - a01 * a10) / det;
  return det;
}

// Offset in the value array of entry (row field i, column field j) at closed-form position pos (seg_position) of a row whose
// blocks start at base.  BAIJ (block = 1) stores dof x dof blocks column-major; AIJ expands the row into dof scalar rows of
// W012 * dof columns, W012 = W0 W1 W2 the row's width.
__host__ __device__ __forceinline__ size_t value_offset(int64_t base, int pos, int dof, int block, int i, int j, int W012) {
  if (dof == 1) return (size_t)(base + pos);
  if (block) return (size_t)(base + pos) * dof * dof + j * dof + i;
  return (size_t)base * dof * dof + (size_t)i * W012 * dof + (size_t)pos * dof + j;
}

}  // namespace pc
