/* tests/hostemu/transform_emu.cpp -- DEVELOPMENT/TEST HARNESS, NOT A PRODUCT PATH.
 *
 * The per-vertex body of kzgpu_mesh_transform (kz_transform.h, the code k_transform_vertices runs) compiled for the host, so that the
 * CPU suite can hold it to a numpy restatement of the C++ host's Transform::point / Transform::normal and the OBJ loader's
 * normalisation, bit for bit (transform_emu.py).
 */
#include "../../nano-kazen_b200/csrc/kz_transform.h"
#include <stddef.h>

extern "C" {

/* n positions (and normals, if nrm != NULL) placed by the row-major matrix m and inverse inv, as k_transform_vertices places them */
int kzemu_transform(const float *m, const float *inv, const float *pos, const float *nrm, size_t n, float *out_pos, float *out_nrm) {
    for (size_t i = 0; i < n; ++i) {
        kz_transform_point(m, pos + 3 * i, out_pos + 3 * i);
        if (nrm) kz_transform_normal(inv, nrm + 3 * i, out_nrm + 3 * i);
    }
    return 0;
}

}  // extern "C"
