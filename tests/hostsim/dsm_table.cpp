// dsm_table.cpp -- TEST INFRASTRUCTURE ONLY.
//
// The table phase of the verification ladder (item_dsm_table, kernels.cuh) on the CPU, compiled with g++ from the same
// headers as hostsim.cpp, so that the rows the ladder reads can be checked against Python integers.  It is never linked
// into, or called by, the product library.
#include <cstddef>
#include <vector>

#include "../../secp256k1-voi_b200/csrc/kernels.cuh"

using namespace s256;
#define EXPORT extern "C" __attribute__((visibility("default")))

EXPORT int sim_dsm_table_rows() { return DSM_TS; }

// pt65: n SEC 1 uncompressed keys, decoded as the kernels decode them (an invalid key becomes G; valid[i] = 0).
// rows: n x TS x 64 bytes, row k of item i at (i TS + k - 1) 64 as x || y, canonical big-endian; zall: n x 32 bytes.
EXPORT void sim_dsm_table(const uint8_t *pt65, size_t n, uint8_t *rows, uint8_t *zall, uint8_t *valid) {
    std::vector<apt> aff(n);
    std::vector<pt> tbl(n * DSM_TSTRIDE);
    fe_ops<DSM_VT> f;
    for (size_t i = 0; i < n; i++) {
        valid[i] = item_decode_uncompressed(aff[i], pt65 + 65 * i);
        item_dsm_table(f, i, aff.data(), tbl.data());
        const char *base = reinterpret_cast<const char *>(tbl.data() + i * (size_t)DSM_TSTRIDE);
        const apt *A = reinterpret_cast<const apt *>(base);
        for (int k = 0; k < DSM_TS; k++) {
            fe x, y;
            fe_normalize(x, A[k].x);
            fe_normalize(y, A[k].y);
            fe_to_be32(rows + (i * DSM_TS + k) * 64, x);
            fe_to_be32(rows + (i * DSM_TS + k) * 64 + 32, y);
        }
        fe z;
        fe_normalize(z, reinterpret_cast<const fe *>(base + DSM_U_OFF)[0]);
        fe_to_be32(zall + 32 * i, z);
    }
}
