// Explicit instantiation of the prover-side kernels and drivers for G1 (Fp).
#include "prover_impl.cuh"

namespace gsi {
template void fixed_table_release<FpOps>(gs_ctx*);
template int fixed_table_rebuild<FpOps>(gs_ctx*, int);
template int batch_commit_impl<FpOps>(gs_ctx*, size_t, int, int, const gs_fr*, size_t, const gs_fr*, size_t, size_t, const void*, void*);
template int proof_element<FpOps>(gs_ctx*, Scratch&, size_t, int, bool, const fr*, const void*, size_t, const void*, size_t, bool, int,
                               const fr*, size_t, const fr*, Aff<FpOps>*);
template int rerand_commit<FpOps>(gs_ctx*, size_t, int, const fr*, const Aff<FpOps>*, Aff<FpOps>*);
template int rerand_element<FpOps>(gs_ctx*, Scratch&, size_t, int, bool, const fr*, const fr*, const void*, size_t,
                                const Aff<FpOps>*, size_t, bool, int, const fr*, const fr*, const Aff<FpOps>*, Aff<FpOps>*);
template int fixed_com_add<FpOps>(gs_ctx*, size_t, int, int, const fr*, size_t, const fr*, size_t, const Aff<FpOps>*, Aff<FpOps>*);
template int com_matmul_impl<FpOps>(gs_ctx*, size_t, size_t, size_t, const gs_fr*, const void*, void*);
}  // namespace gsi
