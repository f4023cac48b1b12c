// Explicit instantiation of the prover-side kernels and drivers for G2 (Fp2).
#include "prover_impl.cuh"

namespace gsi {
template void fixed_table_release<Fp2Ops>(gs_ctx*);
template int fixed_table_rebuild<Fp2Ops>(gs_ctx*, int);
template int batch_commit_impl<Fp2Ops>(gs_ctx*, size_t, int, int, const gs_fr*, size_t, const gs_fr*, size_t, size_t, const void*, void*);
template int proof_element<Fp2Ops>(gs_ctx*, Scratch&, size_t, int, bool, const fr*, const void*, size_t, const void*, size_t, bool, int,
                               const fr*, size_t, const fr*, Aff<Fp2Ops>*);
template int rerand_commit<Fp2Ops>(gs_ctx*, size_t, int, const fr*, const Aff<Fp2Ops>*, Aff<Fp2Ops>*);
template int rerand_element<Fp2Ops>(gs_ctx*, Scratch&, size_t, int, bool, const fr*, const fr*, const void*, size_t,
                                const Aff<Fp2Ops>*, size_t, bool, int, const fr*, const fr*, const Aff<Fp2Ops>*, Aff<Fp2Ops>*);
template int fixed_com_add<Fp2Ops>(gs_ctx*, size_t, int, int, const fr*, size_t, const fr*, size_t, const Aff<Fp2Ops>*, Aff<Fp2Ops>*);
template int com_matmul_impl<Fp2Ops>(gs_ctx*, size_t, size_t, size_t, const gs_fr*, const void*, void*);
}  // namespace gsi
