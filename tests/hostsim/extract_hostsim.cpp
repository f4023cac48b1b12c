// Host instantiation of csrc/extract.cuh (tests only; never linked into the product): the key recoding and the
// fixed-key walk that k_extract runs, checked against the big-integer oracle by tests/test_extract_hostsim.py.
#include <cstring>
#include "../../groth-sahai-rs_b200/csrc/extract.cuh"
using namespace gs;

#define LD(T, v, p) T v; memcpy(&v, p, sizeof(T))
#define ST(p, v) memcpy(p, &v, sizeof(v))
extern "C" {
// c.1 - key * c.0 (com = two points, key in Montgomery form)
void hs_extract_g1(void* r, const void* com /* two G1 */, const void* key_mont) {
  LD(fr, k, key_mont); uint32_t kk[8]; fr_from_mont(kk, k);
  const g1_aff* c = (const g1_aff*)com; g1_aff o;
  extract_single<FpOps>(o, c[0], c[1], make_extract_digits<FpOps>(kk)); ST(r, o); }
void hs_extract_g2(void* r, const void* com /* two G2 */, const void* key_mont) {
  LD(fr, k, key_mont); uint32_t kk[8]; fr_from_mont(kk, k);
  const g2_aff* c = (const g2_aff*)com; g2_aff o;
  extract_single<Fp2Ops>(o, c[0], c[1], make_extract_digits<Fp2Ops>(kk)); ST(r, o); }
// the digits of a key: 4 parts x 33 digits, then the number of positions as one byte
void hs_extract_digits(void* out /* 133 B */, const void* key_mont, int g2) {
  LD(fr, k, key_mont); uint32_t kk[8]; fr_from_mont(kk, k);
  extract_digits d = g2 ? make_extract_digits<Fp2Ops>(kk) : make_extract_digits<FpOps>(kk);
  memcpy(out, d.d, 132); ((uint8_t*)out)[132] = (uint8_t)d.npos; }
}
