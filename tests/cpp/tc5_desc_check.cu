// The tcgen05 descriptors built by sdk_b200/csrc/tc5_layout.cuh, printed in the format of tests/golden/tc5_descriptors.json
// (the same fields packed by CUTLASS's bit-field structs, tests/golden/make_tc5_descriptors.cu).  Host-only; compiled with nvcc.
#include <cstdio>
#include <cstdint>
#include "../../sdk_b200/csrc/tc5_layout.cuh"
int main() {
  printf("{\"instr_desc\": \"0x%08x\",\n \"smem_desc\": {", b200pir::tc5_instr_desc());
  const char* sep = "";
  for (uint32_t addr : {0x0u, 0x400u, 0x12340u, 0x3FFF0u}) {
    printf("%s\"0x%x\": \"0x%016llx\"", sep, addr, (unsigned long long)b200pir::tc5_smem_desc(addr));
    sep = ", ";
  }
  printf("}}\n");
  return 0;
}
