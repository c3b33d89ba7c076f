// Freeze the tcgen05 descriptors as CUTLASS packs them: the fields sdk_b200/csrc/tc5_layout.cuh sets, written through the
// bit-field structs of cute/arch/mma_sm100_desc.hpp.  tests/cpp/tc5_desc_check.cu prints the same descriptors as
// tc5_layout.cuh packs them by hand, and tests/test_host_and_abi.py compares the two.  Host-only:
//   nvcc -std=c++17 -I<cutlass>/include -o make_tc5_descriptors tests/golden/make_tc5_descriptors.cu
//   ./make_tc5_descriptors > tests/golden/tc5_descriptors.json
#include <cstdio>
#include <cstdint>
#include <cutlass/version.h>
#include <cute/arch/mma_sm100_desc.hpp>
#include "../../sdk_b200/csrc/tc5_layout.cuh"
int main() {
  cute::UMMA::InstrDescriptor d = {};
  d.desc_ = 0;
  d.c_format_ = uint8_t(cute::UMMA::CFormat::S32);
  d.a_format_ = uint8_t(cute::UMMA::S8Format::UINT8);
  d.b_format_ = uint8_t(cute::UMMA::S8Format::UINT8);
  d.a_major_ = uint8_t(cute::UMMA::Major::K);
  d.b_major_ = uint8_t(cute::UMMA::Major::K);
  d.n_dim_ = b200pir::TC5_N >> 3;
  d.m_dim_ = b200pir::TC5_M >> 4;
  printf("{\"source\": \"CUTLASS %d.%d.%d, cute/arch/mma_sm100_desc.hpp: UMMA::InstrDescriptor, UMMA::SmemDescriptor "
         "(tests/golden/make_tc5_descriptors.cu)\",\n \"instr_desc\": \"0x%08x\",\n \"smem_desc\": {",
         CUTLASS_MAJOR, CUTLASS_MINOR, CUTLASS_PATCH, d.desc_);
  const char* sep = "";
  for (uint32_t addr : {0x0u, 0x400u, 0x12340u, 0x3FFF0u}) {
    cute::UMMA::SmemDescriptor s;
    s.desc_ = 0;
    s.start_address_ = addr >> 4;
    s.leading_byte_offset_ = b200pir::TC5_LBO >> 4;
    s.stride_byte_offset_ = b200pir::TC5_SBO >> 4;
    s.version_ = 1;
    s.base_offset_ = 0;
    s.lbo_mode_ = 0;
    s.layout_type_ = uint8_t(cute::UMMA::LayoutType::SWIZZLE_NONE);
    printf("%s\"0x%x\": \"0x%016llx\"", sep, addr, (unsigned long long)s.desc_);
    sep = ", ";
  }
  printf("}}\n");
  return 0;
}
