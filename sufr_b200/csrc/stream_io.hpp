// File <-> device streaming through rings of pinned host buffers: the sections of a `.sufr` file into device memory
// (sufr_b200_index_open) and a device result into its `.sufr` file (sufr_b200_create, sufr_b200_create_multi).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/sufr_b200.h"

namespace sufr {

struct FileSection {
    uint64_t file_off;
    uint64_t len;
    void* dev;
};
void upload_file_sections(int fd, const std::string& path, int device, cudaStream_t stream,
                          const std::vector<FileSection>& sections);

void stream_result_to_file(int device, cudaStream_t stream, const SufrB200Args& args, const SufrB200Result& r,
                           uint8_t** host_text);

}  // namespace sufr
