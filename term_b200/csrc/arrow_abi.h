// Arrow C Data Interface (https://arrow.apache.org/docs/format/CDataInterface.html) and C Device Data Interface
// (https://arrow.apache.org/docs/format/CDeviceDataInterface.html) structs: row ingestion (tables.cu) and row-mask export (capi.cpp)
#pragma once
#include <cstddef>
#include <cstdint>

namespace tg {

struct ArrowSchema {
    const char* format;
    const char* name;
    const char* metadata;
    int64_t flags;
    int64_t n_children;
    struct ArrowSchema** children;
    struct ArrowSchema* dictionary;
    void (*release)(struct ArrowSchema*);
    void* private_data;
};
struct ArrowArray {
    int64_t length;
    int64_t null_count;
    int64_t offset;
    int64_t n_buffers;
    int64_t n_children;
    const void** buffers;
    struct ArrowArray** children;
    struct ArrowArray* dictionary;
    void (*release)(struct ArrowArray*);
    void* private_data;
};

struct ArrowDeviceArray {
    ArrowArray array;
    int64_t device_id;
    int32_t device_type;
    void* sync_event;
    int64_t reserved[3];
};
static_assert(sizeof(ArrowDeviceArray) == 128 && offsetof(ArrowDeviceArray, device_type) == 88 && offsetof(ArrowDeviceArray, sync_event) == 96,
              "ArrowDeviceArray layout");
constexpr int32_t ARROW_DEVICE_CPU = 1, ARROW_DEVICE_CUDA = 2, ARROW_DEVICE_CUDA_HOST = 3, ARROW_DEVICE_CUDA_MANAGED = 13;


}  // namespace tg
