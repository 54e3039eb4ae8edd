/* Minimal declaration of the DLPack in-memory tensor ABI (DLPack v0.x / v1.0 unversioned
 * struct: the object behind the "dltensor" PyCapsule of torch.utils.dlpack.to_dlpack and
 * tf.experimental.dlpack.to_dlpack).  Layout-compatible with dmlc/dlpack's dlpack.h; guarded so
 * that the real header can be included alongside.  libiris only READS these structs: tensors
 * stay owned by the producing framework (its deleter is never called here).
 */
#ifndef IRIS_DLPACK_H_
#define IRIS_DLPACK_H_

#include <stdint.h>

#ifndef DLPACK_DLPACK_H_
#ifdef __cplusplus
extern "C" {
#endif

enum { kDLCPU = 1, kDLCUDA = 2, kDLCUDAHost = 3, kDLCUDAManaged = 13 };
enum { kDLInt = 0, kDLUInt = 1, kDLFloat = 2, kDLBfloat = 4 };

typedef struct {
    int32_t device_type;
    int32_t device_id;
} DLDevice;

typedef struct {
    uint8_t code;
    uint8_t bits;
    uint16_t lanes;
} DLDataType;

typedef struct {
    void* data;
    DLDevice device;
    int32_t ndim;
    DLDataType dtype;
    int64_t* shape;
    int64_t* strides; /* in elements; NULL = compact row-major */
    uint64_t byte_offset;
} DLTensor;

typedef struct DLManagedTensor {
    DLTensor dl_tensor;
    void* manager_ctx;
    void (*deleter)(struct DLManagedTensor* self);
} DLManagedTensor;

#ifdef __cplusplus
}
#endif
#endif /* DLPACK_DLPACK_H_ */
#endif /* IRIS_DLPACK_H_ */
