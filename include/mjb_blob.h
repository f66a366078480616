/*
 * mjb_blob.h — packed model blob format (public, header-only, plain C).
 *
 * The MJCF compiler (csrc/mjcf_compile.cpp) turns an MJCF file into ONE packed,
 * position-independent blob: a header, a directory of named fields and the
 * field payloads (int32 or float64).  It plays the role of `MjModel` in the
 * reference (MuJoCo_Gym/mujoco_parent.py:126 `mj.MjModel.from_xml_path`).
 * Consumers: the CUDA batch (converts to fp32 SoA device constants), the host
 * Python layer (index tables, name lookups) and the fp64 CPU oracle (oracle/).
 */
#ifndef MJB_BLOB_H_
#define MJB_BLOB_H_

#if defined(__CUDACC_RTC__)
/* NVRTC (the step kernel specialised at batch creation) compiles without host headers */
typedef signed char int8_t; typedef unsigned char uint8_t; typedef short int16_t; typedef unsigned short uint16_t;
typedef int int32_t; typedef unsigned int uint32_t; typedef long long int64_t; typedef unsigned long long uint64_t;
#else
#include <stdint.h>
#include <string.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MJB_BLOB_MAGIC "MJBLOB1"
#define MJB_FIELD_NAME_LEN 32

enum { MJB_DTYPE_I32 = 0, MJB_DTYPE_F64 = 1 };

typedef struct mjb_blob_header {
  char magic[8];       /* "MJBLOB1\0" */
  int32_t nfields;
  int32_t reserved;
  int64_t total_bytes;
} mjb_blob_header;

typedef struct mjb_blob_field {
  char name[MJB_FIELD_NAME_LEN];
  int32_t dtype;       /* MJB_DTYPE_* */
  int32_t count;       /* number of elements */
  int64_t offset;      /* byte offset from blob start, 8-byte aligned */
} mjb_blob_field;

/* geom / joint / sensor / object type codes (values follow MuJoCo's enums so
 * that `model.geom(n).type` style queries keep their meaning). */
enum { MJB_GEOM_PLANE = 0, MJB_GEOM_SPHERE = 2, MJB_GEOM_CAPSULE = 3, MJB_GEOM_BOX = 6 };
enum { MJB_JNT_FREE = 0, MJB_JNT_SLIDE = 2, MJB_JNT_HINGE = 3 };
enum { MJB_SENS_TOUCH = 0, MJB_SENS_ACCELEROMETER = 1, MJB_SENS_VELOCIMETER = 2, MJB_SENS_GYRO = 3,
       MJB_SENS_RANGEFINDER = 7, MJB_SENS_JOINTPOS = 9, MJB_SENS_JOINTVEL = 10, MJB_SENS_FRAMEPOS = 26,
       MJB_SENS_FRAMEQUAT = 27, MJB_SENS_FRAMEXAXIS = 28, MJB_SENS_FRAMEYAXIS = 29, MJB_SENS_FRAMEZAXIS = 30,
       MJB_SENS_FRAMELINVEL = 31, MJB_SENS_FRAMEANGVEL = 32 };
/* sensor_datatype: MuJoCo's mjtDataType */
enum { MJB_DATA_REAL = 0, MJB_DATA_POSITIVE = 1, MJB_DATA_AXIS = 2, MJB_DATA_QUATERNION = 3 };
/* object types: MuJoCo's mjtObj (XBODY = the body frame, BODY = its inertial frame for frame sensors) */
enum { MJB_OBJ_BODY = 1, MJB_OBJ_XBODY = 2, MJB_OBJ_JOINT = 3, MJB_OBJ_GEOM = 5, MJB_OBJ_SITE = 6, MJB_OBJ_CAMERA = 7,
       MJB_OBJ_ACTUATOR = 19, MJB_OBJ_SENSOR = 20 };
enum { MJB_INT_EULER = 0, MJB_INT_RK4 = 1 };

#if !defined(__CUDACC_RTC__)
static inline const mjb_blob_field* mjb_blob_find(const void* blob, const char* name) {
  const mjb_blob_header* h = (const mjb_blob_header*)blob;
  const mjb_blob_field* f = (const mjb_blob_field*)((const char*)blob + sizeof(mjb_blob_header));
  for (int i = 0; i < h->nfields; i++)
    if (strncmp(f[i].name, name, MJB_FIELD_NAME_LEN) == 0) return &f[i];
  return 0;
}
static inline const int32_t* mjb_blob_i32(const void* blob, const char* name, int* count) {
  const mjb_blob_field* f = mjb_blob_find(blob, name);
  if (!f || f->dtype != MJB_DTYPE_I32) { if (count) *count = -1; return 0; }
  if (count) *count = f->count;
  return (const int32_t*)((const char*)blob + f->offset);
}
static inline const double* mjb_blob_f64(const void* blob, const char* name, int* count) {
  const mjb_blob_field* f = mjb_blob_find(blob, name);
  if (!f || f->dtype != MJB_DTYPE_F64) { if (count) *count = -1; return 0; }
  if (count) *count = f->count;
  return (const double*)((const char*)blob + f->offset);
}
#endif

#ifdef __cplusplus
}
#endif
#endif  /* MJB_BLOB_H_ */
