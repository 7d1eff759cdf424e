/* Type-only stand-in for <CL/cl_gl.h> / <CL/cl.h>.
 *
 * TEST INFRASTRUCTURE.  This image has no OpenCL headers.  The reference's
 * host files (list/vector/matrix/camera/kd_tree/model .c) use nothing from
 * OpenCL except these scalar and 16-byte vector typedefs, so this shim is all
 * that is needed to compile them UNMODIFIED from $CLPT_REFERENCE (see
 * oracle/Makefile).  Layouts follow the Khronos cl_platform.h: 16-byte
 * unions addressed as .s[i]; the 3-component types alias the 4-component ones.
 */
#ifndef ORACLE_SHIM_CL_H
#define ORACLE_SHIM_CL_H
#include <stddef.h>
#include <stdint.h>
typedef int32_t cl_int;
typedef uint32_t cl_uint;
typedef float cl_float;
typedef union { cl_float s[4]; } __attribute__((aligned(16))) cl_float4;
typedef cl_float4 cl_float3;
typedef union { cl_int s[4]; } __attribute__((aligned(16))) cl_int4;
typedef cl_int4 cl_int3;
#endif
