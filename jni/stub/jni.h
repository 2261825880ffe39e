/*
 * jni/stub/jni.h — COMPILE-CHECK STUB of the Java Native Interface header.
 *
 * This image has no JDK (no jni.h on disk), so siesta_gpu_jni.c is compiled here against this stub: the type names and
 * the signatures of the JNIEnv functions the shim uses follow the JNI specification (Java SE "JNI Functions"), but the
 * function table below holds ONLY those functions and NOT in the specification's slot order - a library built against
 * this file must never be loaded into a JVM.  For deployment build with the JDK's header:
 *     make -C jni JNI_INCLUDES="-I$JAVA_HOME/include -I$JAVA_HOME/include/linux"
 */
#ifndef SIESTA_STUB_JNI_H
#define SIESTA_STUB_JNI_H
#include <stdint.h>

#define SIESTA_JNI_STUB 1
#define JNIEXPORT __attribute__((visibility("default")))
#define JNICALL
#define JNI_ABORT 2

typedef int32_t jint;
typedef int64_t jlong;
typedef uint8_t jboolean;
typedef jint jsize;
struct _jobject;
typedef struct _jobject* jobject;
typedef jobject jclass;
typedef jobject jarray;
typedef jarray jintArray;
typedef jarray jlongArray;
typedef jobject jthrowable;

struct JNINativeInterface_;
typedef const struct JNINativeInterface_* JNIEnv;

struct JNINativeInterface_ {
    jclass (*FindClass)(JNIEnv* env, const char* name);
    jint (*ThrowNew)(JNIEnv* env, jclass clazz, const char* msg);
    jboolean (*ExceptionCheck)(JNIEnv* env);
    jsize (*GetArrayLength)(JNIEnv* env, jarray array);
    jintArray (*NewIntArray)(JNIEnv* env, jsize len);
    jlongArray (*NewLongArray)(JNIEnv* env, jsize len);
    jint* (*GetIntArrayElements)(JNIEnv* env, jintArray array, jboolean* isCopy);
    jlong* (*GetLongArrayElements)(JNIEnv* env, jlongArray array, jboolean* isCopy);
    void (*ReleaseIntArrayElements)(JNIEnv* env, jintArray array, jint* elems, jint mode);
    void (*ReleaseLongArrayElements)(JNIEnv* env, jlongArray array, jlong* elems, jint mode);
    void (*SetIntArrayRegion)(JNIEnv* env, jintArray array, jsize start, jsize len, const jint* buf);
    void (*SetLongArrayRegion)(JNIEnv* env, jlongArray array, jsize start, jsize len, const jlong* buf);
    void (*GetIntArrayRegion)(JNIEnv* env, jintArray array, jsize start, jsize len, jint* buf);
    void (*GetLongArrayRegion)(JNIEnv* env, jlongArray array, jsize start, jsize len, jlong* buf);
    void* (*GetPrimitiveArrayCritical)(JNIEnv* env, jarray array, jboolean* isCopy);
    void (*ReleasePrimitiveArrayCritical)(JNIEnv* env, jarray array, void* carray, jint mode);
};
#endif
