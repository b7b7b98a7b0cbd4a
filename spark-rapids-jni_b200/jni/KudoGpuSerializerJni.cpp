// KudoGpuSerializerJni.cpp -- JNI binding of com.nvidia.spark.rapids.jni.kudo.KudoGpuSerializer over libsrj_b200.so.
// Split takes flat tables; assemble takes flat and nested (LIST / STRUCT) schemas.  Replaces src/main/cpp/src/KudoGpuSerializerJni.cpp:22-140 of the reference: the same two symbols and the
// same return conventions (splitAndSerializeToDevice: six longs = {address, size, rmm::device_buffer*} of the partitions
// and of the size_t offsets; assembleFromDeviceRawNative: an AssembleResult(buffer handle, buffer size, column_view
// handles) whose columns, nested ones included, are views into ONE shared rmm buffer).
#include "srj_jni_common.hpp"

using namespace srjshim;

namespace {
size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
constexpr size_t kSplitAlign = 64;   // shuffle_split_detail.hpp:89: every output column buffer starts 64-byte aligned

// one flattened column of the assembled table: where its buffers lie in the shared buffer
struct Slot {
  size_t mask, offsets, data;
};

bool has_offsets(int32_t t) { return t == SRJ_STRING || t == SRJ_LIST; }

// the srj_column tree rooted at flattened column pos++ (children descriptors kept in kids[c])
srj_column build_srj(int& pos, const std::vector<int32_t>& types, const std::vector<int32_t>& scales, const std::vector<int32_t>& nch,
                     const std::vector<int64_t>& rows, const std::vector<Slot>& at, uint8_t* base, std::vector<std::vector<srj_column>>& kids)
{
  const int c = pos++;
  srj_column s{};
  s.type_id   = types[c];
  s.scale     = scales[c];
  s.size      = rows[c];
  s.null_mask = reinterpret_cast<uint32_t*>(base + at[c].mask);
  s.offsets   = has_offsets(types[c]) ? reinterpret_cast<int32_t*>(base + at[c].offsets) : nullptr;
  s.data      = (types[c] == SRJ_LIST || types[c] == SRJ_STRUCT) ? nullptr : base + at[c].data;
  if (types[c] == SRJ_LIST || types[c] == SRJ_STRUCT) {
    for (int k = 0; k < nch[c]; ++k) kids[c].push_back(build_srj(pos, types, scales, nch, rows, at, base, kids));
    s.children     = kids[c].data();
    s.num_children = nch[c];
  }
  return s;
}

// the cudf::column_view of a filled srj_column tree (LIST: {offsets, child}; STRING: {offsets} over the chars)
cudf::column_view to_view(const srj_column& s)
{
  const auto n = static_cast<cudf::size_type>(s.size);
  std::vector<cudf::column_view> children;
  if (has_offsets(s.type_id)) children.emplace_back(cudf::data_type{cudf::type_id::INT32}, n + 1, s.offsets, nullptr, 0);
  for (int k = 0; k < s.num_children; ++k) children.push_back(to_view(s.children[k]));
  return cudf::column_view(cudf::data_type{static_cast<cudf::type_id>(s.type_id), s.scale}, n, s.data, s.null_mask, -1 /* UNKNOWN_NULL_COUNT */, 0,
                           children);
}
}  // namespace

extern "C" {

JNIEXPORT jlongArray JNICALL Java_com_nvidia_spark_rapids_jni_kudo_KudoGpuSerializer_splitAndSerializeToDevice(JNIEnv* env, jclass, jlong j_table_view,
                                                                                                              jintArray j_splits)
{
  if (!j_table_view) { throw_java(env, "java/lang/NullPointerException", "table is null"); return nullptr; }
  if (!j_splits) { throw_java(env, "java/lang/NullPointerException", "splits is null"); return nullptr; }
  cudf::jni::auto_set_device(env);
  auto const* tbl = reinterpret_cast<cudf::table_view const*>(j_table_view);
  auto stream     = cudf::get_default_stream();
  const int nc    = tbl->num_columns();
  const int64_t n = tbl->num_rows();
  std::vector<srj_column> cols(nc);
  for (int c = 0; c < nc; ++c) cols[c] = to_srj(tbl->column(c));
  // Java passes the INTERIOR split indices (cudf::split semantics, shuffle_split.hpp:110-118): the C ABI takes 0 ... n
  const int ns = env->GetArrayLength(j_splits);
  std::vector<int32_t> splits(ns + 2, 0);
  {
    jint* h = env->GetIntArrayElements(j_splits, nullptr);
    for (int i = 0; i < ns; ++i) splits[i + 1] = h[i];
    env->ReleaseIntArrayElements(j_splits, h, JNI_ABORT);
  }
  splits[ns + 1] = static_cast<int32_t>(n);
  const int P    = ns + 1;
  rmm::device_buffer d_splits(splits.size() * 4, stream);
  if (!copy_from_host(d_splits.data(), splits.data(), splits.size() * 4, stream)) { throw_java(env, "ai/rapids/cudf/CudaException", "copy of the splits failed"); return nullptr; }
  rmm::device_buffer ws(static_cast<size_t>(srj_kudo_workspace_bytes(nc, P)), stream);
  auto offsets  = std::make_unique<rmm::device_buffer>(static_cast<size_t>(P + 1) * sizeof(size_t), stream);
  int64_t total = 0;
  if (throw_if_error(env, srj_kudo_split_sizes(cols.data(), nc, n, static_cast<int32_t*>(d_splits.data()), P, static_cast<int64_t*>(offsets->data()), &total,
                                               ws.data(), stream.value())))
    return nullptr;
  auto partitions = std::make_unique<rmm::device_buffer>(static_cast<size_t>(total), stream);
  if (throw_if_error(env, srj_kudo_split(cols.data(), nc, n, static_cast<int32_t*>(d_splits.data()), P, static_cast<int64_t*>(offsets->data()),
                                         static_cast<uint8_t*>(partitions->data()), ws.data(), stream.value())))
    return nullptr;
  stream.synchronize();   // ws / d_splits are released on return
  jlong r[6];
  r[0] = reinterpret_cast<jlong>(partitions->data());
  r[1] = static_cast<jlong>(partitions->size());
  r[2] = reinterpret_cast<jlong>(partitions.release());
  r[3] = reinterpret_cast<jlong>(offsets->data());
  r[4] = static_cast<jlong>(offsets->size());
  r[5] = reinterpret_cast<jlong>(offsets.release());
  jlongArray out = env->NewLongArray(6);
  if (out) env->SetLongArrayRegion(out, 0, 6, r);
  return out;
}

JNIEXPORT jobject JNICALL Java_com_nvidia_spark_rapids_jni_kudo_KudoGpuSerializer_assembleFromDeviceRawNative(JNIEnv* env, jclass, jlong part_addr, jlong part_len,
                                                                                                             jlong offset_addr, jlong offset_len,
                                                                                                             jintArray flat_num_children, jintArray flat_type_ids,
                                                                                                             jintArray flat_scale)
{
  if (!part_addr || !offset_addr || !flat_num_children || !flat_type_ids || !flat_scale) { throw_java(env, "java/lang/NullPointerException", "null argument"); return nullptr; }
  cudf::jni::auto_set_device(env);
  (void)part_len;
  auto stream  = cudf::get_default_stream();
  const int nc = env->GetArrayLength(flat_type_ids);
  std::vector<int32_t> types(nc), scales(nc), nch(nc);
  {
    jint* t  = env->GetIntArrayElements(flat_type_ids, nullptr);
    jint* sc = env->GetIntArrayElements(flat_scale, nullptr);
    jint* ch = env->GetIntArrayElements(flat_num_children, nullptr);
    for (int c = 0; c < nc; ++c) { types[c] = t[c]; scales[c] = sc[c]; nch[c] = ch[c]; }
    env->ReleaseIntArrayElements(flat_type_ids, t, JNI_ABORT);
    env->ReleaseIntArrayElements(flat_scale, sc, JNI_ABORT);
    env->ReleaseIntArrayElements(flat_num_children, ch, JNI_ABORT);
  }
  const int P = static_cast<int>(offset_len / sizeof(size_t)) - 1;
  rmm::device_buffer ws(static_cast<size_t>(srj_kudo_nested_workspace_bytes(nc, P)), stream);
  std::vector<int64_t> rows(nc, 0), chars(nc, 0);
  // checks the flattened schema (a forest of nc columns, a LIST with one child) and every partition against it
  if (throw_if_error(env, srj_kudo_assemble_nested_sizes(reinterpret_cast<const uint8_t*>(part_addr), reinterpret_cast<const int64_t*>(offset_addr), P, types.data(),
                                                         nch.data(), nc, rows.data(), chars.data(), ws.data(), stream.value())))
    return nullptr;
  // one shared buffer, every column buffer 64-byte aligned inside it (shuffle_assemble's layout, shuffle_split.hpp:160-172)
  std::vector<Slot> at(nc);
  size_t total = 0;
  for (int c = 0; c < nc; ++c) {
    const auto n = static_cast<size_t>(rows[c]);
    at[c].mask = total;  total = align_up(total + (n + 31) / 32 * 4, kSplitAlign);
    if (has_offsets(types[c])) { at[c].offsets = total; total = align_up(total + (n + 1) * 4, kSplitAlign); }
    at[c].data = total;
    if (types[c] != SRJ_LIST && types[c] != SRJ_STRUCT)
      total = align_up(total + (types[c] == SRJ_STRING ? static_cast<size_t>(chars[c]) : n * size_of_type(types[c])), kSplitAlign);
  }
  auto shared = std::make_unique<rmm::device_buffer>(total, stream);
  auto* base  = static_cast<uint8_t*>(shared->data());
  std::vector<std::vector<srj_column>> kids(nc);
  std::vector<srj_column> out;
  for (int pos = 0; pos < nc;) out.push_back(build_srj(pos, types, scales, nch, rows, at, base, kids));
  const int nroots = static_cast<int>(out.size());
  if (throw_if_error(env, srj_kudo_assemble_nested(reinterpret_cast<const uint8_t*>(part_addr), reinterpret_cast<const int64_t*>(offset_addr), P, out.data(), nroots,
                                                   ws.data(), stream.value())))
    return nullptr;
  stream.synchronize();
  std::vector<jlong> handles(nroots);
  for (int c = 0; c < nroots; ++c) handles[c] = reinterpret_cast<jlong>(new cudf::column_view(to_view(out[c])));
  const jlong buffer_size   = static_cast<jlong>(shared->size());
  const jlong buffer_handle = release_as_jlong(std::move(shared));
  jlongArray jhandles       = env->NewLongArray(nroots);
  if (jhandles) env->SetLongArrayRegion(jhandles, 0, nroots, handles.data());
  jclass cls    = env->FindClass("com/nvidia/spark/rapids/jni/kudo/KudoGpuSerializer$AssembleResult");
  jmethodID ctr = env->GetMethodID(cls, "<init>", "(JJ[J)V");
  return env->NewObject(cls, ctr, buffer_handle, buffer_size, jhandles);
}

}  // extern "C"
