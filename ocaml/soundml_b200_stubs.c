/* soundml_b200_stubs.c — OCaml foreign stubs over libsoundml_b200.so.
 *
 * NOT LINKED HERE: the build container has no OCaml toolchain (ocaml, dune, opam all
 * absent).  What is verified: the file compiles as C against stand-ins for
 * the caml headers (tests/test_ocaml_layer.py: gcc -fsyntax-only -Wall -Werror with
 * oracle/caml_shim), and every smb_* call matches include/soundml_b200.h.  It follows
 * the conventions of the reference's own stubs:
 *   - Bigarray storage is shared, never copied      (resample.ml:94, resample_stubs.c:220-226)
 *   - every pointer is extracted before the runtime lock is released and no
 *     OCaml value is touched until it is re-acquired (resample_stubs.c:284-295)
 *   - raises happen only while the lock is held     (resample_stubs.c:49-52)
 *   - externals with more than five arguments get a bytecode twin
 *                                                    (resample_stubs.c:410-422)
 *   - handles are custom blocks whose finalizer is the GC backstop for an
 *     explicit destroy                               (soundml_io_stubs.c:202-229)
 * Precondition failures (SMB_EINVAL) become Invalid_argument with the
 * reference's wording; CUDA/runtime failures become Failure.
 */
#include <stdint.h>
#include <string.h>

#include <caml/alloc.h>
#include <caml/bigarray.h>
#include <caml/custom.h>
#include <caml/fail.h>
#include <caml/memory.h>
#include <caml/mlvalues.h>
#include <caml/threads.h>

#include "soundml_b200.h"

static void smb_ml_raise(int status) {
  if (status == SMB_OK) return;
  if (status == SMB_EINVAL) caml_invalid_argument(smb_last_error());
  if (status == SMB_ENOMEM) caml_raise_out_of_memory();
  caml_failwith(smb_last_error());
}

/* ---- handles ------------------------------------------------------------- */
#define HANDLE(v) (*((void **)Data_custom_val(v)))

static void stft_finalize(value v) { if (HANDLE(v)) { smb_stft_plan_destroy(HANDLE(v)); HANDLE(v) = NULL; } }
static void mel_finalize(value v) { if (HANDLE(v)) { smb_mel_plan_destroy(HANDLE(v)); HANDLE(v) = NULL; } }
static void rs_finalize(value v) { if (HANDLE(v)) { smb_resample_plan_destroy(HANDLE(v)); HANDLE(v) = NULL; } }

static struct custom_operations stft_ops = {"soundml_b200.stft", stft_finalize,
  custom_compare_default, custom_hash_default, custom_serialize_default,
  custom_deserialize_default, custom_compare_ext_default, custom_fixed_length_default};
static struct custom_operations mel_ops = {"soundml_b200.mel", mel_finalize,
  custom_compare_default, custom_hash_default, custom_serialize_default,
  custom_deserialize_default, custom_compare_ext_default, custom_fixed_length_default};
static struct custom_operations rs_ops = {"soundml_b200.resample", rs_finalize,
  custom_compare_default, custom_hash_default, custom_serialize_default,
  custom_deserialize_default, custom_compare_ext_default, custom_fixed_length_default};

static void rk_finalize(value v) { if (HANDLE(v)) { smb_resample_kernel_destroy(HANDLE(v)); HANDLE(v) = NULL; } }
static struct custom_operations rk_ops = {"soundml_b200.resample_kernel", rk_finalize,
  custom_compare_default, custom_hash_default, custom_serialize_default,
  custom_deserialize_default, custom_compare_ext_default, custom_fixed_length_default};

/* `mem`: bytes the handle keeps outside the OCaml heap (device tables, staging), so
 * that the GC's pacing sees them (caml_alloc_custom_mem, OCaml >= 4.08). */
static value wrap(struct custom_operations *ops, void *h, uintnat mem) {
  value v = caml_alloc_custom_mem(ops, sizeof(void *), mem);
  HANDLE(v) = h;
  return v;
}

/* Flat storage must hold `elems` elements (complex Bigarrays count complex elements).
 * Raised while the runtime lock is held, like the reference's geometry checks
 * (resample_stubs.c:253-276). */
static void need(value ba, int64_t elems, const char *what) {
  if ((int64_t)Caml_ba_array_val(ba)->dim[0] < elems) caml_failwith(what);
}
static void *live(value v_plan) {
  void *h = HANDLE(v_plan);
  if (!h) caml_invalid_argument("soundml_b200: the plan has been destroyed");
  return h;
}

/* Explicit release (the finalizer stays as the backstop): destroy : plan -> unit */
CAMLprim value soundml_b200_stft_destroy(value v) { stft_finalize(v); return Val_unit; }
CAMLprim value soundml_b200_mel_destroy(value v) { mel_finalize(v); return Val_unit; }
CAMLprim value soundml_b200_resample_destroy(value v) { rs_finalize(v); return Val_unit; }
CAMLprim value soundml_b200_resample_kernel_destroy(value v) { rk_finalize(v); return Val_unit; }

static int dtype_of(value ba) {
  int kind = Caml_ba_array_val(ba)->flags & CAML_BA_KIND_MASK;
  if (kind == CAML_BA_FLOAT32 || kind == CAML_BA_COMPLEX32) return SMB_F32;
  if (kind == CAML_BA_FLOAT64 || kind == CAML_BA_COMPLEX64) return SMB_F64;
  caml_invalid_argument("soundml_b200: unsupported dtype (float32 and float64 are carried)");
}

/* ---- Stft ------------------------------------------------------------------
 * The OCaml Stft.Config.t already holds the float64 analysis window
 * (stft.ml:57-59), so the plan is created from it.
 * soundml_b200_stft_create : fft_size -> hop -> alignment -> pad_kind -> pad_value
 *                            -> (float, float64_elt, c_layout) Array1.t -> stft_plan */
CAMLprim value soundml_b200_stft_create(value v_fft, value v_hop, value v_align, value v_pad,
                                        value v_pad_value, value v_window) {
  CAMLparam1(v_window);
  smb_stft_plan *h = NULL;
  need(v_window, Long_val(v_fft), "soundml_b200: the analysis window is shorter than fft_size");
  int st = smb_stft_plan_create_with_window(&h, Long_val(v_fft), Long_val(v_hop),
                                            Int_val(v_align), Int_val(v_pad),
                                            Double_val(v_pad_value),
                                            (const double *)Caml_ba_data_val(v_window));
  smb_ml_raise(st);
  /* window, twiddles and fast-path tables on the device, plus host-call staging */
  CAMLreturn(wrap(&stft_ops, h, (uintnat)Long_val(v_fft) * 64 + (1u << 20)));
}
CAMLprim value soundml_b200_stft_create_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_stft_create(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* Stft.analyse replacement (stft.ml:356-364 + 670-674):
 * soundml_b200_power_spectrum : stft_plan -> x:ba -> batch -> n -> power -> out:ba -> unit
 * x and out are the flat storage of caller-allocated Nx tensors (host memory). */
CAMLprim value soundml_b200_power_spectrum(value v_plan, value v_x, value v_batch, value v_n,
                                           value v_power, value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const double power = Double_val(v_power);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_stft_bins(h) * smb_stft_frames(h, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_stft_power_spectrum(h, x, batch, n, dtype, power, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_power_spectrum_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_power_spectrum(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* Stft.transform: out is a complex Bigarray (complex32 for float32 audio). */
CAMLprim value soundml_b200_transform(value v_plan, value v_x, value v_batch, value v_n,
                                      value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_stft_bins(h) * smb_stft_frames(h, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_stft_transform(h, x, batch, n, dtype, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}

/* ---- Mel ------------------------------------------------------------------- */
CAMLprim value soundml_b200_mel_create(value v_n_mels, value v_fft, value v_weights) {
  CAMLparam1(v_weights);
  smb_mel_plan *h = NULL;
  need(v_weights, Long_val(v_n_mels) * (Long_val(v_fft) / 2 + 1),
       "soundml_b200: the weight matrix is smaller than n_mels x bins");
  int st = smb_mel_plan_create_with_weights(&h, Long_val(v_n_mels), Long_val(v_fft),
                                            (const double *)Caml_ba_data_val(v_weights));
  smb_ml_raise(st);
  CAMLreturn(wrap(&mel_ops, h, (uintnat)Long_val(v_n_mels) * (Long_val(v_fft) / 2 + 1) * 8 + (1u << 16)));
}

/* Mel.apply (mel.ml:202-231): s [batch; bins; frames] -> out [batch; n_mels; frames] */
CAMLprim value soundml_b200_mel_apply(value v_plan, value v_s, value v_batch, value v_frames,
                                      value v_out) {
  CAMLparam3(v_plan, v_s, v_out);
  smb_mel_plan *h = live(v_plan);
  const void *s = Caml_ba_data_val(v_s);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_s);
  const int64_t batch = Long_val(v_batch), frames = Long_val(v_frames);
  need(v_s, batch * smb_mel_bins(h) * frames, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_mel_n_mels(h) * frames, "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_mel_apply(h, s, batch, frames, dtype, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}

/* Soundml.mel_spectrogram (soundml.ml:22-24), fused. */
CAMLprim value soundml_b200_mel_spectrogram(value v_stft, value v_mel, value v_x, value v_batch,
                                            value v_n, value v_power, value v_out) {
  CAMLparam5(v_stft, v_mel, v_x, v_out, v_power);
  smb_stft_plan *hs = live(v_stft);
  smb_mel_plan *hm = live(v_mel);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const double power = Double_val(v_power);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_mel_n_mels(hm) * smb_stft_frames(hs, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_mel_spectrogram(hs, hm, x, batch, n, dtype, power, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_mel_spectrogram_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_mel_spectrogram(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5],
                                      argv[6]);
}

/* ---- Resample ---------------------------------------------------------------
 * quality: 0 fast, 1 high, 2 best, 3 custom (attenuation, passband). */
CAMLprim value soundml_b200_resample_create(value v_sr, value v_target, value v_quality,
                                            value v_att, value v_passband) {
  CAMLparam0();
  smb_resample_plan *h = NULL;
  int st = smb_resample_plan_create(&h, Long_val(v_sr), Long_val(v_target), Int_val(v_quality),
                                    Double_val(v_att), Double_val(v_passband));
  smb_ml_raise(st);
  CAMLreturn(wrap(&rs_ops, h, 4u << 20));      /* banks, plan spectra, tensor-core images */
}

/* Resample.apply (resample.ml:1913-1936): x [batch; n] -> out [batch; ceil(n L / M)] */
CAMLprim value soundml_b200_resample_apply(value v_plan, value v_x, value v_batch, value v_n,
                                           value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_resample_plan *h = live(v_plan);
  const float *x = (const float *)Caml_ba_data_val(v_x);
  float *out = (float *)Caml_ba_data_val(v_out);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  if ((Caml_ba_array_val(v_x)->flags & CAML_BA_KIND_MASK) != CAML_BA_FLOAT32)
    caml_invalid_argument("apply: this entry carries float32 audio (float64 has its own)");
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_resample_output_frames(h, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_resample_apply(h, x, batch, n, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}

/* Resample.apply for float64 audio (resample.ml:72-84 carries both widths). */
CAMLprim value soundml_b200_resample_apply_f64(value v_plan, value v_x, value v_batch, value v_n,
                                               value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_resample_plan *h = live(v_plan);
  const double *x = (const double *)Caml_ba_data_val(v_x);
  double *out = (double *)Caml_ba_data_val(v_out);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * smb_resample_output_frames(h, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_resample_apply_f64(h, x, batch, n, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}

/* ---- entry points added after the first slice ------------------------------- */

/* Stft.transform_range ~p0 ~p1 (stft.ml:652-666): out [batch; bins; p1 - p0]. */
CAMLprim value soundml_b200_transform_range(value v_plan, value v_x, value v_batch, value v_n,
                                            value v_p0, value v_p1, value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const int64_t p0 = Long_val(v_p0), p1 = Long_val(v_p1);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  if (p1 >= p0) need(v_out, batch * smb_stft_bins(h) * (p1 - p0),
                     "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_stft_transform_range(h, x, batch, n, dtype, p0, p1, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_transform_range_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_transform_range(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5],
                                      argv[6]);
}

/* Stft.invert dtype c ?length z (stft.ml:693-939): z [batch; bins; frames] complex ->
 * out [batch; length].  length < 0 stands for None (the natural length). */
CAMLprim value soundml_b200_invert(value v_plan, value v_z, value v_batch, value v_frames,
                                   value v_length, value v_out) {
  CAMLparam3(v_plan, v_z, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *z = Caml_ba_data_val(v_z);
  void *out = Caml_ba_data_val(v_out);
  const int in_dtype = dtype_of(v_z), out_dtype = dtype_of(v_out);
  const int64_t batch = Long_val(v_batch), frames = Long_val(v_frames);
  const int64_t length = Long_val(v_length);
  need(v_z, batch * smb_stft_bins(h) * frames, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * (length >= 0 ? length : smb_stft_output_length(h, frames)),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_stft_invert(h, z, batch, frames, in_dtype, length >= 0, length >= 0 ? length : 0,
                           out_dtype, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_invert_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_invert(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* ---- Effects (effects.ml; librosa 0.11 phase_vocoder / time_stretch) ----------
 * phase_vocoder: z [batch; bins; frames] complex -> out [batch; bins; T'] of the same
 * kind, T' = time_stretch_frames plan frames rate.  A bad rate is Invalid_argument with
 * the reference's wording, raised by the library before any extent is trusted. */
CAMLprim value soundml_b200_phase_vocoder(value v_plan, value v_z, value v_batch, value v_frames,
                                          value v_rate, value v_out) {
  CAMLparam3(v_plan, v_z, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *z = Caml_ba_data_val(v_z);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_z);
  const int64_t batch = Long_val(v_batch), frames = Long_val(v_frames);
  const double rate = Double_val(v_rate);
  const int64_t out_frames = smb_time_stretch_frames(h, frames, rate);
  if (out_frames >= 0) {
    need(v_z, batch * smb_stft_bins(h) * frames, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * smb_stft_bins(h) * out_frames,
         "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_phase_vocoder(h, z, batch, frames, dtype, rate, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_phase_vocoder_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_phase_vocoder(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* time_stretch: x [batch; n] real -> out [batch; time_stretch_length n rate], same kind. */
CAMLprim value soundml_b200_time_stretch(value v_plan, value v_x, value v_batch, value v_n,
                                         value v_rate, value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const double rate = Double_val(v_rate);
  const int64_t length = smb_time_stretch_length(n, rate);
  if (length >= 0) {
    need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * length, "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_time_stretch(h, x, batch, n, dtype, rate, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_time_stretch_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_time_stretch(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* Output sizes, Invalid_argument on a bad rate or a negative count. */
CAMLprim value soundml_b200_time_stretch_frames(value v_plan, value v_frames, value v_rate) {
  const int64_t r = smb_time_stretch_frames(live(v_plan), Long_val(v_frames), Double_val(v_rate));
  if (r < 0) smb_ml_raise(SMB_EINVAL);
  return Val_long(r);
}
CAMLprim value soundml_b200_time_stretch_length(value v_n, value v_rate) {
  const int64_t r = smb_time_stretch_length(Long_val(v_n), Double_val(v_rate));
  if (r < 0) smb_ml_raise(SMB_EINVAL);
  return Val_long(r);
}

/* ---- Hpss (librosa 0.11 decompose.hpss / effects.hpss; the reference's hpss.ml) ----
 * Outputs per item: 2 for SMB_HPSS_BOTH and SMB_HPSS_MASKS, 1 for one part; an unknown
 * `what` is left to the library, which names it after the parameters' errors. */
static int64_t hpss_parts(int what) {
  return what == SMB_HPSS_BOTH || what == SMB_HPSS_MASKS ? 2 : 1;
}

/* hpss: s [batch; bins; frames] real or complex -> out [batch; parts; bins; frames], of
 * s's kind, or real masks for SMB_HPSS_MASKS. */
CAMLprim value soundml_b200_hpss(value v_s, value v_batch, value v_bins, value v_frames,
                                 value v_win_harm, value v_win_perc, value v_power,
                                 value v_margin_harm, value v_margin_perc, value v_what, value v_out) {
  CAMLparam2(v_s, v_out);
  const void *s = Caml_ba_data_val(v_s);
  void *out = Caml_ba_data_val(v_out);
  const int kind = Caml_ba_array_val(v_s)->flags & CAML_BA_KIND_MASK;
  const int complex_in = kind == CAML_BA_COMPLEX32 || kind == CAML_BA_COMPLEX64;
  const int dtype = dtype_of(v_s);
  const int64_t batch = Long_val(v_batch), bins = Long_val(v_bins), frames = Long_val(v_frames);
  const int what = Int_val(v_what);
  if (batch >= 0 && bins >= 0 && frames >= 0) {
    need(v_s, batch * bins * frames, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * hpss_parts(what) * bins * frames,
         "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_hpss(s, batch, bins, frames, dtype, complex_in, Long_val(v_win_harm), Long_val(v_win_perc),
                    Double_val(v_power), Double_val(v_margin_harm), Double_val(v_margin_perc), what, out,
                    SMB_MEM_HOST, SMB_STREAM_OWN);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_hpss_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_hpss(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6], argv[7],
                           argv[8], argv[9], argv[10]);
}

/* hpss_audio: x [batch; n] real -> out [batch; parts; n], same kind. */
CAMLprim value soundml_b200_hpss_audio(value v_plan, value v_x, value v_batch, value v_n,
                                       value v_win_harm, value v_win_perc, value v_power,
                                       value v_margin_harm, value v_margin_perc, value v_what,
                                       value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const int what = Int_val(v_what);
  if (batch >= 0 && n >= 0) {
    need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * hpss_parts(what) * n, "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_hpss_audio(h, x, batch, n, dtype, Long_val(v_win_harm), Long_val(v_win_perc),
                          Double_val(v_power), Double_val(v_margin_harm), Double_val(v_margin_perc),
                          what, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_hpss_audio_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_hpss_audio(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6],
                                 argv[7], argv[8], argv[9], argv[10]);
}

/* ---- Spectral (librosa 0.11 feature.spectral_*; the reference's spectral.ml) ----
 * Rows per item: one per bit of `what`; unknown bits are left to the library, which names
 * them first. */
static int64_t spectral_rows(int what) {
  return __builtin_popcount((unsigned)what & 15u);
}

/* spectral: s [batch; bins; frames] real -> out [batch; rows; frames], same kind. */
CAMLprim value soundml_b200_spectral(value v_s, value v_batch, value v_bins, value v_frames, value v_n_fft,
                                     value v_sample_rate, value v_what, value v_p, value v_norm,
                                     value v_roll_percent, value v_amin, value v_power, value v_out) {
  CAMLparam2(v_s, v_out);
  const void *s = Caml_ba_data_val(v_s);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_s);
  const int64_t batch = Long_val(v_batch), bins = Long_val(v_bins), frames = Long_val(v_frames);
  const int what = Int_val(v_what);
  if (batch >= 0 && bins >= 0 && frames >= 0) {
    need(v_s, batch * bins * frames, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * spectral_rows(what) * frames, "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_spectral(s, batch, bins, frames, dtype, Long_val(v_n_fft), Double_val(v_sample_rate), what,
                        Double_val(v_p), Bool_val(v_norm), Double_val(v_roll_percent), Double_val(v_amin),
                        Double_val(v_power), out, SMB_MEM_HOST, SMB_STREAM_OWN);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_spectral_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_spectral(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6], argv[7],
                               argv[8], argv[9], argv[10], argv[11], argv[12]);
}

/* spectral_audio: x [batch; n] real -> out [batch; rows; frames], same kind. */
CAMLprim value soundml_b200_spectral_audio(value v_plan, value v_x, value v_batch, value v_n,
                                           value v_sample_rate, value v_what, value v_p, value v_norm,
                                           value v_roll_percent, value v_amin, value v_power, value v_out) {
  CAMLparam3(v_plan, v_x, v_out);
  smb_stft_plan *h = live(v_plan);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n);
  const int what = Int_val(v_what);
  if (batch >= 0 && n >= 0) {
    need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
    need(v_out, batch * spectral_rows(what) * smb_stft_frames(h, n),
         "soundml_b200: output extent disagrees with geometry");
  }
  caml_release_runtime_system();
  int st = smb_spectral_audio(h, x, batch, n, dtype, Double_val(v_sample_rate), what, Double_val(v_p),
                              Bool_val(v_norm), Double_val(v_roll_percent), Double_val(v_amin),
                              Double_val(v_power), out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_spectral_audio_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_spectral_audio(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6], argv[7],
                                     argv[8], argv[9], argv[10], argv[11]);
}

/* Convert.power_to_db / amplitude_to_db (convert.ml:20-56).  top_db = nan stands
 * for None; amplitude selects the 20 log10 form. */
CAMLprim value soundml_b200_to_db(value v_amplitude, value v_x, value v_reference, value v_amin,
                                  value v_top_db, value v_out) {
  CAMLparam2(v_x, v_out);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t count = Caml_ba_array_val(v_x)->dim[0];
  const double reference = Double_val(v_reference), amin = Double_val(v_amin);
  const double top_db = Double_val(v_top_db);
  const int amplitude = Bool_val(v_amplitude);
  need(v_out, count, "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = amplitude
      ? smb_amplitude_to_db(x, count, dtype, reference, amin, top_db, out, SMB_MEM_HOST, SMB_STREAM_OWN)
      : smb_power_to_db(x, count, dtype, reference, amin, top_db, out, SMB_MEM_HOST, SMB_STREAM_OWN);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_to_db_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_to_db(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}

/* Soundml.mfcc stft mel ?n_mfcc ?lifter x (soundml.ml:50-95): out [batch; n_mfcc; frames];
 * lifter = 0 stands for None. */
CAMLprim value soundml_b200_mfcc(value v_stft, value v_mel, value v_x, value v_batch, value v_n,
                                 value v_n_mfcc, value v_lifter, value v_out) {
  CAMLparam4(v_stft, v_mel, v_x, v_out);
  smb_stft_plan *hs = live(v_stft);
  smb_mel_plan *hm = live(v_mel);
  const void *x = Caml_ba_data_val(v_x);
  void *out = Caml_ba_data_val(v_out);
  const int dtype = dtype_of(v_x);
  const int64_t batch = Long_val(v_batch), n = Long_val(v_n), n_mfcc = Long_val(v_n_mfcc);
  const double lifter = Double_val(v_lifter);
  need(v_x, batch * n, "soundml_b200: input extent disagrees with geometry");
  need(v_out, batch * n_mfcc * smb_stft_frames(hs, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_mfcc(hs, hm, x, batch, n, dtype, n_mfcc, lifter, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_mfcc_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_mfcc(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6],
                           argv[7]);
}

/* soundml-io device ingest: the layout pass of stub_readf's staging block on the
 * device (soundml_io_stubs.c:832-872).  staging: the interleaved block libsndfile
 * just filled (host Bigarray, [frames * channels]); dst: the planar destination
 * (host Bigarray here; a device pointer when the caller keeps the signal on the
 * GPU for Resample.Kernel.step).  mode: 1 planar, 2 downmix, as SOUNDML_IO_MODE_*. */
CAMLprim value soundml_b200_ingest_layout(value v_staging, value v_frames, value v_channels,
                                          value v_mode, value v_dst, value v_total, value v_off) {
  CAMLparam2(v_staging, v_dst);
  const void *staging = Caml_ba_data_val(v_staging);
  void *dst = Caml_ba_data_val(v_dst);
  const int dtype = dtype_of(v_staging);
  const int64_t frames = Long_val(v_frames), channels = Long_val(v_channels);
  const int64_t total = Long_val(v_total), off = Long_val(v_off);
  const int mode = Int_val(v_mode);
  need(v_staging, frames * channels, "soundml_b200: staging extent disagrees with geometry");
  need(v_dst, (mode == 2 ? 1 : channels) * total,
       "soundml_b200: destination extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_ingest_layout(staging, frames, channels, mode, dtype, dst, total, off,
                             SMB_MEM_HOST, SMB_MEM_HOST, NULL);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_ingest_layout_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_ingest_layout(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5], argv[6]);
}

/* ---- Resample.Kernel (resample.ml:1343-1424, 1844-1909; soundml_io.ml:639, 768, 798) -----
 * prepare : resample_plan -> dtype:int (0 = float32, 1 = float64) -> channels -> max_block -> kernel */
CAMLprim value soundml_b200_resample_kernel_create(value v_plan, value v_dtype, value v_channels,
                                                   value v_max_block) {
  CAMLparam1(v_plan);
  smb_resample_kernel *k = NULL;
  int st = smb_resample_kernel_create(&k, live(v_plan), Int_val(v_dtype), Long_val(v_channels),
                                      Long_val(v_max_block));
  smb_ml_raise(st);
  /* the carry: two rows of (max_block + cone) samples per channel, plus the window and its image */
  CAMLreturn(wrap(&rk_ops, k, (uintnat)Long_val(v_channels) * (uintnat)Long_val(v_max_block) * 8 * 6));
}
/* frames the next step / the flush will emit: exact integers, asked before the call so
 * that OCaml allocates the result (the stub allocates nothing on the OCaml heap) */
CAMLprim value soundml_b200_resample_kernel_step_frames(value v_k, value v_n) {
  return Val_long(smb_resample_kernel_step_frames(live(v_k), Long_val(v_n)));
}
CAMLprim value soundml_b200_resample_kernel_flush_frames(value v_k) {
  return Val_long(smb_resample_kernel_flush_frames(live(v_k)));
}
/* step : kernel -> chunk:ba ([channels; n] flat) -> channels -> n -> out:ba ([channels; frames] flat) -> unit */
CAMLprim value soundml_b200_resample_kernel_step(value v_k, value v_chunk, value v_channels,
                                                 value v_n, value v_out) {
  CAMLparam3(v_k, v_chunk, v_out);
  smb_resample_kernel *k = live(v_k);
  const void *chunk = Caml_ba_data_val(v_chunk);
  void *out = Caml_ba_data_val(v_out);
  const int64_t channels = Long_val(v_channels), n = Long_val(v_n);
  need(v_chunk, channels * n, "soundml_b200: chunk extent disagrees with geometry");
  need(v_out, channels * smb_resample_kernel_step_frames(k, n),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_resample_kernel_step(k, chunk, n, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_resample_kernel_flush(value v_k, value v_channels, value v_out) {
  CAMLparam2(v_k, v_out);
  smb_resample_kernel *k = live(v_k);
  void *out = Caml_ba_data_val(v_out);
  need(v_out, Long_val(v_channels) * smb_resample_kernel_flush_frames(k),
       "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_resample_kernel_flush(k, out, SMB_MEM_HOST);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
CAMLprim value soundml_b200_resample_kernel_reset(value v_k) {
  smb_ml_raise(smb_resample_kernel_reset(live(v_k)));
  return Val_unit;
}

/* ---- the fused read's decode loop on the device (soundml_io.ml:742-807) ------------------
 * reader = two pinned staging blocks + the streaming resampler; the OCaml side decodes with
 * sf_readf_* straight into the Bigarray `ingest_staging` returns (it aliases the pinned
 * block: CAML_BA_EXTERNAL, nothing for the GC to free), submits, and collects the planar
 * result from a device buffer it owns (`ingest_result_*`). */
static void ing_finalize(value v) { if (HANDLE(v)) { smb_ingest_destroy(HANDLE(v)); HANDLE(v) = NULL; } }
static struct custom_operations ing_ops = {"soundml_b200.ingest", ing_finalize,
  custom_compare_default, custom_hash_default, custom_serialize_default,
  custom_deserialize_default, custom_compare_ext_default, custom_fixed_length_default};

/* channels -> sample_rate -> target (0 = native) -> mode -> quality -> max_block (0 = rule) -> reader
 * (float32 frames: what sf_readf_float delivers) */
CAMLprim value soundml_b200_ingest_create(value v_channels, value v_sr, value v_target, value v_mode,
                                          value v_quality, value v_max_block) {
  CAMLparam0();
  smb_ingest *r = NULL;
  smb_ml_raise(smb_ingest_create(&r, Long_val(v_channels), Long_val(v_sr), Long_val(v_target),
                                 Int_val(v_mode), Int_val(v_quality), Long_val(v_max_block), SMB_F32));
  const int64_t block = smb_ingest_max_block(r) * Long_val(v_channels) * 4;
  CAMLreturn(wrap(&ing_ops, r, (uintnat)(4 * block)));   /* two pinned blocks, two device copies */
}
CAMLprim value soundml_b200_ingest_create_bc(value *argv, int argn) {
  (void)argn;
  return soundml_b200_ingest_create(argv[0], argv[1], argv[2], argv[3], argv[4], argv[5]);
}
CAMLprim value soundml_b200_ingest_destroy(value v) { ing_finalize(v); return Val_unit; }
CAMLprim value soundml_b200_ingest_max_block(value v) { return Val_long(smb_ingest_max_block(live(v))); }
/* reader -> channels -> (float, float32_elt) Array1.t over the block to decode into next */
CAMLprim value soundml_b200_ingest_staging(value v_r, value v_channels) {
  CAMLparam1(v_r);
  smb_ingest *r = live(v_r);
  void *block = NULL;
  caml_release_runtime_system();               /* may wait for the upload of two submits ago */
  int st = smb_ingest_staging(r, &block);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  intnat dim[1] = {(intnat)(smb_ingest_max_block(r) * Long_val(v_channels))};
  CAMLreturn(caml_ba_alloc(CAML_BA_FLOAT32 | CAML_BA_C_LAYOUT | CAML_BA_EXTERNAL, 1, block, dim));
}
CAMLprim value soundml_b200_ingest_submit_frames(value v_r, value v_frames) {
  return Val_long(smb_ingest_submit_frames(live(v_r), Long_val(v_frames)));
}
CAMLprim value soundml_b200_ingest_finish_frames(value v_r) {
  return Val_long(smb_ingest_finish_frames(live(v_r)));
}
/* The planar result lives in a device buffer [width, total] the OCaml side allocates once
 * (it knows the file's frame count): a piece of `released` frames is written as
 * [width, released] C-contiguous at `at`; ingest_result_read strides them back into place. */
CAMLprim value soundml_b200_device_alloc(value v_bytes) {
  void *p = NULL;
  smb_ml_raise(smb_device_alloc(&p, (size_t)Long_val(v_bytes)));
  return caml_copy_nativeint((intnat)p);
}
CAMLprim value soundml_b200_device_free(value v_ptr) {
  smb_ml_raise(smb_device_free((void *)Nativeint_val(v_ptr)));
  return Val_unit;
}
/* reader -> frames -> device base -> byte offset -> unit (only enqueues) */
CAMLprim value soundml_b200_ingest_submit(value v_r, value v_frames, value v_dev, value v_off) {
  smb_ingest *r = live(v_r);
  smb_ml_raise(smb_ingest_submit(r, Long_val(v_frames), (char *)Nativeint_val(v_dev) + Long_val(v_off)));
  return Val_unit;
}
CAMLprim value soundml_b200_ingest_finish(value v_r, value v_dev, value v_off) {
  smb_ingest *r = live(v_r);
  smb_ml_raise(smb_ingest_finish(r, (char *)Nativeint_val(v_dev) + Long_val(v_off)));
  return Val_unit;
}
/* reader -> device base -> bytes -> dst:ba -> unit: waits for the reader, then one copy down */
CAMLprim value soundml_b200_ingest_result_read(value v_r, value v_dev, value v_bytes, value v_dst) {
  CAMLparam2(v_r, v_dst);
  smb_ingest *r = live(v_r);
  void *dst = Caml_ba_data_val(v_dst);
  const size_t bytes = (size_t)Long_val(v_bytes);
  need(v_dst, (int64_t)(bytes / 4), "soundml_b200: output extent disagrees with geometry");
  caml_release_runtime_system();
  int st = smb_ingest_sync(r);
  if (st == SMB_OK) st = smb_memcpy_d2h(dst, (const void *)Nativeint_val(v_dev), bytes);
  caml_acquire_runtime_system();
  smb_ml_raise(st);
  CAMLreturn(Val_unit);
}
