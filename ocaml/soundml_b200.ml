(* soundml_b200.ml — the OCaml side of the drop-in: externals over
   libsoundml_b200.so and the three functions of the reference that change.

   NOT COMPILED HERE (no OCaml toolchain in the build container); the C stubs it
   binds are syntax-checked against stand-in caml headers and every external below
   is checked to name a CAMLprim of soundml_b200_stubs.c with the right arity
   (tests/test_ocaml_layer.py).  The intent is a patch to soundml/lib that leaves every signature of stft.mli / mel.mli /
   resample.mli / soundml.mli untouched:

     Stft.power_spectrum   stft.ml:687-691   -> B200.power_spectrum
     Stft.transform        stft.ml:632-650   -> B200.transform
     Mel.apply             mel.ml:202-231    -> B200.mel_apply
     Soundml.mel_spectrogram soundml.ml:22-24 -> B200.mel_spectrogram (fused)
     Resample.apply        resample.ml:1913-1936 -> B200.resample_apply
     Stft.transform_range  stft.ml:652-666   -> B200.transform_range
     Stft.invert           stft.ml:937-939   -> B200.invert
     Effects.time_stretch  effects.ml:296    -> B200.time_stretch (and B200.phase_vocoder)
     hpss / effects.hpss   hpss.ml           -> B200.Hpss
     spectral.ml                             -> B200.Spectral
     Convert.power_to_db / amplitude_to_db  convert.ml:20-56 -> B200.to_db
     Soundml.mfcc          soundml.ml:50-95  -> B200.mfcc
     Resample.Kernel.prepare / step / flush / reset
                           resample.ml:1343-1424, 1844-1909 -> B200.Kernel

   Config.create stays in OCaml: the plan is built from the float64 window /
   weights the config already owns, so the two sides cannot disagree. *)

type stft_plan
type mel_plan
type resample_plan
type resample_kernel

type ('a, 'b) ba = ('a, 'b, Bigarray.c_layout) Bigarray.Array1.t

external stft_create :
  int -> int -> int -> int -> float -> (float, Bigarray.float64_elt) ba -> stft_plan
  = "soundml_b200_stft_create_bc" "soundml_b200_stft_create"

external power_spectrum_c :
  stft_plan -> (float, 'a) ba -> int -> int -> float -> (float, 'a) ba -> unit
  = "soundml_b200_power_spectrum_bc" "soundml_b200_power_spectrum"

external transform_c :
  stft_plan -> (float, 'a) ba -> int -> int -> (Complex.t, 'c) ba -> unit
  = "soundml_b200_transform"

external mel_create : int -> int -> (float, Bigarray.float64_elt) ba -> mel_plan
  = "soundml_b200_mel_create"

external mel_apply_c : mel_plan -> (float, 'a) ba -> int -> int -> (float, 'a) ba -> unit
  = "soundml_b200_mel_apply"

external mel_spectrogram_c :
  stft_plan -> mel_plan -> (float, 'a) ba -> int -> int -> float -> (float, 'a) ba -> unit
  = "soundml_b200_mel_spectrogram_bc" "soundml_b200_mel_spectrogram"

external resample_create : int -> int -> int -> float -> float -> resample_plan
  = "soundml_b200_resample_create"

external resample_apply_c :
  resample_plan -> (float, Bigarray.float32_elt) ba -> int -> int
  -> (float, Bigarray.float32_elt) ba -> unit
  = "soundml_b200_resample_apply"

external resample_apply_f64_c :
  resample_plan -> (float, Bigarray.float64_elt) ba -> int -> int
  -> (float, Bigarray.float64_elt) ba -> unit
  = "soundml_b200_resample_apply_f64"

external transform_range_c :
  stft_plan -> (float, 'a) ba -> int -> int -> int -> int -> (Complex.t, 'c) ba -> unit
  = "soundml_b200_transform_range_bc" "soundml_b200_transform_range"

(* length < 0 stands for None *)
external invert_c :
  stft_plan -> (Complex.t, 'c) ba -> int -> int -> int -> (float, 'a) ba -> unit
  = "soundml_b200_invert_bc" "soundml_b200_invert"

(* plan -> z -> batch -> frames -> rate -> out *)
external phase_vocoder_c :
  stft_plan -> (Complex.t, 'c) ba -> int -> int -> float -> (Complex.t, 'c) ba -> unit
  = "soundml_b200_phase_vocoder_bc" "soundml_b200_phase_vocoder"

(* plan -> x -> batch -> n -> rate -> out *)
external time_stretch_c :
  stft_plan -> (float, 'a) ba -> int -> int -> float -> (float, 'a) ba -> unit
  = "soundml_b200_time_stretch_bc" "soundml_b200_time_stretch"

external time_stretch_frames : stft_plan -> int -> float -> int
  = "soundml_b200_time_stretch_frames"

external time_stretch_length : int -> float -> int = "soundml_b200_time_stretch_length"

(* s -> batch -> bins -> frames -> win_harm -> win_perc -> power -> margin_harm
   -> margin_perc -> what -> out; s real or complex, out of s's kind or real masks *)
external hpss_c :
  ('a, 'b) ba -> int -> int -> int -> int -> int -> float -> float -> float -> int
  -> ('c, 'd) ba -> unit
  = "soundml_b200_hpss_bc" "soundml_b200_hpss"

(* plan -> x -> batch -> n -> win_harm -> win_perc -> power -> margin_harm -> margin_perc
   -> what -> out *)
external hpss_audio_c :
  stft_plan -> (float, 'a) ba -> int -> int -> int -> int -> float -> float -> float -> int
  -> (float, 'a) ba -> unit
  = "soundml_b200_hpss_audio_bc" "soundml_b200_hpss_audio"

(* s -> batch -> bins -> frames -> n_fft -> sample_rate -> what -> p -> norm -> roll_percent
   -> amin -> power -> out; out [batch; popcount what; frames] of s's kind *)
external spectral_c :
  (float, 'a) ba -> int -> int -> int -> int -> float -> int -> float -> bool -> float -> float
  -> float -> (float, 'a) ba -> unit
  = "soundml_b200_spectral_bc" "soundml_b200_spectral"

(* plan -> x -> batch -> n -> sample_rate -> what -> p -> norm -> roll_percent -> amin
   -> power -> out *)
external spectral_audio_c :
  stft_plan -> (float, 'a) ba -> int -> int -> float -> int -> float -> bool -> float -> float
  -> float -> (float, 'a) ba -> unit
  = "soundml_b200_spectral_audio_bc" "soundml_b200_spectral_audio"

(* amplitude -> x -> reference -> amin -> top_db (nan = None) -> out *)
external to_db_c :
  bool -> (float, 'a) ba -> float -> float -> float -> (float, 'a) ba -> unit
  = "soundml_b200_to_db_bc" "soundml_b200_to_db"

(* lifter = 0. stands for None *)
external mfcc_c :
  stft_plan -> mel_plan -> (float, 'a) ba -> int -> int -> int -> float -> (float, 'a) ba
  -> unit
  = "soundml_b200_mfcc_bc" "soundml_b200_mfcc"

(* soundml-io: the layout pass after stub_readf (soundml_io_stubs.c:832-872) on the
   device; mode 1 = planar, 2 = downmix. *)
external ingest_layout_c :
  (float, 'a) ba -> int -> int -> int -> (float, 'a) ba -> int -> int -> unit
  = "soundml_b200_ingest_layout_bc" "soundml_b200_ingest_layout"

external stft_destroy : stft_plan -> unit = "soundml_b200_stft_destroy"
external mel_destroy : mel_plan -> unit = "soundml_b200_mel_destroy"
external resample_destroy : resample_plan -> unit = "soundml_b200_resample_destroy"

(* dtype: 0 = float32, 1 = float64 *)
external resample_kernel_create : resample_plan -> int -> int -> int -> resample_kernel
  = "soundml_b200_resample_kernel_create"
external resample_kernel_step_frames : resample_kernel -> int -> int
  = "soundml_b200_resample_kernel_step_frames"
external resample_kernel_flush_frames : resample_kernel -> int
  = "soundml_b200_resample_kernel_flush_frames"
external resample_kernel_step_c :
  resample_kernel -> (float, 'a) ba -> int -> int -> (float, 'a) ba -> unit
  = "soundml_b200_resample_kernel_step"
external resample_kernel_flush_c : resample_kernel -> int -> (float, 'a) ba -> unit
  = "soundml_b200_resample_kernel_flush"
external resample_kernel_reset : resample_kernel -> unit = "soundml_b200_resample_kernel_reset"
external resample_kernel_destroy : resample_kernel -> unit
  = "soundml_b200_resample_kernel_destroy"

(* The flat storage of a contiguous tensor, shared (resample.ml:94). *)
type ingest

external ingest_create : int -> int -> int -> int -> int -> int -> ingest
  = "soundml_b200_ingest_create_bc" "soundml_b200_ingest_create"
external ingest_destroy : ingest -> unit = "soundml_b200_ingest_destroy"
external ingest_max_block : ingest -> int = "soundml_b200_ingest_max_block"
external ingest_staging : ingest -> int -> (float, Bigarray.float32_elt) ba
  = "soundml_b200_ingest_staging"
external ingest_submit_frames : ingest -> int -> int = "soundml_b200_ingest_submit_frames"
external ingest_finish_frames : ingest -> int = "soundml_b200_ingest_finish_frames"
external device_alloc : int -> nativeint = "soundml_b200_device_alloc"
external device_free : nativeint -> unit = "soundml_b200_device_free"
external ingest_submit : ingest -> int -> nativeint -> int -> unit = "soundml_b200_ingest_submit"
external ingest_finish : ingest -> nativeint -> int -> unit = "soundml_b200_ingest_finish"
external ingest_result_read : ingest -> nativeint -> int -> (float, Bigarray.float32_elt) ba -> unit
  = "soundml_b200_ingest_result_read"

let array1_of t = Nx_buffer.to_bigarray1 (Nx.to_buffer t)

let leading_shape t =
  let shape = Nx.shape t in
  Array.sub shape 0 (Array.length shape - 1)

let alignment_code = function `Centered -> 0 | `Left -> 1 | `Right -> 2

let pad_code = function `Reflect -> (0, 0.) | `Constant v -> (1, v) | `Edge -> (2, 0.)

(* One plan per configuration, created on first use and kept: Config.t values are
   immutable, so physical identity keys the cache (an ephemeron table: the plan goes
   when its configuration does; [release_plans] frees the device memory at once
   instead of waiting for the finalizers).  Like the reference's lazies
   (resample.ml:427, 492) the caches are not domain-safe. *)
module Cache (K : sig type t end) = struct
  module T = Ephemeron.K1.Make (struct
    type t = K.t
    let equal = ( == )
    let hash = Hashtbl.hash
  end)
  let make () : 'plan T.t = T.create 8
end

module Stft_cache = Cache (struct type t = Stft.Config.t end)
module Mel_cache = Cache (struct type t = Mel.Config.t end)

let stft_plans : stft_plan Stft_cache.T.t = Stft_cache.make ()
let mel_plans : mel_plan Mel_cache.T.t = Mel_cache.make ()
let resample_plans : (int * int * int * float * float, resample_plan) Hashtbl.t = Hashtbl.create 8

let stft_plan_of (c : Stft.Config.t) =
  match Stft_cache.T.find_opt stft_plans c with
  | Some p -> p
  | None ->
      let pad, pad_value = pad_code (Stft.Config.pad c) in
      let p =
        stft_create (Stft.Config.fft_size c) (Stft.Config.hop c)
          (alignment_code (Stft.Config.alignment c))
          pad pad_value
          (array1_of (Stft.Config.analysis_window c))
      in
      Stft_cache.T.replace stft_plans c p ;
      p

let mel_plan_of (c : Mel.Config.t) =
  match Mel_cache.T.find_opt mel_plans c with
  | Some p -> p
  | None ->
      let p =
        mel_create (Mel.Config.n_mels c) (Mel.Config.fft_size c)
          (array1_of (Mel.filterbank Nx.float64 c))
      in
      Mel_cache.T.replace mel_plans c p ;
      p

let quality_code = function
  | `Fast -> (0, 0., 0.)
  | `High -> (1, 0., 0.)
  | `Best -> (2, 0., 0.)
  | `Custom (att, pb) -> (3, att, pb)

let resample_plan_of ~sample_rate ~target ~quality =
  let q, att, pb = quality_code quality in
  let key = (sample_rate, target, q, att, pb) in
  match Hashtbl.find_opt resample_plans key with
  | Some p -> p
  | None ->
      let p = resample_create sample_rate target q att pb in
      Hashtbl.replace resample_plans key p ;
      p

(* Free every cached plan's device memory now. *)
let release_plans () =
  Stft_cache.T.iter (fun _ p -> stft_destroy p) stft_plans ;
  Stft_cache.T.reset stft_plans ;
  Mel_cache.T.iter (fun _ p -> mel_destroy p) mel_plans ;
  Mel_cache.T.reset mel_plans ;
  Hashtbl.iter (fun _ p -> resample_destroy p) resample_plans ;
  Hashtbl.reset resample_plans

(* Replacement body of Stft.power_spectrum: same checks, same result shape
   [...; bins; frames]; the arithmetic is the fused B200 kernel. *)
let power_spectrum ?(power = 2.) c x =
  let n = Nx.dim (Nx.ndim x - 1) x in
  let lead = leading_shape x in
  let batch = Array.fold_left ( * ) 1 lead in
  let frames = Stft.frames c ~n in
  let out = Nx.zeros (Nx.dtype x) (Array.append lead [|Stft.Config.bins c; frames|]) in
  if batch > 0 && frames > 0 then
    power_spectrum_c (stft_plan_of c) (array1_of (Nx.contiguous x)) batch n power
      (array1_of out) ;
  out

let mel_spectrogram stft_config mel_config ?(power = 2.) x =
  let n = Nx.dim (Nx.ndim x - 1) x in
  let lead = leading_shape x in
  let batch = Array.fold_left ( * ) 1 lead in
  let frames = Stft.frames stft_config ~n in
  let n_mels = Mel.Config.n_mels mel_config in
  let out = Nx.zeros (Nx.dtype x) (Array.append lead [|n_mels; frames|]) in
  if batch > 0 && frames > 0 then
    mel_spectrogram_c (stft_plan_of stft_config) (mel_plan_of mel_config)
      (array1_of (Nx.contiguous x))
      batch n power (array1_of out) ;
  out

(* Replacement body of Resample.apply: the result has the dtype of [x], float32 or
   float64 (resample.ml:72-84 carries both widths). *)
let resample_apply (type a b) ~sample_rate ~target ~quality (x : (a, b) Nx.t) : (a, b) Nx.t =
  let plan = resample_plan_of ~sample_rate ~target ~quality in
  let n = Nx.dim (Nx.ndim x - 1) x in
  let lead = leading_shape x in
  let batch = Array.fold_left ( * ) 1 lead in
  let g = let rec gcd a b = if b = 0 then a else gcd b (a mod b) in gcd sample_rate target in
  let l = target / g and m = sample_rate / g in
  let total = if n <= 0 then 0 else (((n * l) - 1) / m) + 1 in
  let out = Nx.zeros (Nx.dtype x) (Array.append lead [|total|]) in
  ( if batch > 0 && n > 0 then
      match Nx.dtype x with
      | Nx.Float32 -> resample_apply_c plan (array1_of (Nx.contiguous x)) batch n (array1_of out)
      | Nx.Float64 ->
          resample_apply_f64_c plan (array1_of (Nx.contiguous x)) batch n (array1_of out)
      | _ -> invalid_arg "apply: cannot resample this sample type (float32 and float64 are carried)" ) ;
  out

(* Replacement of Resample.Kernel (resample.ml:1343-1424, 1844-1909), the face
   soundml-io's decode loop binds (soundml_io.ml:639, 768, 798): the carry lives on the
   device, step returns the samples that became computable ([None] when there are
   none), flush the delayed tail.  Single owner, not domain-safe (resample.mli:271-273). *)
module Kernel = struct
  type t = { k : resample_kernel; channels : int }

  let prepare ~sample_rate ~target ~quality dtype ~channels ~max_block =
    let code =
      match dtype with
      | `Float32 -> 0
      | `Float64 -> 1
    in
    { k = resample_kernel_create (resample_plan_of ~sample_rate ~target ~quality) code channels max_block;
      channels }

  let step t chunk =
    let n = Nx.dim (Nx.ndim chunk - 1) chunk in
    let frames = resample_kernel_step_frames t.k n in
    let lead = leading_shape chunk in
    let out = Nx.zeros (Nx.dtype chunk) (Array.append lead [|frames|]) in
    if n > 0 then
      resample_kernel_step_c t.k (array1_of (Nx.contiguous chunk)) t.channels n (array1_of out) ;
    if frames = 0 then None else Some out

  let flush t dtype lead =
    let frames = resample_kernel_flush_frames t.k in
    let out = Nx.zeros dtype (Array.append lead [|frames|]) in
    resample_kernel_flush_c t.k t.channels (array1_of out) ;
    if frames = 0 then None else Some out

  let reset t = resample_kernel_reset t.k
  let destroy t = resample_kernel_destroy t.k
end

(* Replacement body of Stft.invert: the preconditions (check_synthesis,
   stft.ml:787) stay in OCaml; the library re-validates and raises the same
   messages. *)
let invert dtype c ?length z =
  let rank = Nx.ndim z in
  let frames = Nx.dim (rank - 1) z in
  let lead = Array.sub (Nx.shape z) 0 (rank - 2) in
  let batch = Array.fold_left ( * ) 1 lead in
  let out_len =
    match length with Some n -> n | None -> Stft.output_length c ~frames
  in
  let out = Nx.zeros dtype (Array.append lead [|out_len|]) in
  if batch > 0 && out_len > 0 && frames > 0 then
    invert_c (stft_plan_of c) (array1_of (Nx.contiguous z)) batch frames
      (match length with Some n -> n | None -> -1)
      (array1_of out) ;
  out

(* Replacement bodies of the phase vocoder and Effects.time_stretch (effects.ml:296):
   the library checks the rate (positive and finite) and, for time_stretch,
   invertibility, with the reference's wording. *)
let phase_vocoder c ~rate z =
  let rank = Nx.ndim z in
  if rank < 2 then
    invalid_arg
      (Printf.sprintf
         "phase_vocoder: cannot stretch a rank-%d tensor (the bin and frame axes must exist)"
         rank) ;
  let frames = Nx.dim (rank - 1) z in
  let bins = Nx.dim (rank - 2) z in
  let lead = Array.sub (Nx.shape z) 0 (rank - 1) in
  let batch = Array.fold_left ( * ) 1 (Array.sub lead 0 (rank - 2)) in
  let plan = stft_plan_of c in
  (* the rate first, then the bin axis, as the Python face orders them *)
  let out_frames = time_stretch_frames plan frames rate in
  let want = Stft.Config.bins c in
  if bins <> want then
    invalid_arg
      (Printf.sprintf
         "phase_vocoder: cannot stretch %d frequency bins of a %d-point transform (the bin \
          axis must hold fft_size / 2 + 1 = %d values)"
         bins (Stft.Config.fft_size c) want) ;
  let out = Nx.zeros (Nx.dtype z) (Array.append lead [|out_frames|]) in
  if batch > 0 && out_frames > 0 then
    phase_vocoder_c plan (array1_of (Nx.contiguous z)) batch frames rate (array1_of out) ;
  out

let time_stretch c ~rate x =
  let rank = Nx.ndim x in
  let n = Nx.dim (rank - 1) x in
  let lead = Array.sub (Nx.shape x) 0 (rank - 1) in
  let batch = Array.fold_left ( * ) 1 lead in
  let plan = stft_plan_of c in
  let length = time_stretch_length n rate in
  let out = Nx.zeros (Nx.dtype x) (Array.append lead [|length|]) in
  (* batch 0: the preconditions (invertibility) even when there is nothing to compute *)
  time_stretch_c plan (array1_of (Nx.contiguous x)) 0 n rate (array1_of out) ;
  if batch > 0 && length > 0 then
    time_stretch_c plan (array1_of (Nx.contiguous x)) batch n rate (array1_of out) ;
  out

(* Harmonic-percussive separation, librosa 0.11 decompose.hpss and effects.hpss /
   harmonic / percussive (the reference's hpss.ml).  kernel_size and margin are
   (harmonic, percussive) pairs; power = infinity gives hard masks.  The library checks
   the parameters (and, for audio, invertibility) with its own wording. *)
module Hpss = struct
  let both = 0 and harmonic_only = 1 and percussive_only = 2 and masks_only = 3

  (* [lead; parts; rest] -> the part's [lead; rest] *)
  let part t lead rest i =
    let batch = Array.fold_left ( * ) 1 lead in
    let flat = Nx.reshape (Array.append [|batch; 2|] rest) t in
    Nx.reshape (Array.append lead rest) (Nx.slice [Nx.A; Nx.R (i, i + 1)] flat)

  let run ~what ~kernel_size ~power ~margin dtype s =
    let rank = Nx.ndim s in
    if rank < 2 then
      invalid_arg
        (Printf.sprintf
           "hpss: cannot separate a rank-%d tensor (the bin and frame axes must exist)" rank) ;
    let frames = Nx.dim (rank - 1) s and bins = Nx.dim (rank - 2) s in
    let lead = Array.sub (Nx.shape s) 0 (rank - 2) in
    let batch = Array.fold_left ( * ) 1 lead in
    let win_harm, win_perc = kernel_size and margin_harm, margin_perc = margin in
    let out = Nx.zeros dtype (Array.append lead [|2; bins; frames|]) in
    let s = Nx.contiguous s in
    (* batch 0: the parameter checks even when there is nothing to compute *)
    hpss_c (array1_of s) 0 bins frames win_harm win_perc power margin_harm margin_perc what
      (array1_of out) ;
    if batch * bins * frames > 0 then
      hpss_c (array1_of s) batch bins frames win_harm win_perc power margin_harm margin_perc
        what (array1_of out) ;
    (part out lead [|bins; frames|] 0, part out lead [|bins; frames|] 1)

  (* (harmonic, percussive) of a real or complex spectrogram [...; bins; frames] *)
  let hpss ?(kernel_size = (31, 31)) ?(power = 2.) ?(margin = (1., 1.)) s =
    run ~what:both ~kernel_size ~power ~margin (Nx.dtype s) s

  (* (mask_harm, mask_perc) in the real dtype [dtype] of s *)
  let masks ?(kernel_size = (31, 31)) ?(power = 2.) ?(margin = (1., 1.)) dtype s =
    run ~what:masks_only ~kernel_size ~power ~margin dtype s

  let audio ~what ~kernel_size ~power ~margin c x =
    let n = Nx.dim (Nx.ndim x - 1) x in
    let lead = leading_shape x in
    let batch = Array.fold_left ( * ) 1 lead in
    let parts = if what = both then 2 else 1 in
    let win_harm, win_perc = kernel_size and margin_harm, margin_perc = margin in
    let plan = stft_plan_of c in
    let out = Nx.zeros (Nx.dtype x) (Array.append lead [|parts; n|]) in
    let x = Nx.contiguous x in
    hpss_audio_c plan (array1_of x) 0 n win_harm win_perc power margin_harm margin_perc what
      (array1_of out) ;
    if batch > 0 && n > 0 then
      hpss_audio_c plan (array1_of x) batch n win_harm win_perc power margin_harm margin_perc
        what (array1_of out) ;
    (out, lead, n)

  (* effects.hpss: (harmonic, percussive) signals of x [...; n] *)
  let separate ?(kernel_size = (31, 31)) ?(power = 2.) ?(margin = (1., 1.)) c x =
    let out, lead, n = audio ~what:both ~kernel_size ~power ~margin c x in
    (part out lead [|n|] 0, part out lead [|n|] 1)

  let harmonic ?(kernel_size = (31, 31)) ?(power = 2.) ?(margin = (1., 1.)) c x =
    let out, lead, n = audio ~what:harmonic_only ~kernel_size ~power ~margin c x in
    Nx.reshape (Array.append lead [|n|]) out

  let percussive ?(kernel_size = (31, 31)) ?(power = 2.) ?(margin = (1., 1.)) c x =
    let out, lead, n = audio ~what:percussive_only ~kernel_size ~power ~margin c x in
    Nx.reshape (Array.append lead [|n|]) out
end

(* Per-frame spectral descriptors, librosa 0.11 feature.spectral_centroid / _bandwidth /
   _rolloff / _flatness (the reference's spectral.ml).  [which] lists SMB_SPECTRAL_* flags;
   the result holds one [...; 1; frames] tensor per flag, in flag order.  n_fft = None
   means 2 (bins - 1); the library checks every parameter with its own wording. *)
module Spectral = struct
  let centroid = 1 and bandwidth = 2 and rolloff = 4 and flatness = 8

  let what_of which = List.fold_left ( lor ) 0 which

  let rows what = List.length (List.filter (fun f -> what land f <> 0) [centroid; bandwidth; rolloff; flatness])

  (* [lead; rows; frames] -> one [lead; 1; frames] tensor per row *)
  let split out lead frames what =
    let batch = Array.fold_left ( * ) 1 lead and k = rows what in
    let flat = Nx.reshape [|batch; k; frames|] out in
    List.init k (fun i ->
        Nx.reshape (Array.append lead [|1; frames|]) (Nx.slice [Nx.A; Nx.R (i, i + 1)] flat))

  let features ?(sample_rate = 22050.) ?n_fft ?(p = 2.) ?(norm = true) ?(roll_percent = 0.85)
      ?(amin = 1e-10) ?(power = 2.) which s =
    let rank = Nx.ndim s in
    if rank < 2 then
      invalid_arg
        (Printf.sprintf
           "spectral: cannot describe a rank-%d tensor (the bin and frame axes must exist)" rank) ;
    let frames = Nx.dim (rank - 1) s and bins = Nx.dim (rank - 2) s in
    let lead = Array.sub (Nx.shape s) 0 (rank - 2) in
    let batch = Array.fold_left ( * ) 1 lead in
    let what = what_of which in
    let n_fft = match n_fft with Some n -> n | None -> 2 * (bins - 1) in
    let out = Nx.zeros (Nx.dtype s) (Array.append lead [|rows what; frames|]) in
    let s = Nx.contiguous s in
    (* batch 0: the parameter checks even when there is nothing to compute *)
    spectral_c (array1_of s) 0 bins frames n_fft sample_rate what p norm roll_percent amin power
      (array1_of out) ;
    if batch * frames > 0 then
      spectral_c (array1_of s) batch bins frames n_fft sample_rate what p norm roll_percent amin
        power (array1_of out) ;
    split out lead frames what

  let features_audio ?(sample_rate = 22050.) ?(p = 2.) ?(norm = true) ?(roll_percent = 0.85)
      ?(amin = 1e-10) ?(power = 2.) c which x =
    let n = Nx.dim (Nx.ndim x - 1) x in
    let lead = leading_shape x in
    let batch = Array.fold_left ( * ) 1 lead in
    let what = what_of which in
    let plan = stft_plan_of c in
    let x = Nx.contiguous x in
    let probe = Nx.zeros (Nx.dtype x) [|0|] in
    spectral_audio_c plan (array1_of x) 0 n sample_rate what p norm roll_percent amin power
      (array1_of probe) ;
    let frames = Stft.frames c ~n in
    let out = Nx.zeros (Nx.dtype x) (Array.append lead [|rows what; frames|]) in
    if batch > 0 && frames > 0 then
      spectral_audio_c plan (array1_of x) batch n sample_rate what p norm roll_percent amin power
        (array1_of out) ;
    split out lead frames what
end

(* Replacement body of Convert.power_to_db / amplitude_to_db: elementwise over
   the flat storage, the top_db clamp is one whole-tensor maximum on the GPU. *)
let to_db ~amplitude ?(reference = 1.) ~amin ?top_db s =
  let out = Nx.zeros (Nx.dtype s) (Nx.shape s) in
  if Nx.numel s > 0 then
    to_db_c amplitude (array1_of (Nx.contiguous s)) reference amin
      (match top_db with Some t -> t | None -> Float.nan)
      (array1_of out) ;
  out

let mfcc stft_config mel_config ?(n_mfcc = 20) ?lifter x =
  let n = Nx.dim (Nx.ndim x - 1) x in
  let lead = leading_shape x in
  let batch = Array.fold_left ( * ) 1 lead in
  let frames = Stft.frames stft_config ~n in
  let out = Nx.zeros (Nx.dtype x) (Array.append lead [|n_mfcc; frames|]) in
  if batch > 0 && frames > 0 then
    mfcc_c (stft_plan_of stft_config) (mel_plan_of mel_config) (array1_of (Nx.contiguous x))
      batch n n_mfcc
      (match lifter with Some l -> l | None -> 0.)
      (array1_of out) ;
  out

(* The fused read of soundml-io (Soundml_io.read ~sample_rate, soundml_io.ml:742-807) on the
   device: [decode] is the caller's sf_readf_float -- it fills the staging block it is handed
   and returns the frames it wrote (0 at EOF).  Block i + 1 is decoded while block i is
   uploaded, laid out and resampled; pieces land in a device buffer and come back once, as
   planar [width; total] float32 ([total] = ceil (frames * L / M), from the file's frame
   count as Soundml_io knows it). *)
module Reader = struct
  let read ~channels ~sample_rate ~target ~mono ~quality ~frames
      ~(decode : (float, Bigarray.float32_elt) ba -> int -> int) =
    let width = if mono then 1 else channels in
    let r =
      ingest_create channels sample_rate (if target = sample_rate then 0 else target)
        (if mono then 2 else 1) (quality_code quality) 0
    in
    let block = ingest_max_block r in
    (* an upper bound of what the pieces can add up to: every piece is [width; released] *)
    let total =
      if target = sample_rate then frames
      else
        let g = let rec gcd a b = if b = 0 then a else gcd b (a mod b) in gcd sample_rate target in
        ((frames * (target / g)) + (sample_rate / g) - 1) / (sample_rate / g)
    in
    let dev = device_alloc (Stdlib.max 1 (4 * width * total)) in
    Fun.protect
      ~finally:(fun () -> device_free dev ; ingest_destroy r)
      (fun () ->
        let pieces = ref [] and at = ref 0 in
        let rec loop () =
          let got = decode (ingest_staging r channels) block in
          if got > 0 then begin
            let released = ingest_submit_frames r got in
            ingest_submit r got dev (4 * width * !at) ;
            if released > 0 then pieces := (!at, released) :: !pieces ;
            at := !at + released ;
            loop ()
          end
        in
        loop () ;
        let tail = ingest_finish_frames r in
        ingest_finish r dev (4 * width * !at) ;
        if tail > 0 then pieces := (!at, tail) :: !pieces ;
        at := !at + tail ;
        (* pieces are [width; n_i] blocks one after the other: stride them into [width; total] *)
        let flat = Nx.zeros Nx.float32 [|width * !at|] in
        ingest_result_read r dev (4 * width * !at) (array1_of flat) ;
        let out = Nx.zeros Nx.float32 [|width; !at|] in
        List.iter
          (fun (p, n) ->
            let piece = Nx.reshape [|width; n|] (Nx.slice [Nx.R (width * p, width * (p + n))] flat) in
            Nx.set_slice [Nx.A; Nx.R (p, p + n)] out piece )
          (List.rev !pieces) ;
        out )
end
