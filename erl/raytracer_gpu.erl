%% raytracer_gpu.erl -- GPU tracing functions for plouj/eraytracer (B200, sm_100a).
%%
%% Drop-in for the 4-arity "tracing function" seam of raytracer.erl:
%%     Fun(Width, Height, Scene, Recursion_depth) -> [{Index, {R,G,B}}]
%% (tracing_function/1, raytracer.erl:714-719; called at raytracer.erl:728-732).
%%
%% The only change needed in raytracer.erl is two clauses in tracing_function/1:
%%     tracing_function(gpu) -> fun raytracer_gpu:raytraced_pixel_list_gpu/4;
%%     tracing_function(gpu_distributed) -> fun raytracer_gpu:raytraced_pixel_list_gpu_distributed/4;
%% after which   erl -noinput -run raytracer standalone 1920 1080 out.ppm 1 gpu   works.
%%
%% NOTE: written without an Erlang/OTP installation (none in the build image): it has never been
%% compiled by erlc or loaded by a BEAM.  Its sequential functions ARE evaluated by oracle/erlref.py
%% (the Erlang evaluator the reference's own run_tests/0 passes under) with stand-ins for the NIFs:
%% the tracing function returns the reference's pixel list, error tuples become exits, and
%% write_binary_to_ppm/4 writes the reference writer's text, and render_binary/5 (one linked process
%% per GPU, selective receive) uploads once, clones for the other GPUs and deals the row bands into
%% one frame under the evaluator's sequential process model (tests/test_erl_reference.py).
-module(raytracer_gpu).
-export([raytraced_pixel_list_gpu/4,
         raytraced_pixel_list_gpu_distributed/4,
         render_binary/5,
         write_binary_to_ppm/4,
         device_count/0, scene_info/1, scene_upload/2, scene_clone/2, render/5, render_pixel_list/5,
         frame_alloc/3, render_into/4, frame_binary/1,
         look_at/2]).
-on_load(init/0).

init() ->
    PrivDir = case code:priv_dir(?MODULE) of
                  {error, _} -> "priv";
                  Dir -> Dir
              end,
    erlang:load_nif(filename:join(PrivDir, "raytracer_gpu"), 0).

%% ---- NIF stubs (c_src/raytracer_gpu_nif.c) ---------------------------------
%% Opts of render/5, render_into/4, render_pixel_list/5 (and so of render_binary/5): a proplist of
%%   {format, rgb8|f32|f64}, {accel, auto|exact|linear|bvh|bvh_mega|grid}, {part, {BandRows, NParts, Part}},
%%   {camera, #camera{}}, {supersample, N}: N x N rays per pixel (N an integer in 1..8), each pixel the
%%   average of the N*N pixels of the (N*Width) x (N*Height) frame that fall in it, and {camera_rotation, true}:
%%   the primary rays turned by the camera's rotation {vector, Rx, Ry, Rz} in degrees, M = Ry . Rx . Rz about the
%%   world axes (+y is down: {vector, 0, 90, 0} looks along +x, {vector, 90, 0, 0} up; see look_at/2).  The
%%   reference ignores the rotation, and so does the default {camera_rotation, false}.  Anything else is badarg.
device_count() -> erlang:nif_error(nif_not_loaded).
scene_info(_Scene) -> erlang:nif_error(nif_not_loaded).
scene_upload(_Scene, _Device) -> erlang:nif_error(nif_not_loaded).
scene_clone(_Handle, _Device) -> erlang:nif_error(nif_not_loaded).
frame_alloc(_Width, _Height, _Format) -> erlang:nif_error(nif_not_loaded).
render_into(_Handle, _Frame, _Depth, _Opts) -> erlang:nif_error(nif_not_loaded).
frame_binary(_Frame) -> erlang:nif_error(nif_not_loaded).
render(_Handle, _Width, _Height, _Depth, _Opts) -> erlang:nif_error(nif_not_loaded).
render_pixel_list(_Handle, _Width, _Height, _Depth, _Opts) -> erlang:nif_error(nif_not_loaded).

%% ---- tracing functions -------------------------------------------------------
%% Same clauses and guards as raytraced_pixel_list_simple/4 (raytracer.erl:86-99).
raytraced_pixel_list_gpu(0, 0, _, _) ->
    done;
raytraced_pixel_list_gpu(Width, Height, Scene, Recursion_depth)
  when Width > 0, Height > 0 ->
    {ok, Handle} = ok_or_exit(scene_upload(Scene, 0)),
    case render_pixel_list(Handle, Width, Height, Recursion_depth, []) of
        {error, Reason} -> exit({raytracer_gpu, Reason});
        Pixels when is_list(Pixels) -> Pixels
    end.

%% Row bands dealt round-robin to every GPU of the box; one Erlang process per GPU calls
%% the dirty NIF and its GPU fills its rows of ONE shared frame (the role of
%% distribute_work/7 + master/3, raytracer.erl:139-161, without one message per pixel).
raytraced_pixel_list_gpu_distributed(0, 0, _, _) ->
    done;
raytraced_pixel_list_gpu_distributed(Width, Height, Scene, Recursion_depth)
  when Width > 0, Height > 0 ->
    Frame = render_binary(Width, Height, Scene, Recursion_depth, [{format, f64}]),
    pixel_list_from_f64(Frame, 0, []).

%% Whole frame as a binary (rgb8 by default): the scalable return type.
%% The scene term is decoded and its acceleration structures are built ONCE (scene_upload on device 0);
%% the other GPUs get copies (scene_clone).  One page-locked frame is shared by all parts: every GPU copies
%% its row bands to their place in it, and the result is that memory as a binary — no per-part frames and
%% no stitching on the Erlang side.
render_binary(Width, Height, Scene, Recursion_depth, Opts) when Width > 0, Height > 0 ->
    {ok, N} = ok_or_exit(device_count()),
    Format = proplists:get_value(format, Opts, rgb8),
    {ok, H0} = ok_or_exit(scene_upload(Scene, 0)),
    Handles = [H0 | [begin {ok, H} = ok_or_exit(scene_clone(H0, Dev)), H end || Dev <- lists:seq(1, N - 1)]],
    {ok, Frame} = ok_or_exit(frame_alloc(Width, Height, Format)),
    BandRows = 8,
    Parent = self(),
    Pids = [spawn_link(fun() ->
                Parent ! {self(), render_into(H, Frame, Recursion_depth,
                                              [{part, {BandRows, N, Part}} | Opts])}
            end) || {Part, H} <- lists:zip(lists:seq(0, N - 1), Handles)],
    [receive {Pid, ok} -> ok;
             {Pid, {error, Reason}} -> exit({raytracer_gpu, Reason})
     end || Pid <- Pids],
    frame_binary(Frame).

pixel_list_from_f64(<<>>, _I, Acc) ->
    lists:reverse(Acc);
pixel_list_from_f64(<<R:64/float-native, G:64/float-native, B:64/float-native, Rest/binary>>, I, Acc) ->
    pixel_list_from_f64(Rest, I + 1, [{I, {R, G, B}} | Acc]).

%% P3 writer over an rgb8 frame binary: the bytes write_pixels_to_ppm/5 (raytracer.erl:668-685)
%% produces, without the W*H-element pixel list and the io:format per pixel.
write_binary_to_ppm(Width, Height, FrameRgb8, Filename) ->
    Body = [[integer_to_list(V), $\s] || <<V:8>> <= FrameRgb8],
    file:write_file(Filename,
                    [io_lib:format("P3~n~p ~p~n~p~n", [Width, Height, 255]), Body]).

%% The camera rotation whose forward axis points from Location to Target, for {camera_rotation, true}:
%% Ry = atan2(Fx, Fz), Rx = atan2(-Fy, sqrt(Fx*Fx + Fz*Fz)) of F = Target - Location, in degrees, no roll.
look_at({vector, Lx, Ly, Lz}, {vector, Tx, Ty, Tz}) ->
    Fx = Tx - Lx,
    Fy = Ty - Ly,
    Fz = Tz - Lz,
    Ry = math:atan2(Fx, Fz),
    Rx = math:atan2(-Fy, math:sqrt(Fx * Fx + Fz * Fz)),
    {vector, Rx * 180.0 / math:pi(), Ry * 180.0 / math:pi(), 0.0}.

ok_or_exit({ok, _} = Ok) -> Ok;
ok_or_exit({error, Reason}) -> exit({raytracer_gpu, Reason}).
