!> Drop-in replacement for the reference's `lbfgsb_module` (src/lbfgsb.f90:46-58) that forwards
!! `setulb` to the B200 engine through the C ABI of include/lbfgsb_b200.h.
!!
!! * `setulb`      -- same name, argument list and `task` protocol as src/lbfgsb.f90:88-89.
!!                    Host arrays in / out; the engine stages them on the GPU.  `wa` / `iwa` are
!!                    accepted and ignored (the workspace lives in HBM).
!! * `setulb_dev`  -- x, l, u, nbd, g are CUDA device pointers (type(c_ptr), value); the caller's
!!                    f/g evaluation and the whole iteration stay on the device.
!! * `lbfgsp_wp`   -- the real kind, as exported by the reference (src/lbfgsb.f90:50).
!!
!! Build: compile with -DREAL32 for the single-precision engine (the analogue of
!! src/lbfgsb_kinds_module.F90:29-37), default is real64; link with -llbfgsb_b200.
!!
!! NOTE: this image has no Fortran compiler, so this file is shipped as source only; the same C
!! symbols are exercised with Fortran-shaped arguments (by-reference scalars, blank-padded
!! character(60), 4-byte logicals) by tests/ through ctypes.  See INTEGRATION.md.
module lbfgsb_module

   use, intrinsic :: iso_c_binding
   use, intrinsic :: iso_fortran_env, only: real32, real64

   implicit none
   private

#ifdef REAL32
   integer, parameter, public :: lbfgsp_wp = real32
#else
   integer, parameter, public :: lbfgsp_wp = real64
#endif
   integer, parameter :: wp = lbfgsp_wp

   public :: setulb, setulb_dev
   public :: lbfgsb_dev_create, lbfgsb_dev_destroy, lbfgsb_host_release
   public :: lbfgsb_dev_set_tie_limit, lbfgsb_dev_checkpoint_write, lbfgsb_dev_checkpoint_read
   public :: lbfgsb_minimize_graph_dev, lbfgsb_batch_minimize_graph_dev
   public :: lbfgsb_batch_create, lbfgsb_batch_destroy, setulb_batch_dev, lbfgsb_batch_counts, lbfgsb_batch_get_iwhere

   interface

#ifdef REAL32
      subroutine c_setulb(n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, &
                          isave, dsave, itfile, itfile_len) bind(C, name='lbfgsb_setulb_f32')
#else
      subroutine c_setulb(n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, &
                          isave, dsave, itfile, itfile_len) bind(C, name='lbfgsb_setulb_f64')
#endif
         import :: c_int32_t, c_char, c_ptr, wp
         integer(c_int32_t), intent(in) :: n, m, iprint
         real(wp), intent(inout) :: x(*), f, g(*), wa(*), dsave(29)
         real(wp), intent(in) :: l(*), u(*), factr, pgtol
         integer(c_int32_t), intent(in) :: nbd(*)
         integer(c_int32_t), intent(inout) :: iwa(*), lsave(4), isave(44)
         character(kind=c_char), intent(inout) :: task(60), csave(60)
         type(c_ptr), value :: itfile
         integer(c_int32_t), value :: itfile_len
      end subroutine c_setulb

#ifdef REAL32
      subroutine c_setulb_dev(h, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave) &
         bind(C, name='lbfgsb_setulb_dev_f32')
#else
      subroutine c_setulb_dev(h, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave) &
         bind(C, name='lbfgsb_setulb_dev_f64')
#endif
         import :: c_int32_t, c_char, c_ptr, wp
         type(c_ptr), value :: h, x, l, u, nbd, g      ! opaque handle and CUDA device pointers
         real(wp), intent(inout) :: f, dsave(29)
         real(wp), intent(in) :: factr, pgtol
         integer(c_int32_t), intent(in) :: iprint
         integer(c_int32_t), intent(inout) :: lsave(4), isave(44)
         character(kind=c_char), intent(inout) :: task(60), csave(60)
      end subroutine c_setulb_dev

      function lbfgsb_dev_create(n, m, real_kind, cuda_stream) result(h) bind(C, name='lbfgsb_dev_create')
         import :: c_int64_t, c_int32_t, c_ptr
         integer(c_int64_t), value :: n
         integer(c_int32_t), value :: m, real_kind
         type(c_ptr), value :: cuda_stream
         type(c_ptr) :: h
      end function lbfgsb_dev_create

      subroutine lbfgsb_dev_destroy(h) bind(C, name='lbfgsb_dev_destroy')
         import :: c_ptr
         type(c_ptr), value :: h
      end subroutine lbfgsb_dev_destroy

      subroutine lbfgsb_host_release(isave) bind(C, name='lbfgsb_host_release')
         import :: c_int32_t
         integer(c_int32_t), intent(inout) :: isave(44)
      end subroutine lbfgsb_host_release

      !> Heap replay of equal breakpoints at the exit of the Cauchy search (hpsolb's pop order, src/lbfgsb.f90:2079-2157):
      !> up to max_breakpoints breakpoints per call (default 2**28, 2**26 on a sharded workspace; 0 = ties in variable order).
      subroutine lbfgsb_dev_set_tie_limit(h, max_breakpoints) bind(C, name='lbfgsb_dev_set_tie_limit')
         import :: c_ptr, c_int64_t
         type(c_ptr), value :: h
         integer(c_int64_t), value :: max_breakpoints
      end subroutine lbfgsb_dev_set_tie_limit

      !> Device workspace to / from a file (the reference's wa, iwa); path is a C string (trim(name)//c_null_char).
      function lbfgsb_dev_checkpoint_write(h, path) result(rc) bind(C, name='lbfgsb_dev_checkpoint_write')
         import :: c_ptr, c_char, c_int
         type(c_ptr), value :: h
         character(kind=c_char), intent(in) :: path(*)
         integer(c_int) :: rc
      end function lbfgsb_dev_checkpoint_write
      function lbfgsb_dev_checkpoint_read(h, path) result(rc) bind(C, name='lbfgsb_dev_checkpoint_read')
         import :: c_ptr, c_char, c_int
         type(c_ptr), value :: h
         character(kind=c_char), intent(in) :: path(*)
         integer(c_int) :: rc
      end function lbfgsb_dev_checkpoint_read

      !> The caller's loop kept on the device (one CUDA-graph launch per iteration step): fg is a C function pointer
      !> int fg(void* user, int64_t n, const real* x_dev, real* g_dev, real* f_dev, void* cuda_stream) that only enqueues
      !> kernels and leaves f in device memory (c_funloc of a bind(C) procedure).
#ifdef REAL32
      function lbfgsb_minimize_graph_dev(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, f, g, task, csave, &
                                         lsave, isave, dsave) result(rc) bind(C, name='lbfgsb_minimize_graph_dev_f32')
#else
      function lbfgsb_minimize_graph_dev(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, f, g, task, csave, &
                                         lsave, isave, dsave) result(rc) bind(C, name='lbfgsb_minimize_graph_dev_f64')
#endif
         import :: c_int32_t, c_char, c_ptr, c_funptr, c_int, wp
         type(c_ptr), value :: h, x, l, u, nbd, g, user
         type(c_funptr), value :: fg
         real(wp), value :: factr, pgtol
         integer(c_int32_t), value :: max_iter, max_fg
         real(wp), intent(inout) :: f, dsave(29)
         character(kind=c_char), intent(inout) :: task(60), csave(60)
         integer(c_int32_t), intent(inout) :: lsave(4), isave(44)
         integer(c_int) :: rc
      end function lbfgsb_minimize_graph_dev

      !> The whole task loop of a batch on the device (CUDA-graph launches of up to 128 calls each); every problem starts
      !> from 'START'.  fg is a C function pointer int fg(void* user, int32_t nprob, int64_t n, const real* x_dev,
      !> real* g_dev, real* f_dev, const int32_t* mask_dev, void* cuda_stream) that only enqueues kernels for the problems
      !> with mask_dev(p) = 1 (c_funloc of a bind(C) procedure).  Arrays as for setulb_batch_dev; f is a device pointer.
#ifdef REAL32
      function lbfgsb_batch_minimize_graph_dev(h, x, l, u, nbd, f, g, fg, user, factr, pgtol, max_iter, max_fg, task, &
         csave, lsave, isave, dsave) result(rc) bind(C, name='lbfgsb_batch_minimize_graph_f32')
#else
      function lbfgsb_batch_minimize_graph_dev(h, x, l, u, nbd, f, g, fg, user, factr, pgtol, max_iter, max_fg, task, &
         csave, lsave, isave, dsave) result(rc) bind(C, name='lbfgsb_batch_minimize_graph_f64')
#endif
         import :: c_int32_t, c_char, c_ptr, c_funptr, c_int, wp
         type(c_ptr), value :: h, x, l, u, nbd, f, g, user
         type(c_funptr), value :: fg
         real(wp), value :: factr, pgtol
         integer(c_int32_t), value :: max_iter, max_fg
         character(kind=c_char), intent(inout) :: task(60, *), csave(60, *)
         integer(c_int32_t), intent(inout) :: lsave(4, *), isave(44, *)
         real(wp), intent(inout) :: dsave(29, *)
         integer(c_int) :: rc
      end function lbfgsb_batch_minimize_graph_dev

      !> Batched small problems: nprob independent problems of the same n and m, one call advances every problem from
      !> its own task to its next return point (the caller's loop of test/driver1.f90:263-292, many times over).
      !> task, csave are (60, nprob) characters, lsave (4, nprob), isave (44, nprob), dsave (29, nprob); x, l, u, g, nbd
      !> are CUDA device pointers to (n, nprob) arrays and f to a device array (nprob).
      function lbfgsb_batch_create(nprob, n, m, real_kind, cuda_stream) result(h) bind(C, name='lbfgsb_batch_create')
         import :: c_int64_t, c_int32_t, c_ptr
         integer(c_int32_t), value :: nprob, m, real_kind
         integer(c_int64_t), value :: n
         type(c_ptr), value :: cuda_stream
         type(c_ptr) :: h
      end function lbfgsb_batch_create
      subroutine lbfgsb_batch_destroy(h) bind(C, name='lbfgsb_batch_destroy')
         import :: c_ptr
         type(c_ptr), value :: h
      end subroutine lbfgsb_batch_destroy
#ifdef REAL32
      subroutine setulb_batch_dev(h, x, l, u, nbd, f, g, factr, pgtol, task, csave, lsave, isave, dsave) &
         bind(C, name='lbfgsb_batch_setulb_dev_f32')
#else
      subroutine setulb_batch_dev(h, x, l, u, nbd, f, g, factr, pgtol, task, csave, lsave, isave, dsave) &
         bind(C, name='lbfgsb_batch_setulb_dev_f64')
#endif
         import :: c_int32_t, c_char, c_ptr, wp
         type(c_ptr), value :: h, x, l, u, nbd, f, g
         real(wp), intent(in) :: factr, pgtol
         character(kind=c_char), intent(inout) :: task(60, *), csave(60, *)
         integer(c_int32_t), intent(inout) :: lsave(4, *), isave(44, *)
         real(wp), intent(inout) :: dsave(29, *)
      end subroutine setulb_batch_dev
      function lbfgsb_batch_counts(h, n_fg, n_newx, n_done) result(rc) bind(C, name='lbfgsb_batch_counts')
         import :: c_ptr, c_int32_t, c_int
         type(c_ptr), value :: h
         integer(c_int32_t), intent(out) :: n_fg, n_newx, n_done
         integer(c_int) :: rc
      end function lbfgsb_batch_counts
      !> iwhere of every problem, (n, nprob) on the host: what the reference keeps in iwa(2n+1:3n).
      function lbfgsb_batch_get_iwhere(h, iwhere) result(rc) bind(C, name='lbfgsb_batch_get_iwhere')
         import :: c_ptr, c_int32_t, c_int
         type(c_ptr), value :: h
         integer(c_int32_t), intent(out) :: iwhere(*)
         integer(c_int) :: rc
      end function lbfgsb_batch_get_iwhere

   end interface

contains

   !> Same interface as the reference's setulb (src/lbfgsb.f90:88-89).
   subroutine setulb(n, m, x, l, u, Nbd, f, g, Factr, Pgtol, Wa, Iwa, Task, Iprint, Csave, Lsave, Isave, Dsave, &
                     iteration_file)
      integer, intent(in) :: n, m
      real(wp), intent(inout) :: x(n), f, g(n)
      real(wp), intent(in) :: l(n), u(n), Factr, Pgtol
      integer, intent(in) :: Nbd(n), Iprint
      real(wp) :: Wa(*)
      integer :: Iwa(*)
      character(len=60) :: Task, Csave
      logical :: Lsave(4)
      integer :: Isave(44)
      real(wp) :: Dsave(29)
      character(len=*), intent(in), optional :: iteration_file

      character(kind=c_char) :: ctask(60), ccsave(60)
      integer(c_int32_t) :: clsave(4)
      character(kind=c_char, len=:), allocatable, target :: fname
      integer :: i

      do i = 1, 60
         ctask(i) = Task(i:i)
         ccsave(i) = Csave(i:i)
      end do
      clsave = merge(1_c_int32_t, 0_c_int32_t, Lsave)
      if (present(iteration_file)) then
         fname = iteration_file
         call c_setulb(int(n, c_int32_t), int(m, c_int32_t), x, l, u, Nbd, f, g, Factr, Pgtol, Wa, Iwa, ctask, &
                       int(Iprint, c_int32_t), ccsave, clsave, Isave, Dsave, c_loc(fname), &
                       int(len(fname), c_int32_t))
      else
         call c_setulb(int(n, c_int32_t), int(m, c_int32_t), x, l, u, Nbd, f, g, Factr, Pgtol, Wa, Iwa, ctask, &
                       int(Iprint, c_int32_t), ccsave, clsave, Isave, Dsave, c_null_ptr, 0_c_int32_t)
      end if
      do i = 1, 60
         Task(i:i) = ctask(i)
         Csave(i:i) = ccsave(i)
      end do
      Lsave = clsave /= 0
   end subroutine setulb

   !> Device-pointer variant: `h` from lbfgsb_dev_create(n, m, kind, stream); x, l, u, nbd, g are
   !! CUDA device addresses (e.g. c_devloc of CUDA Fortran arrays, or pointers obtained from C).
   subroutine setulb_dev(h, x, l, u, nbd, f, g, Factr, Pgtol, Task, Iprint, Csave, Lsave, Isave, Dsave)
      type(c_ptr), intent(in) :: h, x, l, u, nbd, g
      real(wp), intent(inout) :: f
      real(wp), intent(in) :: Factr, Pgtol
      integer, intent(in) :: Iprint
      character(len=60) :: Task, Csave
      logical :: Lsave(4)
      integer :: Isave(44)
      real(wp) :: Dsave(29)

      character(kind=c_char) :: ctask(60), ccsave(60)
      integer(c_int32_t) :: clsave(4)
      integer :: i

      do i = 1, 60
         ctask(i) = Task(i:i)
         ccsave(i) = Csave(i:i)
      end do
      clsave = merge(1_c_int32_t, 0_c_int32_t, Lsave)
      call c_setulb_dev(h, x, l, u, nbd, f, g, Factr, Pgtol, ctask, int(Iprint, c_int32_t), ccsave, clsave, &
                        Isave, Dsave)
      do i = 1, 60
         Task(i:i) = ctask(i)
         Csave(i:i) = ccsave(i)
      end do
      Lsave = clsave /= 0
   end subroutine setulb_dev

end module lbfgsb_module
