module qcoh_fortran_api
! ISO_C_BINDING interfaces for the qcoh_* extension of libqcoh.so (include/qcoh.h, group 2).
!
! The reference's own interface module, Shared/xgb_fortran_api.F90, needs NO change: its eleven
! bind(C) names (XGBoosterLoadModel ... XGBoosterFree) are exported by libqcoh.so with libxgboost's
! signatures, so `predict_OH_with_XGB` (OH_GridComp/OH_GridCompMod.F90:123-398) links against
! libqcoh.so as is.  This module adds the fused, device-resident path a patched Run1 calls
! (see fortran/OH_Run1_fused.F90 and INTEGRATION.md).
!
! NOTE: this build box has no Fortran compiler; the module is delivered as source and has been
! checked against include/qcoh.h by hand (field order / kinds) — the executable stand-in is the
! ctypes binding quickchem_b200/capi.py, which declares the same structs.
  use iso_c_binding
  implicit none

  ! qcoh_oh_config (include/qcoh.h) — OH_GridComp state + MAPL constants
  type, bind(C) :: qcoh_oh_config
     integer(c_int) :: ncol                    ! im*jm, i fastest
     integer(c_int) :: km
     real(c_float)  :: mapl_epsilon, mapl_avogad, mapl_runiv
     real(c_float)  :: mapl_radians_to_degrees, mapl_degrees_to_radians
     real(c_float)  :: ohscale                 ! self%OHscale
     integer(c_int) :: compute_once_per_day    ! 1 / 0
     real(c_float)  :: tropp_min               ! 40 hPa = 4000 Pa
     real(c_float)  :: missing                 ! -999.0
  end type qcoh_oh_config

  ! qcoh_run1_in — every pointer may be host (c_loc of the MAPL array) or device memory
  type, bind(C) :: qcoh_run1_in
     integer(c_int) :: nymd
     integer(c_int) :: need_to_call_boost
     type(c_ptr) :: T_MOD, Q_MOD, PLE_MOD, TROPP
     type(c_ptr) :: T_BST, Q_BST, PLE_BST, ZLE_BST
     type(c_ptr) :: TAUCLW, TAUCLI, FCLD, CH4, CO
     type(c_ptr) :: SCA(7)                     ! BC OC BR DU SU SS NI at wavelength_index
     type(c_ptr) :: NO2, O3, ISOP, ACET, C2H6, C3H8, PRPE, ALK4, MP, H2O2, CH2O
     type(c_ptr) :: GMITO3, GMITTO3, ALBUV, LATS, LONS
     type(c_ptr) :: OH_CLIM
     type(c_ptr) :: AREA                       ! c_null_ptr: no global-mean diagnostic
  end type qcoh_run1_in

  type, bind(C) :: qcoh_run1_out
     type(c_ptr) :: OH, OH_boost, NDWET, X, pred   ! c_null_ptr = not wanted
     type(c_ptr) :: LOSS_CH4, LOSS_CO              ! k(T)[OH] in 1/s for the CH4 / CO consumers (build-defined)
     integer(c_int) :: k1
     real(c_double) :: diag(4)
  end type qcoh_run1_out

  interface
     integer(c_int) function qcoh_set_device(device) bind(C, name="qcoh_set_device")
       import :: c_int
       integer(c_int), value :: device
     end function

     integer(c_int) function qcoh_oh_create(booster, cfg, out) bind(C, name="qcoh_oh_create")
       import :: c_int, c_ptr, qcoh_oh_config
       type(c_ptr), value   :: booster   ! BoosterHandle from XGBoosterCreate_f / XGBoosterLoadModel_f
       type(qcoh_oh_config) :: cfg
       type(c_ptr)          :: out       ! qcoh_oh_handle*
     end function

     integer(c_int) function qcoh_oh_run1(h, rin, rout) bind(C, name="qcoh_oh_run1")
       import :: c_int, c_ptr, qcoh_run1_in, qcoh_run1_out
       type(c_ptr), value  :: h
       type(qcoh_run1_in)  :: rin
       type(qcoh_run1_out) :: rout
     end function

     ! DIAG_* exports: name = "TAUCLWDN"//c_null_char etc. (include/qcoh.h)
     integer(c_int) function qcoh_oh_get_diag(h, name, out) bind(C, name="qcoh_oh_get_diag")
       import :: c_int, c_ptr, c_char
       type(c_ptr), value :: h
       character(len=1, kind=c_char), dimension(*) :: name
       type(c_ptr), value :: out   ! c_loc of the export array (host) or a device pointer
     end function

     integer(c_int) function qcoh_oh_free(h) bind(C, name="qcoh_oh_free")
       import :: c_int, c_ptr
       type(c_ptr), value :: h
     end function

     ! Opt-in month roll-over (the reference keeps the first month's booster for the whole run,
     ! OH_GridCompMod.F90:182,209,1187): pattern = self%XGBoostFilePattern//c_null_char; expands the
     ! template, takes the booster of that file from the process-wide cache and switches the handle to it.
     integer(c_int) function qcoh_oh_select_model(h, pattern, nymd, nhms, changed) bind(C, name="qcoh_oh_select_model")
       import :: c_int, c_ptr, c_char
       type(c_ptr), value :: h
       character(len=1, kind=c_char), dimension(*) :: pattern
       integer(c_int), value :: nymd, nhms
       integer(c_int)        :: changed
     end function

     integer(c_int) function qcoh_oh_set_booster(h, booster) bind(C, name="qcoh_oh_set_booster")
       import :: c_int, c_ptr
       type(c_ptr), value :: h, booster
     end function

     integer(c_int) function qcoh_model_cache_get(fname, out) bind(C, name="qcoh_model_cache_get")
       import :: c_int, c_ptr, c_char
       character(len=1, kind=c_char), dimension(*) :: fname
       type(c_ptr) :: out   ! BoosterHandle*, owned by the cache
     end function

     integer(c_int) function qcoh_expand_template(pattern, nymd, nhms, out, cap) bind(C, name="qcoh_expand_template")
       import :: c_int, c_char, c_size_t
       character(len=1, kind=c_char), dimension(*) :: pattern
       integer(c_int), value    :: nymd, nhms
       character(len=1, kind=c_char), dimension(*) :: out
       integer(c_size_t), value :: cap
     end function

     integer(c_int) function qcoh_partition_columns(ncol_global, nranks, rank, col0, ncol_local) &
          bind(C, name="qcoh_partition_columns")
       import :: c_int, c_int64_t
       integer(c_int64_t), value :: ncol_global
       integer(c_int), value     :: nranks, rank
       integer(c_int64_t)        :: col0, ncol_local
     end function

     ! NCCL all-reduce of the diagnostic partial sums: rank 0 gets the id, MPI_Bcast it, every rank joins
     integer(c_int) function qcoh_comm_get_unique_id(id) bind(C, name="qcoh_comm_get_unique_id")
       import :: c_int, c_char
       character(len=1, kind=c_char), dimension(128) :: id
     end function
     integer(c_int) function qcoh_comm_init(nranks, rank, id) bind(C, name="qcoh_comm_init")
       import :: c_int, c_char
       integer(c_int), value :: nranks, rank
       character(len=1, kind=c_char), dimension(128) :: id
     end function
     integer(c_int) function qcoh_comm_allreduce_sum_f64(values, n) bind(C, name="qcoh_comm_allreduce_sum_f64")
       import :: c_int, c_double
       real(c_double), dimension(*) :: values
       integer(c_int), value :: n
     end function
     integer(c_int) function qcoh_comm_destroy() bind(C, name="qcoh_comm_destroy")
       import :: c_int
     end function

     ! libxgboost 1.6.0's JSON-configured predict; config = '{"type": 2, "training": false, "iteration_begin": 0, '//
     ! '"iteration_end": 0, "strict_shape": false}'//c_null_char gives per-feature contributions (type 3: approximate).
     ! out_shape / out_result point at booster-owned buffers (c_f_pointer them; valid until the next predict / free):
     ! contributions are row-major [nrow][num_feature + 1], the last column the bias, i.e. shape (num_feature + 1, nrow)
     ! in Fortran order.
     integer(c_int) function XGBoosterPredictFromDMatrix(handle, dmat, config, out_shape, out_dim, out_result) &
          bind(C, name="XGBoosterPredictFromDMatrix")
       import :: c_int, c_ptr, c_char, c_int64_t
       type(c_ptr), value :: handle, dmat
       character(len=1, kind=c_char), dimension(*) :: config
       type(c_ptr) :: out_shape      ! const bst_ulong**
       integer(c_int64_t) :: out_dim ! bst_ulong*
       type(c_ptr) :: out_result     ! const float**
     end function

     ! Inplace prediction straight from a REAL(4) array, without a DMatrix (include/qcoh.h).  values is a JSON array
     ! interface, e.g. for a field XX(nrow, ncol) held feature-major as Fortran does ('//' joins):
     !   '{"data": [<address>, false], "shape": [nrow, ncol], "strides": [4, <4 * nrow>], "typestr": "<f4", "version": 3}'
     ! and config '{"type": 0, "missing": -999.0, "iteration_begin": 0, "iteration_end": 0, "strict_shape": false}',
     ! both ending in c_null_char; m must be c_null_ptr.  FromDense takes a C-contiguous host array ([nrow][ncol] in C
     ! order, i.e. XX(ncol, nrow) in Fortran) and returns a booster-owned host buffer; FromCudaArray takes device memory
     ! with any strides (the feature-major layout above) and returns a booster-owned DEVICE buffer.
     integer(c_int) function XGBoosterPredictFromDense(handle, values, config, m, out_shape, out_dim, out_result) &
          bind(C, name="XGBoosterPredictFromDense")
       import :: c_int, c_ptr, c_char, c_int64_t
       type(c_ptr), value :: handle, m
       character(len=1, kind=c_char), dimension(*) :: values, config
       type(c_ptr) :: out_shape      ! const bst_ulong**
       integer(c_int64_t) :: out_dim ! bst_ulong*
       type(c_ptr) :: out_result     ! const float**
     end function

     integer(c_int) function XGBoosterPredictFromCudaArray(handle, values, config, m, out_shape, out_dim, out_result) &
          bind(C, name="XGBoosterPredictFromCudaArray")
       import :: c_int, c_ptr, c_char, c_int64_t
       type(c_ptr), value :: handle, m
       character(len=1, kind=c_char), dimension(*) :: values, config
       type(c_ptr) :: out_shape      ! const bst_ulong**
       integer(c_int64_t) :: out_dim ! bst_ulong*
       type(c_ptr) :: out_result     ! const float** (device memory)
     end function

     ! SHAP interaction values of a DMatrix into a DEVICE buffer of nrow * (num_feature + 1)**2 floats (out_dev, e.g. from
     ! qcoh_device_alloc): row-major [nrow][i][j], i the conditioning feature, index num_feature the bias, i.e.
     ! M(j, i, row) in Fortran order.  approximate /= 0 gives libxgboost's type 5; ntree_limit 0 = all trees (C unsigned:
     ! pass a non-negative value).  Asynchronous: qcoh_device_synchronize before reading.  Explain a slab of rows at a
     ! time: each row takes 3136 B of output at 27 features.
     integer(c_int) function qcoh_booster_predict_interactions_device(handle, dmat, approximate, ntree_limit, out_dev) &
          bind(C, name="qcoh_booster_predict_interactions_device")
       import :: c_int, c_ptr
       type(c_ptr), value :: handle, dmat
       integer(c_int), value :: approximate, ntree_limit
       type(c_ptr), value :: out_dev
     end function

     function XGBGetLastError_c() bind(C, name="XGBGetLastError") result(msg)
       import :: c_ptr
       type(c_ptr) :: msg
     end function
  end interface

contains

  ! Fortran string copy of the library's last error (for _ASSERT messages)
  function qcoh_last_error() result(s)
    character(len=:), allocatable :: s
    character(kind=c_char), pointer :: p(:)
    type(c_ptr) :: cp
    integer :: n
    cp = XGBGetLastError_c()
    s = ''
    if (.not. c_associated(cp)) return
    call c_f_pointer(cp, p, [1024])
    n = 0
    do while (n < 1024)
       if (p(n+1) == c_null_char) exit
       n = n + 1
    end do
    allocate(character(len=n) :: s)
    s = transfer(p(1:n), s)
  end function qcoh_last_error

end module qcoh_fortran_api
